"""numpy restatement of mmm_gam_add: bead i lies in slice k iff |s| <= h with s = ((nx*x + ny*y) + nz*z) - o in
FP64, in this order (numpy rounds every ufunc operation on its own, no FMA); bin p is detected in slice k iff a bead
with bin p lies in it (bin -1: left out); the count of the bin pair p <= q at row tri(p, q) of np.triu_indices(B)
is the number of slices in which both are detected, and empty the number of slices in which no bin is.  Blocked
over slices so that memory stays bounded."""
from __future__ import annotations

import numpy as np


def detection(x, bins, n_bins, planes, h, block_slices=None):
    """bool [S, B]: bin p detected in slice k."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    bins = np.asarray(bins, np.int64)
    planes = np.asarray(planes, np.float64).reshape(-1, 4)
    keep = np.flatnonzero(bins >= 0)
    xk, bk = x[keep], bins[keep]
    s_total = len(planes)
    if block_slices is None:
        block_slices = max(1, (1 << 22) // max(len(keep), 1))
    det = np.zeros((s_total, n_bins), bool)
    for k0 in range(0, s_total, block_slices):
        p = planes[k0:k0 + block_slices]
        s = ((p[:, None, 0] * xk[None, :, 0] + p[:, None, 1] * xk[None, :, 1]) + p[:, None, 2] * xk[None, :, 2]) \
            - p[:, None, 3]
        inside = np.abs(s) <= h  # [block, beads]
        kk, ii = np.nonzero(inside)
        det[k0 + kk, bk[ii]] = True
    return det


def gam_add(x, bins, n_bins, planes, h):
    """(counts uint64 [B (B + 1) / 2], empty) of one add, as mmm_gam_read returns them after it."""
    det = detection(x, bins, n_bins, planes, h)
    d = det.astype(np.float32)
    gram = d.T @ d  # exact: sums of 0 / 1 of at most 65536 slices, below 2^24
    iu = np.triu_indices(n_bins)
    return np.rint(gram[iu]).astype(np.uint64), int(np.count_nonzero(~det.any(axis=1)))


def brute_gam(x, bins, n_bins, planes, h):
    """The same by plain loops over slices, beads and bin pairs (small inputs only)."""
    x = np.asarray(x, np.float64)
    planes = np.asarray(planes, np.float64).reshape(-1, 4)
    counts = np.zeros(n_bins * (n_bins + 1) // 2, np.uint64)
    empty = 0
    for nx, ny, nz, o in planes:
        hit = set()
        for i in range(len(x)):
            b = int(bins[i])
            if b < 0:
                continue
            s = ((float(nx) * float(x[i, 0]) + float(ny) * float(x[i, 1])) + float(nz) * float(x[i, 2])) - float(o)
            if abs(s) <= h:
                hit.add(b)
        if not hit:
            empty += 1
        row = 0
        for p in range(n_bins):
            for q in range(p, n_bins):
                if p in hit and q in hit:
                    counts[row] += 1
                row += 1
    return counts, empty
