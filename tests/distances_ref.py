"""numpy restatement of mmm_distance_map: for every pair i < j whose beads both have a bin,
d2 = (dx*dx + dy*dy) + dz*dz in FP64, in this order (numpy rounds every ufunc operation on its own, no FMA),
d = np.sqrt(d2) (correctly rounded, as __dsqrt_rn), each quantised with np.rint(v * 2^24) (half to even, as
__double2ll_rn; the scaling is exact), summed in uint64 with np.add.at at (bin_i, bin_j) and, off the
diagonal, at (bin_j, bin_i).  Blocked over rows of the pair triangle so that memory stays bounded."""
from __future__ import annotations

import numpy as np

SCALE = 2.0 ** 24


def _q(v):
    return np.rint(v * SCALE).astype(np.int64).astype(np.uint64)


def pair_terms(x, i, j):
    """(qd, qd2) uint64 of the pairs (i, j)."""
    d = x[i] - x[j]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    return _q(np.sqrt(d2)), _q(d2)


def add_pairs(dsum, d2sum, bi, bj, qd, qd2):
    """np.add.at of the pair terms into both orientations of the maps (the diagonal once)."""
    np.add.at(dsum, (bi, bj), qd)
    np.add.at(d2sum, (bi, bj), qd2)
    off = bi != bj
    np.add.at(dsum, (bj[off], bi[off]), qd[off])
    np.add.at(d2sum, (bj[off], bi[off]), qd2[off])


def distance_sums(x, bins, n_bins, block_pairs=1 << 22):
    """(dist_sum, dist2_sum) uint64 (n_bins, n_bins) as mmm_distance_map returns them."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    bins = np.asarray(bins, np.int64)
    keep = np.flatnonzero(bins >= 0)  # pairs of binned beads only; i < j in the original order
    xk, bk = x[keep], bins[keep]
    m = len(keep)
    dsum = np.zeros((n_bins, n_bins), np.uint64)
    d2sum = np.zeros((n_bins, n_bins), np.uint64)
    r0 = 0
    while r0 < m - 1:
        rows = max(1, min(m - 1 - r0, block_pairs // max(m - r0, 1)))
        ii, jj = np.nonzero(np.arange(r0, r0 + rows)[:, None] < np.arange(r0, m)[None, :])
        ii += r0
        jj += r0
        qd, qd2 = pair_terms(xk, ii, jj)
        add_pairs(dsum, d2sum, bk[ii], bk[jj], qd, qd2)
        r0 += rows
    return dsum, d2sum


def brute_distance_sums(x, bins, n_bins):
    """The same by a plain double loop over the pairs, Python integers (small n only)."""
    x = np.asarray(x, np.float64)
    dsum = np.zeros((n_bins, n_bins), np.uint64)
    d2sum = np.zeros((n_bins, n_bins), np.uint64)
    n = len(x)
    for i in range(n):
        for j in range(i + 1, n):
            p, q = int(bins[i]), int(bins[j])
            if p < 0 or q < 0:
                continue
            dx, dy, dz = x[i, 0] - x[j, 0], x[i, 1] - x[j, 1], x[i, 2] - x[j, 2]
            d2 = (dx * dx + dy * dy) + dz * dz
            qd, qd2 = np.uint64(round(float(np.sqrt(d2)) * SCALE)), np.uint64(round(d2 * SCALE))
            dsum[p, q] += qd
            d2sum[p, q] += qd2
            if p != q:
                dsum[q, p] += qd
                d2sum[q, p] += qd2
    return dsum, d2sum


def block_sums(x, bins, p, q):
    """(dist_sum, dist2_sum) of the single entry (p, q): every pair with one bead in bin p, the other in q."""
    x = np.asarray(x, np.float64)
    bins = np.asarray(bins)
    a, b = np.flatnonzero(bins == p), np.flatnonzero(bins == q)
    if p == q:
        ii, jj = np.triu_indices(len(a), k=1)
        i, j = a[ii], a[jj]
    else:
        i, j = np.repeat(a, len(b)), np.tile(b, len(a))
    qd, qd2 = pair_terms(x, i, j)
    return int(qd.sum(dtype=np.uint64)), int(qd2.sum(dtype=np.uint64))
