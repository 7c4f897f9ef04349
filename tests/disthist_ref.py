"""numpy restatement of mmm_disthist_add: for every pair i < j whose beads both have a bin, d2 = (dx*dx + dy*dy) +
dz*dz in FP64, in this order (numpy rounds every ufunc operation on its own, no FMA), falls in the cell
h = #{k : e_k * e_k <= d2} (np.searchsorted on the FP64 squares, side="right"), and the count of the bin pair
p = min(bin_i, bin_j), q = max at row tri(p, q) of np.triu_indices(B) and column h grows by one.  Blocked over rows
of the pair triangle so that memory stays bounded."""
from __future__ import annotations

import numpy as np


def tri_index(p, q, n_bins):
    """Row of the bin pair p <= q in np.triu_indices(n_bins) order."""
    p, q = np.asarray(p, np.int64), np.asarray(q, np.int64)
    return p * n_bins - p * (p - 1) // 2 + (q - p)


def hist_counts(x, bins, n_bins, edges, block_pairs=1 << 22):
    """counts uint64 [B (B + 1) / 2, E + 1] as mmm_disthist_read returns them after one add."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    bins = np.asarray(bins, np.int64)
    e2 = np.asarray(edges, np.float64) ** 2
    h_cells = len(e2) + 1
    rows_total = n_bins * (n_bins + 1) // 2
    keep = np.flatnonzero(bins >= 0)  # pairs of binned beads only; i < j in the original order
    xk, bk = x[keep], bins[keep]
    m = len(keep)
    counts = np.zeros(rows_total * h_cells, np.uint64)
    r0 = 0
    while r0 < m - 1:
        rows = max(1, min(m - 1 - r0, block_pairs // max(m - r0, 1)))
        ii, jj = np.nonzero(np.arange(r0, r0 + rows)[:, None] < np.arange(r0, m)[None, :])
        ii += r0
        jj += r0
        d = xk[ii] - xk[jj]
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        h = np.searchsorted(e2, d2, side="right")
        row = tri_index(np.minimum(bk[ii], bk[jj]), np.maximum(bk[ii], bk[jj]), n_bins)
        counts += np.bincount(row * h_cells + h, minlength=rows_total * h_cells).astype(np.uint64)
        r0 += rows
    return counts.reshape(rows_total, h_cells)


def brute_hist(x, bins, n_bins, edges):
    """The same by a plain double loop over the pairs and a linear scan of the edges (small n only)."""
    x = np.asarray(x, np.float64)
    edges = [float(e) for e in edges]
    counts = np.zeros((n_bins * (n_bins + 1) // 2, len(edges) + 1), np.uint64)
    n = len(x)
    for i in range(n):
        for j in range(i + 1, n):
            p, q = int(bins[i]), int(bins[j])
            if p < 0 or q < 0:
                continue
            dx, dy, dz = x[i, 0] - x[j, 0], x[i, 1] - x[j, 1], x[i, 2] - x[j, 2]
            d2 = (dx * dx + dy * dy) + dz * dz
            h = sum(1 for e in edges if e * e <= d2)
            counts[int(tri_index(min(p, q), max(p, q), n_bins)), h] += 1
    return counts
