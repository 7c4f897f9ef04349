"""numpy restatement of mmm_contacts: a contact is a pair i < j with d2 < rc * rc, where
d2 = (dx*dx + dy*dy) + dz*dz in FP64, in this order.  numpy rounds every ufunc operation on its own (no
FMA), which is what the kernel does with __dmul_rn / __dadd_rn, so the two agree pair for pair.

Candidates come from scipy's cKDTree at a slightly larger radius; the exact test above decides."""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree


def _exact(x, i, j, rc):
    d = x[i] - x[j]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    return d2 < rc * rc


def contact_pairs(x, rc):
    """(i, j), i < j, of every contact."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    cand = cKDTree(x).query_pairs(rc * (1.0 + 1e-6) + 1e-12, output_type="ndarray")
    if len(cand) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    i, j = np.minimum(cand[:, 0], cand[:, 1]).astype(np.int64), np.maximum(cand[:, 0], cand[:, 1]).astype(np.int64)
    keep = _exact(x, i, j, rc)
    return i[keep], j[keep]


def brute_pairs(x, rc):
    """The same by brute force over all N (N - 1) / 2 pairs (small N only)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    i, j = np.triu_indices(len(x), k=1)
    keep = _exact(x, i, j, rc)
    return i[keep].astype(np.int64), j[keep].astype(np.int64)


def counts_from_pairs(n, i, j, bins=None, n_bins=1, chrom=None):
    """(map uint64 (B, B) or None, sep uint64[n], pairs) as mmm_contacts returns them."""
    cmap = None
    if bins is not None:
        bins = np.asarray(bins, np.int64)
        bi, bj = bins[i], bins[j]
        ok = (bi >= 0) & (bj >= 0)
        cmap = np.zeros((n_bins, n_bins), np.uint64)
        np.add.at(cmap, (bi[ok], bj[ok]), np.uint64(1))
        off = ok & (bi != bj)
        np.add.at(cmap, (bj[off], bi[off]), np.uint64(1))
    same = np.ones(len(i), bool) if chrom is None else np.asarray(chrom)[i] == np.asarray(chrom)[j]
    sep = np.bincount(j[same] - i[same], minlength=n).astype(np.uint64)[:n]
    return cmap, sep, int(len(i))


def contact_counts(x, rc, bins=None, n_bins=1, chrom=None):
    i, j = contact_pairs(x, rc)
    return counts_from_pairs(len(x), i, j, bins, n_bins, chrom)


def near_threshold_pairs(x, rc, tol):
    """Number of pairs whose distance lies within tol of rc (those rounding of the coordinates can flip)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    cand = cKDTree(x).query_pairs(rc + tol, output_type="ndarray")
    if len(cand) == 0:
        return 0
    d = np.linalg.norm(x[cand[:, 0]] - x[cand[:, 1]], axis=1)
    return int(np.count_nonzero(np.abs(d - rc) <= tol))
