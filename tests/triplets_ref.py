"""numpy restatement of mmm_triplets_add: every bead triple i < j < k whose three pairs are contacts of
contacts_ref.contact_pairs (the FP64 expression of mmm_contacts), counted once, binned with p <= q <= r.

Forward adjacency in CSR order (fwd(i) = the j > i in contact with i); the wedges (i, j, k) with j in fwd(i) and
k in fwd(j) are built with np.repeat, a batch of edges at a time so that memory stays bounded, and a wedge is a
triangle when the key i * N + k is among the sorted contact keys (searchsorted)."""
from __future__ import annotations

import numpy as np

from contacts_ref import contact_pairs

WEDGES_PER_BATCH = 1 << 24


def globule(n, density, seed=0):
    """n beads uniform in a ball of ``density`` beads per nm^3: about 11 contact pairs per bead at rc = 0.2 nm and
    density 680 (as a minimised genome-wide structure has)."""
    rng = np.random.default_rng(seed)
    radius = (3.0 * n / (4.0 * np.pi * density)) ** (1.0 / 3.0)
    v = rng.normal(size=(n, 3))
    v *= (radius * rng.random(n) ** (1.0 / 3.0) / np.linalg.norm(v, axis=1))[:, None]
    return v


def triangles_from_pairs(n, i, j):
    """(i, j, k) int64 arrays, i < j < k, of every triangle of the contact graph with pairs (i, j), i < j."""
    i, j = np.asarray(i, np.int64), np.asarray(j, np.int64)
    key = i * n + j
    order = np.argsort(key, kind="stable")
    key, i, j = key[order], i[order], j[order]
    row = np.searchsorted(i, np.arange(n + 1, dtype=np.int64))
    deg = np.diff(row)
    wedges = deg[j]  # wedges of every edge (i, j): the k in fwd(j)
    ends = np.cumsum(wedges)
    out = []
    e0 = 0
    while e0 < len(i):
        e1 = int(np.searchsorted(ends, (ends[e0 - 1] if e0 else 0) + WEDGES_PER_BATCH, side="right"))
        e1 = max(e1, e0 + 1)
        cnt = wedges[e0:e1]
        if cnt.sum():
            e = np.repeat(np.arange(e0, e1), cnt)
            first = np.cumsum(cnt) - cnt
            t = np.arange(len(e)) - np.repeat(first, cnt)
            k = j[row[j[e]] + t]
            wk = i[e] * n + k
            pos = np.minimum(np.searchsorted(key, wk), len(key) - 1)
            hit = key[pos] == wk
            out.append((i[e][hit], j[e][hit], k[hit]))
        e0 = e1
    if not out:
        z = np.zeros(0, np.int64)
        return z, z, z
    return tuple(np.concatenate([o[a] for o in out]) for a in range(3))


def binned(ti, tj, tk, bins, n_bins):
    """(p, q, r int32, vals uint64) sorted by key, as mmm_triplets_read_entries returns them split."""
    bins = np.asarray(bins, np.int64)
    b = np.stack([bins[ti], bins[tj], bins[tk]], axis=1)
    b = np.sort(b[(b >= 0).all(axis=1)], axis=1)
    keys = (b[:, 0] * n_bins + b[:, 1]) * n_bins + b[:, 2]
    u, c = np.unique(keys, return_counts=True)
    return ((u // (n_bins * n_bins)).astype(np.int32), (u // n_bins % n_bins).astype(np.int32),
            (u % n_bins).astype(np.int32), c.astype(np.uint64))


def triplet_sums(x, rc, bins, n_bins):
    """dict(p, q, r, vals, triples) of one structure."""
    x = np.ascontiguousarray(x, np.float64)
    ti, tj, tk = triangles_from_pairs(len(x), *contact_pairs(x, rc))
    p, q, r, vals = binned(ti, tj, tk, bins, n_bins)
    return dict(p=p, q=q, r=r, vals=vals, triples=len(ti))


def brute_triangles(x, rc):
    """The same triangles by brute force over all N^3 / 6 triples (small N only)."""
    x = np.ascontiguousarray(x, np.float64)
    d = x[:, None, :] - x[None, :, :]
    d2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
    a = d2 < rc * rc
    n = len(x)
    ii, jj, kk = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
    t = (ii < jj) & (jj < kk) & a[ii, jj] & a[ii, kk] & a[jj, kk]
    return ii[t].astype(np.int64), jj[t].astype(np.int64), kk[t].astype(np.int64)
