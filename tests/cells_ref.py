"""numpy restatement of the cell-list grid of cut-off mode (mmm_cells.cu, k_cell_grid / k_cell_keys) and
of the FP32 pair test the kernel and the oracle share.

Every step is FP32 and rounds like the device: numpy's float32 subtraction and division are IEEE
round-to-nearest, as __fdiv_rn is.  The pair test r2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx)) < rc * rc
is emulated exactly (see _fma32).

stencil_misses() finds the pairs inside the cut-off that a walk over the 27 cells around a bead's own
cell cannot reach: their cell coordinates differ by 2 or more on some axis.  On a grid whose edge is
exactly rc such pairs exist (a lattice of 0.1 nm against rc = 0.2 or 0.3 nm has thousands); on the
kernel's grid, whose edge is rc * (1 + CELL_MARGIN), there are none."""
from __future__ import annotations

import numpy as np
from scipy.spatial import cKDTree

from common import O

f32 = np.float32
MAX_DIM = 64
CELL_MARGIN = 2.0 ** -12  # k_cell_grid: cell edge = rc * (1 + 2^-12) before the coarse branch


def centred(x):
    """The engine's centred FP32 copy: FP64 mean in index order (as mmm_set_positions forms it), then
    (float)(x - c)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    c = np.cumsum(x, axis=0)[-1] / float(len(x))  # sequential sum, not numpy's pairwise one
    return (x - c).astype(f32)


def grid(xc, rc, margin=CELL_MARGIN):
    """(cell, dim, origin) as k_cell_grid builds them from the centred FP32 coordinates xc."""
    xc = np.asarray(xc, dtype=f32)
    origin = f32(xc.min())
    extent = max(f32(f32(xc.max()) - origin), f32(0.0))
    cell = f32(f32(rc) * f32(1.0 + margin))
    dim = int(np.floor(f32(extent / cell))) + 1
    if dim > MAX_DIM:  # coarse branch: 64 cells of extent / 63
        cell = f32(extent / f32(MAX_DIM - 1))
        dim = MAX_DIM
    return cell, dim, origin


def cell_coords(xc, cell, dim, origin):
    """(N, 3) int cell coordinates: floorf(__fdiv_rn(x - origin, cell)) clamped to [0, dim - 1]."""
    v = np.floor(f32(f32(np.asarray(xc, dtype=f32) - f32(origin)) / f32(cell))).astype(np.int64)
    return np.clip(v, 0, dim - 1)


def cell_list(xc, rc, margin=CELL_MARGIN):
    """(keys, order, (cell, dim, origin)): sorted Morton keys and the (key, id) order of the grid above."""
    cell, dim, origin = grid(xc, rc, margin)
    keys, order = O.cell_list(xc, cell, dim, origin)
    return keys, order, (cell, dim, origin)


def _fma32(a, b, c):
    """fmaf(a, b, c) for float32 arrays, correctly rounded.  a * b is exact in FP64 and a * b + c is
    exact as s + e (TwoSum); rounding s to FP32 is correct unless s falls on the midpoint of two
    FP32 neighbours, where the sign of e decides."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    r = s.astype(f32)
    rd = r.astype(np.float64)
    toward = np.where(s > rd, f32(np.inf), f32(-np.inf)).astype(f32)
    nb = np.nextafter(r, toward)
    mid = (s != rd) & ((rd + nb.astype(np.float64)) * 0.5 == s) & (e != 0.0)
    # r and nb bracket s; on a midpoint the exact value lies beyond s on the side of e
    pick = np.where((e > 0) == (nb > r), nb, r)
    return np.where(mid, pick, r)


def pair_r2(xc, i, j):
    """r2 of the oracle's pair_in_cut: FP32 differences, fmaf(dz, dz, fmaf(dy, dy, dx * dx))."""
    d = (xc[i] - xc[j]).astype(f32)
    r2 = f32(d[:, 0] * d[:, 0])
    r2 = _fma32(d[:, 1], d[:, 1], r2)
    return _fma32(d[:, 2], d[:, 2], r2)


def in_cut_pairs(xc, rc):
    """(i, j), i < j, of every pair inside the cut-off by the FP32 test (what O.count_pairs counts)."""
    xc = np.asarray(xc, dtype=f32)
    cand = cKDTree(xc.astype(np.float64)).query_pairs(float(rc) * (1.0 + 1e-5), output_type="ndarray")
    if len(cand) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    i, j = cand.min(axis=1).astype(np.int64), cand.max(axis=1).astype(np.int64)
    rcf = f32(rc)
    keep = pair_r2(xc, i, j) < f32(rcf * rcf)
    return i[keep], j[keep]


def stencil_misses(xc, rc, margin=0.0):
    """(i, j) of the pairs inside the cut-off whose cell coordinates, on the grid of edge
    rc * (1 + margin), differ by 2 or more on some axis.  margin 0: the grid with edge exactly rc."""
    i, j = in_cut_pairs(xc, rc)
    cc = cell_coords(xc, *grid(xc, rc, margin))
    far = (np.abs(cc[i] - cc[j]) >= 2).any(axis=1)
    return i[far], j[far]
