"""Distance distributions per genomic bin pair (simulated chromatin tracing and multiplexed FISH: median distance
maps, the fraction of cells with two loci within a threshold, whole distance distributions) — the one module that
owns their format.

Per bead pair i < j whose beads both have a bin, ``d2 = (dx*dx + dy*dy) + dz*dz`` in FP64 (the expression of
``contacts`` and ``distances``) falls in the cell ``h = #{k : e_k * e_k <= d2}`` of the edges e_1 < ... < e_E
(nm, 1 <= E <= 63; the squares in FP64), and the count of (p, q, h) grows by one, p <= q the two bins
(``Engine.disthist_add``, ``mmm_disthist_add``).  Cell 0 is [0, e_1), cell h is [e_h, e_(h+1)) and cell E is
[e_E, inf).  The pairs in the cells below k are exactly the contacts of ``contacts`` at radius e_k, so a
histogram gives the contact map at every edge.  Bins are the canonical genomic bins of ``contacts.genome_bins``;
counts are uint64, so members and MD samples add exactly in any order.

Files (numpy ``.npz``): ``analysis/distance_hist.npz`` of a single run, ``distance_hist/member_<i>.npz`` of an
ensemble member and ``ensemble_distance_hist.npz`` of an ensemble; with ``MD_SAMPLE_STEP`` the same counts over
the structures sampled during MD in ``analysis/distance_hist_md.npz``, ``distance_hist/member_<i>_md.npz`` and
``ensemble_distance_hist_md.npz``.  A file of S structures is their sum exactly as an ensemble file is the sum of
its members.

* ``counts``: uint64 [B (B + 1) / 2, H], rows in ``np.triu_indices(B)`` order, H = E + 1 cells;
* ``edges_nm``: float64 [E];
* ``bin_beads``: uint64 [B], beads in each bin, summed over structures;
* ``members`` (structures), ``resolution_bp``, ``bin_chrom``, ``bin_start_bp``.

The readers return dense symmetric B x B maps.
"""
from __future__ import annotations

import numpy as np

from .contacts import GenomeBins, _write
from .distances import _add

MAX_EDGES = 63              # mmm_disthist_configure: H = E + 1 <= 64 cells
MAX_COUNTERS = 2**27        # B (B + 1) / 2 x H uint64 counters on the device (1 GiB)
DEFAULT_EDGES = "0.1,0.15,0.2,0.3,0.5,0.7,1,1.5,2,3,5,7,10,15,20,30,50,70,100"
KEYS = ("counts", "edges_nm", "bin_beads", "members", "resolution_bp", "bin_chrom", "bin_start_bp")
_MATCH = ("edges_nm", "resolution_bp", "bin_chrom", "bin_start_bp")


def check_edges(edges) -> np.ndarray:
    """The edges as float64 [E]: ValueError unless 1 <= E <= MAX_EDGES and the edges and their FP64 squares are
    finite, > 0 and strictly increasing (what mmm_disthist_configure accepts)."""
    e = np.asarray(edges, np.float64)
    if e.ndim != 1 or not 1 <= len(e) <= MAX_EDGES:
        raise ValueError(f"distance histogram: 1 to {MAX_EDGES} edges are needed, got {e.size}")
    with np.errstate(over="ignore", under="ignore"):
        e2 = e * e
    if not (np.all(np.isfinite(e)) and np.all(e > 0) and np.all(np.isfinite(e2)) and np.all(e2 > 0)):
        raise ValueError(f"distance histogram: the edges must be finite and > 0 (and so must their squares): {e}")
    if np.any(np.diff(e) <= 0) or np.any(np.diff(e2) <= 0):
        raise ValueError(f"distance histogram: the edges must be strictly increasing: {e}")
    return e


def parse_edges(text: str) -> np.ndarray:
    """The edges of a comma-separated string of nm values (DISTANCE_HIST_EDGES), checked by check_edges."""
    try:
        vals = [float(v) for v in str(text).split(",")]
    except ValueError:
        raise ValueError(f"distance histogram edges {text!r} are not a comma-separated list of numbers") from None
    return check_edges(vals)


def max_bins(n_edges: int) -> int:
    """The most bins whose B (B + 1) / 2 x (E + 1) counters fit MAX_COUNTERS."""
    h = int(n_edges) + 1
    b = int(np.floor(np.sqrt(2.0 * MAX_COUNTERS / h)))
    while b * (b + 1) // 2 * h > MAX_COUNTERS:
        b -= 1
    return b


def cells_of(d2, edges) -> np.ndarray:
    """The cell of every squared distance d2 (FP64, nm^2): #{k : e_k * e_k <= d2}."""
    e = np.asarray(edges, np.float64)
    return np.searchsorted(e * e, np.asarray(d2, np.float64), side="right")


def result(counts, edges, gb: GenomeBins, members: int = 1) -> dict:
    """The in-memory form of a distance-histogram file: the counts of Engine.disthist_read over ``members``
    structures binned by ``gb``, with their edges."""
    bins = np.asarray(gb.bins, np.int64)
    n = np.bincount(bins[bins >= 0], minlength=gb.n_bins).astype(np.uint64) * np.uint64(members)
    return dict(counts=np.asarray(counts, np.uint64), edges_nm=np.asarray(edges, np.float64), bin_beads=n,
                members=np.int64(members), resolution_bp=np.int64(gb.resolution_bp),
                bin_chrom=np.asarray(gb.bin_chrom, np.int32), bin_start_bp=np.asarray(gb.bin_start_bp, np.int64))


def save(path: str, d: dict):
    _write(path, {k: d[k] for k in KEYS})


def load(path: str) -> dict:
    with np.load(path) as z:
        if "counts" not in z.files or "edges_nm" not in z.files:
            raise ValueError(f"{path} is not a distance-histogram file")
        return {k: z[k] for k in KEYS}


def aggregate(paths) -> dict:
    """Sum of distance-histogram files: exact uint64, the same bytes in any member order.  ValueError naming the
    file when its bins, resolution or edges differ from the other members', or when a count would overflow
    uint64."""
    paths = list(paths)
    if not paths:
        raise ValueError("no distance-histogram files to aggregate")
    acc = None
    for p in paths:
        d = load(p)
        if acc is None:
            acc = dict(d)
            continue
        for k in _MATCH:
            if np.shape(acc[k]) != np.shape(d[k]) or not np.array_equal(acc[k], d[k]):
                raise ValueError(f"{p}: {k} differs from the other members")
        if acc["counts"].shape != d["counts"].shape:
            raise ValueError(f"{p}: counts differ in shape from the other members")
        acc["counts"] = _add(acc["counts"], d["counts"], p, "counts")
        acc["bin_beads"] = _add(acc["bin_beads"], d["bin_beads"], p, "bin_beads")
        acc["members"] = np.int64(acc["members"] + int(d["members"]))
    return acc


def n_bins(d: dict) -> int:
    return len(d["bin_chrom"])


def _dense(tri: np.ndarray, b: int) -> np.ndarray:
    """Dense symmetric (B, B, ...) of rows in np.triu_indices(B) order."""
    iu = np.triu_indices(b)
    out = np.zeros((b, b) + tri.shape[1:], tri.dtype)
    out[iu] = tri
    out[iu[1], iu[0]] = tri
    return out


def pair_counts(d: dict) -> np.ndarray:
    """uint64 (B, B): bead pairs counted in every bin pair, over all cells."""
    return _dense(np.asarray(d["counts"], np.uint64).sum(axis=1, dtype=np.uint64), n_bins(d))


def cumulative_probability(d: dict) -> np.ndarray:
    """float64 (B, B, E): the fraction of the pairs of every bin pair closer than each edge (d < e_k); NaN where
    there is no pair."""
    c = np.asarray(d["counts"], np.float64)
    cum = np.cumsum(c, axis=1)[:, :-1]
    tot = c.sum(axis=1, keepdims=True)
    with np.errstate(invalid="ignore", divide="ignore"):
        p = np.where(tot > 0, cum / np.where(tot > 0, tot, 1.0), np.nan)
    return _dense(p, n_bins(d))


def contact_probability(d: dict, radius_nm: float) -> np.ndarray:
    """float64 (B, B): the fraction of the pairs of every bin pair closer than ``radius_nm`` (the contact
    frequency of ``contacts`` at that radius); NaN where there is no pair.  The radius must equal one of the edges
    exactly: ValueError otherwise (no interpolation between edges)."""
    e = np.asarray(d["edges_nm"], np.float64)
    k = np.flatnonzero(e == float(radius_nm))
    if len(k) != 1:
        raise ValueError(f"radius {radius_nm} nm is not one of the histogram's edges {list(e)}")
    return cumulative_probability(d)[:, :, int(k[0])]


def quantile_distance(d: dict, q: float) -> np.ndarray:
    """float64 (B, B): the q-quantile of the distances of every bin pair (0 <= q <= 1), in nm.  It is found in
    the cell that holds it, the first cell with pairs whose cumulative count reaches q x pairs, and interpolated
    linearly within that cell (as if its pairs were spread evenly over it; cell 0 spans [0, e_1)).  NaN where the
    bin pair has no pair, or where the quantile falls in the open last cell [e_E, inf)."""
    q = float(q)
    if not 0.0 <= q <= 1.0:
        raise ValueError(f"quantile {q} is outside [0, 1]")
    e = np.asarray(d["edges_nm"], np.float64)
    lo_edge = np.concatenate([[0.0], e])            # lower edge of every cell
    hi_edge = np.concatenate([e, [np.inf]])         # upper edge of every cell
    c = np.asarray(d["counts"], np.float64)
    cum = np.cumsum(c, axis=1)                      # pairs below the upper edge of every cell
    tot = cum[:, -1]
    t = q * tot
    ok = (c > 0) & (cum >= t[:, None])
    h = np.argmax(ok, axis=1)                       # the first cell with pairs that reaches t
    rows = np.arange(len(c))
    ch = c[rows, h]
    below = cum[rows, h] - ch
    last = h == len(e)
    with np.errstate(invalid="ignore", divide="ignore"):
        frac = (t - below) / np.where(ch > 0, ch, 1.0)
        val = lo_edge[h] + frac * np.where(last, 0.0, hi_edge[h] - lo_edge[h])
    val = np.where((tot > 0) & ~last, val, np.nan)
    return _dense(val, n_bins(d))


def median_distance(d: dict) -> np.ndarray:
    """float64 (B, B): the median distance of every bin pair in nm (quantile_distance at 0.5)."""
    return quantile_distance(d, 0.5)


def distance_histogram_sums(V, bins, n_bins: int, edges, device: int = 0) -> np.ndarray:
    """counts (uint64 [B (B + 1) / 2, E + 1]) of any (n, 3) coordinate array in nm, through a temporary Engine on
    `device`."""
    from .engine import Engine

    V = np.ascontiguousarray(V, dtype=np.float64)
    with Engine(len(V), device=device) as eng:
        eng.set_positions(V)
        eng.disthist_configure(bins, n_bins, edges)
        eng.disthist_add()
        return eng.disthist_read()["counts"]
