"""Three-way contact maps (simulated multi-way chromatin capture, as SPRITE, GAM or Pore-C measure it): which
three loci are in contact in the *same* structure — the one module that owns their format.

A three-way contact is an unordered bead triple i < j < k whose three pairs (i, j), (i, k) and (j, k) are all
contacts of ``contacts`` (``d2 < rc * rc``, ``d2 = (dx*dx + dy*dy) + dz*dz`` in FP64): a triangle of the
pairwise contact graph, counted once (``Engine.triplets_add``, ``mmm_triplets_add``).  Beads are binned in the
canonical genomic coordinates of ``contacts.genome_bins``; a triple with a bead outside the map counts only in
``triples``, the others add 1 to the entry of their bins sorted into p <= q <= r (a triple inside one bin is
(p, p, p)).  No minimum index separation is applied: drop near-diagonal entries when reading.

Files (numpy ``.npz``): ``analysis/triplets.npz`` of a single run, ``triplets/member_<i>.npz`` of an ensemble
member and ``ensemble_triplets.npz`` of an ensemble; with ``MD_SAMPLE_STEP`` the same sums over the structures
sampled during MD in ``analysis/triplets_md.npz``, ``triplets/member_<i>_md.npz`` and
``ensemble_triplets_md.npz``.  A file of S structures is their sum exactly as an ensemble file is the sum of
its members.

* the entries: ``p``, ``q``, ``r`` (int32, p <= q <= r) and ``vals`` (uint64 > 0), sorted by the key
  (p * B + q) * B + r;
* the bins: ``n_bins`` (B <= 2^20), ``bin_chrom``, ``bin_start_bp``, ``resolution_bp``;
* the run: ``radius_nm``, ``members`` (structures), ``triples`` (all three-way contacts, binned or not).
"""
from __future__ import annotations

import numpy as np

from . import contacts
from .contacts import GenomeBins, _write
from .distances import _add

MAX_BINS = 2**20    # mmm_triplets_configure: keys (p * B + q) * B + r stay below 2^60
DEFAULT_CHUNK_KEYS = 2**26  # binned triples of one structure sorted at a time on the device (1 GiB)
KEYS = ("p", "q", "r", "vals", "n_bins", "bin_chrom", "bin_start_bp", "resolution_bp", "radius_nm", "members",
        "triples")
_MATCH = ("n_bins", "bin_chrom", "bin_start_bp", "resolution_bp", "radius_nm")


def result(read: dict, radius_nm: float, gb: GenomeBins, members: int = 1) -> dict:
    """The in-memory form of a triplets file: what Engine.triplets_read returns, with its bins."""
    return dict(p=np.asarray(read["p"], np.int32), q=np.asarray(read["q"], np.int32),
                r=np.asarray(read["r"], np.int32), vals=np.asarray(read["vals"], np.uint64),
                n_bins=np.int64(gb.n_bins), bin_chrom=np.asarray(gb.bin_chrom, np.int32),
                bin_start_bp=np.asarray(gb.bin_start_bp, np.int64), resolution_bp=np.int64(gb.resolution_bp),
                radius_nm=np.float64(radius_nm), members=np.int64(members), triples=np.uint64(read["triples"]))


def save(path: str, d: dict):
    _write(path, {k: d[k] for k in KEYS})


def load(path: str) -> dict:
    with np.load(path) as z:
        if "triples" not in z.files or "p" not in z.files:
            raise ValueError(f"{path} is not a triplets file")
        return {k: z[k] for k in KEYS}


def keys(d: dict) -> np.ndarray:
    """int64 key (p * B + q) * B + r of every entry."""
    b = int(d["n_bins"])
    return (np.asarray(d["p"], np.int64) * b + np.asarray(d["q"], np.int64)) * b + np.asarray(d["r"], np.int64)


def _reduce(k: np.ndarray, v: np.ndarray, b: int, path: str = "sum"):
    """Sorted unique (p, q, r, vals) of keys k with counts v (equal keys added, exact uint64)."""
    order = np.argsort(k, kind="stable")
    k, v = k[order], np.asarray(v, np.uint64)[order]
    head = np.ones(len(k), bool)
    head[1:] = k[1:] != k[:-1]
    starts = np.flatnonzero(head)
    vals = np.add.reduceat(v, starts) if len(starts) else v[:0]
    if len(starts) and np.any(vals < np.maximum.reduceat(v, starts)):
        raise ValueError(f"{path}: a count would overflow uint64")
    k = k[starts]
    return ((k // (b * b)).astype(np.int32), (k // b % b).astype(np.int32), (k % b).astype(np.int32),
            vals.astype(np.uint64))


def aggregate(paths) -> dict:
    """Sum of triplets files: exact uint64, the same bytes in any member order (sorted merge of the entries).
    ValueError naming the file when its bins, resolution or radius differ from the other members'."""
    paths = list(paths)
    if not paths:
        raise ValueError("no triplets files to aggregate")
    acc = None
    for p in paths:
        d = load(p)
        if acc is None:
            acc = dict(d)
            continue
        for k in _MATCH:
            if np.shape(acc[k]) != np.shape(d[k]) or not np.array_equal(acc[k], d[k]):
                raise ValueError(f"{p}: {k} differs from the other members")
        acc["p"], acc["q"], acc["r"], acc["vals"] = _reduce(np.concatenate([keys(acc), keys(d)]),
                                                            np.concatenate([acc["vals"], d["vals"]]),
                                                            int(acc["n_bins"]), p)
        acc["members"] = np.int64(acc["members"] + int(d["members"]))
        acc["triples"] = _add(np.uint64(acc["triples"]), np.uint64(d["triples"]), p, "triples")
    return acc


def coarsen(d: dict, resolution_bp: int) -> dict:
    """The triplets file of ``d`` at ``resolution_bp``, a multiple of its resolution giving at most
    contacts.MAX_BINS bins.  Both grids start at each chromosome's ``lo`` (contacts.genome_bins), so coarse bin
    = fine bin // k within a chromosome, the order of bins is kept and the sums are exact."""
    res = int(d["resolution_bp"])
    if resolution_bp <= 0 or resolution_bp % res:
        raise ValueError(f"resolution_bp={resolution_bp} is not a multiple of the resolution {res} bp")
    k = resolution_bp // res
    chrom = np.asarray(d["bin_chrom"])
    start = np.asarray(d["bin_start_bp"], np.int64)
    starts = np.flatnonzero(np.concatenate([[True], chrom[1:] != chrom[:-1]]))  # a chromosome's bins are contiguous
    ends = np.append(starts[1:], len(chrom))
    cmap = np.empty(len(chrom), np.int64)
    first = []  # the first fine bin of every coarse bin
    nb = 0
    for a, b in zip(starts, ends):
        cmap[a:b] = nb + np.arange(b - a) // k
        first.extend(range(a, b, k))
        nb += -(-(b - a) // k)
    if nb > contacts.MAX_BINS:
        raise ValueError(f"resolution_bp={resolution_bp} gives {nb} bins; at most {contacts.MAX_BINS} are supported")
    first = np.asarray(first, np.int64)
    gb = GenomeBins(np.zeros(0, np.int32), chrom[first], start[first], resolution_bp)
    # cmap is non-decreasing, so p <= q <= r stays sorted
    ck = (cmap[d["p"]] * nb + cmap[d["q"]]) * nb + cmap[d["r"]]
    p, q, r, vals = _reduce(ck, d["vals"], nb)
    return result(dict(p=p, q=q, r=r, vals=vals, triples=d["triples"]), float(d["radius_nm"]), gb,
                  int(d["members"]))


def viewpoint(d: dict, bin: int) -> np.ndarray:
    """Dense symmetric uint64 (B, B) M with M[a, b] = the count of the triples whose bin multiset is {bin, a, b}:
    the three-way contacts of ``bin`` with every pair of bins (the conditional map of multi-way analyses).  At
    most contacts.MAX_BINS bins (coarsen a fine map first)."""
    nb = int(d["n_bins"])
    if nb > contacts.MAX_BINS:
        raise ValueError(f"{nb} bins; a viewpoint map holds at most {contacts.MAX_BINS} (coarsen first)")
    v = int(bin)
    if not 0 <= v < nb:
        raise ValueError(f"bin {v} outside [0, {nb})")
    p, q, r = (np.asarray(d[k], np.int64) for k in ("p", "q", "r"))
    vals = np.asarray(d["vals"], np.uint64)
    # drop one occurrence of the viewpoint bin from every entry that holds it: the other two bins remain
    a = np.where(p == v, q, p)
    b = np.where((p == v) | (q == v), r, q)
    sel = (p == v) | (q == v) | (r == v)
    a, b, vals = a[sel], b[sel], vals[sel]
    out = np.zeros((nb, nb), np.uint64)
    np.add.at(out, (a, b), vals)
    off = a != b
    np.add.at(out, (b[off], a[off]), vals[off])
    return out
