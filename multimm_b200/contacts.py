"""Contact frequencies of structures and ensembles (simulated Hi-C) — the one module that owns their format.

A contact is an unordered bead pair i < j with ``d2 < rc * rc``, ``d2 = (dx*dx + dy*dy) + dz*dz`` in FP64
(``Engine.contacts``, ``mmm_contacts``).  Beads are binned in *canonical genomic coordinates*: chromosomes
in ``loaders.CHROM_NAMES`` order whatever the member's shuffle, bins of ``resolution_bp`` that never straddle
a chromosome (as in Hi-C), over the whole chromosome genome-wide and over ``[LOC_START, LOC_END)`` in region
runs.  So bin p means the same locus in every member of an ensemble, and member maps add up.

Files (numpy ``.npz``):

* ``analysis/contacts.npz`` of a single run and ``ensemble_contacts.npz`` of an ensemble: ``counts`` (uint64
  B x B, symmetric), ``members``, ``radius_nm``, ``resolution_bp``, ``bin_chrom``, ``bin_start_bp``,
  ``sep_contacts`` / ``sep_pairs`` (uint64[N]: same-chromosome contacts and bead pairs at index separation s;
  P(s) = sep_contacts / sep_pairs), ``pairs`` (all contacts);
* ``contacts/member_<i>.npz`` of an ensemble member: the same, with the map as the sparse upper triangle
  (``rows``, ``cols``, ``vals``) and ``n_bins``.  Integer sums do not depend on order, so the ensemble file
  is the same bit for bit whichever GPU ran which member;
* the fine map (``CONTACT_FINE_RESOLUTION``, ``Engine.contacts_sparse``): ``analysis/contacts_fine.npz`` of a
  single run, ``contacts/member_<i>_fine.npz`` of an ensemble member and ``ensemble_contacts_fine.npz`` of an
  ensemble.  Always sparse, never a dense ``counts`` (a 5 kb genome-wide map has ~6e5 bins): ``rows``,
  ``cols`` (int32), ``vals`` (uint64), the nonzero upper triangle sorted by (row, col) with rows <= cols;
  ``n_bins``, ``bin_chrom``, ``bin_start_bp``, ``resolution_bp``, ``radius_nm``, ``members``, ``pairs``.
  Read it with ``load_fine``; ``coarsen`` and ``fine_block`` give dense views of it;
* the trajectory maps (``MD_SAMPLE_STEP``, ``Engine.sampler_read``): the same maps summed over the structures
  sampled during MD, in the same formats, named with ``_md`` before ``.npz``: ``analysis/contacts_md.npz`` and
  ``analysis/contacts_fine_md.npz`` of a single run, ``contacts/member_<i>_md.npz`` and
  ``contacts/member_<i>_fine_md.npz`` of an ensemble member, ``ensemble_contacts_md.npz`` and
  ``ensemble_contacts_fine_md.npz`` of an ensemble.  A file of S sampled structures is their sum exactly as an
  ensemble file is the sum of its members: ``members`` = S and ``sep_pairs`` S times one structure's, so
  ``contact_probability``, ``aggregate``, ``aggregate_fine``, ``coarsen`` and ``fine_block`` read it unchanged.
"""
from __future__ import annotations

import os
from typing import NamedTuple

import numpy as np

from . import loaders

MAX_BINS = 4096     # dense map cap of mmm_contacts (128 MB of uint64)
MAX_FINE_BINS = 2**31 - 1  # sparse map (mmm_contacts_sparse): bins are int32
FINE_KEYS = ("rows", "cols", "vals", "n_bins", "bin_chrom", "bin_start_bp", "resolution_bp", "radius_nm",
             "members", "pairs")
AUTO_BINS = 1000    # CONTACT_RESOLUTION = 0: about this many bins over the modelled genome or region


class GenomeBins(NamedTuple):
    bins: np.ndarray          # int32[N]: canonical bin of every bead
    bin_chrom: np.ndarray     # int32[B]: chromosome index (loaders.CHROM_NAMES) of every bin
    bin_start_bp: np.ndarray  # int64[B]: first bp of every bin
    resolution_bp: int

    @property
    def n_bins(self) -> int:
        return len(self.bin_chrom)


def spans(chrom_idxs, start_bp: int = 0, stop_bp: int | None = None) -> list[tuple[int, int, int]]:
    """(chromosome index, lo, hi) of the modelled stretch of every chromosome, in CHROM_NAMES order:
    whole chromosomes genome-wide (stop_bp None), [start_bp, stop_bp) in a region run."""
    out = []
    for c in sorted(int(c) for c in chrom_idxs):
        if stop_bp is None:
            out.append((c, 0, int(loaders.CHROM_LENGTHS[c])))
        else:
            out.append((c, int(start_bp), int(stop_bp)))
    return out


def auto_resolution(sp) -> int:
    """Bin size that gives at most AUTO_BINS bins: ceil(total / (AUTO_BINS - chromosomes)) bp, since every
    chromosome adds at most one partial bin."""
    total = sum(hi - lo for _, lo, hi in sp)
    return max(1, -(-total // (AUTO_BINS - len(sp))))


def bin_count(sp, resolution_bp: int) -> int:
    return int(sum(-(-(hi - lo) // resolution_bp) for _, lo, hi in sp))


def genome_bins(layout: dict, resolution_bp: int = 0, n_beads: int | None = None,
                max_bins: int = MAX_BINS) -> GenomeBins:
    """Canonical bin of every bead of a run whose bead-to-genome mapping is ``layout`` (what
    loaders.import_mns_from_bedpe fills; MultiMM.layout).  Bead i of block k sits at bp
    ``start_bp + i * res + res // 2 - ends[k]`` of chromosome ``chrom_idxs[k]``, clamped to the modelled
    stretch of that chromosome.  resolution_bp 0: automatic (auto_resolution).  ValueError beyond max_bins
    (MAX_BINS for the dense map, MAX_FINE_BINS for the sparse one)."""
    sp = spans(layout["chrom_idxs"], int(layout.get("start_bp", 0)), layout.get("stop_bp"))
    r = int(resolution_bp) if resolution_bp and resolution_bp > 0 else auto_resolution(sp)
    nb = bin_count(sp, r)
    if nb > max_bins:
        raise ValueError(f"CONTACT_RESOLUTION={r} bp gives {nb} bins; at most {max_bins} are supported")
    first = np.zeros(len(loaders.CHROM_LENGTHS), np.int64)
    lo_of = np.zeros(len(loaders.CHROM_LENGTHS), np.int64)
    bin_chrom, bin_start = [], []
    for c, lo, hi in sp:
        first[c], lo_of[c] = len(bin_chrom), lo
        k = -(-(hi - lo) // r)
        bin_chrom.extend([c] * k)
        bin_start.extend(lo + r * np.arange(k, dtype=np.int64))
    chrom, bp = bead_loci(layout, n_beads)
    bins = (first[chrom] + (bp - lo_of[chrom]) // r).astype(np.int32)
    return GenomeBins(bins, np.asarray(bin_chrom, np.int32), np.asarray(bin_start, np.int64), r)


def bead_loci(layout: dict, n_beads: int | None = None) -> tuple[np.ndarray, np.ndarray]:
    """(chromosome index, bp) of every bead, as genome_bins places them."""
    res = int(layout["resolution"])
    ends, chr_ends = np.asarray(layout["ends"], np.int64), np.asarray(layout["chr_ends"], np.int64)
    idxs = np.asarray(layout["chrom_idxs"], np.int64)
    start_bp, stop_bp = int(layout.get("start_bp", 0)), layout.get("stop_bp")
    n = int(chr_ends[-1]) if n_beads is None else int(n_beads)
    chrom, bp = np.empty(n, np.int64), np.empty(n, np.int64)
    i = np.arange(n, dtype=np.int64)
    for k in range(len(idxs)):
        a, b, c = int(chr_ends[k]), int(chr_ends[k + 1]), int(idxs[k])
        lo, hi = (0, int(loaders.CHROM_LENGTHS[c])) if stop_bp is None else (start_bp, int(stop_bp))
        chrom[a:b] = c
        bp[a:b] = np.clip(start_bp + i[a:b] * res + res // 2 - ends[k], lo, hi - 1)
    return chrom, bp


def sep_pairs(chrom_ids) -> np.ndarray:
    """uint64[N]: bead pairs at index separation s inside the same-chromosome blocks (runs of equal ids):
    sum over blocks of max(0, L_b - s); entry 0 is 0."""
    c = np.asarray(chrom_ids)
    n = len(c)
    cuts = np.concatenate([[0], np.flatnonzero(c[1:] != c[:-1]) + 1, [n]])
    s = np.arange(n, dtype=np.int64)
    out = np.zeros(n, dtype=np.int64)
    for L in np.diff(cuts):
        out += np.maximum(0, L - s)
    out[0] = 0
    return out.astype(np.uint64)


def result(counts, sep, pairs, radius_nm, gb: GenomeBins, sep_den, members: int = 1) -> dict:
    """The in-memory form of a contacts file (dense map)."""
    return dict(counts=np.asarray(counts, np.uint64), members=np.int64(members), radius_nm=np.float64(radius_nm),
                resolution_bp=np.int64(gb.resolution_bp), bin_chrom=np.asarray(gb.bin_chrom, np.int32),
                bin_start_bp=np.asarray(gb.bin_start_bp, np.int64), sep_contacts=np.asarray(sep, np.uint64),
                sep_pairs=np.asarray(sep_den, np.uint64), pairs=np.int64(pairs))


def contact_probability(d: dict) -> np.ndarray:
    """P(s) = sep_contacts / sep_pairs (NaN where there is no pair at separation s)."""
    num = np.asarray(d["sep_contacts"], np.float64)
    den = np.asarray(d["sep_pairs"], np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.nan)


def md_path(path: str) -> str:
    """The trajectory-map file beside a structure's map file: ``_md`` before ``.npz``."""
    return path[:-len(".npz")] + "_md.npz"


def _write(path: str, arrays: dict):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    tmp = path + ".tmp.npz"
    np.savez(tmp, **arrays)
    os.replace(tmp, path)


def save_dense(path: str, d: dict):
    _write(path, d)


def save_member(path: str, d: dict):
    """Upper triangle of the map, sparse, plus everything else of the dense form."""
    counts = np.asarray(d["counts"], np.uint64)
    rows, cols = np.nonzero(np.triu(counts))
    out = {k: v for k, v in d.items() if k != "counts"}
    out.update(rows=rows.astype(np.int32), cols=cols.astype(np.int32), vals=counts[rows, cols],
               n_bins=np.int64(counts.shape[0]))
    _write(path, out)


def load(path: str) -> dict:
    """A dense or member contacts file, with the map dense.  ValueError for a fine file (load_fine)."""
    with np.load(path) as z:
        d = {k: z[k] for k in z.files}
    if "sep_contacts" not in d:
        raise ValueError(f"{path} is a fine (sparse) contacts file; read it with contacts.load_fine")
    if "counts" not in d:
        b = int(d.pop("n_bins"))
        rows, cols, vals = d.pop("rows"), d.pop("cols"), d.pop("vals")
        counts = np.zeros((b, b), np.uint64)
        counts[rows, cols] = vals
        counts[cols, rows] = vals
        d["counts"] = counts
    return d


def aggregate(paths) -> dict:
    """Sum of member files (exact integer sums); the bins, radius and resolution must agree."""
    paths = list(paths)
    if not paths:
        raise ValueError("no contact files to aggregate")
    acc = None
    for p in paths:
        d = load(p)
        if acc is None:
            acc = dict(d, members=np.int64(0), pairs=np.int64(0))
        else:
            for k in ("bin_chrom", "bin_start_bp", "radius_nm", "resolution_bp"):
                if not np.array_equal(acc[k], d[k]):
                    raise ValueError(f"{p}: {k} differs from the other members")
            acc["counts"] = acc["counts"] + d["counts"]
            acc["sep_contacts"] = acc["sep_contacts"] + d["sep_contacts"]
            acc["sep_pairs"] = acc["sep_pairs"] + d["sep_pairs"]
        acc["members"] = np.int64(acc["members"] + int(d.get("members", 1)))
        acc["pairs"] = np.int64(acc["pairs"] + int(d["pairs"]))
    return acc


def fine_result(rows, cols, vals, pairs, radius_nm, gb: GenomeBins, members: int = 1) -> dict:
    """The in-memory form of a fine contacts file (what Engine.contacts_sparse returns, with its bins)."""
    return dict(rows=np.asarray(rows, np.int32), cols=np.asarray(cols, np.int32), vals=np.asarray(vals, np.uint64),
                n_bins=np.int64(gb.n_bins), bin_chrom=np.asarray(gb.bin_chrom, np.int32),
                bin_start_bp=np.asarray(gb.bin_start_bp, np.int64), resolution_bp=np.int64(gb.resolution_bp),
                radius_nm=np.float64(radius_nm), members=np.int64(members), pairs=np.int64(pairs))


def save_fine(path: str, d: dict):
    _write(path, {k: d[k] for k in FINE_KEYS})


def load_fine(path: str) -> dict:
    """A fine contacts file, sparse as stored."""
    with np.load(path) as z:
        if "rows" not in z.files or "sep_contacts" in z.files:
            raise ValueError(f"{path} is not a fine contacts file")
        return {k: z[k] for k in FINE_KEYS}


def _merge(rows, cols, vals, r2, c2, v2, n_bins: int):
    """Sum of two sorted sparse upper triangles, sorted (exact uint64; merged, never densified)."""
    k1 = rows.astype(np.int64) * n_bins + cols
    k2 = r2.astype(np.int64) * n_bins + c2
    keys = np.concatenate([k1, k2])
    v = np.concatenate([vals, v2])
    order = np.argsort(keys, kind="stable")
    keys, v = keys[order], v[order]
    head = np.ones(len(keys), bool)
    head[1:] = keys[1:] != keys[:-1]
    starts = np.flatnonzero(head)
    out_v = np.add.reduceat(v, starts) if len(starts) else v[:0]
    k = keys[starts]
    return (k // n_bins).astype(np.int32), (k % n_bins).astype(np.int32), out_v.astype(np.uint64)


def aggregate_fine(paths) -> dict:
    """Sum of fine member files: exact uint64, the same bytes in any member order (sorted merge of sparse
    entries); the bins, radius and resolution must agree."""
    paths = list(paths)
    if not paths:
        raise ValueError("no fine contact files to aggregate")
    acc = None
    for p in paths:
        d = load_fine(p)
        if acc is None:
            acc = dict(d)
            continue
        for k in ("n_bins", "bin_chrom", "bin_start_bp", "radius_nm", "resolution_bp"):
            if not np.array_equal(acc[k], d[k]):
                raise ValueError(f"{p}: {k} differs from the other members")
        acc["rows"], acc["cols"], acc["vals"] = _merge(acc["rows"], acc["cols"], acc["vals"], d["rows"], d["cols"],
                                                       d["vals"], int(acc["n_bins"]))
        acc["members"] = np.int64(acc["members"] + int(d["members"]))
        acc["pairs"] = np.int64(acc["pairs"] + int(d["pairs"]))
    return acc


def coarsen(fine: dict, resolution_bp: int) -> np.ndarray:
    """Dense symmetric uint64 map of a fine map at ``resolution_bp``, a multiple of its resolution giving at
    most MAX_BINS bins.  Both grids start at each chromosome's ``lo``, so coarse bin = fine bin // k within
    a chromosome and the sums are exact; the coarse grid is what genome_bins makes at resolution_bp."""
    r = int(fine["resolution_bp"])
    if resolution_bp <= 0 or resolution_bp % r:
        raise ValueError(f"resolution_bp={resolution_bp} is not a multiple of the fine resolution {r} bp")
    k = resolution_bp // r
    chrom = np.asarray(fine["bin_chrom"])
    starts = np.flatnonzero(np.concatenate([[True], chrom[1:] != chrom[:-1]]))  # a chromosome's bins are contiguous
    ends = np.append(starts[1:], len(chrom))
    cmap = np.empty(len(chrom), np.int64)
    nb = 0
    for a, b in zip(starts, ends):
        cmap[a:b] = nb + np.arange(b - a) // k
        nb += -(-(b - a) // k)
    if nb > MAX_BINS:
        raise ValueError(f"resolution_bp={resolution_bp} gives {nb} bins; at most {MAX_BINS} are supported")
    out = np.zeros((nb, nb), np.uint64)
    p, q = cmap[fine["rows"]], cmap[fine["cols"]]
    vals = np.asarray(fine["vals"], np.uint64)
    np.add.at(out, (p, q), vals)
    off = p != q
    np.add.at(out, (q[off], p[off]), vals[off])
    return out


def fine_block(fine: dict, chrom: str | int, start_bp: int, end_bp: int) -> tuple[np.ndarray, np.ndarray]:
    """(counts, bin_start_bp): the dense symmetric uint64 sub-matrix of the fine map over the bins of
    chromosome ``chrom`` (name or CHROM_NAMES index) that overlap [start_bp, end_bp), and their first bps."""
    c = {v: i for i, v in loaders.CHROM_NAMES.items()}[chrom] if isinstance(chrom, str) else int(chrom)
    r = int(fine["resolution_bp"])
    start = np.asarray(fine["bin_start_bp"], np.int64)
    sel = np.flatnonzero((np.asarray(fine["bin_chrom"]) == c) & (start < end_bp) & (start + r > start_bp))
    if len(sel) == 0:
        return np.zeros((0, 0), np.uint64), start[:0]
    lo, hi = int(sel[0]), int(sel[-1]) + 1   # a chromosome's bins are contiguous
    rows, cols = np.asarray(fine["rows"]), np.asarray(fine["cols"])
    m = (rows >= lo) & (rows < hi) & (cols >= lo) & (cols < hi)
    p, q, v = rows[m] - lo, cols[m] - lo, np.asarray(fine["vals"], np.uint64)[m]
    out = np.zeros((hi - lo, hi - lo), np.uint64)
    out[p, q] = v
    out[q, p] = v
    return out, start[lo:hi]


def contact_counts(V, rc_nm: float, bins=None, n_bins: int = 1, chrom=None, device: int = 0):
    """(map, sep, pairs) of any (n, 3) coordinate array in nm, through a temporary Engine on `device`.
    chrom (int[n], optional): chromosome ids for the separation counts (None = one chromosome)."""
    from .engine import Engine

    V = np.ascontiguousarray(V, dtype=np.float64)
    with Engine(len(V), device=device) as eng:
        if chrom is not None:
            eng.set_bead_params(chrom=np.asarray(chrom, np.int32))
        eng.set_positions(V)
        return eng.contacts(rc_nm, bins, n_bins)
