"""Simulated genome architecture mapping (GAM): thin random slices ("nuclear profiles") through each structure, and
how often two genomic windows are found in the same slice (co-segregation) — the one module that owns the slice
geometry and the file format.

A slice is the slab ``|((nx*x + ny*y) + nz*z) - o| <= h`` (FP64, rounded operation by operation; a bead on the
boundary is inside).  A bin is detected in a slice when any of its beads lies in it; per slice, the count of every
bin pair p <= q grows by one when both are detected (``Engine.gam_add``, ``mmm_gam_add``).  Whether a window is
detected depends on the extent of its beads along the slice normal and on where it sits in the nucleus, so GAM is
a many-body readout that pair distances and contact maps cannot give.  Bins are the canonical genomic bins of
``contacts.genome_bins``; sums are integers, so members and MD samples add exactly in any order.

``slice_planes`` draws isotropic uniform random sections of the structure's envelope sphere: unit normals from
normalised Gaussian 3-vectors, offsets ``o = n.c + u R`` with u ~ U[-1, 1], R the largest distance of a binned
bead from the centre c, and ``h = fraction R``, so a slice is ``fraction`` x the envelope diameter thick (0.025:
about a 220 nm cryosection through a 9 um nucleus).

Files (numpy ``.npz``): ``analysis/gam.npz`` of a single run, ``gam/member_<i>.npz`` of an ensemble member and
``ensemble_gam.npz`` of an ensemble; with ``MD_SAMPLE_STEP`` the same sums over the structures sampled during MD
in ``analysis/gam_md.npz``, ``gam/member_<i>_md.npz`` and ``ensemble_gam_md.npz``.

* ``counts``: uint64 [B (B + 1) / 2], rows in ``np.triu_indices(B)`` order: slices in which both bins are
  detected; the diagonal is each bin's detection count;
* ``structures``, ``slices``, ``empty`` (slices in which no bin is detected): int64;
* ``slice_fraction``: float64, the half-thickness over R;
* ``resolution_bp``, ``bin_chrom``, ``bin_start_bp``.

The readers return dense symmetric B x B maps (``detection_frequency``: [B]).  Frequencies are over the slices
that hit the structure, ``slices - empty``: an empty slice adds to no count, so leaving it out changes only that
denominator.
"""
from __future__ import annotations

import numpy as np

from .contacts import GenomeBins, _write
from .distances import _add

MAX_SLICES = 65536          # mmm_gam_configure: slices of one add
MAX_ROWS = 2**27            # B (B + 1) / 2 uint64 sums on the device (1 GiB)
MAX_BINS = 16383            # the most bins whose pairs fit MAX_ROWS
KEYS = ("counts", "structures", "slices", "empty", "slice_fraction", "resolution_bp", "bin_chrom", "bin_start_bp")
_MATCH = ("slice_fraction", "resolution_bp", "bin_chrom", "bin_start_bp")


def slice_planes(x, center, bins, count: int, fraction: float, rng: np.random.Generator):
    """``count`` isotropic uniform random slices of the envelope sphere of the binned beads of ``x`` (N x 3, nm)
    about ``center``: returns (planes float64 [count, 4] of nx, ny, nz, o, half-thickness h).  R is the largest
    distance of a bead with a bin from the centre (FP64); the unit normals are normalised Gaussian 3-vectors, the
    offsets o = n.c + u R with u ~ U[-1, 1], and h = fraction R.  Draws from ``rng`` only: normals first, then u."""
    x = np.asarray(x, np.float64)
    c = np.asarray(center, np.float64).reshape(3)
    keep = np.asarray(bins) >= 0
    if not keep.any():
        raise ValueError("GAM slices: no bead has a bin")
    d = x[keep] - c
    r = float(np.sqrt(np.max((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])))
    g = rng.standard_normal((int(count), 3))
    n = g / np.linalg.norm(g, axis=1, keepdims=True)
    u = rng.uniform(-1.0, 1.0, int(count))
    planes = np.empty((int(count), 4), np.float64)
    planes[:, :3] = n
    planes[:, 3] = n @ c + u * r
    return planes, float(fraction) * r


def result(r: dict, gb: GenomeBins, fraction: float) -> dict:
    """The in-memory form of a GAM file: the sums of Engine.gam_read binned by ``gb``, sliced with ``fraction``."""
    return dict(counts=np.asarray(r["counts"], np.uint64), structures=np.int64(r["structures"]),
                slices=np.int64(r["slices"]), empty=np.int64(r["empty"]), slice_fraction=np.float64(fraction),
                resolution_bp=np.int64(gb.resolution_bp), bin_chrom=np.asarray(gb.bin_chrom, np.int32),
                bin_start_bp=np.asarray(gb.bin_start_bp, np.int64))


def save(path: str, d: dict):
    _write(path, {k: d[k] for k in KEYS})


def load(path: str) -> dict:
    with np.load(path) as z:
        if "counts" not in z.files or "slice_fraction" not in z.files:
            raise ValueError(f"{path} is not a GAM file")
        return {k: z[k] for k in KEYS}


def aggregate(paths) -> dict:
    """Sum of GAM files: exact, the same bytes in any member order.  ValueError naming the file when its bins,
    resolution or slice fraction differ from the other members', or when a count would overflow uint64."""
    paths = list(paths)
    if not paths:
        raise ValueError("no GAM files to aggregate")
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
        for k in ("structures", "slices", "empty"):
            acc[k] = np.int64(int(acc[k]) + int(d[k]))
    return acc


def n_bins(d: dict) -> int:
    return len(d["bin_chrom"])


def _dense(tri: np.ndarray, b: int) -> np.ndarray:
    """Dense symmetric (B, B) of rows in np.triu_indices(B) order."""
    iu = np.triu_indices(b)
    out = np.zeros((b, b), tri.dtype)
    out[iu] = tri
    out[iu[1], iu[0]] = tri
    return out


def _hit(d: dict) -> float:
    """Slices that hit the structure (slices - empty): the denominator of every frequency; NaN when none did."""
    s = int(d["slices"]) - int(d["empty"])
    return float(s) if s > 0 else np.nan


def cosegregation(d: dict) -> np.ndarray:
    """float64 (B, B): f_pq, the fraction of the non-empty slices in which both bins are detected (the diagonal:
    f_p)."""
    return _dense(np.asarray(d["counts"], np.float64), n_bins(d)) / _hit(d)


def detection_frequency(d: dict) -> np.ndarray:
    """float64 [B]: f_p, the fraction of the non-empty slices in which each bin is detected."""
    return np.diagonal(cosegregation(d)).copy()


def _freqs(d: dict):
    fpq = cosegregation(d)
    fp = np.diagonal(fpq).copy()
    return fpq, fp[:, None], fp[None, :]


def linkage(d: dict) -> np.ndarray:
    """float64 (B, B): the linkage disequilibrium D = f_pq - f_p f_q."""
    fpq, fp, fq = _freqs(d)
    return fpq - fp * fq


def normalized_linkage(d: dict) -> np.ndarray:
    """float64 (B, B): D' = D / D_max with Lewontin's D_max: min(f_p (1 - f_q), (1 - f_p) f_q) where D >= 0,
    min(f_p f_q, (1 - f_p)(1 - f_q)) where D < 0.  NaN where D_max = 0 (a window detected in no slice or in
    every slice)."""
    fpq, fp, fq = _freqs(d)
    dl = fpq - fp * fq
    dmax = np.where(dl >= 0, np.minimum(fp * (1.0 - fq), (1.0 - fp) * fq), np.minimum(fp * fq, (1.0 - fp) * (1.0 - fq)))
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(dmax > 0, dl / np.where(dmax > 0, dmax, 1.0), np.nan)


def npmi(d: dict) -> np.ndarray:
    """float64 (B, B): normalised pointwise mutual information ln(f_pq / (f_p f_q)) / -ln f_pq, in [-1, 1]: -1
    where both windows are detected but never together (f_pq = 0), +1 where f_pq = 1, NaN where a window is
    never detected."""
    fpq, fp, fq = _freqs(d)
    with np.errstate(invalid="ignore", divide="ignore"):
        v = np.log(fpq / (fp * fq)) / -np.log(fpq)
    v = np.where(fpq == 0, -1.0, v)
    v = np.where(fpq == 1, 1.0, v)
    return np.where((fp > 0) & (fq > 0), v, np.nan)
