"""Mean-distance maps and radial profiles of structures and ensembles (simulated chromatin tracing) — the one
module that owns their format.

Per bead pair i < j whose beads both have a bin, ``d2 = (dx*dx + dy*dy) + dz*dz`` in FP64 and ``d =
sqrt(d2)``, each quantised on its own with the quantum Q = 2^-24 (``rint(d / Q)``, half to even) and summed in
uint64 per bin pair (``Engine.distance_map``, ``mmm_distance_map``).  Per bead, its distance r from the
member's container centre (``MultiMM.mass_center``, the centre of the SC / LAM / CF terms) and r^2,
quantised and summed per bin the same way on the host.  Bins are the canonical genomic bins of
``contacts.genome_bins``, so bin p is the same locus in every member and integer sums of members are exact
in any order.

Files (numpy ``.npz``): ``analysis/distances.npz`` of a single run, ``distances/member_<i>.npz`` of an
ensemble member and ``ensemble_distances.npz`` of an ensemble, all in one format.  With ``MD_SAMPLE_STEP``
the same maps summed over the structures sampled during MD (``Engine.sampler_read``) go to
``analysis/distances_md.npz``, ``distances/member_<i>_md.npz`` and ``ensemble_distances_md.npz``: a file of
S sampled structures is their sum exactly as an ensemble file is the sum of its members (``members`` = S,
pair and bead counts S times one structure's), so every function below reads it unchanged.

* ``dist_sum``, ``dist2_sum``: uint64, the upper triangle p <= q of the B x B maps, flattened in
  ``np.triu_indices(B)`` order, in units of Q nm and Q nm^2 (every entry of a distance map is a sum over
  pairs that exist, so a sparse form gains nothing);
* ``pair_count``: uint64, upper triangle in the same order: bead pairs summed into each entry, n_p * n_q
  off the diagonal and n_p (n_p - 1) / 2 on it per member (n = the member's beads per bin);
* ``bin_beads``: uint64[B], beads in each bin, summed over members;
* ``radial_sum``, ``radial2_sum``: uint64[B], quantised r and r^2 summed over the bin's beads;
* ``members``, ``resolution_bp``, ``bin_chrom``, ``bin_start_bp``, ``quantum_log2`` (-24).

Members of a shuffled ensemble model the same loci, but the loader's rounding of the chromosome blocks can
move a bead across a bin edge, so their beads per bin may differ by one here and there.  Each file therefore
carries its own exact pair and bead counts, and the means divide exact sums by exact counts.  ``load``
returns the maps dense and symmetric.
"""
from __future__ import annotations

import numpy as np

from .contacts import GenomeBins, _write

QUANTUM_LOG2 = -24
Q = 2.0 ** QUANTUM_LOG2
MAX_BINS = 4096     # dense maps of mmm_distance_map (2 x 128 MB of uint64)
KEYS = ("dist_sum", "dist2_sum", "pair_count", "bin_beads", "radial_sum", "radial2_sum", "members", "resolution_bp",
        "bin_chrom", "bin_start_bp", "quantum_log2")
_MATCH = ("bin_chrom", "bin_start_bp", "resolution_bp", "quantum_log2")
_SUMS = ("dist_sum", "dist2_sum", "pair_count", "bin_beads", "radial_sum", "radial2_sum")
_MAPS = ("dist_sum", "dist2_sum", "pair_count")


def quantise(v) -> np.ndarray:
    """rint(v / Q) as uint64 (round half to even; the scaling by 2^24 is exact), as the kernel does."""
    return np.rint(np.asarray(v, np.float64) * 2.0 ** -QUANTUM_LOG2).astype(np.int64).astype(np.uint64)


def radial_sums(x, center, bins, n_bins: int) -> tuple[np.ndarray, np.ndarray]:
    """(radial_sum, radial2_sum), uint64[n_bins]: quantised distance r of every binned bead from ``center``
    and r^2 = (dx*dx + dy*dy) + dz*dz (FP64, this order), summed per bin exactly."""
    x = np.asarray(x, np.float64)
    d = x - np.asarray(center, np.float64)[None, :]
    r2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    bins = np.asarray(bins, np.int64)
    ok = bins >= 0
    rs, r2s = np.zeros(n_bins, np.uint64), np.zeros(n_bins, np.uint64)
    np.add.at(rs, bins[ok], quantise(np.sqrt(r2[ok])))
    np.add.at(r2s, bins[ok], quantise(r2[ok]))
    return rs, r2s


def result(dist_sum, dist2_sum, gb: GenomeBins, x, center, members: int = 1) -> dict:
    """The in-memory form of a distances file (dense maps) of one structure: the device maps of
    Engine.distance_map at bins ``gb``, and the radial sums of its positions ``x`` about ``center``."""
    rs, r2s = radial_sums(x, center, gb.bins, gb.n_bins)
    pairs, n = _counts(gb)
    return _result(dist_sum, dist2_sum, gb, pairs, n, rs, r2s, members)


def sampled_result(dist_sum, dist2_sum, gb: GenomeBins, radial_sum, radial2_sum, samples: int) -> dict:
    """The in-memory form of a distances file summed over ``samples`` structures of one run, all binned by
    ``gb`` (Engine.sampler_read, radial sums added per structure): ``members`` = samples, and the pair and
    bead counts are ``samples`` times one structure's, as in an ensemble file of that many members."""
    pairs, n = _counts(gb)
    s = np.uint64(samples)
    return _result(dist_sum, dist2_sum, gb, pairs * s, n * s, radial_sum, radial2_sum, samples)


def _counts(gb: GenomeBins) -> tuple[np.ndarray, np.ndarray]:
    """(pair_count (B, B), bin_beads (B,)) of one structure binned by ``gb``."""
    bins = np.asarray(gb.bins, np.int64)
    n = np.bincount(bins[bins >= 0], minlength=gb.n_bins).astype(np.uint64)
    pairs = np.outer(n, n)
    pairs[np.diag_indices(gb.n_bins)] = n * (n - np.uint64(1)) // np.uint64(2)  # 0 for an empty bin (wraps to 0 * ...)
    return pairs, n


def _result(dist_sum, dist2_sum, gb: GenomeBins, pairs, n, rs, r2s, members: int) -> dict:
    return dict(dist_sum=np.asarray(dist_sum, np.uint64), dist2_sum=np.asarray(dist2_sum, np.uint64),
                pair_count=pairs, bin_beads=n, radial_sum=np.asarray(rs, np.uint64),
                radial2_sum=np.asarray(r2s, np.uint64), members=np.int64(members),
                resolution_bp=np.int64(gb.resolution_bp), bin_chrom=np.asarray(gb.bin_chrom, np.int32),
                bin_start_bp=np.asarray(gb.bin_start_bp, np.int64), quantum_log2=np.int64(QUANTUM_LOG2))


def save(path: str, d: dict):
    b = len(d["bin_beads"])
    iu = np.triu_indices(b)
    out = {k: d[k] for k in KEYS}
    for k in _MAPS:
        out[k] = np.asarray(d[k], np.uint64)[iu]
    _write(path, out)


def load(path: str) -> dict:
    """A distances file, with the maps dense and symmetric."""
    with np.load(path) as z:
        if "dist_sum" not in z.files:
            raise ValueError(f"{path} is not a distances file")
        d = {k: z[k] for k in KEYS}
    b = len(d["bin_beads"])
    iu = np.triu_indices(b)
    for k in _MAPS:
        m = np.zeros((b, b), np.uint64)
        m[iu] = d[k]
        m.T[iu] = d[k]
        d[k] = m
    return d


def _add(a: np.ndarray, b: np.ndarray, path: str, key: str) -> np.ndarray:
    s = a + b  # uint64 wraps: a wrapped sum is smaller than either term
    if np.any(s < a):
        raise ValueError(f"{path}: {key} would overflow uint64 in the sum of the members")
    return s


def aggregate(paths) -> dict:
    """Sum of member files: exact uint64 (distance sums, pair and bead counts, radial sums), the same bytes in
    any member order.  ValueError naming the file when its bins, resolution or quantum differ from the other
    members', or when a sum would overflow uint64."""
    paths = list(paths)
    if not paths:
        raise ValueError("no distance files to aggregate")
    acc = None
    for p in paths:
        d = load(p)
        if acc is None:
            acc = dict(d)
            continue
        for k in _MATCH:
            if not np.array_equal(acc[k], d[k]):
                raise ValueError(f"{p}: {k} differs from the other members")
        for k in _SUMS:
            acc[k] = _add(acc[k], d[k], p, k)
        acc["members"] = np.int64(acc["members"] + int(d["members"]))
    return acc


def pair_counts(d: dict) -> np.ndarray:
    """float64 (B, B): bead pairs summed in every entry (``pair_count``)."""
    return np.asarray(d["pair_count"], np.float64)


def _ratio(num, den) -> np.ndarray:
    num = np.asarray(num, np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.nan)


def _q(d: dict) -> float:
    return 2.0 ** int(d["quantum_log2"])


def mean_distance(d: dict) -> np.ndarray:
    """Mean distance (nm) between the loci of every bin pair; NaN where there is no pair."""
    return _q(d) * _ratio(d["dist_sum"], pair_counts(d))


def rms_distance(d: dict) -> np.ndarray:
    """Root-mean-square distance (nm) of every bin pair; NaN where there is no pair."""
    return np.sqrt(_q(d) * _ratio(d["dist2_sum"], pair_counts(d)))


def std_distance(d: dict) -> np.ndarray:
    """Standard deviation (nm) of the distances of every bin pair (population form); NaN where there is no
    pair."""
    m = mean_distance(d)
    return np.sqrt(np.maximum(rms_distance(d) ** 2 - m * m, 0.0))


def radial_profile(d: dict) -> tuple[np.ndarray, np.ndarray]:
    """(mean, std) in nm of the distance of every bin's beads from the container centre; NaN for empty
    bins."""
    den = np.asarray(d["bin_beads"], np.float64)
    mean = _q(d) * _ratio(d["radial_sum"], den)
    rms2 = _q(d) * _ratio(d["radial2_sum"], den)
    return mean, np.sqrt(np.maximum(rms2 - mean * mean, 0.0))


def distance_sums(V, bins, n_bins: int, device: int = 0) -> tuple[np.ndarray, np.ndarray]:
    """(dist_sum, dist2_sum) of any (n, 3) coordinate array in nm, through a temporary Engine on `device`."""
    from .engine import Engine

    V = np.ascontiguousarray(V, dtype=np.float64)
    with Engine(len(V), device=device) as eng:
        eng.set_positions(V)
        return eng.distance_map(bins, n_bins)
