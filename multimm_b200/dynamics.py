"""Locus dynamics of MD runs (simulated live-cell imaging: tracked loci, two-colour labelled loop anchors, loop
lifetimes) — the one module that owns their format.

The structures sampled every ``MD_SAMPLE_STEP`` steps of a run are numbered s = 0, 1, ..., S - 1 in time order
(MD samples only: the minimised structure is not sample 0).  For a lag tau in the lag set (1, 2, 4, ...,
``DYNAMICS_MAX_LAG`` samples) the sample pairs are (s - tau, s), max(0, S - tau) of them.  On the device
(``Engine.dynamics_add``, ``mmm_dynamics_add``), in FP64 with ``d2 = (dx*dx + dy*dy) + dz*dz`` and the quantum
Q = 2^-24 of ``distances``:

* the **per-bin MSD**: the squared displacement of every bead between the two samples of a pair, summed per lag
  and canonical genomic bin (``contacts.genome_bins``).  No drift or centre-of-mass correction is applied, so a
  drifting or rotating structure adds its drift;
* the **two-anchor MSD** of every loop row of ``loops``: the squared change of the anchor vector R = x_hi - x_lo,
  which needs no drift correction.  2 <R^2> - MSD_rel(tau) is twice the vector autocorrelation at tau, with <R^2>
  the loop readout's ``dist2_sum``;
* the **loop state**: a row is closed in a sample when its anchors are in contact (``CONTACT_RADIUS``, the loop
  readout's verdict) and open otherwise.  A run is a maximal stretch of samples in one state.  A run that begins
  and ends at an observed change is *complete*; one that began before sample 0 and ends at a change is
  *left-censored*; one still in progress at the last sample is *right-censored* when it began at a change, and a
  row that never changed is one *whole-window* run.

Files (numpy ``.npz``): ``analysis/dynamics.npz`` of a single run, ``dynamics/member_<i>.npz`` of an ensemble
member and ``ensemble_dynamics.npz``, the exact sum of the members that succeeded.  State index k: 0 closed,
1 open; group g: 0 enforced, 1 held out (``loops``).

* ``lags`` (int64[L]), ``members`` (runs summed), ``samples`` (structures summed), ``sample_step`` (MD steps
  between samples), ``dt_ps`` (ps per MD step), ``radius_nm``, ``quantum_log2`` (-24), ``bead_bp_min`` /
  ``bead_bp_max``;
* the bins: ``bin_chrom``, ``bin_start_bp``, ``resolution_bp``; ``msd_sum`` and ``msd_pairs`` uint64 [L][B] (Q nm^2
  and bead-sample pairs; members' beads per bin can differ by one, so the pairs are stored);
* the loop table (``loops.TABLE_KEYS``) and per row, uint64 over the whole table: ``measured`` (samples in which the
  row was valid), ``rel_msd_sum`` / ``rel_pairs`` [L][R], ``closed_runs``, ``closed_len``, ``open_runs``,
  ``open_len`` (complete runs), ``right_runs``, ``right_len``, ``whole_runs``, ``whole_len`` [2][R] (by state);
* per group: ``rel_group_sum`` / ``rel_group_pairs`` [2][L]; ``hist`` [2][2][64] (complete runs by floor(log2
  length)), ``hist_len``, ``left_runs``, ``left_len``, ``group_right_runs``, ``group_right_len``,
  ``group_whole_runs``, ``group_whole_len`` [2][2].
"""
from __future__ import annotations

import numpy as np

from .contacts import GenomeBins, _write
from .distances import QUANTUM_LOG2, _add
from .loops import TABLE_KEYS

MAX_BINS = 2**22    # mmm_dynamics_configure: dense [lags][bins] sums, 32 MB per lag at the cap
MAX_LAG = 4096      # samples
DEFAULT_MAX_LAG = 64
BIN_KEYS = ("bin_chrom", "bin_start_bp", "resolution_bp")
ROW_SUMS = ("measured", "rel_msd_sum", "rel_pairs", "closed_runs", "closed_len", "open_runs", "open_len",
            "right_runs", "right_len", "whole_runs", "whole_len")
GROUP_SUMS = ("rel_group_sum", "rel_group_pairs", "hist", "hist_len", "left_runs", "left_len", "group_right_runs",
              "group_right_len", "group_whole_runs", "group_whole_len")
SUMS = ("msd_sum", "msd_pairs") + ROW_SUMS + GROUP_SUMS
KEYS = ("lags", "members", "samples", "sample_step", "dt_ps", "radius_nm", "quantum_log2", "bead_bp_min",
        "bead_bp_max") + BIN_KEYS + TABLE_KEYS + SUMS
_MATCH = ("lags", "sample_step", "dt_ps", "radius_nm", "quantum_log2") + BIN_KEYS + TABLE_KEYS


def lag_set(max_lag: int) -> np.ndarray:
    """int32 lags 1, 2, 4, ..., max_lag (a power of two in [1, MAX_LAG]), in samples."""
    m = int(max_lag)
    if not (1 <= m <= MAX_LAG and m & (m - 1) == 0):
        raise ValueError(f"DYNAMICS_MAX_LAG={m} must be a power of two in [1, {MAX_LAG}] samples")
    return (1 << np.arange(m.bit_length(), dtype=np.int64)).astype(np.int32)


def _open_runs(read: dict, r: int) -> tuple[np.ndarray, ...]:
    """(right_runs, right_len, whole_runs, whole_len) uint64 [2][r] of the runs in progress of a read."""
    k = np.where(np.asarray(read["closed"], bool), 0, 1)
    ln = np.asarray(read["length"], np.int64).astype(np.uint64)
    frm = np.asarray(read["from_transition"], bool)
    out = [np.zeros((2, r), np.uint64) for _ in range(4)]
    idx = np.arange(r)
    for j, sel in ((0, frm & (ln > 0)), (2, ~frm & (ln > 0))):
        out[j][k[sel], idx[sel]] = 1
        out[j + 1][k[sel], idx[sel]] = ln[sel]
    return tuple(out)


def result(read: dict, lags, gb: GenomeBins, tab: dict, mr: dict, radius_nm: float, sample_step: int,
           dt_ps: float) -> dict:
    """The in-memory form of a dynamics file of one run: ``read`` is what Engine.dynamics_read returns after the
    run's S samples, with bins ``gb`` and the device rows of ``loops.device_rows(mr)`` (the valid rows of the
    loop table ``tab``, in table order).  The denominators and the right-censored and whole-window counts are
    computed here; the device state is not changed."""
    lags = np.asarray(lags, np.int64)
    s = int(read["samples"])
    pairs = np.maximum(0, s - lags).astype(np.uint64)  # sample pairs per lag
    beads = np.bincount(np.asarray(gb.bins, np.int64)[np.asarray(gb.bins) >= 0], minlength=gb.n_bins).astype(np.uint64)
    v = np.asarray(mr["valid"], bool)
    R, rv = len(tab["row"]), int(v.sum())
    grp = np.asarray(mr["group"], np.int64)[v]
    d = {k: np.asarray(tab[k]) for k in TABLE_KEYS}
    d.update(lags=lags, members=np.int64(1), samples=np.int64(s), sample_step=np.int64(sample_step),
             dt_ps=np.float64(dt_ps), radius_nm=np.float64(radius_nm), quantum_log2=np.int64(QUANTUM_LOG2),
             bead_bp_min=np.int64(mr["resolution"]), bead_bp_max=np.int64(mr["resolution"]),
             bin_chrom=np.asarray(gb.bin_chrom, np.int32), bin_start_bp=np.asarray(gb.bin_start_bp, np.int64),
             resolution_bp=np.int64(gb.resolution_bp), msd_sum=np.asarray(read["msd_sum"], np.uint64),
             msd_pairs=pairs[:, None] * beads[None, :])
    per_row = dict(measured=np.full(rv, s, np.uint64)[None], rel_msd_sum=np.asarray(read["rel_msd_sum"], np.uint64),
                   rel_pairs=np.repeat(pairs[:, None], rv, axis=1))
    for k in ("closed_runs", "closed_len", "open_runs", "open_len"):
        per_row[k] = np.asarray(read[k], np.uint64)[None]
    right_runs, right_len, whole_runs, whole_len = _open_runs(read, rv)
    per_row.update(right_runs=right_runs, right_len=right_len, whole_runs=whole_runs, whole_len=whole_len)
    for k, a in per_row.items():  # onto the whole table: zero for a row that is not valid for this run
        full = np.zeros((a.shape[0], R), np.uint64)
        full[:, v] = a
        d[k] = full[0] if k in ("measured", "closed_runs", "closed_len", "open_runs", "open_len") else full
    by_group = lambda a: np.stack([a[..., grp == g].sum(axis=-1, dtype=np.uint64) for g in (0, 1)])  # noqa: E731
    d.update(rel_group_sum=by_group(per_row["rel_msd_sum"]), rel_group_pairs=by_group(per_row["rel_pairs"]),
             hist=np.asarray(read["hist"], np.uint64), hist_len=np.asarray(read["hist_len"], np.uint64),
             left_runs=np.asarray(read["left_runs"], np.uint64), left_len=np.asarray(read["left_len"], np.uint64),
             group_right_runs=by_group(right_runs), group_right_len=by_group(right_len),
             group_whole_runs=by_group(whole_runs), group_whole_len=by_group(whole_len))
    return d


def save(path: str, d: dict):
    _write(path, {k: d[k] for k in KEYS})


def load(path: str) -> dict:
    with np.load(path) as z:
        if "rel_msd_sum" not in z.files or "lags" not in z.files:
            raise ValueError(f"{path} is not a dynamics file")
        return {k: z[k] for k in KEYS}


def aggregate(paths) -> dict:
    """Sum of dynamics files: exact uint64, the same bytes in any member order.  ValueError naming the file when
    its lags, bins, loop table, radius, sample step, time step or quantum differ from the other members', or when
    a sum would overflow uint64."""
    paths = list(paths)
    if not paths:
        raise ValueError("no dynamics files to aggregate")
    acc = None
    for p in paths:
        d = load(p)
        if acc is None:
            acc = dict(d)
            continue
        for k in _MATCH:
            if acc[k].shape != d[k].shape or not np.array_equal(acc[k], d[k]):
                raise ValueError(f"{p}: {k} differs from the other members")
        for k in SUMS:
            acc[k] = _add(acc[k], d[k], p, k)
        for k in ("members", "samples"):
            acc[k] = np.int64(acc[k] + int(d[k]))
        acc["bead_bp_min"] = np.int64(min(int(acc["bead_bp_min"]), int(d["bead_bp_min"])))
        acc["bead_bp_max"] = np.int64(max(int(acc["bead_bp_max"]), int(d["bead_bp_max"])))
    return acc


def _ratio(num, den) -> np.ndarray:
    num, den = np.asarray(num, np.float64), np.asarray(den, np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.nan)


def _q(d: dict) -> float:
    return 2.0 ** int(d["quantum_log2"])


def msd(d: dict) -> np.ndarray:
    """float64 [L][B]: mean squared displacement (nm^2) of the beads of every bin at every lag; NaN where no
    bead-sample pair was summed."""
    return _q(d) * _ratio(d["msd_sum"], d["msd_pairs"])


def relative_msd(d: dict) -> tuple[np.ndarray, np.ndarray]:
    """(per row float64 [L][R], per group float64 [2][L]): mean squared change (nm^2) of the anchor vector of
    every loop row, and over the rows of each group (0 enforced, 1 held out); NaN where no pair was summed."""
    return _q(d) * _ratio(d["rel_msd_sum"], d["rel_pairs"]), _q(d) * _ratio(d["rel_group_sum"], d["rel_group_pairs"])


def exponent(lags, m) -> np.ndarray:
    """float64 [L - 1][...]: the local log-log slope of the MSDs ``m`` ([L][...], as msd or relative_msd give
    them) between consecutive lags, d log MSD / d log tau (1 for free diffusion, about 0.5 for a Rouse chain);
    NaN where either MSD is not positive."""
    lags = np.asarray(lags, np.float64)
    m = np.asarray(m, np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        lm = np.where(m > 0, np.log(np.where(m > 0, m, 1.0)), np.nan)
    dl = np.diff(np.log(lags)).reshape((-1,) + (1,) * (m.ndim - 1))
    return np.diff(lm, axis=0) / dl


def lifetimes(d: dict) -> dict:
    """Per group (0 enforced, 1 held out) and state (0 closed, 1 open), arrays [2][2]: ``mean_ps``, the mean
    length of the complete runs in ps (length x MD_SAMPLE_STEP x SIM_INTEGRATOR_STEP; NaN with no complete run);
    ``complete``, ``left``, ``right``, ``whole``, the counts of complete, left-censored, right-censored and
    whole-window runs; and ``hist`` [2][2][64], the complete runs by floor(log2 length in samples)."""
    hist = np.asarray(d["hist"], np.uint64)
    complete = hist.sum(axis=-1, dtype=np.uint64)
    step_ps = float(d["sample_step"]) * float(d["dt_ps"])
    return dict(mean_ps=step_ps * _ratio(d["hist_len"], complete), complete=complete, hist=hist,
                left=np.asarray(d["left_runs"], np.uint64), right=np.asarray(d["group_right_runs"], np.uint64),
                whole=np.asarray(d["group_whole_runs"], np.uint64))
