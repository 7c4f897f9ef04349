"""The loop readout: did the ensemble form the loops it was given, and does it predict the loops it was not
given?  Per-loop contact frequencies and anchor distances and aggregate peak analysis (APA) of the rows of the
loop file (``LOOPS_PATH``) — the one module that owns their format.

**The table** (``table``) holds the rows of the bedpe that ``loaders.import_mns_from_bedpe`` reads, in file
order: all of them genome-wide, the rows its region filter keeps in chromosome, region and gene runs.  Row k
is the same loop in every ensemble member; rows are not deduplicated (two rows on one bead pair are two
entries).

**Per member** (``member_rows``), each row's anchor beads come from the loader's own arithmetic
(``loaders.loop_anchor_beads``: block offset or region start, integer division by the resolution, the
midpoint of each anchor, clamped to N - 1), so they follow the member's chromosome shuffle.  The measured pair
is ``(lo, hi) = (min, max)`` of the two anchor beads.  A row is *valid* for a member when both anchors name
modelled chromosomes and ``hi > lo + 2`` (the loader's ``min_loop_dist``).  Rows on chromosomes that are not
modelled are left out, although the loader aliases them into chr1's beads (SURVEY appendix A, Q5); so are
inter-chromosomal rows that pass a region filter.  A valid row is in group 0, *enforced*, when ``(lo, hi)`` is
one of the member's loop bonds ``(ms, ns)``, and in group 1, *held out*, when it is not: down-sampling
(``DOWNSAMPLING_PROB``) dropped it, its mean count is at or below the loader's threshold, or its second anchor
lies upstream of its first in the member's chain so that the loader drops it (only inter-chromosomal rows can
be oriented so; with shuffling it depends on the member).  Each anchor's APA window is bounded by the block of
the chain that holds its bead (``chr_ends`` clipped to [0, N]).

**Per structure** (``Engine.loops_add``, ``mmm_loops_add``), with ``d2 = (dx*dx + dy*dy) + dz*dz`` in FP64
and the quantum Q = 2^-24 of ``distances``: per row, the contact ``d2 < rc * rc`` and the quantised distance
and squared distance at ``(lo, hi)``; per group and offset (a, b) in [-W, W]^2, the same contact and distance
at ``(lo + a, hi + b)`` over the rows whose window pair lies in the two blocks with ``lo + a < hi + b``.

Files (numpy ``.npz``): ``analysis/loops.npz`` of a single run, ``loops/member_<i>.npz`` of an ensemble member
and ``ensemble_loops.npz`` of an ensemble; with ``MD_SAMPLE_STEP`` the same sums over the structures sampled
during MD in ``analysis/loops_md.npz``, ``loops/member_<i>_md.npz`` and ``ensemble_loops_md.npz``.  A file of
S structures is their sum exactly as an ensemble file is the sum of its members.

* the table: ``row`` (line index in the bedpe), ``chrom1``, ``start1``, ``end1``, ``chrom2``, ``start2``,
  ``end2``;
* per row, uint64[R] over the whole table: ``measured`` (structures in which the row was valid), ``enforced``
  (of those, structures of members that bond it), ``contacts``, ``dist_sum``, ``dist2_sum`` (units Q nm and
  Q nm^2); a row that was never valid is zero everywhere;
* APA, uint64 [2][2W+1][2W+1] (group, a + W, b + W): ``apa_contacts``, ``apa_dist_sum``, ``apa_pairs`` (the
  window pairs summed, computed from the table alone); ``apa_window`` (W);
* ``members`` (structures), ``radius_nm``, ``quantum_log2`` (-24), ``bead_bp_min`` / ``bead_bp_max`` (the
  smallest and largest bead resolution in bp of the members summed: it depends on the shuffle genome-wide).
"""
from __future__ import annotations

import numpy as np
import pandas as pd

from . import loaders
from .contacts import _write
from .distances import QUANTUM_LOG2, _add

MAX_WINDOW = 25     # mmm_loops_configure: the accumulators of both groups stay in shared memory
MIN_LOOP_DIST = 2   # the loader's min_loop_dist: a valid row has hi > lo + 2
TABLE_KEYS = ("row", "chrom1", "start1", "end1", "chrom2", "start2", "end2")
ROW_SUMS = ("measured", "enforced", "contacts", "dist_sum", "dist2_sum")
APA_SUMS = ("apa_contacts", "apa_dist_sum", "apa_pairs")
KEYS = TABLE_KEYS + ROW_SUMS + APA_SUMS + ("apa_window", "members", "radius_nm", "quantum_log2", "bead_bp_min",
                                            "bead_bp_max")
_MATCH = TABLE_KEYS + ("radius_nm", "apa_window", "quantum_log2")


def table(bedpe_file, chrom=None, coords=None) -> dict:
    """The loop table of a run: the rows of ``bedpe_file`` that import_mns_from_bedpe reads with the same
    ``chrom`` and ``coords``, in file order."""
    df = loaders.loop_rows(pd.read_csv(bedpe_file, header=None, sep="\t"), chrom, coords)
    return dict(row=df.index.to_numpy(np.int64), chrom1=df[0].to_numpy().astype(str),
                start1=df[1].to_numpy(np.int64), end1=df[2].to_numpy(np.int64), chrom2=df[3].to_numpy().astype(str),
                start2=df[4].to_numpy(np.int64), end2=df[5].to_numpy(np.int64))


def member_rows(tab: dict, layout: dict, n_beads: int, ms, ns, chrom=None) -> dict:
    """The rows of ``tab`` as one member measures them.  ``layout`` is what import_mns_from_bedpe filled for
    the member (MultiMM.layout), ``ms``, ``ns`` its loop bonds, ``chrom`` the run's chromosome (None
    genome-wide).  Returns int64[R] arrays ``lo``, ``hi``, ``first_lo``, ``end_lo``, ``first_hi``, ``end_hi``,
    ``group`` (0 enforced, 1 held out) and bool[R] ``valid``, plus ``resolution`` (bp per bead); the entries of
    an invalid row are meaningless."""
    n = int(n_beads)
    idxs = np.asarray(layout["chrom_idxs"], np.int64)
    ends = np.asarray(layout["ends"], np.int64)
    coords = None if chrom is None else (int(layout["start_bp"]), int(layout["stop_bp"]))
    df = pd.DataFrame({0: tab["chrom1"], 1: tab["start1"], 2: tab["end1"], 3: tab["chrom2"], 4: tab["start2"],
                       5: tab["end2"]})
    r = len(df)
    if r:
        m, nn, res, _ = loaders.loop_anchor_beads(df, idxs, ends, n, chrom, coords)
        if res != int(layout["resolution"]):
            raise ValueError(f"the loop table gives {res} bp per bead, the member's loader {layout['resolution']}")
    else:
        m = nn = np.zeros(0, np.int64)
    m, nn = np.minimum(m, n - 1), np.minimum(nn, n - 1)
    lo, hi = np.minimum(m, nn), np.maximum(m, nn)
    names = {chrom} if chrom is not None else {loaders.CHROM_NAMES[int(c)] for c in idxs}
    modelled = np.isin(tab["chrom1"], list(names)) & np.isin(tab["chrom2"], list(names))
    valid = modelled & (hi > lo + MIN_LOOP_DIST) & (lo >= 0)
    bonds = np.asarray(ms, np.int64) * n + np.asarray(ns, np.int64)
    group = np.where(np.isin(lo * n + hi, bonds), 0, 1).astype(np.int64)
    # the block of the chain that holds each anchor bead (chr_ends clipped to [0, N]: a monotone table)
    bounds = np.clip(np.asarray(layout["chr_ends"], np.int64), 0, n)
    k_lo = np.clip(np.searchsorted(bounds, lo, side="right") - 1, 0, len(bounds) - 2)
    k_hi = np.clip(np.searchsorted(bounds, hi, side="right") - 1, 0, len(bounds) - 2)
    return dict(lo=lo, hi=hi, first_lo=bounds[k_lo], end_lo=bounds[k_lo + 1], first_hi=bounds[k_hi],
                end_hi=bounds[k_hi + 1], group=group, valid=valid, resolution=int(layout["resolution"]))


def window_pairs(mr: dict, window: int) -> np.ndarray:
    """uint64 [2][2W+1][2W+1]: the window pairs (lo + a, hi + b) of the valid rows of each group that lie in
    the anchors' blocks with lo + a < hi + b — the denominators of one structure's APA sums."""
    w = int(window)
    span = 2 * w + 1
    v = np.asarray(mr["valid"], bool)
    lo, hi, g = mr["lo"][v], mr["hi"][v], mr["group"][v]
    off = np.arange(-w, w + 1)
    pl, ph = lo[:, None] + off, hi[:, None] + off
    in_lo = (pl >= mr["first_lo"][v][:, None]) & (pl < mr["end_lo"][v][:, None])
    in_hi = (ph >= mr["first_hi"][v][:, None]) & (ph < mr["end_hi"][v][:, None])
    out = np.zeros((2, span, span), np.uint64)
    for ia in range(span):
        ok = in_lo[:, ia:ia + 1] & in_hi & (pl[:, ia:ia + 1] < ph)
        for grp in (0, 1):
            out[grp, ia] = ok[g == grp].sum(axis=0)
    return out


def result(tab: dict, mr: dict, sums: dict, radius_nm: float, window: int, samples: int = 1) -> dict:
    """The in-memory form of a loops file of one member over ``samples`` structures: ``sums`` is what
    Engine.loops_read returns for the device rows of ``device_rows(mr)`` (valid rows, in table order)."""
    r = len(tab["row"])
    v = np.asarray(mr["valid"], bool)
    s = np.uint64(samples)
    d = {k: np.asarray(tab[k]) for k in TABLE_KEYS}
    d["measured"] = v.astype(np.uint64) * s
    d["enforced"] = (v & (mr["group"] == 0)).astype(np.uint64) * s
    for k in ("contacts", "dist_sum", "dist2_sum"):
        d[k] = np.zeros(r, np.uint64)
        d[k][v] = np.asarray(sums[k], np.uint64)
    d["apa_contacts"] = np.asarray(sums["apa_contacts"], np.uint64)
    d["apa_dist_sum"] = np.asarray(sums["apa_dist_sum"], np.uint64)
    d["apa_pairs"] = window_pairs(mr, window) * s
    d.update(apa_window=np.int64(window), members=np.int64(samples), radius_nm=np.float64(radius_nm),
             quantum_log2=np.int64(QUANTUM_LOG2), bead_bp_min=np.int64(mr["resolution"]),
             bead_bp_max=np.int64(mr["resolution"]))
    return d


def device_rows(mr: dict) -> dict:
    """The arguments of Engine.loops_configure for the valid rows of ``mr``, in table order."""
    v = np.asarray(mr["valid"], bool)
    return dict(bead_lo=mr["lo"][v], bead_hi=mr["hi"][v], first_lo=mr["first_lo"][v], end_lo=mr["end_lo"][v],
                first_hi=mr["first_hi"][v], end_hi=mr["end_hi"][v], group=mr["group"][v])


def save(path: str, d: dict):
    _write(path, {k: d[k] for k in KEYS})


def load(path: str) -> dict:
    with np.load(path) as z:
        if "apa_pairs" not in z.files:
            raise ValueError(f"{path} is not a loops file")
        return {k: z[k] for k in KEYS}


def aggregate(paths) -> dict:
    """Sum of loops files: exact uint64, the same bytes in any member order.  ValueError naming the file when
    its table, radius, window or quantum differ from the other members', or when a sum would overflow
    uint64."""
    paths = list(paths)
    if not paths:
        raise ValueError("no loops files to aggregate")
    acc = None
    for p in paths:
        d = load(p)
        if acc is None:
            acc = dict(d)
            continue
        for k in _MATCH:
            if acc[k].shape != d[k].shape or not np.array_equal(acc[k], d[k]):
                raise ValueError(f"{p}: {k} differs from the other members")
        for k in ROW_SUMS + APA_SUMS:
            acc[k] = _add(acc[k], d[k], p, k)
        acc["members"] = np.int64(acc["members"] + int(d["members"]))
        acc["bead_bp_min"] = np.int64(min(int(acc["bead_bp_min"]), int(d["bead_bp_min"])))
        acc["bead_bp_max"] = np.int64(max(int(acc["bead_bp_max"]), int(d["bead_bp_max"])))
    return acc


def _ratio(num, den) -> np.ndarray:
    num, den = np.asarray(num, np.float64), np.asarray(den, np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.nan)


def _q(d: dict) -> float:
    return 2.0 ** int(d["quantum_log2"])


def contact_frequency(d: dict) -> np.ndarray:
    """float64[R]: fraction of the structures that measured a row in which its anchors were in contact; NaN for
    a row never measured."""
    return _ratio(d["contacts"], d["measured"])


def mean_distance(d: dict) -> np.ndarray:
    """float64[R]: mean anchor distance (nm) of every row; NaN for a row never measured."""
    return _q(d) * _ratio(d["dist_sum"], d["measured"])


def std_distance(d: dict) -> np.ndarray:
    """float64[R]: standard deviation (nm, population form) of every row's anchor distance; NaN for a row never
    measured."""
    m = mean_distance(d)
    return np.sqrt(np.maximum(_q(d) * _ratio(d["dist2_sum"], d["measured"]) - m * m, 0.0))


def apa(d: dict, group: int) -> tuple[np.ndarray, np.ndarray]:
    """(contact frequency, mean distance in nm) of group ``group`` (0 enforced, 1 held out), float64
    [2W+1][2W+1] indexed by (a + W, b + W); NaN where no window pair was summed."""
    g = int(group)
    den = d["apa_pairs"][g]
    return _ratio(d["apa_contacts"][g], den), _q(d) * _ratio(d["apa_dist_sum"][g], den)


def apa_score(d: dict, group: int) -> float:
    """Peak to lower left (P2LL) of group ``group``'s APA contact frequency: the centre over the mean of the
    lower-left k x k corner, a in [W - k + 1, W] and b in [-W, -W + k - 1] with k = max(1, W // 3) (Juicer's
    3 x 3 corner at W = 10).  NaN when the centre or the corner has no pair, or the corner no contact."""
    freq, _ = apa(d, group)
    w = int(d["apa_window"])
    k = max(1, w // 3)
    corner = float(np.mean(freq[2 * w - k + 1:, :k]))
    centre = float(freq[w, w])
    if not (np.isfinite(corner) and np.isfinite(centre)) or corner == 0.0:
        return float("nan")
    return centre / corner
