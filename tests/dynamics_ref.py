"""numpy restatement of the locus-dynamics accumulator (mmm_dynamics_configure / _add / _read / _read_runs) over an
ordered list of structures: the lag pairs, the exact FP64 expressions and quantisation of the kernels, the per-row
state machine and its censoring.  Returns what Engine.dynamics_read returns (device_ms aside)."""
import numpy as np

from multimm_b200.distances import quantise


def _pair_d2(a, b):
    d = a - b
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def dynamics(xs, lags, rc, bins=None, n_bins=0, lo=None, hi=None, group=None):
    lags = [int(t) for t in lags]
    lo = np.zeros(0, np.int64) if lo is None else np.asarray(lo, np.int64)
    hi = np.zeros(0, np.int64) if hi is None else np.asarray(hi, np.int64)
    group = np.zeros(0, np.int64) if group is None else np.asarray(group, np.int64)
    r = len(lo)
    rc2 = float(rc) * float(rc)
    msd = np.zeros((len(lags), n_bins), np.uint64) if bins is not None else None
    if bins is not None:  # exact per-bin sums: sort the binned beads by bin, add runs in uint64
        bins = np.asarray(bins, np.int64)
        order = np.flatnonzero(bins >= 0)
        order = order[np.argsort(bins[order], kind="stable")]
        head = np.ones(len(order), bool)
        head[1:] = bins[order][1:] != bins[order][:-1]
        starts = np.flatnonzero(head)
        dest = bins[order][starts]
    rel = np.zeros((len(lags), r), np.uint64)
    runs = np.zeros((4, r), np.uint64)
    closed = np.zeros(r, bool)
    length = np.zeros(r, np.int64)
    frm = np.zeros(r, bool)
    hist = np.zeros((2, 2, 64), np.uint64)
    hist_len, left_runs, left_len = (np.zeros((2, 2), np.uint64) for _ in range(3))
    xs = [np.asarray(x, np.float64) for x in xs]
    for s, x in enumerate(xs):
        R = x[hi] - x[lo]
        for k, tau in enumerate(lags):
            if tau > s:
                break
            p = xs[s - tau]
            if bins is not None and len(order):
                q = quantise(_pair_d2(x[order], p[order]))
                msd[k, dest] += np.add.reduceat(q, starts)
            if r:
                e = R - (p[hi] - p[lo])
                rel[k] += quantise((e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2])
        if not r:
            continue
        c = _pair_d2(x[lo], x[hi]) < rc2
        first = length == 0
        same = ~first & (c == closed)
        ends = ~first & ~same
        kk = np.where(closed, 0, 1)  # state index of the run that ends: 0 closed, 1 open
        ln = length.astype(np.uint64)
        comp = ends & frm
        left = ends & ~frm
        for kstate in (0, 1):
            m = comp & (kk == kstate)
            runs[2 * kstate, m] += np.uint64(1)
            runs[2 * kstate + 1, m] += ln[m]
        if comp.any():
            bucket = np.floor(np.log2(length[comp].astype(np.float64))).astype(np.int64)
            np.add.at(hist, (group[comp], kk[comp], bucket), np.uint64(1))
            np.add.at(hist_len, (group[comp], kk[comp]), ln[comp])
        if left.any():
            np.add.at(left_runs, (group[left], kk[left]), np.uint64(1))
            np.add.at(left_len, (group[left], kk[left]), ln[left])
        length = np.where(same, length + 1, 1)
        frm = np.where(ends, True, frm)
        closed = c
    return dict(samples=len(xs), msd_sum=msd, rel_msd_sum=rel, closed_runs=runs[0], closed_len=runs[1],
                open_runs=runs[2], open_len=runs[3], closed=closed, length=length, from_transition=frm, hist=hist,
                hist_len=hist_len, left_runs=left_runs, left_len=left_len)


KEYS = ("msd_sum", "rel_msd_sum", "closed_runs", "closed_len", "open_runs", "open_len", "closed", "length",
        "from_transition", "hist", "hist_len", "left_runs", "left_len")
