"""Timing of the locus-dynamics add (mmm_dynamics_add) on one GPU, beside its numpy restatement on the host.

    python scripts/gpu_dynamics_timing.py --out profiles/r09_dynamics.json   (also writes profiles/r09_dynamics.md)

1. Device time of one add (CUDA events of mmm_dynamics_add, from the first kernel to the end of the ring copy) and
   its wall time (the guard's bounding-box pass and both host waits included), at N = 2e4 (tests/common.make_case,
   minimised for 300 L-BFGS iterations) and N = 2e5 (the genome-wide system built as bench.py builds it, after the
   two-stage minimisation, MIN_COARSE_CUTOFF = 0.5 nm), for lags 1, 2, ..., 64 and 1, 2, ..., 1024, with and
   without loop rows (those of a synthetic.write_bedpe file of about 4 000 rows, placed by the loader's own
   arithmetic, DOWNSAMPLING_PROB = 0.5).  Bins: about 1000 canonical genomic bins (N = 2e5) or 1000 runs of beads
   (N = 2e4).  The structures cycle through three perturbations of the minimised one (Gaussian noise of 0.05 nm),
   so that no lag of the set pairs a structure with itself; the timed adds follow L adds that fill the ring, so
   every lag is active.  The bytes an add must move are (2 + lags) 24 N (read x, the lagged ring slots, write the
   ring slot) plus, per row, the row, its state and the anchors' positions now and at every lag; bytes/s is that
   over the device time.  At lags up to 64 the device sums are compared bit for bit with the numpy restatement
   (tests/dynamics_ref.py), whose host time is reported.
2. At N = 2e4, MD wall time of 2000 steps in chunks of 100 with and without an add after every chunk, alternating,
   twice each.
The card's name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")]

from gpu_contacts_timing import card, write  # noqa: E402
from gpu_loops_timing import member_rows  # noqa: E402

RC = 0.2


def lag_set(max_lag):
    from multimm_b200 import dynamics

    return dynamics.lag_set(max_lag)


def bytes_per_add(n, n_lags, n_rows):
    return (2 + n_lags) * 24 * n + n_rows * (16 + 24 + 48 + n_lags * (48 + 16))


def per_add(eng, xs, max_lag, bins, nb, rows, reps, label, log, check):
    import dynamics_ref as DR

    lags = lag_set(max_lag)
    r = 0 if rows is None else len(rows["bead_lo"])
    kw = {} if rows is None else dict(bead_lo=rows["bead_lo"], bead_hi=rows["bead_hi"], group=rows["group"])
    eng.dynamics_configure(RC, lags, bins, nb, **kw)
    seq = [xs[s % len(xs)] for s in range(max_lag + reps)]
    for x in seq[:max_lag]:  # fill the ring: every lag is active in the timed adds
        eng.set_positions(x)
        eng.dynamics_add()
    ms0 = eng.dynamics_read()["device_ms"]
    wall = 0.0
    for x in seq[max_lag:]:
        eng.set_positions(x)
        t0 = time.perf_counter()
        eng.dynamics_add()
        wall += time.perf_counter() - t0
    got = eng.dynamics_read()
    ms = (got["device_ms"] - ms0) / reps
    nbytes = bytes_per_add(eng.n, len(lags), r)
    out = dict(system=label, n=eng.n, max_lag=max_lag, lags=len(lags), rows=r, bins=nb, adds_timed=reps,
               device_ms_per_add=ms, wall_ms_per_add=1e3 * wall / reps, bytes_per_add=nbytes,
               bytes_per_s=nbytes / (ms * 1e-3), ring_bytes=24 * eng.n * max_lag)
    if check:
        t0 = time.perf_counter()
        want = DR.dynamics(seq, lags, RC, bins, nb, kw.get("bead_lo"), kw.get("bead_hi"), kw.get("group"))
        out["host_numpy_s"] = time.perf_counter() - t0
        out["structures"] = len(seq)
        out["device_equals_numpy"] = all(want[k] is None or np.array_equal(np.asarray(got[k]), want[k])
                                         for k in DR.KEYS)
    log(out)
    return out


def perturbed(x, k, seed):
    rng = np.random.default_rng(seed)
    return [x + rng.normal(scale=0.05, size=x.shape) for _ in range(k)]


def md_wall(eng, bins, nb, rows, chunks, log):
    runs = []
    for order in ((False, True), (True, False)):
        for added in order:
            eng.md_configure("langevin", dt_ps=0.001, seed=5)
            eng.set_velocities_to_temperature(310.0, seed=6)
            eng.dynamics_configure(RC, lag_set(64), bins, nb, rows["bead_lo"], rows["bead_hi"], rows["group"])
            eng.md_run(100, want_report=True)  # warm-up
            t0 = time.perf_counter()
            for _ in range(chunks):
                eng.md_run(100, want_report=False)
                if added:
                    eng.dynamics_add()
            eng.get_positions()  # ends in a device synchronise
            wall = time.perf_counter() - t0
            runs.append(dict(added=added, steps=100 * chunks, wall_s=wall, adds=eng.dynamics_read()["samples"]))
            log(runs[-1])
    off = [r["wall_s"] for r in runs if not r["added"]]
    on = [r["wall_s"] for r in runs if r["added"]]
    return dict(runs=runs, overhead=float(np.mean(on) / np.mean(off) - 1.0))


def markdown(result) -> str:
    c = result["card"]
    lines = [f"# Locus dynamics: one add (mmm_dynamics_add)", "",
             f"Measured by `scripts/gpu_dynamics_timing.py` on one {c['name']} at a {c['power_limit']} power limit "
             f"(max SM clock {c['max_sm_clock']}).", "",
             "| system | N | lags (max) | rows | bins | device ms / add | wall ms / add | MB moved | GB/s | numpy s | equal |",
             "|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in result["per_add"]:
        lines.append(f"| {r['system']} | {r['n']} | {r['lags']} ({r['max_lag']}) | {r['rows']} | {r['bins']} | "
                     f"{r['device_ms_per_add']:.4f} | {r['wall_ms_per_add']:.3f} | {r['bytes_per_add'] / 1e6:.1f} | "
                     f"{r['bytes_per_s'] / 1e9:.0f} | {r.get('host_numpy_s', float('nan')):.2f} | "
                     f"{r.get('device_equals_numpy', '-')} |")
    md = result["md_wall_20k"]
    lines += ["", f"MD at N = 2e4, 2000 steps in chunks of 100, an add (lags to 64, rows and bins) after every chunk: "
                  f"{md['overhead']:.2%} more wall time (alternated, twice each):", ""]
    lines += [f"- add {r['added']}: {r['wall_s']:.3f} s" for r in md["runs"]]
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    opt = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing measured")
    import bench
    from common import make_case, to_engine
    from multimm_b200 import contacts

    def log(msg):
        print(msg, flush=True)

    result = dict(card=card(), per_add=[])
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        eng = to_engine(make_case(20_000, n_chrom=2, seed=1))
        eng.minimize(tol=10.0, max_iter=300)
        bins20 = (np.arange(20_000) * 1000 // 20_000).astype(np.int32)
        rows20, _ = member_rows(20_000, 4_000, 2, tmp)
        xs = perturbed(eng.get_positions(), 3, 1)
        for max_lag in (64, 1024):
            for rows in (None, rows20):
                result["per_add"].append(per_add(eng, xs, max_lag, bins20, 1000, rows, opt.reps,
                                                 "N=2e4 make_case, minimised", log, max_lag == 64))
        eng.set_positions(xs[0])
        result["md_wall_20k"] = md_wall(eng, bins20, 1000, rows20, 20, log)
        log(f"MD overhead of a dynamics add every 100 steps: {result['md_wall_20k']['overhead']:.2%}")
        eng.close()
        m = bench.build_model("gw", 0, 0, tmp)
        try:
            m.args.MIN_COARSE_CUTOFF = 0.5
            m.min_energy(write_files=False)
            n = m.engine.n
            gb = contacts.genome_bins(m.layout, 0, n_beads=n)
            rows, table_rows = member_rows(n, 4_000, 1, tmp)
            log(f"{table_rows} table rows, {len(rows['bead_lo'])} valid at N = {n}, {gb.n_bins} bins")
            xs = perturbed(m.engine.get_positions(), 3, 2)
            for max_lag in (64, 1024):
                for rw in (None, rows):
                    result["per_add"].append(per_add(m.engine, xs, max_lag, gb.bins, gb.n_bins, rw, opt.reps,
                                                     "N=2e5 genome-wide, two-stage minimised", log, max_lag == 64))
        finally:
            m.close()
    write(opt.out, result, log)
    md_path = os.path.splitext(opt.out)[0] + ".md"
    with open(md_path, "w") as fh:
        fh.write(markdown(result))
    log(f"wrote {md_path}")


if __name__ == "__main__":
    main()
