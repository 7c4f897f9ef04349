"""Timing of the loop readout (mmm_loops_add) on one GPU, beside its numpy restatement on the host.

    python scripts/gpu_loops_timing.py --out profiles/r07_loops.json

1. Device time of one add (CUDA events of mmm_loops_add, summed by mmm_loops_read over `reps` adds after a
   warm-up) at N = 2e5: the genome-wide system built as bench.py builds it, after the two-stage minimisation
   (MIN_COARSE_CUTOFF = 0.5 nm).  The rows are those of synthetic.write_bedpe files of about 4 000 rows (the
   size of the reference's ENCODE loop fixture) and 1e5 rows, placed on the 2e5 beads by the loader's own
   arithmetic (genome-wide, no shuffle, DOWNSAMPLING_PROB = 0.5 so both groups are populated), at W = 10 and
   W = 25.  The counted work is R (2W + 1)^2 pair tests (tests/loops_ref.py counts the same pairs); pairs/s is
   that over the device time.  The same add in the numpy restatement, timed on the host, and compared bit for
   bit with the device sums.
2. At N = 2e4 (tests/common.make_case, minimised for 300 L-BFGS iterations, 4 000 rows on its beads, W = 10),
   MD wall time of 2000 steps in chunks of 100 with and without an add after every chunk, alternating, twice
   each.
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

RC = 0.2


def member_rows(n, n_rows, seed, tmp):
    """Device rows of a synthetic loop file of about n_rows rows, as a genome-wide member of n beads measures it."""
    from multimm_b200 import loaders, loops, synthetic

    path = os.path.join(tmp, f"loops_{n_rows}.bedpe")
    synthetic.write_bedpe(path, n_rows, seed=seed)
    lay = {}
    ms, ns, *_ = loaders.import_mns_from_bedpe(path, N_beads=n, path=None, down_prob=0.5, seed=seed, layout=lay)
    mr = loops.member_rows(loops.table(path), lay, n, ms, ns)
    return loops.device_rows(mr), len(mr["valid"])


def pairs_tested(rows, w):
    """Window pairs of the rows inside their blocks with lo + a < hi + b: the pairs the kernel tests."""
    from multimm_b200 import loops

    mr = dict(lo=rows["bead_lo"], hi=rows["bead_hi"], first_lo=rows["first_lo"], end_lo=rows["end_lo"],
              first_hi=rows["first_hi"], end_hi=rows["end_hi"], group=rows["group"],
              valid=np.ones(len(rows["bead_lo"]), bool))
    return int(loops.window_pairs(mr, w).sum())


def per_add(eng, rows, w, reps, label, log):
    import loops_ref as LR

    r = len(rows["bead_lo"])
    eng.loops_configure(RC, w, **rows)
    eng.loops_add()  # warm-up: buffers, module load, shared-memory attribute
    eng.loops_configure(RC, w, **rows)
    t0 = time.perf_counter()
    for _ in range(reps):
        eng.loops_add()
    wall = time.perf_counter() - t0
    got = eng.loops_read()
    ms = got["device_ms"] / reps
    x = eng.get_positions()
    t0 = time.perf_counter()
    want = LR.loop_sums(x, rows, RC, w)
    host = time.perf_counter() - t0
    equal = all(np.array_equal(got[k], np.uint64(reps) * want[k]) for k in want)
    work = r * (2 * w + 1) ** 2
    out = dict(system=label, n=eng.n, rows=r, window=w, adds=reps, device_ms_per_add=ms, wall_ms_per_add=1e3 * wall / reps,
               pair_tests=work, pairs_in_blocks=pairs_tested(rows, w), pair_tests_per_s=work / (ms * 1e-3),
               host_numpy_ms=1e3 * host, host_over_device=1e3 * host / ms, device_equals_numpy=equal)
    log(out)
    return out


def md_wall(eng, rows, chunks, log):
    runs = []
    for order in ((False, True), (True, False)):
        for sampled in order:
            eng.md_configure("langevin", dt_ps=0.001, seed=5)
            eng.set_velocities_to_temperature(310.0, seed=6)
            eng.loops_configure(RC, 10, **rows)
            eng.md_run(100, want_report=True)  # warm-up
            t0 = time.perf_counter()
            for _ in range(chunks):
                eng.md_run(100, want_report=False)
                if sampled:
                    eng.loops_add()
            eng.get_positions()  # ends in a device synchronise
            wall = time.perf_counter() - t0
            runs.append(dict(sampled=sampled, steps=100 * chunks, wall_s=wall,
                             adds=eng.loops_read()["samples"]))
            log(runs[-1])
    off = [r["wall_s"] for r in runs if not r["sampled"]]
    on = [r["wall_s"] for r in runs if r["sampled"]]
    return dict(runs=runs, overhead=float(np.mean(on) / np.mean(off) - 1.0))


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

    def log(msg):
        print(msg, flush=True)

    result = dict(card=card())
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        m = bench.build_model("gw", 0, 0, tmp)
        try:
            m.args.MIN_COARSE_CUTOFF = 0.5
            m.min_energy(write_files=False)
            result["per_add_200k"] = []
            for n_rows in (4_000, 100_000):
                rows, table_rows = member_rows(m.engine.n, n_rows, 1, tmp)
                log(f"{table_rows} table rows, {len(rows['bead_lo'])} valid at N = {m.engine.n}")
                for w in (10, 25):
                    result["per_add_200k"].append(per_add(m.engine, rows, w, opt.reps,
                                                          "N=2e5 genome-wide, two-stage minimised", log))
        finally:
            m.close()
        eng = to_engine(make_case(20_000, n_chrom=2, seed=1))
        eng.minimize(tol=10.0, max_iter=300)
        rows, _ = member_rows(20_000, 4_000, 2, tmp)
        result["md_wall_20k"] = md_wall(eng, rows, 20, log)
        log(f"MD overhead of a loop add every 100 steps: {result['md_wall_20k']['overhead']:.2%}")
        eng.close()
    write(opt.out, result, log)


if __name__ == "__main__":
    main()
