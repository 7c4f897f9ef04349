"""Timing of the trajectory sampler (mmm_sample) on one GPU, and its outputs against the host alternative.

    python scripts/gpu_md_sampling_timing.py --out profiles/r06_md_sampling.json

1. Device time per sample of each map alone (CUDA events of mmm_sample, summed by mmm_sampler_read, over
   `reps` samples of one structure after a warm-up): dense contact map (1000 bins), fine map (one bin per
   bead), distance maps (1000 bins), and all three together, at
   * N = 2e4, a synthetic system (tests/common.make_case) minimised for 300 L-BFGS iterations;
   * N = 2e5, the genome-wide system built as bench.py builds it, after the two-stage minimisation
     (MIN_COARSE_CUTOFF = 0.5 nm).
2. At N = 2e4 over an MD run (Langevin, 100 steps between samples, 100 samples): the fine map's device
   time per sample against the accumulated entries, beside the host alternative (mmm_contacts_sparse at the
   same positions, then contacts._merge into the host-side sum), timed per sample; the two results
   compared for equality at the end.
3. At N = 2e4, MD wall time of 2000 steps in chunks of 100 with and without a sample of all three maps after
   every chunk (with the driver's host-side radial sums), alternating, twice each.
The card's name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scripts"), os.path.join(ROOT, "tests")]

from gpu_contacts_timing import card, write  # noqa: E402

RC = 0.2


def fine_entries(eng):
    e, ms = C.c_int64(), C.c_float()
    eng._ck(eng._lib.mmm_sampler_read(eng._h, None, None, None, None, C.byref(e), None, None, C.byref(ms)))
    return int(e.value), float(ms.value)


def per_map(eng, reps, label):
    n = eng.n
    coarse = (np.arange(n) * 1000 // n).astype(np.int32)
    bead = np.arange(n, dtype=np.int32)
    cases = {"dense contacts (1000 bins)": dict(contact_bins=coarse, n_contact_bins=1000),
             "dense + fine contacts (one bin per bead)": dict(contact_bins=coarse, n_contact_bins=1000,
                                                               fine_bins=bead, n_fine_bins=n),
             "distances (1000 bins)": dict(distance_bins=coarse, n_distance_bins=1000),
             "all three": dict(contact_bins=coarse, n_contact_bins=1000, fine_bins=bead, n_fine_bins=n,
                               distance_bins=coarse, n_distance_bins=1000)}
    out = []
    for name, kw in cases.items():
        eng.sampler_configure(RC, **kw)
        eng.sample()  # warm-up: scratch, module load
        eng.sampler_configure(RC, **kw)
        t0 = time.perf_counter()
        for _ in range(reps):
            eng.sample()
        wall = time.perf_counter() - t0
        r = eng.sampler_read()
        out.append(dict(system=label, n=n, maps=name, samples=reps, device_ms_per_sample=r["device_ms"] / reps,
                        wall_ms_per_sample=1e3 * wall / reps, fine_entries=None if r["vals"] is None else len(r["vals"])))
    return out


def merge_growth(eng, samples, log):
    from multimm_b200 import contacts

    n = eng.n
    bead = np.arange(n, dtype=np.int32)
    eng.md_configure("langevin", dt_ps=0.001, seed=3)
    eng.set_velocities_to_temperature(310.0, seed=4)
    eng.sampler_configure(RC, np.zeros(n, np.int32), 1, bead, n)
    rows = []
    acc = None
    last_ms = 0.0
    for k in range(samples):
        eng.md_run(100, want_report=False)
        eng.sample()
        entries, ms = fine_entries(eng)
        t0 = time.perf_counter()
        r, c, v, _ = eng.contacts_sparse(RC, bead, n)
        t1 = time.perf_counter()
        acc = (r, c, v) if acc is None else contacts._merge(*acc, r, c, v, n)
        t2 = time.perf_counter()
        rows.append(dict(sample=k + 1, accumulated_entries=entries, structure_entries=len(v),
                         device_ms=ms - last_ms, host_one_shot_ms=1e3 * (t1 - t0), host_merge_ms=1e3 * (t2 - t1)))
        last_ms = ms
        if (k + 1) % 20 == 0:
            log(rows[-1])
    got = eng.sampler_read()
    equal = all(np.array_equal(g, w) for g, w in zip((got["rows"], got["cols"], got["vals"]), acc))
    log(f"device fine map == host merge of the one-shot maps over {samples} samples: {equal}")
    return dict(per_sample=rows, equal=equal, samples=samples, entries=len(got["vals"]))


def md_wall(eng, chunks, log):
    from multimm_b200 import distances

    n = eng.n
    coarse = (np.arange(n) * 1000 // n).astype(np.int32)
    runs = []
    for order in ((False, True), (True, False)):
        for sampled in order:
            eng.md_configure("langevin", dt_ps=0.001, seed=5)
            eng.set_velocities_to_temperature(310.0, seed=6)
            eng.sampler_configure(RC, coarse, 1000, np.arange(n, dtype=np.int32), n, coarse, 1000)
            eng.md_run(100, want_report=True)  # warm-up
            t0 = time.perf_counter()
            for _ in range(chunks):
                eng.md_run(100, want_report=False)
                if sampled:
                    eng.sample()
                    distances.radial_sums(eng.get_positions(), np.zeros(3), coarse, 1000)
            eng.get_positions()  # ends in a device synchronise
            wall = time.perf_counter() - t0
            runs.append(dict(sampled=sampled, steps=100 * chunks, wall_s=wall))
            log(runs[-1])
    off = [r["wall_s"] for r in runs if not r["sampled"]]
    on = [r["wall_s"] for r in runs if r["sampled"]]
    return dict(runs=runs, overhead=float(np.mean(on) / np.mean(off) - 1.0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--samples", type=int, default=100)
    opt = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing measured")
    from common import make_case, to_engine

    def log(msg):
        print(msg, flush=True)

    result = dict(card=card())
    log(f"card: {result['card']}")
    eng = to_engine(make_case(20_000, n_chrom=2, seed=1))
    eng.minimize(tol=10.0, max_iter=300)
    result["per_map_20k"] = per_map(eng, opt.reps, "N=2e4, 300 L-BFGS iterations")
    for r in result["per_map_20k"]:
        log(r)
    result["merge_growth_20k"] = merge_growth(eng, opt.samples, log)
    result["md_wall_20k"] = md_wall(eng, 20, log)
    log(f"MD overhead of sampling every 100 steps: {result['md_wall_20k']['overhead']:.2%}")
    eng.close()
    import bench

    with tempfile.TemporaryDirectory() as tmp:
        m = bench.build_model("gw", 0, 0, tmp)
        try:
            m.args.MIN_COARSE_CUTOFF = 0.5
            m.min_energy(write_files=False)
            result["per_map_200k"] = per_map(m.engine, max(3, opt.reps // 3), "N=2e5 genome-wide, two-stage minimised")
            for r in result["per_map_200k"]:
                log(r)
        finally:
            m.close()
    write(opt.out, result, log)


if __name__ == "__main__":
    main()
