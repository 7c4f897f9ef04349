"""Timing of simulated GAM (mmm_gam_add) on one GPU, beside the numpy restatement.

    python scripts/gpu_gam_timing.py --out profiles/r11_gam.json

writes the JSON and, beside it, the same numbers as a Markdown report (.md).

1. Device time of one add at N = 2e5 (the genome-wide system bench.py builds, after the two-stage minimisation,
   MIN_COARSE_CUTOFF = 0.5 nm), at the canonical bins of contacts.genome_bins (about 990 bins, and about 4096 at a
   finer resolution), with S = 1024 and S = 16384 slices of gam.slice_planes (GAM_SLICE_FRACTION 0.025) about the
   container centre.  The add's time is its CUDA events (mmm_gam_read's device_ms: plane upload, clears, both
   passes, the read-back of the slice bitset), mean over `reps` adds after a warm-up add.  The two passes are timed
   apart from the kernel durations torch.profiler records (CUDA activities) in a separate run of `reps` adds;
   from them, slab tests per second (N S over the detection pass) and POPC per second (B (B + 1) / 2 ceil(S / 32)
   over the co-segregation pass).  At S = 1024 the numpy restatement (tests/gam_ref.py) is timed on the host and
   compared with the device sums.
2. At N = 2e4 (tests/common.make_case, minimised for 300 L-BFGS iterations), MD wall time of 2000 steps in chunks
   of 100 with and without a GAM add after every chunk (1000 bins, S = 1024, the planes drawn on the host from the
   positions as the driver does), alternating, twice each.
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

FRACTION = 0.025


def pass_ms(eng, planes, h, reps):
    """Mean duration of k_gam_detect and k_gam_coseg per add, from torch.profiler's CUDA kernel records."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            eng.gam_add(planes, h)
        torch.cuda.synchronize()
    out = {"k_gam_detect": None, "k_gam_coseg": None}
    for ev in prof.key_averages():
        for name in out:
            if name in ev.key:
                total = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                out[name] = (out[name] or 0.0) + total / 1e3 / reps  # us -> ms per add
    return out


def per_add(eng, system, center, gb, slices, reps, log, check=False):
    import gam_ref as GR
    from multimm_b200 import gam

    x = eng.get_positions()
    planes, h = gam.slice_planes(x, center, gb.bins, slices, FRACTION, np.random.default_rng([0, slices]))
    eng.gam_configure(gb.bins, gb.n_bins, slices)
    eng.gam_add(planes, h)  # warm-up: module load
    eng.gam_configure(gb.bins, gb.n_bins, slices)
    for _ in range(reps):
        eng.gam_add(planes, h)
    r = eng.gam_read()
    ms = r["device_ms"] / reps
    split = pass_ms(eng, planes, h, reps)
    n, nb = int(eng.n), int(gb.n_bins)
    binned = int(np.count_nonzero(gb.bins >= 0))
    tests = n * slices
    popc = nb * (nb + 1) // 2 * ((slices + 31) // 32)
    one = r["counts"] // np.uint64(reps)
    diag = one[np.cumsum(np.r_[0, np.arange(nb, 1, -1)])]
    out = dict(system=system, n=n, binned_beads=binned, n_bins=nb, slices=slices, half_thickness_nm=h,
               adds=reps, device_ms_per_add=ms, detect_ms=split["k_gam_detect"], coseg_ms=split["k_gam_coseg"],
               slab_tests=tests, popc=popc, empty_share=r["empty"] / r["slices"],
               mean_detection=float(diag.mean()) / (slices - r["empty"] / reps),
               host_numpy_ms=None, device_equals_numpy=None)
    out["slab_tests_per_s"] = None if out["detect_ms"] is None else tests / (out["detect_ms"] * 1e-3)
    out["popc_per_s"] = None if out["coseg_ms"] is None else popc / (out["coseg_ms"] * 1e-3)
    if check:
        t0 = time.perf_counter()
        want, empty = GR.gam_add(x, gb.bins, nb, planes, h)
        out["host_numpy_ms"] = 1e3 * (time.perf_counter() - t0)
        out["device_equals_numpy"] = bool(np.array_equal(one, want) and r["empty"] == reps * empty)
        out["host_over_device"] = out["host_numpy_ms"] / ms
    log(out)
    return out


def md_wall(eng, bins, nb, chunks, log):
    from multimm_b200 import gam

    center = eng.get_positions().mean(axis=0)
    runs = []
    for order in ((False, True), (True, False)):
        for sampled in order:
            eng.md_configure("langevin", dt_ps=0.001, seed=5)
            eng.set_velocities_to_temperature(310.0, seed=6)
            eng.gam_configure(bins, nb, 1024)
            eng.md_run(100, want_report=True)  # warm-up
            t0 = time.perf_counter()
            for k in range(chunks):
                eng.md_run(100, want_report=False)
                if sampled:
                    planes, h = gam.slice_planes(eng.get_positions(), center, bins, 1024, FRACTION,
                                                 np.random.default_rng([0, k]))
                    eng.gam_add(planes, h)
            eng.get_positions()  # ends in a device synchronise
            wall = time.perf_counter() - t0
            r = eng.gam_read()
            runs.append(dict(sampled=sampled, steps=100 * chunks, wall_s=wall, adds=r["structures"],
                             device_ms=r["device_ms"]))
            log(runs[-1])
    off = [r["wall_s"] for r in runs if not r["sampled"]]
    on = [r["wall_s"] for r in runs if r["sampled"]]
    return dict(runs=runs, overhead=float(np.mean(on) / np.mean(off) - 1.0))


def _f(v, fmt):
    return "not measured" if v is None else format(v, fmt)


def report(result) -> str:
    c = result["card"]
    lines = ["# Simulated GAM (mmm_gam_add): timing on one GPU", "",
             f"Measured on one {c['name']} at a power limit of {c['power_limit']} (max SM clock {c['max_sm_clock']}), "
             "with `python scripts/gpu_gam_timing.py --out profiles/r11_gam.json`, which reads the card's name and "
             "power limit in the same run and writes this file beside `r11_gam.json`.", "",
             "## Device time of one add (N = 2·10⁵, genome-wide, two-stage minimised)", "",
             "Add: CUDA events of `mmm_gam_add` (plane upload, clears of the bitsets, both passes, read-back of the "
             "slice bitset), summed by `mmm_gam_read`, mean over the adds after a warm-up add. Detection and "
             "co-segregation: kernel durations of `k_gam_detect` and `k_gam_coseg` recorded by `torch.profiler` "
             "(CUDA activities) in a separate run of the same adds. Slab tests: N · S; POPC: B (B + 1) / 2 · ⌈S / 32⌉. "
             "Slices of `gam.slice_planes` with `GAM_SLICE_FRACTION` 0.025 about the container centre. The numpy "
             "restatement (`tests/gam_ref.py`) ran on the host at S = 1024 only.", "",
             "| bins | S | add | detection | slab tests/s | co-segregation | POPC/s | numpy on the host | equal | "
             "empty slices | mean detection |", "|---|---|---|---|---|---|---|---|---|---|---|"]
    for r in result["per_add"]:
        host = "not measured" if r["host_numpy_ms"] is None else f"{r['host_numpy_ms'] / 1e3:.1f} s"
        eq = "not measured" if r["device_equals_numpy"] is None else ("yes" if r["device_equals_numpy"] else "NO")
        lines.append(f"| {r['n_bins']} | {r['slices']} | {r['device_ms_per_add']:.3f} ms | {_f(r['detect_ms'], '.3f')} ms | "
                     f"{_f(r['slab_tests_per_s'], '.3g')} | {_f(r['coseg_ms'], '.3f')} ms | {_f(r['popc_per_s'], '.3g')} | "
                     f"{host} | {eq} | {r['empty_share']:.3g} | {r['mean_detection']:.3g} |")
    md = result["md_wall_20k"]
    lines += ["", "## MD wall time with and without an add every 100 steps (N = 2·10⁴)", "",
              "2000 MD steps in chunks of 100 (Langevin), with and without a GAM add after every chunk (1000 bins, "
              "S = 1024; the positions read back and the planes drawn on the host, as the driver does), "
              "alternating, twice each.", "",
              "| adds | wall time | device time of the adds |", "|---|---|---|"]
    for r in md["runs"]:
        lines.append(f"| {r['adds']} | {r['wall_s']:.3f} s | {r['device_ms']:.1f} ms |")
    lines += ["", f"Overhead of an add every 100 steps: {100 * md['overhead']:.2f} % of the MD wall time.", ""]
    return "\n".join(lines)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    opt = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing measured")
    import bench
    from common import make_case, to_engine
    from multimm_b200 import contacts, gam

    def log(msg):
        print(msg, flush=True)

    result = dict(card=card(), per_add=[])
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        m = bench.build_model("gw", 0, 0, tmp)
        try:
            m.args.MIN_COARSE_CUTOFF = 0.5
            m.min_energy(write_files=False)
            n = m.engine.n
            gb = contacts.genome_bins(m.layout, 0, n_beads=n)
            fine = contacts.genome_bins(m.layout, int(gb.resolution_bp * gb.n_bins / 4096), n_beads=n,
                                        max_bins=gam.MAX_BINS)
            for b in (gb, fine):
                for s in (1024, 16384):
                    result["per_add"].append(per_add(m.engine, "N=2e5 genome-wide, two-stage minimised",
                                                     m.mass_center, b, s, opt.reps, log, check=s == 1024))
        finally:
            m.close()
    eng = to_engine(make_case(20_000, n_chrom=2, seed=1))
    eng.minimize(tol=10.0, max_iter=300)
    bins = (np.arange(20_000) * 1000 // 20_000).astype(np.int32)
    result["md_wall_20k"] = md_wall(eng, bins, 1000, 20, log)
    log(f"MD overhead of a GAM add every 100 steps: {result['md_wall_20k']['overhead']:.2%}")
    eng.close()
    write(opt.out, result, log)
    md_path = os.path.splitext(opt.out)[0] + ".md"
    with open(md_path, "w") as fh:
        fh.write(report(result))
    log(f"wrote {md_path}")


if __name__ == "__main__":
    main()
