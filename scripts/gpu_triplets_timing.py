"""Timing of the three-way contact map (mmm_triplets_add) on one GPU, beside its numpy restatement on the host.

    python scripts/gpu_triplets_timing.py --out profiles/r08_triplets.json

writes the JSON and, beside it, the same numbers as a Markdown report (.md).

1. Device time of one add (CUDA events of mmm_triplets_add, summed by mmm_triplets_read over `reps` adds after a
   warm-up add) at N = 2e5: the genome-wide system built as bench.py builds it, after the two-stage minimisation
   (MIN_COARSE_CUTOFF = 0.5 nm), at rc = 0.2 and 0.5 nm, with the canonical bins of contacts.genome_bins at the
   automatic resolution (about 1000 bins) and at 5 kb.  Per case: triples, entries, chunks per add, the
   device memory the accumulator holds (cudaMemGetInfo before the first configure and after the case: sort
   buffers, adjacency, per-bead arrays and the accumulated list), and, at rc = 0.2 nm, the numpy restatement
   (tests/triplets_ref.py) timed on the host and compared bit for bit.  At rc = 0.5 nm the restatement is not
   run: its wedge arrays do not fit a test machine's memory in reasonable time.
2. At N = 2e4 (tests/common.make_case, minimised for 300 L-BFGS iterations, about 1000 contiguous bins), MD wall
   time of 2000 steps in chunks of 100 with and without an add after every chunk, alternating, twice each.
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


def per_add(eng, rc, gb, label, reps, free0, tri, log):
    import torch

    import triplets_ref as TR

    eng.triplets_configure(rc, gb.bins, gb.n_bins)
    eng.triplets_add()  # warm-up: buffers, module load
    eng.triplets_configure(rc, gb.bins, gb.n_bins)
    t0 = time.perf_counter()
    for _ in range(reps):
        eng.triplets_add()
    wall = time.perf_counter() - t0
    got = eng.triplets_read()
    held = free0 - torch.cuda.mem_get_info()[0]
    ms = got["device_ms"] / reps
    out = dict(system="N=2e5 genome-wide, two-stage minimised", n=eng.n, rc_nm=rc, bins=label, n_bins=gb.n_bins,
               resolution_bp=gb.resolution_bp, adds=reps, device_ms_per_add=ms, wall_ms_per_add=1e3 * wall / reps,
               triples=got["triples"] // reps, entries=len(got["vals"]), chunks_per_add=got["chunks"] / reps,
               accumulator_device_bytes=int(held), host_numpy_ms=None, device_equals_numpy=None)
    if tri is not None:
        t0 = time.perf_counter()
        p, q, r, vals = TR.binned(*tri["t"], gb.bins, gb.n_bins)
        host = tri["s"] + time.perf_counter() - t0
        out.update(host_numpy_ms=1e3 * host, host_over_device=1e3 * host / ms,
                   device_equals_numpy=bool(got["triples"] == reps * len(tri["t"][0]) and
                                            all(np.array_equal(got[k], w) for k, w in zip("pqr", (p, q, r))) and
                                            np.array_equal(got["vals"], np.uint64(reps) * vals)))
    log(out)
    return out


def md_wall(eng, bins, nb, chunks, log):
    runs = []
    for order in ((False, True), (True, False)):
        for sampled in order:
            eng.md_configure("langevin", dt_ps=0.001, seed=5)
            eng.set_velocities_to_temperature(310.0, seed=6)
            eng.triplets_configure(0.2, bins, nb)
            eng.md_run(100, want_report=True)  # warm-up
            t0 = time.perf_counter()
            for _ in range(chunks):
                eng.md_run(100, want_report=False)
                if sampled:
                    eng.triplets_add()
            eng.get_positions()  # ends in a device synchronise
            wall = time.perf_counter() - t0
            r = eng.triplets_read()
            runs.append(dict(sampled=sampled, steps=100 * chunks, wall_s=wall, adds=r["samples"],
                             device_ms=r["device_ms"], triples_per_add=r["triples"] / max(r["samples"], 1)))
            log(runs[-1])
    off = [r["wall_s"] for r in runs if not r["sampled"]]
    on = [r["wall_s"] for r in runs if r["sampled"]]
    return dict(runs=runs, overhead=float(np.mean(on) / np.mean(off) - 1.0))


def report(result) -> str:
    c = result["card"]
    lines = ["# Three-way contact map (mmm_triplets_add): timing on one GPU", "",
             f"Measured on one {c['name']} at a power limit of {c['power_limit']} (max SM clock {c['max_sm_clock']}), "
             "with `python scripts/gpu_triplets_timing.py --out profiles/r08_triplets.json`, which reads the card's "
             "name and power limit in the same run and writes this file beside `r08_triplets.json`.", "",
             "## Device time of one add at N = 2·10⁵", "",
             "The system is the genome-wide one `bench.py` builds, after the two-stage minimisation "
             "(MIN_COARSE_CUTOFF = 0.5 nm). Device time: CUDA events of `mmm_triplets_add`, summed by "
             "`mmm_triplets_read`, mean over the adds after a warm-up add (the host waits between the chunks are "
             "inside it). Memory: device memory the accumulator holds after the case (cudaMemGetInfo), cumulative "
             "over the cases in table order, since buffers only grow. The numpy restatement (`tests/triplets_ref.py`: "
             "pairs, triangles and binning) ran on the host at rc = 0.2 nm only; at rc = 0.5 nm it was not measured.",
             "", "| rc | bins | triples per add | entries | chunks per add | device time | device memory | numpy on the "
             "host | equal |", "|---|---|---|---|---|---|---|---|---|"]
    for r in result["per_add_200k"]:
        host = "not measured" if r["host_numpy_ms"] is None else f"{r['host_numpy_ms'] / 1e3:.2f} s"
        eq = "not measured" if r["device_equals_numpy"] is None else ("yes" if r["device_equals_numpy"] else "NO")
        lines.append(f"| {r['rc_nm']} nm | {r['n_bins']} ({r['resolution_bp']} bp) | {r['triples']:.3g} | "
                     f"{r['entries']:.3g} | {r['chunks_per_add']:g} | {r['device_ms_per_add']:.2f} ms | "
                     f"{r['accumulator_device_bytes'] / 2**20:.0f} MiB | {host} | {eq} |")
    md = result["md_wall_20k"]
    lines += ["", "## MD wall time with and without an add every 100 steps (N = 2·10⁴)", "",
              "2000 MD steps in chunks of 100 (Langevin), with and without `mmm_triplets_add` after every chunk "
              "(rc = 0.2 nm, about 1000 bins), alternating, twice each.", "",
              "| adds | triples per add | wall time | device time of the adds |", "|---|---|---|---|"]
    for r in md["runs"]:
        lines.append(f"| {r['adds']} | {r['triples_per_add']:.3g} | {r['wall_s']:.3f} s | {r['device_ms']:.1f} ms |")
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
    import contacts_ref as CR
    import triplets_ref as TR
    from common import make_case, to_engine
    from multimm_b200 import contacts, triplets

    def log(msg):
        print(msg, flush=True)

    result = dict(card=card())
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        m = bench.build_model("gw", 0, 0, tmp)
        try:
            m.args.MIN_COARSE_CUTOFF = 0.5
            m.min_energy(write_files=False)
            n = m.engine.n
            tables = [("auto", contacts.genome_bins(m.layout, 0, n_beads=n)),
                      ("5 kb", contacts.genome_bins(m.layout, 5_000, n_beads=n, max_bins=triplets.MAX_BINS))]
            torch.cuda.init()
            free0 = torch.cuda.mem_get_info()[0]
            result["per_add_200k"] = []
            for rc in (0.2, 0.5):
                tri = None
                if rc == 0.2:
                    x = m.engine.get_positions()
                    t0 = time.perf_counter()
                    t = TR.triangles_from_pairs(n, *CR.contact_pairs(x, rc))
                    tri = dict(t=t, s=time.perf_counter() - t0)
                for label, gb in tables:
                    result["per_add_200k"].append(per_add(m.engine, rc, gb, label, opt.reps if rc == 0.2 else 2,
                                                          free0, tri, log))
        finally:
            m.close()
        eng = to_engine(make_case(20_000, n_chrom=2, seed=1))
        eng.minimize(tol=10.0, max_iter=300)
        bins = (np.arange(20_000) * 1000 // 20_000).astype(np.int32)
        result["md_wall_20k"] = md_wall(eng, bins, 1000, 20, log)
        log(f"MD overhead of a three-way add every 100 steps: {result['md_wall_20k']['overhead']:.2%}")
        eng.close()
    write(opt.out, result, log)
    md_path = os.path.splitext(opt.out)[0] + ".md"
    with open(md_path, "w") as fh:
        fh.write(report(result))
    log(f"wrote {md_path}")


if __name__ == "__main__":
    main()
