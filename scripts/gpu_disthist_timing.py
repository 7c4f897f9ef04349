"""Timing of the distance histograms (mmm_disthist_add) on one GPU, beside the distance pass and the numpy
restatement.

    python scripts/gpu_disthist_timing.py --out profiles/r10_disthist.json

writes the JSON and, beside it, the same numbers as a Markdown report (.md).

1. Device time of one add (CUDA events of mmm_disthist_add, summed by mmm_disthist_read over `reps` adds after a
   warm-up add) at N = 2e4 (tests/common.make_case, minimised for 300 L-BFGS iterations) and at N = 2e5 (the
   genome-wide system bench.py builds, after the two-stage minimisation, MIN_COARSE_CUTOFF = 0.5 nm), at the
   canonical bins of contacts.genome_bins where the layout is known (about 1000 bins) or 1000 contiguous bins,
   with the 19 default edges and with 63 edges.  Beside it, the device time of the distance pass
   (mmm_distance_map) at the same bins, and pairs per second of both.  At N = 2e4 the counts are compared with the
   numpy restatement (tests/disthist_ref.py), timed on the host.  At N = 2e5 with the default edges: the share of
   pairs in each cell, so the open last cell's share, and the median of all pair distances.
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
from multimm_b200.disthist import DEFAULT_EDGES as DEFAULT  # noqa: E402

EDGES_63 = np.geomspace(0.05, 60.0, 63)


def per_add(eng, system, bins, nb, edges, label, reps, log, check=False):
    import disthist_ref as HR

    eng.disthist_configure(bins, nb, edges)
    eng.disthist_add()  # warm-up: module load, attribute
    eng.disthist_configure(bins, nb, edges)
    for _ in range(reps):
        eng.disthist_add()
    got = eng.disthist_read()
    one = got["counts"] // np.uint64(reps)
    ms = got["device_ms"] / reps
    eng.distance_map(bins, nb)  # warm-up
    dist = []
    for _ in range(reps):
        eng.distance_map(bins, nb)
        dist.append(eng._distance_ms)
    dist_ms = float(np.mean(dist))
    n, nb = int(eng.n), int(nb)
    binned = int(np.count_nonzero(np.asarray(bins) >= 0))
    pairs = binned * (binned - 1) // 2
    out = dict(system=system, n=n, n_bins=nb, edges=label, n_edges=len(edges), adds=reps, device_ms_per_add=ms,
               pairs=pairs, pairs_per_s=float(pairs / (ms * 1e-3)), distance_pass_ms=dist_ms,
               distance_pass_pairs_per_s=float(pairs / (dist_ms * 1e-3)), counts_total=int(one.sum()),
               host_numpy_ms=None, device_equals_numpy=None)
    assert out["counts_total"] == pairs
    cells = one.sum(axis=0, dtype=np.uint64).astype(np.float64)
    out["cell_share"] = (cells / cells.sum()).tolist()
    out["open_last_cell_share"] = float(cells[-1] / cells.sum())
    cum = np.cumsum(cells) / cells.sum()
    h = int(np.searchsorted(cum, 0.5))
    lo = 0.0 if h == 0 else float(edges[h - 1])
    hi = float(edges[h]) if h < len(edges) else float("nan")
    below = 0.0 if h == 0 else cum[h - 1]
    out["median_all_pairs_nm"] = float(lo + (0.5 - below) / (cells[h] / cells.sum()) * (hi - lo))
    if check:
        x = eng.get_positions()
        t0 = time.perf_counter()
        want = HR.hist_counts(x, bins, nb, edges)
        out.update(host_numpy_ms=1e3 * (time.perf_counter() - t0), device_equals_numpy=bool(np.array_equal(one, want)))
        out["host_over_device"] = out["host_numpy_ms"] / ms
    log(out)
    return out


def md_wall(eng, bins, nb, chunks, log):
    runs = []
    for order in ((False, True), (True, False)):
        for sampled in order:
            eng.md_configure("langevin", dt_ps=0.001, seed=5)
            eng.set_velocities_to_temperature(310.0, seed=6)
            eng.disthist_configure(bins, nb, np.asarray([float(v) for v in DEFAULT.split(",")]))
            eng.md_run(100, want_report=True)  # warm-up
            t0 = time.perf_counter()
            for _ in range(chunks):
                eng.md_run(100, want_report=False)
                if sampled:
                    eng.disthist_add()
            eng.get_positions()  # ends in a device synchronise
            wall = time.perf_counter() - t0
            r = eng.disthist_read()
            runs.append(dict(sampled=sampled, steps=100 * chunks, wall_s=wall, adds=r["samples"],
                             device_ms=r["device_ms"]))
            log(runs[-1])
    off = [r["wall_s"] for r in runs if not r["sampled"]]
    on = [r["wall_s"] for r in runs if r["sampled"]]
    return dict(runs=runs, overhead=float(np.mean(on) / np.mean(off) - 1.0))


def report(result) -> str:
    c = result["card"]
    lines = ["# Distance histograms (mmm_disthist_add): timing on one GPU", "",
             f"Measured on one {c['name']} at a power limit of {c['power_limit']} (max SM clock {c['max_sm_clock']}), "
             "with `python scripts/gpu_disthist_timing.py --out profiles/r10_disthist.json`, which reads the card's "
             "name and power limit in the same run and writes this file beside `r10_disthist.json`.", "",
             "## Device time of one add", "",
             "Device time: CUDA events of `mmm_disthist_add`, summed by `mmm_disthist_read`, mean over the adds after "
             "a warm-up add. The distance pass (`mmm_distance_map`, mean sums over the same pairs) ran in the same "
             "process at the same bins. Default edges: 0.1 … 100 nm (19 edges, 20 cells); 63 edges: geometric from "
             "0.05 to 60 nm. The numpy restatement (`tests/disthist_ref.py`) ran on the host at N = 2·10⁴ only; at "
             "N = 2·10⁵ it was not measured.", "",
             "| system | bins | edges | device time | pairs/s | distance pass | its pairs/s | numpy on the host | "
             "equal |", "|---|---|---|---|---|---|---|---|---|"]
    for r in result["per_add"]:
        host = "not measured" if r["host_numpy_ms"] is None else f"{r['host_numpy_ms'] / 1e3:.1f} s"
        eq = "not measured" if r["device_equals_numpy"] is None else ("yes" if r["device_equals_numpy"] else "NO")
        lines.append(f"| {r['system']} | {r['n_bins']} | {r['n_edges']} | {r['device_ms_per_add']:.2f} ms | "
                     f"{r['pairs_per_s']:.3g} | {r['distance_pass_ms']:.2f} ms | {r['distance_pass_pairs_per_s']:.3g} | "
                     f"{host} | {eq} |")
    d = next(r for r in result["per_add"] if r["n"] >= 100_000 and r["n_edges"] == 19)
    lines += ["", "## Distance scale of the genome-wide minimised structure (N = 2·10⁵, default edges)", "",
              f"Median of all pair distances (interpolated in its cell): {d['median_all_pairs_nm']:.2f} nm. "
              f"Share of pairs in the open last cell [100 nm, ∞): {d['open_last_cell_share']:.3g}.", "",
              "| cell | share of pairs |", "|---|---|"]
    e = [0.0] + [float(v) for v in DEFAULT.split(",")] + [float("inf")]
    for k, s in enumerate(d["cell_share"]):
        lines.append(f"| [{e[k]:g}, {e[k + 1]:g}) nm | {s:.3g} |")
    md = result["md_wall_20k"]
    lines += ["", "## MD wall time with and without an add every 100 steps (N = 2·10⁴)", "",
              "2000 MD steps in chunks of 100 (Langevin), with and without `mmm_disthist_add` after every chunk "
              "(1000 bins, default edges), alternating, twice each.", "",
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
    from multimm_b200 import contacts

    def log(msg):
        print(msg, flush=True)

    default = np.asarray([float(v) for v in DEFAULT.split(",")])
    result = dict(card=card(), per_add=[])
    log(f"card: {result['card']}")
    eng = to_engine(make_case(20_000, n_chrom=2, seed=1))
    eng.minimize(tol=10.0, max_iter=300)
    bins = (np.arange(20_000) * 1000 // 20_000).astype(np.int32)
    for label, edges in (("default", default), ("63", EDGES_63)):
        result["per_add"].append(per_add(eng, "N=2e4 minimised", bins, 1000, edges, label, opt.reps, log, check=True))
    result["md_wall_20k"] = md_wall(eng, bins, 1000, 20, log)
    log(f"MD overhead of a distance-histogram add every 100 steps: {result['md_wall_20k']['overhead']:.2%}")
    eng.close()
    with tempfile.TemporaryDirectory() as tmp:
        m = bench.build_model("gw", 0, 0, tmp)
        try:
            m.args.MIN_COARSE_CUTOFF = 0.5
            m.min_energy(write_files=False)
            gb = contacts.genome_bins(m.layout, 0, n_beads=m.engine.n)
            for label, edges in (("default", default), ("63", EDGES_63)):
                result["per_add"].append(per_add(m.engine, "N=2e5 genome-wide, two-stage minimised", gb.bins,
                                                 gb.n_bins, edges, label, opt.reps, log))
        finally:
            m.close()
    write(opt.out, result, log)
    md_path = os.path.splitext(opt.out)[0] + ".md"
    with open(md_path, "w") as fh:
        fh.write(report(result))
    log(f"wrote {md_path}")


if __name__ == "__main__":
    main()
