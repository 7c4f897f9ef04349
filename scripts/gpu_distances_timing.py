"""Timing of the distance-map pass (mmm_distance_map) and of SAVE_DISTANCES in the ensemble driver, on one GPU.

    python scripts/gpu_distances_timing.py --out profiles/r05_distances.json [--members 8] [--rounds 2]

1. Distance pass, ms per structure (CUDA events around the clearing of the maps and the kernel, median
   over repeated calls; the host wall time of the whole call, bin check, guard and copies included, beside
   it), with the bead pairs per second it reaches:
   * N = 2e5 genome-wide system built as bench.py builds it, after the two-stage minimisation
     (MIN_COARSE_CUTOFF = 0.5 nm, as bench.py's ensemble metric), at the automatic bins (about 1000) and
     at 4096 bins — with its two-stage time;
   * N = 5000 (the region preset's size) at 4096 bins, the finest the dense map allows (about 1.2 beads per
     bin; one bead per bin would need 5000), on the Hilbert start (the pass has no culling, so its cost
     depends on N and the bins, not on the structure);
   * N = 2e6 on the Hilbert start, 1000 bins.
2. Ensembles of `members` genome-wide members on this GPU with SAVE_DISTANCES on and off, alternating,
   `rounds` times each: structures / hour, and distances.aggregate over the members of the last one.
The card's name and power limit are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from gpu_contacts_timing import card, write  # noqa: E402


def time_pass(eng, bins, n_bins, reps, label):
    eng.distance_map(bins, n_bins)  # warm-up (scratch allocation, module load)
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        eng.distance_map(bins, n_bins)
        wall.append(1e3 * (time.perf_counter() - t0))
        dev.append(eng.distance_stats()["device_ms"])
    n = eng.n
    pairs = n * (n - 1) / 2
    med = float(np.median(dev))
    return dict(system=label, n=n, n_bins=int(n_bins), device_ms_median=med, device_ms_min=float(np.min(dev)),
                device_ms_max=float(np.max(dev)), call_wall_ms_median=float(np.median(wall)), repeats=reps,
                bead_pairs=pairs, bead_pairs_per_s=pairs / (med * 1e-3))


def passes(tmp, reps, log):
    import bench
    from multimm_b200 import contacts
    from multimm_b200.engine import Engine

    out = {}
    m = bench.build_model("gw", 0, 0, tmp)
    try:
        m.args.MIN_COARSE_CUTOFF = 0.5
        t0 = time.perf_counter()
        m.min_energy(write_files=False)
        out["two_stage_minimisation_s"] = time.perf_counter() - t0
        n = m.args.N_BEADS
        gb = contacts.genome_bins(m.layout, 0, n_beads=n)
        gb4 = contacts.genome_bins(m.layout, contacts.auto_resolution(contacts.spans(range(22))) // 4 + 1, n_beads=n)
        out["gw_200k"] = [time_pass(m.engine, gb.bins, gb.n_bins, reps, "N=2e5 minimised, auto bins"),
                          time_pass(m.engine, (np.arange(n) * 4096 // n).astype(np.int32), 4096, reps,
                                    "N=2e5 minimised, 4096 equal bead blocks")]
        out["gw_200k_genomic_4x"] = time_pass(m.engine, gb4.bins, gb4.n_bins, reps, "N=2e5 minimised, genomic bins at 1/4 of the auto resolution")
        for r in out["gw_200k"] + [out["gw_200k_genomic_4x"]]:
            log(r)
        out["pass_share_of_minimisation"] = out["gw_200k"][0]["call_wall_ms_median"] / (1e3 * out["two_stage_minimisation_s"])
        log(f"two-stage minimisation {out['two_stage_minimisation_s']:.2f} s; pass share {out['pass_share_of_minimisation']:.4%}")
    finally:
        m.close()
    with Engine(5000) as eng:
        eng.hilbert_init(8, 0.1)
        out["region_5000"] = time_pass(eng, (np.arange(5000) * 4096 // 5000).astype(np.int32), 4096, reps,
                                       "N=5000 Hilbert start, 4096 bins")
        log(out["region_5000"])
    n = 2_000_000
    with Engine(n) as eng:
        eng.hilbert_init(8, 0.1)
        out["hilbert_2m"] = time_pass(eng, (np.arange(n) * 1000 // n).astype(np.int32), 1000, 3,
                                      "N=2e6 Hilbert start, 1000 bins")
        log(out["hilbert_2m"])
    return out


def ensemble(tmp, members, save, tag):
    import bench
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    kw = bench.config_kwargs("gw", 0, tmp)
    out = os.path.join(tmp, f"ens_{tag}")
    kw.update(PLATFORM="B200", GENERATE_ENSEMBLE=True, N_ENSEMBLE=members, MIN_COARSE_CUTOFF=0.5, OUT_PATH=out,
              SAVE_DISTANCES=save)
    args = SimulationConfig(**kw)
    t0 = time.perf_counter()
    reps = run.run_ensemble(args, devices=[0])
    wall = time.perf_counter() - t0
    return out, dict(save_distances=save, members=len(reps), wall_s=wall,
                     structures_per_hour=3600.0 * len(reps) / wall, distances_s=[r.get("distances_s") for r in reps])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--members", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    opt = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing measured")
    from multimm_b200 import distances

    def log(msg):
        print(msg, flush=True)

    result = dict(card=card())
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        result["passes"] = passes(tmp, opt.reps, log)
        runs, last_on = [], None
        for r in range(opt.rounds):
            for save in ((False, True) if r % 2 == 0 else (True, False)):
                out, res = ensemble(tmp, opt.members, save, f"{r}_{int(save)}")
                log(f"ensemble round {r} SAVE_DISTANCES={save}: {res['structures_per_hour']:.1f} structures/hour "
                    f"(distances_s {res['distances_s']})")
                runs.append(res)
                if save:
                    last_on = out
        result["ensemble"] = runs
        for save in (False, True):
            result[f"ensemble_{'on' if save else 'off'}_structures_per_hour"] = [
                r["structures_per_hour"] for r in runs if r["save_distances"] == save]
        paths = sorted(os.path.join(last_on, "distances", f) for f in os.listdir(os.path.join(last_on, "distances")))
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            agg = distances.aggregate(paths)
            times.append(time.perf_counter() - t0)
        mean = distances.mean_distance(agg)
        rmean, _ = distances.radial_profile(agg)
        result["aggregate"] = dict(members=len(paths), n_bins=int(len(agg["bin_beads"])), wall_s=times,
                                   mean_distance_nm_range=[float(np.nanmin(mean)), float(np.nanmax(mean))],
                                   radial_mean_nm_range=[float(np.nanmin(rmean)), float(np.nanmax(rmean))])
        log(f"aggregate: {result['aggregate']}")
    write(opt.out, result, log)


if __name__ == "__main__":
    main()
