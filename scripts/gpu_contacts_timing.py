"""Timing of the contact pass (mmm_contacts) and of SAVE_CONTACTS in the ensemble driver, on one GPU.

    python scripts/gpu_contacts_timing.py --out profiles/r03_contacts.json [--members 8] [--rounds 2]

1. Contact pass, ms per structure (CUDA events around its kernels, median over repeated calls; the host
   wall time of the whole call, copies and bin check included, beside it), candidates tested in FP64,
   contacts found, hit rate, at rc = 0.2 and 0.5 nm:
   * N = 2e5 genome-wide system built as bench.py builds it, at the Hilbert start and after the two-stage
     minimisation (MIN_COARSE_CUTOFF = 0.5 nm, as bench.py's ensemble metric) — with its two-stage time;
   * N = 2e6 on the Hilbert start (22 chromosome blocks of equal length, 1000 bins).
2. mmm_contact_map (the structure report's block-mean proxy) at N = 2e5, 1000 bins, for scale.
3. Ensembles of `members` genome-wide members on this GPU with SAVE_CONTACTS on and off, alternating,
   `rounds` times each: structures / hour.
The card's name and power limit are read in the same run and stored with the numbers.

    python scripts/gpu_contacts_timing.py --fine --out profiles/r04_contacts_fine.json

measures the sparse map (mmm_contacts_sparse) instead: device and call ms, contacts, entries and scratch
bytes at N = 2e5 minimised (bead resolution and 50 kb) and N = 2e6 on the Hilbert start; ensembles with
CONTACT_FINE_RESOLUTION = 5 kb and 0 (SAVE_CONTACTS on in both), alternating; contacts.aggregate_fine
over the members of the last ensemble with the fine map.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    name, power, clock = [t.strip() for t in out.split(",")] if out.count(",") == 2 else (out, "", "")
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def time_pass(eng, rc, bins, n_bins, reps):
    eng.contacts(rc, bins, n_bins)  # warm-up (scratch allocation, module load)
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        _, _, pairs = eng.contacts(rc, bins, n_bins)
        wall.append(1e3 * (time.perf_counter() - t0))
        dev.append(eng.contacts_stats()["device_ms"])
    cand = eng.contacts_stats()["candidates"]
    return dict(rc_nm=rc, n_bins=int(n_bins), device_ms_median=float(np.median(dev)), device_ms_min=float(np.min(dev)),
                device_ms_max=float(np.max(dev)), call_wall_ms_median=float(np.median(wall)), repeats=reps,
                candidates=int(cand), contacts=int(pairs), hit_rate=float(pairs / max(cand, 1)),
                contacts_per_bead=float(pairs / eng.n))


def gw_passes(tmp, reps, log):
    import bench
    from multimm_b200 import contacts

    m = bench.build_model("gw", 0, 0, tmp)
    out = {}
    try:
        gb = contacts.genome_bins(m.layout, 0, n_beads=m.args.N_BEADS)
        out["hilbert_start"] = [time_pass(m.engine, rc, gb.bins, gb.n_bins, reps) for rc in (0.2, 0.5)]
        log(f"N=2e5 Hilbert start: {out['hilbert_start']}")
        m.args.MIN_COARSE_CUTOFF = 0.5
        t0 = time.perf_counter()
        m.min_energy(write_files=False)
        out["two_stage_minimisation_s"] = time.perf_counter() - t0
        out["minimisation_report"] = {k: (float(v) if isinstance(v, (float, np.floating)) else int(v))
                                      for k, v in m.report.items()}
        out["minimised"] = [time_pass(m.engine, rc, gb.bins, gb.n_bins, reps) for rc in (0.2, 0.5)]
        log(f"N=2e5 minimised ({out['two_stage_minimisation_s']:.2f} s two-stage): {out['minimised']}")
        out["pass_share_of_minimisation"] = out["minimised"][0]["call_wall_ms_median"] / (1e3 * out["two_stage_minimisation_s"])
        x = m.engine.get_positions()
    finally:
        m.close()
    return out, x


def big_pass(reps, log):
    from multimm_b200.engine import Engine

    n = 2_000_000
    with Engine(n) as eng:
        eng.hilbert_init(8, 0.1)
        eng.set_bead_params(chrom=(np.arange(n) * 22 // n).astype(np.int32))
        bins = (np.arange(n) * 1000 // n).astype(np.int32)
        res = [time_pass(eng, rc, bins, 1000, reps) for rc in (0.2, 0.5)]
    log(f"N=2e6 Hilbert start: {res}")
    return res


def contact_map_proxy(x, log):
    import ctypes as C

    from multimm_b200 import _lib

    lib = _lib.load()
    xs = np.ascontiguousarray(x)
    m = np.empty((1000, 1000))
    mean = C.c_double()
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        rc = lib.mmm_contact_map(0, xs.ctypes.data_as(C.c_void_p), len(xs), 1000, 1, m.ctypes.data_as(C.c_void_p),
                                 C.byref(mean))
        times.append(1e3 * (time.perf_counter() - t0))
        assert rc == 0
    res = dict(n=len(xs), bins=1000, wall_ms=times, note="host wall clock of the whole call (allocation, copies, kernel)")
    log(f"mmm_contact_map N=2e5, 1000 bins: {times} ms")
    return res


def ensemble(tmp, members, save, tag):
    import bench
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    kw = bench.config_kwargs("gw", 0, tmp)
    out = os.path.join(tmp, f"ens_{tag}")
    kw.update(PLATFORM="B200", GENERATE_ENSEMBLE=True, N_ENSEMBLE=members, MIN_COARSE_CUTOFF=0.5, OUT_PATH=out,
              SAVE_CONTACTS=save)
    args = SimulationConfig(**kw)
    t0 = time.perf_counter()
    reps = run.run_ensemble(args, devices=[0])
    wall = time.perf_counter() - t0
    res = dict(save_contacts=save, members=len(reps), wall_s=wall, structures_per_hour=3600.0 * len(reps) / wall,
               contacts_s=[r.get("contacts_s") for r in reps])
    if save:
        from multimm_b200 import contacts

        d = contacts.load(os.path.join(out, "ensemble_contacts.npz"))
        p = contacts.contact_probability(d)
        res.update(ensemble_members=int(d["members"]), ensemble_pairs=int(d["pairs"]),
                   symmetric=bool(np.array_equal(d["counts"], d["counts"].T)),
                   p_of_s={str(s): float(p[s]) for s in (1, 2, 5, 10, 100, 1000, 10000)})
    return res


def sparse_scratch_bytes(keys: int, n: int) -> int:
    """Device scratch of mmm_contacts_sparse for `keys` binned contacts (mmm_contacts.cu): two sort buffers,
    the digit x chunk table with its scan parts, the per-tile offsets."""
    blocks = max(1, -(-keys // 4096))
    tiles = -(-n // 32)
    return 16 * keys + 8 * (256 * blocks * 17 // 16 + 2) + 8 * (tiles + max(1, -(-tiles // 4096)) + 1)


def time_sparse(eng, rc, bins, n_bins, reps, label):
    eng.contacts_sparse(rc, bins, n_bins)  # warm-up (scratch allocation, module load)
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        rows, _, _, pairs = eng.contacts_sparse(rc, bins, n_bins)
        wall.append(1e3 * (time.perf_counter() - t0))
        dev.append(eng.contacts_stats()["device_ms"])
    keys = pairs if int(np.min(bins)) >= 0 else None  # every contact is binned when no bead is left out
    return dict(system=label, rc_nm=rc, n_bins=int(n_bins), device_ms_median=float(np.median(dev)),
                device_ms_min=float(np.min(dev)), device_ms_max=float(np.max(dev)),
                call_wall_ms_median=float(np.median(wall)), repeats=reps, contacts=int(pairs), entries=int(len(rows)),
                candidates=int(eng.contacts_stats()["candidates"]),
                scratch_bytes=sparse_scratch_bytes(keys, eng.n) if keys is not None else None)


def fine_passes(tmp, reps, log):
    import bench
    from multimm_b200 import contacts
    from multimm_b200.engine import Engine

    res = []
    m = bench.build_model("gw", 0, 0, tmp)
    try:
        m.args.MIN_COARSE_CUTOFF = 0.5
        m.min_energy(write_files=False)
        n = m.args.N_BEADS
        bead = np.arange(n, dtype=np.int32)
        gb = contacts.genome_bins(m.layout, 50_000, n_beads=n, max_bins=contacts.MAX_FINE_BINS)
        for rc in (0.2, 0.5):
            res.append(time_sparse(m.engine, rc, bead, n, reps, "N=2e5 minimised, bead bins"))
            log(res[-1])
            res.append(time_sparse(m.engine, rc, gb.bins, gb.n_bins, reps, "N=2e5 minimised, 50 kb"))
            log(res[-1])
    finally:
        m.close()
    n = 2_000_000
    with Engine(n) as eng:
        eng.hilbert_init(8, 0.1)
        bins = (np.arange(n) * 1000 // n).astype(np.int32)
        for rc in (0.2, 0.5):
            res.append(time_sparse(eng, rc, bins, 1000, max(3, reps // 4), "N=2e6 Hilbert start, 1000 bins"))
            log(res[-1])
        res.append(time_sparse(eng, 0.2, np.arange(n, dtype=np.int32), n, max(3, reps // 4),
                               "N=2e6 Hilbert start, bead bins"))
        log(res[-1])
    return res


def fine_ensemble(tmp, members, fine_bp, tag):
    import bench
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    kw = bench.config_kwargs("gw", 0, tmp)
    out = os.path.join(tmp, f"ens_{tag}")
    kw.update(PLATFORM="B200", GENERATE_ENSEMBLE=True, N_ENSEMBLE=members, MIN_COARSE_CUTOFF=0.5, OUT_PATH=out,
              SAVE_CONTACTS=True, CONTACT_FINE_RESOLUTION=fine_bp)
    args = SimulationConfig(**kw)
    t0 = time.perf_counter()
    reps = run.run_ensemble(args, devices=[0])
    wall = time.perf_counter() - t0
    return out, dict(fine_resolution_bp=fine_bp, members=len(reps), wall_s=wall,
                     structures_per_hour=3600.0 * len(reps) / wall,
                     contacts_fine_s=[r.get("contacts_fine_s") for r in reps])


def main_fine(opt, log):
    from multimm_b200 import contacts

    result = dict(card=card())
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        result["passes"] = fine_passes(tmp, opt.reps, log)
        runs, last_fine = [], None
        for r in range(opt.rounds):
            for fine in ((0, 5000) if r % 2 == 0 else (5000, 0)):
                out, res = fine_ensemble(tmp, opt.members, fine, f"{r}_{fine}")
                log(f"ensemble round {r} CONTACT_FINE_RESOLUTION={fine}: {res['structures_per_hour']:.1f} structures/hour")
                runs.append(res)
                if fine:
                    last_fine = out
        result["ensemble"] = runs
        for fine in (0, 5000):
            result[f"ensemble_fine_{fine}_structures_per_hour"] = [
                r["structures_per_hour"] for r in runs if r["fine_resolution_bp"] == fine]
        paths = sorted(os.path.join(last_fine, "contacts", f) for f in os.listdir(os.path.join(last_fine, "contacts"))
                       if f.endswith("_fine.npz"))
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            agg = contacts.aggregate_fine(paths)
            times.append(time.perf_counter() - t0)
        result["aggregate_fine"] = dict(members=len(paths), n_bins=int(agg["n_bins"]), entries=int(len(agg["vals"])),
                                        member_entries=[int(len(contacts.load_fine(p)["vals"])) for p in paths],
                                        wall_s=times)
        log(f"aggregate_fine: {result['aggregate_fine']}")
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--members", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--fine", action="store_true", help="measure the sparse map (mmm_contacts_sparse) instead")
    opt = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing measured")
    lines = []

    def log(msg):
        print(msg, flush=True)
        lines.append(msg)

    if opt.fine:
        write(opt.out, main_fine(opt, log), log)
        return
    result = dict(card=card())
    log(f"card: {result['card']}")
    with tempfile.TemporaryDirectory() as tmp:
        result["gw_200k"], x = gw_passes(tmp, opt.reps, log)
        result["hilbert_2m"] = big_pass(max(3, opt.reps // 4), log)
        result["contact_map_proxy_200k"] = contact_map_proxy(x, log)
        runs = []
        for r in range(opt.rounds):
            for save in ((False, True) if r % 2 == 0 else (True, False)):
                res = ensemble(tmp, opt.members, save, f"{r}_{int(save)}")
                log(f"ensemble round {r} SAVE_CONTACTS={save}: {res['structures_per_hour']:.1f} structures/hour")
                runs.append(res)
        result["ensemble"] = runs
        for save in (False, True):
            rates = [r["structures_per_hour"] for r in runs if r["save_contacts"] == save]
            result[f"ensemble_{'on' if save else 'off'}_structures_per_hour"] = rates
    write(opt.out, result, log)


def write(path, result, log):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as fh:
        json.dump(result, fh, indent=1)
    log(f"wrote {path}")


if __name__ == "__main__":
    main()
