#!/usr/bin/env python
"""bench.py — force evaluations per second of the genome-wide MultiMM model on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload gw|chrom|region|stress] [--decompose] [--dump-outputs DIR]

Metric (BASELINE.json: "genome-wide minimization wall-time; force evals/s; ensemble
structures/hour"): the headline `value` is metric 2, combined energy+force evaluations per second
of the genome-wide system (N = 2e5 beads, flags of examples/config_gw.ini).  A step is ONE fused
evaluation of every term (prepare -> exact all-pairs kernel -> bonded/external pass -> energy
reduction) — the thing OpenMM does once per L-BFGS line-search trial.  The workload is built the
way a user builds it: synthetic .bedpe/.bed files in the reference's formats -> loaders ->
MultiMM.add_* -> engine (C-ABI).  Metrics 1 and 3 ride on the same line:

`value`  : inputs resident in HBM, K evaluations timed with CUDA events on the engine's stream.
`e2e`    : the same evaluation through the C-ABI with HOST buffers: positions copied host->device
           and forces device->host every step (what LocalEnergyMinimizer does per evaluation).
`roofline`: the exact pair kernel against the FP32-FMA peak: `frac` against the FFMA micro-benchmark
           run inside this bench, `frac_nominal` against 148 SM x 128 lanes x 2 x the maximum SM clock
           (MEASURED_PEAKS.json carries only HBM and bf16; this kernel is bound by the FP32 / MUFU
           pipes, not by HBM or tensor cores).  Algorithmic flops: SURVEY.md 8(d).
`minimize_full` (N = 1): metric 1 — the genome-wide system minimised to OpenMM's default tolerance
           with unlimited iterations on the exact potential: wall seconds, iterations, evaluations,
           final energy; and the opt-in two-stage variant (taken from the ensemble member below).
`ensemble`: metric 3 — every rank runs ONE ensemble member through the driver's own per-replica
           pipeline (run.run_replica: loaders, init CIF/PSF, force field, minimisation, minimised
           CIF, per-chromosome CIFs, tar.gz) on its GPU; structures/hour = ranks x 3600 / slowest.
--dump-outputs DIR: what the last timed evaluation returned, DIR/energy_terms.npy (10,) kJ/mol and
           DIR/forces.npy (N, 3) kJ/mol/nm, float64 (rank 0).  The inputs are seeded, so two builds run
           with the same arguments can be compared array for array.
`decomposed` (N > 1): the N = 2e6 stress system with its pair work shared by the ranks
           (mmm_dist.cu): ms per evaluation, pair-kernel share, ms in the exchange step.
`cpu_baseline`: the CPU oracle (FP64 restatement of the OpenMM Reference semantics, OpenMP, thread
           count set explicitly and reported as measured) on a bounded sample of the same system.
--impl reference: OpenMM through the unmodified reference (bench_openmm.py) when it imports; else
           the oracle port, each step a bounded sample scaled by pair count, plus ONE real full-size
           evaluation timed once.
N > 1 (torchrun): one independent replica per GPU (ensemble members, seeds = rank), no data-path
collective; value = evaluations of all ranks / max-over-ranks device time; scaling "weak".
--decompose (N > 1): headline = ONE system (use --workload stress) whose pair work is shared by the
ranks; scaling "strong".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (synthetic config key, flags)
    "gw": dict(key="S3_gw", n_beads=200_000, chrom=None, region=None, n_loops=10_000,
               flags=dict(SC_USE_SPHERICAL_CONTAINER=True, CHB_USE_CHROMOSOMAL_BLOCKS=True,
                          SCB_USE_SUBCOMPARTMENT_BLOCKS=True, IBL_USE_B_LAMINA_INTERACTION=True,
                          CF_USE_CENTRAL_FORCE=True, COB_USE_COMPARTMENT_BLOCKS=False, SHUFFLE_CHROMS=True),
               name="genome-wide, N=200000, 22 chromosomes, EV+SCB+CHB+SC+LAM+CF+bonds+loops+angles "
                    "(examples/config_gw.ini flags), exact all-pairs"),
    "chrom": dict(key="S2_chrom", n_beads=50_000, chrom="chr1", region=None, n_loops=2_000,
                  flags=dict(SCB_USE_SUBCOMPARTMENT_BLOCKS=True),
                  name="single chromosome chr1, N=50000, EV+SCB+bonds+loops+angles, exact all-pairs"),
    "stress": dict(key="S5_stress", n_beads=2_000_000, chrom=None, region=None, n_loops=100_000,
                   flags=dict(SC_USE_SPHERICAL_CONTAINER=True, CHB_USE_CHROMOSOMAL_BLOCKS=True,
                              SCB_USE_SUBCOMPARTMENT_BLOCKS=True, IBL_USE_B_LAMINA_INTERACTION=True,
                              CF_USE_CENTRAL_FORCE=True, COB_USE_COMPARTMENT_BLOCKS=False, SHUFFLE_CHROMS=True),
                   name="high-resolution genome-wide stress test, N=2000000, 22 chromosomes, EV+SCB+CHB+SC+LAM+CF+"
                        "bonds+loops+angles, exact all-pairs"),
    "region": dict(key="S1_region", n_beads=10_000, chrom="chr1", region=(10_000_000, 110_000_000), n_loops=400,
                   flags=dict(), name="specific region chr1:10-110Mb, N=10000, EV+bonds+loops+angles, exact all-pairs"),
}


def config_kwargs(workload: str, seed: int, tmp: str) -> dict:
    """Synthetic input files (the reference's formats) and the SimulationConfig fields of a workload."""
    from multimm_b200 import synthetic

    w = WORKLOADS[workload]
    bedpe = os.path.join(tmp, f"loops_{seed}.bedpe")
    bed = os.path.join(tmp, f"comps_{seed}.bed")
    if not os.path.exists(bedpe):
        synthetic.write_bedpe(bedpe, n_loops=w["n_loops"], seed=100 + seed, chrom=w["chrom"], region=w["region"])
        synthetic.write_bed(bed, seed=100 + seed, chrom=w["chrom"])
    kw = dict(N_BEADS=w["n_beads"], LOOPS_PATH=bedpe, COMPARTMENT_PATH=bed,
              OUT_PATH=os.path.join(tmp, f"out_{seed}"), SHUFFLING_SEED=seed, SAVE_PLOTS=False, **w["flags"])
    if w["chrom"]:
        kw["CHROM"] = w["chrom"]
    if w["region"]:
        kw["LOC_START"], kw["LOC_END"] = w["region"]
    return kw


def build_model(workload: str, seed: int, device: int, tmp: str, with_engine: bool = True):
    """Synthetic input files -> SimulationConfig -> MultiMM with its force field on the device."""
    from multimm_b200.config import SimulationConfig
    from multimm_b200.model import MultiMM

    args = SimulationConfig(PLATFORM="B200", **config_kwargs(workload, seed, tmp))
    m = MultiMM(args, device=device)
    m.set_radiuses()
    if with_engine:
        m.initialize_simulation()
        m.add_forcefield()
    return m


def oracle_system(m, n_sub: int):
    """The first n_sub beads of the model as an oracle System (same parameters, same start)."""
    from multimm_b200 import structures
    from multimm_b200.model import _f, backbone_angles, backbone_bonds
    from oracle import oracle as O

    a = m.args
    n = a.N_BEADS
    x = structures.hilbert_points_host(n, 8).astype(np.float64) * 0.1
    center = x.mean(axis=0)
    sub = slice(0, n_sub)
    bi = backbone_bonds(n, m.chr_ends)
    bi = bi[bi + 1 < n_sub]
    ai = backbone_angles(n, m.chr_ends)
    ai = ai[ai + 2 < n_sub]
    keep = np.asarray(m.ns) < n_sub
    lm, ln, lr0 = np.asarray(m.ms)[keep], np.asarray(m.ns)[keep], np.asarray(m.ds)[keep]
    s = np.zeros(n, dtype=np.int8) if m.Cs is None else np.asarray(m.Cs, dtype=np.int8)
    sysd = O.System(
        n=n_sub,
        ev=(0, [a.EV_EPSILON, a.EV_R_SMALL, _f(a.LE_HARMONIC_BOND_R0), a.EV_POWER]) if a.EV_USE_EXCLUDED_VOLUME else None,
        cob=(0, [m.r_comp, a.COB_EA, a.COB_EB]) if a.COB_USE_COMPARTMENT_BLOCKS else None,
        scb=(0, [m.r_comp, a.SCB_EA1, a.SCB_EA2, a.SCB_EB1, a.SCB_EB2]) if a.SCB_USE_SUBCOMPARTMENT_BLOCKS else None,
        chb=(0, [a.CHB_KC, a.CHB_DE]) if a.CHB_USE_CHROMOSOMAL_BLOCKS else None,
        sc=(0, [a.SC_SCALE, m.radius1, m.radius2, *center]) if a.SC_USE_SPHERICAL_CONTAINER else None,
        lam=(0, [a.IBL_SCALE, m.radius1, m.radius2, *center]) if a.IBL_USE_B_LAMINA_INTERACTION else None,
        cf=(0, [a.CF_STRENGTH, m.radius1, *center]) if a.CF_USE_CENTRAL_FORCE else None,
        s=s[sub], chrom=m.chrom_spin[sub].astype(np.int32), cstr=m.chrom_strength[sub],
        bonds=(bi, bi + 1, np.full(len(bi), _f(a.POL_HARMONIC_BOND_R0)), np.full(len(bi), _f(a.POL_HARMONIC_BOND_K))),
        loops=(lm, ln, lr0, np.full(len(lm), _f(a.LE_HARMONIC_BOND_K))),
        angles=(ai, ai + 1, ai + 2, np.full(len(ai), _f(a.POL_HARMONIC_ANGLE_R0)),
                np.full(len(ai), _f(a.POL_HARMONIC_ANGLE_CONSTANT_K))),
    )
    return sysd, x[sub].copy()


def openmm_probe() -> str:
    """BASELINE.md section 3, step 1: is the real reference backend importable (also from a
    driver-provided baseline/_ref)?  The answer is recorded in the JSON line."""
    import bench_openmm

    ok, why = bench_openmm.available()
    return ("importable: `bench.py --impl reference` times the unmodified reference on it" if ok
            else f"not importable ({why}): OpenMM-CPU and OpenMM-CUDA are unmeasured")


def oracle_threads() -> tuple[int, int]:
    """(threads asked for, threads the OpenMP runtime really gives).  Asked for = the hardware threads
    of the affinity mask, passed EXPLICITLY: under torchrun OMP_NUM_THREADS=1 is exported, and an
    oracle left at its default would run on one core while the line says 32."""
    from oracle import oracle as O

    want = O.host_threads()
    return want, O.threads_used(want)


def cpu_baseline(m, target_seconds: float = 12.0, reps: int = 1):
    """Oracle timed on all host cores on a bounded sample; extrapolated to the full system by
    pair count (the O(N^2) pair loop is > 99.9 % of the oracle's time)."""
    from oracle import oracle as O

    n = m.args.N_BEADS
    want, cores = oracle_threads()
    sysd, x = oracle_system(m, min(n, 6000))
    O.energy_forces(sysd, x, nthreads=want)  # warm
    t0 = time.perf_counter()
    O.energy_forces(sysd, x, nthreads=want)
    probe = time.perf_counter() - t0
    rate = (sysd.n * (sysd.n - 1) / 2) / max(probe, 1e-9)  # pairs/s
    n_sub = int(min(n, max(6000, np.sqrt(2.0 * rate * target_seconds / max(reps, 1)))))
    sysd, x = oracle_system(m, n_sub)
    t0 = time.perf_counter()
    for _ in range(reps):
        O.energy_forces(sysd, x, nthreads=want)
    dt = (time.perf_counter() - t0) / reps
    pairs_sub = n_sub * (n_sub - 1) / 2
    pairs_full = n * (n - 1) / 2
    evals_per_s = (pairs_sub / dt) / pairs_full
    return dict(value=evals_per_s, unit="force_evals/s", cores=cores, kind="port",
                sample=f"CPU oracle (FP64 restatement of OpenMM Reference semantics, OpenMP x{cores} threads measured, "
                       f"{want} requested explicitly) on the first "
                       f"{n_sub} beads of the same system ({pairs_sub:.3g} pairs in {dt:.2f} s), EXTRAPOLATED to "
                       f"{pairs_full:.3g} pairs by pair count; OpenMM itself is not installable here (no wheel, no network)",
                extrapolated=n_sub < n, pairs_per_s=pairs_sub / dt, sample_beads=n_sub, sample_seconds=dt,
                omp_num_threads_env=os.environ.get("OMP_NUM_THREADS"), openmm=openmm_probe())


def oracle_full_evaluation(m) -> dict:
    """ONE real evaluation of the whole system by the oracle (no sample, no extrapolation)."""
    from oracle import oracle as O

    want, cores = oracle_threads()
    sysd, x = oracle_system(m, m.args.N_BEADS)
    t0 = time.perf_counter()
    e, _ = O.energy_forces(sysd, x, nthreads=want)
    dt = time.perf_counter() - t0
    return dict(seconds=dt, force_evals_per_s=1.0 / dt, cores=cores, beads=int(m.args.N_BEADS),
                energy_kj_mol=float(e.sum()), note="timed, not extrapolated: every pair of the full system")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md).  nvidia-smi takes
    a few hundred ms to deliver its first line, longer than a short timed region, so the sampler is started
    ahead of it (before the warm-up); `mark_start` / `mark_end` bracket the timed region and the summary
    keeps the samples that arrived inside the bracket (plus one sampling period)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD_MS = 50

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines: list[tuple[float, str]] = []
        self.t0 = self.t1 = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.PERIOD_MS)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            t_wait = time.perf_counter()
            while not self.lines and time.perf_counter() - t_wait < 3.0:  # the first line: nvidia-smi is up
                time.sleep(0.01)
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark_start(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(1.5 * self.PERIOD_MS / 1e3)  # let the sample of the last period arrive
            self.proc.kill()  # exact PID we started
            self.proc.wait()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        lo = self.t0 if self.t0 is not None else -1e30
        hi = (self.t1 if self.t1 is not None else 1e30) + self.PERIOD_MS / 1e3
        for when, ln in self.lines:
            if not (lo <= when <= hi):
                continue
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, name in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(np.max(mx)), reasons=sorted(reasons),
                    samples=len(sm))


def pair_flops(m) -> tuple[float, float]:
    """Algorithmic flops of one evaluation of the pair kernel (SURVEY.md 8d): per unordered pair
    16 (geometry + accumulation) + (body + 2) per active term: EV power-law 12, each Gaussian block
    term 6, CHB polynomial 12 charged on same-chromosome pairs only.  Returns (flops, pairs)."""
    a = m.args
    n = a.N_BEADS
    pairs = n * (n - 1) / 2.0
    per = 16.0
    if a.EV_USE_EXCLUDED_VOLUME:
        per += 12.0
    per += 6.0 * (bool(a.COB_USE_COMPARTMENT_BLOCKS) + bool(a.SCB_USE_SUBCOMPARTMENT_BLOCKS))
    flops = pairs * per
    if a.CHB_USE_CHROMOSOMAL_BLOCKS:
        sizes = np.diff(np.asarray(m.chr_ends)).astype(np.float64)
        flops += 12.0 * float((sizes * (sizes - 1) / 2.0).sum())
    return flops, pairs


NOMINAL_SM, NOMINAL_LANES = 148, 128


def nominal_fp32_tflops(sm_max_mhz: float | None) -> float:
    """148 SMs x 128 FP32 lanes x 2 flop x the maximum SM clock (1965 MHz on this pool: 74.4)."""
    mhz = sm_max_mhz if sm_max_mhz and sm_max_mhz > 0 else 1965.0
    return NOMINAL_SM * NOMINAL_LANES * 2 * mhz * 1e6 / 1e12


def max_over_ranks(values, device):
    """Device timings are reduced with MAX over ranks (no-op for one process)."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def min_over_ranks(values, device):
    """MIN over ranks: e.g. the exchange step without the wait for the slowest rank."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return [float(v) for v in t]


def whole_job_rate(world: int, steps: int, total_ms: float) -> float:
    """Evaluations of all ranks per second of the slowest rank (weak scaling: one replica per GPU)."""
    return world * steps / (total_ms * 1e-3)


def replica_seed(rank: int) -> int:
    """Rank r runs ensemble member r (SHUFFLING_SEED = r, run.py:473-476)."""
    return rank


def structures_per_hour(world: int, slowest_seconds: float) -> float:
    """One ensemble member per rank, all at once: members x 3600 / wall of the slowest."""
    return world * 3600.0 / slowest_seconds


def run_pipeline_on() -> bool:
    from multimm_b200 import run

    return run.pipeline_enabled()


def ensemble_members(workload: str, rank: int, world: int, device: int, tmp: str, coarse_cutoff: float, count: int) -> dict:
    """`count` ensemble members on this rank's GPU through the driver's per-replica pipeline
    (multimm_b200.run.run_replicas_on_device == the loop at run.py:473-485): parse inputs, Hilbert
    start, init CIF + PSF, force field, minimisation to OpenMM's default tolerance, minimised CIF,
    per-chromosome CIFs, tar.gz — the archive of member k is written while member k + 1 minimises.
    Member seeds: rank, rank + world, ... (replica i -> GPU i mod G, as run.assign_replicas deals them)."""
    from multimm_b200 import run
    from multimm_b200.config import SimulationConfig

    seeds = [replica_seed(rank) + world * k for k in range(count)]
    kw = config_kwargs(workload, seeds[0], tmp)
    kw.update(PLATFORM="B200", GENERATE_ENSEMBLE=True, N_ENSEMBLE=max(seeds) + 1, MIN_COARSE_CUTOFF=coarse_cutoff)
    params = SimulationConfig(**kw).model_dump()
    paths = {i: os.path.join(tmp, f"ens_{coarse_cutoff}_{i}") for i in seeds}
    got = []
    t0 = time.perf_counter()
    run.run_replicas_on_device(params, paths, seeds, device, True, got.append)
    wall = time.perf_counter() - t0
    bad = [p for kind, p in got if kind != "ok"]
    if bad:
        raise RuntimeError(f"ensemble member failed: {bad}")
    reps = [p for kind, p in got if kind == "ok"]
    run.check_archives(reps)
    return dict(wall_seconds=wall, members=reps)


def dump_outputs(path: str, e_terms: np.ndarray, forces: np.ndarray) -> None:
    """The arrays a caller of the evaluation receives, as float64 .npy (N = 2e6, the largest
    workload, makes 48 MB of forces)."""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "energy_terms.npy"), np.asarray(e_terms, dtype=np.float64))
    np.save(os.path.join(path, "forces.npy"), np.asarray(forces, dtype=np.float64))


def run_ours(opt):
    import torch
    import torch.distributed as dist

    from multimm_b200.engine import measure_fp32_peak

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    K, W = opt.steps, max(opt.warmup, 3)
    w = WORKLOADS[opt.workload]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def share_dist_id(eng):
        from multimm_b200.engine import Engine

        box = [Engine.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.dist_init(rank, world, box[0])

    with tempfile.TemporaryDirectory(prefix="mmm_bench_") as tmp:
        t_build0 = time.perf_counter()
        decomposed = bool(opt.decompose) and world > 1
        # replicas (default): rank r is ensemble member r.  --decompose: every rank builds the SAME
        # system and the ranks share its pair work (one exchange step per evaluation, mmm_dist.cu)
        m = build_model(opt.workload, seed=0 if decomposed else replica_seed(rank), device=local, tmp=tmp)
        eng = m.engine
        if decomposed:
            share_dist_id(eng)
        build_s = time.perf_counter() - t_build0
        n = m.args.N_BEADS

        # ---- device-resident: K evaluations, CUDA events on the engine's stream -----------------
        with ClockSampler(local) as clk:
            eng.evaluate_timed(W, flush_l2=True)
            launches0 = eng.launch_count
            barrier()
            clk.mark_start()
            total_ms, pair_ms = eng.evaluate_timed(K, flush_l2=True)
            barrier()
            clk.mark_end()
        launches = eng.launch_count - launches0
        if opt.dump_outputs and rank == 0:
            dump_outputs(opt.dump_outputs, *eng.last_result())
        coll_ms = eng.last_collective_ms if decomposed else 0.0
        total_ms, pair_ms_max, coll_ms = max_over_ranks([total_ms, pair_ms, coll_ms], device=dev)
        value = whole_job_rate(1 if decomposed else world, K, total_ms)

        # ---- end to end through the C-ABI with host buffers ------------------------------------
        x_host = torch.from_numpy(m.positions.copy()).pin_memory()
        x_np = x_host.numpy()
        f_host = torch.empty((n, 3), dtype=torch.float64).pin_memory()
        f_np = f_host.numpy()
        for _ in range(2):
            eng.set_positions(x_np)
            eng.energy_forces(out=f_np)
        barrier()
        t0 = time.perf_counter()
        for _ in range(K):
            eng.set_positions(x_np)
            e_terms, forces = eng.energy_forces(out=f_np)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_value = whole_job_rate(1 if decomposed else world, K,
                                   1e3 * max_over_ranks([e2e_s], device=dev)[0])

        # ---- metric 1 (N = 1): the whole minimisation, exact potential, OpenMM's defaults -----------
        mini = mini_full = None
        pair_kernel = eng.pair_kernel_in_use
        # (these objects ride on the contract line: a failure in one of them must not cost the line)
        if world == 1 and opt.minimize_iters > 0:
            try:
                eng.set_positions(x_np)
                mini = dict(max_iter=opt.minimize_iters, **eng.minimize(tol=10.0, max_iter=opt.minimize_iters))
            except Exception as e:
                mini = dict(error=f"{type(e).__name__}: {e}")
        if world == 1 and not opt.no_minimize_full and opt.workload != "stress":
            try:
                eng.set_positions(x_np)
                rep = eng.minimize(tol=10.0, max_iter=0)
                mini_full = dict(exact=dict(rep, tolerance_kj_mol_nm=10.0, max_iter="unlimited",
                                            potential="exact all-pairs (reference semantics, model.py:886)"))
            except Exception as e:
                mini_full = dict(exact=dict(error=f"{type(e).__name__}: {e}"))
        flops, pairs = pair_flops(m)
        m.close()

        # ---- metric 3: one ensemble member per rank through the driver's pipeline ----------------
        ens = None
        if not opt.no_ensemble and opt.workload != "stress" and not decomposed:
            barrier()
            ens_error = None
            try:
                mine = ensemble_members(opt.workload, rank, world, local, tmp, opt.coarse_cutoff, opt.ensemble_members)
            except Exception as e:  # this object is an add-on to the contract line: a failure must not cost the line
                mine, ens_error = dict(wall_seconds=1e30, members=[]), f"{type(e).__name__}: {e}"
            slow = max_over_ranks([mine["wall_seconds"]], device=dev)[0]
            keep = ("replica", "seconds", "iterations", "evaluations", "e_final", "converged", "initialize_s",
                    "forcefield_s", "minimize_s", "write_cif_s", "coarse_iterations", "coarse_seconds", "coarse_rounds",
                    "exact_iterations", "archive_inline_s", "prepare_s", "compute_s", "finish_s")
            members = world * opt.ensemble_members
            if slow >= 1e29:
                ens = dict(error=ens_error or "an ensemble member failed on another rank", members=members, gpus=world)
            else:
                ens = dict(structures_per_hour=members * 3600.0 / slow, members=members, members_per_gpu=opt.ensemble_members,
                           gpus=world, slowest_rank_seconds=slow, unit="structures/hour",
                           mode=(f"opt-in two-stage minimisation (MIN_COARSE_CUTOFF = {opt.coarse_cutoff} nm, then the exact "
                                 "potential to the same stopping rule)" if opt.coarse_cutoff > 0 else
                                 "reference semantics (exact potential throughout)"),
                           pipeline="run.run_replicas_on_device: loaders, Hilbert start, init CIF + PSF, force field, minimisation, "
                                    "minimised CIF, per-chromosome CIFs, tar.gz (run.py:473-485); member k + 1 is prepared and "
                                    "member k - 1 written out and archived on background threads while member k minimises"
                                    if run_pipeline_on() else
                                    "run.run_replicas_on_device, MMM_ENSEMBLE_PIPELINE=0: members one after another, only the "
                                    "tar.gz in the background",
                           rank0_members=[{k: r[k] for k in keep if k in r} for r in mine["members"]])
            if mini_full is not None and opt.coarse_cutoff > 0 and ens.get("rank0_members"):
                mini_full["two_stage"] = dict(ens["rank0_members"][0], coarse_cutoff_nm=opt.coarse_cutoff,
                                              note="minimize_s = both stages; same stopping rule met on the exact potential")

        # ---- N > 1: the N = 2e6 stress system, pair work shared by the ranks ----------------------
        deco = None
        if world > 1 and not decomposed and not opt.no_decomposed:
            barrier()
            t0 = time.perf_counter()
            ms_ = build_model("stress", seed=0, device=local, tmp=tmp)
            share_dist_id(ms_.engine)
            ms_.engine.evaluate_timed(3, flush_l2=True)
            barrier()
            d_tot, d_pair = ms_.engine.evaluate_timed(opt.decomposed_steps, flush_l2=True)
            barrier()
            d_coll = ms_.engine.last_collective_ms
            d_pair_min, d_coll_min = min_over_ranks([d_pair, d_coll], device=dev)
            d_tot, d_pair, d_coll = max_over_ranks([d_tot, d_pair, d_coll], device=dev)
            ks = opt.decomposed_steps
            deco = dict(workload=WORKLOADS["stress"]["name"], n_beads=ms_.args.N_BEADS, gpus=world, steps=ks,
                        ms_per_evaluation=d_tot / ks, force_evals_per_s=ks / (d_tot * 1e-3), scaling="strong",
                        pair_kernel_ms=d_pair / ks, pair_kernel_share=d_pair / d_tot,
                        pair_kernel_ms_fastest_rank=d_pair_min / ks,
                        exchange_ms=d_coll, exchange_ms_fastest_rank=d_coll_min,
                        exchange="one NCCL all-reduce (uint64 sum) of the fixed-point force planes and the per-item energy "
                        "slots; CUDA events around it on the engine's stream, last evaluation.  A rank's figure includes its "
                        "wait for the slowest rank's pair kernel: the smallest over ranks is the collective itself",
                        work_queue=("one queue for all GPUs (ticket counters in rank 0's memory, CUDA IPC, system-scope "
                                    "atomics over NVLink)" if ms_.engine.dist_queue_mode else "static round-robin dealing"),
                        build_seconds=time.perf_counter() - t0,
                        single_gpu_reference="profiles/: 1 GPU runs the same system in ms_per_evaluation x speed-up")
            ms_.close()

        if rank != 0:
            if world > 1:
                dist.destroy_process_group()
            return

        # ---- rank 0 only: roofline, CPU baseline ------------------------------------------------
        if decomposed:  # this rank's kernel evaluates 1 / world of the pairs
            flops, pairs = flops / world, pairs / world
        peak_tflops, mufu_tops = measure_fp32_peak(local)
        clocks = clk.summary()
        nominal = nominal_fp32_tflops(clocks.get("sm_max_mhz"))
        pair_ms_avg = pair_ms / K
        achieved = flops / (pair_ms_avg * 1e-3) / 1e12
        traffic = None
        try:  # DRAM bytes of one launch from the committed ncu --set full capture of this kernel
            with open(os.path.join(ROOT, "profiles", "pair_n3_traffic.json")) as fh:
                tj = json.load(fh)
            if pair_kernel == 2 and opt.workload == "gw" and not decomposed:
                traffic = tj["dram_bytes_per_launch"]
        except (OSError, KeyError, ValueError):
            pass
        kernel_name = {1: "k_pair_exact (gather)", 2: "k_pair_n3 (Newton-3)", 3: "k_pair_cells"}.get(pair_kernel, "none")
        roofline = dict(
            bound="fp32", kernel=kernel_name, achieved=achieved, peak=peak_tflops, unit="TFLOP/s",
            frac=achieved / peak_tflops if peak_tflops > 0 else None,
            peak_nominal=nominal, frac_nominal=achieved / nominal, traffic=traffic,
            traffic_unit="bytes of DRAM per launch (ncu capture under profiles/); the kernel is FMA-pipe bound",
            peak_source="`peak`: FFMA micro-benchmark run inside this bench (MEASURED_PEAKS.json has no FP32 entry; SASS "
                        "of its loop under profiles/); `peak_nominal`: 148 SM x 128 lanes x 2 x max SM clock; "
                        f"MUFU peak measured likewise: {mufu_tops:.2f} Tera-op/s",
            algorithmic_flops_per_launch=flops, unordered_pairs_per_launch=pairs,
            pair_kernel_ms=pair_ms_avg, pairs_per_s=pairs / (pair_ms_avg * 1e-3),
            kernel_share_of_step=pair_ms / total_ms)
        base = None
        if world == 1 and not opt.no_cpu:
            base = cpu_baseline(m, target_seconds=opt.cpu_seconds)
        out = dict(
            metric="force_evals_per_s", value=value, unit="force_evals/s", n_gpus=world, steps=K, warmup=W,
            ms_per_step=total_ms / K, higher_is_better=True, scaling="strong" if decomposed else "weak",
            vs_baseline=None, dtype="f32",
            data="synthetic",
            config=dict(workload=w["name"], n_beads=n, n_loops=int(len(m.ms)), n_bonds=int(m.n_bonds),
                        n_angles=int(m.n_angles), replicas=1 if decomposed else world,
                        parallelism=(f"one system, pair work sharded over {world} GPUs, 1 exchange step per evaluation"
                                     if decomposed else f"{world} independent replica(s), no collective"), l2="flushed between steps (256 MiB memset inside "
                        "the timed region)", start="Hilbert lattice (0.1 nm)", build_seconds=build_s),
            clocks=clocks,
            e2e=dict(value=e2e_value, unit="force_evals/s", h2d_bytes_per_step=24 * n,
                     d2h_bytes_per_step=24 * n + 8 * len(e_terms)),
            gpu_launches=int(launches),
            roofline=roofline, cpu_baseline=base, minimize=mini, minimize_full=mini_full, ensemble=ens,
            decomposed=deco, exchange_ms=coll_ms if decomposed else None,
            energy_terms={k: float(v) for k, v in zip(("EV", "COB", "SCB", "CHB", "SC", "LAM", "CF", "BOND", "LOOP",
                                                        "ANGLE"), e_terms)},
        )
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_reference_openmm(opt, w, tmp):
    """The real reference: OpenMM through multimm.model.MultiMM, CPU platform on all host threads
    (the headline of this arm) and, when the platform exists, CUDA on the same GPU."""
    import bench_openmm

    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    kw = config_kwargs(opt.workload, 0, tmp)
    kw["SIM_RUN_MD"] = False
    cap = max(10.0, min(opt.openmm_minimize_cap, 600.0))
    arms = {}
    for plat in ("CPU", "CUDA"):
        if plat not in bench_openmm.platforms():
            arms[plat] = dict(unavailable=f"OpenMM has no {plat} platform on this box")
            continue
        steps = opt.steps if plat == "CUDA" else max(1, min(opt.steps, 3))  # a CPU evaluation of 2e10 pairs is long
        try:
            arms[plat] = bench_openmm.time_arm(kw, plat, steps, min(opt.warmup, 1) if plat == "CPU" else opt.warmup,
                                               threads, minimize_cap_s=cap)
        except Exception as e:
            arms[plat] = dict(unavailable=f"{type(e).__name__}: {e}")
    cpu = arms["CPU"]
    if "force_evals_per_s" not in cpu:
        return None
    value = cpu["force_evals_per_s"]
    return dict(
        impl="reference", metric="force_evals_per_s", value=value, unit="force_evals/s",
        n_gpus=int(os.environ.get("WORLD_SIZE", "1")), steps=opt.steps, warmup=opt.warmup, ms_per_step=1e3 / value,
        higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64/f32 (OpenMM CPU platform)", data="synthetic",
        config=dict(workload=w["name"], n_beads=w["n_beads"], note="unmodified reference (multimm.model.MultiMM) on OpenMM"),
        cpu_baseline=dict(value=value, unit="force_evals/s", cores=threads, kind="reference",
                          sample="full system, every evaluation timed (setPositions + getState(energy, forces))"),
        e2e=dict(value=value, unit="force_evals/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
        gpu_launches=0, openmm=arms)


def run_reference(opt):
    """The reference arm.  With OpenMM and the reference package importable: the unmodified
    reference on OpenMM's CPU (and CUDA) platform.  Otherwise (this image): the reference's CPU
    implementation is represented by the oracle port on all host threads; each step is a bounded
    sample scaled by pair count, and ONE real full-size evaluation is timed beside them."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import bench_openmm

    K, W = opt.steps, opt.warmup
    w = WORKLOADS[opt.workload]
    with tempfile.TemporaryDirectory(prefix="mmm_bench_ref_") as tmp:
        ok, why = bench_openmm.available()
        if ok:
            out = run_reference_openmm(opt, w, tmp)
            if out is not None:
                print(json.dumps(out), flush=True)
                return
        m = build_model(opt.workload, seed=0, device=0, tmp=tmp, with_engine=False)
        budget = max(1.0, min(opt.cpu_seconds, 120.0 / max(K + W, 1)))
        for _ in range(W):
            base = cpu_baseline(m, target_seconds=budget)
        vals, secs = [], []
        t0 = time.perf_counter()
        for _ in range(K):
            base = cpu_baseline(m, target_seconds=budget)
            vals.append(base["value"])
            secs.append(base["sample_seconds"])
        wall = time.perf_counter() - t0
        value = float(np.mean(vals))
        full = None
        if not opt.no_ref_full and m.args.N_BEADS <= 250_000:
            full = oracle_full_evaluation(m)
        out = dict(
            impl="reference", metric="force_evals_per_s", value=value, unit="force_evals/s",
            n_gpus=int(os.environ.get("WORLD_SIZE", "1")), steps=K, warmup=W, ms_per_step=1e3 / value,
            higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
            config=dict(workload=w["name"], n_beads=m.args.N_BEADS,
                        note="EXTRAPOLATED: each step times a bounded bead sample and scales by pair count; ms_per_step "
                             "is the extrapolated time of one full evaluation, not a timed step.  `full_evaluation` is "
                             "one real evaluation of the whole system, timed once."),
            value_is="extrapolated from bounded samples by pair count" if base["extrapolated"] else "timed on the full system",
            sample_seconds_per_step=float(np.mean(secs)), full_evaluation=full,
            cpu_baseline=dict(base, value=value),
            e2e=dict(value=value, unit="force_evals/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
            gpu_launches=0, wall_seconds=wall, openmm=f"not used: {why}")
        print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--workload", default="gw", choices=tuple(WORKLOADS))
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--decompose", action="store_true",
                    help="N > 1: one system whose pair work is shared by the ranks (default: one replica per rank)")
    ap.add_argument("--minimize-iters", type=int, default=50, help="bounded L-BFGS run reported as `minimize` (0: skip)")
    ap.add_argument("--no-minimize-full", action="store_true", help="skip the full minimisation (metric 1, N = 1 only)")
    ap.add_argument("--no-ensemble", action="store_true", help="skip the ensemble member per rank (metric 3)")
    ap.add_argument("--ensemble-members", type=int, default=2, help="ensemble members per rank (metric 3)")
    ap.add_argument("--coarse-cutoff", type=float, default=0.5,
                    help="MIN_COARSE_CUTOFF of the ensemble member in nm (0: reference semantics, exact throughout)")
    ap.add_argument("--no-decomposed", action="store_true", help="N > 1: skip the sharded N = 2e6 system")
    ap.add_argument("--decomposed-steps", type=int, default=5)
    ap.add_argument("--no-ref-full", action="store_true", help="reference arm: skip the one real full-size evaluation")
    ap.add_argument("--openmm-minimize-cap", type=float, default=120.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the energies and forces of the last timed evaluation to DIR/<name>.npy")
    opt = ap.parse_args()
    if opt.dump_outputs and opt.impl != "ours":
        ap.error("--dump-outputs writes what the engine computed: it needs --impl ours")
    if opt.impl == "reference":
        run_reference(opt)
    else:
        run_ours(opt)


if __name__ == "__main__":
    main()
