"""Command line and ensemble driver — mirror of the reference's ``run.py``
(src/multimm/run.py:60-500) on the minimisation path.

    python -m multimm_b200.run -c config.ini [--field value ...] [--gpus 0,1,...]

Same precedence (defaults < ini < CLI, run.py:367-382), same MODELLING_LEVEL presets
(run.py:128-213), same cross-field checks (run.py:219-331), same ``metadata/config_auto.ini`` /
``metadata/output.log`` side products, same ensemble semantics (run.py:471-485: replica i runs
with SHUFFLING_SEED = i in ``run_<i>``, is archived to ``run_<i>.tar.gz`` and its directory
removed).  What changes: ensemble members are independent, so they are dealt to the visible
B200s, one worker process per GPU, replica i -> GPU i mod G, with no communication between
workers (the reference runs them one after the other in a single Python loop).
"""
from __future__ import annotations

import argparse
import configparser
import logging
import multiprocessing as mp
import os
import shutil
import sys
import tarfile
import time
from enum import Enum


def _early_cuda_start():
    """Ensemble worker processes only (run_ensemble exports MMM_WORKER_WARMUP=1 to them): CUDA
    initialisation — several seconds per process when eight start at once on an 8-GPU box — begins on a
    background thread BEFORE this module's own imports (pandas, pydantic: ~3 s) and the first member's
    input ingestion, instead of after them.  ctypes releases the GIL, so the two overlap.  The thread only
    creates and destroys a two-bead handle; whatever is wrong with the device is reported by the member's
    own mmm_create later."""
    if os.environ.get("MMM_WORKER_WARMUP") != "1":
        return None
    import threading

    def warm():
        try:
            import ctypes

            from . import _lib
            lib = _lib.load()
            h = ctypes.c_void_p()
            if lib.mmm_create(0, 2, ctypes.byref(h)) == 0:
                lib.mmm_destroy(h)
        except Exception:  # noqa: BLE001
            pass

    t = threading.Thread(target=warm, name="mmm-cuda-warmup", daemon=True)
    t.start()
    return t


_WARMUP = _early_cuda_start()

from . import loaders  # noqa: E402
from .config import EXTRA_FIELDS, SimulationConfig, contact_setting  # noqa: E402
from .units import Quantity  # noqa: E402

logger = logging.getLogger("multimm_b200")


class Tee:
    """run.py:60-71"""

    def __init__(self, *streams):
        self.streams = streams

    def write(self, data):
        for s in self.streams:
            s.write(data)
            s.flush()

    def flush(self):
        for s in self.streams:
            s.flush()


# MODELLING_LEVEL presets (run.py:137-213).  `None` = "on iff a compartment file was given".
_OFF5 = dict(SC_USE_SPHERICAL_CONTAINER=False, CHB_USE_CHROMOSOMAL_BLOCKS=False, SCB_USE_SUBCOMPARTMENT_BLOCKS=False,
             IBL_USE_B_LAMINA_INTERACTION=False, CF_USE_CENTRAL_FORCE=False)
PRESETS = {
    "gene": dict(N_BEADS=1000, **_OFF5, COB_USE_COMPARTMENT_BLOCKS=False, SHUFFLE_CHROMS=False, SIM_RUN_MD=True,
                 SIM_N_STEPS=10000),
    "region": dict(N_BEADS=5000, **_OFF5, COB_USE_COMPARTMENT_BLOCKS=None, SIM_RUN_MD=True, SIM_N_STEPS=10000),
    "chromosome": dict(N_BEADS=20000, **_OFF5, COB_USE_COMPARTMENT_BLOCKS=None, SIM_RUN_MD=True, SIM_N_STEPS=10000),
    "gw": dict(N_BEADS=200000, SC_USE_SPHERICAL_CONTAINER=True, CHB_USE_CHROMOSOMAL_BLOCKS=False,
               SCB_USE_SUBCOMPARTMENT_BLOCKS=False, COB_USE_COMPARTMENT_BLOCKS=None, IBL_USE_B_LAMINA_INTERACTION=None,
               CF_USE_CENTRAL_FORCE=False, SIM_RUN_MD=False, SIM_N_STEPS=10000),
}
_ALIASES = {"loc": "region", "chrom": "chromosome", "genome": "gw"}


class ArgumentChanger:
    """run.py:73-217: presets that silently override flags; every change is reported."""

    def __init__(self, args, chrom_sizes=None):
        self.args = args
        self.chrom_sizes = chrom_sizes or loaders.CHROM_SIZES
        self.changed: dict = {}

    def set_arg(self, name, value):
        if not hasattr(self.args, name):
            logger.warning(f"Argument '{name}' not found in args object.")
            return
        self.changed.setdefault(name, getattr(self.args, name))
        setattr(self.args, name, value)

    def convenient_argument_changer(self):
        # nucleosome interpolation is always forced off (run.py:130-131)
        self.set_arg("NUC_DO_INTERPOLATION", False)
        self.set_arg("ATACSEQ_PATH", None)
        level = str(self.args.MODELLING_LEVEL or "").lower()
        level = _ALIASES.get(level, level)
        preset = PRESETS.get(level)
        if preset:
            logger.warning(f"{level}-level modelling activated. This will overwrite parameters.")
            has_comps = bool(self.args.COMPARTMENT_PATH)
            for name, value in preset.items():
                self.set_arg(name, has_comps if value is None else value)
            if level == "chromosome":
                self.set_arg("LOC_START", 1)
                self.set_arg("LOC_END", self.chrom_sizes[self.args.CHROM])
            self.report()

    def report(self):
        rows = [(k, old, getattr(self.args, k)) for k, old in self.changed.items() if old != getattr(self.args, k)]
        if rows:
            logger.warning("MODELLING LEVEL OVERRIDE ACTIVE: parameters have been overwritten.")
            print("\nChanged parameters:\n" + "-" * 60)
            for k, old, new in rows:
                print(f"{k:35s} : {old}  ->  {new}")
            print("-" * 60 + "\n")


def _empty(v) -> bool:
    return v is None or v == ""


def args_tests(args):
    """Cross-field validation, run.py:219-331: same conditions, same order, same exception type."""

    def check_file(path, name, hint):
        if not _empty(path) and not os.path.exists(path):
            raise ValueError(f"{name} file was provided but not found: {path} (expected {hint})")

    if _empty(args.LOOPS_PATH):
        raise ValueError("Loops interaction data is required to run MultiMM. "
                         "Please provide a valid .bedpe file via LOOPS_PATH.")
    check_file(args.LOOPS_PATH, "Loops (.bedpe)", ".bedpe")
    check_file(args.COMPARTMENT_PATH, "Compartment data", ".bed")
    check_file(args.ATACSEQ_PATH, "Nucleosome/ATAC data", ".bigwig")

    no_comps = _empty(args.COMPARTMENT_PATH)
    if no_comps and args.COB_USE_COMPARTMENT_BLOCKS:
        raise ValueError("Compartment modeling is enabled, but no compartment data was provided. "
                         "Please supply a .bed file or disable COB_USE_COMPARTMENT_BLOCKS.")
    elif args.NUC_DO_INTERPOLATION and args.ATACSEQ_PATH is None:
        raise ValueError("Nucleosome interpolation is enabled, but no occupancy data was found. "
                         "Provide a .bigwig file via ATACSEQ_PATH or disable NUC_DO_INTERPOLATION.")
    elif no_comps and args.SCB_USE_SUBCOMPARTMENT_BLOCKS:
        raise ValueError("Subcompartment modeling requires input data. "
                         "Please provide a .bed file or disable SCB_USE_SUBCOMPARTMENT_BLOCKS.")
    elif args.COMPARTMENT_PATH is None and args.IBL_USE_B_LAMINA_INTERACTION:
        raise ValueError("Lamina interactions depend on compartment annotations. "
                         "Please provide a compartment .bed file or disable IBL_USE_B_LAMINA_INTERACTION.")
    elif args.IBL_USE_B_LAMINA_INTERACTION and not (args.SCB_USE_SUBCOMPARTMENT_BLOCKS or args.COB_USE_COMPARTMENT_BLOCKS):
        raise ValueError("Lamina interactions are enabled but no compartment-based forces are active. Enable "
                         "COB_USE_COMPARTMENT_BLOCKS or SCB_USE_SUBCOMPARTMENT_BLOCKS, or disable lamina interactions.")
    elif args.CF_USE_CENTRAL_FORCE and args.CHROM is not None:
        raise ValueError("Central force attraction to the nucleolus is typically used for whole-genome simulations. "
                         "Since you are modeling a single chromosome or region, consider disabling CF_USE_CENTRAL_FORCE.")
    elif args.CHB_USE_CHROMOSOMAL_BLOCKS and args.CHROM is not None:
        # the reference only warns here (run.py:296-300), although its own test expects a raise
        logger.warning("Chromosomal block interactions are more meaningful in multi-chromosome systems. "
                       "You may want to disable CHB_USE_CHROMOSOMAL_BLOCKS for single-chromosome simulations.")

    single = args.CHROM is not None and args.CHROM != ""
    if args.SHUFFLE_CHROMS and single:
        logger.warning("Chromosome shuffling is enabled, but you are simulating a specific chromosomal region.")
    if single and args.IBL_USE_B_LAMINA_INTERACTION:
        logger.warning("Lamina interactions are enabled; they are typically more relevant in whole-genome simulations.")
    if single and args.SC_USE_SPHERICAL_CONTAINER:
        logger.warning("A spherical container is being used; it is generally more meaningful for the full genome.")
    if not (args.POL_USE_HARMONIC_BOND and args.POL_USE_HARMONIC_ANGLE and args.EV_USE_EXCLUDED_VOLUME):
        logger.warning("Some fundamental backbone forces are disabled. Make sure this is intentional.")
    if args.CHB_USE_CHROMOSOMAL_BLOCKS:
        logger.warning("Chromosomal block forces are enabled. These are approximate.")

    # checks the reference makes later (or never): here they fail before any I/O or GPU work
    from . import _lib
    from .model import resolve_platform

    resolve_platform(args.PLATFORM)  # ValueError for anything that is neither B200 nor an OpenMM platform name
    if args.SIM_RUN_MD and str(args.SIM_INTEGRATOR_TYPE).lower() not in _lib.MD_INTEGRATORS:
        # the reference builds its integrator in initialize_simulation (model.py:768-808); a config
        # that asks for one this engine does not have must not run a whole minimisation first
        raise ValueError(f"SIM_INTEGRATOR_TYPE={args.SIM_INTEGRATOR_TYPE!r} is not available "
                         f"(supported: {', '.join(_lib.MD_INTEGRATORS)})")
    check_contact_fields(args)
    check_distance_fields(args)
    check_loop_fields(args)
    check_triplet_fields(args)
    check_md_sample_fields(args)


def check_triplet_fields(args):
    """TRIPLET_RESOLUTION >= 0 and, where the modelled stretch is known from the config alone, at most
    triplets.MAX_BINS bins."""
    from . import contacts, triplets

    res = int(contact_setting(args, "TRIPLET_RESOLUTION"))
    if res < 0:
        raise ValueError(f"TRIPLET_RESOLUTION={res} must be >= 0 (0 = automatic)")
    sp = _modelled_spans(args)
    if res > 0 and sp is not None:
        nb = contacts.bin_count(sp, res)
        if nb > triplets.MAX_BINS:
            raise ValueError(f"TRIPLET_RESOLUTION={res} bp gives {nb} three-way map bins; at most {triplets.MAX_BINS} "
                             "are supported (0 = automatic)")


def check_loop_fields(args):
    """LOOP_APA_WINDOW in [0, loops.MAX_WINDOW]."""
    from . import loops

    w = int(contact_setting(args, "LOOP_APA_WINDOW"))
    if not 0 <= w <= loops.MAX_WINDOW:
        raise ValueError(f"LOOP_APA_WINDOW={w} must be in [0, {loops.MAX_WINDOW}] beads")


def check_md_sample_fields(args):
    """MD_SAMPLE_STEP >= 0; when > 0, MD must run, a map must be on (SAVE_CONTACTS or SAVE_DISTANCES, the loop
    readout SAVE_LOOPS or the three-way map SAVE_TRIPLETS), and the MD loop, which runs
    (SIM_N_STEPS // SIM_SAMPLING_STEP) * SIM_SAMPLING_STEP steps, must reach the first sample."""
    step = int(contact_setting(args, "MD_SAMPLE_STEP"))
    if step < 0:
        raise ValueError(f"MD_SAMPLE_STEP={step} must be >= 0 (0 = no trajectory maps)")
    if step == 0:
        return
    if not args.SIM_RUN_MD:
        raise ValueError(f"MD_SAMPLE_STEP={step} samples the MD run, but SIM_RUN_MD is off")
    if not any(contact_setting(args, k) for k in ("SAVE_CONTACTS", "SAVE_DISTANCES", "SAVE_LOOPS", "SAVE_TRIPLETS")):
        raise ValueError(f"MD_SAMPLE_STEP={step} needs a map to sample: enable SAVE_CONTACTS or SAVE_DISTANCES "
                         "(or SAVE_LOOPS, SAVE_TRIPLETS)")
    every = max(1, int(args.SIM_SAMPLING_STEP))
    steps = (int(args.SIM_N_STEPS) // every) * every
    if step > steps:
        raise ValueError(f"MD_SAMPLE_STEP={step} exceeds the {steps} MD steps that run "
                         "((SIM_N_STEPS // SIM_SAMPLING_STEP) * SIM_SAMPLING_STEP): no structure would be sampled")


def check_distance_fields(args):
    """DISTANCE_RESOLUTION >= 0 and, where the modelled stretch is known from the config alone, at most
    distances.MAX_BINS bins."""
    from . import contacts, distances

    res = int(contact_setting(args, "DISTANCE_RESOLUTION"))
    if res < 0:
        raise ValueError(f"DISTANCE_RESOLUTION={res} must be >= 0 (0 = automatic)")
    sp = _modelled_spans(args)
    if res > 0 and sp is not None:
        nb = contacts.bin_count(sp, res)
        if nb > distances.MAX_BINS:
            raise ValueError(f"DISTANCE_RESOLUTION={res} bp gives {nb} distance-map bins; at most {distances.MAX_BINS} "
                             "are supported (0 = automatic)")


def check_contact_fields(args):
    """CONTACT_RADIUS finite and > 0; CONTACT_RESOLUTION >= 0 and CONTACT_FINE_RESOLUTION >= 0 and, where the
    modelled stretch is known from the config alone (not for gene-level runs), at most contacts.MAX_BINS
    and contacts.MAX_FINE_BINS bins."""
    import math

    from . import contacts

    rc = float(contact_setting(args, "CONTACT_RADIUS"))
    if not (math.isfinite(rc) and rc > 0.0):
        raise ValueError(f"CONTACT_RADIUS={rc!r} must be a finite distance > 0 (nm)")
    res = int(contact_setting(args, "CONTACT_RESOLUTION"))
    if res < 0:
        raise ValueError(f"CONTACT_RESOLUTION={res} must be >= 0 (0 = automatic)")
    fine = int(contact_setting(args, "CONTACT_FINE_RESOLUTION"))
    if fine < 0:
        raise ValueError(f"CONTACT_FINE_RESOLUTION={fine} must be >= 0 (0 = no fine map)")
    sp = _modelled_spans(args)
    if sp is None:
        return
    if res > 0:
        nb = contacts.bin_count(sp, res)
        if nb > contacts.MAX_BINS:
            raise ValueError(f"CONTACT_RESOLUTION={res} bp gives {nb} contact-map bins; at most {contacts.MAX_BINS} "
                             "are supported (0 = automatic)")
    if fine > 0:
        nb = contacts.bin_count(sp, fine)
        if nb > contacts.MAX_FINE_BINS:
            raise ValueError(f"CONTACT_FINE_RESOLUTION={fine} bp gives {nb} fine contact-map bins; at most "
                             f"{contacts.MAX_FINE_BINS} are supported")


def _modelled_spans(args):
    """contacts.spans of the modelled stretch where the config alone determines it, else None."""
    from . import contacts

    if str(args.MODELLING_LEVEL or "").lower() == "gene":
        return None
    if args.CHROM is None:
        return contacts.spans(range(22))
    if args.LOC_START is not None and args.LOC_END is not None:
        return contacts.spans([loaders._chrom_index(args.CHROM)], int(args.LOC_START), int(args.LOC_END))
    if args.CHROM in loaders.CHROM_SIZES:
        return contacts.spans([loaders._chrom_index(args.CHROM)], 0, loaders.CHROM_SIZES[args.CHROM])
    return None


def read_ini(path: str) -> dict:
    """Flat {UPPER_NAME: value} over all sections, DEFAULT last (run.py:334-346, 372-377)."""
    cp = configparser.ConfigParser()
    cp.read(path)
    raw: dict = {}
    for section in cp.sections():
        for name, value in dict(cp[section]).items():
            raw[name.upper()] = value
    for name, value in dict(cp.defaults()).items():
        raw[name.upper()] = value
    return raw


def get_config(argv=None):
    """defaults < ini < CLI, then the MODELLING_LEVEL presets, then config_auto.ini (run.py:349-395)."""
    ap = argparse.ArgumentParser(prog="multimm_b200")
    ap.add_argument("-c", "--config_file", metavar="FILE", help="config file (ini format)")
    ap.add_argument("--gpus", default=None, help="comma-separated CUDA device indices for ensemble workers "
                                                 "(default: DEVICE, or every visible GPU for ensembles)")
    for name in (*SimulationConfig.model_fields, *EXTRA_FIELDS):
        ap.add_argument(f"--{name.lower()}")
    ns = vars(ap.parse_args(argv))
    raw = read_ini(ns["config_file"]) if ns.get("config_file") else {}
    for name, value in ns.items():
        if name not in ("config_file", "gpus") and value is not None:
            raw[name.upper()] = value
    try:
        args = SimulationConfig(**raw)
    except Exception as e:
        logger.error(f"Configuration validation failed: {e}")
        raise
    ArgumentChanger(args).convenient_argument_changer()
    write_config(args)
    return args, ns.get("gpus")


def write_config(args) -> str:
    """metadata/config_auto.ini (run.py:398-420)."""
    meta = os.path.join(args.OUT_PATH, "metadata")
    os.makedirs(meta, exist_ok=True)
    path = os.path.join(meta, "config_auto.ini")
    cp = configparser.ConfigParser()
    cp["DEFAULT"] = {}
    for name, value in args.model_dump().items():
        if isinstance(value, Quantity):
            cp["DEFAULT"][name] = f"{value._value} {value.unit.get_name()}"
        elif isinstance(value, Enum):
            cp["DEFAULT"][name] = value.value
        elif value is None:
            cp["DEFAULT"][name] = ""
        else:
            cp["DEFAULT"][name] = str(value)
    with open(path, "w") as fh:
        cp.write(fh)
    logger.info(f"Configuration saved to {path}")
    return path


def archive_run(run_path: str) -> str:
    """tar.gz the run directory, delete it only if the archive exists and is non-empty (run.py:423-445)."""
    tar_path = run_path + ".tar.gz"
    with tarfile.open(tar_path, "w:gz") as tar:
        tar.add(run_path, arcname=os.path.basename(run_path))
    if os.path.exists(tar_path) and os.path.getsize(tar_path) > 0:
        shutil.rmtree(run_path)
    else:
        raise RuntimeError(f"Archive creation failed ({tar_path}). Original directory was NOT deleted.")
    return tar_path


# ---------------------------------------------------------------------------------------------
# ensemble: replicas dealt to GPUs, one worker process per GPU, no communication
# ---------------------------------------------------------------------------------------------
def replica_paths(out_path: str, n_ensemble: int) -> list[str]:
    width = len(str(max(n_ensemble - 1, 0)))
    return [os.path.join(out_path, f"run_{i:0{width}d}") for i in range(n_ensemble)]


def assign_replicas(n_ensemble: int, devices: list[int]) -> dict[int, list[int]]:
    """The static plan, replica i -> devices[i mod G]: the order in which the GPUs take their FIRST
    replicas.  run_ensemble hands the replicas out from one queue (a worker takes the next index when it
    is free), because members differ a lot in cost (the exact stage of the two-stage minimisation takes 3
    iterations in most replicas and hundreds in a few); with equal costs the two coincide."""
    plan: dict[int, list[int]] = {d: [] for d in devices}
    for i in range(n_ensemble):
        plan[devices[i % len(devices)]].append(i)
    return plan


class Archiver:
    """tar.gz of finished run directories on a background thread, so that replica k is archived while
    replica k + 1 minimises on the GPU (gzip and the engine's C calls both release the GIL).  The
    reference archives inline (run.py:478-485); the files written are the same."""

    def __init__(self):
        from concurrent.futures import ThreadPoolExecutor

        self.pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="mmm-archive")
        self.pending = []

    def submit(self, run_path: str):
        t0 = time.time()

        def job():
            tar = archive_run(run_path)
            return tar, time.time() - t0

        self.pending.append(self.pool.submit(job))

    def wait(self) -> float:
        """Block until every archive is written; returns the seconds spent archiving (summed).
        Re-raises the first failure (a run directory that was not deleted because its archive failed)."""
        spent = 0.0
        try:
            for fut in self.pending:
                spent += fut.result()[1]
        finally:
            self.pending = []
            self.pool.shutdown(wait=True)
        return spent


def build_replica(params: dict, i: int, run_path: str, device: int):
    """Host side of one ensemble member up to the point where the GPU is needed: config with
    SHUFFLING_SEED = i and OUT_PATH = run_<i> (run.py:473-476), output tree, input ingestion
    (MultiMM.__init__: the loaders)."""
    from .model import MultiMM

    cfg = SimulationConfig(**{**params, "SHUFFLING_SEED": i, "OUT_PATH": run_path})
    os.makedirs(run_path, exist_ok=True)
    t0 = time.time()
    md = MultiMM(cfg, device=device)
    # outside run_<i>, so that archiving does not take it away; summed by run_ensemble
    md.contacts_file = member_contacts_path(params["OUT_PATH"], i)
    md.contacts_fine_file = member_contacts_fine_path(params["OUT_PATH"], i)
    md.distances_file = member_distances_path(params["OUT_PATH"], i)
    md.loops_file = member_loops_path(params["OUT_PATH"], i)
    md.triplets_file = member_triplets_path(params["OUT_PATH"], i)
    md.timings["ingest_s"] = time.time() - t0
    return md


def member_contacts_path(out_path: str, i: int) -> str:
    return os.path.join(out_path, "contacts", f"member_{i}.npz")


def member_contacts_fine_path(out_path: str, i: int) -> str:
    return os.path.join(out_path, "contacts", f"member_{i}_fine.npz")


def member_distances_path(out_path: str, i: int) -> str:
    return os.path.join(out_path, "distances", f"member_{i}.npz")


def member_loops_path(out_path: str, i: int) -> str:
    return os.path.join(out_path, "loops", f"member_{i}.npz")


def member_triplets_path(out_path: str, i: int) -> str:
    return os.path.join(out_path, "triplets", f"member_{i}.npz")


def _sampled_md(args) -> bool:
    """The run writes trajectory maps (MD_SAMPLE_STEP with MD on)."""
    return bool(args.SIM_RUN_MD) and int(contact_setting(args, "MD_SAMPLE_STEP")) > 0


def write_ensemble_distances(args, results: list[dict]) -> str | None:
    """SAVE_DISTANCES: OUT_PATH/ensemble_distances.npz, the sum of the distance files of the members that
    succeeded (exact integer sums: the same bits whichever GPU ran which member); with MD_SAMPLE_STEP also
    ensemble_distances_md.npz, the sum of their trajectory maps."""
    if not contact_setting(args, "SAVE_DISTANCES") or not results:
        return None
    from . import contacts, distances

    out = None
    for md in (False, True) if _sampled_md(args) else (False,):
        name = contacts.md_path if md else (lambda p: p)
        paths = [name(member_distances_path(args.OUT_PATH, r["replica"]))
                 for r in sorted(results, key=lambda r: r["replica"])]
        agg = distances.aggregate(paths)
        path = name(os.path.join(args.OUT_PATH, "ensemble_distances.npz"))
        distances.save(path, agg)
        logger.info(f"ensemble distances{' (MD samples)' if md else ''}: {int(agg['members'])} "
                    f"{'structures' if md else 'members'}, {len(agg['bin_beads'])} bins at "
                    f"{int(agg['resolution_bp'])} bp -> {path}")
        out = out or path
    return out


def write_ensemble_loops(args, results: list[dict]) -> str | None:
    """SAVE_LOOPS: OUT_PATH/ensemble_loops.npz, the sum of the loops files of the members that succeeded (exact
    integer sums: the same bits whichever GPU ran which member); with MD_SAMPLE_STEP also ensemble_loops_md.npz,
    the sum of their MD samples."""
    if not contact_setting(args, "SAVE_LOOPS") or not results:
        return None
    from . import contacts, loops

    out = None
    for md in (False, True) if _sampled_md(args) else (False,):
        name = contacts.md_path if md else (lambda p: p)
        paths = [name(member_loops_path(args.OUT_PATH, r["replica"])) for r in sorted(results, key=lambda r: r["replica"])]
        agg = loops.aggregate(paths)
        path = name(os.path.join(args.OUT_PATH, "ensemble_loops.npz"))
        loops.save(path, agg)
        logger.info(f"ensemble loops{' (MD samples)' if md else ''}: {int(agg['members'])} structures, "
                    f"{len(agg['row'])} rows, APA window {int(agg['apa_window'])} beads -> {path}")
        out = out or path
    return out


def write_ensemble_triplets(args, results: list[dict]) -> str | None:
    """SAVE_TRIPLETS: OUT_PATH/ensemble_triplets.npz, the sum of the triplets files of the members that succeeded
    (exact integer sums: the same bits whichever GPU ran which member); with MD_SAMPLE_STEP also
    ensemble_triplets_md.npz, the sum of their MD samples."""
    if not contact_setting(args, "SAVE_TRIPLETS") or not results:
        return None
    from . import contacts, triplets

    out = None
    for md in (False, True) if _sampled_md(args) else (False,):
        name = contacts.md_path if md else (lambda p: p)
        paths = [name(member_triplets_path(args.OUT_PATH, r["replica"]))
                 for r in sorted(results, key=lambda r: r["replica"])]
        agg = triplets.aggregate(paths)
        path = name(os.path.join(args.OUT_PATH, "ensemble_triplets.npz"))
        triplets.save(path, agg)
        logger.info(f"ensemble three-way contacts{' (MD samples)' if md else ''}: {int(agg['members'])} structures, "
                    f"{int(agg['triples'])} triples, {len(agg['vals'])} entries -> {path}")
        out = out or path
    return out


def write_ensemble_contacts(args, results: list[dict]) -> str | None:
    """SAVE_CONTACTS: OUT_PATH/ensemble_contacts.npz, the sum of the contact files of the members that
    succeeded (exact integer sums: the same bits whichever GPU ran which member); with MD_SAMPLE_STEP also
    ensemble_contacts_md.npz (and _fine_md), the sum of their trajectory maps."""
    if not contact_setting(args, "SAVE_CONTACTS") or not results:
        return None
    from . import contacts

    out = None
    members = sorted(results, key=lambda r: r["replica"])
    for md in (False, True) if _sampled_md(args) else (False,):
        name = contacts.md_path if md else (lambda p: p)
        what, unit = (" (MD samples)", "structures") if md else ("", "members")
        paths = [name(member_contacts_path(args.OUT_PATH, r["replica"])) for r in members]
        agg = contacts.aggregate(paths)
        path = name(os.path.join(args.OUT_PATH, "ensemble_contacts.npz"))
        contacts.save_dense(path, agg)
        logger.info(f"ensemble contacts{what}: {int(agg['members'])} {unit}, {agg['counts'].shape[0]} bins at "
                    f"{int(agg['resolution_bp'])} bp, {int(agg['pairs'])} contacts (rc = {float(agg['radius_nm'])} nm) "
                    f"-> {path}")
        out = out or path
        if int(contact_setting(args, "CONTACT_FINE_RESOLUTION")) > 0:
            paths = [name(member_contacts_fine_path(args.OUT_PATH, r["replica"])) for r in members]
            fine = contacts.aggregate_fine(paths)
            out_fine = name(os.path.join(args.OUT_PATH, "ensemble_contacts_fine.npz"))
            contacts.save_fine(out_fine, fine)
            logger.info(f"ensemble fine contacts{what}: {int(fine['members'])} {unit}, {int(fine['n_bins'])} bins at "
                        f"{int(fine['resolution_bp'])} bp, {len(fine['vals'])} entries, {int(fine['pairs'])} contacts "
                        f"-> {out_fine}")
    return out


def prepare_replica(params: dict, i: int, run_path: str, device: int):
    """build_replica + MultiMM.prepare(): everything of member i that precedes its first force
    evaluation, in ONE task — __init__ seeds numpy's global random stream with the member's
    SHUFFLING_SEED and the random start curves of prepare() go on drawing from it, so nothing else that
    draws may come between the two (the pipelined driver runs these tasks one after another on one thread,
    and no other stage draws)."""
    t0 = time.time()
    md = build_replica(params, i, run_path, device)
    try:
        md.prepare()
    except BaseException:
        md.close()
        raise
    md.timings["prepare_s"] = time.time() - t0
    return md


def finish_replica(md, i: int, run_path: str, device: int, compute_s: float, archive: bool,
                   archiver: Archiver | None) -> dict:
    """Write-out of a computed member: structure files, reports, engine released, archive queued."""
    t0 = time.time()
    try:
        rep = md.finish()
    finally:
        md.close()
    finish_s = time.time() - t0
    prepare_s = md.timings.get("prepare_s", 0.0)
    out = dict(replica=i, device=device, seconds=prepare_s + compute_s + finish_s, compute_s=compute_s,
               finish_s=finish_s, **(rep or {}), **md.timings)
    if archive:
        t1 = time.time()
        if archiver is not None:
            archiver.submit(run_path)
            out["archive"] = run_path + ".tar.gz"
        else:
            out["archive"] = archive_run(run_path)
        out["archive_inline_s"] = time.time() - t1
    return out


def run_replica(params: dict, i: int, run_path: str, device: int, archive: bool = True, archiver: Archiver | None = None,
                prebuilt=None) -> dict:
    """One ensemble member from start to end on the calling thread (run.py:473-485).  With an `archiver`
    the tar.gz is written in the background (the report names the file it will be)."""
    md = prebuilt if prebuilt is not None else prepare_replica(params, i, run_path, device)
    t0 = time.time()
    try:
        md.compute()
    except BaseException:
        md.close()
        raise
    return finish_replica(md, i, run_path, device, time.time() - t0, archive, archiver)


def pipeline_enabled() -> bool:
    """MMM_ENSEMBLE_PIPELINE=0: every member runs from start to end on one thread (only the tar.gz of the
    previous member is written in the background)."""
    return os.environ.get("MMM_ENSEMBLE_PIPELINE", "1") != "0"


def run_replicas_on_device(params: dict, paths: list[str], todo, device: int, archive: bool, emit):
    """The replicas one GPU takes.  Three stages run side by side so that the GPU goes from one
    minimisation straight into the next: member k + 1 is PREPARED (inputs read, start structure and its
    files, engine, force field) on one background thread, member k COMPUTES (minimisation, MD) on the
    calling thread, member k - 1 is WRITTEN OUT (structure files, reports; then its tar.gz by the Archiver)
    on another.  pandas' parsers, file writes, gzip and every engine call release the GIL; the engine's
    graph capture is thread-local.  At most one member waits in each stage (bounded memory)."""
    from concurrent.futures import ThreadPoolExecutor

    archiver = Archiver() if archive else None
    if not pipeline_enabled():
        try:
            for i in todo:
                try:
                    emit(("ok", run_replica(params, i, paths[i], device, archive, archiver)))
                except Exception as e:  # report and keep going with the next replica
                    emit(("error", dict(replica=i, device=device, error=f"{type(e).__name__}: {e}")))
        finally:
            _wait_archiver(archiver, emit, device)
        return

    prep = ThreadPoolExecutor(max_workers=1, thread_name_prefix="mmm-prepare")
    fin = ThreadPoolExecutor(max_workers=1, thread_name_prefix="mmm-finish")
    it = iter(todo)

    def start_next():
        i = next(it, None)
        return None if i is None else (i, prep.submit(prepare_replica, params, i, paths[i], device))

    def finish_and_emit(md, i, compute_s):
        try:
            emit(("ok", finish_replica(md, i, paths[i], device, compute_s, archive, archiver)))
        except Exception as e:
            emit(("error", dict(replica=i, device=device, error=f"{type(e).__name__}: {e}")))

    finishing = None
    try:
        pending = start_next()
        while pending is not None:
            i, fut = pending
            try:
                md = fut.result()
            except Exception as e:
                pending = start_next()
                emit(("error", dict(replica=i, device=device, error=f"{type(e).__name__}: {e}")))
                continue
            pending = start_next()  # member k + 1 is prepared while member k computes
            t0 = time.time()
            try:
                md.compute()
            except Exception as e:  # report and keep going with the next replica
                md.close()
                emit(("error", dict(replica=i, device=device, error=f"{type(e).__name__}: {e}")))
                continue
            if finishing is not None:
                finishing.result()  # never more than one member behind
            finishing = fin.submit(finish_and_emit, md, i, time.time() - t0)
    finally:
        if finishing is not None:
            finishing.result()
        prep.shutdown(wait=True)
        fin.shutdown(wait=True)
        _wait_archiver(archiver, emit, device)


def _wait_archiver(archiver, emit, device):
    if archiver is None:
        return
    try:
        archiver.wait()
    except Exception as e:
        emit(("error", dict(replica=-1, device=device, error=f"archive failed: {type(e).__name__}: {e}")))


def _take(todo_queue):
    """Replica indices from the shared queue until it is empty."""
    import queue as _q

    while True:
        try:
            yield todo_queue.get(timeout=1.0)  # (not get_nowait: the parent's feeder thread may still be flushing)
        except _q.Empty:
            return


def worker_environment(device: int, base: dict | None = None) -> tuple[dict, int]:
    """Environment of the worker process that drives GPU `device`, and the device index it will use.
    One GPU per worker: with only its own device visible, CUDA initialisation does not touch the other
    seven.  The restriction is exported by the PARENT before the worker starts (run_ensemble), because the
    worker begins to initialise CUDA while it is still importing (_early_cuda_start)."""
    env = dict(os.environ if base is None else base)
    visible = env.get("CUDA_VISIBLE_DEVICES")
    local = 0
    if visible is None:
        env["CUDA_VISIBLE_DEVICES"] = str(device)
    else:  # the parent already runs under a restriction: `device` indexes into it
        ids = [t for t in visible.split(",") if t.strip()]
        if device < len(ids):
            env["CUDA_VISIBLE_DEVICES"] = ids[device]
        else:
            local = device  # nothing sensible to narrow to: let mmm_create report it
    # MMM_NO_EARLY_CUDA=1 switches the early start off (A/B timing)
    env["MMM_WORKER_WARMUP"] = "1" if local == 0 and os.environ.get("MMM_NO_EARLY_CUDA") != "1" else "0"
    env["MMM_WORKER_LOCAL_DEVICE"] = str(local)
    return env, local


def _worker(params: dict, paths: list[str], todo_queue, device: int, archive: bool, queue):
    # the parent exported this worker's CUDA_VISIBLE_DEVICES (worker_environment); a worker started by
    # other means narrows the visible devices itself, before anything has touched CUDA
    if "MMM_WORKER_LOCAL_DEVICE" in os.environ:
        local = int(os.environ["MMM_WORKER_LOCAL_DEVICE"])
    else:
        env, local = worker_environment(device)
        os.environ["CUDA_VISIBLE_DEVICES"] = env["CUDA_VISIBLE_DEVICES"]

    def emit(msg):
        kind, payload = msg
        if isinstance(payload, dict) and "device" in payload:
            payload["device"] = device  # the physical index, not the worker's local 0
        queue.put((kind, payload))

    run_replicas_on_device(params, paths, _take(todo_queue), local, archive, emit)


def run_ensemble(args, devices: list[int] | None = None, archive: bool = True) -> list[dict]:
    """All N_ENSEMBLE members; returns one report per replica, ordered by replica index."""
    n = int(args.N_ENSEMBLE or 0)
    if n <= 0:
        raise ValueError("GENERATE_ENSEMBLE is set but N_ENSEMBLE is not a positive integer")
    if not devices:
        devices = visible_devices(args)
    params = {k: v for k, v in args.model_dump().items()}
    paths = replica_paths(args.OUT_PATH, n)
    if len(devices) == 1:
        got = []
        run_replicas_on_device(params, paths, list(range(n)), devices[0], archive, got.append)
        errors = [p for kind, p in got if kind != "ok"]
        results = [p for kind, p in got if kind == "ok"]
        write_ensemble_contacts(args, results)
        write_ensemble_distances(args, results)
        write_ensemble_loops(args, results)
        write_ensemble_triplets(args, results)
        if errors:
            raise RuntimeError(f"{len(errors)} ensemble member(s) failed: {errors}")
        check_archives(results)
        return results
    ctx = mp.get_context("spawn")  # CUDA contexts must not be forked
    queue = ctx.Queue()
    todo_queue = ctx.Queue()
    for i in range(n):
        todo_queue.put(i)
    procs = [ctx.Process(target=_worker, args=(params, paths, todo_queue, dev, archive, queue))
             for dev in devices[:n]]
    # a spawned child inherits os.environ as it is at start(): export each worker's own restriction
    # (and the early CUDA start) around its start, then put the parent's environment back
    keys = ("CUDA_VISIBLE_DEVICES", "MMM_WORKER_WARMUP", "MMM_WORKER_LOCAL_DEVICE")
    saved = {k: os.environ.get(k) for k in keys}
    try:
        for p, dev in zip(procs, devices[:n]):
            env, _ = worker_environment(dev, base={k: v for k, v in saved.items() if v is not None})
            for k in keys:
                os.environ[k] = env[k]
            p.start()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    try:
        results, errors = collect_reports(procs, queue, n)
    finally:
        for p in procs:
            p.join(timeout=900)  # workers exit by themselves once their replicas are reported and archived
            if p.is_alive():
                p.terminate()  # exact processes we started
                p.join()
    write_ensemble_contacts(args, [r for r in results if r.get("replica", -1) >= 0])
    write_ensemble_distances(args, [r for r in results if r.get("replica", -1) >= 0])
    write_ensemble_loops(args, [r for r in results if r.get("replica", -1) >= 0])
    write_ensemble_triplets(args, [r for r in results if r.get("replica", -1) >= 0])
    if errors:
        raise RuntimeError(f"{len(errors)} ensemble member(s) failed: {errors}")
    check_archives(results)
    return sorted(results, key=lambda r: r["replica"])


def check_archives(results: list[dict]):
    """Archives are written in the background: once the workers are done every tarball must exist and
    be non-empty (archive_run keeps the run directory otherwise, run.py:436-443)."""
    bad = [r["archive"] for r in results if "archive" in r and not (os.path.exists(r["archive"]) and os.path.getsize(r["archive"]) > 0)]
    if bad:
        raise RuntimeError(f"archive(s) missing after the ensemble finished: {bad}")


def collect_reports(procs, queue, n: int, poll_seconds: float = 2.0):
    """Gather one report per replica from the workers.  A worker that dies without reporting
    (killed, crashed inside native code) must not leave the parent waiting forever: when every worker
    has exited and the queue is drained, the missing replicas are reported as failed."""
    import queue as _q

    results, errors = [], []
    while len(results) + len(errors) < n:
        try:
            kind, payload = queue.get(timeout=poll_seconds)
        except _q.Empty:
            if any(p.is_alive() for p in procs):
                continue
            try:  # the workers are gone: one last look at what they left behind
                kind, payload = queue.get(timeout=poll_seconds)
            except _q.Empty:
                seen = {r["replica"] for r in results} | {e["replica"] for e in errors}
                codes = [p.exitcode for p in procs]
                errors.extend(dict(replica=i, error=f"worker exited without a report (exit codes {codes})")
                              for i in range(n) if i not in seen)
                break
        (results if kind == "ok" else errors).append(payload)
    return results, errors


def visible_devices(args) -> list[int]:
    dev = str(getattr(args, "DEVICE", "") or "").strip()
    if dev.isdigit():
        return [int(dev)]
    if args.GENERATE_ENSEMBLE:
        try:
            import torch

            n = torch.cuda.device_count()
        except Exception:
            n = 0
        return list(range(n)) if n > 0 else [0]
    return [0]


def main(argv=None) -> int:
    try:
        args, gpus = get_config(argv)
        args_tests(args)
        log_dir = os.path.join(args.OUT_PATH, "metadata")
        os.makedirs(log_dir, exist_ok=True)
        with open(os.path.join(log_dir, "output.log"), "w") as log_file:
            out, err = sys.stdout, sys.stderr
            sys.stdout, sys.stderr = Tee(out, log_file), Tee(err, log_file)
            try:
                devices = [int(t) for t in gpus.split(",")] if gpus else visible_devices(args)
                if args.GENERATE_ENSEMBLE:
                    t0 = time.time()
                    reports = run_ensemble(args, devices)
                    dt = time.time() - t0
                    print(f"ensemble of {len(reports)} structures on {len(devices)} GPU(s) in {dt:.1f} s "
                          f"({3600.0 * len(reports) / dt:.1f} structures/hour)")
                else:
                    from .model import MultiMM

                    md = MultiMM(args, device=devices[0])
                    try:
                        md.run()
                    finally:
                        md.close()
            finally:
                sys.stdout, sys.stderr = out, err
        return 0
    except Exception as e:
        logger.error(f"ERROR: {e}")
        return 1


if __name__ == "__main__":
    sys.exit(main())
