"""MultiMM — the model driver, mirroring ``class MultiMM`` of the reference
(src/multimm/model.py:24-1248) method for method on the minimisation path:

    set_radiuses -> initialize_simulation -> add_forcefield (ten add_*) -> min_energy
    -> save_chromosomes

Everything that was an OpenMM object is now one ``Engine`` handle on a B200: the ``add_*``
methods pack the same parameters, read from the same config fields, into bulk C-ABI calls
(one call per term instead of one SWIG call per particle), ``min_energy`` runs the on-device
L-BFGS, ``run_md`` the on-device integrators, and the structure files are written in the reference's
formats.  Out of scope here (see DESIGN.md): plots, nucleosome interpolation.
"""
from __future__ import annotations

import logging
import os
import time

import numpy as np

from . import _lib, analysis, cif, loaders, structures
from .config import contact_setting
from .engine import Engine
from .units import Quantity

logger = logging.getLogger(__name__)


def _is_empty(val) -> bool:
    return val is None or str(val).strip() == "" or str(val).lower() == "none"


def _f(v) -> float:
    """Config value -> float in MD units (Quantity or bare float, model.py:176-179)."""
    return v.md if isinstance(v, Quantity) else float(v)


def backbone_bonds(n: int, chr_ends) -> np.ndarray:
    """Start indices i of the bonds (i, i+1): every i in [0, N-2] that is not in chr_ends
    (model.py:628-635).  Bond (0,1) and each (e_k, e_k+1) are absent; (e_k-1, e_k) joins
    consecutive chromosomes."""
    i = np.arange(n - 1)
    return i[~np.isin(i, np.asarray(chr_ends))].astype(np.int32)


def backbone_angles(n: int, chr_ends) -> np.ndarray:
    """Start indices i of the angles (i, i+1, i+2): i in [0, N-3], i not in chr_ends and not in
    chr_ends - 1 (model.py:711-719)."""
    ce = np.asarray(chr_ends)
    i = np.arange(n - 2)
    return i[~np.isin(i, ce) & ~np.isin(i, ce - 1)].astype(np.int32)


OPENMM_PLATFORMS = ("CUDA", "OPENCL", "CPU", "REFERENCE", "HIP")


def resolve_platform(name) -> str:
    """"B200", or an OpenMM platform name (taken as a preference, like model.py:862-871) -> "B200";
    anything else is a ValueError.  Called by run.args_tests too, so that a bad value fails before any I/O."""
    p = str(name).strip().upper()
    if p == "B200" or p in OPENMM_PLATFORMS:
        return "B200"
    raise ValueError(f"PLATFORM={name!r} is neither B200 nor an OpenMM platform name "
                     f"({', '.join(OPENMM_PLATFORMS)}); this engine runs on a B200 only")


class MultiMM:
    # the loop readout (SAVE_LOOPS): the loop table and how this member measures it (built in __init__ from the
    # loader's inputs), the sums of the minimised structure and of the MD samples, and where finish() writes
    # them (the ensemble driver points loops_file outside run_<i>)
    loop_table = loop_rows = loops = loops_md = loops_file = None
    # the three-way contact map (SAVE_TRIPLETS): the sums of the minimised structure and of the MD samples, and
    # where finish() writes them (the ensemble driver points triplets_file outside run_<i>)
    triplets = triplets_md = triplets_file = None
    # the locus dynamics of the MD samples (SAVE_DYNAMICS) and where finish() writes them (the ensemble driver
    # points dynamics_file outside run_<i>)
    dynamics = dynamics_file = None
    # the distance histograms (SAVE_DISTANCE_HIST): the counts of the minimised structure and of the MD samples,
    # and where finish() writes them (the ensemble driver points distance_hist_file outside run_<i>)
    distance_hist = distance_hist_md = distance_hist_file = None
    # GAM co-segregation (SAVE_GAM): the sums of the minimised structure and of the MD samples, and where finish()
    # writes them (the ensemble driver points gam_file outside run_<i>)
    gam = gam_md = gam_file = None

    def __init__(self, args, device: int | None = None):
        self.args = args
        self.ms = self.ns = self.ds = self.chr_ends = self.Cs = None
        self.chrom_idxs = None
        self.engine: Engine | None = None
        self.report: dict | None = None
        self.timings: dict = {}
        if device is None:
            device = int(args.DEVICE) if str(getattr(args, "DEVICE", "")).strip().isdigit() else 0
        self.device = device

        if str(args.MODELLING_LEVEL or "").lower() == "gene" and not _is_empty(args.GENE_TSV) \
                and not os.path.exists(args.GENE_TSV):
            # before the output tree is made or any file is parsed (upstream ships the table as package data)
            raise ValueError(f"MODELLING_LEVEL=gene needs the gene annotation table, but GENE_TSV={args.GENE_TSV!r} "
                             "does not exist. The 4 MB hg38 table is not shipped with this package: point GENE_TSV "
                             "at MultiMM's src/multimm/data/hg38_gtf_annotations.tsv (any TSV with its columns).")
        # output tree (model.py:46-55)
        self.save_path = args.OUT_PATH + "/"
        for sub in ("md_frames", "plots", "metadata", "model"):
            os.makedirs(os.path.join(self.save_path, sub), exist_ok=True)
        self._whole = _is_empty(args.GENE_ID) and _is_empty(args.GENE_NAME) and args.LOC_START is None
        if self._whole:
            os.makedirs(os.path.join(self.save_path, "plots", "chromosomes"), exist_ok=True)
            os.makedirs(os.path.join(self.save_path, "model", "chromosomes"), exist_ok=True)

        chrom = None if _is_empty(args.CHROM) else args.CHROM
        coords = [args.LOC_START, args.LOC_END] if (args.LOC_START is not None and args.LOC_END is not None) else None
        if chrom is not None and coords is None and chrom in loaders.CHROM_SIZES:
            coords = [0, loaders.CHROM_SIZES[chrom]]

        # gene-level region (model.py:65-97)
        if args.GENE_TSV is not None and str(args.MODELLING_LEVEL).lower() == "gene":
            if not _is_empty(args.GENE_ID):
                chrom, coords, gene = loaders.get_gene_region(args.GENE_TSV, gene_id=args.GENE_ID,
                                                              window_size=args.GENE_WINDOW)
            elif not _is_empty(args.GENE_NAME):
                chrom, coords, gene = loaders.get_gene_region(args.GENE_TSV, gene_name=args.GENE_NAME,
                                                              window_size=args.GENE_WINDOW)
            else:
                raise ValueError("You did not provide gene name or ID.")
            span = coords[1] - coords[0]
            self.gene_start = ((gene[0] - coords[0]) * args.N_BEADS) // span
            self.gene_end = ((gene[1] - coords[0]) * args.N_BEADS) // span

        if args.COMPARTMENT_PATH:
            if not args.COMPARTMENT_PATH.lower().endswith(".bed"):
                raise ValueError("Compartments file should be in .bed format.")
            self.Cs, self.chr_ends, self.chrom_idxs = loaders.import_bed(
                bed_file=args.COMPARTMENT_PATH, N_beads=args.N_BEADS, chrom=chrom, coords=coords,
                save_path=self.save_path, shuffle=args.SHUFFLE_CHROMS, seed=args.SHUFFLING_SEED,
                flip_prob=args.COMPARTMENT_FLIP_PROB, noise_strength=args.COMPARTMENT_NOISE_STD)
        if not str(args.LOOPS_PATH).lower().endswith(".bedpe"):
            raise ValueError("You did not provide appropriate loop file. Loop .bedpe file is obligatory.")
        # chr_ends / chrom_idxs of the bed loader are overwritten here (appendix A, Q4); the loop loader's
        # bead-to-genome mapping is what places beads in genomic coordinates (contacts.genome_bins)
        self.layout = {}
        self.ms, self.ns, self.ds, self.chr_ends, self.chrom_idxs = loaders.import_mns_from_bedpe(
            bedpe_file=args.LOOPS_PATH, N_beads=args.N_BEADS, coords=coords, chrom=chrom, path=self.save_path,
            shuffle=args.SHUFFLE_CHROMS, seed=args.SHUFFLING_SEED, down_prob=args.DOWNSAMPLING_PROB,
            layout=self.layout)
        self.contacts = None        # counts of the minimised structure (SAVE_CONTACTS)
        self.contacts_file = None   # where finish() writes them; the ensemble driver points it outside run_<i>
        self.contacts_fine = None   # sparse map of the same contacts (CONTACT_FINE_RESOLUTION)
        self.contacts_fine_file = None
        self.distances = None       # distance sums of the minimised structure (SAVE_DISTANCES)
        self.distances_file = None  # where finish() writes them; the ensemble driver points it outside run_<i>
        # the same maps summed over the structures sampled during MD (MD_SAMPLE_STEP); written beside the
        # files above, named by contacts.md_path
        self.contacts_md = self.contacts_fine_md = self.distances_md = None
        if contact_setting(args, "SAVE_LOOPS") or contact_setting(args, "SAVE_DYNAMICS"):
            from . import loops

            self.loop_table = loops.table(args.LOOPS_PATH, chrom, coords)
            self.loop_rows = loops.member_rows(self.loop_table, self.layout, args.N_BEADS, self.ms, self.ns, chrom)

        # chrom_spin: chromosome id per bead; chrom_strength: indexed by POSITION in the (possibly
        # shuffled) order, not by chromosome id (model.py:158-162; appendix A, Q8)
        n = args.N_BEADS
        self.chrom_spin, self.chrom_strength = np.zeros(n), np.zeros(n)
        if _is_empty(args.CHROM):
            for k in range(len(self.chr_ends) - 1):
                self.chrom_spin[self.chr_ends[k]:self.chr_ends[k + 1]] = self.chrom_idxs[k]
                self.chrom_strength[self.chr_ends[k]:self.chr_ends[k + 1]] = loaders.CHROM_STRENGTH[k]

    # ------------------------------------------------------------------------------------------
    def set_radiuses(self):
        """model.py:1016-1067: R2 = b0 N^(1/3), R1 = R2 * 0.2^(1/3), r_comp = 1.5 b0."""
        b0 = _f(self.args.POL_HARMONIC_BOND_R0)
        n = float(self.args.N_BEADS)
        self.radius2 = b0 * n ** (1.0 / 3.0)
        self.radius1 = self.radius2 * 0.20 ** (1.0 / 3.0)
        self.r_comp = 1.5 * b0
        logger.info(f"[Radiuses] b0={b0:.4f} nm | N={n:.0f} | R1={self.radius1:.4f} nm | "
                    f"R2={self.radius2:.4f} nm | r_comp={self.r_comp:.4f} nm")

    def initialize_simulation(self):
        """model.py:722-810: start structure -> init CIF -> positions (nm) -> mass centre -> system."""
        a = self.args
        # PLATFORM is a preference in the reference (model.py:862-871 falls back when the named
        # platform is unavailable); every config.ini it ships says OpenCL, its default is CPU.  Here
        # every OpenMM platform name maps to the one backend there is; nothing ever runs on the CPU.
        platform = resolve_platform(a.PLATFORM)
        if platform != str(a.PLATFORM):
            logger.warning(f"PLATFORM={a.PLATFORM!r} is an OpenMM platform name; running on the B200 engine "
                           "(the only backend; there is no CPU/OpenCL/Reference path)")
        t0 = time.time()
        self.engine = Engine(a.N_BEADS, device=self.device)
        init_cif = self.save_path + "metadata/MultiMM_init.cif"
        on_device = False
        if a.BUILD_INITIAL_STRUCTURE:
            pts = structures.compute_init_struct(a.N_BEADS, a.INITIAL_STRUCTURE_TYPE, engine=self.engine)
            cif.write_mmcif(pts, self.chr_ends, init_cif, hetatm_ends=True, connections=True, decimals=3)
            cif.write_psf(a.N_BEADS, self.save_path + "metadata/MultiMM.psf")
            # what PDBxFile would read back: the %.3f text, Angstrom -> nm.  Lattice points are
            # integers, so the text is exact and the file need not be parsed again.
            if getattr(a.INITIAL_STRUCTURE_TYPE, "value", a.INITIAL_STRUCTURE_TYPE) == "hilbert":
                self.positions = pts * 0.1
                self.engine.hilbert_init(8, 0.1)  # positions written in place on the device
                on_device = True
            else:
                self.positions = cif.read_cif_coordinates(init_cif, include_hetatm=True) / 10.0
        else:
            path = init_cif if _is_empty(a.INITIAL_STRUCTURE_PATH) else a.INITIAL_STRUCTURE_PATH
            self.positions = cif.read_cif_coordinates(path, include_hetatm=True) / 10.0
            if len(self.positions) != a.N_BEADS:
                raise ValueError(f"{path} holds {len(self.positions)} beads, N_BEADS is {a.N_BEADS}")
        self.mass_center = np.average(self.positions, axis=0)  # model.py:759
        if not on_device:
            self.engine.set_positions(self.positions)
        self.timings["initialize_s"] = time.time() - t0

    # -- the ten add_* methods (model.py:164-720) -----------------------------------------------
    def _form(self, table, field, default, what):
        mode = getattr(self.args, field, default)
        if mode not in table:
            raise ValueError(f"Unknown {what}: {mode}")
        return table[mode]

    def add_evforce(self):
        a = self.args
        form = self._form(_lib.EV_FORMS, "EV_FORCE_TYPE", "powerlaw", "EV_FORCE_TYPE")
        sigma = _f(a.LE_HARMONIC_BOND_R0)  # sigma is the LOOP bond length (model.py:175; appendix A, Q7)
        self.engine.set_pair_term("EV", form, [a.EV_EPSILON, a.EV_R_SMALL, sigma, a.EV_POWER])

    def add_compartment_blocks(self):
        form = self._form(_lib.BLOCK_FORMS, "COB_FORCE_TYPE", "gaussian", "COB_FORCE_TYPE")
        self.engine.set_pair_term("COB", form, [self.r_comp, self.args.COB_EA, self.args.COB_EB])

    def add_subcompartment_blocks(self):
        a = self.args
        form = self._form(_lib.BLOCK_FORMS, "SCB_FORCE_TYPE", "gaussian", "SCB_FORCE_TYPE")
        self.engine.set_pair_term("SCB", form, [self.r_comp, a.SCB_EA1, a.SCB_EA2, a.SCB_EB1, a.SCB_EB2])

    def add_chromosomal_blocks(self):
        form = self._form(_lib.CHB_FORMS, "CHB_FORCE_TYPE", "polynomial", "CHB_FORCE_TYPE")
        self.engine.set_pair_term("CHB", form, [self.args.CHB_KC, self.args.CHB_DE])

    def add_spherical_container(self):
        self.engine.set_external_term("SC", 0, [self.args.SC_SCALE, self.radius1, self.radius2, *self.mass_center])

    def add_Blamina_interaction(self):
        form = self._form(_lib.LAM_FORMS, "BLAMINA_FORCE_TYPE", "sin", "BLAMINA_FORCE_TYPE")
        self.engine.set_external_term("LAM", form, [self.args.IBL_SCALE, self.radius1, self.radius2,
                                                    *self.mass_center])

    def add_central_force(self):
        form = self._form(_lib.CF_FORMS, "CENTRAL_FORCE_TYPE", "harmonic", "CENTRAL_FORCE_TYPE")
        self.engine.set_external_term("CF", form, [self.args.CF_STRENGTH, self.radius1, *self.mass_center])

    def add_harmonic_bonds(self):
        a = self.args
        i = backbone_bonds(a.N_BEADS, self.chr_ends)
        self.engine.set_bonds(i, i + 1, _f(a.POL_HARMONIC_BOND_R0), _f(a.POL_HARMONIC_BOND_K))
        self.n_bonds = len(i)

    def add_loops(self):
        a = self.args
        mode = getattr(a, "LE_LOOP_FORCE_TYPE", "harmonic")
        if mode not in _lib.LOOP_FORMS:
            raise ValueError(f"Unknown loop force type: {mode}")
        # r0 is the fixed loop length or ds[i] taken as nm (model.py:656-659)
        r0 = np.full(len(self.ms), _f(a.LE_HARMONIC_BOND_R0)) if a.LE_FIXED_DISTANCES else np.asarray(self.ds, float)
        self.engine.set_loops(self.ms, self.ns, r0, _f(a.LE_HARMONIC_BOND_K), form=_lib.LOOP_FORMS[mode])

    def add_stiffness(self):
        a = self.args
        i = backbone_angles(a.N_BEADS, self.chr_ends)
        self.engine.set_angles(i, i + 1, i + 2, _f(a.POL_HARMONIC_ANGLE_R0), _f(a.POL_HARMONIC_ANGLE_CONSTANT_K))
        self.n_angles = len(i)

    def add_forcefield(self):
        """model.py:812-857: same gating, same order."""
        a = self.args
        t0 = time.time()
        n = a.N_BEADS
        s = np.zeros(n, dtype=np.int8) if self.Cs is None else np.asarray(self.Cs, dtype=np.int8)
        self.engine.set_bead_params(s, self.chrom_spin.astype(np.int32), self.chrom_strength)
        needs_cs = a.COB_USE_COMPARTMENT_BLOCKS or a.SCB_USE_SUBCOMPARTMENT_BLOCKS or a.IBL_USE_B_LAMINA_INTERACTION
        if needs_cs and self.Cs is None:
            raise ValueError("a compartment-dependent force is enabled but no COMPARTMENT_PATH was loaded")
        if a.EV_USE_EXCLUDED_VOLUME: self.add_evforce()
        if a.COB_USE_COMPARTMENT_BLOCKS: self.add_compartment_blocks()
        if a.SCB_USE_SUBCOMPARTMENT_BLOCKS: self.add_subcompartment_blocks()
        if a.CHB_USE_CHROMOSOMAL_BLOCKS: self.add_chromosomal_blocks()
        if a.SC_USE_SPHERICAL_CONTAINER: self.add_spherical_container()
        if a.IBL_USE_B_LAMINA_INTERACTION: self.add_Blamina_interaction()
        if a.CF_USE_CENTRAL_FORCE: self.add_central_force()
        if a.POL_USE_HARMONIC_BOND: self.add_harmonic_bonds()
        if a.LE_USE_HARMONIC_BOND: self.add_loops()
        if a.POL_USE_HARMONIC_ANGLE: self.add_stiffness()
        cutoff = float(getattr(a, "PAIR_CUTOFF", 0.0) or 0.0)
        if cutoff > 0:
            self.engine.set_cutoff(cutoff)
        self.timings["forcefield_s"] = time.time() - t0

    def _two_stage_minimize(self, tol: float, max_iter: int, coarse: float) -> dict:
        """Opt-in two-stage minimisation (MIN_COARSE_CUTOFF > 0; not in the reference).  L-BFGS on a cheap
        coarse potential — pair terms truncated at `coarse` nm, plus what truncation misses at long range
        (CHB's polynomial, the EV tail) evaluated between cluster centroids (MIN_COARSE_FAR_FIELD = exact:
        the exact same-chromosome pass for CHB and no tail) — gets close to a minimum at a fraction of the
        cost per evaluation; the SAME stopping rule is then met on the exact all-pairs potential, so the
        result satisfies exactly what minimizeEnergy() guarantees.

        The two potentials' minima are close but not equal.  Most replicas need 0-15 exact iterations after
        the coarse stage; some would need hundreds (measured: 10 of 64).  So the exact stage is first run as
        a PROBE of MIN_EXACT_PROBE_ITERATIONS; if that does not converge, the coarse stage goes on from there
        to a tighter tolerance (x 0.7 per round) and the exact probe is repeated; the last round's exact
        stage is unbounded (or bounded by MIN_MAX_ITERATIONS).  The coarse stage itself is bounded
        (MIN_COARSE_MAX_ITERATIONS): a truncated potential jumps at the cut-off, so L-BFGS on it is not
        guaranteed to reach a gradient tolerance."""
        a = self.args
        cap = int(getattr(a, "MIN_COARSE_MAX_ITERATIONS", 20000) or 20000)
        far = str(getattr(a, "MIN_COARSE_FAR_FIELD", "clusters")).lower() == "clusters"
        frac = min(max(float(getattr(a, "MIN_COARSE_TOLERANCE", 1.0) or 1.0), 0.05), 1.0)
        rounds = max(1, int(getattr(a, "MIN_COARSE_ROUNDS", 4) or 1))
        probe = max(1, int(getattr(a, "MIN_EXACT_PROBE_ITERATIONS", 30) or 30))
        c_it = c_ev = e_it = e_ev = 0
        c_s = 0.0
        rep = None
        self.coarse_report = None
        for r in range(rounds):
            last = r == rounds - 1
            self.engine.set_cutoff(coarse)
            self.engine.set_chb_surrogate(far)
            rep_c = self.engine.minimize(tol=tol * frac, max_iter=min(max_iter, cap) if max_iter > 0 else cap)
            self.engine.set_cutoff(0.0)
            self.engine.set_chb_surrogate(False)
            self.coarse_report = rep_c if self.coarse_report is None else self.coarse_report
            c_it += int(rep_c["iterations"]); c_ev += int(rep_c["evaluations"]); c_s += float(rep_c["wall_seconds"])
            bound = max_iter if last else (min(probe, max_iter) if max_iter > 0 else probe)
            rep = self.engine.minimize(tol=tol, max_iter=bound)
            e_it += int(rep["iterations"]); e_ev += int(rep["evaluations"])
            if rep["converged"] or rep["ls_status"] != 0:
                break
            frac *= 0.7
        self.timings["coarse_iterations"], self.timings["coarse_evaluations"] = c_it, c_ev
        self.timings["coarse_seconds"] = c_s
        self.timings["coarse_rounds"] = r + 1
        self.timings["exact_iterations"], self.timings["exact_evaluations"] = e_it, e_ev
        return rep

    def min_energy(self, write_files: bool = True):
        """model.py:859-897: minimise with OpenMM's defaults (10 kJ/mol/nm, unlimited iterations)
        and write model/MultiMM_minimized.cif (Angstrom).  write_files False: the file is left to
        write_minimized() (the ensemble driver writes it while the next member minimises)."""
        a = self.args
        t0 = time.time()
        tol, max_iter = float(getattr(a, "MIN_TOLERANCE", 10.0)), int(getattr(a, "MIN_MAX_ITERATIONS", 0))
        coarse = float(getattr(a, "MIN_COARSE_CUTOFF", 0.0) or 0.0)
        final_cutoff = float(getattr(a, "PAIR_CUTOFF", 0.0) or 0.0)
        self.coarse_report = None
        if final_cutoff > 0.0 and max_iter == 0:
            # a truncated potential jumps at the cut-off: unlimited iterations could go on for ever
            max_iter = int(getattr(a, "MIN_COARSE_MAX_ITERATIONS", 20000) or 20000)
            logger.warning(f"PAIR_CUTOFF > 0 with unlimited iterations: bounded at {max_iter} L-BFGS iterations")
        if coarse > 0.0 and final_cutoff == 0.0:
            self.report = self._two_stage_minimize(tol, max_iter, coarse)
        else:
            self.report = self.engine.minimize(tol=tol, max_iter=max_iter)
        self.positions = self.engine.get_positions()
        self.positions_minimized = self.positions
        self.timings["minimize_s"] = time.time() - t0
        if write_files:
            self.write_minimized()
        dt = time.time() - t0
        logger.info(f"--- Energy minimization done!! Executed in {dt // 3600:.0f} hours, {dt % 3600 // 60:.0f} "
                    f"minutes and  {dt % 60:.0f} seconds. :D --- {self.report}")

    def write_minimized(self):
        """model/MultiMM_minimized.cif (model.py:889-896), Angstrom."""
        t1 = time.time()
        cif.write_mmcif(10.0 * self.positions_minimized, self.chr_ends, self.save_path + "model/MultiMM_minimized.cif",
                        hetatm_ends=True, connections=False, decimals=4)
        self.timings["write_cif_s"] = time.time() - t1

    def run_md(self):
        """model.py:907-995: relaxation with the configured integrator, a thermodynamic record every
        SIM_SAMPLING_STEP steps (printed like OpenMM's StateDataReporter), a CIF per sample in
        md_frames/, a DCD every SIM_N_STEPS // TRJ_FRAMES steps, model/MultiMM_afterMD.cif at the end."""
        a = self.args
        kind = str(a.SIM_INTEGRATOR_TYPE).lower()
        if kind not in _lib.MD_INTEGRATORS:
            raise ValueError(f"SIM_INTEGRATOR_TYPE={a.SIM_INTEGRATOR_TYPE!r} is not available "
                             f"(supported: {', '.join(_lib.MD_INTEGRATORS)})")
        dt = _f(a.SIM_INTEGRATOR_STEP)  # ps
        temp = _f(a.SIM_TEMPERATURE)
        seed = int(a.SHUFFLING_SEED)
        self.engine.md_configure(kind, dt, temp, float(a.SIM_FRICTION_COEFF), loaders.BEAD_MASS, seed,
                                 amd_alpha=_f(a.SIM_AMD_ALPHA), amd_e=_f(a.SIM_AMD_E))  # model.py:796-800
        self.engine.set_velocities_to_temperature(temp, seed)  # model.py:878
        self.md_history = {"step": [], "potential": [], "kinetic": [], "total": [], "temperature": []}
        n_steps, every = int(a.SIM_N_STEPS), max(1, int(a.SIM_SAMPLING_STEP))
        dcd_every = max(1, n_steps // max(1, int(a.TRJ_FRAMES)))
        dcd = cif.DCDWriter(self.save_path + "metadata/MultiMM_annealing.dcd", a.N_BEADS, dt, dcd_every)
        sample_every = int(contact_setting(a, "MD_SAMPLE_STEP"))
        maps = contact_setting(a, "SAVE_CONTACTS") or contact_setting(a, "SAVE_DISTANCES")
        sampling = self._configure_sampler() if sample_every > 0 and maps else None
        loop_sampling = sample_every > 0 and bool(contact_setting(a, "SAVE_LOOPS"))
        if loop_sampling:
            self._configure_loops()
        triplet_sampling = sample_every > 0 and bool(contact_setting(a, "SAVE_TRIPLETS"))
        tb = self._configure_triplets() if triplet_sampling else None
        dyn = self._configure_dynamics() if sample_every > 0 and contact_setting(a, "SAVE_DYNAMICS") else None
        hist_sampling = sample_every > 0 and bool(contact_setting(a, "SAVE_DISTANCE_HIST"))
        hb = self._configure_distance_hist() if hist_sampling else None
        gam_sampling = sample_every > 0 and bool(contact_setting(a, "SAVE_GAM"))
        gg = self._configure_gam() if gam_sampling else None
        chunk = int(np.gcd.reduce([every, dcd_every] +
                                  ([sample_every] if sampling or loop_sampling or triplet_sampling or dyn or hist_sampling
                                   or gam_sampling else [])))
        t0 = time.time()
        print('#"Step"\t"Potential Energy (kJ/mole)"\t"Kinetic Energy (kJ/mole)"\t"Total Energy (kJ/mole)"\t"Temperature (K)"')
        done = 0
        try:
            while done < (n_steps // every) * every:
                done += chunk
                want_frame, want_dcd = done % every == 0, done % dcd_every == 0
                # energies (one more force evaluation and a host read) only where a sample is recorded
                rep = self.engine.md_run(chunk, want_report=want_frame)
                if want_frame or want_dcd:
                    self.positions = self.engine.get_positions()
                if want_dcd:
                    dcd.write(10.0 * self.positions)
                if want_frame:
                    h = self.md_history
                    h["step"].append(done); h["potential"].append(rep["potential"]); h["kinetic"].append(rep["kinetic"])
                    h["total"].append(rep["potential"] + rep["kinetic"]); h["temperature"].append(rep["temperature"])
                    print(f"{done}\t{rep['potential']}\t{rep['kinetic']}\t{rep['potential'] + rep['kinetic']}\t{rep['temperature']}")
                    cif.write_mmcif(10.0 * self.positions, self.chr_ends,
                                    self.save_path + f"md_frames/frame_{done // every}.cif", hetatm_ends=True,
                                    connections=False, decimals=4)
                if sampling and done % sample_every == 0:
                    self._sample(sampling)
                if loop_sampling and done % sample_every == 0:
                    self.engine.loops_add()
                if triplet_sampling and done % sample_every == 0:
                    self.engine.triplets_add()
                if dyn and done % sample_every == 0:
                    self.engine.dynamics_add()
                if hist_sampling and done % sample_every == 0:
                    self.engine.disthist_add()
                if gam_sampling and done % sample_every == 0:
                    self._gam_add(gg, done // sample_every)
        finally:
            dcd.close()
        if sampling:
            self._read_samples(sampling, sample_every)
        if loop_sampling:
            self._read_loops(md=True)
        if triplet_sampling:
            self._read_triplets(tb, md=True)
        if dyn:
            self._read_dynamics(dyn, sample_every)
        if hist_sampling:
            self._read_distance_hist(hb, md=True)
        if gam_sampling:
            self._read_gam(gg, md=True)
        self.positions = self.engine.get_positions()
        cif.write_mmcif(10.0 * self.positions, self.chr_ends, self.save_path + "model/MultiMM_afterMD.cif",
                        hetatm_ends=True, connections=False, decimals=4)
        with open(self.save_path + "metadata/md_thermodynamics.tsv", "w") as fh:
            fh.write("step\tpotential\tkinetic\ttotal\ttemperature\n")
            for row in zip(*(self.md_history[k] for k in ("step", "potential", "kinetic", "total", "temperature"))):
                fh.write("\t".join(str(v) for v in row) + "\n")
        self.timings["md_s"] = time.time() - t0
        logger.info(f"MD finished in {self.timings['md_s']:.1f} s ({n_steps} steps, {kind})")

    def save_chromosomes(self):
        """model.py:899-905."""
        for k in range(len(self.chr_ends) - 1):
            name = loaders.CHROM_NAMES[int(self.chrom_idxs[k])]
            cif.write_mmcif_chrom(10.0 * self.positions_minimized[self.chr_ends[k]:self.chr_ends[k + 1]],
                                  self.save_path + f"model/chromosomes/MultiMM_minimized_{name}.cif")

    def make_reports(self):
        """The numeric part of make_plots (model.py:1069-1213): for single-chromosome / region runs
        the reference analyses the initial, minimised and post-MD structures (analyze_structure,
        plots.py:630-829); genome-wide runs return before that step.  Figures are not drawn here."""
        multi = self._whole and self.chrom_idxs is not None and len(self.chrom_idxs) > 1
        if multi:
            return
        todo = [("initial_structure", "metadata/MultiMM_init.cif"), ("minimized_structure", "model/MultiMM_minimized.cif")]
        if self.args.SIM_RUN_MD:
            todo.append(("structure_afterMD", "model/MultiMM_afterMD.cif"))
        for name, rel in todo:
            # get_coordinates_cif keeps ATOM rows only (utils.py:184-190), so V is shorter than N_BEADS
            # (the chromosome-end beads are HETATM): the device pass takes any number of rows
            V = cif.read_cif_coordinates(self.save_path + rel, include_hetatm=False)
            analysis.analyze_structure(V, self.save_path, name=name, device=self.device)

    def save_args_to_txt(self, filename):
        """utils.py:733-742."""
        with open(filename, "w") as f:
            for name, value in self.args.model_dump().items():
                if isinstance(value, Quantity):
                    f.write(f"{name} = {value._value} {value.unit.get_name()}\n")
                elif value is None:
                    f.write(f"{name} = \n")
                else:
                    f.write(f"{name} = {getattr(value, 'value', value)}\n")

    # run() = prepare() -> compute() -> finish() (model.py:1216-1248).  The split is what the ensemble
    # driver pipelines: member k + 1 is prepared and member k - 1 written out while member k computes.
    def prepare(self):
        """Everything up to the first force evaluation: radii, start structure and its files, the engine,
        the force field.  The only stage (besides __init__) that draws from numpy's global random stream
        (the random start curves), so it must follow the member's own __init__ with nothing in between."""
        self.set_radiuses()
        self.initialize_simulation()
        self.add_forcefield()

    def compute(self):
        """The GPU-bound stage: minimisation, MD relaxation if configured.  No structure files except MD's."""
        self.min_energy(write_files=False)
        if contact_setting(self.args, "SAVE_CONTACTS"):
            self.count_contacts()
        if contact_setting(self.args, "SAVE_DISTANCES"):
            self.count_distances()
        if contact_setting(self.args, "SAVE_LOOPS"):
            self.measure_loops()
        if contact_setting(self.args, "SAVE_TRIPLETS"):
            self.count_triplets()
        if contact_setting(self.args, "SAVE_DISTANCE_HIST"):
            self.count_distance_hist()
        if contact_setting(self.args, "SAVE_GAM"):
            self.count_gam()
        if self.args.SIM_RUN_MD:
            self.run_md()

    def _contact_bins(self, fine: bool = False):
        """Canonical bins of the contact map (fine: of the fine map, None when CONTACT_FINE_RESOLUTION is 0)."""
        from . import contacts

        a = self.args
        if not fine:
            return contacts.genome_bins(self.layout, int(contact_setting(a, "CONTACT_RESOLUTION")), n_beads=a.N_BEADS)
        fine_res = int(contact_setting(a, "CONTACT_FINE_RESOLUTION"))
        if fine_res <= 0:
            return None
        return contacts.genome_bins(self.layout, fine_res, n_beads=a.N_BEADS, max_bins=contacts.MAX_FINE_BINS)

    def _distance_bins(self):
        from . import contacts, distances

        res = int(contact_setting(self.args, "DISTANCE_RESOLUTION"))
        try:
            return contacts.genome_bins(self.layout, res, n_beads=self.args.N_BEADS, max_bins=distances.MAX_BINS)
        except ValueError as e:
            raise ValueError(f"DISTANCE_RESOLUTION={res}: {e}") from None

    def count_contacts(self):
        """Contacts of the minimised structure (SAVE_CONTACTS), counted by this member's own engine at the
        positions the minimisation left on the device, binned in canonical genomic coordinates."""
        from . import contacts

        t0 = time.time()
        a = self.args
        gb = self._contact_bins()
        rc = float(contact_setting(a, "CONTACT_RADIUS"))
        cmap, sep, pairs = self.engine.contacts(rc, gb.bins, gb.n_bins)
        self.contacts = contacts.result(cmap, sep, pairs, rc, gb, contacts.sep_pairs(self.chrom_spin))
        self.timings["contacts_s"] = time.time() - t0
        fb = self._contact_bins(fine=True)
        if fb is not None:
            t0 = time.time()
            rows, cols, vals, pairs = self.engine.contacts_sparse(rc, fb.bins, fb.n_bins)
            self.contacts_fine = contacts.fine_result(rows, cols, vals, pairs, rc, fb)
            self.timings["contacts_fine_s"] = time.time() - t0

    def count_distances(self):
        """Distance sums of the minimised structure (SAVE_DISTANCES): the all-pairs map summed by this member's
        own engine at the positions the minimisation left on the device, and the radial sums about the
        container centre on the host, binned in canonical genomic coordinates."""
        from . import contacts, distances

        t0 = time.time()
        gb = self._distance_bins()
        dsum, d2sum = self.engine.distance_map(gb.bins, gb.n_bins)
        self.distances = distances.result(dsum, d2sum, gb, self.engine.get_positions(), self.mass_center)
        self.timings["distances_s"] = time.time() - t0

    def _configure_loops(self):
        """Set up the engine's loop accumulator with this member's valid rows (SAVE_LOOPS)."""
        from . import loops

        a = self.args
        self.engine.loops_configure(float(contact_setting(a, "CONTACT_RADIUS")), int(contact_setting(a, "LOOP_APA_WINDOW")),
                                    **loops.device_rows(self.loop_rows))

    def _read_loops(self, md: bool = False):
        from . import loops

        a = self.args
        r = self.engine.loops_read()
        if md:
            logger.info(f"loop readout: {r['samples']} MD structures ({r['device_ms']:.1f} ms on the device)")
            if r["samples"] == 0:
                return
        d = loops.result(self.loop_table, self.loop_rows, r, float(contact_setting(a, "CONTACT_RADIUS")),
                         int(contact_setting(a, "LOOP_APA_WINDOW")), r["samples"])
        if md:
            self.loops_md = d
        else:
            self.loops = d

    def measure_loops(self):
        """The loop readout of the minimised structure (SAVE_LOOPS): per-row sums and APA of the rows of the loop
        table that are valid for this member, measured by its own engine at the positions the minimisation
        left on the device."""
        t0 = time.time()
        self._configure_loops()
        self.engine.loops_add()
        self._read_loops()
        self.timings["loops_s"] = time.time() - t0

    def _configure_triplets(self):
        """Set up the engine's three-way accumulator with the canonical bins of TRIPLET_RESOLUTION; returns them."""
        from . import contacts, triplets

        a = self.args
        res = int(contact_setting(a, "TRIPLET_RESOLUTION"))
        try:
            gb = contacts.genome_bins(self.layout, res, n_beads=a.N_BEADS, max_bins=triplets.MAX_BINS)
        except ValueError as e:
            raise ValueError(f"TRIPLET_RESOLUTION={res}: {e}") from None
        self.engine.triplets_configure(float(contact_setting(a, "CONTACT_RADIUS")), gb.bins, gb.n_bins)
        return gb

    def _read_triplets(self, gb, md: bool = False):
        from . import triplets

        r = self.engine.triplets_read()
        if md:
            logger.info(f"three-way contacts: {r['samples']} MD structures ({r['device_ms']:.1f} ms on the device)")
            if r["samples"] == 0:
                return
        d = triplets.result(r, float(contact_setting(self.args, "CONTACT_RADIUS")), gb, r["samples"])
        if md:
            self.triplets_md = d
        else:
            self.triplets = d

    def count_triplets(self):
        """Three-way contacts of the minimised structure (SAVE_TRIPLETS): bead triples in mutual contact,
        enumerated by this member's own engine at the positions the minimisation left on the device, binned in
        canonical genomic coordinates."""
        t0 = time.time()
        gb = self._configure_triplets()
        self.engine.triplets_add()
        self._read_triplets(gb)
        self.timings["triplets_s"] = time.time() - t0

    def _configure_distance_hist(self):
        """Set up the engine's distance-histogram accumulator with the canonical bins of DISTANCE_HIST_RESOLUTION
        and the edges of DISTANCE_HIST_EDGES; returns the bins and edges."""
        from . import contacts, disthist

        a = self.args
        edges = disthist.parse_edges(contact_setting(a, "DISTANCE_HIST_EDGES"))
        res = int(contact_setting(a, "DISTANCE_HIST_RESOLUTION"))
        try:
            gb = contacts.genome_bins(self.layout, res, n_beads=a.N_BEADS, max_bins=disthist.max_bins(len(edges)))
        except ValueError as e:
            raise ValueError(f"DISTANCE_HIST_RESOLUTION={res}: {e}") from None
        self.engine.disthist_configure(gb.bins, gb.n_bins, edges)
        return gb, edges

    def _read_distance_hist(self, hb, md: bool = False):
        from . import disthist

        gb, edges = hb
        r = self.engine.disthist_read()
        if md:
            logger.info(f"distance histograms: {r['samples']} MD structures ({r['device_ms']:.1f} ms on the device)")
            if r["samples"] == 0:
                return
        d = disthist.result(r["counts"], edges, gb, r["samples"])
        if md:
            self.distance_hist_md = d
        else:
            self.distance_hist = d

    def count_distance_hist(self):
        """Distance histograms of the minimised structure (SAVE_DISTANCE_HIST): every bead pair counted per bin
        pair and distance cell by this member's own engine at the positions the minimisation left on the device,
        binned in canonical genomic coordinates."""
        t0 = time.time()
        hb = self._configure_distance_hist()
        self.engine.disthist_add()
        self._read_distance_hist(hb)
        self.timings["distance_hist_s"] = time.time() - t0

    def _configure_gam(self):
        """Set up the engine's GAM accumulator with the canonical bins of GAM_RESOLUTION and room for GAM_SLICES
        slices per add; returns the bins."""
        from . import contacts, gam

        a = self.args
        res = int(contact_setting(a, "GAM_RESOLUTION"))
        try:
            gb = contacts.genome_bins(self.layout, res, n_beads=a.N_BEADS, max_bins=gam.MAX_BINS)
        except ValueError as e:
            raise ValueError(f"GAM_RESOLUTION={res}: {e}") from None
        self.engine.gam_configure(gb.bins, gb.n_bins, int(contact_setting(a, "GAM_SLICES")))
        return gb

    def _gam_add(self, gb, k: int):
        """Slice the structure on the device with GAM_SLICES random planes about the container centre, drawn from
        the private stream default_rng([SHUFFLING_SEED, k]) (k = 0: the minimised structure, k = s: MD sample s),
        never from numpy's global stream, whose order the ensemble driver keeps."""
        from . import gam

        a = self.args
        rng = np.random.default_rng([int(a.SHUFFLING_SEED), int(k)])
        planes, h = gam.slice_planes(self.engine.get_positions(), self.mass_center, gb.bins,
                                     int(contact_setting(a, "GAM_SLICES")), float(contact_setting(a, "GAM_SLICE_FRACTION")),
                                     rng)
        self.engine.gam_add(planes, h)

    def _read_gam(self, gb, md: bool = False):
        from . import gam

        r = self.engine.gam_read()
        if md:
            logger.info(f"GAM: {r['structures']} MD structures, {r['slices']} slices ({r['empty']} empty; "
                        f"{r['device_ms']:.1f} ms on the device)")
            if r["structures"] == 0:
                return
        d = gam.result(r, gb, float(contact_setting(self.args, "GAM_SLICE_FRACTION")))
        if md:
            self.gam_md = d
        else:
            self.gam = d

    def count_gam(self):
        """GAM co-segregation of the minimised structure (SAVE_GAM): GAM_SLICES random slices through the
        positions the minimisation left on the device, bins co-detected counted by this member's own engine in
        canonical genomic coordinates."""
        t0 = time.time()
        gb = self._configure_gam()
        self._gam_add(gb, 0)
        self._read_gam(gb)
        self.timings["gam_s"] = time.time() - t0

    def _configure_dynamics(self) -> dict:
        """SAVE_DYNAMICS: set up the engine's dynamics accumulator with the canonical bins of DYNAMICS_RESOLUTION,
        the lags 1, 2, ..., DYNAMICS_MAX_LAG and this member's valid loop rows.  Returns the bins and lags."""
        from . import contacts, dynamics, loops

        a = self.args
        res = int(contact_setting(a, "DYNAMICS_RESOLUTION"))
        try:
            gb = contacts.genome_bins(self.layout, res, n_beads=a.N_BEADS, max_bins=dynamics.MAX_BINS)
        except ValueError as e:
            raise ValueError(f"DYNAMICS_RESOLUTION={res}: {e}") from None
        lags = dynamics.lag_set(int(contact_setting(a, "DYNAMICS_MAX_LAG")))
        rows = loops.device_rows(self.loop_rows)
        self.engine.dynamics_configure(float(contact_setting(a, "CONTACT_RADIUS")), lags, gb.bins, gb.n_bins,
                                       rows["bead_lo"], rows["bead_hi"], rows["group"])
        return dict(gb=gb, lags=lags)

    def _read_dynamics(self, st: dict, sample_every: int):
        from . import dynamics

        a = self.args
        r = self.engine.dynamics_read()
        logger.info(f"locus dynamics: {r['samples']} MD structures, lags up to {int(st['lags'][-1])} samples "
                    f"({r['device_ms']:.1f} ms on the device)")
        self.dynamics = dynamics.result(r, st["lags"], st["gb"], self.loop_table, self.loop_rows,
                                        float(contact_setting(a, "CONTACT_RADIUS")), sample_every,
                                        _f(a.SIM_INTEGRATOR_STEP))

    def _configure_sampler(self) -> dict:
        """MD_SAMPLE_STEP: set up the engine's sampler with the maps that are on (SAVE_CONTACTS with its fine map,
        SAVE_DISTANCES), binned as the minimised structure's.  Returns the bins and the host-side radial sums."""
        a = self.args
        st = dict(rc=float(contact_setting(a, "CONTACT_RADIUS")), gb=None, fb=None, db=None)
        if contact_setting(a, "SAVE_CONTACTS"):
            st["gb"], st["fb"] = self._contact_bins(), self._contact_bins(fine=True)
        if contact_setting(a, "SAVE_DISTANCES"):
            db = st["db"] = self._distance_bins()
            st["radial"] = [np.zeros(db.n_bins, np.uint64), np.zeros(db.n_bins, np.uint64)]
        gb, fb, db = st["gb"], st["fb"], st["db"]
        self.engine.sampler_configure(st["rc"], None if gb is None else gb.bins, 0 if gb is None else gb.n_bins,
                                      None if fb is None else fb.bins, 0 if fb is None else fb.n_bins,
                                      None if db is None else db.bins, 0 if db is None else db.n_bins)
        return st

    def _sample(self, st: dict):
        """Add the structure on the device to the trajectory maps; the radial sums (O(N)) on the host."""
        from . import distances

        self.engine.sample()
        if st["db"] is not None:
            rs, r2s = distances.radial_sums(self.engine.get_positions(), self.mass_center, st["db"].bins,
                                            st["db"].n_bins)
            st["radial"][0] += rs
            st["radial"][1] += r2s

    def _read_samples(self, st: dict, sample_every: int):
        from . import contacts, distances

        r = self.engine.sampler_read()
        s = r["samples"]
        logger.info(f"trajectory maps: {s} structures sampled every {sample_every} MD steps "
                    f"({r['device_ms']:.1f} ms on the device)")
        if s == 0:
            return
        if st["gb"] is not None:
            self.contacts_md = contacts.result(r["counts"], r["sep"], r["pairs"], st["rc"], st["gb"],
                                               np.uint64(s) * contacts.sep_pairs(self.chrom_spin), members=s)
        if st["fb"] is not None:
            self.contacts_fine_md = contacts.fine_result(r["rows"], r["cols"], r["vals"], r["pairs"], st["rc"],
                                                         st["fb"], members=s)
        if st["db"] is not None:
            self.distances_md = distances.sampled_result(r["dist_sum"], r["dist2_sum"], st["db"], *st["radial"], s)

    def finish(self):
        """Structure files, per-chromosome files, reports, parameters.  Host work (the report's device
        pass takes the device index, not this member's engine)."""
        self.write_minimized()
        if self._whole:
            self.save_chromosomes()  # the minimised structure, as model.py:1222-1224 (before MD)
        if self.args.SAVE_PLOTS:
            self.make_reports()
        from . import contacts, distances

        dense_path = self.contacts_file or os.path.join(self.save_path, "analysis", "contacts.npz")
        fine_path = self.contacts_fine_file or os.path.join(self.save_path, "analysis", "contacts_fine.npz")
        dist_path = self.distances_file or os.path.join(self.save_path, "analysis", "distances.npz")
        save_dense = contacts.save_dense if self.contacts_file is None else contacts.save_member
        for d, md_path in ((self.contacts, dense_path), (self.contacts_md, contacts.md_path(dense_path))):
            if d is not None:
                save_dense(md_path, d)
        for d, path in ((self.contacts_fine, fine_path), (self.contacts_fine_md, contacts.md_path(fine_path))):
            if d is not None:
                contacts.save_fine(path, d)
        for d, path in ((self.distances, dist_path), (self.distances_md, contacts.md_path(dist_path))):
            if d is not None:
                distances.save(path, d)
        if self.loops is not None or self.loops_md is not None:
            from . import loops

            loop_path = self.loops_file or os.path.join(self.save_path, "analysis", "loops.npz")
            for d, path in ((self.loops, loop_path), (self.loops_md, contacts.md_path(loop_path))):
                if d is not None:
                    loops.save(path, d)
        if self.triplets is not None or self.triplets_md is not None:
            from . import triplets

            tri_path = self.triplets_file or os.path.join(self.save_path, "analysis", "triplets.npz")
            for d, path in ((self.triplets, tri_path), (self.triplets_md, contacts.md_path(tri_path))):
                if d is not None:
                    triplets.save(path, d)
        if self.distance_hist is not None or self.distance_hist_md is not None:
            from . import disthist

            hist_path = self.distance_hist_file or os.path.join(self.save_path, "analysis", "distance_hist.npz")
            for d, path in ((self.distance_hist, hist_path), (self.distance_hist_md, contacts.md_path(hist_path))):
                if d is not None:
                    disthist.save(path, d)
        if self.gam is not None or self.gam_md is not None:
            from . import gam

            gam_path = self.gam_file or os.path.join(self.save_path, "analysis", "gam.npz")
            for d, path in ((self.gam, gam_path), (self.gam_md, contacts.md_path(gam_path))):
                if d is not None:
                    gam.save(path, d)
        if self.dynamics is not None:
            from . import dynamics

            dynamics.save(self.dynamics_file or os.path.join(self.save_path, "analysis", "dynamics.npz"), self.dynamics)
        self.save_args_to_txt(self.args.OUT_PATH + "/metadata/parameters.txt")
        return self.report

    def run(self):
        """model.py:1216-1248."""
        self.prepare()
        self.compute()
        return self.finish()

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
