/*
 * multimm_b200.h — C-ABI of the B200-native MultiMM energy-minimisation engine.
 *
 * This is the drop-in boundary for the one hot path of SFGLab/MultiMM: the set of OpenMM
 * calls that `src/multimm/model.py` makes between `createSystem` and `minimizeEnergy()`.
 * The reference has no FFI of its own; every entry point below cites the reference lines
 * whose effect it replaces.  Plain pointers and sizes only: no torch / numpy types.
 *
 * Conventions
 *   - lengths nm, energies kJ/mol, angles rad (OpenMM's unit system, model.py passes raw
 *     floats / Quantities in these units);
 *   - every call returns 0 on success, a negative mmm_status otherwise; the text is
 *     available from mmm_last_error().  Device failures contain the substring "CUDA error"
 *     so callers in the style of bridge.py:70-75 still classify them;
 *   - all input arrays are HOST pointers and are copied during the call unless the name
 *     ends in `_device`;
 *   - a handle owns one CUDA device + one stream and is not thread-safe; handles are
 *     independent of each other (ensemble = one handle per replica).
 */
#ifndef MULTIMM_B200_H
#define MULTIMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMM_ABI_VERSION 1

typedef struct mmm_system *mmm_handle;

typedef enum {
  MMM_OK = 0,
  MMM_ERR_ARG = -1,      /* bad argument / unknown form (ValueError in the Python shim) */
  MMM_ERR_CUDA = -2,     /* device failure; message contains "CUDA error" */
  MMM_ERR_STATE = -3,    /* call sequence error (e.g. minimise before positions set) */
  MMM_ERR_NUMERIC = -4,  /* NaN/Inf energy or force */
  MMM_ERR_NOMEM = -5
} mmm_status;

/* Energy terms, in the order add_forcefield builds them (model.py:812-857). The
 * per-term energy array of mmm_energy_forces() is indexed by this enum. */
typedef enum {
  MMM_TERM_EV = 0,     /* add_evforce                 model.py:164-217 */
  MMM_TERM_COB = 1,    /* add_compartment_blocks      model.py:219-294 */
  MMM_TERM_SCB = 2,    /* add_subcompartment_blocks   model.py:296-384 */
  MMM_TERM_CHB = 3,    /* add_chromosomal_blocks      model.py:386-451 */
  MMM_TERM_SC = 4,     /* add_spherical_container     model.py:453-466 */
  MMM_TERM_LAM = 5,    /* add_Blamina_interaction     model.py:468-550 */
  MMM_TERM_CF = 6,     /* add_central_force           model.py:552-623 */
  MMM_TERM_BOND = 7,   /* add_harmonic_bonds          model.py:625-636 */
  MMM_TERM_LOOP = 8,   /* add_loops                   model.py:638-706 */
  MMM_TERM_ANGLE = 9,  /* add_stiffness               model.py:708-720 */
  MMM_NUM_TERMS = 10
} mmm_term;

/* Functional forms are enumerated, not parsed (the reference hands Lepton strings to
 * OpenMM; the strings are fixed per mode so an enum is equivalent). MMM_FORM_OFF disables. */
#define MMM_FORM_OFF (-1)

/* EV forms (model.py:195-215).  globals: {epsilon, r_small, sigma, power} */
#define MMM_EV_POWERLAW 0      /* epsilon*(sigma/(r+r_small))^power        model.py:199 */
#define MMM_EV_GAUSSIAN_CORE 1 /* epsilon*exp(-r^2/(2 sigma^2))            model.py:209 */

/* COB forms (model.py:242-292).  globals: {rc, Ea, Eb} */
/* SCB forms (model.py:318-382).  globals: {rsc, Ea1, Ea2, Eb1, Eb2} */
#define MMM_BLOCK_GAUSSIAN 0 /* -E*exp(-r^2/(2 rc^2))        model.py:246-250, 322-328 */
#define MMM_BLOCK_YUKAWA 1   /* -E*exp(-r/lambda)/r          model.py:262-266, 342-348 */
#define MMM_BLOCK_THETA 2    /* -E*step(rc-r)                model.py:279-283, 363-369 */

/* CHB forms (model.py:412-449).  globals: {k_C, dE} */
#define MMM_CHB_POLYNOMIAL 0 /* dE*delta*(kC r^4 - r^3 + r^2)   model.py:416-419 */
#define MMM_CHB_GAUSSIAN 1   /* -dE*delta*exp(-kC r^2)          model.py:428-431 */
#define MMM_CHB_SATURATING 2 /* -dE*delta/(1+kC r^2)            model.py:440-443 */

/* SC form (model.py:454-456).  globals: {C, R1, R2, x0, y0, z0} */
#define MMM_SC_DOUBLE_WALL 0

/* LAM forms (model.py:499-544).  globals: {B, R1, R2, x0, y0, z0} */
#define MMM_LAM_SIN 0             /* model.py:503-505 */
#define MMM_LAM_GAUSSIAN_SHELL 1  /* sigma = 0.1 (R2-R1)       model.py:513-517 */
#define MMM_LAM_HARMONIC_SHELL 2  /* r0 = (R1+R2)/2            model.py:524-527 */
#define MMM_LAM_LOGISTIC_SHELL 3  /* lambda = 0.05 (R2-R1)     model.py:534-538 */

/* CF forms (model.py:581-615).  globals: {G, R1, x0, y0, z0} */
#define MMM_CF_HARMONIC 0 /* model.py:584-586 */
#define MMM_CF_GAUSSIAN 1 /* sigma = 0.5 R1        model.py:594-599 */
#define MMM_CF_LOGISTIC 2 /* lambda = 0.2 R1       model.py:607-612 */

/* Loop forms (model.py:651-704) */
#define MMM_LOOP_HARMONIC 0        /* 0.5 k (r-r0)^2 (HarmonicBondForce)           model.py:653-659 */
#define MMM_LOOP_FENE_SOFT 1       /* k (r-r0)^2/(1+(r-r0)^2/r0^2)                 model.py:664-680 */
#define MMM_LOOP_GAUSSIAN_TETHER 2 /* k (1-exp(-(r-r0)^2/(r0/2)^2))                model.py:685-701 */

/* Result of mmm_minimize (replaces the silent return of Simulation.minimizeEnergy(),
 * model.py:886). */
typedef struct {
  int64_t iterations;   /* accepted L-BFGS iterations */
  int64_t evaluations;  /* energy+force evaluations, incl. line-search trials */
  double e_initial;     /* total energy at the start */
  double e_final;       /* total energy at the returned positions */
  double rms_force;     /* sqrt(|g|^2 / N) at the returned positions, kJ/mol/nm */
  double wall_seconds;  /* entry to converged positions on device */
  int32_t converged;    /* 1: gradient test met; 0: max_iter hit or line search gave up */
  int32_t ls_status;    /* 0 or the line-search failure code */
} mmm_min_report;

/* ---- lifetime ------------------------------------------------------------------ */
/* Replaces Platform.getPlatformByName + Simulation(...) (model.py:862-876). `device` is the
 * now-honoured DEVICE field (config.py:131). There is no CPU fallback: without a usable
 * sm_100 device this returns MMM_ERR_CUDA.  2 <= n_beads <= 2^24, the number of points of the
 * order-8 Hilbert curve the reference starts from (initial_structure_tools.py:157-166). */
int mmm_create(int device, int64_t n_beads, mmm_handle *out);
int mmm_destroy(mmm_handle h);
/* Text of the last failure on `h` (or of the last failed mmm_create when h is NULL). */
const char *mmm_last_error(mmm_handle h);
int mmm_abi_version(void);

/* ---- topology and parameters (replace the add_* loops of model.py:164-720) -------- */
/* HarmonicBondForce.addBond per backbone bond, model.py:628-635. */
int mmm_set_bonds(mmm_handle h, const int32_t *i, const int32_t *j, const double *r0,
                  const double *k, int64_t n_bonds);
/* Loop bonds, model.py:656-701; `form` is an MMM_LOOP_* value. */
int mmm_set_loops(mmm_handle h, const int32_t *i, const int32_t *j, const double *r0,
                  const double *k, int64_t n_loops, int form);
/* HarmonicAngleForce.addAngle, model.py:711-719. */
int mmm_set_angles(mmm_handle h, const int32_t *i, const int32_t *j, const int32_t *k,
                   const double *theta0, const double *k_theta, int64_t n_angles);
/* Per-bead parameters: compartment label s in {-2..2} (Cs, model.py:239,315,548), chromosome
 * id (chrom_spin, model.py:409) and central-force weight (chrom_strength, model.py:621).
 * Any pointer may be NULL (= all zero). */
int mmm_set_bead_params(mmm_handle h, const int8_t *s, const int32_t *chrom,
                        const double *chrom_strength);
/* Pair terms EV/COB/SCB/CHB. `form` MMM_FORM_OFF removes the term. */
int mmm_set_pair_term(mmm_handle h, int term, int form, const double *globals, int n_globals);
/* External terms SC/LAM/CF. */
int mmm_set_external_term(mmm_handle h, int term, int form, const double *globals,
                          int n_globals);
/* 0 = exact all-pairs (the reference's NoCutoff); > 0 = plain truncation at rc (OpenMM
 * CutoffNonPeriodic semantics) evaluated over a cell list. */
int mmm_set_cutoff(mmm_handle h, double rc_nm);

/* ---- state (context.setPositions / getState, model.py:877, 889) ------------------ */
int mmm_set_positions(mmm_handle h, const double *xyz_nm /* N x 3 row-major */);
int mmm_get_positions(mmm_handle h, double *xyz_nm_out);
/* Same, for a device pointer on the handle's device (torch tensor hand-off). */
int mmm_set_positions_device(mmm_handle h, const double *d_xyz_nm);
int mmm_get_positions_device(mmm_handle h, double *d_xyz_nm_out);
/* On-device Hilbert start (generate_hilbert_curve, initial_structure_tools.py:157-166):
 * the first N points of the 3-D Hilbert curve of order p, times spacing_nm. */
int mmm_hilbert_init(mmm_handle h, int p, double spacing_nm);
/* Integer lattice points only (device generator, host output), int32 N x 3. */
int mmm_hilbert_points(mmm_handle h, int p, int32_t *ijk_out);

/* ---- evaluation ------------------------------------------------------------------- */
/* One fused energy+force evaluation at the current positions. e_terms[MMM_NUM_TERMS]
 * receives per-term energies; forces (N x 3, = -dE/dx) may be NULL. */
int mmm_energy_forces(mmm_handle h, double *e_terms, double *forces);
/* Device-resident variant: no host copy of forces; e_terms still returned to the host. */
int mmm_energy_forces_device(mmm_handle h, double *e_terms, double *d_forces /* may be NULL */);
/* Launch `n` evaluations back to back without host synchronisation in between (bench). */
int mmm_evaluate_n(mmm_handle h, int n);

/* `n` evaluations timed with CUDA events on the handle's own stream (where the kernels are
 * launched).  flush_l2 != 0 overwrites a 256 MiB scratch buffer before every evaluation, inside
 * the timed region.  total_ms: all n evaluations (flushes included); pair_ms: sum of the n pair
 * kernel launches alone (per-launch events). Either output may be NULL. */
int mmm_evaluate_timed(mmm_handle h, int n, int flush_l2, float *total_ms, float *pair_ms);
/* What the most recent evaluation (mmm_energy_forces, mmm_evaluate_n, mmm_evaluate_timed)
 * computed, without evaluating again: per-term energies and forces (N x 3, = -dE/dx), as
 * mmm_energy_forces returns them, for the positions and parameters that evaluation ran with
 * (setting new ones does not recompute them). mmm_minimize and mmm_md_run reuse these buffers:
 * after either, MMM_ERR_STATE until the next evaluation, as before the first. Either output may
 * be NULL. */
int mmm_last_result(mmm_handle h, double *e_terms, double *forces);

/* ---- minimisation (Simulation.minimizeEnergy(), model.py:886) -------------------- */
/* L-BFGS (m = 6, strong-Wolfe backtracking) until the per-particle RMS-force rule of
 * OpenMM's LocalEnergyMinimizer is met: |g| / max(1,|x|) < tol / max(1, rms|x_i|).
 * max_iter 0 = unlimited (the reference's default). No host round trip per iteration. */
int mmm_minimize(mmm_handle h, double tol_kj_mol_nm, int64_t max_iter, mmm_min_report *out);

/* ---- MD relaxation (model.py:768-808 integrators, model.py:907-995 run_md) -------------------- */
#define MMM_MD_LANGEVIN 0 /* mm.LangevinIntegrator(T, friction, dt)   model.py:781-787 */
#define MMM_MD_VERLET 1   /* mm.VerletIntegrator(dt)                  model.py:770-772 */
#define MMM_MD_BROWNIAN 2 /* mm.BrownianIntegrator(T, friction, dt)   model.py:801-807 */
#define MMM_MD_AMD 3      /* mm.amd.AMDIntegrator(dt, alpha, E)       model.py:794-800 */
typedef struct {
  int64_t step;        /* steps taken since mmm_md_configure */
  double potential;    /* kJ/mol at the current positions */
  double kinetic;      /* 1/2 m sum v^2, kJ/mol (leapfrog velocities) */
  double temperature;  /* 2 K / (3 N kB), K */
} mmm_md_report;
/* mass_amu: the single bead mass of forcefields/ff.xml:5 (16427.889). seed: noise stream. */
int mmm_md_configure(mmm_handle h, int integrator, double dt_ps, double temperature_k,
                     double friction_per_ps, double mass_amu, uint64_t seed);
/* The two globals of the accelerated-MD integrator (SIM_AMD_ALPHA, SIM_AMD_E; config.py:255-256:
 * 100 and 1000 kJ/mol, the values a handle starts with).  Used by MMM_MD_AMD only. */
int mmm_md_set_amd(mmm_handle h, double alpha_kj_mol, double e_boost_kj_mol);
/* context.setVelocitiesToTemperature(T, seed), model.py:878. */
int mmm_set_velocities_to_temperature(mmm_handle h, double temperature_k, uint64_t seed);
int mmm_set_velocities(mmm_handle h, const double *v_nm_ps /* N x 3 */);
int mmm_get_velocities(mmm_handle h, double *v_out);
/* simulation.step(n) + getState(getEnergy=True), model.py:929-936: n steps enqueued back to back
 * (one fused force evaluation + one integrator launch each), energies read once at the end. */
int mmm_md_run(mmm_handle h, int64_t n_steps, mmm_md_report *out /* NULL: no energies, no extra evaluation, no host read */);

/* ---- structure report (plots.py:630-829 analyze_structure) ------------------------------------- */
/* Mean of the full N x N distance matrix at the current positions (np.mean(cdist(V, V)),
 * plots.py:663-664) without materialising it. */
int mmm_mean_pair_distance(mmm_handle h, double *mean_out);
/* Block means of the contact map get_heatmap draws (plots.py:540-561: 1 / (d + 1)^(2/3) per bead pair,
 * log1p if log_scale) over bins x bins blocks of consecutive beads (edges as np.linspace(0, n, bins + 1)
 * .astype(int)), for ANY (n, 3) coordinate array — no handle: the structures the report reads back from
 * .cif files are shorter than N_BEADS (HETATM rows dropped, utils.py:184-190).  The N x N matrix never
 * exists, which lifts the reference's N < 50 000 limit (model.py:1095-1104).  mean_dist_out (may be NULL):
 * np.mean(cdist(V, V)) from the same pass. */
int mmm_contact_map(int device, const double *xyz, int64_t n, int bins, int log_scale, double *map_out,
                    double *mean_dist_out);

/* ---- one system on several GPUs of one box (exact mode only) -------------------------------- */
/* The reference has no multi-GPU path (DeviceIndex is never set, model.py:862-876).  Here the
 * O(N^2) pair work of ONE system is dealt to `world` handles, one per GPU / process, each holding
 * the full (replicated) state; ONE NCCL all-reduce (uint64 sum) of the fixed-point force planes and
 * the per-item energy slots follows the pair kernel of every evaluation.  All ranks must make the same
 * calls in the same order.  Results are bit-identical to a single-GPU run.
 *   rank 0: mmm_dist_unique_id(buf, 128); ship buf to the other ranks by any means;
 *   every rank: mmm_dist_init(h, rank, world, buf, 128). */
int mmm_dist_unique_id(void *out, int nbytes);
int mmm_dist_init(mmm_handle h, int rank, int world, const void *unique_id, int nbytes);
/* Single-GPU emulation of the sharding (tests): the shares of all `world` ranks are run one
 * after another on this handle's GPU into the same accumulators. */
int mmm_dist_emulate(mmm_handle h, int world);
/* 1 if the ranks draw their work items from ONE queue (two ticket counters in rank 0's memory, opened by
 * the other ranks through CUDA IPC, advanced with system-scope atomics over NVLink — a slower GPU simply
 * takes fewer items), 0 if the items are dealt round-robin (IPC unavailable, or MMM_DIST_STATIC=1). */
int mmm_dist_queue_mode(mmm_handle h);
/* Milliseconds the exchange step of the most recent evaluation took on this rank (CUDA events on
 * the handle's stream around the all-reduce; includes the wait for the slowest rank).  0 without a
 * communicator. */
int mmm_dist_last_exchange_ms(mmm_handle h, float *ms_out);

/* ---- introspection (tests, bench) ---------------------------------------------------- */
/* Number of kernels this handle has launched since creation. */
int64_t mmm_launch_count(mmm_handle h);
/* Pair-kernel selection (tests, A/B timing): 0 = automatic (Newton-3 kernel for the reference's
 * default forms, gather kernel otherwise), 1 = always the gather kernel. */
int mmm_set_pair_kernel(mmm_handle h, int which);
/* Coarse-stage far field (cut-off mode with the default forms only; never the default, not the
 * reference's potential): the two long-range pieces a truncated evaluation misses — CHB's polynomial
 * (model.py:416-419), which otherwise costs an exact pass over every same-chromosome pair, and the tail
 * of the EV power law beyond the cut-off (model.py:199) — evaluated between the centroids of clusters of
 * <= 32 consecutive same-chromosome beads (O(N + clusters^2)).  A proper potential with an exact gradient;
 * used by the opt-in two-stage minimisation (MIN_COARSE_CUTOFF, MIN_COARSE_FAR_FIELD), whose exact stage
 * follows. */
int mmm_set_chb_surrogate(mmm_handle h, int on);
/* mmm_minimize replays one captured CUDA graph per evaluation (per Morton-order period in cut-off
 * mode) instead of 6-7 separate launches; on = 0 goes back to plain launches (A/B timing, debugging).
 * Results are identical either way. */
int mmm_set_graph(mmm_handle h, int on);
/* Kernel the last evaluation used: 0 none, 1 gather, 2 Newton-3, 3 cut-off cell list. */
int mmm_pair_kernel_in_use(mmm_handle h);
/* Time of the most recent mmm_evaluate_n / mmm_energy_forces pair kernel, ms (CUDA events
 * on the handle's stream). */
int mmm_last_pair_kernel_ms(mmm_handle h, float *ms_out);
/* Cell-list contents of the last cutoff-mode evaluation (bit-exact parity): sorted bead
 * order (int32[N]) and the cell key of each sorted bead (uint32[N]). */
int mmm_get_cell_list(mmm_handle h, int32_t *order_out, uint32_t *key_out);
/* Grid of that cell list (cell edge >= cut-off, cells per axis, common origin of the centred FP32
 * coordinates) and the number of unordered pairs with r2 < rc^2 the pair kernel found: with these
 * the oracle rebuilds keys, order and the neighbour count bit for bit. Any output may be NULL. */
int mmm_get_cell_grid(mmm_handle h, float *cell_out, int32_t *dim_out, float *origin_out,
                      int64_t *pairs_in_cutoff);
/* Micro-benchmarks that measure this GPU's FP32-FMA and MUFU peaks (the roofline
 * denominators of the pair kernel; MEASURED_PEAKS.json has only HBM and bf16). */
int mmm_measure_fp32_peak(int device, double *tflops_out, double *mufu_tops_out);

#ifdef __cplusplus
}
#endif
#endif /* MULTIMM_B200_H */
