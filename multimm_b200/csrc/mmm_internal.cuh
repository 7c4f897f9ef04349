// mmm_internal.cuh — internal declarations shared by the sm_100a translation units of
// libmultimm_b200.so.  Not part of the public ABI (that is include/multimm_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/multimm_b200.h"

// ---------------------------------------------------------------------------------------
// constants of the data layout
// ---------------------------------------------------------------------------------------
constexpr int MMM_TILE = 32;          // beads per tile (one warp's worth); bbox granularity
constexpr int MMM_IBLOCK = 256;       // i-beads per work item of the exact pair kernel
constexpr int MMM_STAGE = 256;        // j-beads staged in shared memory at a time
constexpr int MMM_ASM_BLOCK = 128;    // threads per block of the O(N) assemble kernel
#ifndef MMM_LBFGS_M_VALUE
#define MMM_LBFGS_M_VALUE 6
#endif
constexpr int MMM_LBFGS_M = MMM_LBFGS_M_VALUE;  // history length (6 = liblbfgs default used by OpenMM)
constexpr int MMM_NDOT = 6 * MMM_LBFGS_M + 7;  // dot products per evaluation (vector-free L-BFGS)
constexpr int MMM_PAD_TO = 512;       // npad is a multiple of this (i-block of the Newton-3 pair kernel)
// Padding bead k (k = i - n < MMM_PAD_TO) sits at x = y = z = MMM_PAD_COORD + k * MMM_PAD_STEP, so
// far away that every pair term with a real bead underflows to 0, and pads are also far from each
// other (no r = 0 pair).  It carries the chromosome id MMM_PAD_CHROM + k: equal to no real id and
// to no other pad, so chromosome-block work never sees a pad pair as "same chromosome".
constexpr float MMM_PAD_COORD = 1.0e10f;
constexpr float MMM_PAD_STEP = 1.0e7f;
constexpr int MMM_PAD_CHROM = 0xFC00;  // real chromosome ids are < this

// bead type bits carried in pos4.w (bit pattern of an int):
//   [2:0]  s + 2                (sub-compartment label, model.py Cs in {-2..2})
//   [4:3]  class: 1 = A (s > 0), 2 = B (s < 0), 3 = none (s == 0)
//   [23:8] chromosome id (chrom_spin, model.py:158-161), 0xFFFF for padding
__host__ __device__ inline int mmm_pack_type(int s, int chrom) {
  int cls = s > 0 ? 1 : (s < 0 ? 2 : 3);
  return ((s + 2) & 7) | (cls << 3) | ((chrom & 0xFFFF) << 8);
}

// ---------------------------------------------------------------------------------------
// parameters handed to kernels by value
// ---------------------------------------------------------------------------------------
struct PairParams {
  int ev_form, cob_form, scb_form, chb_form;  // MMM_FORM_OFF (-1) = absent
  float ev_eps, ev_rs, ev_sigma, ev_power;
  float cob_rc, cob_ea, cob_eb;
  float scb_rc, scb_e[4];  // Ea1 (s=2), Ea2 (s=1), Eb1 (s=-1), Eb2 (s=-2)
  float chb_kc, chb_de;
  // derived
  float ev_pref;    // eps * sigma^p
  float g_c;        // -log2(e) / (2 rc^2): exp(-r^2/(2 rc^2)) = ex2(r2 * g_c)
  float g_inv_rc2;  // 1 / rc^2
  float rg2;        // squared range beyond which the Gaussian block terms are < 2^-26
  float cutoff2;    // cutoff^2 (cutoff mode) or 0
  // the same globals in FP64, as handed to mmm_set_pair_term (generic any-form path)
  double d_ev[4], d_cob[3], d_scb[5], d_chb[2];
};

struct ExternalParams {
  int sc_form, lam_form, cf_form;
  double sc[6], lam[6], cf[5];
};

// per-tile bounding box + chromosome range (2 x float4 per tile of 32 beads)
struct __align__(16) TileInfo {
  float lox, loy, loz;
  int cmin;
  float hix, hiy, hiz;
  int cmax;
};

// L-BFGS controller state, device resident (one per handle)
struct LbfgsState {
  // control
  int phase;       // 0 = idle, 1 = first evaluation pending, 2 = line search
  int flag;        // what the next apply kernel must do (ApplyFlag)
  int done;        // 0 running, 1 converged, 2 max_iter, 3 line-search failure, 4 non-finite
  int ls_status;   // liblbfgs-style error code when done == 3
  int slot;        // history slot written by the pending ACCEPT
  int end;         // next slot to write
  int bound;       // number of valid history pairs
  int ls_count;
  long long k;     // liblbfgs iteration counter (starts at 1)
  long long iterations, evaluations, max_iter;
  // scalars
  double step, finit, dginit, fx, e_initial, epsilon, gnorm, xnorm;
  double delta[2 * MMM_LBFGS_M + 1];  // coefficients of the next direction over {s_l, y_l, g}
  double ys[MMM_LBFGS_M];
  // Gram matrix of the stored history
  double Gss[MMM_LBFGS_M][MMM_LBFGS_M], Gsy[MMM_LBFGS_M][MMM_LBFGS_M], Gyy[MMM_LBFGS_M][MMM_LBFGS_M];
  double e_terms[MMM_NUM_TERMS];  // per-term energies of the most recent evaluation
};

enum ApplyFlag { APPLY_NONE = 0, APPLY_INIT = 1, APPLY_RETRY = 2, APPLY_ACCEPT = 3, APPLY_RESTORE = 4 };

// ---------------------------------------------------------------------------------------
// the handle
// ---------------------------------------------------------------------------------------
struct mmm_system {
  int device = 0;
  int64_t n = 0;       // beads
  int64_t npad = 0;    // padded to a multiple of MMM_PAD_TO
  int64_t ntiles = 0;  // npad / MMM_TILE
  cudaStream_t stream = nullptr;
  int sm_count = 148;
  std::string err;
  int64_t launches = 0;
  bool capturing = false;          // a CUDA graph capture is in progress: no event records, no allocations
  bool no_graph = false;           // mmm_set_graph(h, 0): plain launches in mmm_minimize (A/B timing)
  int64_t launches_per_period = 0; // kernels in one replay of the captured period

  // parameters (host copies)
  PairParams pp{};
  ExternalParams ep{};
  double cutoff = 0.0;
  bool positions_set = false;
  bool types_dirty = true;

  // per-bead parameters
  int* d_type = nullptr;         // packed type bits [npad]
  double* d_cstr = nullptr;      // chrom_strength [n]
  signed char* d_s = nullptr;    // compartment label [n]

  // topology in gather (CSR) form
  int64_t n_bonds = 0, n_loops = 0, n_angles = 0;
  int loop_form = 0;
  int* d_bl_ptr = nullptr;       // [n+1]
  int* d_bl_partner = nullptr;   // [2*(nb+nl)]
  int* d_bl_flags = nullptr;     // bit0: entry owns the energy; bits 1-2: 0 backbone bond, else 1 + loop form
  double* d_bl_r0 = nullptr;
  double* d_bl_k = nullptr;
  int* d_an_ptr = nullptr;       // [n+1]
  int4* d_an_ijk = nullptr;      // [3*na] (i, j, k, role)
  double2* d_an_par = nullptr;   // [3*na] (theta0, k)
  std::vector<int32_t> h_bond_i, h_bond_j, h_loop_i, h_loop_j;
  std::vector<double> h_bond_r0, h_bond_k, h_loop_r0, h_loop_k;
  bool topo_dirty = true;

  // state
  double* d_x = nullptr;         // [3n] master positions (nm), row-major N x 3
  double* d_center = nullptr;    // [3] centre used for the FP32 copy
  float4* d_pos4 = nullptr;      // [npad] centred FP32 xyz + type bits
  float* d_soa = nullptr;        // [3][npad] the same coordinates as planes
  TileInfo* d_tiles = nullptr;   // [ntiles]
  double* d_g = nullptr;         // [3n] gradient (= -force)

  // pair-kernel scratch
  int nchunk = 1;
  int n_planes = 0;              // planes of d_fpair the assemble pass sums (gather chunks + cell-list plane)
  int chunk_tiles = 0;           // j-tiles per chunk (a whole number of stages)
  int scratch_sig = -1;
  double* d_fpair = nullptr;     // [nchunk][3][npad]
  double* d_epair = nullptr;     // [items][4]
  int64_t n_items = 0;
  int* d_counter = nullptr;      // dynamic work counter
  // pair_mode: which kernel the scratch is sized for. 0 none, 1 gather (mmm_pair.cu),
  // 2 Newton-3 (mmm_pair_n3.cu), 3 cut-off cell list (mmm_cells.cu)
  int pair_mode = 0;
  int pair_kernel_pref = 0;      // 0 auto, 1 force the gather kernel (tests / A-B timing)
  unsigned long long* d_facc = nullptr;  // [3][npad] fixed-point force accumulator (Newton-3, cells)
  int2* d_items = nullptr;       // Newton-3 work items
  // several GPUs, one system (mmm_dist.cu): Newton-3 items are dealt round-robin to the ranks
  int dist_rank = 0, dist_world = 1;
  bool dist_emulate = false;     // run every rank's share on this GPU, one after another (tests)
  void* nccl_comm = nullptr;
  int* d_gqueue = nullptr;       // two ticket counters in rank 0's memory (CUDA IPC): one work queue for all GPUs
  bool gqueue_owner = false;
  int64_t gqueue_eval = 0;       // evaluations drawn from the queue so far (selects the counter)
  bool epair_aliased = false;    // dist: d_epair is the tail of the d_facc allocation (one all-reduce covers both)
  cudaEvent_t ev_c0 = nullptr, ev_c1 = nullptr;  // around the exchange step of the last evaluation (dist)
  int n3_items = 0;              // number of Newton-3 work items (their energy slots come first in d_epair)
  bool n3_chb_only = false;      // the item list is the cut-off mode's CHB-only list
  std::vector<int32_t> h_chrom;  // host copy of the chromosome ids (static; sizes the CHB-only item list)

  // reductions
  int n_red_blocks = 0;
  int n_dot_blocks = 0;
  double* d_epart = nullptr;     // [n_red_blocks][6] external+bonded energy partials
  double* d_dpart = nullptr;     // [n_red_blocks][MMM_NDOT] dot partials
  double* d_eterms = nullptr;    // [MMM_NUM_TERMS] result of the last evaluation
  bool have_result = false;      // d_eterms / d_g hold a finished stand-alone evaluation (mmm_last_result)

  // L-BFGS
  LbfgsState* d_lb = nullptr;
  double *d_xp = nullptr, *d_gp = nullptr, *d_d = nullptr;
  double *d_S = nullptr, *d_Y = nullptr;  // [m][3n]
  int* h_done = nullptr;         // pinned mirror of LbfgsState::done / counters

  // MD relaxation (mmm_md.cu)
  double* d_v = nullptr;         // [3n] velocities, nm/ps
  bool md_configured = false;
  int md_integrator = 0;
  double md_dt = 0.001, md_temperature = 310.0, md_gamma = 0.5, md_mass = 16427.889;
  double md_amd_alpha = 100.0, md_amd_e = 1000.0;  // config.py:255-256
  uint64_t md_seed = 0;
  int64_t md_step = 0;

  // cell list (cutoff mode)
  uint32_t* d_keys = nullptr;    // [n] sorted keys
  int* d_order = nullptr;        // [n] sorted bead order
  uint32_t* d_keys_tmp = nullptr;
  int* d_order_tmp = nullptr;
  float4* d_pos4_sorted = nullptr;
  int* d_cell_start = nullptr;   // [ncells+1]
  void* d_sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0;
  void* d_cell_grid = nullptr;   // device CellGrid {origin, cell, dim, bits}
  unsigned long long* d_cell_npairs = nullptr;  // ordered pairs inside the cut-off, per CTA
  // cut-off mode on the Newton-3 machinery (mmm_cutoff.cu; default functional forms)
  bool cut_n3 = false;           // the cut-off pass runs the CUT variant of k_pair_n3 (else k_pair_cells)
  float* d_soa_sorted = nullptr;       // [3][npad] coordinate planes in Morton-sorted order
  TileInfo* d_tiles_sorted = nullptr;  // [npad / 32] boxes of the sorted tiles
  TileInfo* d_stage_boxes = nullptr;   // [npad / 256] boxes of the sorted stages
  int* d_sort_table = nullptr;         // radix-sort digit x block table
  int2* d_items_cut = nullptr;         // all-pairs item table the CUT kernel culls from
  int n_items_cut = 0;
  std::vector<int32_t> h_cut_iblk;     // i-block of every item of d_items_cut (slab boundaries of the sharded mode)
  double* d_cut_npairs = nullptr;      // [n_items_cut] pairs inside the cut-off (warp kernel: one per rank)
  bool cut_warp = false;               // the one-warp-per-item kernel serves the cut-off pass (else the CTA-level CUT variant)
  int n_cut_slots = 0;                 // energy slots of the cut-off pass
  unsigned long long* d_cut_eacc = nullptr;  // [4] fixed-point energies + pair count (warp kernel)
  int sort_age = 0;                    // evaluations since the Morton order was rebuilt (0: rebuild now)
  // CHB on cluster centroids (mmm_chb_clusters.cu): coarse-stage surrogate, cut-off mode only
  bool chb_surrogate = false;    // requested (mmm_set_chb_surrogate)
  bool chb_clusters = false;     // in force for the current scratch
  int n_clusters = 0;
  int* d_cl_start = nullptr;     // [n_clusters + 1] first bead of every cluster
  int* d_cl_of_bead = nullptr;   // [n] cluster of every bead
  int* d_cl_by_chrom = nullptr;  // [n_clusters] clusters sorted by chromosome id
  int2* d_cl_range = nullptr;    // [n_clusters] slots of by_chrom that hold the same chromosome
  double* d_cl_cen = nullptr;    // [n_clusters][4] centroid, bead count
  double* d_cl_force = nullptr;  // [n_clusters][3] force on every bead of the cluster
  int64_t cl_item0 = 0;          // first d_epair item of the cluster pass
  int cells_plane = 0;           // plane of d_fpair the cell-list pass writes
  int64_t cells_item0 = 0;       // first d_epair item of the cell-list pass

  // timing
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  std::vector<cudaEvent_t> ev_pool;  // per-launch event pairs while a timed batch runs
  int ev_cursor = -1;                // -1: not collecting
  void* d_flush = nullptr;           // 256 MiB L2-flush scratch (bench only)
  double* d_fout = nullptr;          // [3n] forces (= -gradient) staged for mmm_energy_forces' host copy
  float last_pair_ms = 0.f;
};

// ---------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------
int mmm_fail(mmm_system* h, int code, const std::string& msg);
#define MMM_CUDA(h, call)                                                                  \
  do {                                                                                     \
    cudaError_t _e = (call);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return mmm_fail((h), MMM_ERR_CUDA,                                                   \
                      std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " #call); \
  } while (0)

// ---------------------------------------------------------------------------------------
// kernel launchers (defined in the other .cu files)
// ---------------------------------------------------------------------------------------
// mmm_prepare.cu
int mmm_launch_prepare(mmm_system* h, const int* d_skip);  // d_x -> d_pos4, d_tiles
int mmm_launch_hilbert(mmm_system* h, int p, double spacing, int32_t* d_ijk);
// mmm_pair.cu
int mmm_launch_pair_exact(mmm_system* h, const int* d_skip, const PairParams* pp_override = nullptr);  // d_pos4 -> d_fpair, d_epair
bool mmm_pair_fast_path(const mmm_system* h);
bool mmm_pair_fast_path_pp(const PairParams& p);
// mmm_pair_n3.cu
bool mmm_pair_n3_eligible(const mmm_system* h);
bool mmm_pair_n3_generic(const mmm_system* h);
int mmm_n3_build_items(mmm_system* h, std::vector<int2>& items, bool chb_only);
int mmm_launch_pair_n3(mmm_system* h, const int* d_skip, bool chb_only = false);  // d_pos4 -> d_facc, d_epair
// mmm_dist.cu
int mmm_dist_allreduce(mmm_system* h);
void mmm_dist_destroy(mmm_system* h);
int mmm_launch_pair_n3_cut(mmm_system* h, const int* d_skip);
int mmm_cut_warp_build_items(mmm_system* h, std::vector<int2>& items);  // sorted arrays -> d_facc, d_epair (cut-off mode)
// mmm_cutoff.cu
int mmm_launch_pair_cutoff_n3(mmm_system* h, const int* d_skip);
int mmm_cutoff_read_grid(mmm_system* h, float* cell, int32_t* dim, float* origin);
int mmm_cutoff_resort_period();
// mmm_chb_clusters.cu
int mmm_chb_clusters_build(mmm_system* h);
int mmm_chb_clusters_blocks(const mmm_system* h);
int mmm_launch_chb_clusters(mmm_system* h, const int* d_skip);
// mmm_cells.cu
int mmm_launch_pair_cutoff(mmm_system* h, const int* d_skip);
int64_t mmm_cells_energy_slots(const mmm_system* h);
// mmm_bonded.cu
int mmm_upload_topology(mmm_system* h);
int mmm_upload_angles(mmm_system* h, const int32_t* ai, const int32_t* aj, const int32_t* ak,
                      const double* t0, const double* kt, int64_t na);
int mmm_launch_assemble(mmm_system* h, const int* d_skip);  // -> d_g, d_epart
int mmm_launch_finalize_energy(mmm_system* h);  // -> d_eterms (stand-alone evaluation)
// mmm_lbfgs.cu
int mmm_run_minimize(mmm_system* h, double tol, int64_t max_iter, mmm_min_report* out);

// one full evaluation at the positions in d_x: prepare -> pair -> assemble.  d_skip (may be
// NULL) points at a device flag; when it is non-zero every kernel returns immediately.
int mmm_evaluate(mmm_system* h, const int* d_skip);
