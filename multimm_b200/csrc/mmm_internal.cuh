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

// Grid of the cut-off mode's cell keys, written on the device by k_cut_grid (mmm_cutoff.cu) or
// k_cell_grid (mmm_cells.cu) into the one d_cell_grid of the handle, and read back by mmm_get_cell_grid.
struct CellGrid {
  float origin, cell;  // lower corner (every axis) and edge of a cubic cell
  int dim, bits;       // cells per axis, key bits per axis
};

// One valid row of the loop table (mmm_loops.cu): anchor beads lo < hi, the chromosome block [first, end)
// of each anchor, group 0 (enforced) or 1 (held out).
struct LoopRow {
  int lo, hi, first_lo, end_lo, first_hi, end_hi, group, pad;
};

// ---------------------------------------------------------------------------------------
// the FP64 pair arithmetic of the analysis passes (mmm_contacts, mmm_distance_map, mmm_loops)
// ---------------------------------------------------------------------------------------
// d2 = (dx*dx + dy*dy) + dz*dz rounded operation by operation (no FMA contraction), so that a numpy
// evaluation of the same expression gives the same bits; a pair is a contact when d2 < rc^2.
__device__ __forceinline__ double mmm_pair_d2(double xi, double yi, double zi, double xj, double yj, double zj) {
  const double dx = __dadd_rn(xi, -xj);
  const double dy = __dadd_rn(yi, -yj);
  const double dz = __dadd_rn(zi, -zj);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}
constexpr double MMM_DIST_SCALE = 0x1p24;  // 1 / Q: distances are summed in units of Q = 2^-24 nm (nm^2)
// rint(v / Q), half to even (the scaling is exact): v = d (correctly rounded sqrt of d2) or d2
__device__ __forceinline__ unsigned long long mmm_quantise(double v) {
  return (unsigned long long)__double2ll_rn(__dmul_rn(v, MMM_DIST_SCALE));
}

// ---------------------------------------------------------------------------------------
// device memory
// ---------------------------------------------------------------------------------------
template <class T> class DevBuf;
template <class T> int mmm_reserve(mmm_system* h, DevBuf<T>& buf, size_t count, const char* what);

// An owning device buffer of up to cap_ elements of T.  It converts to T*, so kernel arguments and
// pointer arithmetic read as for a raw pointer.  It grows only through mmm_reserve; the destructor
// and reset() free it.
template <class T>
class DevBuf {
 public:
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { reset(); }
  operator T*() const { return p_; }
  T* get() const { return p_; }  // for a conditional expression or a cast
  T* operator->() const { return p_; }
  void reset() {
    if (p_) cudaFree(p_);
    p_ = nullptr;
    cap_ = 0;
  }
  T* release() {  // the caller frees what it gets
    T* p = p_;
    p_ = nullptr;
    cap_ = 0;
    return p;
  }

 private:
  friend int mmm_reserve<T>(mmm_system* h, DevBuf<T>& buf, size_t count, const char* what);
  T* p_ = nullptr;
  size_t cap_ = 0;
};

// A sorted unique (key, count) list summed over structures on the device (mmm_list_accumulate: the trajectory
// sampler's fine map, the three-way contact map): key[0], val[0] hold the n entries; [1] receives the merge.
struct KeyCountList {
  DevBuf<unsigned long long> key[2], val[2];
  DevBuf<unsigned long long> sval;   // counts of the list being added
  DevBuf<long long> part;            // merge partition, then run offsets of the merge
  int64_t n = 0;
};

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
  DevBuf<int> d_type;            // packed type bits [npad]
  DevBuf<double> d_cstr;         // chrom_strength [n]
  DevBuf<signed char> d_s;       // compartment label [n]

  // topology in gather (CSR) form
  int64_t n_bonds = 0, n_loops = 0, n_angles = 0;
  int loop_form = 0;
  DevBuf<int> d_bl_ptr;          // [n+1]
  DevBuf<int> d_bl_partner;      // [2*(nb+nl)]
  DevBuf<int> d_bl_flags;        // bit0: entry owns the energy; bits 1-2: 0 backbone bond, else 1 + loop form
  DevBuf<double> d_bl_r0;
  DevBuf<double> d_bl_k;
  DevBuf<int> d_an_ptr;          // [n+1]
  DevBuf<int4> d_an_ijk;         // [3*na] (i, j, k, role)
  DevBuf<double2> d_an_par;      // [3*na] (theta0, k)
  std::vector<int32_t> h_bond_i, h_bond_j, h_loop_i, h_loop_j;
  std::vector<double> h_bond_r0, h_bond_k, h_loop_r0, h_loop_k;
  bool topo_dirty = true;

  // state
  DevBuf<double> d_x;            // [3n] master positions (nm), row-major N x 3
  DevBuf<double> d_center;       // [3] centre used for the FP32 copy
  DevBuf<float4> d_pos4;         // [npad] centred FP32 xyz + type bits
  DevBuf<float> d_soa;           // [3][npad] the same coordinates as planes
  DevBuf<TileInfo> d_tiles;      // [ntiles]
  DevBuf<double> d_g;            // [3n] gradient (= -force)

  // pair-kernel scratch
  int nchunk = 1;
  int n_planes = 0;              // planes of d_fpair the assemble pass sums (gather chunks + cell-list plane)
  int chunk_tiles = 0;           // j-tiles per chunk (a whole number of stages)
  int scratch_sig = -1;
  DevBuf<double> d_fpair;        // [nchunk][3][npad]
  DevBuf<double> d_epair_buf;    // [items][4] energy slots (single GPU)
  double* d_epair = nullptr;     // d_epair_buf; several GPUs: the tail of d_facc (one all-reduce covers both)
  int64_t n_items = 0;
  DevBuf<int> d_counter;         // dynamic work counter
  // pair_mode: which kernel the scratch is sized for. 0 none, 1 gather (mmm_pair.cu),
  // 2 Newton-3 (mmm_pair_n3.cu), 3 cut-off cell list (mmm_cells.cu)
  int pair_mode = 0;
  int pair_kernel_pref = 0;      // 0 auto, 1 force the gather kernel (tests / A-B timing)
  DevBuf<unsigned long long> d_facc;  // [3][npad] fixed-point force accumulator (Newton-3, cells)
  DevBuf<int2> d_items;          // Newton-3 work items
  // several GPUs, one system (mmm_dist.cu): Newton-3 items are dealt round-robin to the ranks
  int dist_rank = 0, dist_world = 1;
  bool dist_emulate = false;     // run every rank's share on this GPU, one after another (tests)
  void* nccl_comm = nullptr;
  int* d_gqueue = nullptr;       // two ticket counters in rank 0's memory (CUDA IPC): one work queue for all GPUs
  bool gqueue_owner = false;
  int64_t gqueue_eval = 0;       // evaluations drawn from the queue so far (selects the counter)
  cudaEvent_t ev_c0 = nullptr, ev_c1 = nullptr;  // around the exchange step of the last evaluation (dist)
  int n3_items = 0;              // number of Newton-3 work items (their energy slots come first in d_epair)
  bool n3_chb_only = false;      // the item list is the cut-off mode's CHB-only list
  std::vector<int32_t> h_chrom;  // host copy of the chromosome ids (static; sizes the CHB-only item list)

  // reductions
  int n_red_blocks = 0;
  int n_dot_blocks = 0;
  DevBuf<double> d_epart;        // [n_red_blocks][6] external+bonded energy partials
  DevBuf<double> d_dpart;        // [n_red_blocks][MMM_NDOT] dot partials
  DevBuf<double> d_eterms;       // [MMM_NUM_TERMS] result of the last evaluation
  bool have_result = false;      // d_eterms / d_g hold a finished stand-alone evaluation (mmm_last_result)

  // L-BFGS
  DevBuf<LbfgsState> d_lb;
  DevBuf<double> d_xp, d_gp, d_d;
  DevBuf<double> d_S, d_Y;       // [m][3n]
  int* h_done = nullptr;         // pinned mirror of LbfgsState::done / counters

  // MD relaxation (mmm_md.cu)
  DevBuf<double> d_v;            // [3n] velocities, nm/ps
  bool md_configured = false;
  int md_integrator = 0;
  double md_dt = 0.001, md_temperature = 310.0, md_gamma = 0.5, md_mass = 16427.889;
  double md_amd_alpha = 100.0, md_amd_e = 1000.0;  // config.py:255-256
  uint64_t md_seed = 0;
  int64_t md_step = 0;

  // cell list (cutoff mode)
  DevBuf<uint32_t> d_keys;       // [n] sorted keys
  DevBuf<int> d_order;           // [n] sorted bead order
  DevBuf<uint32_t> d_keys_tmp;
  DevBuf<int> d_order_tmp;
  DevBuf<float4> d_pos4_sorted;
  DevBuf<int> d_cell_start;      // [ncells+1]
  DevBuf<int> d_sort_tmp;        // [2][cells] per-cell histogram, placement cursor
  DevBuf<CellGrid> d_cell_grid;
  DevBuf<unsigned long long> d_cell_npairs;  // ordered pairs inside the cut-off, per CTA
  // cut-off mode on the Newton-3 machinery (mmm_cutoff.cu; default functional forms)
  bool cut_n3 = false;           // the cut-off pass runs the CUT variant of k_pair_n3 (else k_pair_cells)
  DevBuf<float> d_soa_sorted;          // [3][npad] coordinate planes in Morton-sorted order
  DevBuf<TileInfo> d_tiles_sorted;     // [npad / 32] boxes of the sorted tiles
  DevBuf<TileInfo> d_stage_boxes;      // [npad / 256] boxes of the sorted stages
  DevBuf<int> d_sort_table;            // radix-sort digit x block table
  DevBuf<int2> d_items_cut;            // all-pairs item table the CUT kernel culls from
  int n_items_cut = 0;
  std::vector<int32_t> h_cut_iblk;     // i-block of every item of d_items_cut (slab boundaries of the sharded mode)
  DevBuf<double> d_cut_npairs;         // [n_items_cut] pairs inside the cut-off (warp kernel: one per rank)
  bool cut_warp = false;               // the one-warp-per-item kernel serves the cut-off pass (else the CTA-level CUT variant)
  int n_cut_slots = 0;                 // energy slots of the cut-off pass
  DevBuf<unsigned long long> d_cut_eacc;  // [4] fixed-point energies + pair count (warp kernel)
  int sort_age = 0;                    // evaluations since the Morton order was rebuilt (0: rebuild now)
  // CHB on cluster centroids (mmm_chb_clusters.cu): coarse-stage surrogate, cut-off mode only
  bool chb_surrogate = false;    // requested (mmm_set_chb_surrogate)
  bool chb_clusters = false;     // in force for the current scratch
  int n_clusters = 0;
  DevBuf<int> d_cl_start;        // [n_clusters + 1] first bead of every cluster
  DevBuf<int> d_cl_of_bead;      // [n] cluster of every bead
  DevBuf<int> d_cl_by_chrom;     // [n_clusters] clusters sorted by chromosome id
  DevBuf<double> d_cl_cen;       // [n_clusters][4] centroid, bead count
  DevBuf<double> d_cl_force;     // [n_clusters][3] force on every bead of the cluster
  int64_t cl_item0 = 0;          // first d_epair item of the cluster pass
  int cells_plane = 0;           // plane of d_fpair the cell-list pass writes
  int64_t cells_item0 = 0;       // first d_epair item of the cell-list pass

  // timing
  cudaEvent_t ev_a = nullptr, ev_b = nullptr;
  std::vector<cudaEvent_t> ev_pool;  // per-launch event pairs while a timed batch runs
  int ev_cursor = -1;                // -1: not collecting
  DevBuf<unsigned char> d_flush;     // 256 MiB L2-flush scratch (bench only)
  DevBuf<double> d_fout;             // [3n] forces (= -gradient) staged for mmm_energy_forces' host copy
  float last_pair_ms = 0.f;

  // contact counting (mmm_contacts.cu): scratch kept for the handle's lifetime
  DevBuf<int> d_ct_bin;                    // [n] bin of every bead
  DevBuf<unsigned long long> d_ct_map;     // [n_bins^2] dense bin x bin counts
  DevBuf<unsigned long long> d_ct_sep;     // [n] same-chromosome contacts by index separation
  DevBuf<TileInfo> d_ct_stage;             // [stages] boxes of the chain-order 256-bead stages
  DevBuf<unsigned long long> d_ct_cnt;     // [2] contacts, candidate pairs tested
  int64_t ct_candidates = 0;               // candidate pairs the last call tested in FP64
  float ct_ms = 0.f;                       // device time of the last call's kernels (events below)
  cudaEvent_t ct_ev0 = nullptr, ct_ev1 = nullptr;
  // sparse map (mmm_contacts_sparse): grown to the binned contacts of the largest call so far
  DevBuf<long long> d_cs_tile;                          // [tiles + scan parts] int64 key counts -> offsets
  DevBuf<unsigned long long> d_cs_keys[2];              // [keys] each: the radix sort's buffers
  DevBuf<long long> d_cs_table;                         // digit x chunk table + scan parts; then run offsets
  int64_t cs_keys = 0, cs_entries = 0;                  // of the last call: binned contacts, entries
  int cs_src = 0;                                       // which d_cs_keys holds the sorted keys
  int32_t cs_nbins = 0;
  bool cs_valid = false;                                // a call succeeded; mmm_contacts_sparse_read may run

  // mean-distance maps (mmm_distances.cu): scratch kept for the handle's lifetime
  DevBuf<int> d_dm_bin;                    // [n] bin of every bead
  DevBuf<unsigned long long> d_dm_map;     // [2][n_bins^2] quantised distance sums, then squared-distance sums
  DevBuf<double> d_dm_box;                 // per-block bounding boxes of the beads (overflow guard)
  cudaEvent_t dm_ev0 = nullptr, dm_ev1 = nullptr;

  // trajectory sampler (mmm_sampler.cu): maps summed over many structures, on the device until read.  Its
  // own buffers, so that sampling leaves the one-shot calls' results (mmm_contacts_sparse_read) alone
  bool sp_configured = false;
  double sp_rc = 0.0;
  int32_t sp_ct_bins = 0, sp_fine_bins = 0, sp_dm_bins = 0;  // 0: that map is off
  DevBuf<int> d_sp_ct_bin, d_sp_fine_bin, d_sp_dm_bin;      // [n] bins of every bead, uploaded once
  std::vector<int64_t> sp_dm_occ;                          // beads per distance bin (overflow guard)
  int64_t sp_samples = 0;
  double sp_dm_bound = 0.0;                                // summed per-structure bounds of the distance sums
  float sp_ms = 0.f;                                       // device time of all samples
  cudaEvent_t sp_ev0 = nullptr, sp_ev1 = nullptr;
  DevBuf<unsigned long long> d_sp_map;     // [n_bins^2] dense contact map
  DevBuf<unsigned long long> d_sp_sep;     // [n] contacts by index separation
  DevBuf<unsigned long long> d_sp_cnt;     // [4] contacts, candidates (summed); the fine pass's own two
  DevBuf<unsigned long long> d_sp_dist;    // [2][n_bins^2] distance sums, squared-distance sums
  // fine map: the sparse pass into these buffers, then its entries added to sp_fine
  DevBuf<long long> d_sp_tile, d_sp_table;             // the sparse pass's scratch (as d_cs_tile, d_cs_table)
  DevBuf<unsigned long long> d_sp_keys[2];             // the sparse pass's sort buffers
  KeyCountList sp_fine;                                // accumulated fine entries

  // loop readout (mmm_loops.cu): per-row and APA sums over structures, on the device until read
  bool lp_configured = false;
  double lp_rc = 0.0;
  int lp_w = 0;                            // APA window: offsets [-lp_w, lp_w] on each anchor
  int64_t lp_rows = 0;
  int64_t lp_samples = 0;
  double lp_bound = 0.0;                   // summed per-structure bounds of the sums (overflow guard)
  float lp_ms = 0.f;                       // device time of all adds
  cudaEvent_t lp_ev0 = nullptr, lp_ev1 = nullptr;
  DevBuf<LoopRow> d_lp_row;                // [rows]
  DevBuf<unsigned long long> d_lp_sum;     // [3][rows] contacts, dist_sum, dist2_sum; [2 sums][2 groups][(2W+1)^2] APA

  // three-way contact map (mmm_triplets.cu): bead triples in mutual contact, summed over structures
  bool tp_configured = false;
  double tp_rc = 0.0;
  int32_t tp_bins = 0;
  int64_t tp_max_chunk = 0;                // keys per chunk of triples (a chunk holds one bead at least)
  int64_t tp_samples = 0, tp_chunks = 0;
  uint64_t tp_triples = 0;                 // all three-way contacts, binned or not
  float tp_ms = 0.f;                       // device time of all adds
  cudaEvent_t tp_ev0 = nullptr, tp_ev1 = nullptr;
  DevBuf<int> d_tp_ident, d_tp_bin;        // [n] identity bins (the bead-level contact list), the caller's bins
  DevBuf<long long> d_tp_tile, d_tp_table; // the sparse pass's scratch, then the chunks' sort table
  DevBuf<unsigned long long> d_tp_adj[2];  // the sparse pass's sort buffers: forward adjacency i * n + j, i < j
  DevBuf<unsigned long long> d_tp_cnt;     // [3] contacts, candidates, triples of the add
  DevBuf<long long> d_tp_row;              // [n + 1] first adjacency entry of every bead
  DevBuf<long long> d_tp_off;              // [n + 1 + scan parts] binned triples per bead -> their offsets
  DevBuf<unsigned long long> d_tp_keys[2]; // one chunk's keys: the radix sort's buffers
  KeyCountList tp_acc;                     // the accumulated (key, count) list
};

// the sorted keys of one sparse pass (mmm_contacts_sparse_pass)
struct CsSorted {
  long long keys = 0, entries = 0;  // binned contacts, distinct keys
  int src = 0;                      // which sort buffer holds the sorted keys
  unsigned long long cnt[2] = {0, 0};  // contacts, candidates
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

// Make buf hold at least count elements.  A buffer that is large enough is left alone (same
// pointer: captured graphs and earlier views stay valid); otherwise it is replaced by exactly
// count elements, after the handle's stream is done with the old one.  Nothing allocates while a
// graph is captured.  h may be NULL for a temporary of a call without a handle.
template <class T>
int mmm_reserve(mmm_system* h, DevBuf<T>& buf, size_t count, const char* what) {
  if (count <= buf.cap_) return MMM_OK;
  if (h && h->capturing)
    return mmm_fail(h, MMM_ERR_STATE, std::string("allocation of ") + what + " while a CUDA graph is captured");
  if (h && buf.p_) cudaStreamSynchronize(h->stream);
  buf.reset();
  cudaError_t e = cudaMalloc((void**)&buf.p_, count * sizeof(T));
  if (e != cudaSuccess) {
    buf.p_ = nullptr;
    return mmm_fail(h, MMM_ERR_NOMEM, std::string("CUDA error: ") + cudaGetErrorString(e) + " (cudaMalloc, " + what + ")");
  }
  buf.cap_ = count;
  return MMM_OK;
}

// Reserve and copy v from the host; an empty v leaves buf NULL.
template <class T>
int mmm_upload(mmm_system* h, DevBuf<T>& buf, const std::vector<T>& v, const char* what) {
  if (v.empty()) {
    buf.reset();
    return MMM_OK;
  }
  int rc = mmm_reserve(h, buf, v.size(), what);
  if (rc) return rc;
  MMM_CUDA(h, cudaMemcpyAsync(buf, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

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

// mmm_contacts.cu
int mmm_contacts_dense_pass(mmm_system* h, double rc_nm, const int* d_bin, int32_t n_bins, unsigned long long* map,
                            unsigned long long* sep, unsigned long long* cnt, bool clear, cudaEvent_t ev0);
int mmm_contacts_sparse_pass(mmm_system* h, double rc_nm, const int* d_bin, int32_t n_bins, DevBuf<long long>& tile,
                             DevBuf<unsigned long long>* keys, DevBuf<long long>& table, unsigned long long* cnt,
                             cudaEvent_t ev0, cudaEvent_t ev1, CsSorted* out);
void cs_scan(mmm_system* h, long long* a, long long len, long long* part);  // exclusive, in place
long long cs_blocks(long long nkeys);       // 4096-key chunks of the sort, scan and run kernels
size_t cs_table_len(long long nkeys);       // the sort table of nkeys keys
int cs_key_bits(unsigned long long kmax);   // significant bits of the largest key
// LSD radix sort of keys[0][0, m) (< 2^bits) and the run offsets of the sorted keys in table[0, cs_blocks(m));
// returns which buffer holds the sorted keys; the entry count lands at cs_run_total(table, m)
int cs_sort_runs(mmm_system* h, DevBuf<unsigned long long>* keys, long long m, int bits, long long* table);
long long* cs_run_total(long long* table, long long nkeys);
int mmm_list_accumulate(mmm_system* h, const unsigned long long* keys, long long m, const long long* off,
                        long long entries, unsigned long long* spare, KeyCountList& acc);
int mmm_contacts_fine_accumulate(mmm_system* h);  // the sampler's fine map += the current structure's
int mmm_contacts_fine_read(mmm_system* h, int32_t* rows_out, int32_t* cols_out, uint64_t* vals_out);
// mmm_distances.cu
int mmm_distance_qmax(mmm_system* h, const char* who, double* dpad, double* qmax);
int mmm_distance_guard(mmm_system* h, const char* who, const std::vector<int64_t>& occ, double prior, double* bound);
int mmm_distance_pass(mmm_system* h, const int* d_bin, int32_t n_bins, unsigned long long* dmap,
                      unsigned long long* d2map, bool clear);

// one full evaluation at the positions in d_x: prepare -> pair -> assemble.  d_skip (may be
// NULL) points at a device flag; when it is non-zero every kernel returns immediately.
int mmm_evaluate(mmm_system* h, const int* d_skip);
