// mmm_cells.cu — cut-off mode (opt-in, mmm_set_cutoff(rc > 0)): Morton-sorted cell list and the
// pair kernel over neighbouring cells, for sm_100a.
//
// The reference itself never sets a cut-off (every CustomNonbondedForce stays at NoCutoff,
// model.py:181,231,307,397), so this path is the north star's "pair interactions over a cell list"
// as an explicit extension: plain truncation (OpenMM CutoffNonPeriodic semantics, no shift, no
// switch) of EV / COB / SCB at r < rc; the oracle applies the same truncation with the same FP32
// inclusion test, so cell contents, sorted order and the number of pairs inside the cut-off are
// bit-exact (tests/test_gpu_parity.py; grid, keys and order against the numpy restatement
// tests/cells_ref.py, every form and the cell-boundary edge in tests/test_gpu_cutoff_reference.py).  CHB's polynomial grows with r and cannot be truncated:
// when CHB is on, an exact all-pairs pass restricted to CHB runs beside the cell-list pass.
//
// Per evaluation (all hand-written; the sort is a counting sort by cell, which the cell structure
// gives for free, followed by an id-rank inside each cell so that the order is exactly (key, id) —
// the oracle's stable sort — whatever order the atomics landed in):
//   k_cell_grid   (1 block)  bounding box of the real tiles -> origin, cell edge rc (1 + 2^-12) or
//                            coarser, dim <= 64 (the margin keeps every in-cut pair in neighbouring cells)
//   k_cell_keys   30-bit Morton key of the bead's cell + histogram (RED.ADD per bead)      16 B read,  4 B written per bead
//   k_cell_scan   (1 block)  exclusive scan of the 8^bits cell counts in use -> [start, end) per cell
//   k_cell_place  unstable placement: slot = start[key] + atomic cursor                    8 B written per bead
//   k_cell_rank   rank of the bead's id inside its cell segment -> final slot; writes the sorted
//                 keys, ids and the sorted float4 copy                                     16 B read, 24 B written per bead
//   k_pair_cells  one warp per 32 consecutive sorted beads, one bead per lane; every lane walks the 27
//                 cells around its own cell in fixed order (neighbouring lanes share most
//                 j-addresses), gather formulation => fixed summation order, no atomics.  FP32 inside
//                 a neighbour cell, FP64 across cells.  Default forms specialised; every other form
//                 of every term through pairmath::pair_generic.
#include "mmm_internal.cuh"
#include "mmm_pairmath.cuh"

namespace {

using namespace pairmath;

constexpr int kMaxDim = 64;
constexpr int kMaxCodes = kMaxDim * kMaxDim * kMaxDim;  // 8^6
constexpr int kCellWarps = 8;
constexpr float kCellMargin = 0x1p-12f;  // cell edge = rc * (1 + kCellMargin): see k_cell_grid

__host__ __device__ inline uint32_t spread3(uint32_t v) {
  v &= 0x3ff;
  v = (v | (v << 16)) & 0x030000FF;
  v = (v | (v << 8)) & 0x0300F00F;
  v = (v | (v << 4)) & 0x030C30C3;
  v = (v | (v << 2)) & 0x09249249;
  return v;
}
__host__ __device__ inline uint32_t compact3(uint32_t v) {
  v &= 0x09249249;
  v = (v | (v >> 2)) & 0x030C30C3;
  v = (v | (v >> 4)) & 0x0300F00F;
  v = (v | (v >> 8)) & 0x030000FF;
  v = (v | (v >> 16)) & 0x3ff;
  return v;
}

__global__ void __launch_bounds__(256) k_cell_grid(const TileInfo* __restrict__ tiles, int ntiles, float rc,
                                                   CellGrid* __restrict__ g, const int* __restrict__ skip) {
  if (skip && *skip) return;
  __shared__ float s_lo[256], s_hi[256];
  float lo = 3.0e38f, hi = -3.0e38f;
  for (int t = threadIdx.x; t < ntiles; t += 256) {
    const TileInfo ti = tiles[t];
    if (ti.cmin >= MMM_PAD_CHROM) continue;  // padding only
    lo = fminf(lo, fminf(ti.lox, fminf(ti.loy, ti.loz)));
    hi = fmaxf(hi, fmaxf(ti.hix, fmaxf(ti.hiy, ti.hiz)));
  }
  s_lo[threadIdx.x] = lo;
  s_hi[threadIdx.x] = hi;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_lo[threadIdx.x] = fminf(s_lo[threadIdx.x], s_lo[threadIdx.x + o]);
      s_hi[threadIdx.x] = fmaxf(s_hi[threadIdx.x], s_hi[threadIdx.x + o]);
    }
    __syncthreads();
  }
  // The cell edge is strictly larger than rc, so that every pair the FP32 test accepts lies in
  // neighbouring cells.  A pair with fmaf(dz, dz, fmaf(dy, dy, dx * dx)) < fl(rc * rc) has, on every axis,
  // |fl(x_i - x_j)| < rc (1 + 2^-23), so |x_i - x_j| < rc (1 + 2^-22), which is below (1 - 2^-13) cells of
  // rc (1 + 2^-12).  The cell coordinate floorf(__fdiv_rn(x - origin, cell)) rounds twice, each time by
  // at most 2^-24 of a value below 64 cells, so it moves by less than 2^-17 cells per bead; the two
  // beads' coordinates then differ by less than 1 - 2^-13 + 2^-16 < 1 cell, and their cells by at most
  // one.  (With an edge of exactly rc, pairs on cell boundaries — any lattice of rc / k — land two
  // cells apart and the 27-cell walk never meets them.)  The coarse branch has even more room.
  if (threadIdx.x == 0) {
    const float origin = s_lo[0];
    const float extent = fmaxf(s_hi[0] - origin, 0.0f);
    float cell = rc * (1.0f + kCellMargin);
    int dim = (int)floorf(__fdiv_rn(extent, cell)) + 1;
    if (dim > kMaxDim) {  // coarser cells are still correct (cell > rc); keys are clamped anyway
      cell = __fdiv_rn(extent, (float)(kMaxDim - 1));
      dim = kMaxDim;
    }
    int bits = 0;
    while ((1 << bits) < dim) ++bits;
    g->origin = origin;
    g->cell = cell;
    g->dim = dim;
    g->bits = bits;
  }
}

__device__ __forceinline__ uint32_t cell_coord(float x, const CellGrid& g) {
  int v = (int)floorf(__fdiv_rn(x - g.origin, g.cell));
  v = v < 0 ? 0 : v;
  v = v > g.dim - 1 ? g.dim - 1 : v;
  return (uint32_t)v;
}

__global__ void __launch_bounds__(256) k_cell_keys(const float4* __restrict__ pos4, int64_t n,
                                                   const CellGrid* __restrict__ gp, uint32_t* __restrict__ keys,
                                                   int* __restrict__ count, const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const CellGrid g = *gp;
  const float4 p = pos4[i];
  const uint32_t k = spread3(cell_coord(p.x, g)) | (spread3(cell_coord(p.y, g)) << 1) | (spread3(cell_coord(p.z, g)) << 2);
  keys[i] = k;
  atomicAdd(count + k, 1);
}

// Exclusive scan of the cell counts over the codes in use (8^bits <= kMaxCodes), one block of 1024
// threads, a run of consecutive cells each.
__global__ void __launch_bounds__(1024) k_cell_scan(const CellGrid* __restrict__ gp, const int* __restrict__ count,
                                                    int* __restrict__ cstart, int* __restrict__ cend,
                                                    const int* __restrict__ skip) {
  if (skip && *skip) return;
  __shared__ int s_sum[1024];
  const int ncodes = 1 << (3 * gp->bits);
  const int per = (ncodes + 1023) / 1024;
  const int t = threadIdx.x;
  const int lo = min(t * per, ncodes), hi = min(lo + per, ncodes);
  int local = 0;
  for (int idx = lo; idx < hi; ++idx) local += count[idx];
  s_sum[t] = local;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan of the 1024 partial sums
    const int v = t >= o ? s_sum[t - o] : 0;
    __syncthreads();
    s_sum[t] += v;
    __syncthreads();
  }
  int run = s_sum[t] - local;  // exclusive prefix of this thread's first cell
  for (int idx = lo; idx < hi; ++idx) {
    const int cnt = count[idx];
    cstart[idx] = run;
    run += cnt;
    cend[idx] = run;
  }
}

__global__ void __launch_bounds__(256) k_cell_place(int64_t n, const uint32_t* __restrict__ keys,
                                                    const int* __restrict__ cstart, int* __restrict__ cursor,
                                                    int* __restrict__ slot_id, const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t k = keys[i];
  slot_id[cstart[k] + atomicAdd(cursor + k, 1)] = (int)i;
}

// Final slot of bead i = start of its cell + number of beads of the same cell with a smaller id.
__global__ void __launch_bounds__(256) k_cell_rank(const float4* __restrict__ pos4, int64_t n,
                                                   const uint32_t* __restrict__ keys, const int* __restrict__ cstart,
                                                   const int* __restrict__ cend, const int* __restrict__ slot_id,
                                                   uint32_t* __restrict__ keys_sorted, int* __restrict__ order,
                                                   float4* __restrict__ pos4s, const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  const int i = slot_id[s];
  const uint32_t k = keys[i];
  const int j0 = cstart[k], j1 = cend[k];
  int rank = 0;
  for (int j = j0; j < j1; ++j) rank += slot_id[j] < i ? 1 : 0;
  const int dst = j0 + rank;
  keys_sorted[dst] = k;
  order[dst] = i;
  pos4s[dst] = pos4[i];
}

struct CellArgs {
  const float4* pos4s;
  const uint32_t* keys;
  const int* order;
  const int* cstart;
  const int* cend;
  const CellGrid* grid;
  double* fplane;   // [3][npad], indexed by ORIGINAL bead id
  double* epair;    // [n_cell_items][4]
  unsigned long long* npairs;  // [n_cell_items] ordered pairs inside the cut-off
  int64_t n, npad;
  const int* skip;
  PairParams pp;    // CHB switched off (handled by the exact pass)
};

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int P>
__device__ __forceinline__ float powi(float w) {
  if constexpr (P == 1) {
    return w;
  } else if constexpr (P % 2 == 0) {
    const float hf = powi<P / 2>(w);
    return hf * hf;
  } else {
    return w * powi<P - 1>(w);
  }
}

// Default forms, specialised: power-law EV with integer power EVP, Gaussian SCB (GK & 1) / COB
// (GK & 2).  ~30 instructions per candidate.  Forces in real units.
template <int EVP, int GK>
__device__ __forceinline__ bool pair_fast(const float4 pj, const IBead& b, const PairParams& c, bool live,
                                          float& fx, float& fy, float& fz, float e4[4]) {
  const float dx = b.x - pj.x, dy = b.y - pj.y, dz = b.z - pj.z;
  float r2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
  live = live && (r2 < c.cutoff2);
  r2 = live ? r2 : 1.0f;
  const float inv_r = fast_rsqrt(r2);
  const float r = r2 * inv_r;
  const float w = fast_rcp(r + c.ev_rs);
  const float wp = live ? powi<EVP>(w) : 0.0f;
  e4[0] += wp;  // x eps sigma^p at the end
  float fs = ((float)EVP * c.ev_pref) * wp * w * inv_r;
  if (GK != 0) {
    const float g = live ? fast_ex2(r2 * c.g_c) : 0.0f;
    const int xr = b.w ^ __float_as_int(pj.w);
    if (GK & 1) {
      const float g1 = ((xr & 0x7) == 0) ? g : 0.0f;
      e4[2] += g1;  // x -eps_i at the end
      fs = fmaf(-b.a_scb, g1, fs);
    }
    if (GK & 2) {
      const float g2 = ((xr & 0x18) == 0) ? g : 0.0f;
      e4[1] += g2;
      fs = fmaf(-b.a_cob, g2, fs);
    }
  }
  fx = fmaf(fs, dx, fx);
  fy = fmaf(fs, dy, fy);
  fz = fmaf(fs, dz, fz);
  return live;
}

// One warp per 32 consecutive SORTED beads, one bead per lane, gather formulation (fixed summation
// order per bead, no atomics).
// EVP = 0: any functional form (pair_generic).
template <int EVP, int GK>
__global__ void __launch_bounds__(kCellWarps * 32) k_pair_cells(const CellArgs A) {
  __shared__ double s_red[5][kCellWarps];
  if (A.skip && *A.skip) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const CellGrid g = *A.grid;
  const PairParams& c = A.pp;
  const int64_t i = ((int64_t)blockIdx.x * kCellWarps + warp) * 32 + lane;
  const bool valid = i < A.n;
  double de[4] = {0.0, 0.0, 0.0, 0.0};
  double dfx = 0.0, dfy = 0.0, dfz = 0.0;
  unsigned long long cnt = 0;
  const float4 pi = A.pos4s[valid ? i : 0];
  const int oi = A.order[valid ? i : 0];
  const uint32_t mykey = A.keys[valid ? i : 0];
  IBead b;
  b.x = pi.x; b.y = pi.y; b.z = pi.z; b.w = __float_as_int(pi.w);
  const int si = (b.w & 7) - 2;
  float e_scb_i = 0.0f, e_cob_i = 0.0f;
  if (c.scb_form >= 0 && si != 0) e_scb_i = c.scb_e[si == 2 ? 0 : (si == 1 ? 1 : (si == -1 ? 2 : 3))];
  if (c.cob_form >= 0 && si != 0) e_cob_i = si > 0 ? c.cob_ea : c.cob_eb;
  b.a_scb = e_scb_i * c.g_inv_rc2;
  b.a_cob = e_cob_i * c.g_inv_rc2;

  // Every lane walks the 27 cells around ITS OWN cell (the beads of a warp lie in one or a few
  // adjacent cells, so most lanes share each j-address: the loads coalesce to a broadcast or two);
  // the warp iterates to the longest of its lanes' ranges.  Fixed (z, y, x) order per bead.
  const int cx = (int)compact3(mykey), cy = (int)compact3(mykey >> 1), cz = (int)compact3(mykey >> 2);
  for (int dz = -1; dz <= 1; ++dz) {
    for (int dy = -1; dy <= 1; ++dy) {
      for (int dx = -1; dx <= 1; ++dx) {
        const int nx = cx + dx, ny = cy + dy, nz = cz + dz;
        const bool inside = valid && nx >= 0 && nx < g.dim && ny >= 0 && ny < g.dim && nz >= 0 && nz < g.dim;
        int j0 = 0, j1 = 0;
        if (inside) {
          const uint32_t nc = spread3((uint32_t)nx) | (spread3((uint32_t)ny) << 1) | (spread3((uint32_t)nz) << 2);
          j0 = A.cstart[nc];
          j1 = A.cend[nc];
        }
        const int len = j1 - j0;
        const int maxlen = __reduce_max_sync(0xffffffffu, len);
        float fx = 0.f, fy = 0.f, fz = 0.f, e4[4] = {0.f, 0.f, 0.f, 0.f};
        double gx = 0.0, gy = 0.0, gz = 0.0, g4[4] = {0.0, 0.0, 0.0, 0.0};  // generic (FP64) path
        unsigned hits = 0;
#pragma unroll 4
        for (int t = 0; t < maxlen; ++t) {
          const bool have = t < len;
          const int j = have ? j0 + t : 0;
          const float4 pj = A.pos4s[j];
          bool in;
          if (EVP > 0) {
            in = pair_fast<EVP, GK>(pj, b, c, have && j != i, fx, fy, fz, e4);
          } else {
            const int oj = A.order[j];
            in = pair_generic(pj, b, si, oi < oj, c, have && j != i, gx, gy, gz, g4, c.cutoff2);
          }
          hits += in ? 1u : 0u;
        }
        cnt += hits;
        if (EVP > 0) {
          dfx += (double)fx; dfy += (double)fy; dfz += (double)fz;
          de[0] += (double)e4[0]; de[1] += (double)e4[1]; de[2] += (double)e4[2]; de[3] += (double)e4[3];
        } else {
          dfx += gx; dfy += gy; dfz += gz;
          de[0] += g4[0]; de[1] += g4[1]; de[2] += g4[2]; de[3] += g4[3];
        }
      }
    }
  }
  if (valid) {
    A.fplane[oi] = dfx;
    A.fplane[(size_t)A.npad + oi] = dfy;
    A.fplane[2 * (size_t)A.npad + oi] = dfz;
  }
  if (EVP > 0) {
    de[0] *= (double)c.ev_pref;
    de[1] *= -(double)e_cob_i;
    de[2] *= -(double)e_scb_i;
  }
  // each unordered pair was seen from both sides
  double v[5] = {0.5 * de[0], 0.5 * de[1], 0.5 * de[2], 0.5 * de[3], (double)cnt};
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    v[q] = warp_sum_d(v[q]);
    if (lane == 0) s_red[q][warp] = v[q];
  }
  __syncthreads();
  if (threadIdx.x < 5) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kCellWarps; ++w) s += s_red[threadIdx.x][w];
    if (threadIdx.x < 4) A.epair[(size_t)blockIdx.x * 4 + threadIdx.x] = s;
    else A.npairs[blockIdx.x] = (unsigned long long)(s + 0.5);
  }
}

template <int EVP>
void launch_cells_evp(const CellArgs& A, int gk, int blocks, cudaStream_t st) {
  switch (gk) {
    case 0: k_pair_cells<EVP, 0><<<blocks, kCellWarps * 32, 0, st>>>(A); break;
    case 1: k_pair_cells<EVP, 1><<<blocks, kCellWarps * 32, 0, st>>>(A); break;
    case 2: k_pair_cells<EVP, 2><<<blocks, kCellWarps * 32, 0, st>>>(A); break;
    default: k_pair_cells<EVP, 3><<<blocks, kCellWarps * 32, 0, st>>>(A); break;
  }
}

}  // namespace

int64_t mmm_cells_energy_slots(const mmm_system* h) { return (h->n + kCellWarps * 32 - 1) / (kCellWarps * 32); }

static int mmm_cells_alloc(mmm_system* h) {
  const size_t npad = (size_t)h->npad;
  int rc;
  // keys, order, sorted positions and grid are shared with mmm_cutoff.cu: both reserve npad (the most either uses)
  if ((rc = mmm_reserve(h, h->d_keys, npad, "cell keys")) || (rc = mmm_reserve(h, h->d_keys_tmp, npad, "cell keys")) ||
      (rc = mmm_reserve(h, h->d_order, npad, "sorted order")) ||
      (rc = mmm_reserve(h, h->d_order_tmp, npad, "sorted order")) ||
      (rc = mmm_reserve(h, h->d_pos4_sorted, npad, "sorted positions")) ||
      (rc = mmm_reserve(h, h->d_cell_grid, 1, "cell grid")) ||
      (rc = mmm_reserve(h, h->d_cell_start, (size_t)2 * kMaxCodes, "cell ranges")) ||
      (rc = mmm_reserve(h, h->d_cell_npairs, (size_t)mmm_cells_energy_slots(h), "cell pair counts")) ||
      (rc = mmm_reserve(h, h->d_sort_tmp, (size_t)2 * kMaxCodes, "cell histogram")))
    return rc;
  return MMM_OK;
}

// Cell-list pass: EV / COB / SCB truncated at the cut-off, forces into plane `plane` of d_fpair,
// energies into d_epair at item offset `item0`.
int mmm_launch_pair_cutoff(mmm_system* h, const int* d_skip) {
  int rc;
  if ((rc = mmm_cells_alloc(h))) return rc;
  const int n = (int)h->n;
  const int blocks = (n + 255) / 256;
  CellGrid* grid = h->d_cell_grid;
  int* cstart = h->d_cell_start;
  int* cend = h->d_cell_start + kMaxCodes;

  const bool collect = h->ev_cursor >= 0 && (size_t)(2 * h->ev_cursor + 1) < h->ev_pool.size();
  cudaEvent_t ea = collect ? h->ev_pool[2 * h->ev_cursor] : h->ev_a;
  cudaEvent_t eb = collect ? h->ev_pool[2 * h->ev_cursor + 1] : h->ev_b;
  if (collect) h->ev_cursor++;
  if (!h->capturing) MMM_CUDA(h, cudaEventRecord(ea, h->stream));

  int* count = h->d_sort_tmp;  // per-cell histogram, then placement cursor
  int* cursor = count + kMaxCodes;
  MMM_CUDA(h, cudaMemsetAsync(count, 0, sizeof(int) * 2 * kMaxCodes, h->stream));
  k_cell_grid<<<1, 256, 0, h->stream>>>(h->d_tiles, (int)h->ntiles, (float)h->cutoff, grid, d_skip);
  k_cell_keys<<<blocks, 256, 0, h->stream>>>(h->d_pos4, h->n, grid, h->d_keys_tmp, count, d_skip);
  k_cell_scan<<<1, 1024, 0, h->stream>>>(grid, count, cstart, cend, d_skip);
  k_cell_place<<<blocks, 256, 0, h->stream>>>(h->n, h->d_keys_tmp, cstart, cursor, h->d_order_tmp, d_skip);
  k_cell_rank<<<blocks, 256, 0, h->stream>>>(h->d_pos4, h->n, h->d_keys_tmp, cstart, cend, h->d_order_tmp, h->d_keys,
                                             h->d_order, h->d_pos4_sorted, d_skip);
  CellArgs A;
  A.pos4s = h->d_pos4_sorted;
  A.keys = h->d_keys;
  A.order = h->d_order;
  A.cstart = cstart;
  A.cend = cend;
  A.grid = grid;
  A.fplane = h->d_fpair + (size_t)h->cells_plane * 3 * (size_t)h->npad;
  A.epair = h->d_epair + (size_t)h->cells_item0 * 4;
  A.npairs = h->d_cell_npairs;
  A.n = h->n;
  A.npad = h->npad;
  A.skip = d_skip;
  A.pp = h->pp;
  A.pp.chb_form = MMM_FORM_OFF;
  const int cblocks = (int)mmm_cells_energy_slots(h);
  if (mmm_pair_fast_path_pp(A.pp) && A.pp.ev_form == MMM_EV_POWERLAW) {
    const int gk = (A.pp.scb_form >= 0 ? 1 : 0) | (A.pp.cob_form >= 0 ? 2 : 0);
    if (A.pp.ev_power == 6.0f) launch_cells_evp<6>(A, gk, cblocks, h->stream);
    else launch_cells_evp<3>(A, gk, cblocks, h->stream);
  } else {
    k_pair_cells<0, 0><<<cblocks, kCellWarps * 32, 0, h->stream>>>(A);
  }
  h->launches += 6;
  MMM_CUDA(h, cudaGetLastError());
  if (!h->capturing) MMM_CUDA(h, cudaEventRecord(eb, h->stream));
  return MMM_OK;
}

extern "C" {

int mmm_get_cell_list(mmm_handle h, int32_t* order_out, uint32_t* key_out) {
  if (!h) return MMM_ERR_ARG;
  if (h->pair_mode != 3 || !h->d_keys)
    return mmm_fail(h, MMM_ERR_STATE, "mmm_get_cell_list: no cut-off evaluation has run on this handle");
  cudaSetDevice(h->device);
  if (order_out)
    MMM_CUDA(h, cudaMemcpyAsync(order_out, h->d_order, sizeof(int) * h->n, cudaMemcpyDeviceToHost, h->stream));
  if (key_out)
    MMM_CUDA(h, cudaMemcpyAsync(key_out, h->d_keys, sizeof(uint32_t) * h->n, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_get_cell_grid(mmm_handle h, float* cell_out, int32_t* dim_out, float* origin_out, int64_t* pairs_in_cutoff) {
  if (!h) return MMM_ERR_ARG;
  if (h->pair_mode != 3 || !h->d_keys)
    return mmm_fail(h, MMM_ERR_STATE, "mmm_get_cell_grid: no cut-off evaluation has run on this handle");
  cudaSetDevice(h->device);
  CellGrid g;
  MMM_CUDA(h, cudaMemcpyAsync(&g, h->d_cell_grid, sizeof(g), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (cell_out) *cell_out = g.cell;
  if (dim_out) *dim_out = g.dim;
  if (origin_out) *origin_out = g.origin;
  if (h->cut_n3) {
    if (pairs_in_cutoff) {
      std::vector<double> per_item((size_t)h->n_cut_slots);
      MMM_CUDA(h, cudaMemcpyAsync(per_item.data(), h->d_cut_npairs, per_item.size() * sizeof(double),
                                  cudaMemcpyDeviceToHost, h->stream));
      MMM_CUDA(h, cudaStreamSynchronize(h->stream));
      double s = 0.0;
      for (double v : per_item) s += v;  // halves of diagonal stages (ordered pairs) add up to integers
      *pairs_in_cutoff = (int64_t)(s + 0.5);
    }
    return MMM_OK;
  }
  if (pairs_in_cutoff) {
    std::vector<unsigned long long> cnt((size_t)mmm_cells_energy_slots(h));
    MMM_CUDA(h, cudaMemcpyAsync(cnt.data(), h->d_cell_npairs, cnt.size() * sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, h->stream));
    MMM_CUDA(h, cudaStreamSynchronize(h->stream));
    unsigned long long s = 0;
    for (unsigned long long v : cnt) s += v;
    *pairs_in_cutoff = (int64_t)(s / 2);  // the gather kernel sees each unordered pair twice
  }
  return MMM_OK;
}

}  // extern "C"
