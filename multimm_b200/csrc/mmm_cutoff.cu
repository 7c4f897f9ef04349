// mmm_cutoff.cu — cut-off mode for the reference's default functional forms: Morton-sorted beads,
// bounding boxes of 32-bead tiles, and the Newton-3 pair kernel (mmm_pair_n3.cu, CUT variant) over the
// tile pairs that lie within the cut-off.  This is the north star's "cell list / neighbour list,
// Morton-sorted beads, shared-memory tile staging, warp-shuffle force reduction, deterministic
// per-bead accumulation" kernel; the reference itself never truncates (model.py:181,231,307,397), so
// the mode is an explicit extension (mmm_set_cutoff) whose oracle applies the same truncation.
//
// Per list rebuild (every evaluation after new positions arrive from the host, every kResortEvery
// evaluations inside a minimisation — results never depend on the age of the sort, only speed does):
//   k_cut_grid     bounding box of the real tiles -> origin, key cell edge = rc / 4 exactly, <= 1024 cells per
//                  axis (10 key bits per axis; beads beyond that share the edge cell — the order is only a
//                  locality heuristic, the pair kernel culls on the real bounding boxes)
//   k_cut_keys     30-bit Morton key of the bead's cell                       16 B read, 8 B written per bead
//   LSD radix sort of (key, bead id), 3 passes of 10 bits, each: k_sort_hist (per-block digit
//                  histogram), k_sort_scan (exclusive scan of the digit x block table, 1 block),
//                  k_sort_scatter (stable ranks by warp match_any + per-warp digit counters)
//                  — stable, so the order is exactly the oracle's (key, id) order.   16 B read + 16 B written per bead per pass
// Per evaluation:
//   k_gather_sorted  sorted FP32 copy of the beads (float4 + planes), bounding boxes of the sorted
//                    32-bead tiles and of the 256-bead stages                48 B per bead
//   k_pair_n3<.., CUT>  (mmm_pair_n3.cu) stages whose box is farther than rc from the i-block are culled
//                    by one ballot per work item, tiles by the per-step classification, pairs by the
//                    r^2 < rc^2 mask; forces leave as 64-bit fixed point through the sort permutation.
// CHB's polynomial grows with r and is never truncated: the CHB-only Newton-3 pass over
// same-chromosome tile pairs (chain order) runs beside this one, into the same accumulators.
// Integer outputs stay bit-exact against the oracle: keys, order, number of pairs with r^2 < rc^2.
#include <algorithm>

#include "mmm_internal.cuh"

namespace {

constexpr int kMaxDim = 1024;
constexpr int kDigitBits = 10, kDigits = 1 << kDigitBits, kPasses = 3;
constexpr int kSortThreads = 256, kSortPer = 8, kSortChunk = kSortThreads * kSortPer;  // 2048 keys per block
constexpr int kResortEvery = 8;
// The Morton key is taken on cells of a QUARTER of the cut-off: the pair kernel culls on the bounding
// boxes of 32 consecutive sorted beads, and with keys on cells of the full cut-off the ~100 beads of a
// cell keep their bead-id order, which after a few hundred L-BFGS iterations is no spatial order at all
// (tile boxes as large as the cell: measured 1.30 ms per pass against 1.02 ms on the Hilbert start).
constexpr float kKeyCellFraction = 0.25f;

__host__ __device__ inline uint32_t spread3(uint32_t v) {
  v &= 0x3ff;
  v = (v | (v << 16)) & 0x030000FF;
  v = (v | (v << 8)) & 0x0300F00F;
  v = (v | (v << 4)) & 0x030C30C3;
  v = (v | (v << 2)) & 0x09249249;
  return v;
}

__global__ void __launch_bounds__(256) k_cut_grid(const TileInfo* __restrict__ tiles, int ntiles, float rc,
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
  if (threadIdx.x == 0) {
    const float origin = s_lo[0];
    const float extent = fmaxf(s_hi[0] - origin, 0.0f);
    const float cell = rc * kKeyCellFraction;  // a fixed fraction of the cut-off: the geometry of the structure never coarsens it
    int dim = (int)fminf(floorf(__fdiv_rn(extent, cell)), (float)(kMaxDim - 1)) + 1;
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
  v = v > g.dim - 1 ? g.dim - 1 : v;  // beads beyond 1024 cells share the edge cell (a contraction)
  return (uint32_t)v;
}

__global__ void __launch_bounds__(256) k_cut_keys(const float4* __restrict__ pos4, int n, const CellGrid* __restrict__ gp,
                                                  uint32_t* __restrict__ keys, int* __restrict__ ids,
                                                  const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const CellGrid g = *gp;
  const float4 p = pos4[i];
  keys[i] = spread3(cell_coord(p.x, g)) | (spread3(cell_coord(p.y, g)) << 1) | (spread3(cell_coord(p.z, g)) << 2);
  ids[i] = i;
}

// ---- LSD radix sort, one pass = hist + scan + scatter --------------------------------------
__global__ void __launch_bounds__(kSortThreads) k_sort_hist(const uint32_t* __restrict__ keys, int n, int shift,
                                                            int* __restrict__ table, int nblocks,
                                                            const int* __restrict__ skip) {
  if (skip && *skip) return;
  __shared__ int s_cnt[kDigits];
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) s_cnt[d] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortChunk;
  for (int q = threadIdx.x; q < kSortChunk; q += kSortThreads) {
    const int e = base + q;
    if (e < n) atomicAdd(&s_cnt[(keys[e] >> shift) & (kDigits - 1)], 1);
  }
  __syncthreads();
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) table[(size_t)blockIdx.x * kDigits + d] = s_cnt[d];
}

// Exclusive scan of the digit x block counts in digit-major order (all blocks of digit 0, then digit
// 1, ...), in place; one block, thread d owns digit d.  The table is stored block-major
// (table[b * 1024 + d]) so that both sweeps over the blocks are coalesced across the threads.
__global__ void __launch_bounds__(kDigits) k_sort_scan(int* __restrict__ table, int nblocks, const int* __restrict__ skip) {
  if (skip && *skip) return;
  __shared__ int s_sum[kDigits];
  const int d = threadIdx.x;
  int total = 0;
  for (int b = 0; b < nblocks; ++b) total += table[(size_t)b * kDigits + d];
  s_sum[d] = total;
  __syncthreads();
  for (int o = 1; o < kDigits; o <<= 1) {  // Hillis-Steele inclusive scan of the digit totals
    const int v = d >= o ? s_sum[d - o] : 0;
    __syncthreads();
    s_sum[d] += v;
    __syncthreads();
  }
  int run = s_sum[d] - total;  // beads with a smaller digit
  for (int b = 0; b < nblocks; ++b) {
    const int c = table[(size_t)b * kDigits + d];
    table[(size_t)b * kDigits + d] = run;
    run += c;
  }
}

// Stable scatter.  Warp w owns elements [w * 256, (w + 1) * 256) of the block's chunk and visits them
// in 8 rounds of 32 consecutive elements, so (round, lane) order is the element order.  Per round the
// lanes with equal digits find each other with match_any; the lowest of them advances the warp's
// counter of that digit (distinct digits -> distinct addresses, no conflict).
__global__ void __launch_bounds__(kSortThreads) k_sort_scatter(const uint32_t* __restrict__ keys_in,
                                                               const int* __restrict__ ids_in, int n, int shift,
                                                               const int* __restrict__ table, int nblocks,
                                                               uint32_t* __restrict__ keys_out, int* __restrict__ ids_out,
                                                               const int* __restrict__ skip) {
  if (skip && *skip) return;
  constexpr int kWarps = kSortThreads / 32;
  __shared__ int s_cnt[kWarps][kDigits];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int d = threadIdx.x; d < kWarps * kDigits; d += kSortThreads) (&s_cnt[0][0])[d] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortChunk + warp * (kSortChunk / kWarps);
  uint32_t key[kSortPer];
  int id[kSortPer], rank[kSortPer];
#pragma unroll
  for (int r = 0; r < kSortPer; ++r) {
    const int e = base + r * 32 + lane;
    const bool have = e < n;
    key[r] = have ? keys_in[e] : 0xFFFFFFFFu;
    id[r] = have ? ids_in[e] : -1;
    const int d = have ? (int)((key[r] >> shift) & (kDigits - 1)) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int before = __popc(peers & ((1u << lane) - 1u));
    int old = 0;
    if (have && before == 0) {
      old = s_cnt[warp][d];
      s_cnt[warp][d] = old + __popc(peers);
    }
    old = __shfl_sync(0xffffffffu, old, __ffs(peers) - 1);
    rank[r] = old + before;
    __syncwarp();
  }
  __syncthreads();
  // exclusive prefix over the warps, per digit
  for (int d = threadIdx.x; d < kDigits; d += kSortThreads) {
    int run = table[(size_t)blockIdx.x * kDigits + d];
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      const int c = s_cnt[w][d];
      s_cnt[w][d] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kSortPer; ++r) {
    if (id[r] < 0) continue;
    const int d = (int)((key[r] >> shift) & (kDigits - 1));
    const int dst = s_cnt[warp][d] + rank[r];
    keys_out[dst] = key[r];
    ids_out[dst] = id[r];
  }
}

// pads keep their own slots behind the real beads: order[s] = s for s >= n
__global__ void __launch_bounds__(256) k_order_tail(int* __restrict__ order, int n, int npad) {
  const int s = n + blockIdx.x * blockDim.x + threadIdx.x;
  if (s < npad) order[s] = s;
}

// Sorted FP32 copy (float4 + planes) and the boxes of the sorted 32-bead tiles; one warp per tile.
__global__ void __launch_bounds__(256) k_gather_sorted(const float4* __restrict__ pos4, const int* __restrict__ order,
                                                       int n, int npad, float4* __restrict__ pos4s,
                                                       float* __restrict__ soas, TileInfo* __restrict__ tiles,
                                                       const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int lane = threadIdx.x & 31;
  const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int s = tile * MMM_TILE + lane;
  if (s >= npad) return;
  const bool real = s < n;
  const float4 p = pos4[order[s]];
  pos4s[s] = p;
  soas[s] = p.x;
  soas[npad + s] = p.y;
  soas[2 * (size_t)npad + s] = p.z;
  const float big = 3.0e38f;
  float lox = real ? p.x : big, loy = real ? p.y : big, loz = real ? p.z : big;
  float hix = real ? p.x : -big, hiy = real ? p.y : -big, hiz = real ? p.z : -big;
  const int ch = (__float_as_int(p.w) >> 8) & 0xFFFF;
  int cmin = real ? ch : 0x7fffffff, cmax = real ? ch : -1;
  const bool mixed = __any_sync(0xffffffffu, real) && !__all_sync(0xffffffffu, real);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lox = fminf(lox, __shfl_xor_sync(0xffffffffu, lox, o));
    loy = fminf(loy, __shfl_xor_sync(0xffffffffu, loy, o));
    loz = fminf(loz, __shfl_xor_sync(0xffffffffu, loz, o));
    hix = fmaxf(hix, __shfl_xor_sync(0xffffffffu, hix, o));
    hiy = fmaxf(hiy, __shfl_xor_sync(0xffffffffu, hiy, o));
    hiz = fmaxf(hiz, __shfl_xor_sync(0xffffffffu, hiz, o));
    cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
    cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
  }
  if (lane == 0) {
    TileInfo t;
    if (cmax < 0) {
      t.lox = t.loy = t.loz = t.hix = t.hiy = t.hiz = MMM_PAD_COORD;
      t.cmin = t.cmax = MMM_PAD_CHROM;
    } else {
      t.lox = lox; t.loy = loy; t.loz = loz;
      t.hix = hix; t.hiy = hiy; t.hiz = hiz;
      t.cmin = cmin; t.cmax = mixed ? MMM_PAD_CHROM : cmax;
    }
    tiles[tile] = t;
  }
}

// boxes of the 256-bead stages (8 tiles each): what the pair kernel's per-item ballot tests
__global__ void __launch_bounds__(256) k_stage_boxes(const TileInfo* __restrict__ tiles, int nstages,
                                                     TileInfo* __restrict__ stages, const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nstages) return;
  TileInfo b;
  b.lox = b.loy = b.loz = 3.0e38f;
  b.hix = b.hiy = b.hiz = -3.0e38f;
  b.cmin = MMM_PAD_CHROM;
  b.cmax = -1;
  for (int q = 0; q < MMM_STAGE / MMM_TILE; ++q) {
    const TileInfo t = tiles[s * (MMM_STAGE / MMM_TILE) + q];
    if (t.cmin >= MMM_PAD_CHROM) continue;  // padding only
    b.lox = fminf(b.lox, t.lox); b.loy = fminf(b.loy, t.loy); b.loz = fminf(b.loz, t.loz);
    b.hix = fmaxf(b.hix, t.hix); b.hiy = fmaxf(b.hiy, t.hiy); b.hiz = fmaxf(b.hiz, t.hiz);
    b.cmin = min(b.cmin, t.cmin);
    b.cmax = max(b.cmax, t.cmax);
  }
  stages[s] = b;  // cmin == MMM_PAD_CHROM: nothing real in the stage
}

}  // namespace

static int mmm_cutoff_alloc(mmm_system* h) {
  const size_t n = (size_t)h->n, npad = (size_t)h->npad;
  const int nblocks = (int)((n + kSortChunk - 1) / kSortChunk);
  int rc;
  // keys, order, sorted positions and grid are shared with mmm_cells.cu: both reserve npad (the most either uses)
  if ((rc = mmm_reserve(h, h->d_keys, npad, "cell keys")) || (rc = mmm_reserve(h, h->d_keys_tmp, npad, "cell keys")) ||
      (rc = mmm_reserve(h, h->d_order, npad, "sorted order")) ||
      (rc = mmm_reserve(h, h->d_order_tmp, npad, "sorted order")) ||
      (rc = mmm_reserve(h, h->d_pos4_sorted, npad, "sorted positions")) ||
      (rc = mmm_reserve(h, h->d_cell_grid, 1, "cell grid")) ||
      (rc = mmm_reserve(h, h->d_soa_sorted, 3 * npad, "sorted coordinate planes")) ||
      (rc = mmm_reserve(h, h->d_tiles_sorted, npad / MMM_TILE, "sorted tile boxes")) ||
      (rc = mmm_reserve(h, h->d_stage_boxes, npad / MMM_STAGE, "sorted stage boxes")) ||
      (rc = mmm_reserve(h, h->d_sort_table, (size_t)kDigits * nblocks, "radix-sort table")))
    return rc;
  return MMM_OK;
}

// Rebuild the Morton order from the current (chain-order) FP32 copy.
static int rebuild_order(mmm_system* h, const int* d_skip) {
  const int n = (int)h->n, npad = (int)h->npad;
  const int nblocks = (n + kSortChunk - 1) / kSortChunk;
  CellGrid* grid = h->d_cell_grid;
  k_cut_grid<<<1, 256, 0, h->stream>>>(h->d_tiles, (int)h->ntiles, (float)h->cutoff, grid, d_skip);
  k_cut_keys<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_pos4, n, grid, h->d_keys_tmp, h->d_order_tmp, d_skip);
  uint32_t* kin = h->d_keys_tmp; uint32_t* kout = h->d_keys;
  int* iin = h->d_order_tmp; int* iout = h->d_order;
  for (int pass = 0; pass < kPasses; ++pass) {
    const int shift = pass * kDigitBits;
    k_sort_hist<<<nblocks, kSortThreads, 0, h->stream>>>(kin, n, shift, h->d_sort_table, nblocks, d_skip);
    k_sort_scan<<<1, kDigits, 0, h->stream>>>(h->d_sort_table, nblocks, d_skip);
    k_sort_scatter<<<nblocks, kSortThreads, 0, h->stream>>>(kin, iin, n, shift, h->d_sort_table, nblocks, kout, iout, d_skip);
    std::swap(kin, kout);
    std::swap(iin, iout);
  }
  // an odd number of passes leaves the result in (d_keys, d_order): kin / iin point at it now
  if (kin != h->d_keys) {
    MMM_CUDA(h, cudaMemcpyAsync(h->d_keys, kin, sizeof(uint32_t) * n, cudaMemcpyDeviceToDevice, h->stream));
    MMM_CUDA(h, cudaMemcpyAsync(h->d_order, iin, sizeof(int) * n, cudaMemcpyDeviceToDevice, h->stream));
  }
  if (npad > n) k_order_tail<<<(npad - n + 255) / 256, 256, 0, h->stream>>>(h->d_order, n, npad);
  h->launches += 2 + 3 * kPasses + (npad > n ? 1 : 0);
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}

// The cut-off pass for the default forms: (re)sort, gather, Newton-3 kernel with the CUT variant.
int mmm_launch_pair_cutoff_n3(mmm_system* h, const int* d_skip) {
  int rc;
  if ((rc = mmm_cutoff_alloc(h))) return rc;
  const bool collect = h->ev_cursor >= 0 && (size_t)(2 * h->ev_cursor + 1) < h->ev_pool.size();
  cudaEvent_t ea = collect ? h->ev_pool[2 * h->ev_cursor] : h->ev_a;
  cudaEvent_t eb = collect ? h->ev_pool[2 * h->ev_cursor + 1] : h->ev_b;
  if (collect) h->ev_cursor++;
  if (!h->capturing) MMM_CUDA(h, cudaEventRecord(ea, h->stream));
  // a converged minimisation skips every kernel (d_skip): the counter still advances, harmless
  if (h->sort_age <= 0 || h->sort_age >= kResortEvery) {
    if ((rc = rebuild_order(h, d_skip))) return rc;
    h->sort_age = 0;
  }
  h->sort_age++;
  const int npad = (int)h->npad, ntiles = (int)h->ntiles, nstages = npad / MMM_STAGE;
  k_gather_sorted<<<(ntiles + 7) / 8, 256, 0, h->stream>>>(h->d_pos4, h->d_order, (int)h->n, npad, h->d_pos4_sorted,
                                                          h->d_soa_sorted, h->d_tiles_sorted, d_skip);
  k_stage_boxes<<<(nstages + 255) / 256, 256, 0, h->stream>>>(h->d_tiles_sorted, nstages, h->d_stage_boxes, d_skip);
  h->launches += 2;
  MMM_CUDA(h, cudaGetLastError());
  if ((rc = mmm_launch_pair_n3_cut(h, d_skip))) return rc;
  if (!h->capturing) MMM_CUDA(h, cudaEventRecord(eb, h->stream));
  return MMM_OK;
}

int mmm_cutoff_resort_period() { return kResortEvery; }
