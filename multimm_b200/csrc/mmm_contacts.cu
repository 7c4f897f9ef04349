// mmm_contacts.cu — contact counting at the handle's current positions (simulated Hi-C):
//   every unordered bead pair i < j with d2 < rc^2, decided in FP64 on the master positions d_x with
//   d2 = (dx*dx + dy*dy) + dz*dz rounded operation by operation (no FMA contraction), so that a numpy
//   evaluation of the same expression gives the same verdict for every pair, the boundary included.
// mmm_contacts counts them three ways with integer atomics (bit-identical however the work is scheduled):
// per (bin_i, bin_j) in a dense symmetric map, per index separation j - i for same-chromosome pairs
// (P(s)), and in total.  mmm_contacts_sparse stores the map sparse, for any int32 number of bins: the
// same kernel (k_contacts, sink kKeys) writes the key p * n_bins + q (p <= q) of every binned contact,
// an LSD radix sort over the significant bits orders them, and runs of equal keys become the entries.
//
// Culling is two-level over the chain-order tiles mmm_launch_prepare builds (32 beads, FP32 boxes of
// the centred copy): one warp per i-tile tests its box against 256-bead stage boxes, 32 stages at a time,
// then against the 8 tile boxes of every stage that survives, and runs the exact FP64 test over the
// 32 x 32 beads of every tile pair that survives.  The cut-off mode's Morton order is not used: rebuilding
// it at rc would change the handle's sorted state.  The pass writes only the FP32 copy (d_pos4, d_soa,
// d_tiles, which every evaluation rewrites from d_x before reading) and its own scratch.
//
// Sparse pass, per call (M = binned contacts, E = entries):
//   k_contacts<kTileCount>  binned contacts of every i-tile -> exclusive scan -> each warp's key offset
//   k_contacts<kKeys>       keys of warp a at [off_a, off_a+1): no atomics, deterministic order
//   k_rs_hist / scan / k_rs_scatter   LSD radix sort, 8-bit digits, ceil(log2(n_bins^2)) bits
//   k_rle<kCount>           heads (first key of a run) per 4096-key chunk -> scan -> E
// and in mmm_contacts_sparse_read, into the other sort buffer: k_rle<kVals> (run lengths), then
// k_rle<kSplit> (row = key / n_bins, col = key % n_bins of every head).
// Scratch: 2 x 8 B per binned contact (the two sort buffers; the read reuses the free one), a digit x
// chunk table of 8 B x 256 per 4096 keys, and O(N) for the per-tile offsets.
//
// The trajectory sampler (mmm_sampler.cu) runs the dense pass and the sparse pass through the same functions
// (mmm_contacts_dense_pass, mmm_contacts_sparse_pass) into its own buffers; its fine map adds
//   k_rle<kKeyVals>         sorted keys -> unique (key, count) list of the structure
//   k_merge_part, k_merge   merge-path merge with the accumulated (key, count) list
//   k_rle<kCount>, scan, k_rle<kKeyVals>   equal keys (at most two, adjacent) -> one entry, counts added
#include <math.h>

#include <algorithm>

#include "mmm_internal.cuh"

namespace {

constexpr int CT_WARPS = 8;                              // i-tiles per CTA
constexpr int CT_TILES_PER_STAGE = MMM_STAGE / MMM_TILE;  // 8
constexpr int CT_MAX_BINS = 4096;
constexpr int CS_THREADS = 256, CS_PER = 16, CS_CHUNK = CS_THREADS * CS_PER;  // sort / scan / run blocks: 4096 keys
constexpr int CS_DIGIT_BITS = 8, CS_DIGITS = 1 << CS_DIGIT_BITS;

// what k_contacts does with a contact: the dense map + P(s) + totals; the binned-contact count of the
// i-tile (sparse pass 1); the key of every binned contact at the tile's offset (sparse pass 2) + totals
enum CtSink { kDense, kTileCount, kKeys };

// Gap between [lo_a, hi_a] and [lo_b, hi_b], shrunk by 2^-20 of the largest coordinate involved.  An FP32
// coordinate of the centred copy is within 2^-24 |p| of the FP64 one and the subtraction adds 2^-24 of
// the result, so the shrunk gap is never larger than the FP64 |dx| of any bead pair of the two boxes.
__device__ __forceinline__ float ct_gap(float lo_a, float hi_a, float lo_b, float hi_b) {
  const float g = fmaxf(fmaxf(lo_b - hi_a, lo_a - hi_b), 0.0f);
  const float m = fmaxf(fmaxf(fabsf(lo_a), fabsf(hi_a)), fmaxf(fabsf(lo_b), fabsf(hi_b)));
  return fmaxf(g - m * 0x1p-20f, 0.0f);
}

// true unless no bead pair of the two boxes can be within rc; rcm2 = rc^2 (1 + 2^-16) covers the
// rounding of the FP32 sum of squares (a few 2^-24) and of rc^2 itself
__device__ __forceinline__ bool ct_near(const TileInfo& a, const TileInfo& b, float rcm2) {
  const float gx = ct_gap(a.lox, a.hix, b.lox, b.hix);
  const float gy = ct_gap(a.loy, a.hiy, b.loy, b.hiy);
  const float gz = ct_gap(a.loz, a.hiz, b.loz, b.hiz);
  return gx * gx + gy * gy + gz * gz <= rcm2;
}

// stage box = union of the boxes of its real tiles (an all-padding tile sits at the pad point)
__global__ void __launch_bounds__(256) k_ct_stage_boxes(const TileInfo* __restrict__ tiles, int ntr, int nst,
                                                        TileInfo* __restrict__ stages) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nst) return;
  TileInfo b = tiles[s * CT_TILES_PER_STAGE];
  for (int k = 1; k < CT_TILES_PER_STAGE; ++k) {
    const int t = s * CT_TILES_PER_STAGE + k;
    if (t >= ntr) break;
    const TileInfo o = tiles[t];
    b.lox = fminf(b.lox, o.lox); b.loy = fminf(b.loy, o.loy); b.loz = fminf(b.loz, o.loz);
    b.hix = fmaxf(b.hix, o.hix); b.hiy = fmaxf(b.hiy, o.hiy); b.hiz = fmaxf(b.hiz, o.hiz);
  }
  stages[s] = b;
}

// One warp per i-tile a; j-tiles b >= a.  Lane l holds bead i = 32 a + l; the beads of the current j-tile
// are staged in shared memory and read as broadcasts.  kDense: map increments are aggregated over the lanes
// that hit the same bin pair in the same step (consecutive i-beads mostly share a bin).  kTileCount /
// kKeys see the same candidates in the same order, so pass 2 writes exactly the keys pass 1 counted.
template <CtSink kSink>
__global__ void __launch_bounds__(CT_WARPS * 32) k_contacts(
    const double* __restrict__ x, const int* __restrict__ type, const int* __restrict__ bin,
    const TileInfo* __restrict__ tiles, const TileInfo* __restrict__ stages, int n, int ntr, int nst, double rc2,
    float rcm2, int nbins, unsigned long long* __restrict__ map, unsigned long long* __restrict__ sep,
    unsigned long long* __restrict__ counts, long long* __restrict__ tile_keys,
    unsigned long long* __restrict__ keys) {
  __shared__ double s_x[CT_WARPS][3][32];
  __shared__ int s_bin[CT_WARPS][32], s_chr[CT_WARPS][32];
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int a = blockIdx.x * CT_WARPS + w;
  if (a >= ntr) return;  // whole warps only; no CTA-wide barrier below
  const int i = a * MMM_TILE + lane;
  const bool ireal = i < n;
  double xi = 0.0, yi = 0.0, zi = 0.0;
  int bi = -1, ci = -1;
  if (ireal) {
    xi = x[3 * (size_t)i]; yi = x[3 * (size_t)i + 1]; zi = x[3 * (size_t)i + 2];
    bi = bin ? bin[i] : -1;
    ci = (type[i] >> 8) & 0xFFFF;
  }
  const TileInfo A = tiles[a];
  unsigned long long npairs = 0, ncand = 0;
  long long kpos = kSink == kKeys ? tile_keys[a] : 0;  // next key slot of this warp (warp-uniform)
  for (int t0 = a / CT_TILES_PER_STAGE; t0 < nst; t0 += 32) {
    const int t = t0 + lane;
    unsigned sm = __ballot_sync(full, t < nst && ct_near(A, stages[t], rcm2));
    while (sm) {
      const int ts = t0 + __ffs(sm) - 1;
      sm &= sm - 1;
      const int b = ts * CT_TILES_PER_STAGE + lane;
      unsigned bm = __ballot_sync(full, lane < CT_TILES_PER_STAGE && b >= a && b < ntr && ct_near(A, tiles[b], rcm2));
      while (bm) {
        const int tb = ts * CT_TILES_PER_STAGE + __ffs(bm) - 1;
        bm &= bm - 1;
        const int j = tb * MMM_TILE + lane;
        __syncwarp();
        if (j < n) {
          s_x[w][0][lane] = x[3 * (size_t)j];
          s_x[w][1][lane] = x[3 * (size_t)j + 1];
          s_x[w][2][lane] = x[3 * (size_t)j + 2];
          s_bin[w][lane] = bin ? bin[j] : -1;
          if (kSink == kDense) s_chr[w][lane] = (type[j] >> 8) & 0xFFFF;
        }
        __syncwarp();
        const int jn = min(MMM_TILE, n - tb * MMM_TILE);
        const int jstart = tb == a ? lane + 1 : 0;  // i < j inside the diagonal tile
        if (ireal && jn > jstart) ncand += (unsigned long long)(jn - jstart);
        for (int jj = 0; jj < jn; ++jj) {  // every lane runs every step: the votes below see the whole warp
          const double d2 = mmm_pair_d2(xi, yi, zi, s_x[w][0][jj], s_x[w][1][jj], s_x[w][2][jj]);
          const bool hit = ireal && jj >= jstart && d2 < rc2;
          if (!__any_sync(full, hit)) continue;
          const int bj = s_bin[w][jj];
          if constexpr (kSink == kDense) {
            if (hit) {
              ++npairs;
              if (sep && ci == s_chr[w][jj]) atomicAdd(&sep[tb * MMM_TILE + jj - i], 1ull);
            }
            if (map) {
              const int key = hit && bi >= 0 && bj >= 0 ? bi * nbins + bj : -1;
              const unsigned grp = __match_any_sync(full, key);
              if (key >= 0 && lane == __ffs(grp) - 1) {
                const unsigned long long c = (unsigned long long)__popc(grp);
                atomicAdd(&map[(size_t)key], c);
                if (bi != bj) atomicAdd(&map[(size_t)bj * nbins + bi], c);
              }
            }
          } else {
            if (hit) ++npairs;
            const bool binned = hit && bi >= 0 && bj >= 0;
            const unsigned em = __ballot_sync(full, binned);
            if (kSink == kKeys && binned) {
              const unsigned p = (unsigned)min(bi, bj), q = (unsigned)max(bi, bj);
              keys[kpos + __popc(em & ((1u << lane) - 1u))] = (unsigned long long)p * (unsigned)nbins + q;
            }
            kpos += __popc(em);
          }
        }
      }
    }
  }
  if constexpr (kSink == kTileCount) {
    if (lane == 0) tile_keys[a] = kpos;
  } else {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      npairs += __shfl_xor_sync(full, npairs, o);
      ncand += __shfl_xor_sync(full, ncand, o);
    }
    if (lane == 0) {
      atomicAdd(&counts[0], npairs);
      atomicAdd(&counts[1], ncand);
    }
  }
}

// ---- exclusive scan of an int64 array of any length, in place; the total lands in part[nparts] ----------
// (nparts = ceil(len / CS_CHUNK); part holds nparts + 1 entries)
__device__ __forceinline__ long long cs_block_exclusive(long long v, long long* s_warp, long long* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  long long inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) s_warp[w] = inc;
  __syncthreads();
  long long before = 0, all = 0;
  for (int k = 0; k < CS_THREADS / 32; ++k) {
    if (k < w) before += s_warp[k];
    all += s_warp[k];
  }
  __syncthreads();  // s_warp is reused by the next call
  *total = all;
  return before + inc - v;
}

__global__ void __launch_bounds__(CS_THREADS) k_scan_parts(const long long* __restrict__ a, long long len,
                                                           long long* __restrict__ part) {
  __shared__ long long s_warp[CS_THREADS / 32];
  const long long base = (long long)blockIdx.x * CS_CHUNK + (long long)threadIdx.x * CS_PER;
  long long v = 0;
  for (int k = 0; k < CS_PER; ++k)
    if (base + k < len) v += a[base + k];
  long long total;
  cs_block_exclusive(v, s_warp, &total);
  if (threadIdx.x == 0) part[blockIdx.x] = total;
}

__global__ void __launch_bounds__(CS_THREADS) k_scan_top(long long* __restrict__ part, int nparts) {
  __shared__ long long s_warp[CS_THREADS / 32];
  long long carry = 0;
  for (int b0 = 0; b0 < nparts; b0 += CS_THREADS) {
    const int b = b0 + threadIdx.x;
    const long long v = b < nparts ? part[b] : 0;
    long long total;
    const long long ex = cs_block_exclusive(v, s_warp, &total);
    if (b < nparts) part[b] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) part[nparts] = carry;
}

__global__ void __launch_bounds__(CS_THREADS) k_scan_apply(long long* __restrict__ a, long long len,
                                                           const long long* __restrict__ part) {
  __shared__ long long s_warp[CS_THREADS / 32];
  const long long base = (long long)blockIdx.x * CS_CHUNK + (long long)threadIdx.x * CS_PER;
  long long v[CS_PER], sum = 0;
#pragma unroll
  for (int k = 0; k < CS_PER; ++k) {
    v[k] = base + k < len ? a[base + k] : 0;
    sum += v[k];
  }
  long long total;
  long long run = part[blockIdx.x] + cs_block_exclusive(sum, s_warp, &total);
#pragma unroll
  for (int k = 0; k < CS_PER; ++k) {
    if (base + k < len) a[base + k] = run;
    run += v[k];
  }
}

// ---- LSD radix sort of 64-bit keys, one pass = hist + scan + scatter ------------------------------------
// The table is digit-major (table[d * nblocks + b]), so that one flat exclusive scan gives every (digit,
// block) its first output slot.
__global__ void __launch_bounds__(CS_THREADS) k_rs_hist(const unsigned long long* __restrict__ keys, long long n,
                                                        int shift, long long* __restrict__ table, int nblocks) {
  __shared__ int s_cnt[CS_DIGITS];
  for (int d = threadIdx.x; d < CS_DIGITS; d += CS_THREADS) s_cnt[d] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * CS_CHUNK;
  for (int q = threadIdx.x; q < CS_CHUNK; q += CS_THREADS) {  // whole warps every round: match_any below
    const long long e = base + q;
    const int d = e < n ? (int)((keys[e] >> shift) & (CS_DIGITS - 1)) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (d >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_cnt[d], __popc(peers));
  }
  __syncthreads();
  for (int d = threadIdx.x; d < CS_DIGITS; d += CS_THREADS) table[(size_t)d * nblocks + blockIdx.x] = s_cnt[d];
}

// Stable scatter.  Warp w owns keys [w * 512, (w + 1) * 512) of the block's chunk and visits them in 16
// rounds of 32 consecutive keys, so (round, lane) order is the key order.  Per round the lanes with equal
// digits find each other with match_any; the lowest of them advances the warp's counter of that digit.
__global__ void __launch_bounds__(CS_THREADS) k_rs_scatter(const unsigned long long* __restrict__ keys_in, long long n,
                                                           int shift, const long long* __restrict__ table, int nblocks,
                                                           unsigned long long* __restrict__ keys_out) {
  constexpr int kWarps = CS_THREADS / 32;
  __shared__ int s_cnt[kWarps][CS_DIGITS];
  __shared__ long long s_base[CS_DIGITS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int d = threadIdx.x; d < kWarps * CS_DIGITS; d += CS_THREADS) (&s_cnt[0][0])[d] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * CS_CHUNK + warp * (CS_CHUNK / kWarps);
  unsigned long long key[CS_PER];
  int rank[CS_PER];
#pragma unroll
  for (int r = 0; r < CS_PER; ++r) {
    const long long e = base + r * 32 + lane;
    const bool have = e < n;
    key[r] = have ? keys_in[e] : 0ull;
    const int d = have ? (int)((key[r] >> shift) & (CS_DIGITS - 1)) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int before = __popc(peers & ((1u << lane) - 1u));
    int old = 0;
    if (have && before == 0) {
      old = s_cnt[warp][d];
      s_cnt[warp][d] = old + __popc(peers);
    }
    old = __shfl_sync(0xffffffffu, old, __ffs(peers) - 1);
    rank[r] = have ? old + before : -1;
    __syncwarp();
  }
  __syncthreads();
  for (int d = threadIdx.x; d < CS_DIGITS; d += CS_THREADS) {  // exclusive prefix over the warps, per digit
    int run = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      const int c = s_cnt[w][d];
      s_cnt[w][d] = run;
      run += c;
    }
    s_base[d] = table[(size_t)d * nblocks + blockIdx.x];
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < CS_PER; ++r) {
    if (rank[r] < 0) continue;
    const int d = (int)((key[r] >> shift) & (CS_DIGITS - 1));
    keys_out[s_base[d] + s_cnt[warp][d] + rank[r]] = key[r];
  }
}

// ---- runs of equal sorted keys -> entries -------------------------------------------------------------
// Thread t of block b owns keys [b * 4096 + 16 t, + 16); a head is a key unlike its predecessor, and entry
// e(k) of key k = (heads at or before k) - 1.  kCount: heads of the chunk -> cnt[b].  kVals: vals[e] +=
// the weight of every piece of a run the thread holds, a key weighing in_vals[k] (1 when in_vals is NULL;
// integer atomics: exact in any order; vals zeroed).  kKeyVals: kVals, and out_keys[e] = key at every head
// (a sorted, unique (key, value) list).  kSplit: rows[e] = key / n_bins, cols[e] = key % n_bins at every
// head.  off = the scanned kCount output.
enum RleMode { kCount, kVals, kKeyVals, kSplit };
template <RleMode kMode>
__global__ void __launch_bounds__(CS_THREADS) k_rle(const unsigned long long* __restrict__ keys, long long n,
                                                    long long* __restrict__ cnt, const long long* __restrict__ off,
                                                    unsigned nbins, const unsigned long long* __restrict__ in_vals,
                                                    unsigned long long* __restrict__ vals,
                                                    unsigned long long* __restrict__ out_keys, int* __restrict__ rows,
                                                    int* __restrict__ cols) {
  __shared__ long long s_warp[CS_THREADS / 32];
  const long long base = (long long)blockIdx.x * CS_CHUNK + (long long)threadIdx.x * CS_PER;
  unsigned long long prev = base > 0 && base - 1 < n ? keys[base - 1] : ~0ull;  // no key is ~0 (< 2^62)
  unsigned long long k[CS_PER];
  long long heads = 0;
#pragma unroll
  for (int q = 0; q < CS_PER; ++q) {
    k[q] = base + q < n ? keys[base + q] : prev;  // past the end: a repeat, never a head
    heads += (base + q < n && k[q] != (q ? k[q - 1] : prev)) ? 1 : 0;
  }
  long long total;
  const long long before = cs_block_exclusive(heads, s_warp, &total);
  if constexpr (kMode == kCount) {
    if (threadIdx.x == 0) cnt[blockIdx.x] = total;
    return;
  }
  constexpr bool kSum = kMode == kVals || kMode == kKeyVals;
  long long e = off[blockIdx.x] + before - 1;  // entry of the key before this thread's first
  unsigned long long len = 0;
#pragma unroll
  for (int q = 0; q < CS_PER; ++q) {
    if (base + q >= n) break;
    if (k[q] != (q ? k[q - 1] : prev)) {
      if (kSum && len) atomicAdd(&vals[e], len);
      ++e;
      len = 0;
      if (kMode == kKeyVals) out_keys[e] = k[q];
      if (kMode == kSplit) {
        rows[e] = (int)(k[q] / nbins);
        cols[e] = (int)(k[q] % nbins);
      }
    }
    if (kSum) len += in_vals ? in_vals[base + q] : 1ull;
  }
  if (kSum && len) atomicAdd(&vals[e], len);
}

// ---- merge of two sorted (key, value) lists (the trajectory sampler's fine map) -------------------------
// Merge path: output position d of the merge of A (na keys) and B (nb keys) takes i keys from A and d - i
// from B, i the smallest with A[i] > B[d - 1 - i] (A first among equal keys).  k_merge_part finds i at the
// first output of every CTA; k_merge stages the CTA's slices of A and B in shared memory, and each thread
// finds its own diagonal there and merges MG_PER outputs.  Keys are unique within each list, so a key
// appears at most twice in the output, adjacent; k_rle<kKeyVals> then adds the two values.
constexpr int MG_THREADS = 256, MG_PER = 8, MG_TILE = MG_THREADS * MG_PER;

__device__ __forceinline__ long long mg_diag(const unsigned long long* a, long long na, const unsigned long long* b,
                                             long long nb, long long d) {
  long long lo = d > nb ? d - nb : 0, hi = d < na ? d : na;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (a[mid] <= b[d - 1 - mid]) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256) k_merge_part(const unsigned long long* __restrict__ a, long long na,
                                                    const unsigned long long* __restrict__ b, long long nb, int nparts,
                                                    long long* __restrict__ part) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p > nparts) return;
  const long long d = (long long)p * MG_TILE;
  part[p] = mg_diag(a, na, b, nb, d < na + nb ? d : na + nb);
}

__global__ void __launch_bounds__(MG_THREADS) k_merge(const unsigned long long* __restrict__ akey,
                                                      const unsigned long long* __restrict__ aval, long long na,
                                                      const unsigned long long* __restrict__ bkey,
                                                      const unsigned long long* __restrict__ bval, long long nb,
                                                      const long long* __restrict__ part,
                                                      unsigned long long* __restrict__ okey,
                                                      unsigned long long* __restrict__ oval) {
  __shared__ unsigned long long s_key[MG_TILE], s_val[MG_TILE];
  const long long d0 = (long long)blockIdx.x * MG_TILE, d1 = d0 + MG_TILE < na + nb ? d0 + MG_TILE : na + nb;
  const long long a0 = part[blockIdx.x], a1 = part[blockIdx.x + 1];
  const int la = (int)(a1 - a0), lb = (int)((d1 - a1) - (d0 - a0));
  for (int t = threadIdx.x; t < la + lb; t += MG_THREADS) {  // A's slice, then B's
    const long long g = t < la ? a0 + t : d0 - a0 + (t - la);
    s_key[t] = t < la ? akey[g] : bkey[g];
    s_val[t] = t < la ? aval[g] : bval[g];
  }
  __syncthreads();
  const int d = min((int)threadIdx.x * MG_PER, la + lb);
  int i = (int)mg_diag(s_key, la, s_key + la, lb, d), j = d - i;
  for (int q = 0; q < MG_PER && d + q < la + lb; ++q) {
    const bool take_a = i < la && (j >= lb || s_key[i] <= s_key[la + j]);
    const int s = take_a ? i++ : la + j++;
    okey[d0 + d + q] = s_key[s];
    oval[d0 + d + q] = s_val[s];
  }
}

}  // namespace

// exclusive scan of a[0, len) in place; part: ceil(len / CS_CHUNK) + 1 entries, the last receives the total
void cs_scan(mmm_system* h, long long* a, long long len, long long* part) {
  const int nparts = (int)std::max<long long>(1, (len + CS_CHUNK - 1) / CS_CHUNK);
  k_scan_parts<<<nparts, CS_THREADS, 0, h->stream>>>(a, len, part);
  k_scan_top<<<1, CS_THREADS, 0, h->stream>>>(part, nparts);
  k_scan_apply<<<nparts, CS_THREADS, 0, h->stream>>>(a, len, part);
  h->launches += 3;
}

long long cs_blocks(long long nkeys) { return std::max<long long>(1, (nkeys + CS_CHUNK - 1) / CS_CHUNK); }
// sort table (digit x chunk) followed by the partial sums of its scan
size_t cs_table_len(long long nkeys) { return (size_t)(CS_DIGITS * cs_blocks(nkeys)) * 17 / 16 + 2; }

int cs_key_bits(unsigned long long kmax) {
  int bits = 0;
  while (bits < 64 && (kmax >> bits)) ++bits;
  return bits;
}

long long* cs_run_total(long long* table, long long nkeys) {
  const long long nblocks = cs_blocks(nkeys);
  return table + nblocks + cs_blocks(nblocks);
}

int cs_sort_runs(mmm_system* h, DevBuf<unsigned long long>* keys, long long m, int bits, long long* table) {
  const int nblocks = (int)cs_blocks(m);
  long long* table_part = table + (size_t)CS_DIGITS * nblocks;
  int src = 0;
  for (int shift = 0; shift < bits; shift += CS_DIGIT_BITS) {
    k_rs_hist<<<nblocks, CS_THREADS, 0, h->stream>>>(keys[src], m, shift, table, nblocks);
    cs_scan(h, table, (long long)CS_DIGITS * nblocks, table_part);
    k_rs_scatter<<<nblocks, CS_THREADS, 0, h->stream>>>(keys[src], m, shift, table, nblocks, keys[1 - src]);
    h->launches += 2;
    src = 1 - src;
  }
  // entries: heads per chunk -> offsets (the first nblocks slots of the table, kept for the read)
  k_rle<kCount><<<nblocks, CS_THREADS, 0, h->stream>>>(keys[src], m, table, nullptr, 0u, nullptr, nullptr, nullptr,
                                                       nullptr, nullptr);
  h->launches++;
  cs_scan(h, table, nblocks, table + nblocks);
  return src;
}

namespace {

// the argument checks of mmm_contacts and mmm_contacts_sparse (max_bins: 4096 for the dense map)
int ct_check_args(mmm_system* h, const char* who, double rc_nm, const int32_t* bin_of_bead, int32_t n_bins, int max_bins,
             bool need_bins) {
  if (!(rc_nm > 0.0) || !isfinite(rc_nm)) return mmm_fail(h, MMM_ERR_ARG, std::string(who) + ": rc must be finite and > 0");
  if (n_bins < 1 || n_bins > max_bins)
    return mmm_fail(h, MMM_ERR_ARG, std::string(who) + (max_bins == CT_MAX_BINS ? ": n_bins must be in [1, 4096]"
                                                                              : ": n_bins must be >= 1"));
  if (need_bins && !bin_of_bead) return mmm_fail(h, MMM_ERR_ARG, std::string(who) + ": a map needs bin_of_bead");
  if (bin_of_bead)
    for (int64_t i = 0; i < h->n; ++i)
      if (bin_of_bead[i] < -1 || bin_of_bead[i] >= n_bins)
        return mmm_fail(h, MMM_ERR_ARG, std::string(who) + ": bin id outside [-1, n_bins)");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

}  // namespace

// The dense pass: contacts at the current positions added into map (n_bins^2; NULL: none, and then d_bin may
// be NULL), sep (n) and cnt[2] (contacts, candidates), which are zeroed first when clear.  ev0 (may be NULL)
// is recorded after the clearing.  mmm_contacts and the trajectory sampler run it.
int mmm_contacts_dense_pass(mmm_system* h, double rc_nm, const int* d_bin, int32_t n_bins, unsigned long long* map,
                            unsigned long long* sep, unsigned long long* cnt, bool clear, cudaEvent_t ev0) {
  const int n = (int)h->n;
  const int ntr = (n + MMM_TILE - 1) / MMM_TILE;                    // tiles holding a real bead
  const int nst = (ntr + CT_TILES_PER_STAGE - 1) / CT_TILES_PER_STAGE;  // stages holding a real tile
  int rc;
  if ((rc = mmm_reserve(h, h->d_ct_stage, (size_t)nst, "contact stage boxes"))) return rc;
  if (clear) {
    if (map)
      MMM_CUDA(h, cudaMemsetAsync(map, 0, sizeof(unsigned long long) * (size_t)n_bins * (size_t)n_bins, h->stream));
    if (sep) MMM_CUDA(h, cudaMemsetAsync(sep, 0, sizeof(unsigned long long) * (size_t)n, h->stream));
    MMM_CUDA(h, cudaMemsetAsync(cnt, 0, sizeof(unsigned long long) * 2, h->stream));
  }
  if (ev0) MMM_CUDA(h, cudaEventRecord(ev0, h->stream));
  if ((rc = mmm_launch_prepare(h, nullptr))) return rc;  // d_x -> FP32 copy and its tile boxes
  k_ct_stage_boxes<<<(nst + 255) / 256, 256, 0, h->stream>>>(h->d_tiles, ntr, nst, h->d_ct_stage);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  const float rcm2 = (float)(rc_nm * rc_nm) * (1.0f + 0x1p-16f);
  k_contacts<kDense><<<(ntr + CT_WARPS - 1) / CT_WARPS, CT_WARPS * 32, 0, h->stream>>>(
      h->d_x, h->d_type, map ? d_bin : nullptr, h->d_tiles, h->d_ct_stage, n, ntr, nst, rc_nm * rc_nm, rcm2, n_bins, map,
      sep, cnt, nullptr, nullptr);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}

// The sparse pass up to the run count: the key of every binned contact, radix-sorted into keys[out->src], and
// table[0, nblocks) = the first entry of every 4096-key chunk.  tile, keys and table are grown as needed;
// cnt[2] (device) is cleared before ev0 and holds contacts and candidates after ev1 (either event may be NULL).  One host
// synchronisation for the key count, one for the entry count.
int mmm_contacts_sparse_pass(mmm_system* h, double rc_nm, const int* d_bin, int32_t n_bins, DevBuf<long long>& tile,
                             DevBuf<unsigned long long>* keys, DevBuf<long long>& table, unsigned long long* cnt,
                             cudaEvent_t ev0, cudaEvent_t ev1, CsSorted* out) {
  const int n = (int)h->n;
  const int ntr = (n + MMM_TILE - 1) / MMM_TILE;
  const int nst = (ntr + CT_TILES_PER_STAGE - 1) / CT_TILES_PER_STAGE;
  int rc;
  if ((rc = mmm_reserve(h, h->d_ct_stage, (size_t)nst, "contact stage boxes")) ||
      (rc = mmm_reserve(h, tile, (size_t)ntr + cs_blocks(ntr) + 1, "contact tile counts")))  // counts, then scan parts
    return rc;
  long long* tile_part = tile + ntr;
  MMM_CUDA(h, cudaMemsetAsync(cnt, 0, sizeof(unsigned long long) * 2, h->stream));
  if (ev0) MMM_CUDA(h, cudaEventRecord(ev0, h->stream));
  if ((rc = mmm_launch_prepare(h, nullptr))) return rc;
  k_ct_stage_boxes<<<(nst + 255) / 256, 256, 0, h->stream>>>(h->d_tiles, ntr, nst, h->d_ct_stage);
  const float rcm2 = (float)(rc_nm * rc_nm) * (1.0f + 0x1p-16f);
  const int ctas = (ntr + CT_WARPS - 1) / CT_WARPS;
  k_contacts<kTileCount><<<ctas, CT_WARPS * 32, 0, h->stream>>>(
      h->d_x, h->d_type, d_bin, h->d_tiles, h->d_ct_stage, n, ntr, nst, rc_nm * rc_nm, rcm2, n_bins, nullptr,
      nullptr, nullptr, tile, nullptr);
  h->launches += 2;
  cs_scan(h, tile, ntr, tile_part);
  MMM_CUDA(h, cudaGetLastError());
  long long m = 0;  // binned contacts = keys
  MMM_CUDA(h, cudaMemcpyAsync(&m, tile_part + cs_blocks(ntr), sizeof(m), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  // grown to exactly this call's keys when they do not fit
  if ((rc = mmm_reserve(h, keys[0], (size_t)m, "contact keys")) ||
      (rc = mmm_reserve(h, keys[1], (size_t)m, "contact keys")) ||
      (rc = mmm_reserve(h, table, cs_table_len(m), "contact sort table")))
    return rc;
  long long* tab = table;
  k_contacts<kKeys><<<ctas, CT_WARPS * 32, 0, h->stream>>>(
      h->d_x, h->d_type, d_bin, h->d_tiles, h->d_ct_stage, n, ntr, nst, rc_nm * rc_nm, rcm2, n_bins, nullptr,
      nullptr, cnt, tile, keys[0]);
  h->launches++;
  // keys < n_bins^2: sort on ceil(log2(n_bins^2)) bits, 8 per pass
  const int bits = cs_key_bits((unsigned long long)n_bins * (unsigned long long)n_bins - 1ull);
  int src = 0;
  if (m > 0) src = cs_sort_runs(h, keys, m, bits, tab);
  MMM_CUDA(h, cudaGetLastError());
  if (ev1) MMM_CUDA(h, cudaEventRecord(ev1, h->stream));
  long long entries = 0;
  MMM_CUDA(h, cudaMemcpyAsync(out->cnt, cnt, sizeof(out->cnt), cudaMemcpyDeviceToHost, h->stream));
  if (m > 0)
    MMM_CUDA(h, cudaMemcpyAsync(&entries, cs_run_total(tab, m), sizeof(entries), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  out->keys = m;
  out->entries = entries;
  out->src = src;
  return MMM_OK;
}

// Capacity for n entries of a list that grows by a few per cent a sample (the accumulated fine map): n rounded
// up to the next of eight steps per power of two, so that the buffers are reallocated every ~12 % of growth
// rather than at every sample.
static size_t sp_capacity(long long n) {
  size_t step = 1;
  while (step * 16 <= (size_t)n) step <<= 1;
  return ((size_t)n + step - 1) / step * step;
}

// Adds the sorted keys[0, m) to the list acc: the runs of equal keys (off: their offsets per 4096-key chunk, as
// cs_sort_runs leaves them; entries of them) become a sorted unique (key, count) list in spare (>= entries
// slots) and acc.sval, which is merged with acc's entries [0] into [1], and equal keys (at most two, adjacent)
// are added back into [0].  Work and memory O(acc.n + entries).
int mmm_list_accumulate(mmm_system* h, const unsigned long long* keys, long long m, const long long* off,
                        long long entries, unsigned long long* spare, KeyCountList& acc) {
  const long long nb = entries, na = acc.n, nm = na + nb;
  if (nb == 0) return MMM_OK;
  int rc;
  if ((rc = mmm_reserve(h, acc.sval, sp_capacity(nb), "sorted list counts")) ||
      (rc = mmm_reserve(h, acc.key[1], sp_capacity(nm), "sorted list keys")) ||
      (rc = mmm_reserve(h, acc.val[1], sp_capacity(nm), "sorted list counts")))
    return rc;
  MMM_CUDA(h, cudaMemsetAsync(acc.sval, 0, sizeof(unsigned long long) * (size_t)nb, h->stream));
  k_rle<kKeyVals><<<(int)cs_blocks(m), CS_THREADS, 0, h->stream>>>(keys, m, nullptr, off, 0u, nullptr, acc.sval, spare,
                                                                   nullptr, nullptr);
  const int nparts = (int)((nm + MG_TILE - 1) / MG_TILE);
  const long long nchunks = cs_blocks(nm);
  if ((rc = mmm_reserve(h, acc.part, sp_capacity(std::max<long long>(nparts + 1, nchunks + cs_blocks(nchunks) + 1)),
                        "sorted list merge table")))
    return rc;
  long long* part = acc.part;
  k_merge_part<<<(nparts + 1 + 255) / 256, 256, 0, h->stream>>>(acc.key[0], na, spare, nb, nparts, part);
  k_merge<<<nparts, MG_THREADS, 0, h->stream>>>(acc.key[0], acc.val[0], na, spare, acc.sval, nb, part, acc.key[1],
                                                acc.val[1]);
  // equal keys -> one entry: heads per chunk, their offsets, then keys and summed counts
  k_rle<kCount><<<(int)nchunks, CS_THREADS, 0, h->stream>>>(acc.key[1], nm, part, nullptr, 0u, nullptr, nullptr,
                                                            nullptr, nullptr, nullptr);
  h->launches += 4;
  cs_scan(h, part, nchunks, part + nchunks);
  MMM_CUDA(h, cudaGetLastError());
  long long ne = 0;
  MMM_CUDA(h, cudaMemcpyAsync(&ne, part + nchunks + cs_blocks(nchunks), sizeof(ne), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if ((rc = mmm_reserve(h, acc.key[0], sp_capacity(ne), "sorted list keys")) ||
      (rc = mmm_reserve(h, acc.val[0], sp_capacity(ne), "sorted list counts")))
    return rc;
  MMM_CUDA(h, cudaMemsetAsync(acc.val[0], 0, sizeof(unsigned long long) * (size_t)ne, h->stream));
  k_rle<kKeyVals><<<(int)nchunks, CS_THREADS, 0, h->stream>>>(acc.key[1], nm, nullptr, part, 0u, acc.val[1], acc.val[0],
                                                              acc.key[0], nullptr, nullptr);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  acc.n = ne;
  return MMM_OK;
}

// The trajectory sampler's fine map: this structure's sparse map added to the accumulated list h->sp_fine.
int mmm_contacts_fine_accumulate(mmm_system* h) {
  CsSorted srt;
  int rc = mmm_contacts_sparse_pass(h, h->sp_rc, h->d_sp_fine_bin, h->sp_fine_bins, h->d_sp_tile, h->d_sp_keys,
                                    h->d_sp_table, h->d_sp_cnt + 2, nullptr, nullptr, &srt);
  if (rc) return rc;
  // the spare sort buffer (free after the sort, keys >= entries slots) takes this structure's list
  return mmm_list_accumulate(h, h->d_sp_keys[srt.src], srt.keys, h->d_sp_table, srt.entries,
                             h->d_sp_keys[1 - srt.src], h->sp_fine);
}

namespace {
// rows[e] = key / n_bins, cols[e] = key % n_bins of the sampler's fine entries
__global__ void __launch_bounds__(256) k_split_keys(const unsigned long long* __restrict__ keys, long long n,
                                                    unsigned nbins, int* __restrict__ rows, int* __restrict__ cols) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  rows[e] = (int)(keys[e] / nbins);
  cols[e] = (int)(keys[e] % nbins);
}
}  // namespace

int mmm_contacts_fine_read(mmm_system* h, int32_t* rows_out, int32_t* cols_out, uint64_t* vals_out) {
  const long long e = h->sp_fine.n;
  if (e == 0) return MMM_OK;
  if (vals_out)
    MMM_CUDA(h, cudaMemcpyAsync(vals_out, h->sp_fine.val[0], sizeof(uint64_t) * (size_t)e, cudaMemcpyDeviceToHost,
                                h->stream));
  if (rows_out || cols_out) {  // rows then cols as int32 in the free merge buffer (>= e slots of 8 B)
    int* rows = reinterpret_cast<int*>(h->sp_fine.key[1].get());
    int* cols = rows + e;
    k_split_keys<<<(unsigned)((e + 255) / 256), 256, 0, h->stream>>>(h->sp_fine.key[0], e, (unsigned)h->sp_fine_bins,
                                                                      rows, cols);
    h->launches++;
    MMM_CUDA(h, cudaGetLastError());
    if (rows_out) MMM_CUDA(h, cudaMemcpyAsync(rows_out, rows, sizeof(int32_t) * (size_t)e, cudaMemcpyDeviceToHost, h->stream));
    if (cols_out) MMM_CUDA(h, cudaMemcpyAsync(cols_out, cols, sizeof(int32_t) * (size_t)e, cudaMemcpyDeviceToHost, h->stream));
  }
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

extern "C" int mmm_contacts(mmm_handle h, double rc_nm, const int32_t* bin_of_bead, int32_t n_bins, uint64_t* map_out,
                            uint64_t* sep_out, int64_t* pairs_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = ct_check_args(h, "mmm_contacts", rc_nm, bin_of_bead, n_bins, CT_MAX_BINS, map_out != nullptr))) return rc;
  cudaSetDevice(h->device);
  const int n = (int)h->n;
  const bool want_map = map_out != nullptr;
  const size_t cells = (size_t)n_bins * (size_t)n_bins;
  // scratch lives as long as the handle and only grows (the map when a call needs a larger one), so
  // that a call does not synchronise the device while another handle minimises beside it
  if ((rc = mmm_reserve(h, h->d_ct_bin, (size_t)n, "contact bins")) ||
      (rc = mmm_reserve(h, h->d_ct_sep, (size_t)n, "contacts by separation")) ||
      (rc = mmm_reserve(h, h->d_ct_cnt, 2, "contact counters")) ||
      (want_map && (rc = mmm_reserve(h, h->d_ct_map, cells, "contact map"))))
    return rc;
  if (!h->ct_ev0) MMM_CUDA(h, cudaEventCreate(&h->ct_ev0));
  if (!h->ct_ev1) MMM_CUDA(h, cudaEventCreate(&h->ct_ev1));
  if (want_map)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_ct_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  if ((rc = mmm_contacts_dense_pass(h, rc_nm, h->d_ct_bin, n_bins, want_map ? h->d_ct_map.get() : nullptr,
                                    sep_out ? h->d_ct_sep.get() : nullptr, h->d_ct_cnt, true, h->ct_ev0)))
    return rc;
  MMM_CUDA(h, cudaEventRecord(h->ct_ev1, h->stream));
  unsigned long long cnt[2];
  MMM_CUDA(h, cudaMemcpyAsync(cnt, h->d_ct_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, h->stream));
  if (want_map)
    MMM_CUDA(h, cudaMemcpyAsync(map_out, h->d_ct_map, sizeof(uint64_t) * cells, cudaMemcpyDeviceToHost, h->stream));
  if (sep_out)
    MMM_CUDA(h, cudaMemcpyAsync(sep_out, h->d_ct_sep, sizeof(uint64_t) * (size_t)n, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (pairs_out) *pairs_out = (int64_t)cnt[0];
  h->ct_candidates = (int64_t)cnt[1];
  cudaEventElapsedTime(&h->ct_ms, h->ct_ev0, h->ct_ev1);
  return MMM_OK;
}

extern "C" int mmm_contacts_sparse(mmm_handle h, double rc_nm, const int32_t* bin_of_bead, int32_t n_bins,
                                   int64_t* n_entries_out, int64_t* pairs_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = ct_check_args(h, "mmm_contacts_sparse", rc_nm, bin_of_bead, n_bins, INT32_MAX, true))) return rc;
  cudaSetDevice(h->device);
  h->cs_valid = false;
  const int n = (int)h->n;
  if ((rc = mmm_reserve(h, h->d_ct_bin, (size_t)n, "contact bins")) ||
      (rc = mmm_reserve(h, h->d_ct_cnt, 2, "contact counters")))
    return rc;
  if (!h->ct_ev0) MMM_CUDA(h, cudaEventCreate(&h->ct_ev0));
  if (!h->ct_ev1) MMM_CUDA(h, cudaEventCreate(&h->ct_ev1));
  MMM_CUDA(h, cudaMemcpyAsync(h->d_ct_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  CsSorted srt;
  if ((rc = mmm_contacts_sparse_pass(h, rc_nm, h->d_ct_bin, n_bins, h->d_cs_tile, h->d_cs_keys, h->d_cs_table,
                                     h->d_ct_cnt, h->ct_ev0, h->ct_ev1, &srt)))
    return rc;
  h->cs_keys = srt.keys;
  h->cs_entries = srt.entries;
  h->cs_src = srt.src;
  h->cs_nbins = n_bins;
  h->cs_valid = true;
  if (n_entries_out) *n_entries_out = srt.entries;
  if (pairs_out) *pairs_out = (int64_t)srt.cnt[0];
  h->ct_candidates = (int64_t)srt.cnt[1];
  cudaEventElapsedTime(&h->ct_ms, h->ct_ev0, h->ct_ev1);
  return MMM_OK;
}

extern "C" int mmm_contacts_sparse_read(mmm_handle h, int32_t* rows_out, int32_t* cols_out, uint64_t* vals_out) {
  if (!h) return MMM_ERR_ARG;
  if (!h->cs_valid) return mmm_fail(h, MMM_ERR_STATE, "mmm_contacts_sparse_read: no mmm_contacts_sparse call to read");
  const long long m = h->cs_keys, e = h->cs_entries;
  if (e == 0) return MMM_OK;
  cudaSetDevice(h->device);
  const int nblocks = (int)cs_blocks(m);
  const unsigned long long* keys = h->d_cs_keys[h->cs_src];
  unsigned long long* spare = h->d_cs_keys[1 - h->cs_src];  // free after the sort; m >= e slots
  const long long* off = h->d_cs_table;
  if (vals_out) {
    MMM_CUDA(h, cudaMemsetAsync(spare, 0, sizeof(unsigned long long) * (size_t)e, h->stream));
    k_rle<kVals><<<nblocks, CS_THREADS, 0, h->stream>>>(keys, m, nullptr, off, 0u, nullptr, spare, nullptr, nullptr,
                                                        nullptr);
    h->launches++;
    MMM_CUDA(h, cudaGetLastError());
    MMM_CUDA(h, cudaMemcpyAsync(vals_out, spare, sizeof(uint64_t) * (size_t)e, cudaMemcpyDeviceToHost, h->stream));
  }
  if (rows_out || cols_out) {  // rows then cols as int32 in the same spare buffer (8 B per entry)
    int* rows = reinterpret_cast<int*>(spare);
    int* cols = rows + e;
    k_rle<kSplit><<<nblocks, CS_THREADS, 0, h->stream>>>(keys, m, nullptr, off, (unsigned)h->cs_nbins, nullptr, nullptr,
                                                         nullptr, rows, cols);
    h->launches++;
    MMM_CUDA(h, cudaGetLastError());
    if (rows_out) MMM_CUDA(h, cudaMemcpyAsync(rows_out, rows, sizeof(int32_t) * (size_t)e, cudaMemcpyDeviceToHost, h->stream));
    if (cols_out) MMM_CUDA(h, cudaMemcpyAsync(cols_out, cols, sizeof(int32_t) * (size_t)e, cudaMemcpyDeviceToHost, h->stream));
  }
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

extern "C" int mmm_contacts_stats(mmm_handle h, int64_t* candidates_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  if (candidates_out) *candidates_out = h->ct_candidates;
  if (device_ms_out) *device_ms_out = h->ct_ms;
  return MMM_OK;
}
