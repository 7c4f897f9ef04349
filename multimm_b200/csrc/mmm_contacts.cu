// mmm_contacts.cu — contact counting at the handle's current positions (simulated Hi-C):
//   every unordered bead pair i < j with d2 < rc^2, decided in FP64 on the master positions d_x with
//   d2 = (dx*dx + dy*dy) + dz*dz rounded operation by operation (no FMA contraction), so that a numpy
//   evaluation of the same expression gives the same verdict for every pair, the boundary included.
// Contacts are counted three ways with integer atomics (bit-identical however the work is scheduled):
// per (bin_i, bin_j) in a dense symmetric map, per index separation j - i for same-chromosome pairs
// (P(s)), and in total.
//
// Culling is two-level over the chain-order tiles mmm_launch_prepare builds (32 beads, FP32 boxes of
// the centred copy): one warp per i-tile tests its box against 256-bead stage boxes, 32 stages at a time,
// then against the 8 tile boxes of every stage that survives, and runs the exact FP64 test over the
// 32 x 32 beads of every tile pair that survives.  The cut-off mode's Morton order is not used: rebuilding
// it at rc would change the handle's sorted state.  The pass writes only the FP32 copy (d_pos4, d_soa,
// d_tiles, which every evaluation rewrites from d_x before reading) and its own scratch.
#include <math.h>

#include "mmm_internal.cuh"

namespace {

constexpr int CT_WARPS = 8;                              // i-tiles per CTA
constexpr int CT_TILES_PER_STAGE = MMM_STAGE / MMM_TILE;  // 8
constexpr int CT_MAX_BINS = 4096;

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
// are staged in shared memory and read as broadcasts.  Map increments are aggregated over the lanes that
// hit the same bin pair in the same step (consecutive i-beads mostly share a bin).
__global__ void __launch_bounds__(CT_WARPS * 32) k_contacts(
    const double* __restrict__ x, const int* __restrict__ type, const int* __restrict__ bin,
    const TileInfo* __restrict__ tiles, const TileInfo* __restrict__ stages, int n, int ntr, int nst, double rc2,
    float rcm2, int nbins, unsigned long long* __restrict__ map, unsigned long long* __restrict__ sep,
    unsigned long long* __restrict__ counts) {
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
          s_chr[w][lane] = (type[j] >> 8) & 0xFFFF;
        }
        __syncwarp();
        const int jn = min(MMM_TILE, n - tb * MMM_TILE);
        const int jstart = tb == a ? lane + 1 : 0;  // i < j inside the diagonal tile
        if (ireal && jn > jstart) ncand += (unsigned long long)(jn - jstart);
        for (int jj = 0; jj < jn; ++jj) {  // every lane runs every step: the votes below see the whole warp
          const double dx = __dadd_rn(xi, -s_x[w][0][jj]);
          const double dy = __dadd_rn(yi, -s_x[w][1][jj]);
          const double dz = __dadd_rn(zi, -s_x[w][2][jj]);
          const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
          const bool hit = ireal && jj >= jstart && d2 < rc2;
          if (!__any_sync(full, hit)) continue;
          const int bj = s_bin[w][jj];
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
        }
      }
    }
  }
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

// scratch that lives as long as the handle: allocated on the first call (the map when a larger one is
// needed), so that a call does not synchronise the device while another handle minimises beside it
template <typename T>
int ct_alloc(mmm_system* h, T** p, size_t count) {
  if (*p) return MMM_OK;
  cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
  if (e != cudaSuccess) {
    *p = nullptr;
    return mmm_fail(h, MMM_ERR_NOMEM, std::string("CUDA error: ") + cudaGetErrorString(e) + " (cudaMalloc, contacts)");
  }
  return MMM_OK;
}

}  // namespace

void mmm_contacts_free(mmm_system* h) {
  void* ptrs[] = {h->d_ct_bin, h->d_ct_map, h->d_ct_sep, h->d_ct_stage, h->d_ct_cnt};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  if (h->ct_ev0) cudaEventDestroy(h->ct_ev0);
  if (h->ct_ev1) cudaEventDestroy(h->ct_ev1);
  h->ct_ev0 = h->ct_ev1 = nullptr;
  h->d_ct_bin = nullptr; h->d_ct_map = nullptr; h->d_ct_sep = nullptr; h->d_ct_stage = nullptr; h->d_ct_cnt = nullptr;
  h->ct_map_cap = 0;
}

extern "C" int mmm_contacts(mmm_handle h, double rc_nm, const int32_t* bin_of_bead, int32_t n_bins, uint64_t* map_out,
                            uint64_t* sep_out, int64_t* pairs_out) {
  if (!h) return MMM_ERR_ARG;
  if (!(rc_nm > 0.0) || !isfinite(rc_nm)) return mmm_fail(h, MMM_ERR_ARG, "mmm_contacts: rc must be finite and > 0");
  if (n_bins < 1 || n_bins > CT_MAX_BINS)
    return mmm_fail(h, MMM_ERR_ARG, "mmm_contacts: n_bins must be in [1, 4096]");
  if (map_out && !bin_of_bead) return mmm_fail(h, MMM_ERR_ARG, "mmm_contacts: a map needs bin_of_bead");
  if (bin_of_bead)
    for (int64_t i = 0; i < h->n; ++i)
      if (bin_of_bead[i] < -1 || bin_of_bead[i] >= n_bins)
        return mmm_fail(h, MMM_ERR_ARG, "mmm_contacts: bin id outside [-1, n_bins)");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  cudaSetDevice(h->device);
  const int n = (int)h->n;
  const int ntr = (n + MMM_TILE - 1) / MMM_TILE;                    // tiles holding a real bead
  const int nst = (ntr + CT_TILES_PER_STAGE - 1) / CT_TILES_PER_STAGE;  // stages holding a real tile
  const bool want_map = map_out != nullptr;
  const size_t cells = (size_t)n_bins * (size_t)n_bins;
  int rc;
  if ((rc = ct_alloc(h, &h->d_ct_bin, (size_t)n))) return rc;
  if ((rc = ct_alloc(h, &h->d_ct_sep, (size_t)n))) return rc;
  if ((rc = ct_alloc(h, &h->d_ct_stage, (size_t)nst))) return rc;
  if ((rc = ct_alloc(h, &h->d_ct_cnt, 2))) return rc;
  if (!h->ct_ev0) MMM_CUDA(h, cudaEventCreate(&h->ct_ev0));
  if (!h->ct_ev1) MMM_CUDA(h, cudaEventCreate(&h->ct_ev1));
  if (want_map && h->ct_map_cap < cells) {
    if (h->d_ct_map) {
      MMM_CUDA(h, cudaStreamSynchronize(h->stream));
      cudaFree(h->d_ct_map);
      h->d_ct_map = nullptr;
    }
    if ((rc = ct_alloc(h, &h->d_ct_map, cells))) return rc;
    h->ct_map_cap = cells;
  }
  if (want_map) {
    MMM_CUDA(h, cudaMemcpyAsync(h->d_ct_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
    MMM_CUDA(h, cudaMemsetAsync(h->d_ct_map, 0, sizeof(unsigned long long) * cells, h->stream));
  }
  if (sep_out) MMM_CUDA(h, cudaMemsetAsync(h->d_ct_sep, 0, sizeof(unsigned long long) * (size_t)n, h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_ct_cnt, 0, sizeof(unsigned long long) * 2, h->stream));
  MMM_CUDA(h, cudaEventRecord(h->ct_ev0, h->stream));
  if ((rc = mmm_launch_prepare(h, nullptr))) return rc;  // d_x -> FP32 copy and its tile boxes
  k_ct_stage_boxes<<<(nst + 255) / 256, 256, 0, h->stream>>>(h->d_tiles, ntr, nst, h->d_ct_stage);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  const float rcm2 = (float)(rc_nm * rc_nm) * (1.0f + 0x1p-16f);
  k_contacts<<<(ntr + CT_WARPS - 1) / CT_WARPS, CT_WARPS * 32, 0, h->stream>>>(
      h->d_x, h->d_type, want_map ? h->d_ct_bin : nullptr, h->d_tiles, h->d_ct_stage, n, ntr, nst, rc_nm * rc_nm, rcm2,
      n_bins, want_map ? h->d_ct_map : nullptr, sep_out ? h->d_ct_sep : nullptr, h->d_ct_cnt);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
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

extern "C" int mmm_contacts_stats(mmm_handle h, int64_t* candidates_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  if (candidates_out) *candidates_out = h->ct_candidates;
  if (device_ms_out) *device_ms_out = h->ct_ms;
  return MMM_OK;
}
