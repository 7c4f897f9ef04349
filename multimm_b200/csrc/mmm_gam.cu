// mmm_gam.cu — simulated genome architecture mapping (GAM): random thin slices ("nuclear profiles") through a
// structure, and how often two genomic bins are found in the same slice (co-segregation), summed over structures.
// Slice k is the slab |s| <= h of the plane (n_k, o_k), with
//   s = ((n_x*x + n_y*y) + n_z*z) - o  (FP64, rounded operation by operation, no FMA contraction)
// so a numpy evaluation of the same expression gives the same bits; a bead exactly on the boundary is inside.  Bin
// p is detected in slice k when any bead of bin p lies in it (bin -1: left out).  Per add of S slices,
// counts[tri(p, q)] += #{k : p and q both detected in k} for p <= q (tri the row-major upper-triangle index), so
// the diagonal holds each bin's detections; slices += S, empty += #{k : no bin detected}.  Integer sums do not
// depend on order: bit-identical however the work is scheduled, and exact over adds, members and MD samples.
//
// Two passes per add:
//  * k_gam_detect, over beads x slice words: the planes of GM_WPB words (32 slices each) are staged in shared
//    memory; a lane tests its bead against the 32 slices of a word and builds a mask; lanes of equal bins are
//    grouped once (__match_any_sync) and their masks OR-reduced (__reduce_or_sync), and the group head ORs the
//    result into the bitset X[bin][word] with one atomicOr.  The warp's OR of all binned masks goes through
//    shared memory into any[word], so empty = S - popc(any) on the host.  X and any are cleared at the start of
//    every add, and bits >= S are never set.
//  * k_gam_coseg: the binary Gram matrix X X^T over bins by popc(a & b), on the upper triangle of 64 x 64 bin
//    tiles.  Chunks of GM_KW words of both row blocks are staged in shared memory; each thread owns a 4 x 4
//    micro-tile of uint32 sums (S <= 2^16, so a sum cannot overflow) and adds them to the uint64 triangle with a
//    plain load-add-store: every pair has exactly one owner.  This is POPC work that takes microseconds at the
//    default sizes; tcgen05 has no b1 kind, so tensor cores are not used.
//
// The passes read d_x and write only the accumulator's own buffers (planes, X, any, counts; the positions'
// check uses the bounding-box partials of mmm_positions_box): nothing an evaluation, a minimisation, an MD step
// or another readout reads.
#include <math.h>

#include <algorithm>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int GM_THREADS = 256;              // beads per detection CTA
constexpr int GM_WPB = 8;                    // slice words per detection CTA (256 planes in shared memory)
constexpr int GM_TILE = 64;                  // bins per side of a co-segregation tile
constexpr int GM_KW = 32;                    // words per staged chunk of the co-segregation pass
constexpr int32_t GM_MAX_SLICES = 65536;     // per add: a uint32 micro-tile sum stays below 2^32
constexpr int64_t GM_MAX_ROWS = 1 << 27;     // B (B + 1) / 2 uint64 sums: 1 GiB

__global__ void __launch_bounds__(GM_THREADS) k_gam_detect(const double* __restrict__ x, const int* __restrict__ bin,
                                                           int n, const double4* __restrict__ planes, int nslices,
                                                           int nwords, double half, unsigned* __restrict__ X,
                                                           unsigned* __restrict__ any) {
  __shared__ double4 s_pl[GM_WPB * 32];
  __shared__ unsigned s_any[GM_WPB];
  const int w0 = blockIdx.y * GM_WPB;
  const int nw = min(GM_WPB, nwords - w0);
  for (int k = threadIdx.x; k < GM_WPB * 32; k += blockDim.x) {
    const int s = w0 * 32 + k;
    s_pl[k] = s < nslices ? planes[s] : make_double4(0.0, 0.0, 0.0, 0.0);  // masked off below
  }
  if (threadIdx.x < GM_WPB) s_any[threadIdx.x] = 0u;
  __syncthreads();
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * GM_THREADS + threadIdx.x;
  double xi = 0.0, yi = 0.0, zi = 0.0;
  int b = -1;
  if (i < n) {
    xi = x[3 * (size_t)i];
    yi = x[3 * (size_t)i + 1];
    zi = x[3 * (size_t)i + 2];
    b = bin[i];
  }
  if (__any_sync(full, b >= 0)) {  // warp-uniform
    const unsigned grp = __match_any_sync(full, b);
    const bool head = b >= 0 && lane == __ffs(grp) - 1;
    for (int w = 0; w < nw; ++w) {
      unsigned m = 0u;
      if (b >= 0) {
        const double4* p = s_pl + w * 32;
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
          const double4 pl = p[k];  // a broadcast
          const double s = __dsub_rn(__dadd_rn(__dadd_rn(__dmul_rn(pl.x, xi), __dmul_rn(pl.y, yi)), __dmul_rn(pl.z, zi)), pl.w);
          m |= (fabs(s) <= half ? 1u : 0u) << k;
        }
        const int left = nslices - (w0 + w) * 32;
        if (left < 32) m &= (1u << left) - 1u;
      }
      const unsigned g = __reduce_or_sync(grp, m);
      if (head && g) atomicOr(&X[(size_t)b * nwords + w0 + w], g);
      const unsigned a = __reduce_or_sync(full, m);
      if (lane == 0 && a) atomicOr(&s_any[w], a);
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < nw && s_any[threadIdx.x]) atomicOr(&any[w0 + threadIdx.x], s_any[threadIdx.x]);
}

// first tile pair of tile row a: rows 0 .. a-1 hold nt, nt - 1, ..., nt - a + 1 pairs
__device__ __forceinline__ long long gm_row_start(long long a, long long nt) { return a * nt - a * (a - 1) / 2; }

__global__ void __launch_bounds__(256) k_gam_coseg(const unsigned* __restrict__ X, int nbins, int nwords, int ntiles,
                                                   unsigned long long* __restrict__ counts) {
  __shared__ unsigned s_a[GM_TILE][GM_KW + 1];  // padded: the 16 rows a warp reads lie in 16 banks
  __shared__ unsigned s_b[GM_TILE][GM_KW + 1];
  // tile pair (tp, tq), tp <= tq, of the row-major upper triangle: the largest tp with gm_row_start(tp) <= t
  const long long t = blockIdx.x;
  const double tt = 2.0 * ntiles + 1.0;
  long long tp = (long long)((tt - sqrt(fmax(tt * tt - 8.0 * (double)t, 0.0))) * 0.5);
  tp = min(max(tp, 0ll), (long long)ntiles - 1);
  while (tp > 0 && gm_row_start(tp, ntiles) > t) --tp;
  while (tp + 1 < ntiles && gm_row_start(tp + 1, ntiles) <= t) ++tp;
  const long long tq = tp + (t - gm_row_start(tp, ntiles));
  const int p0 = (int)tp * GM_TILE, q0 = (int)tq * GM_TILE;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // rows p0 + ty + 16 r, columns q0 + tx + 16 c
  unsigned acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0u;
  for (int k0 = 0; k0 < nwords; k0 += GM_KW) {
    for (int e = threadIdx.x; e < GM_TILE * GM_KW; e += blockDim.x) {
      const int r = e / GM_KW, k = e % GM_KW, w = k0 + k;  // a warp reads 32 consecutive words of one row
      const int p = p0 + r, q = q0 + r;
      s_a[r][k] = p < nbins && w < nwords ? X[(size_t)p * nwords + w] : 0u;
      s_b[r][k] = q < nbins && w < nwords ? X[(size_t)q * nwords + w] : 0u;
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < GM_KW; ++k) {
      unsigned a[4], b[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) a[r] = s_a[ty + 16 * r][k];
#pragma unroll
      for (int c = 0; c < 4; ++c) b[c] = s_b[tx + 16 * c][k];
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] += __popc(a[r] & b[c]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int p = p0 + ty + 16 * r;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int q = q0 + tx + 16 * c;
      if (p < nbins && q < nbins && p <= q) {
        const size_t row = (size_t)p * nbins - (size_t)p * (p - 1) / 2 + (size_t)(q - p);
        counts[row] += acc[r][c];  // the one owner of this pair
      }
    }
  }
}

int gm_ready(mmm_system* h, const char* who) {
  if (!h->gm_configured) return mmm_fail(h, MMM_ERR_STATE, std::string(who) + ": call mmm_gam_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

}  // namespace

extern "C" int mmm_gam_configure(mmm_handle h, const int32_t* bin_of_bead, int32_t n_bins, int32_t max_slices) {
  if (!h) return MMM_ERR_ARG;
  h->gm_configured = false;
  const std::string who = "mmm_gam_configure: ";
  if (n_bins < 1) return mmm_fail(h, MMM_ERR_ARG, who + "n_bins must be >= 1");
  if (!bin_of_bead) return mmm_fail(h, MMM_ERR_ARG, who + "bin_of_bead is NULL");
  if (max_slices < 1 || max_slices > GM_MAX_SLICES)
    return mmm_fail(h, MMM_ERR_ARG, who + "max_slices must be in [1, " + std::to_string(GM_MAX_SLICES) + "]");
  const int64_t rows = (int64_t)n_bins * ((int64_t)n_bins + 1) / 2;
  if (rows > GM_MAX_ROWS)
    return mmm_fail(h, MMM_ERR_ARG, who + std::to_string(rows) + " bin pairs exceed the 2^27 sums (1 GiB) of the "
                                          "accumulator; use fewer bins");
  const int64_t n = h->n;
  for (int64_t i = 0; i < n; ++i)
    if (bin_of_bead[i] < -1 || bin_of_bead[i] >= n_bins) return mmm_fail(h, MMM_ERR_ARG, who + "bin id outside [-1, n_bins)");
  const int64_t wmax = ((int64_t)max_slices + 31) / 32;
  cudaSetDevice(h->device);
  int rc;
  if ((rc = mmm_reserve(h, h->d_gm_bin, (size_t)std::max<int64_t>(n, 1), "GAM bins")) ||
      (rc = mmm_reserve(h, h->d_gm_planes, (size_t)max_slices * 4, "GAM planes")) ||
      (rc = mmm_reserve(h, h->d_gm_x, (size_t)(n_bins * wmax), "GAM detection bitset")) ||
      (rc = mmm_reserve(h, h->d_gm_any, (size_t)wmax, "GAM slice bitset")) ||
      (rc = mmm_reserve(h, h->d_gm_cnt, (size_t)rows, "GAM co-segregation counts")))
    return rc;
  if (!h->gm_ev0) MMM_CUDA(h, cudaEventCreate(&h->gm_ev0));
  if (!h->gm_ev1) MMM_CUDA(h, cudaEventCreate(&h->gm_ev1));
  if (n > 0)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_gm_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_gm_cnt, 0, sizeof(unsigned long long) * (size_t)rows, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));  // the host table may go away after the call
  h->gm_bins = n_bins;
  h->gm_max_slices = max_slices;
  h->gm_structures = 0;
  h->gm_slices = 0;
  h->gm_empty = 0;
  h->gm_ms = 0.f;
  h->gm_configured = true;
  return MMM_OK;
}

extern "C" int mmm_gam_add(mmm_handle h, const double* planes, int32_t n_slices, double half_thickness) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = gm_ready(h, "mmm_gam_add"))) return rc;
  // every check comes before the first copy, so a refused add leaves every sum as it was
  const std::string who = "mmm_gam_add: ";
  if (n_slices < 1 || n_slices > h->gm_max_slices)
    return mmm_fail(h, MMM_ERR_ARG, who + "n_slices must be in [1, max_slices = " + std::to_string(h->gm_max_slices) + "]");
  if (!planes) return mmm_fail(h, MMM_ERR_ARG, who + "planes is NULL");
  for (int64_t k = 0; k < 4 * (int64_t)n_slices; ++k)
    if (!std::isfinite(planes[k]))
      return mmm_fail(h, MMM_ERR_ARG, who + "plane " + std::to_string(k / 4) + " is not finite");
  if (!std::isfinite(half_thickness) || half_thickness < 0.0)
    return mmm_fail(h, MMM_ERR_ARG, who + "the half-thickness must be finite and >= 0");
  if ((uint64_t)h->gm_slices + (uint64_t)n_slices >= (1ull << 63))
    return mmm_fail(h, MMM_ERR_ARG, who + "the slice total would reach 2^63");
  cudaSetDevice(h->device);
  const int n = (int)h->n;
  double box[6];
  if ((rc = mmm_positions_box(h, box))) return rc;
  for (int c = 0; c < 6 && n > 0; ++c)
    if (!std::isfinite(box[c])) return mmm_fail(h, MMM_ERR_ARG, who + "positions are not finite");
  const int nwords = (n_slices + 31) / 32;
  const int nbins = h->gm_bins;
  const int ntiles = (nbins + GM_TILE - 1) / GM_TILE;
  std::vector<unsigned> any((size_t)nwords);
  MMM_CUDA(h, cudaEventRecord(h->gm_ev0, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(h->d_gm_planes, planes, sizeof(double) * 4 * (size_t)n_slices, cudaMemcpyHostToDevice,
                              h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_gm_x, 0, sizeof(unsigned) * (size_t)nbins * (size_t)nwords, h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_gm_any, 0, sizeof(unsigned) * (size_t)nwords, h->stream));
  if (n > 0) {
    const dim3 grid((unsigned)((n + GM_THREADS - 1) / GM_THREADS), (unsigned)((nwords + GM_WPB - 1) / GM_WPB));
    k_gam_detect<<<grid, GM_THREADS, 0, h->stream>>>(h->d_x, h->d_gm_bin, n,
                                                     reinterpret_cast<const double4*>(h->d_gm_planes.get()), n_slices,
                                                     nwords, half_thickness, h->d_gm_x, h->d_gm_any);
    h->launches++;
  }
  const long long tile_pairs = (long long)ntiles * (ntiles + 1) / 2;
  k_gam_coseg<<<(unsigned)tile_pairs, 256, 0, h->stream>>>(h->d_gm_x, nbins, nwords, ntiles, h->d_gm_cnt);
  h->launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    h->gm_configured = false;  // the counts may hold part of this add: unusable until reconfigured
    return mmm_fail(h, MMM_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e) + " (k_gam_detect, k_gam_coseg)");
  }
  MMM_CUDA(h, cudaMemcpyAsync(any.data(), h->d_gm_any, sizeof(unsigned) * any.size(), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaEventRecord(h->gm_ev1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->gm_ev0, h->gm_ev1);
  int64_t detected = 0;
  for (unsigned v : any) detected += __builtin_popcount(v);
  h->gm_ms += ms;
  h->gm_empty += (int64_t)n_slices - detected;
  h->gm_slices += n_slices;
  h->gm_structures++;
  return MMM_OK;
}

extern "C" int mmm_gam_read(mmm_handle h, int64_t* structures_out, int64_t* slices_out, int64_t* empty_out,
                            uint64_t* counts_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = gm_ready(h, "mmm_gam_read"))) return rc;
  if (counts_out) {
    cudaSetDevice(h->device);
    const size_t rows = (size_t)h->gm_bins * ((size_t)h->gm_bins + 1) / 2;
    MMM_CUDA(h, cudaMemcpyAsync(counts_out, h->d_gm_cnt, sizeof(uint64_t) * rows, cudaMemcpyDeviceToHost, h->stream));
    MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  if (structures_out) *structures_out = h->gm_structures;
  if (slices_out) *slices_out = h->gm_slices;
  if (empty_out) *empty_out = h->gm_empty;
  if (device_ms_out) *device_ms_out = h->gm_ms;
  return MMM_OK;
}
