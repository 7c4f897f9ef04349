// mmm_disthist.cu — distance distributions per genomic bin pair (simulated chromatin tracing: median distance
// maps, contact probability at any radius), summed over structures.  For every unordered bead pair i < j whose
// beads both have a bin, the FP64 squared distance
//   d2 = (dx*dx + dy*dy) + dz*dz  (rounded operation by operation, mmm_pair_d2, as mmm_contacts)
// falls in the cell h = #{k : e2[k] <= d2} of the squared edges e2[0] < ... < e2[E-1] (no sqrt: the cells below
// k hold exactly the contacts of mmm_contacts at rc = e_k), and counts[tri(p, q)][h] += 1 with p <= q the two
// bins, tri the row-major upper-triangle index.  Integer counts do not depend on order, so they are
// bit-identical however the work is scheduled, equal to a numpy restatement, and add up exactly over structures.
//
// The traversal is k_distance_map's (mmm_distances.cu): the upper triangle of the chain-order 32-bead tile pairs,
// cut into chunks of DH_CHUNK consecutive tile pairs taken grid-stride by warps; lane l holds bead i = 32 a + l
// and the j-tile is staged in shared memory, read as broadcasts.  What differs is the per-pair work: the cell
// comes from a branch-free binary search over the squared edges in shared memory (compared as the bit patterns
// of non-negative doubles, which order as the values do; the table is padded to a power of two with ~0, which
// no d2 reaches), and the count goes into a lane-owned uint32 counter s_cnt[warp][cell][lane] (bank = lane: no
// conflicts, no atomics).  A run of equal j-bins holds at most DH_CHUNK * 32 pairs per lane, so uint32 cannot
// overflow.  When the j-bin or the i-tile changes (warp-uniform events) the counters are flushed cell by cell
// with the distance kernel's grouping by bin_i (__match_any_sync; contiguous groups summed by a segmented
// shuffle, one 64-bit atomic per group) and zeroed.
//
// The pass reads d_x and writes only its own buffers (bin table, counts, and the bounding-box partials of
// mmm_positions_box): nothing an evaluation, a minimisation, an MD step or another readout reads.
#include <math.h>

#include <algorithm>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int DH_WARPS = 8;                  // warps per CTA
constexpr int DH_CHUNK = 8;                  // consecutive tile pairs per work item
constexpr int DH_MAX_EDGES = 63;             // H = E + 1 <= 64 cells
constexpr int DH_TABLE = 64;                 // squared-edge table, padded to a power of two
constexpr int64_t DH_MAX_COUNTERS = 1 << 27; // B (B + 1) / 2 x H uint64 counters: 1 GiB

// first tile pair of row a: rows 0 .. a-1 hold ntr, ntr - 1, ..., ntr - a + 1 pairs
__device__ __forceinline__ long long dh_row_start(long long a, long long ntr) { return a * ntr - a * (a - 1) / 2; }

// row-major upper-triangle index of the bin pair p <= q among B bins (numpy.triu_indices order)
__device__ __forceinline__ int dh_tri(int p, int q, int nbins) {
  return (int)((long long)p * nbins - (long long)p * (p - 1) / 2 + (q - p));
}

// flush the warp's run counters cnt[cell][lane] into counts[key][cell] and zero them: key = the lane's bin-pair
// row (-1: no bin, and then its counters are zero).  Called by the whole warp.
__device__ __forceinline__ void dh_flush(int key, bool dirty, unsigned* cnt, int ncells,
                                         unsigned long long* __restrict__ counts) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (!__any_sync(full, dirty)) return;
  const unsigned grp = __match_any_sync(full, key);
  const int head = __ffs(grp) - 1;
  const unsigned span = grp >> head;  // contiguous: span + 1 is a power of two
  const bool contiguous = __all_sync(full, key < 0 || (span & (span + 1)) == 0);
  for (int c = 0; c < ncells; ++c) {
    unsigned v = cnt[c * 32 + lane];
    if (!__any_sync(full, v != 0)) continue;
    cnt[c * 32 + lane] = 0;
    if (contiguous) {
      // segmented suffix sums: lane l adds lane l + o while both are in one (contiguous) group
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned u = __shfl_down_sync(full, v, o);
        if (lane + o < 32 && ((grp >> (lane + o)) & 1u)) v += u;
      }
      if (lane != head) continue;
    }
    if (key >= 0 && v) atomicAdd(&counts[(size_t)key * ncells + c], (unsigned long long)v);
  }
}

__global__ void __launch_bounds__(DH_WARPS * 32) k_disthist(const double* __restrict__ x, const int* __restrict__ bin,
                                                            int n, int ntr, long long npairs_t, long long nchunks,
                                                            int nbins, const unsigned long long* __restrict__ e2,
                                                            int ncells, int half,
                                                            unsigned long long* __restrict__ counts) {
  __shared__ double s_x[DH_WARPS][3][32];
  __shared__ int s_bin[DH_WARPS][32];
  __shared__ unsigned long long s_e2[DH_TABLE];
  extern __shared__ unsigned s_cnt_all[];  // [DH_WARPS][ncells][32]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int k = threadIdx.x; k < DH_TABLE; k += blockDim.x) s_e2[k] = k < ncells - 1 ? e2[k] : ~0ull;
  unsigned* cnt = s_cnt_all + (size_t)w * ncells * 32;
  for (int c = 0; c < ncells; ++c) cnt[c * 32 + lane] = 0;
  __syncthreads();
  const long long nwarps = (long long)gridDim.x * DH_WARPS;
  for (long long c = (long long)blockIdx.x * DH_WARPS + w; c < nchunks; c += nwarps) {  // warp-uniform
    // row a of the first tile pair of the chunk: the largest a with dh_row_start(a) <= k
    const long long k0 = c * DH_CHUNK;
    const double t = 2.0 * ntr + 1.0;
    long long a = (long long)((t - sqrt(fmax(t * t - 8.0 * (double)k0, 0.0))) * 0.5);
    a = min(max(a, 0ll), (long long)ntr - 1);
    while (a > 0 && dh_row_start(a, ntr) > k0) --a;
    while (a + 1 < ntr && dh_row_start(a + 1, ntr) <= k0) ++a;
    long long b = a + (k0 - dh_row_start(a, ntr));
    const long long kend = min(k0 + DH_CHUNK, npairs_t);
    long long cur_a = -1;
    int bi = -1, run = -1;  // run: j-bin of the current run (-1: none; its counters are zero)
    double xi = 0.0, yi = 0.0, zi = 0.0;
    bool ireal = false, dirty = false;
    for (long long k = k0; k < kend; ++k) {
      if (a != cur_a) {  // a new i-tile: flush the run of the old one
        if (cur_a >= 0) dh_flush(bi >= 0 && run >= 0 ? dh_tri(min(bi, run), max(bi, run), nbins) : -1, dirty, cnt, ncells, counts);
        dirty = false;
        run = -1;
        cur_a = a;
        const int i = (int)a * MMM_TILE + lane;
        ireal = i < n;
        bi = -1;
        if (ireal) {
          xi = x[3 * (size_t)i]; yi = x[3 * (size_t)i + 1]; zi = x[3 * (size_t)i + 2];
          bi = bin[i];
        }
      }
      const int j = (int)b * MMM_TILE + lane;
      __syncwarp();
      if (j < n) {
        s_x[w][0][lane] = x[3 * (size_t)j];
        s_x[w][1][lane] = x[3 * (size_t)j + 1];
        s_x[w][2][lane] = x[3 * (size_t)j + 2];
        s_bin[w][lane] = bin[j];
      }
      __syncwarp();
      const int jn = min(MMM_TILE, n - (int)b * MMM_TILE);
      const int jstart = b == a ? lane + 1 : 0;  // i < j inside the diagonal tile
      for (int jj = 0; jj < jn; ++jj) {
        const int bj = s_bin[w][jj];  // warp-uniform
        if (bj != run) {
          dh_flush(bi >= 0 && run >= 0 ? dh_tri(min(bi, run), max(bi, run), nbins) : -1, dirty, cnt, ncells, counts);
          dirty = false;
          run = bj;
        }
        if (ireal && jj >= jstart && bi >= 0 && bj >= 0) {
          const double d2 = mmm_pair_d2(xi, yi, zi, s_x[w][0][jj], s_x[w][1][jj], s_x[w][2][jj]);
          const unsigned long long u = (unsigned long long)__double_as_longlong(d2);  // d2 >= 0: bits order as values
          int pos = 0;
          for (int s = half; s > 0; s >>= 1) pos += s_e2[pos + s - 1] <= u ? s : 0;
          ++cnt[pos * 32 + lane];
          dirty = true;
        }
      }
      if (++b == ntr) {
        ++a;
        b = a;
      }
    }
    dh_flush(bi >= 0 && run >= 0 ? dh_tri(min(bi, run), max(bi, run), nbins) : -1, dirty, cnt, ncells, counts);
  }
}

size_t dh_smem(int ncells) { return sizeof(unsigned) * DH_WARPS * 32 * (size_t)ncells; }

int dh_ready(mmm_system* h, const char* who) {
  if (!h->dh_configured) return mmm_fail(h, MMM_ERR_STATE, std::string(who) + ": call mmm_disthist_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

}  // namespace

extern "C" int mmm_disthist_configure(mmm_handle h, const int32_t* bin_of_bead, int32_t n_bins, const double* edges_nm,
                                      int32_t n_edges) {
  if (!h) return MMM_ERR_ARG;
  h->dh_configured = false;
  const std::string who = "mmm_disthist_configure: ";
  if (n_bins < 1) return mmm_fail(h, MMM_ERR_ARG, who + "n_bins must be >= 1");
  if (!bin_of_bead) return mmm_fail(h, MMM_ERR_ARG, who + "bin_of_bead is NULL");
  if (!edges_nm) return mmm_fail(h, MMM_ERR_ARG, who + "edges_nm is NULL");
  if (n_edges < 1 || n_edges > DH_MAX_EDGES)
    return mmm_fail(h, MMM_ERR_ARG, who + "n_edges must be in [1, " + std::to_string(DH_MAX_EDGES) + "]");
  std::vector<double> e2((size_t)n_edges);
  for (int32_t k = 0; k < n_edges; ++k) {
    const double e = edges_nm[k];
    if (!std::isfinite(e) || !(e > 0.0))
      return mmm_fail(h, MMM_ERR_ARG, who + "edge " + std::to_string(k) + " must be finite and > 0");
    e2[(size_t)k] = e * e;
    if (!std::isfinite(e2[(size_t)k]) || !(e2[(size_t)k] > 0.0) || (k > 0 && !(e2[(size_t)k] > e2[(size_t)k - 1])))
      return mmm_fail(h, MMM_ERR_ARG, who + "the edges and their squares must be strictly increasing, finite and > 0 "
                                            "(edge " + std::to_string(k) + ")");
  }
  const int64_t ncells = (int64_t)n_edges + 1;
  const int64_t rows = (int64_t)n_bins * ((int64_t)n_bins + 1) / 2;
  if (rows > DH_MAX_COUNTERS / ncells)
    return mmm_fail(h, MMM_ERR_ARG, who + std::to_string(rows) + " bin pairs x " + std::to_string(ncells) +
                                        " cells exceed the 2^27 counters (1 GiB) of the accumulator; use fewer bins or edges");
  const int64_t n = h->n;
  std::vector<int64_t> occ((size_t)n_bins, 0);  // beads per bin: the fullest bin pair bounds one add
  for (int64_t i = 0; i < n; ++i) {
    const int32_t b = bin_of_bead[i];
    if (b < -1 || b >= n_bins) return mmm_fail(h, MMM_ERR_ARG, who + "bin id outside [-1, n_bins)");
    if (b >= 0) ++occ[(size_t)b];
  }
  uint64_t pmax = 0, top1 = 0, top2 = 0;  // a diagonal bin pair, or the two fullest bins
  for (int64_t c : occ) {
    const uint64_t v = (uint64_t)c;
    pmax = std::max(pmax, v > 1 ? v * (v - 1) / 2 : 0);
    if (v > top1) {
      top2 = top1;
      top1 = v;
    } else if (v > top2) {
      top2 = v;
    }
  }
  pmax = std::max(pmax, top1 * top2);
  cudaSetDevice(h->device);
  int rc;
  if ((rc = mmm_reserve(h, h->d_dh_bin, (size_t)std::max<int64_t>(n, 1), "distance-histogram bins")) ||
      (rc = mmm_reserve(h, h->d_dh_e2, (size_t)DH_MAX_EDGES, "distance-histogram edges")) ||
      (rc = mmm_reserve(h, h->d_dh_cnt, (size_t)(rows * ncells), "distance-histogram counts")))
    return rc;
  if (!h->dh_ev0) MMM_CUDA(h, cudaEventCreate(&h->dh_ev0));
  if (!h->dh_ev1) MMM_CUDA(h, cudaEventCreate(&h->dh_ev1));
  if (n > 0)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_dh_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(h->d_dh_e2, e2.data(), sizeof(double) * e2.size(), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_dh_cnt, 0, sizeof(unsigned long long) * (size_t)(rows * ncells), h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));  // the host tables may go away after the call
  h->dh_bins = n_bins;
  h->dh_cells = (int32_t)ncells;
  h->dh_pmax = pmax;
  h->dh_total = 0;
  h->dh_samples = 0;
  h->dh_ms = 0.f;
  h->dh_configured = true;
  return MMM_OK;
}

extern "C" int mmm_disthist_add(mmm_handle h) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = dh_ready(h, "mmm_disthist_add"))) return rc;
  // checked before the kernel runs, so a refused structure leaves every count as it was
  if (h->dh_total + h->dh_pmax >= (1ull << 63))
    return mmm_fail(h, MMM_ERR_ARG,
                    "mmm_disthist_add: the counts could overflow int64 (" + std::to_string(h->dh_pmax) +
                        " bead pairs in the fullest bin pair, on top of the " + std::to_string(h->dh_samples) +
                        " structures already counted)");
  cudaSetDevice(h->device);
  const int n = (int)h->n;
  double box[6];
  if ((rc = mmm_positions_box(h, box))) return rc;
  for (int c = 0; c < 6 && n > 0; ++c)
    if (!std::isfinite(box[c])) return mmm_fail(h, MMM_ERR_ARG, "mmm_disthist_add: positions are not finite");
  const int ncells = h->dh_cells;
  int half = 1;  // the binary search's first step: half of the smallest power of two >= H
  while (2 * half < ncells) half *= 2;
  const int ntr = (n + MMM_TILE - 1) / MMM_TILE;
  const long long npairs_t = (long long)ntr * (ntr + 1) / 2;
  const long long nchunks = (npairs_t + DH_CHUNK - 1) / DH_CHUNK;
  MMM_CUDA(h, cudaEventRecord(h->dh_ev0, h->stream));
  if (nchunks > 0) {
    const size_t smem = dh_smem(ncells);
    MMM_CUDA(h, cudaFuncSetAttribute(k_disthist, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    MMM_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_disthist, DH_WARPS * 32, smem));
    const long long want = (nchunks + DH_WARPS - 1) / DH_WARPS;
    const int ctas = (int)std::min<long long>(want, (long long)std::max(h->sm_count, 1) * std::max(per_sm, 1));
    k_disthist<<<ctas, DH_WARPS * 32, smem, h->stream>>>(h->d_x, h->d_dh_bin, n, ntr, npairs_t, nchunks, h->dh_bins,
                                                         h->d_dh_e2, ncells, half, h->d_dh_cnt);
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      h->dh_configured = false;  // the counts may hold part of this structure: unusable until reconfigured
      return mmm_fail(h, MMM_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e) + " (k_disthist)");
    }
  }
  MMM_CUDA(h, cudaEventRecord(h->dh_ev1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->dh_ev0, h->dh_ev1);
  h->dh_ms += ms;
  h->dh_total += h->dh_pmax;
  h->dh_samples++;
  return MMM_OK;
}

extern "C" int mmm_disthist_read(mmm_handle h, int64_t* samples_out, uint64_t* counts_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = dh_ready(h, "mmm_disthist_read"))) return rc;
  if (counts_out) {
    cudaSetDevice(h->device);
    const size_t len = (size_t)h->dh_bins * ((size_t)h->dh_bins + 1) / 2 * (size_t)h->dh_cells;
    MMM_CUDA(h, cudaMemcpyAsync(counts_out, h->d_dh_cnt, sizeof(uint64_t) * len, cudaMemcpyDeviceToHost, h->stream));
    MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  if (samples_out) *samples_out = h->dh_samples;
  if (device_ms_out) *device_ms_out = h->dh_ms;
  return MMM_OK;
}
