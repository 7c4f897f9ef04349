// mmm_distances.cu — ensemble mean-distance maps (simulated chromatin tracing) at the handle's current
// positions: for every unordered bead pair i < j whose beads both have a bin, the FP64 distance
//   d2 = (dx*dx + dy*dy) + dz*dz  (rounded operation by operation, as mmm_contacts), d = sqrt(d2) (correctly
//   rounded), quantised on its own with Q = 2^-24: qd = rint(d / Q), qd2 = rint(d2 / Q) (half to even),
// added into two dense symmetric uint64 maps at (bin_i, bin_j) and, off the diagonal, at (bin_j, bin_i).
// Integer sums do not depend on order, so the maps are bit-identical however the work is scheduled and
// equal to a numpy restatement, and the maps of ensemble members add up exactly.
//
// All pairs, no culling: the upper triangle of the chain-order 32-bead tile pairs (b >= a), numbered row by
// row and cut into chunks of DM_CHUNK consecutive tile pairs; warps take chunks grid-stride (every tile pair
// off the diagonal costs the same 1024 pairs, so equal chunks are equal work).  Lane l holds bead
// i = 32 a + l; the j-tile is staged in shared memory and read as broadcasts.  Every lane keeps register
// sums over the current run of equal j-bins and flushes them when the j-bin or the i-tile changes (a
// warp-uniform event, also across the consecutive tile pairs of a chunk).  A flush groups the lanes by
// (bin_i, bin_j) with __match_any_sync: contiguous groups (canonical bins are runs of beads in chain order)
// are summed by a segmented shuffle and their first lane adds them with one atomic per map and orientation;
// scattered groups (any other bin assignment) add lane by lane.  A tile pair whose beads sit in one bin on
// each side thus ends in one warp reduction and at most four atomics.
//
// The pass reads d_x and writes only its own scratch (bin table, the two maps, bounding-box partials):
// nothing an evaluation, a minimisation or mmm_last_result reads.
#include <math.h>

#include <algorithm>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int DM_WARPS = 8;          // warps per CTA
constexpr int DM_CHUNK = 8;          // consecutive tile pairs per work item
constexpr int DM_MAX_BINS = 4096;    // two dense maps of 128 MB each
constexpr int DM_BOX_BLOCKS = 256;   // partial bounding boxes

// first tile pair of row a: rows 0 .. a-1 hold ntr, ntr - 1, ..., ntr - a + 1 pairs
__device__ __forceinline__ long long dm_row_start(long long a, long long ntr) { return a * ntr - a * (a - 1) / 2; }

// flush one lane's run sums: group the lanes by key (bin_i * n_bins + bin_j; -1: no bin, and then the sums
// are zero).  Called by the whole warp.
__device__ __forceinline__ void dm_flush(int key, int bi, int bj, int nbins, unsigned long long sd,
                                         unsigned long long sd2, unsigned long long* __restrict__ dmap,
                                         unsigned long long* __restrict__ d2map) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (!__any_sync(full, (sd | sd2) != 0)) return;
  const unsigned grp = __match_any_sync(full, key);
  const int head = __ffs(grp) - 1;
  const unsigned span = grp >> head;  // contiguous: span + 1 is a power of two
  if (__all_sync(full, key < 0 || (span & (span + 1)) == 0)) {
    // segmented suffix sums: lane l adds lane l + o while both are in one (contiguous) group
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long u = __shfl_down_sync(full, sd, o);
      const unsigned long long u2 = __shfl_down_sync(full, sd2, o);
      if (lane + o < 32 && ((grp >> (lane + o)) & 1u)) {
        sd += u;
        sd2 += u2;
      }
    }
    if (lane != head) return;
  }
  if (key < 0 || (sd | sd2) == 0) return;
  atomicAdd(&dmap[key], sd);
  atomicAdd(&d2map[key], sd2);
  if (bi != bj) {
    const size_t mirror = (size_t)bj * nbins + bi;
    atomicAdd(&dmap[mirror], sd);
    atomicAdd(&d2map[mirror], sd2);
  }
}

__global__ void __launch_bounds__(DM_WARPS * 32) k_distance_map(const double* __restrict__ x, const int* __restrict__ bin,
                                                                int n, int ntr, long long npairs_t, long long nchunks,
                                                                int nbins, unsigned long long* __restrict__ dmap,
                                                                unsigned long long* __restrict__ d2map) {
  __shared__ double s_x[DM_WARPS][3][32];
  __shared__ int s_bin[DM_WARPS][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long nwarps = (long long)gridDim.x * DM_WARPS;
  for (long long c = (long long)blockIdx.x * DM_WARPS + w; c < nchunks; c += nwarps) {  // warp-uniform
    // row a of the first tile pair of the chunk: the largest a with dm_row_start(a) <= k
    const long long k0 = c * DM_CHUNK;
    const double t = 2.0 * ntr + 1.0;
    long long a = (long long)((t - sqrt(fmax(t * t - 8.0 * (double)k0, 0.0))) * 0.5);
    a = min(max(a, 0ll), (long long)ntr - 1);
    while (a > 0 && dm_row_start(a, ntr) > k0) --a;
    while (a + 1 < ntr && dm_row_start(a + 1, ntr) <= k0) ++a;
    long long b = a + (k0 - dm_row_start(a, ntr));
    const long long kend = min(k0 + DM_CHUNK, npairs_t);
    long long cur_a = -1;
    int bi = -1, run = -1;  // run: j-bin of the current run (-1: none; its sums are zero)
    double xi = 0.0, yi = 0.0, zi = 0.0;
    bool ireal = false;
    unsigned long long sd = 0, sd2 = 0;
    for (long long k = k0; k < kend; ++k) {
      if (a != cur_a) {  // a new i-tile: flush the run of the old one
        if (cur_a >= 0) dm_flush(bi >= 0 && run >= 0 ? bi * nbins + run : -1, bi, run, nbins, sd, sd2, dmap, d2map);
        sd = sd2 = 0;
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
          dm_flush(bi >= 0 && run >= 0 ? bi * nbins + run : -1, bi, run, nbins, sd, sd2, dmap, d2map);
          sd = sd2 = 0;
          run = bj;
        }
        const double d2 = mmm_pair_d2(xi, yi, zi, s_x[w][0][jj], s_x[w][1][jj], s_x[w][2][jj]);
        if (ireal && jj >= jstart && bi >= 0 && bj >= 0) {
          sd += mmm_quantise(__dsqrt_rn(d2));
          sd2 += mmm_quantise(d2);
        }
      }
      if (++b == ntr) {
        ++a;
        b = a;
      }
    }
    dm_flush(bi >= 0 && run >= 0 ? bi * nbins + run : -1, bi, run, nbins, sd, sd2, dmap, d2map);
  }
}

// per-block FP64 bounding box of the beads: part[block] = {min x, min y, min z, max x, max y, max z}
__global__ void __launch_bounds__(256) k_dm_bbox(const double* __restrict__ x, int n, double* __restrict__ part) {
  __shared__ double s[6][256];
  double v[6] = {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    for (int c = 0; c < 3; ++c) {
      const double p = x[3 * (size_t)i + c];
      v[c] = fmin(v[c], p);
      v[3 + c] = fmax(v[3 + c], p);
      if (p != p) v[c] = v[3 + c] = p;  // NaN stays visible to the host check
    }
  for (int c = 0; c < 6; ++c) s[c][threadIdx.x] = v[c];
  __syncthreads();
  if (threadIdx.x < 6) {
    const int c = threadIdx.x;
    double r = s[c][0];
    for (int t = 1; t < 256; ++t) {
      const double p = s[c][t];
      r = (p != p || r != r) ? NAN : (c < 3 ? fmin(r, p) : fmax(r, p));
    }
    part[(size_t)blockIdx.x * 6 + c] = r;
  }
}

}  // namespace

// The FP64 bounding box of the current positions: box = {min x, min y, min z, max x, max y, max z}, NaN on an
// axis where a coordinate is NaN.  Launches one kernel and synchronises; writes nothing else.
int mmm_positions_box(mmm_system* h, double box[6]) {
  const int n = (int)h->n;
  int rc;
  if ((rc = mmm_reserve(h, h->d_dm_box, (size_t)DM_BOX_BLOCKS * 6, "distance-map boxes"))) return rc;
  const int box_blocks = std::max(1, std::min(DM_BOX_BLOCKS, (n + 255) / 256));
  k_dm_bbox<<<box_blocks, 256, 0, h->stream>>>(h->d_x, n, h->d_dm_box);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  std::vector<double> part((size_t)box_blocks * 6);
  MMM_CUDA(h, cudaMemcpyAsync(part.data(), h->d_dm_box, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  for (int c = 0; c < 3; ++c) {
    double lo = INFINITY, hi = -INFINITY;
    for (int b = 0; b < box_blocks; ++b) {
      lo = std::min(lo, part[(size_t)b * 6 + c]);
      hi = std::max(hi, part[(size_t)b * 6 + 3 + c]);
      if (std::isnan(part[(size_t)b * 6 + c]) || std::isnan(part[(size_t)b * 6 + 3 + c])) lo = hi = NAN;
    }
    box[c] = lo;
    box[3 + c] = hi;
  }
  return MMM_OK;
}

// *dpad: a distance of at most sqrt(d2max), padded for the rounding of d2 and d; *qmax bounds its quantised
// value and that of its square.
void mmm_qmax_of(double d2max, double* dpad, double* qmax) {
  *dpad = sqrt(d2max) * (1.0 + 0x1p-40) + 0x1p-60;
  *qmax = ceil(MMM_DIST_SCALE * std::max(*dpad * *dpad, *dpad)) + 1.0;
}

// The quantised-distance bound of the current positions: *dpad bounds every bead pair's distance (the diagonal
// of the beads' FP64 bounding box, padded for the rounding of d2 and d) and *qmax the quantised distance and
// squared distance of every pair.  MMM_ERR_ARG (message prefixed by who) when the positions are not finite.
// Launches one kernel and synchronises; writes nothing else.  The distance maps and mmm_loops_add guard with it.
int mmm_distance_qmax(mmm_system* h, const char* who, double* dpad, double* qmax) {
  const int n = (int)h->n;
  double box[6];
  int rc;
  if ((rc = mmm_positions_box(h, box))) return rc;
  double d2max = 0.0;
  for (int c = 0; c < 3; ++c) {
    const double ext = n > 0 ? box[3 + c] - box[c] : 0.0;
    d2max += ext * ext;
  }
  if (!std::isfinite(d2max))
    return mmm_fail(h, MMM_ERR_ARG, std::string(who) + ": positions are not finite (no distance can be quantised)");
  mmm_qmax_of(d2max, dpad, qmax);  // D and the bound of qd and qd2 of every pair
  return MMM_OK;
}

// Overflow guard of the distance sums: *bound = (pairs of the fullest bin pair) x (largest quantised value of
// one pair, mmm_distance_qmax), occ = beads per bin.  MMM_ERR_ARG (message prefixed by who) when the positions
// are not finite or when prior + *bound reaches 2^63: the one-shot map passes prior = 0, the trajectory
// sampler the bounds of the structures it has already summed.  Launches one kernel and synchronises; writes
// nothing else.
int mmm_distance_guard(mmm_system* h, const char* who, const std::vector<int64_t>& occ, double prior, double* bound) {
  double dpad, qmax;
  int rc;
  if ((rc = mmm_distance_qmax(h, who, &dpad, &qmax))) return rc;
  double pmax = 0.0, top1 = 0.0, top2 = 0.0;  // pairs of the fullest bin pair: a diagonal one or the two fullest bins
  for (int64_t c : occ) {
    const double v = (double)c;
    pmax = std::max(pmax, v * (v - 1.0) * 0.5);
    if (v > top1) {
      top2 = top1;
      top1 = v;
    } else if (v > top2) {
      top2 = v;
    }
  }
  pmax = std::max(pmax, top1 * top2);
  *bound = pmax * qmax;
  if (prior + *bound >= 0x1p63)
    return mmm_fail(h, MMM_ERR_ARG,
                    std::string(who) + ": the sums could overflow int64 (" + std::to_string((long long)pmax) +
                        " bead pairs in the fullest bin pair, distances up to " + std::to_string(dpad) +
                        " nm at a quantum of 2^-24 nm" +
                        (prior > 0.0 ? ", on top of the structures already summed" : "") +
                        "); use more bins or a more compact structure");
  return MMM_OK;
}

// The distance pass: sums at the current positions added into dmap and d2map (n_bins^2 each), zeroed first
// when clear.  d_bin: the bin of every bead on the device.  mmm_distance_map and the sampler run it.
int mmm_distance_pass(mmm_system* h, const int* d_bin, int32_t n_bins, unsigned long long* dmap,
                      unsigned long long* d2map, bool clear) {
  const int n = (int)h->n;
  const size_t cells = (size_t)n_bins * (size_t)n_bins;
  if (clear) {
    MMM_CUDA(h, cudaMemsetAsync(dmap, 0, sizeof(unsigned long long) * cells, h->stream));
    MMM_CUDA(h, cudaMemsetAsync(d2map, 0, sizeof(unsigned long long) * cells, h->stream));
  }
  const int ntr = (n + MMM_TILE - 1) / MMM_TILE;
  const long long npairs_t = (long long)ntr * (ntr + 1) / 2;
  const long long nchunks = (npairs_t + DM_CHUNK - 1) / DM_CHUNK;
  if (nchunks > 0) {
    const long long want = (nchunks + DM_WARPS - 1) / DM_WARPS;
    const int ctas = (int)std::min<long long>(want, (long long)std::max(h->sm_count, 1) * 8);
    k_distance_map<<<ctas, DM_WARPS * 32, 0, h->stream>>>(h->d_x, d_bin, n, ntr, npairs_t, nchunks, n_bins, dmap,
                                                          d2map);
    h->launches++;
    MMM_CUDA(h, cudaGetLastError());
  }
  return MMM_OK;
}

extern "C" int mmm_distance_map(mmm_handle h, const int32_t* bin_of_bead, int32_t n_bins, uint64_t* dist_sum_out,
                                uint64_t* dist2_sum_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  if (n_bins < 1 || n_bins > DM_MAX_BINS) return mmm_fail(h, MMM_ERR_ARG, "mmm_distance_map: n_bins must be in [1, 4096]");
  if (!bin_of_bead) return mmm_fail(h, MMM_ERR_ARG, "mmm_distance_map: bin_of_bead is NULL");
  const int n = (int)h->n;
  std::vector<int64_t> occ((size_t)n_bins, 0);  // beads per bin: the largest bin pair bounds every sum
  for (int i = 0; i < n; ++i) {
    const int32_t b = bin_of_bead[i];
    if (b < -1 || b >= n_bins) return mmm_fail(h, MMM_ERR_ARG, "mmm_distance_map: bin id outside [-1, n_bins)");
    if (b >= 0) ++occ[(size_t)b];
  }
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  cudaSetDevice(h->device);
  int rc;
  const size_t cells = (size_t)n_bins * (size_t)n_bins;
  if ((rc = mmm_reserve(h, h->d_dm_bin, (size_t)std::max(n, 1), "distance-map bins")) ||
      (rc = mmm_reserve(h, h->d_dm_map, 2 * cells, "distance map")))
    return rc;
  if (!h->dm_ev0) MMM_CUDA(h, cudaEventCreate(&h->dm_ev0));
  if (!h->dm_ev1) MMM_CUDA(h, cudaEventCreate(&h->dm_ev1));
  unsigned long long* dmap = h->d_dm_map;
  unsigned long long* d2map = h->d_dm_map + cells;
  double bound;
  if ((rc = mmm_distance_guard(h, "mmm_distance_map", occ, 0.0, &bound))) return rc;

  MMM_CUDA(h, cudaMemcpyAsync(h->d_dm_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaEventRecord(h->dm_ev0, h->stream));
  if ((rc = mmm_distance_pass(h, h->d_dm_bin, n_bins, dmap, d2map, true))) return rc;
  MMM_CUDA(h, cudaEventRecord(h->dm_ev1, h->stream));
  if (dist_sum_out)
    MMM_CUDA(h, cudaMemcpyAsync(dist_sum_out, dmap, sizeof(uint64_t) * cells, cudaMemcpyDeviceToHost, h->stream));
  if (dist2_sum_out)
    MMM_CUDA(h, cudaMemcpyAsync(dist2_sum_out, d2map, sizeof(uint64_t) * cells, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->dm_ev0, h->dm_ev1);
  if (device_ms_out) *device_ms_out = ms;
  return MMM_OK;
}
