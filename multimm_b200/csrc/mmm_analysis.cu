// mmm_analysis.cu — the O(N^2) part of the structure report (SURVEY 8(f) N4):
// plots.py:663 `dmat = distance.cdist(V, V); mean_dist = np.mean(dmat)` materialises an N x N FP64
// matrix (320 GB at N = 2e5; the reference's own heat-map is switched off at N >= 50 000,
// model.py:1095).  Here the sum of all pair distances is a tiled gather pass over the centred FP32
// copy: j-beads staged 256 at a time in shared memory, FP32 within a stage, FP64 across, fixed
// summation order.  Issue-bound like the gather pair kernel (7 instructions per ordered pair).
#include "mmm_internal.cuh"

namespace {

__global__ void __launch_bounds__(256) k_sum_distances(const float4* __restrict__ pos4, int64_t n, int64_t npad,
                                                       double* __restrict__ part) {
  __shared__ float4 s_j[256];
  __shared__ double s_red[8];
  const int tid = threadIdx.x;
  const int64_t i = (int64_t)blockIdx.x * 256 + tid;
  const float4 pi = pos4[i < npad ? i : 0];
  double acc = 0.0;
  for (int64_t j0 = 0; j0 < n; j0 += 256) {
    __syncthreads();
    s_j[tid] = pos4[j0 + tid];  // npad is a multiple of 256
    __syncthreads();
    const int cnt = (int)(n - j0 < 256 ? n - j0 : 256);
    float a = 0.0f;
#pragma unroll 8
    for (int jj = 0; jj < cnt; ++jj) {
      const float dx = pi.x - s_j[jj].x, dy = pi.y - s_j[jj].y, dz = pi.z - s_j[jj].z;
      a += sqrtf(fmaf(dz, dz, fmaf(dy, dy, dx * dx)));
    }
    acc += (double)a;
  }
  if (i >= n) acc = 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((tid & 31) == 0) s_red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += s_red[w];
    part[blockIdx.x] = s;
  }
}

// Block means of the contact map the reference's get_heatmap draws (plots.py:540-561): strength
// 1 / (d + 1)^(2/3) of every bead pair, log1p-transformed.  One CTA per bin pair (p <= q) sums its
// (beads of bin p) x (beads of bin q) rectangle in FP64 with a fixed order and writes the mean to both
// (p, q) and (q, p): the N x N matrix never exists, which is what lifts the reference's N < 5e4 limit
// (model.py:1095-1104).  The same pass returns the sum of all pair distances (np.mean(cdist(V, V))).
__global__ void __launch_bounds__(256) k_contact_bins(const double* __restrict__ x, const long long* __restrict__ edges,
                                                      int bins, int log_scale, double* __restrict__ map,
                                                      double* __restrict__ dist_part) {
  __shared__ double s_red[2][8];
  // upper-triangular enumeration of (p, q), q >= p
  const long long t = blockIdx.x;
  int p = (int)((2.0 * bins + 1.0 - sqrt((2.0 * bins + 1.0) * (2.0 * bins + 1.0) - 8.0 * (double)t)) * 0.5);
  while ((long long)p * (2 * bins - p + 1) / 2 > t) --p;
  while ((long long)(p + 1) * (2 * bins - p) / 2 <= t) ++p;
  const int q = p + (int)(t - (long long)p * (2 * bins - p + 1) / 2);
  const long long a0 = edges[p], a1 = edges[p + 1], b0 = edges[q], b1 = edges[q + 1];
  const long long wa = a1 - a0, wb = b1 - b0, cells = wa * wb;
  double acc = 0.0, dsum = 0.0;
  for (long long c = threadIdx.x; c < cells; c += 256) {
    const long long i = a0 + c / wb, j = b0 + c % wb;
    const double dx = x[3 * i] - x[3 * j], dy = x[3 * i + 1] - x[3 * j + 1], dz = x[3 * i + 2] - x[3 * j + 2];
    const double d = sqrt(dx * dx + dy * dy + dz * dz);
    const double m = 1.0 / cbrt((d + 1.0) * (d + 1.0));
    acc += log_scale ? log1p(m) : m;
    dsum += d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
  }
  if ((threadIdx.x & 31) == 0) { s_red[0][threadIdx.x >> 5] = acc; s_red[1][threadIdx.x >> 5] = dsum; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0, sd = 0.0;
    for (int w = 0; w < 8; ++w) { s += s_red[0][w]; sd += s_red[1][w]; }
    const double mean = s / (double)cells;
    map[(size_t)p * bins + q] = mean;
    map[(size_t)q * bins + p] = mean;
    dist_part[blockIdx.x] = p == q ? sd : 2.0 * sd;  // off-diagonal rectangles stand for both orders
  }
}

}  // namespace

// Stand-alone (no handle): any (n, 3) coordinate array, e.g. what get_coordinates_cif returns, which
// drops the HETATM chromosome-end beads and is therefore shorter than N_BEADS.
extern "C" int mmm_contact_map(int device, const double* xyz, int64_t n, int bins, int log_scale, double* map_out,
                               double* mean_dist_out) {
  if (!xyz || n < 1 || bins < 1 || bins > n || !map_out) return MMM_ERR_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return MMM_ERR_CUDA;
  // np.linspace(0, n, bins + 1).astype(int64): edges[k] = floor(k * n / bins) computed as numpy does
  std::vector<long long> edges((size_t)bins + 1);
  const double step = (double)n / (double)bins;
  for (int k = 0; k <= bins; ++k) edges[(size_t)k] = (long long)(k == bins ? (double)n : (double)k * step);
  const long long nblocks = (long long)bins * (bins + 1) / 2;
  if (nblocks > 2147483647LL) return MMM_ERR_ARG;
  DevBuf<double> d_x, d_map, d_part;
  DevBuf<long long> d_edges;
  int rc;
  if ((rc = mmm_reserve(nullptr, d_x, 3 * (size_t)n, "contact-map coordinates")) ||
      (rc = mmm_reserve(nullptr, d_map, (size_t)bins * bins, "contact map")) ||
      (rc = mmm_reserve(nullptr, d_part, (size_t)nblocks, "contact-map partial sums")) ||
      (rc = mmm_reserve(nullptr, d_edges, edges.size(), "contact-map bin edges")))
    return rc;
  MMM_CUDA(nullptr, cudaMemcpy(d_x, xyz, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice));
  MMM_CUDA(nullptr, cudaMemcpy(d_edges, edges.data(), sizeof(long long) * edges.size(), cudaMemcpyHostToDevice));
  k_contact_bins<<<(unsigned)nblocks, 256>>>(d_x, d_edges, bins, log_scale, d_map, d_part);
  MMM_CUDA(nullptr, cudaGetLastError());
  MMM_CUDA(nullptr, cudaMemcpy(map_out, d_map, sizeof(double) * (size_t)bins * bins, cudaMemcpyDeviceToHost));
  if (mean_dist_out) {
    std::vector<double> part((size_t)nblocks);
    MMM_CUDA(nullptr, cudaMemcpy(part.data(), d_part, sizeof(double) * (size_t)nblocks, cudaMemcpyDeviceToHost));
    double s = 0.0;
    for (double v : part) s += v;
    *mean_dist_out = s / ((double)n * (double)n);  // zero diagonal included, as np.mean(cdist(V, V))
  }
  return MMM_OK;
}

extern "C" int mmm_mean_pair_distance(mmm_handle h, double* mean_out) {
  if (!h || !mean_out) return MMM_ERR_ARG;
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  cudaSetDevice(h->device);
  int rc = mmm_launch_prepare(h, nullptr);  // d_x -> centred FP32 copy
  if (rc) return rc;
  const int blocks = (int)((h->n + 255) / 256);
  DevBuf<double> d_part;
  if ((rc = mmm_reserve(h, d_part, (size_t)blocks, "mean-distance partial sums"))) return rc;
  k_sum_distances<<<blocks, 256, 0, h->stream>>>(h->d_pos4, h->n, h->npad, d_part);
  h->launches++;
  std::vector<double> part((size_t)blocks);
  MMM_CUDA(h, cudaMemcpyAsync(part.data(), d_part, sizeof(double) * blocks, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  double s = 0.0;
  for (double p : part) s += p;
  // np.mean over the full N x N matrix, zero diagonal included (plots.py:664)
  *mean_out = s / ((double)h->n * (double)h->n);
  return MMM_OK;
}
