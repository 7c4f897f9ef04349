// mmm_loops.cu — the loop readout: how the ensemble's structures realise the loops of the input table, summed
// over any number of structures (the minimised one, the states of an MD run) on the device and read back once.
//
// The host uploads the rows of the loop table that are valid for this member (multimm_b200/loops.py): the
// anchor beads lo < hi, the chromosome block [first, end) of each anchor and the row's group (0 enforced:
// (lo, hi) is one of the member's loop bonds; 1 held out).  Per structure, in FP64 on the master positions
// with the arithmetic of mmm_contacts and mmm_distance_map (mmm_pair_d2, mmm_quantise):
//   per row r:  contacts[r] += (d2 < rc^2), dist_sum[r] += qd, dist2_sum[r] += qd2 at (lo, hi);
//   per group g and offset (a, b) in [-W, W]^2, over the rows of g whose window pair (lo + a, hi + b) lies in
//   the two blocks with lo + a < hi + b:  apa_contacts[g][a][b] += (d2 < rc^2), apa_dist_sum[g][a][b] += qd
// (aggregate peak analysis: the mean contact frequency and distance in a (2W+1)^2 bead window around the loops).
// Integer sums, so the result is bit-identical however the work is scheduled and equal to a numpy restatement.
//
// k_loops: contiguous row ranges per CTA.  LP_STAGE rows at a time have both anchor windows (2 (2W+1) beads)
// staged in shared memory; thread t owns the offsets t, t + LP_THREADS, ... and adds into its own slots of the
// CTA's accumulators in shared memory (both groups, both sums: 4 (2W+1)^2 uint64, 83 KB at W = 25), so no
// atomic runs inside the loop.  The thread that owns offset (0, 0) adds the per-row sums in place (each row
// belongs to one CTA).  At the end one atomicAdd per nonzero accumulator and CTA.
//
// The add reads d_x and writes only its own buffers: nothing an evaluation, a minimisation, an MD step,
// mmm_last_result or the trajectory sampler reads.
#include <math.h>

#include <algorithm>
#include <string>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int LP_THREADS = 256;
constexpr int LP_STAGE = 8;        // rows staged in shared memory at a time
constexpr int LP_MAX_W = 25;       // keeps the accumulators of both groups in shared memory
constexpr int LP_MIN_ROWS = 64;    // rows per CTA at least: the final atomics stay few beside the pairs
constexpr int LP_CTAS_PER_SM = 2;  // the shared memory of W = 25 allows two

// dynamic shared memory of k_loops at window w
size_t lp_smem(int w) {
  const size_t span = 2 * (size_t)w + 1;
  return 4 * span * span * sizeof(unsigned long long) + (size_t)LP_STAGE * 2 * span * (3 * sizeof(double) + sizeof(int));
}

__global__ void __launch_bounds__(LP_THREADS) k_loops(const double* __restrict__ x, const LoopRow* __restrict__ rows,
                                                      int nrows, int rows_per_cta, int w, double rc2,
                                                      unsigned long long* __restrict__ row_sum,
                                                      unsigned long long* __restrict__ apa) {
  extern __shared__ unsigned long long s_acc[];  // [2 sums: contacts, dist][2 groups][K]
  const int span = 2 * w + 1, K = span * span;
  double* s_x = (double*)(s_acc + 4 * K);                  // [LP_STAGE][2 sides][3][span]
  int* s_bead = (int*)(s_x + (size_t)LP_STAGE * 2 * 3 * span);  // [LP_STAGE][2 sides][span]; -1 outside the block
  __shared__ int s_grp[LP_STAGE];
  const int tid = threadIdx.x;
  for (int o = tid; o < 4 * K; o += LP_THREADS) s_acc[o] = 0;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(nrows, r0 + rows_per_cta);
  const int oc = w * span + w;  // offset (0, 0): the loop's own pair
  for (int s0 = r0; s0 < r1; s0 += LP_STAGE) {
    const int ns = min(LP_STAGE, r1 - s0);
    __syncthreads();  // the previous stage is read (and the accumulators are zero)
    for (int t = tid; t < ns * 2 * span; t += LP_THREADS) {
      const int q = t / (2 * span), side = (t / span) & 1, k = t % span;
      const LoopRow R = rows[s0 + q];
      const int c = (side ? R.hi : R.lo) + k - w;
      const bool in = side ? (c >= R.first_hi && c < R.end_hi) : (c >= R.first_lo && c < R.end_lo);
      s_bead[(q * 2 + side) * span + k] = in ? c : -1;
      if (in)
        for (int d = 0; d < 3; ++d) s_x[((q * 2 + side) * 3 + d) * span + k] = x[3 * (size_t)c + d];
    }
    if (tid < ns) s_grp[tid] = rows[s0 + tid].group;
    __syncthreads();
    for (int q = 0; q < ns; ++q) {
      const int g = s_grp[q];  // CTA-uniform
      const int* bl_of = s_bead + q * 2 * span;
      const int* bh_of = bl_of + span;
      const double* xl = s_x + (size_t)q * 2 * 3 * span;
      const double* xh = xl + 3 * span;
      for (int o = tid; o < K; o += LP_THREADS) {
        const int ia = o / span, ib = o - ia * span;
        const int bl = bl_of[ia], bh = bh_of[ib];
        if (bl < 0 || bh < 0 || bl >= bh) continue;
        const double d2 = mmm_pair_d2(xl[ia], xl[span + ia], xl[2 * span + ia], xh[ib], xh[span + ib], xh[2 * span + ib]);
        const unsigned long long hit = d2 < rc2 ? 1ull : 0ull;
        const unsigned long long qd = mmm_quantise(__dsqrt_rn(d2));
        s_acc[g * K + o] += hit;
        s_acc[(2 + g) * K + o] += qd;
        if (o == oc) {
          const size_t r = (size_t)(s0 + q);
          row_sum[r] += hit;
          row_sum[nrows + r] += qd;
          row_sum[2 * (size_t)nrows + r] += mmm_quantise(d2);
        }
      }
    }
  }
  __syncthreads();
  for (int o = tid; o < 4 * K; o += LP_THREADS)
    if (s_acc[o]) atomicAdd(&apa[o], s_acc[o]);
}

int lp_ready(mmm_system* h, const char* who) {
  if (!h->lp_configured) return mmm_fail(h, MMM_ERR_STATE, std::string(who) + ": call mmm_loops_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

}  // namespace

extern "C" int mmm_loops_configure(mmm_handle h, double rc_nm, int32_t window, int32_t n_loops, const int32_t* bead_lo,
                                   const int32_t* bead_hi, const int32_t* first_lo, const int32_t* end_lo,
                                   const int32_t* first_hi, const int32_t* end_hi, const int8_t* group) {
  if (!h) return MMM_ERR_ARG;
  h->lp_configured = false;
  if (!(rc_nm > 0.0) || !isfinite(rc_nm)) return mmm_fail(h, MMM_ERR_ARG, "mmm_loops_configure: rc must be finite and > 0");
  if (window < 0 || window > LP_MAX_W)
    return mmm_fail(h, MMM_ERR_ARG, "mmm_loops_configure: window must be in [0, " + std::to_string(LP_MAX_W) + "]");
  if (n_loops < 0) return mmm_fail(h, MMM_ERR_ARG, "mmm_loops_configure: n_loops must be >= 0");
  if (n_loops > 0 && (!bead_lo || !bead_hi || !first_lo || !end_lo || !first_hi || !end_hi || !group))
    return mmm_fail(h, MMM_ERR_ARG, "mmm_loops_configure: a row array is NULL");
  const int64_t n = h->n;
  std::vector<LoopRow> rows((size_t)n_loops);
  for (int32_t r = 0; r < n_loops; ++r) {
    const LoopRow R{bead_lo[r], bead_hi[r], first_lo[r], end_lo[r], first_hi[r], end_hi[r], group[r], 0};
    auto bad = [&](const char* why) {
      return mmm_fail(h, MMM_ERR_ARG, "mmm_loops_configure: row " + std::to_string(r) + ": " + why);
    };
    if (R.first_lo < 0 || R.end_lo > n || R.first_lo >= R.end_lo || R.first_hi < 0 || R.end_hi > n ||
        R.first_hi >= R.end_hi)
      return bad("a chromosome block is empty or outside [0, N)");
    if (R.lo < R.first_lo || R.lo >= R.end_lo || R.hi < R.first_hi || R.hi >= R.end_hi)
      return bad("an anchor bead lies outside its block");
    if (R.lo >= R.hi) return bad("bead_lo must be < bead_hi");
    if (R.group != 0 && R.group != 1) return bad("group must be 0 or 1");
    rows[(size_t)r] = R;
  }
  cudaSetDevice(h->device);
  const size_t span = 2 * (size_t)window + 1;
  const size_t sums = 3 * (size_t)n_loops + 4 * span * span;
  int rc;
  if ((rc = mmm_reserve(h, h->d_lp_row, (size_t)n_loops, "loop rows")) ||
      (rc = mmm_reserve(h, h->d_lp_sum, sums, "loop sums")))
    return rc;
  if (!h->lp_ev0) MMM_CUDA(h, cudaEventCreate(&h->lp_ev0));
  if (!h->lp_ev1) MMM_CUDA(h, cudaEventCreate(&h->lp_ev1));
  if (n_loops > 0)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_lp_row, rows.data(), sizeof(LoopRow) * rows.size(), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_lp_sum, 0, sizeof(unsigned long long) * sums, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));  // rows is a host temporary
  h->lp_rc = rc_nm;
  h->lp_w = window;
  h->lp_rows = n_loops;
  h->lp_samples = 0;
  h->lp_bound = 0.0;
  h->lp_ms = 0.f;
  h->lp_configured = true;
  return MMM_OK;
}

extern "C" int mmm_loops_add(mmm_handle h) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = lp_ready(h, "mmm_loops_add"))) return rc;
  cudaSetDevice(h->device);
  // every sum of one structure is at most max(rows, 1) quantised distances: checked before the kernel runs, so
  // a refused structure leaves every sum as it was
  double dpad, qmax;
  if ((rc = mmm_distance_qmax(h, "mmm_loops_add", &dpad, &qmax))) return rc;
  const double bound = (double)std::max<int64_t>(h->lp_rows, 1) * qmax;
  if (h->lp_bound + bound >= 0x1p63)
    return mmm_fail(h, MMM_ERR_ARG,
                    "mmm_loops_add: the sums could overflow int64 (" + std::to_string((long long)h->lp_rows) +
                        " rows, distances up to " + std::to_string(dpad) + " nm at a quantum of 2^-24 nm" +
                        (h->lp_samples > 0 ? ", on top of the structures already summed" : "") + ")");
  const int w = h->lp_w, nrows = (int)h->lp_rows;
  MMM_CUDA(h, cudaEventRecord(h->lp_ev0, h->stream));
  if (nrows > 0) {
    const size_t smem = lp_smem(w);
    MMM_CUDA(h, cudaFuncSetAttribute(k_loops, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ctas = std::max(1, std::min((nrows + LP_MIN_ROWS - 1) / LP_MIN_ROWS,
                                          std::max(h->sm_count, 1) * LP_CTAS_PER_SM));
    const int per = (nrows + ctas - 1) / ctas;
    k_loops<<<(nrows + per - 1) / per, LP_THREADS, smem, h->stream>>>(
        h->d_x, h->d_lp_row, nrows, per, w, h->lp_rc * h->lp_rc, h->d_lp_sum, h->d_lp_sum + 3 * (size_t)nrows);
    h->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      h->lp_configured = false;  // the sums may hold part of this structure: unusable until reconfigured
      return mmm_fail(h, MMM_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e) + " (k_loops)");
    }
  }
  MMM_CUDA(h, cudaEventRecord(h->lp_ev1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->lp_ev0, h->lp_ev1);
  h->lp_ms += ms;
  h->lp_bound += bound;
  h->lp_samples++;
  return MMM_OK;
}

extern "C" int mmm_loops_read(mmm_handle h, int64_t* samples_out, uint64_t* contacts_out, uint64_t* dist_sum_out,
                              uint64_t* dist2_sum_out, uint64_t* apa_contacts_out, uint64_t* apa_dist_sum_out,
                              float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = lp_ready(h, "mmm_loops_read"))) return rc;
  cudaSetDevice(h->device);
  const size_t nr = (size_t)h->lp_rows;
  const size_t span = 2 * (size_t)h->lp_w + 1, K = span * span;
  const unsigned long long* s = h->d_lp_sum;
  const unsigned long long* apa = s + 3 * nr;
  uint64_t* outs[5] = {contacts_out, dist_sum_out, dist2_sum_out, apa_contacts_out, apa_dist_sum_out};
  const unsigned long long* srcs[5] = {s, s + nr, s + 2 * nr, apa, apa + 2 * K};
  const size_t counts[5] = {nr, nr, nr, 2 * K, 2 * K};
  for (int k = 0; k < 5; ++k)
    if (outs[k] && counts[k])
      MMM_CUDA(h, cudaMemcpyAsync(outs[k], srcs[k], sizeof(uint64_t) * counts[k], cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (samples_out) *samples_out = h->lp_samples;
  if (device_ms_out) *device_ms_out = h->lp_ms;
  return MMM_OK;
}
