// mmm_dynamics.cu — locus dynamics of an ordered run of structures (the samples of an MD run, as live-cell
// imaging sees a nucleus): mean squared displacements at fixed lags and the lifetimes of the loops' closed and
// open states, summed on the device and read back once.
//
// Structures are numbered s = 0, 1, ... in add order.  For every lag tau of the lag set with tau <= s, the add of
// structure s pairs it with structure s - tau, in FP64 on the master positions:
//   per bead i with a bin:  msd_sum[tau][bin_i] += rint(2^24 d2),  d2 = mmm_pair_d2(x_i(s), x_i(s - tau));
//   per loop row (lo, hi):  rel_msd_sum[tau][r] += rint(2^24 d2),  d2 = (ex*ex + ey*ey) + ez*ez with
//                           e = R(s) - R(s - tau), R = x_hi - x_lo per component (the two-anchor MSD, free of
//                           drift by construction; the per-bead MSD has no drift correction).
// Per row the add also steps a state machine: the row is closed when mmm_pair_d2(lo, hi) < rc^2 (the loop
// readout's contact) and open otherwise.  A run is a maximal stretch of samples in one state; when a transition
// ends a run of length l, the run is complete if it began at a transition (per row: count and summed length by
// state; per group and state: a histogram over floor(log2 l) and the summed length) and left-censored otherwise
// (per group and state: count and summed length).  The run still open stays in the row's state for the host.
// Integer sums, so the results are bit-identical however the work is scheduled and equal to a numpy restatement.
//
// The ring keeps the master positions of the last L = max lag structures (slot s mod L).  An add runs
//   k_dyn_rows:  one thread per row; it owns its row's sums and state (no atomics), the group sums take atomics;
//   k_dyn_bins:  one thread per bead looping over the lags, reducing per (lag, bin) with __match_any_sync groups
//                and a segmented shuffle (bins are runs of beads in chain order: one atomic per warp and lag),
//                lane by lane for scattered bins;
//   a device-to-device copy of d_x into slot s mod L.
// The add reads d_x and writes only its own buffers: nothing an evaluation, a minimisation, an MD step,
// mmm_last_result, the trajectory sampler, the loop readout or the three-way map reads.
#include <math.h>

#include <algorithm>
#include <string>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int DY_THREADS = 256;
constexpr int DY_ROW_THREADS = 128;
constexpr int DY_MAX_LAG = 4096;
constexpr int32_t DY_MAX_BINS = 1 << 22;  // dense [lags][bins] sums: 32 MB per lag at the cap
constexpr int DY_BUCKETS = 64;            // floor(log2 l) of a run length l < 2^64
// the group sums after the per-row ones: hist [2 groups][2 states][64], hist_len, left_runs, left_len [2][2]
// (state 0 closed, 1 open)
constexpr size_t DY_GROUP_SUMS = 4 * DY_BUCKETS + 3 * 4;

__device__ __forceinline__ size_t dy_slot(long long s, int tau, int ring_len) { return (size_t)((s - tau) % ring_len); }

__global__ void __launch_bounds__(DY_ROW_THREADS) k_dyn_rows(const double* __restrict__ x, const double* __restrict__ ring,
                                                            size_t plane, int ring_len, long long s,
                                                            const int* __restrict__ lags, int n_active,
                                                            const int4* __restrict__ rows, int nrows, double rc2,
                                                            long long* __restrict__ state,
                                                            unsigned long long* __restrict__ rel,
                                                            unsigned long long* __restrict__ runs,
                                                            unsigned long long* __restrict__ grp) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nrows) return;
  const int4 R = rows[r];
  const size_t lo = 3 * (size_t)R.x, hi = 3 * (size_t)R.y;
  const double lx = x[lo], ly = x[lo + 1], lz = x[lo + 2];
  const double hx = x[hi], hy = x[hi + 1], hz = x[hi + 2];
  const double rx = __dsub_rn(hx, lx), ry = __dsub_rn(hy, ly), rz = __dsub_rn(hz, lz);
  for (int k = 0; k < n_active; ++k) {
    const double* p = ring + dy_slot(s, lags[k], ring_len) * plane;
    const double ex = __dsub_rn(rx, __dsub_rn(p[hi], p[lo]));
    const double ey = __dsub_rn(ry, __dsub_rn(p[hi + 1], p[lo + 1]));
    const double ez = __dsub_rn(rz, __dsub_rn(p[hi + 2], p[lo + 2]));
    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)), __dmul_rn(ez, ez));
    rel[(size_t)k * nrows + r] += mmm_quantise(d2);
  }
  const long long closed = mmm_pair_d2(lx, ly, lz, hx, hy, hz) < rc2 ? 1 : 0;
  long long* st = state + r;           // closed
  long long* len = state + nrows + r;  // length of the run in progress (0: no sample yet)
  long long* from = state + 2 * (size_t)nrows + r;  // it began at a transition
  if (*len == 0) {
    *st = closed;
    *len = 1;
  } else if (*st == closed) {
    ++*len;
  } else {  // a transition ends the run in progress
    const int k = *st ? 0 : 1;
    const unsigned long long l = (unsigned long long)*len;
    const int g = R.z;
    if (*from) {
      runs[(size_t)(2 * k) * nrows + r] += 1;
      runs[(size_t)(2 * k + 1) * nrows + r] += l;
      atomicAdd(&grp[(g * 2 + k) * DY_BUCKETS + (63 - __clzll((long long)l))], 1ull);
      atomicAdd(&grp[4 * DY_BUCKETS + g * 2 + k], l);
    } else {
      atomicAdd(&grp[4 * DY_BUCKETS + 4 + g * 2 + k], 1ull);
      atomicAdd(&grp[4 * DY_BUCKETS + 8 + g * 2 + k], l);
    }
    *st = closed;
    *len = 1;
    *from = 1;
  }
}

// add one lane's value v at out[key] (key -1: none, and then v is 0).  Called by the whole warp.
__device__ __forceinline__ void dy_flush(int key, unsigned long long v, unsigned long long* __restrict__ out) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  if (!__any_sync(full, v != 0)) return;
  const unsigned grp = __match_any_sync(full, key);
  const int head = __ffs(grp) - 1;
  const unsigned span = grp >> head;  // contiguous: span + 1 is a power of two
  if (__all_sync(full, key < 0 || (span & (span + 1)) == 0)) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {  // segmented suffix sums inside each contiguous group
      const unsigned long long u = __shfl_down_sync(full, v, o);
      if (lane + o < 32 && ((grp >> (lane + o)) & 1u)) v += u;
    }
    if (lane != head) return;
  }
  if (key < 0 || v == 0) return;
  atomicAdd(&out[key], v);
}

__global__ void __launch_bounds__(DY_THREADS) k_dyn_bins(const double* __restrict__ x, const double* __restrict__ ring,
                                                        int n, int ring_len, long long s, const int* __restrict__ lags,
                                                        int n_active, const int* __restrict__ bin, int nbins,
                                                        unsigned long long* __restrict__ msd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // every lane of the warp takes part in the flushes
  const int b = i < n ? bin[i] : -1;
  const size_t o = 3 * (size_t)i;
  double xi = 0.0, yi = 0.0, zi = 0.0;
  if (b >= 0) {
    xi = x[o];
    yi = x[o + 1];
    zi = x[o + 2];
  }
  for (int k = 0; k < n_active; ++k) {
    unsigned long long q = 0;
    if (b >= 0) {
      const double* p = ring + dy_slot(s, lags[k], ring_len) * 3 * (size_t)n + o;
      q = mmm_quantise(mmm_pair_d2(xi, yi, zi, p[0], p[1], p[2]));
    }
    dy_flush(b, q, msd + (size_t)k * nbins);
  }
}

int dy_ready(mmm_system* h, const char* who) {
  if (!h->dy_configured) return mmm_fail(h, MMM_ERR_STATE, std::string(who) + ": call mmm_dynamics_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

}  // namespace

extern "C" int mmm_dynamics_configure(mmm_handle h, double rc_nm, const int32_t* lags, int32_t n_lags,
                                      const int32_t* bin_of_bead, int32_t n_bins, int32_t n_rows,
                                      const int32_t* bead_lo, const int32_t* bead_hi, const int8_t* group) {
  if (!h) return MMM_ERR_ARG;
  h->dy_configured = false;
  auto bad = [&](const std::string& why) { return mmm_fail(h, MMM_ERR_ARG, "mmm_dynamics_configure: " + why); };
  if (!(rc_nm > 0.0) || !isfinite(rc_nm)) return bad("rc must be finite and > 0");
  if (n_lags < 1 || !lags) return bad("the lag set is empty");
  for (int32_t k = 0; k < n_lags; ++k) {
    if (lags[k] < 1 || lags[k] > DY_MAX_LAG) return bad("lags must lie in [1, " + std::to_string(DY_MAX_LAG) + "]");
    if (k > 0 && lags[k] <= lags[k - 1]) return bad("lags must be strictly increasing");
  }
  if (n_rows < 0) return bad("n_rows must be >= 0");
  if (!bin_of_bead && n_rows == 0) return bad("neither bins nor rows: nothing to measure");
  const int64_t n = h->n;
  int64_t fullest = 0;
  if (bin_of_bead) {
    if (n_bins < 1 || n_bins > DY_MAX_BINS) return bad("n_bins must be in [1, 2^22]");
    std::vector<int64_t> occ((size_t)n_bins, 0);
    for (int64_t i = 0; i < n; ++i) {
      const int32_t b = bin_of_bead[i];
      if (b < -1 || b >= n_bins) return bad("bin id outside [-1, n_bins)");
      if (b >= 0) fullest = std::max(fullest, ++occ[(size_t)b]);
    }
  }
  if (n_rows > 0 && (!bead_lo || !bead_hi || !group)) return bad("a row array is NULL");
  std::vector<int4> rows((size_t)n_rows);
  for (int32_t r = 0; r < n_rows; ++r) {
    const std::string row = "row " + std::to_string(r) + ": ";
    if (bead_lo[r] < 0 || bead_hi[r] >= n) return bad(row + "an anchor bead lies outside [0, N)");
    if (bead_lo[r] >= bead_hi[r]) return bad(row + "bead_lo must be < bead_hi");
    if (group[r] != 0 && group[r] != 1) return bad(row + "group must be 0 or 1");
    rows[(size_t)r] = make_int4(bead_lo[r], bead_hi[r], group[r], 0);
  }
  cudaSetDevice(h->device);
  const int32_t nb = bin_of_bead ? n_bins : 0;
  const size_t ring_len = (size_t)lags[n_lags - 1];
  const size_t sums = (size_t)n_lags * ((size_t)nb + (size_t)n_rows) + 4 * (size_t)n_rows + DY_GROUP_SUMS;
  int rc;
  if ((rc = mmm_reserve(h, h->d_dy_ring, ring_len * 3 * (size_t)n, "dynamics ring")) ||
      (rc = mmm_reserve(h, h->d_dy_bin, (size_t)std::max<int64_t>(n, 1), "dynamics bins")) ||
      (rc = mmm_reserve(h, h->d_dy_lag, (size_t)n_lags, "dynamics lags")) ||
      (rc = mmm_reserve(h, h->d_dy_row, (size_t)std::max(n_rows, 1), "dynamics rows")) ||
      (rc = mmm_reserve(h, h->d_dy_state, 3 * (size_t)std::max(n_rows, 1), "dynamics run states")) ||
      (rc = mmm_reserve(h, h->d_dy_sum, sums, "dynamics sums"))) {
    cudaGetLastError();  // a failed cudaMalloc is not sticky: clear it, or the next launch check reports it
    return rc;
  }
  if (!h->dy_ev0) MMM_CUDA(h, cudaEventCreate(&h->dy_ev0));
  if (!h->dy_ev1) MMM_CUDA(h, cudaEventCreate(&h->dy_ev1));
  MMM_CUDA(h, cudaMemcpyAsync(h->d_dy_lag, lags, sizeof(int32_t) * (size_t)n_lags, cudaMemcpyHostToDevice, h->stream));
  if (nb)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_dy_bin, bin_of_bead, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, h->stream));
  if (n_rows > 0)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_dy_row, rows.data(), sizeof(int4) * rows.size(), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_dy_state, 0, sizeof(long long) * 3 * (size_t)std::max(n_rows, 1), h->stream));
  MMM_CUDA(h, cudaMemsetAsync(h->d_dy_sum, 0, sizeof(unsigned long long) * sums, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));  // rows is a host temporary
  h->dy_rc = rc_nm;
  h->dy_lags.assign(lags, lags + n_lags);
  h->dy_bins = nb;
  h->dy_rows = n_rows;
  h->dy_fullest = fullest;
  h->dy_samples = 0;
  h->dy_bound_bins = h->dy_bound_rows = 0.0;
  h->dy_ms = 0.f;
  h->dy_configured = true;
  return MMM_OK;
}

extern "C" int mmm_dynamics_add(mmm_handle h) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = dy_ready(h, "mmm_dynamics_add"))) return rc;
  cudaSetDevice(h->device);
  // the guard, before any kernel: a refused structure leaves the sums, the ring and the run states as they were.
  // Every position added so far lies in the union box of diagonal D, so one add puts at most qmax(D) into a
  // bead's cell (times the beads of the fullest bin) and qmax(2 D) into a row's: |R(s) - R(s - tau)| <= 2 D.
  double box[6];
  if ((rc = mmm_positions_box(h, box))) return rc;
  for (int c = 0; c < 6; ++c)
    if (!std::isfinite(box[c]))
      return mmm_fail(h, MMM_ERR_ARG, "mmm_dynamics_add: positions are not finite (no distance can be quantised)");
  double u[6], d2max = 0.0;
  for (int c = 0; c < 3; ++c) {
    u[c] = h->dy_samples ? std::min(h->dy_box[c], box[c]) : box[c];
    u[3 + c] = h->dy_samples ? std::max(h->dy_box[3 + c], box[3 + c]) : box[3 + c];
    d2max += (u[3 + c] - u[c]) * (u[3 + c] - u[c]);
  }
  double dpad, q1, q2, dpad2;
  mmm_qmax_of(d2max, &dpad, &q1);
  mmm_qmax_of(4.0 * d2max, &dpad2, &q2);
  const double bb = h->dy_bins ? (double)h->dy_fullest * q1 : 0.0;
  const double br = h->dy_rows ? q2 : 0.0;
  if (!std::isfinite(d2max) || h->dy_bound_bins + bb >= 0x1p63 || h->dy_bound_rows + br >= 0x1p63)
    return mmm_fail(h, MMM_ERR_ARG,
                    "mmm_dynamics_add: the sums could overflow int64 (" + std::to_string((long long)h->dy_fullest) +
                        " beads in the fullest bin, displacements up to " + std::to_string(dpad2) +
                        " nm at a quantum of 2^-24 nm" +
                        (h->dy_samples > 0 ? ", on top of the structures already summed" : "") + ")");
  const long long s = h->dy_samples;
  const int n = (int)h->n, nrows = (int)h->dy_rows, nb = h->dy_bins;
  const int ring_len = h->dy_lags.back();
  const int n_active = (int)(std::upper_bound(h->dy_lags.begin(), h->dy_lags.end(), (int)std::min<long long>(s, DY_MAX_LAG)) -
                             h->dy_lags.begin());  // the lags tau <= s
  const int n_lags = (int)h->dy_lags.size();
  unsigned long long* msd = h->d_dy_sum;
  unsigned long long* rel = msd + (size_t)n_lags * nb;
  unsigned long long* runs = rel + (size_t)n_lags * nrows;
  unsigned long long* grp = runs + 4 * (size_t)nrows;
  const size_t plane = 3 * (size_t)n;
  MMM_CUDA(h, cudaEventRecord(h->dy_ev0, h->stream));
  if (nrows > 0) {
    k_dyn_rows<<<(nrows + DY_ROW_THREADS - 1) / DY_ROW_THREADS, DY_ROW_THREADS, 0, h->stream>>>(
        h->d_x, h->d_dy_ring, plane, ring_len, s, h->d_dy_lag, n_active, h->d_dy_row, nrows, h->dy_rc * h->dy_rc,
        h->d_dy_state, rel, runs, grp);
    h->launches++;
  }
  if (nb > 0 && n_active > 0) {
    k_dyn_bins<<<(n + DY_THREADS - 1) / DY_THREADS, DY_THREADS, 0, h->stream>>>(
        h->d_x, h->d_dy_ring, n, ring_len, s, h->d_dy_lag, n_active, h->d_dy_bin, nb, msd);
    h->launches++;
  }
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(h->d_dy_ring + (size_t)(s % ring_len) * plane, h->d_x, sizeof(double) * plane,
                        cudaMemcpyDeviceToDevice, h->stream);
  if (e != cudaSuccess) {
    h->dy_configured = false;  // the sums may hold part of this structure: unusable until reconfigured
    return mmm_fail(h, MMM_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e) + " (mmm_dynamics_add)");
  }
  MMM_CUDA(h, cudaEventRecord(h->dy_ev1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->dy_ev0, h->dy_ev1);
  h->dy_ms += ms;
  std::copy(u, u + 6, h->dy_box);
  h->dy_bound_bins += bb;
  h->dy_bound_rows += br;
  h->dy_samples++;
  return MMM_OK;
}

extern "C" int mmm_dynamics_read(mmm_handle h, int64_t* samples_out, uint64_t* msd_sum_out, uint64_t* rel_msd_sum_out,
                                 float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = dy_ready(h, "mmm_dynamics_read"))) return rc;
  cudaSetDevice(h->device);
  const size_t nl = h->dy_lags.size(), nb = (size_t)h->dy_bins, nr = (size_t)h->dy_rows;
  if (msd_sum_out && nl * nb)
    MMM_CUDA(h, cudaMemcpyAsync(msd_sum_out, h->d_dy_sum, sizeof(uint64_t) * nl * nb, cudaMemcpyDeviceToHost, h->stream));
  if (rel_msd_sum_out && nl * nr)
    MMM_CUDA(h, cudaMemcpyAsync(rel_msd_sum_out, h->d_dy_sum + nl * nb, sizeof(uint64_t) * nl * nr,
                                cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (samples_out) *samples_out = h->dy_samples;
  if (device_ms_out) *device_ms_out = h->dy_ms;
  return MMM_OK;
}

extern "C" int mmm_dynamics_read_runs(mmm_handle h, uint64_t* row_runs_out, int8_t* closed_out, int64_t* length_out,
                                      int8_t* from_transition_out, uint64_t* hist_out, uint64_t* hist_len_out,
                                      uint64_t* left_runs_out, uint64_t* left_len_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = dy_ready(h, "mmm_dynamics_read_runs"))) return rc;
  cudaSetDevice(h->device);
  const size_t nl = h->dy_lags.size(), nr = (size_t)h->dy_rows;
  const unsigned long long* runs = h->d_dy_sum + nl * ((size_t)h->dy_bins + nr);
  std::vector<unsigned long long> grp(DY_GROUP_SUMS);
  std::vector<long long> st(3 * nr);
  if (row_runs_out && nr)
    MMM_CUDA(h, cudaMemcpyAsync(row_runs_out, runs, sizeof(uint64_t) * 4 * nr, cudaMemcpyDeviceToHost, h->stream));
  if (nr) MMM_CUDA(h, cudaMemcpyAsync(st.data(), h->d_dy_state, sizeof(long long) * st.size(), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(grp.data(), runs + 4 * nr, sizeof(uint64_t) * grp.size(), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  for (size_t r = 0; r < nr; ++r) {
    if (closed_out) closed_out[r] = (int8_t)st[r];
    if (length_out) length_out[r] = st[nr + r];
    if (from_transition_out) from_transition_out[r] = (int8_t)st[2 * nr + r];
  }
  uint64_t* outs[4] = {hist_out, hist_len_out, left_runs_out, left_len_out};
  const size_t at[4] = {0, 4 * DY_BUCKETS, 4 * DY_BUCKETS + 4, 4 * DY_BUCKETS + 8}, len[4] = {4 * DY_BUCKETS, 4, 4, 4};
  for (int k = 0; k < 4; ++k)
    if (outs[k]) std::copy(grp.begin() + at[k], grp.begin() + at[k] + len[k], outs[k]);
  return MMM_OK;
}
