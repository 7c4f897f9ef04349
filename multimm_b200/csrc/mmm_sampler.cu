// mmm_sampler.cu — the trajectory sampler: contact, fine contact and distance maps summed over any number of
// structures (the states of an MD run) on the device, and read back once.
//
// Every sum is an integer sum, so adding structures is exact and independent of order: after K calls of
// mmm_sample the dense map, sep, pairs and both distance maps equal bit for bit the sums of what
// mmm_contacts and mmm_distance_map return at the same K positions (the same passes run, into the sampler's
// accumulators without clearing them), and the fine map equals the sorted union of the K maps of
// mmm_contacts_sparse with the counts of equal keys added (mmm_contacts_fine_accumulate: a per-structure
// run reduction and a merge-path merge into the accumulated list).  The distance pass's int64 guard is
// cumulative: a structure whose bound would take the summed bounds to 2^63 is refused before any pass runs.
//
// Like the one-shot passes the sampler reads d_x and writes only the FP32 copy (which every evaluation
// rewrites from d_x before reading it) and scratch; its accumulators and the fine map's buffers are its own.
#include <math.h>

#include <string>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int SP_MAX_BINS = 4096;  // the dense contact map and the distance maps

// a bin table of n beads: NULL (map off) or ids in [-1, n_bins) with n_bins in [1, max_bins]
int sp_check_bins(mmm_system* h, const char* what, const int32_t* bins, int32_t n_bins, int32_t max_bins) {
  if (!bins) return MMM_OK;
  if (n_bins < 1 || n_bins > max_bins)
    return mmm_fail(h, MMM_ERR_ARG, std::string("mmm_sampler_configure: ") + what + " n_bins must be in [1, " +
                                        std::to_string(max_bins) + "]");
  for (int64_t i = 0; i < h->n; ++i)
    if (bins[i] < -1 || bins[i] >= n_bins)
      return mmm_fail(h, MMM_ERR_ARG, std::string("mmm_sampler_configure: ") + what + " bin id outside [-1, n_bins)");
  return MMM_OK;
}

int sp_ready(mmm_system* h, const char* who) {
  if (!h->sp_configured) return mmm_fail(h, MMM_ERR_STATE, std::string(who) + ": call mmm_sampler_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

// the passes of one structure, into the accumulators
int sp_add(mmm_system* h) {
  int rc;
  if (h->sp_ct_bins &&
      (rc = mmm_contacts_dense_pass(h, h->sp_rc, h->d_sp_ct_bin, h->sp_ct_bins, h->d_sp_map, h->d_sp_sep, h->d_sp_cnt,
                                    false, nullptr)))
    return rc;
  const size_t dcells = (size_t)h->sp_dm_bins * (size_t)h->sp_dm_bins;
  if (h->sp_dm_bins &&
      (rc = mmm_distance_pass(h, h->d_sp_dm_bin, h->sp_dm_bins, h->d_sp_dist, h->d_sp_dist + dcells, false)))
    return rc;
  if (h->sp_fine_bins && (rc = mmm_contacts_fine_accumulate(h))) return rc;
  return MMM_OK;
}

}  // namespace

extern "C" int mmm_sampler_configure(mmm_handle h, double rc_nm, const int32_t* contact_bins, int32_t n_contact_bins,
                                     const int32_t* fine_bins, int32_t n_fine_bins, const int32_t* distance_bins,
                                     int32_t n_distance_bins) {
  if (!h) return MMM_ERR_ARG;
  h->sp_configured = false;
  int rc;
  if (!contact_bins && !distance_bins)
    return mmm_fail(h, MMM_ERR_ARG, "mmm_sampler_configure: no map to sample (contact_bins and distance_bins NULL)");
  if (fine_bins && !contact_bins)
    return mmm_fail(h, MMM_ERR_ARG, "mmm_sampler_configure: the fine map needs contact_bins");
  if (contact_bins && (!(rc_nm > 0.0) || !isfinite(rc_nm)))
    return mmm_fail(h, MMM_ERR_ARG, "mmm_sampler_configure: rc must be finite and > 0");
  if ((rc = sp_check_bins(h, "contact", contact_bins, n_contact_bins, SP_MAX_BINS)) ||
      (rc = sp_check_bins(h, "fine", fine_bins, n_fine_bins, INT32_MAX)) ||
      (rc = sp_check_bins(h, "distance", distance_bins, n_distance_bins, SP_MAX_BINS)))
    return rc;
  cudaSetDevice(h->device);
  const size_t n = (size_t)h->n;
  const size_t ccells = contact_bins ? (size_t)n_contact_bins * (size_t)n_contact_bins : 0;
  const size_t dcells = distance_bins ? (size_t)n_distance_bins * (size_t)n_distance_bins : 0;
  if ((rc = mmm_reserve(h, h->d_sp_cnt, 4, "sampler counters")) ||
      (contact_bins && ((rc = mmm_reserve(h, h->d_sp_ct_bin, n, "sampler contact bins")) ||
                        (rc = mmm_reserve(h, h->d_sp_map, ccells, "sampler contact map")) ||
                        (rc = mmm_reserve(h, h->d_sp_sep, n, "sampler contacts by separation")))) ||
      (fine_bins && (rc = mmm_reserve(h, h->d_sp_fine_bin, n, "sampler fine bins"))) ||
      (distance_bins && ((rc = mmm_reserve(h, h->d_sp_dm_bin, n, "sampler distance bins")) ||
                         (rc = mmm_reserve(h, h->d_sp_dist, 2 * dcells, "sampler distance maps")))))
    return rc;
  if (!h->sp_ev0) MMM_CUDA(h, cudaEventCreate(&h->sp_ev0));
  if (!h->sp_ev1) MMM_CUDA(h, cudaEventCreate(&h->sp_ev1));
  MMM_CUDA(h, cudaMemsetAsync(h->d_sp_cnt, 0, sizeof(unsigned long long) * 4, h->stream));
  if (contact_bins) {
    MMM_CUDA(h, cudaMemcpyAsync(h->d_sp_ct_bin, contact_bins, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
    MMM_CUDA(h, cudaMemsetAsync(h->d_sp_map, 0, sizeof(unsigned long long) * ccells, h->stream));
    MMM_CUDA(h, cudaMemsetAsync(h->d_sp_sep, 0, sizeof(unsigned long long) * n, h->stream));
  }
  if (fine_bins)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_sp_fine_bin, fine_bins, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
  h->sp_dm_occ.assign(distance_bins ? (size_t)n_distance_bins : 0, 0);
  if (distance_bins) {
    for (size_t i = 0; i < n; ++i)
      if (distance_bins[i] >= 0) ++h->sp_dm_occ[(size_t)distance_bins[i]];
    MMM_CUDA(h, cudaMemcpyAsync(h->d_sp_dm_bin, distance_bins, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
    MMM_CUDA(h, cudaMemsetAsync(h->d_sp_dist, 0, sizeof(unsigned long long) * 2 * dcells, h->stream));
  }
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));  // the host tables may go away after the call
  h->sp_rc = rc_nm;
  h->sp_ct_bins = contact_bins ? n_contact_bins : 0;
  h->sp_fine_bins = fine_bins ? n_fine_bins : 0;
  h->sp_dm_bins = distance_bins ? n_distance_bins : 0;
  h->sp_samples = 0;
  h->sp_dm_bound = 0.0;
  h->sp_ms = 0.f;
  h->sp_fine.n = 0;
  h->sp_configured = true;
  return MMM_OK;
}

extern "C" int mmm_sample(mmm_handle h) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = sp_ready(h, "mmm_sample"))) return rc;
  cudaSetDevice(h->device);
  double bound = 0.0;  // checked before any pass runs: a refused structure leaves every accumulator as it was
  if (h->sp_dm_bins && (rc = mmm_distance_guard(h, "mmm_sample", h->sp_dm_occ, h->sp_dm_bound, &bound))) return rc;
  MMM_CUDA(h, cudaEventRecord(h->sp_ev0, h->stream));
  if ((rc = sp_add(h))) {
    h->sp_configured = false;  // the maps may hold part of this structure: unusable until reconfigured
    return rc;
  }
  MMM_CUDA(h, cudaEventRecord(h->sp_ev1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->sp_ev0, h->sp_ev1);
  h->sp_ms += ms;
  h->sp_dm_bound += bound;
  h->sp_samples++;
  return MMM_OK;
}

extern "C" int mmm_sampler_read(mmm_handle h, int64_t* samples_out, uint64_t* contact_map_out, uint64_t* sep_out,
                                int64_t* pairs_out, int64_t* fine_entries_out, uint64_t* dist_sum_out,
                                uint64_t* dist2_sum_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = sp_ready(h, "mmm_sampler_read"))) return rc;
  cudaSetDevice(h->device);
  unsigned long long cnt[2] = {0, 0};
  const size_t ccells = (size_t)h->sp_ct_bins * (size_t)h->sp_ct_bins;
  const size_t dcells = (size_t)h->sp_dm_bins * (size_t)h->sp_dm_bins;
  MMM_CUDA(h, cudaMemcpyAsync(cnt, h->d_sp_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, h->stream));
  if (h->sp_ct_bins && contact_map_out)
    MMM_CUDA(h, cudaMemcpyAsync(contact_map_out, h->d_sp_map, sizeof(uint64_t) * ccells, cudaMemcpyDeviceToHost, h->stream));
  if (h->sp_ct_bins && sep_out)
    MMM_CUDA(h, cudaMemcpyAsync(sep_out, h->d_sp_sep, sizeof(uint64_t) * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
  if (h->sp_dm_bins && dist_sum_out)
    MMM_CUDA(h, cudaMemcpyAsync(dist_sum_out, h->d_sp_dist, sizeof(uint64_t) * dcells, cudaMemcpyDeviceToHost, h->stream));
  if (h->sp_dm_bins && dist2_sum_out)
    MMM_CUDA(h, cudaMemcpyAsync(dist2_sum_out, h->d_sp_dist + dcells, sizeof(uint64_t) * dcells, cudaMemcpyDeviceToHost,
                                h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (samples_out) *samples_out = h->sp_samples;
  if (h->sp_ct_bins && pairs_out) *pairs_out = (int64_t)cnt[0];
  if (fine_entries_out) *fine_entries_out = h->sp_fine.n;
  if (device_ms_out) *device_ms_out = h->sp_ms;
  return MMM_OK;
}

extern "C" int mmm_sampler_read_fine(mmm_handle h, int32_t* rows_out, int32_t* cols_out, uint64_t* vals_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = sp_ready(h, "mmm_sampler_read_fine"))) return rc;
  cudaSetDevice(h->device);
  return mmm_contacts_fine_read(h, rows_out, cols_out, vals_out);
}
