// mmm_triplets.cu — three-way contact maps (simulated multi-way chromatin capture): every unordered bead triple
// i < j < k whose three pairs are contacts of mmm_contacts (d2 < rc^2 in FP64 on the master positions), i.e.
// every triangle of the contact graph, counted once, binned by a caller-given table and summed over any number
// of structures on the device.  A triple with a bead outside the map (bin -1) counts only in the total;
// otherwise its bins sorted into p <= q <= r give the key (p * B + q) * B + r (B <= 2^20, so keys < 2^60 and
// k_rle's "no key is ~0" holds).  uint64 integer sums: exact and independent of schedule and chunking.  No
// overflow guard: one structure adds at most N^3 / 6 to any count (the number of bead triples), and a contact
// graph of beads that exclude each other has a bounded degree, so real counts are orders of magnitude below.
//
// Per add:
//   mmm_contacts_sparse_pass at identity bins (n_bins = N) into the accumulator's own buffers: the sorted unique
//     keys i * N + j (i < j), the forward adjacency in CSR order
//   k_tp_rows              row[i] = first key of bead i (binary search), row[N] = contacts
//   k_triplets<kTpCount>   binned triples per bead i and all triples -> exclusive scan (cs_scan) -> offsets
//   host: bead ranges [i0, i1) of at most max_chunk_keys keys each (a chunk holds one bead at least); per chunk
//     k_triplets<kTpKeys>  the keys of bead i at its offset, no atomics: a deterministic order
//     cs_sort_runs         LSD radix sort over ceil(log2 B^3) bits, runs of equal keys
//     mmm_list_accumulate  run reduction, merge-path merge with the accumulated list, equal keys added
// Scratch: O(N + contacts + chunk keys), never O(triples): the default chunk (2^26 keys) sorts in 1 GiB.
//
// k_triplets: one warp per bead i.  fwd(i) (d entries) is staged in shared memory when d <= TP_ROW_SMEM (else
// read from global memory).  32 j of fwd(i) at a time: lane a holds j and deg(j) = |fwd(j)|, an inclusive warp
// scan of the degrees numbers the wedges (i, j, k in fwd(j)) of the 32, and the lanes take consecutive wedges
// (each finds its j by a 5-step binary search over the scan with shuffles), so every lane works whatever the
// degrees.  A wedge closes when k is in fwd(i), found by binary search over fwd(i) after j's position (k > j).
// Pass 2 sees the same wedges in the same order, so it writes exactly the keys pass 1 counted.
//
// The add reads d_x and writes only the FP32 copy (which every evaluation rewrites from d_x before reading it)
// and the accumulator's own buffers: nothing an evaluation, a minimisation, an MD step, mmm_last_result, the
// one-shot sparse map, the trajectory sampler or the loop readout reads.
#include <math.h>

#include <algorithm>
#include <string>
#include <vector>

#include "mmm_internal.cuh"

namespace {

constexpr int TP_WARPS = 8;            // beads per CTA
constexpr int TP_ROW_SMEM = 512;       // fwd(i) entries staged per warp (16 KB per CTA)
constexpr int32_t TP_MAX_BINS = 1 << 20;
constexpr int64_t TP_DEFAULT_CHUNK = 1ll << 26;

enum TpSink { kTpCount, kTpKeys };

__global__ void __launch_bounds__(256) k_tp_rows(const unsigned long long* __restrict__ adj, long long m, int n,
                                                 long long* __restrict__ row) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  const unsigned long long key = (unsigned long long)i * (unsigned)n;  // first key bead i can have
  long long lo = 0, hi = m;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (adj[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  row[i] = lo;
}

// Beads [i0, i1).  kTpCount: off[i] = binned triples of bead i, total += all its triples.  kTpKeys: the keys of
// bead i at keys[off[i] - key0] (off scanned).
template <TpSink kSink>
__global__ void __launch_bounds__(TP_WARPS * 32) k_triplets(const unsigned long long* __restrict__ adj,
                                                            const long long* __restrict__ row,
                                                            const int* __restrict__ bin, int n, int i0, int i1,
                                                            unsigned long long nb, long long* __restrict__ off,
                                                            unsigned long long* __restrict__ total,
                                                            unsigned long long* __restrict__ keys, long long key0) {
  __shared__ int s_fwd[TP_WARPS][TP_ROW_SMEM];
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = i0 + blockIdx.x * TP_WARPS + w;
  if (i >= i1) return;  // whole warps only; no CTA-wide barrier below
  const long long lo = row[i];
  const int d = (int)(row[i + 1] - lo);
  const unsigned long long ibase = (unsigned long long)i * (unsigned)n;
  const bool staged = d <= TP_ROW_SMEM;
  int* fwd = s_fwd[w];
  if (staged)
    for (int t = lane; t < d; t += 32) fwd[t] = (int)(adj[lo + t] - ibase);
  __syncwarp();
  const int bi = bin[i];
  long long kpos = kSink == kTpKeys ? off[i] - key0 : 0;  // next key slot of this bead (warp-uniform)
  unsigned long long ntri = 0;
  for (int a0 = 0; a0 < d - 1; a0 += 32) {  // j = fwd(i)[a]; the last j closes no triangle (no k > j in fwd(i))
    const int a = a0 + lane;
    int j = 0, dj = 0, bj = -1;
    long long sj = 0;
    if (a < d - 1) {
      j = staged ? fwd[a] : (int)(adj[lo + a] - ibase);
      sj = row[j];
      dj = (int)(row[j + 1] - sj);
      bj = bin[j];
    }
    int inc = dj;  // inclusive scan of the degrees: wedges of lanes 0..lane
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(full, inc, o);
      if (lane >= o) inc += u;
    }
    const int seg = __shfl_sync(full, inc, 31);
    for (int w0 = 0; w0 < seg; w0 += 32) {
      const int pos = w0 + lane;
      int src = 0;  // the lane whose wedges hold pos: the number of lanes with inc <= pos
#pragma unroll
      for (int b = 16; b > 0; b >>= 1)
        if (__shfl_sync(full, inc, src + b - 1) <= pos) src += b;
      const int before = __shfl_sync(full, inc - dj, src);
      const long long s = __shfl_sync(full, sj, src);
      const int jj = __shfl_sync(full, j, src), bjj = __shfl_sync(full, bj, src);
      bool tri = false;
      int k = 0;
      if (pos < seg) {
        k = (int)(adj[s + (pos - before)] - (unsigned long long)jj * (unsigned)n);
        int l = a0 + src + 1, r = d;  // fwd(i) is sorted and k > j = fwd(i)[a0 + src]
        while (l < r) {
          const int mid = (l + r) >> 1;
          const int v = staged ? fwd[mid] : (int)(adj[lo + mid] - ibase);
          if (v < k) l = mid + 1;
          else r = mid;
        }
        tri = l < d && (staged ? fwd[l] : (int)(adj[lo + l] - ibase)) == k;
      }
      ntri += tri ? 1ull : 0ull;
      const int bk = tri ? bin[k] : -1;
      const bool binned = tri && bi >= 0 && bjj >= 0 && bk >= 0;
      const unsigned em = __ballot_sync(full, binned);
      if (kSink == kTpKeys && binned) {
        const int p = min(bi, min(bjj, bk)), r = max(bi, max(bjj, bk));
        const int q = bi + bjj + bk - p - r;
        keys[kpos + __popc(em & ((1u << lane) - 1u))] =
            ((unsigned long long)p * nb + (unsigned long long)q) * nb + (unsigned long long)r;
      }
      kpos += __popc(em);
    }
  }
  if constexpr (kSink == kTpCount) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ntri += __shfl_xor_sync(full, ntri, o);
    if (lane == 0) {
      off[i] = kpos;
      if (ntri) atomicAdd(total, ntri);
    }
  }
}

int tp_ready(mmm_system* h, const char* who) {
  if (!h->tp_configured) return mmm_fail(h, MMM_ERR_STATE, std::string(who) + ": call mmm_triplets_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

// the structure at the current positions, into the accumulator; *chunks = the chunks it used
int tp_add(mmm_system* h, int64_t* chunks) {
  const int n = (int)h->n;
  int rc;
  CsSorted srt;
  if ((rc = mmm_contacts_sparse_pass(h, h->tp_rc, h->d_tp_ident, n, h->d_tp_tile, h->d_tp_adj, h->d_tp_table,
                                     h->d_tp_cnt, nullptr, nullptr, &srt)))
    return rc;
  const unsigned long long* adj = h->d_tp_adj[srt.src];
  const long long nparts = cs_blocks(n + 1);
  if ((rc = mmm_reserve(h, h->d_tp_row, (size_t)n + 1, "triplet rows")) ||
      (rc = mmm_reserve(h, h->d_tp_off, (size_t)(n + 1 + nparts + 1), "triplet offsets")))
    return rc;
  long long* off = h->d_tp_off;
  k_tp_rows<<<(n + 1 + 255) / 256, 256, 0, h->stream>>>(adj, srt.keys, n, h->d_tp_row);
  MMM_CUDA(h, cudaMemsetAsync(h->d_tp_cnt + 2, 0, sizeof(unsigned long long), h->stream));
  MMM_CUDA(h, cudaMemsetAsync(off + n, 0, sizeof(long long), h->stream));  // off[n] becomes the binned total
  const unsigned long long nb = (unsigned long long)h->tp_bins;
  const int ctas = (n + TP_WARPS - 1) / TP_WARPS;
  k_triplets<kTpCount><<<ctas, TP_WARPS * 32, 0, h->stream>>>(adj, h->d_tp_row, h->d_tp_bin, n, 0, n, nb, off,
                                                              h->d_tp_cnt + 2, nullptr, 0);
  h->launches += 2;
  cs_scan(h, off, n + 1, off + n + 1);
  MMM_CUDA(h, cudaGetLastError());
  std::vector<long long> hoff((size_t)n + 1);
  unsigned long long triples = 0;
  MMM_CUDA(h, cudaMemcpyAsync(hoff.data(), off, sizeof(long long) * hoff.size(), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(&triples, h->d_tp_cnt + 2, sizeof(triples), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  // bead ranges of at most tp_max_chunk keys (one bead with keys at least), greedily from bead 0
  std::vector<std::pair<int, int>> ranges;
  long long most = 0;
  for (int i0 = 0; i0 < n && hoff[(size_t)i0] < hoff[(size_t)n];) {
    // from the first bead with keys: the last i with off[i] = off[i0]
    i0 = (int)(std::upper_bound(hoff.begin() + i0, hoff.end(), hoff[(size_t)i0]) - hoff.begin()) - 1;
    int i1 = (int)(std::upper_bound(hoff.begin() + i0 + 1, hoff.end(), hoff[(size_t)i0] + h->tp_max_chunk) -
                   hoff.begin()) - 1;
    i1 = std::max(i1, i0 + 1);
    ranges.emplace_back(i0, i1);
    most = std::max(most, hoff[(size_t)i1] - hoff[(size_t)i0]);
    i0 = i1;
  }
  if ((rc = mmm_reserve(h, h->d_tp_keys[0], (size_t)most, "triplet keys")) ||
      (rc = mmm_reserve(h, h->d_tp_keys[1], (size_t)most, "triplet keys")) ||
      (rc = mmm_reserve(h, h->d_tp_table, cs_table_len(most), "triplet sort table")))
    return rc;
  // keys < B^3: sort on ceil(log2(B^3)) bits
  const int bits = cs_key_bits(nb * nb * nb - 1ull);
  for (const auto& rg : ranges) {
    const long long key0 = hoff[(size_t)rg.first], m = hoff[(size_t)rg.second] - key0;
    k_triplets<kTpKeys><<<(rg.second - rg.first + TP_WARPS - 1) / TP_WARPS, TP_WARPS * 32, 0, h->stream>>>(
        adj, h->d_tp_row, h->d_tp_bin, n, rg.first, rg.second, nb, off, nullptr, h->d_tp_keys[0], key0);
    h->launches++;
    const int src = cs_sort_runs(h, h->d_tp_keys, m, bits, h->d_tp_table);
    MMM_CUDA(h, cudaGetLastError());
    long long entries = 0;
    MMM_CUDA(h, cudaMemcpyAsync(&entries, cs_run_total(h->d_tp_table, m), sizeof(entries), cudaMemcpyDeviceToHost,
                                h->stream));
    MMM_CUDA(h, cudaStreamSynchronize(h->stream));
    if ((rc = mmm_list_accumulate(h, h->d_tp_keys[src], m, h->d_tp_table, entries, h->d_tp_keys[1 - src], h->tp_acc)))
      return rc;
  }
  h->tp_triples += triples;
  *chunks = (int64_t)ranges.size();
  return MMM_OK;
}

}  // namespace

extern "C" int mmm_triplets_configure(mmm_handle h, double rc_nm, const int32_t* bin_of_bead, int32_t n_bins,
                                      int64_t max_chunk_keys) {
  if (!h) return MMM_ERR_ARG;
  h->tp_configured = false;
  const char* who = "mmm_triplets_configure: ";
  if (!(rc_nm > 0.0) || !isfinite(rc_nm)) return mmm_fail(h, MMM_ERR_ARG, std::string(who) + "rc must be finite and > 0");
  if (n_bins < 1 || n_bins > TP_MAX_BINS)
    return mmm_fail(h, MMM_ERR_ARG, std::string(who) + "n_bins must be in [1, 2^20]");
  if (!bin_of_bead) return mmm_fail(h, MMM_ERR_ARG, std::string(who) + "bin_of_bead is NULL");
  for (int64_t i = 0; i < h->n; ++i)
    if (bin_of_bead[i] < -1 || bin_of_bead[i] >= n_bins)
      return mmm_fail(h, MMM_ERR_ARG, std::string(who) + "bin id outside [-1, n_bins)");
  if (max_chunk_keys < 0) return mmm_fail(h, MMM_ERR_ARG, std::string(who) + "max_chunk_keys must be >= 0");
  cudaSetDevice(h->device);
  const size_t n = (size_t)h->n;
  int rc;
  if ((rc = mmm_reserve(h, h->d_tp_ident, n, "triplet identity bins")) ||
      (rc = mmm_reserve(h, h->d_tp_bin, n, "triplet bins")) ||
      (rc = mmm_reserve(h, h->d_tp_cnt, 3, "triplet counters")))
    return rc;
  if (!h->tp_ev0) MMM_CUDA(h, cudaEventCreate(&h->tp_ev0));
  if (!h->tp_ev1) MMM_CUDA(h, cudaEventCreate(&h->tp_ev1));
  std::vector<int32_t> ident(n);
  for (size_t i = 0; i < n; ++i) ident[i] = (int32_t)i;
  MMM_CUDA(h, cudaMemcpyAsync(h->d_tp_ident, ident.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(h->d_tp_bin, bin_of_bead, sizeof(int32_t) * n, cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));  // the host tables may go away after the call
  h->tp_rc = rc_nm;
  h->tp_bins = n_bins;
  h->tp_max_chunk = max_chunk_keys > 0 ? max_chunk_keys : TP_DEFAULT_CHUNK;
  h->tp_samples = h->tp_chunks = 0;
  h->tp_triples = 0;
  h->tp_ms = 0.f;
  h->tp_acc.n = 0;
  h->tp_configured = true;
  return MMM_OK;
}

extern "C" int mmm_triplets_add(mmm_handle h) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = tp_ready(h, "mmm_triplets_add"))) return rc;
  cudaSetDevice(h->device);
  MMM_CUDA(h, cudaEventRecord(h->tp_ev0, h->stream));
  int64_t chunks = 0;
  if ((rc = tp_add(h, &chunks))) {
    h->tp_configured = false;  // the list may hold part of this structure: unusable until reconfigured
    return rc;
  }
  MMM_CUDA(h, cudaEventRecord(h->tp_ev1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, h->tp_ev0, h->tp_ev1);
  h->tp_ms += ms;
  h->tp_chunks += chunks;
  h->tp_samples++;
  return MMM_OK;
}

extern "C" int mmm_triplets_read(mmm_handle h, int64_t* samples_out, uint64_t* triples_out, int64_t* entries_out,
                                 int64_t* chunks_out, float* device_ms_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = tp_ready(h, "mmm_triplets_read"))) return rc;
  if (samples_out) *samples_out = h->tp_samples;
  if (triples_out) *triples_out = h->tp_triples;
  if (entries_out) *entries_out = h->tp_acc.n;
  if (chunks_out) *chunks_out = h->tp_chunks;
  if (device_ms_out) *device_ms_out = h->tp_ms;
  return MMM_OK;
}

extern "C" int mmm_triplets_read_entries(mmm_handle h, uint64_t* keys_out, uint64_t* vals_out) {
  if (!h) return MMM_ERR_ARG;
  int rc;
  if ((rc = tp_ready(h, "mmm_triplets_read_entries"))) return rc;
  const size_t e = (size_t)h->tp_acc.n;
  if (e == 0) return MMM_OK;
  cudaSetDevice(h->device);
  if (keys_out)
    MMM_CUDA(h, cudaMemcpyAsync(keys_out, h->tp_acc.key[0], sizeof(uint64_t) * e, cudaMemcpyDeviceToHost, h->stream));
  if (vals_out)
    MMM_CUDA(h, cudaMemcpyAsync(vals_out, h->tp_acc.val[0], sizeof(uint64_t) * e, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}
