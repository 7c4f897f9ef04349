// mmm_chb_clusters.cu — the far field on cluster centroids: what the COARSE stage of the opt-in
// two-stage minimisation adds to the truncated pair pass (mmm_set_chb_surrogate; never in exact mode,
// never by default in cut-off mode).
//
// A potential truncated at rc = 0.5 nm misses two long-range pieces of the reference's energy, and a
// minimum of the truncated potential is not close to a minimum of the exact one without them:
//   * CHB's polynomial dE (kC r^4 - r^3 + r^2) (model.py:416-419) grows with r and cannot be truncated
//     at all — plain cut-off mode pays an exact pass over every same-chromosome pair for it (1.08e9
//     pairs at N = 2e5, more than the truncated pass itself);
//   * the tail of the EV power law beyond rc (model.py:199) is weak per pair but adds up to an outward
//     pressure on the whole globule; without it the exact stage has to swell the structure, a collective
//     move that costs L-BFGS hundreds of iterations (measured: 460-680 in five replicas of eight).
// Both are smooth at these distances, so they are evaluated between CLUSTERS: runs of at most 32
// consecutive beads of one chromosome (the 32-bead tiles of the chain order, split where the chromosome
// changes), with c_T the centroid and n_T the size,
//     E_far = sum_{T < U} n_T n_U [ same_chromosome(T, U) dE f(R) + S(R) eps (sigma / (R + r_s))^p ],
//     R = |c_T - c_U|,  f(r) = kC r^4 - r^3 + r^2,  S = smoothstep from 0 at 0.7 rc to 1 at 1.3 rc
// (bead pairs with r < rc are the truncated pass's; S hands over around rc).  It is a proper potential
// — a function of the positions through the centroids — whose gradient is exact: every bead of T feels
// -dE_far/dc_T / n_T, so L-BFGS's line search stays consistent.  O(N + clusters^2): 3.9e7 cluster pairs
// at N = 2e5 instead of 1.08e9 + 2e10 bead pairs.
//   k_cl_centroid   one warp per cluster: FP64 centroid of its beads             24 B read per bead
//   k_cl_forces     one warp per cluster, lanes stride over all clusters (FP64), one energy slot per cluster
// k_assemble adds the cluster's force to each of its beads.
// (Measured and dropped, calls 18 / 19: FP32 pair arithmetic on FP64 deltas in k_cl_forces.  The coarse
// evaluation went from 1.161 to 1.095 ms, but 5 of 16 ensemble members then needed a second coarse round
// against 1 of 16 — the rounding noise of the FP32 pair energies, ~1 kJ/mol in the total, is of the order
// of L-BFGS's last decreases, and the coarse stage's line search gives up early.  FP64 stays.)
#include <algorithm>

#include "mmm_internal.cuh"

namespace {

__global__ void __launch_bounds__(256) k_cl_centroid(const double* __restrict__ x, const int* __restrict__ cl_start,
                                                     int ncl, double* __restrict__ cen, const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= ncl) return;
  const int b0 = cl_start[c], b1 = cl_start[c + 1];
  double sx = 0.0, sy = 0.0, sz = 0.0;
  const int i = b0 + lane;
  if (i < b1) { sx = x[3 * (size_t)i]; sy = x[3 * (size_t)i + 1]; sz = x[3 * (size_t)i + 2]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sx += __shfl_xor_sync(0xffffffffu, sx, o);
    sy += __shfl_xor_sync(0xffffffffu, sy, o);
    sz += __shfl_xor_sync(0xffffffffu, sz, o);
  }
  if (lane == 0) {
    const double inv = 1.0 / (double)(b1 - b0);
    cen[4 * (size_t)c] = sx * inv;
    cen[4 * (size_t)c + 1] = sy * inv;
    cen[4 * (size_t)c + 2] = sz * inv;
    cen[4 * (size_t)c + 3] = (double)(b1 - b0);
  }
}

struct FarArgs {
  const double* cen;     // [ncl][4] centroid, size
  const int* chrom;      // [ncl]
  int ncl;
  int chb_on, ev_on;
  double kc, de;                 // CHB
  double eps, rs, sigma, power;  // EV
  int ipower;                    // the power as an integer, 0 if it is not one
  double r_lo, r_hi;             // S(R): 0 below r_lo, 1 above r_hi
  double* force;         // [ncl][3]
  double* epair_slots;   // [ncl][4]: EV tail in slot 0, CHB in slot 3
  const int* skip;
};

// One warp per cluster T; the CTA's 8 warps walk all clusters U together, 256 at a time through shared
// memory (as planes: conflict-free).  Without the staging every warp streamed the whole centroid table
// (200 KB at N = 2e5) from L2 on its own: 1.4 GB per launch, and the kernel was L2-bound at 0.30 ms; lane l
// still takes U = l, l + 32, ... in ascending order (same summation order as before).
constexpr int CL_CHUNK = 256;
__global__ void __launch_bounds__(256) k_cl_forces(const FarArgs A) {
  __shared__ double s_x[CL_CHUNK], s_y[CL_CHUNK], s_z[CL_CHUNK], s_n[CL_CHUNK];
  __shared__ int s_c[CL_CHUNK];
  if (A.skip && *A.skip) return;
  const int tid = threadIdx.x, lane = tid & 31;
  const int T = blockIdx.x * (blockDim.x >> 5) + (tid >> 5);
  const bool live = T < A.ncl;
  const int Tc = live ? T : 0;
  const double cx = A.cen[4 * (size_t)Tc], cy = A.cen[4 * (size_t)Tc + 1], cz = A.cen[4 * (size_t)Tc + 2], nT = A.cen[4 * (size_t)Tc + 3];
  const int chT = A.chrom[Tc];
  const double inv_band = 1.0 / (A.r_hi - A.r_lo);
  double fx = 0.0, fy = 0.0, fz = 0.0, e_ev = 0.0, e_chb = 0.0;
  for (int base = 0; base < A.ncl; base += CL_CHUNK) {
    __syncthreads();  // the previous chunk has been consumed
    if (base + tid < A.ncl) {
      const double2 c01 = *reinterpret_cast<const double2*>(A.cen + 4 * (size_t)(base + tid));
      const double2 c23 = *reinterpret_cast<const double2*>(A.cen + 4 * (size_t)(base + tid) + 2);
      s_x[tid] = c01.x; s_y[tid] = c01.y; s_z[tid] = c23.x; s_n[tid] = c23.y;
      s_c[tid] = A.chrom[base + tid];
    }
    __syncthreads();
    if (!live) continue;
    const int cnt = min(CL_CHUNK, A.ncl - base);
    for (int q = lane; q < cnt; q += 32) {
      if (base + q == T) continue;
      const double dx = cx - s_x[q], dy = cy - s_y[q], dz = cz - s_z[q];
      const double nU = s_n[q];
      // one reciprocal square root instead of a square root and a division by r (the kernel is FP64-bound)
      const double r2 = fmax(dx * dx + dy * dy + dz * dz, 1e-300), inv_r = rsqrt(r2), r = r2 * inv_r;
      double g = 0.0;  // -dE/dR / R per unit n_T
      if (A.chb_on && s_c[q] == chT) {
        e_chb += nU * r2 * (A.kc * r2 - r + 1.0);
        g -= A.de * nU * (4.0 * A.kc * r2 - 3.0 * r + 2.0);
      }
      if (A.ev_on && r > A.r_lo) {
        const double w = 1.0 / (r + A.rs), sw = A.sigma * w;
        double wp;
        if (A.ipower == 6) { const double s2 = sw * sw; wp = s2 * s2 * s2; }
        else if (A.ipower == 3) wp = sw * sw * sw;
        else wp = pow(sw, A.power);
        const double u = A.eps * wp, du = -A.power * u * w;
        double sR = 1.0, dsR = 0.0;
        if (r < A.r_hi) {
          const double t = (r - A.r_lo) * inv_band;
          sR = t * t * (3.0 - 2.0 * t);
          dsR = 6.0 * t * (1.0 - t) * inv_band;
        }
        e_ev += nU * u * sR;
        g -= nU * (du * sR + u * dsR) * inv_r;
      }
      fx += g * dx; fy += g * dy; fz += g * dz;
    }
  }
  if (!live) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    fx += __shfl_xor_sync(0xffffffffu, fx, o);
    fy += __shfl_xor_sync(0xffffffffu, fy, o);
    fz += __shfl_xor_sync(0xffffffffu, fz, o);
    e_ev += __shfl_xor_sync(0xffffffffu, e_ev, o);
    e_chb += __shfl_xor_sync(0xffffffffu, e_chb, o);
  }
  if (lane == 0) {
    A.force[3 * (size_t)T] = fx;
    A.force[3 * (size_t)T + 1] = fy;
    A.force[3 * (size_t)T + 2] = fz;
    double* slot = A.epair_slots + 4 * (size_t)T;
    slot[0] = 0.5 * nT * e_ev;  // every cluster pair is seen from both sides
    slot[1] = 0.0;
    slot[2] = 0.0;
    slot[3] = 0.5 * nT * A.de * e_chb;
  }
}

}  // namespace

int mmm_chb_clusters_blocks(const mmm_system* h) { return h->n_clusters; }  // one energy slot per cluster

// Clusters are static (chromosome ids and the chain order do not change): built once per scratch.
int mmm_chb_clusters_build(mmm_system* h) {
  const int n = (int)h->n;
  std::vector<int> start, chrom, of_bead((size_t)n);
  for (int i = 0; i < n; ++i) {
    const int c = h->h_chrom.empty() ? 0 : h->h_chrom[(size_t)i];
    if (i % MMM_TILE == 0 || c != chrom.back()) { start.push_back(i); chrom.push_back(c); }
    of_bead[(size_t)i] = (int)start.size() - 1;
  }
  const int ncl = (int)start.size();
  start.push_back(n);
  h->n_clusters = ncl;
  int rc;
  if ((rc = mmm_upload(h, h->d_cl_start, start, "cluster starts")) ||
      (rc = mmm_upload(h, h->d_cl_of_bead, of_bead, "cluster of every bead")) ||
      (rc = mmm_upload(h, h->d_cl_by_chrom, chrom, "cluster chromosomes")) ||  // chromosome id of every cluster
      (rc = mmm_reserve(h, h->d_cl_cen, 4 * (size_t)ncl, "cluster centroids")) ||
      (rc = mmm_reserve(h, h->d_cl_force, 3 * (size_t)ncl, "cluster forces")))
    return rc;
  return MMM_OK;
}

int mmm_launch_chb_clusters(mmm_system* h, const int* d_skip) {
  const int ncl = h->n_clusters;
  const PairParams& p = h->pp;
  FarArgs A;
  A.cen = h->d_cl_cen;
  A.chrom = h->d_cl_by_chrom;
  A.ncl = ncl;
  A.chb_on = p.chb_form == MMM_CHB_POLYNOMIAL;
  A.ev_on = p.ev_form == MMM_EV_POWERLAW && h->cutoff > 0.0;
  A.kc = p.d_chb[0]; A.de = p.d_chb[1];
  A.eps = p.d_ev[0]; A.rs = p.d_ev[1]; A.sigma = p.d_ev[2]; A.power = p.d_ev[3];
  A.ipower = (A.power == 6.0) ? 6 : (A.power == 3.0 ? 3 : 0);
  A.r_lo = 0.7 * h->cutoff; A.r_hi = 1.3 * h->cutoff;
  A.force = h->d_cl_force;
  A.epair_slots = h->d_epair + 4 * (size_t)h->cl_item0;
  A.skip = d_skip;
  k_cl_centroid<<<(ncl + 7) / 8, 256, 0, h->stream>>>(h->d_x, h->d_cl_start, ncl, h->d_cl_cen, d_skip);
  k_cl_forces<<<(ncl + 7) / 8, 256, 0, h->stream>>>(A);
  h->launches += 2;
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}
