// mmm_bonded.cu — the fused O(N) pass: backbone bonds, loop bonds, angles, the three external
// terms, and assembly of the gradient from the pair kernel's per-chunk partial forces.
//
// Replaces HarmonicBondForce / CustomBondForce / HarmonicAngleForce / CustomExternalForce as
// built by model.py:453-720.  Gather formulation: one thread per bead walks the bead's own
// CSR lists (<= 2 backbone bonds, its loops, <= 3 angles), so accumulation order is fixed and
// no atomics are needed; each bond is evaluated from both ends and each angle from its three
// beads (O(N) redundant work, irrelevant next to the pair kernel).  All arithmetic here is
// FP64 on the FP64 master positions.  HBM-bound: ~24 B (x) + 24 B (g) + 24 B x nchunk (pair
// partials) + ~40 B per bond end + ~48 B per angle corner per bead.
#include <math.h>

#include <algorithm>

#include "mmm_internal.cuh"

namespace {

constexpr int kAsmBlock = MMM_ASM_BLOCK;

struct AsmArgs {
  const double* x;
  const double* fpair;       // gather kernel: [nchunk][3][npad] partial forces
  unsigned long long* facc;  // Newton-3 kernel: [3][npad] fixed-point force (2^-24), zeroed here after use
  int nchunk;
  int64_t n, npad;
  const int* bl_ptr; const int* bl_partner; const int* bl_flags; const double* bl_r0; const double* bl_k;
  const int* an_ptr; const int4* an_ijk; const double2* an_par;
  const signed char* s; const double* cstr;
  const double* cl_force; const int* cl_of_bead;  // CHB cluster surrogate: force of the bead's cluster (or NULL)
  ExternalParams ep;
  double* g;
  double* epart;  // [blocks][6]: SC, LAM, CF, BOND, LOOP, ANGLE
  const int* skip;
};

// E and dE/dr of a bond-like term; kind 0 = backbone harmonic, 1 + MMM_LOOP_* for loops
__device__ __forceinline__ double bond_like(int kind, double r, double r0, double k, double& dedr) {
  const double d = r - r0;
  if (kind <= 1) {  // [OpenMM] HarmonicBondForce: 1/2 k (r - r0)^2   (model.py:630-635, 653-659)
    dedr = k * d;
    return 0.5 * k * d * d;
  } else if (kind == 2) {  // fene_soft, model.py:664-680
    const double al = 1.0 / (r0 * r0), q = 1.0 + al * d * d;
    dedr = 2.0 * k * d / (q * q);
    return k * d * d / q;
  } else {  // gaussian_tether, model.py:685-701
    const double sg = 0.5 * r0, gg = exp(-d * d / (sg * sg));
    dedr = k * gg * 2.0 * d / (sg * sg);
    return k * (1.0 - gg);
  }
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(kAsmBlock) k_assemble(const AsmArgs A) {
  __shared__ double s_red[6][kAsmBlock / 32];
  if (A.skip && *A.skip) return;
  const int64_t i = (int64_t)blockIdx.x * kAsmBlock + threadIdx.x;
  double e_sc = 0, e_lam = 0, e_cf = 0, e_bond = 0, e_loop = 0, e_ang = 0;
  if (i < A.n) {
    double fx = 0, fy = 0, fz = 0;
    if (A.facc) {
      const double inv = 1.0 / 16777216.0;
      fx = (double)(long long)A.facc[i] * inv;
      fy = (double)(long long)A.facc[(size_t)A.npad + i] * inv;
      fz = (double)(long long)A.facc[2 * (size_t)A.npad + i] * inv;
      A.facc[i] = 0ull;
      A.facc[(size_t)A.npad + i] = 0ull;
      A.facc[2 * (size_t)A.npad + i] = 0ull;
    }
    if (A.fpair) {
      for (int c = 0; c < A.nchunk; ++c) {
        const double* fp = A.fpair + (size_t)c * 3 * (size_t)A.npad;
        fx += fp[i];
        fy += fp[(size_t)A.npad + i];
        fz += fp[2 * (size_t)A.npad + i];
      }
    }
    if (A.cl_force) {
      const size_t c = (size_t)A.cl_of_bead[i];
      fx += A.cl_force[3 * c]; fy += A.cl_force[3 * c + 1]; fz += A.cl_force[3 * c + 2];
    }
    const double xi = A.x[3 * i], yi = A.x[3 * i + 1], zi = A.x[3 * i + 2];

    // bonds and loops
    if (A.bl_ptr) {
      for (int q = A.bl_ptr[i]; q < A.bl_ptr[i + 1]; ++q) {
        const int64_t p = A.bl_partner[q];
        const int fl = A.bl_flags[q];
        const double dx = xi - A.x[3 * p], dy = yi - A.x[3 * p + 1], dz = zi - A.x[3 * p + 2];
        const double r = sqrt(dx * dx + dy * dy + dz * dz);
        double dedr;
        const double e = bond_like(fl >> 1, r, A.bl_r0[q], A.bl_k[q], dedr);
        if (r > 0.0) {
          const double sc = -dedr / r;
          fx += sc * dx; fy += sc * dy; fz += sc * dz;
        }
        if (fl & 1) {
          if ((fl >> 1) == 0) e_bond += e; else e_loop += e;
        }
      }
    }
    // angles: [OpenMM] HarmonicAngleForce, theta = acos(clamped cosine), |u x v| floored at 1e-6
    if (A.an_ptr) {
      for (int q = A.an_ptr[i]; q < A.an_ptr[i + 1]; ++q) {
        const int4 t = A.an_ijk[q];
        const double2 par = A.an_par[q];
        const double ux = A.x[3 * (int64_t)t.x] - A.x[3 * (int64_t)t.y];
        const double uy = A.x[3 * (int64_t)t.x + 1] - A.x[3 * (int64_t)t.y + 1];
        const double uz = A.x[3 * (int64_t)t.x + 2] - A.x[3 * (int64_t)t.y + 2];
        const double vx = A.x[3 * (int64_t)t.z] - A.x[3 * (int64_t)t.y];
        const double vy = A.x[3 * (int64_t)t.z + 1] - A.x[3 * (int64_t)t.y + 1];
        const double vz = A.x[3 * (int64_t)t.z + 2] - A.x[3 * (int64_t)t.y + 2];
        const double uu = ux * ux + uy * uy + uz * uz, vv = vx * vx + vy * vy + vz * vz;
        const double uv = ux * vx + uy * vy + uz * vz;
        const double px = uy * vz - uz * vy, py = uz * vx - ux * vz, pz = ux * vy - uy * vx;
        double rp = sqrt(px * px + py * py + pz * pz);
        if (rp < 1e-6) rp = 1e-6;
        const double cs = uv / sqrt(uu * vv);
        double th;
        if (cs >= 1.0) th = 0.0;
        else if (cs <= -1.0) th = M_PI;
        else th = acos(cs);
        const double dth = th - par.x;
        const double dedth = par.y * dth;
        const double ta = -dedth / (uu * rp), tc = dedth / (vv * rp);
        const double fax = ta * (uy * pz - uz * py), fay = ta * (uz * px - ux * pz), faz = ta * (ux * py - uy * px);
        const double fcx = tc * (vy * pz - vz * py), fcy = tc * (vz * px - vx * pz), fcz = tc * (vx * py - vy * px);
        if (t.w == 0) {
          fx += fax; fy += fay; fz += faz;
          e_ang += 0.5 * par.y * dth * dth;
        } else if (t.w == 2) {
          fx += fcx; fy += fcy; fz += fcz;
        } else {
          fx -= fax + fcx; fy -= fay + fcy; fz -= faz + fcz;
        }
      }
    }
    // external terms (CustomExternalForce): functions of rho = |x - centre|
    const int si = A.s ? (int)A.s[i] : 0;
    const ExternalParams& E = A.ep;
    if (E.sc_form >= 0) {  // model.py:454-456
      const double dx = xi - E.sc[3], dy = yi - E.sc[4], dz = zi - E.sc[5];
      const double rho = sqrt(dx * dx + dy * dy + dz * dz);
      const double a = fmax(0.0, rho - E.sc[2]), b = fmax(0.0, E.sc[1] - rho);
      e_sc = E.sc[0] * (a * a + b * b);
      const double d = 2.0 * E.sc[0] * (a - b);
      if (rho > 0.0) { fx -= d * dx / rho; fy -= d * dy / rho; fz -= d * dz / rho; }
    }
    if (E.lam_form >= 0 && (si == -1 || si == -2)) {
      const double dx = xi - E.lam[3], dy = yi - E.lam[4], dz = zi - E.lam[5];
      const double rho = sqrt(dx * dx + dy * dy + dz * dz);
      const double B = E.lam[0], R1 = E.lam[1], R2 = E.lam[2];
      double d = 0.0;
      if (E.lam_form == MMM_LAM_SIN) {  // model.py:503-505
        const double w = M_PI / (R2 - R1), a = w * (rho - R1);
        double sn, cn;
        sincos(a, &sn, &cn);
        const double s2 = sn * sn, s4 = s2 * s2;
        e_lam = B * (s4 * s4 - 1.0);
        d = B * 8.0 * s4 * s2 * sn * cn * w;
      } else if (E.lam_form == MMM_LAM_GAUSSIAN_SHELL) {  // model.py:513-517
        const double sg = 0.1 * (R2 - R1), qq = 2.0 * sg * sg;
        const double g1 = exp(-(rho - R1) * (rho - R1) / qq), g2 = exp(-(rho - R2) * (rho - R2) / qq);
        e_lam = -B * (g1 + g2);
        d = B * (g1 * 2.0 * (rho - R1) / qq + g2 * 2.0 * (rho - R2) / qq);
      } else if (E.lam_form == MMM_LAM_HARMONIC_SHELL) {  // model.py:524-527
        const double r0 = 0.5 * (R1 + R2);
        e_lam = B * (rho - r0) * (rho - r0);
        d = 2.0 * B * (rho - r0);
      } else {  // model.py:534-538
        const double lm = 0.05 * (R2 - R1);
        const double ea = exp((rho - R2) / lm), eb = exp(-(rho - R1) / lm);
        const double fa = 1.0 / (1.0 + ea), fb = 1.0 / (1.0 + eb);
        e_lam = -B * (fa + fb);
        d = -B * (-ea * fa * fa / lm + eb * fb * fb / lm);
      }
      if (rho > 0.0) { fx -= d * dx / rho; fy -= d * dy / rho; fz -= d * dz / rho; }
    }
    if (E.cf_form >= 0) {
      const double cw = A.cstr ? A.cstr[i] : 0.0;
      const double dx = xi - E.cf[2], dy = yi - E.cf[3], dz = zi - E.cf[4];
      const double rho = sqrt(dx * dx + dy * dy + dz * dz);
      const double G = E.cf[0], R1 = E.cf[1];
      double d;
      if (E.cf_form == MMM_CF_HARMONIC) {  // model.py:584-586
        e_cf = G * cw * (rho - R1) * (rho - R1);
        d = 2.0 * G * cw * (rho - R1);
      } else if (E.cf_form == MMM_CF_GAUSSIAN) {  // model.py:594-599
        const double sg = 0.5 * R1, ee = exp(-rho * rho / (2.0 * sg * sg));
        e_cf = -G * cw * ee;
        d = G * cw * ee * rho / (sg * sg);
      } else {  // model.py:607-612
        const double lm = 0.2 * R1, ea = exp((rho - R1) / lm), qq = 1.0 / (1.0 + ea);
        e_cf = -G * cw * qq;
        d = G * cw * ea * qq * qq / lm;
      }
      if (rho > 0.0) { fx -= d * dx / rho; fy -= d * dy / rho; fz -= d * dz / rho; }
    }
    A.g[3 * i] = -fx;
    A.g[3 * i + 1] = -fy;
    A.g[3 * i + 2] = -fz;
  }
  // deterministic block reduction of the six O(N) energies
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  e_sc = warp_sum_d(e_sc); e_lam = warp_sum_d(e_lam); e_cf = warp_sum_d(e_cf);
  e_bond = warp_sum_d(e_bond); e_loop = warp_sum_d(e_loop); e_ang = warp_sum_d(e_ang);
  if (lane == 0) {
    s_red[0][warp] = e_sc; s_red[1][warp] = e_lam; s_red[2][warp] = e_cf;
    s_red[3][warp] = e_bond; s_red[4][warp] = e_loop; s_red[5][warp] = e_ang;
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double s = 0;
#pragma unroll
    for (int w = 0; w < kAsmBlock / 32; ++w) s += s_red[threadIdx.x][w];
    A.epart[(size_t)blockIdx.x * 6 + threadIdx.x] = s;
  }
}

// Fixed-order final sums: pair energies over work items, O(N) energies over blocks.
__global__ void __launch_bounds__(256) k_finalize_energy(const double* __restrict__ epair, int n_items,
                                                         const double* __restrict__ epart, int n_blocks,
                                                         double* __restrict__ eterms) {
  __shared__ double s[256];
  for (int t = 0; t < MMM_NUM_TERMS; ++t) {
    double acc = 0;
    if (t < 4) {
      for (int q = threadIdx.x; q < n_items; q += 256) acc += epair[(size_t)q * 4 + t];
    } else {
      for (int q = threadIdx.x; q < n_blocks; q += 256) acc += epart[(size_t)q * 6 + (t - 4)];
    }
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) eterms[t] = s[0];
    __syncthreads();
  }
}

template <typename T>
int upload(mmm_system* h, T** dptr, const std::vector<T>& v) {
  if (*dptr) { cudaFree(*dptr); *dptr = nullptr; }
  if (v.empty()) return MMM_OK;
  MMM_CUDA(h, cudaMalloc((void**)dptr, v.size() * sizeof(T)));
  MMM_CUDA(h, cudaMemcpyAsync(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

}  // namespace

// Build the per-bead gather lists from the bond / loop arrays held on the host side of the handle.
int mmm_upload_topology(mmm_system* h) {
  const int64_t n = h->n;
  const int64_t nb = (int64_t)h->h_bond_i.size(), nl = (int64_t)h->h_loop_i.size();
  std::vector<int> ptr(n + 1, 0);
  for (int64_t b = 0; b < nb; ++b) { ptr[h->h_bond_i[b] + 1]++; ptr[h->h_bond_j[b] + 1]++; }
  for (int64_t b = 0; b < nl; ++b) { ptr[h->h_loop_i[b] + 1]++; ptr[h->h_loop_j[b] + 1]++; }
  for (int64_t i = 0; i < n; ++i) ptr[i + 1] += ptr[i];
  const size_t ne = (size_t)ptr[n];
  std::vector<int> partner(ne), flags(ne), fill(ptr.begin(), ptr.end() - 1);
  std::vector<double> r0(ne), kk(ne);
  auto put = [&](int a, int b, int fl, double r, double k) {
    const int q = fill[a]++;
    partner[q] = b; flags[q] = fl; r0[q] = r; kk[q] = k;
  };
  for (int64_t b = 0; b < nb; ++b) {
    put(h->h_bond_i[b], h->h_bond_j[b], 1, h->h_bond_r0[b], h->h_bond_k[b]);
    put(h->h_bond_j[b], h->h_bond_i[b], 0, h->h_bond_r0[b], h->h_bond_k[b]);
  }
  const int lk = (1 + h->loop_form) << 1;
  for (int64_t b = 0; b < nl; ++b) {
    put(h->h_loop_i[b], h->h_loop_j[b], lk | 1, h->h_loop_r0[b], h->h_loop_k[b]);
    put(h->h_loop_j[b], h->h_loop_i[b], lk, h->h_loop_r0[b], h->h_loop_k[b]);
  }
  int rc;
  if (ne == 0) {
    if (h->d_bl_ptr) { cudaFree(h->d_bl_ptr); h->d_bl_ptr = nullptr; }
  } else {
    if ((rc = upload(h, &h->d_bl_ptr, ptr))) return rc;
  }
  if ((rc = upload(h, &h->d_bl_partner, partner))) return rc;
  if ((rc = upload(h, &h->d_bl_flags, flags))) return rc;
  if ((rc = upload(h, &h->d_bl_r0, r0))) return rc;
  if ((rc = upload(h, &h->d_bl_k, kk))) return rc;
  h->topo_dirty = false;
  return MMM_OK;
}

int mmm_upload_angles(mmm_system* h, const int32_t* ai, const int32_t* aj, const int32_t* ak,
                      const double* t0, const double* kt, int64_t na) {
  const int64_t n = h->n;
  std::vector<int> ptr(n + 1, 0);
  for (int64_t a = 0; a < na; ++a) { ptr[ai[a] + 1]++; ptr[aj[a] + 1]++; ptr[ak[a] + 1]++; }
  for (int64_t i = 0; i < n; ++i) ptr[i + 1] += ptr[i];
  std::vector<int> fill(ptr.begin(), ptr.end() - 1);
  std::vector<int4> ijk((size_t)ptr[n]);
  std::vector<double2> par((size_t)ptr[n]);
  for (int64_t a = 0; a < na; ++a) {
    const int who[3] = {ai[a], aj[a], ak[a]};
    for (int role = 0; role < 3; ++role) {
      const int q = fill[who[role]]++;
      ijk[q] = make_int4(ai[a], aj[a], ak[a], role);
      par[q] = make_double2(t0[a], kt[a]);
    }
  }
  int rc;
  if (na == 0) {
    if (h->d_an_ptr) { cudaFree(h->d_an_ptr); h->d_an_ptr = nullptr; }
  } else {
    if ((rc = upload(h, &h->d_an_ptr, ptr))) return rc;
  }
  if ((rc = upload(h, &h->d_an_ijk, ijk))) return rc;
  if ((rc = upload(h, &h->d_an_par, par))) return rc;
  h->n_angles = na;
  return MMM_OK;
}

int mmm_launch_assemble(mmm_system* h, const int* d_skip) {
  AsmArgs A;
  A.x = h->d_x;
  A.fpair = (h->pair_mode == 1 || (h->pair_mode == 3 && !h->cut_n3)) ? h->d_fpair : nullptr;
  A.facc = (h->pair_mode == 2 || (h->pair_mode == 3 && (h->cut_n3 || (h->n3_items > 0 && h->n3_chb_only)))) ? h->d_facc : nullptr;
  A.nchunk = h->n_planes;
  A.n = h->n;
  A.npad = h->npad;
  A.bl_ptr = h->d_bl_ptr; A.bl_partner = h->d_bl_partner; A.bl_flags = h->d_bl_flags;
  A.bl_r0 = h->d_bl_r0; A.bl_k = h->d_bl_k;
  A.an_ptr = h->d_an_ptr; A.an_ijk = h->d_an_ijk; A.an_par = h->d_an_par;
  A.s = h->d_s; A.cstr = h->d_cstr;
  A.cl_force = (h->pair_mode == 3 && h->chb_clusters) ? h->d_cl_force : nullptr;
  A.cl_of_bead = h->d_cl_of_bead;
  A.ep = h->ep;
  A.g = h->d_g;
  A.epart = h->d_epart;
  A.skip = d_skip;
  k_assemble<<<h->n_red_blocks, kAsmBlock, 0, h->stream>>>(A);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}

int mmm_launch_finalize_energy(mmm_system* h) {
  k_finalize_energy<<<1, 256, 0, h->stream>>>(h->d_epair, (int)h->n_items, h->d_epart, h->n_red_blocks,
                                             h->d_eterms);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  h->have_result = true;
  return MMM_OK;
}
