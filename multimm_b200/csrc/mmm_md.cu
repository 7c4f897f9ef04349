// mmm_md.cu — MD relaxation after minimisation (SURVEY §8(f) N1): replaces the OpenMM integrators
// the reference constructs at model.py:768-808 and steps at model.py:907-995, on top of the same
// fused force pass the minimiser uses.  One launch per step beside the force evaluation; no host
// round trip per step (the host enqueues n steps and reads energies once).
//
// Integrators [OpenMM, restated from its documented algorithms; masses amu, nm, ps, kJ/mol]:
//   MMM_MD_LANGEVIN  (LangevinIntegrator)  v <- a v + (1 - a)/gamma F/m + sqrt(kT (1 - a^2)/m) N(0,1),
//                                          a = exp(-gamma dt);  x <- x + dt v
//   MMM_MD_VERLET    (VerletIntegrator)    leapfrog: v <- v + dt F/m;  x <- x + dt v
//   MMM_MD_BROWNIAN  (BrownianIntegrator)  x <- x + dt/(gamma m) F + sqrt(2 kT dt/(gamma m)) N(0,1);
//                                          v <- dx/dt
//   MMM_MD_AMD       (amd.AMDIntegrator)   leapfrog on the boosted potential: with V the TOTAL potential
//                                          energy at x(t), F' = F (alpha / (alpha + E - V))^2 where V <= E
//                                          (CustomIntegrator's step(E - energy)), F' = F above it;
//                                          v <- v + dt F'/m;  x <- x + dt v.  V is read on the device
//                                          from the per-term energies of the same evaluation.
// All beads carry the one mass of forcefields/ff.xml:5 (16427.889 amu) unless overridden.
// Random numbers: Philox4x32-10, counter = (bead, step_lo, step_hi, stream), key = seed: the same
// numbers whatever the launch geometry, reproducible, and restated in numpy by the tests.
// HBM-bound: 24 B (g) + 48 B (x) + 48 B (v) per bead per step.
#include <math.h>

#include "mmm_internal.cuh"

namespace {

constexpr double kBoltz = 0.008314462618;  // kJ/mol/K

__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// three standard normals for (bead, step, stream): Box-Muller in FP64 on 32-bit uniforms
__device__ inline void normals3(uint64_t seed, int64_t bead, int64_t step, uint32_t stream, double n[3]) {
  uint32_t u[4];
  philox4x32_10((uint32_t)bead, (uint32_t)step, (uint32_t)((uint64_t)step >> 32), stream, (uint32_t)seed,
                (uint32_t)(seed >> 32), u);
  const double two_pi = 6.283185307179586, s = 1.0 / 4294967296.0;
  const double u0 = ((double)u[0] + 0.5) * s, u1 = ((double)u[1] + 0.5) * s;
  const double u2 = ((double)u[2] + 0.5) * s, u3 = ((double)u[3] + 0.5) * s;
  const double r0 = sqrt(-2.0 * log(u0)), r1 = sqrt(-2.0 * log(u2));
  n[0] = r0 * cos(two_pi * u1);
  n[1] = r0 * sin(two_pi * u1);
  n[2] = r1 * cos(two_pi * u3);
}

struct MdArgs {
  int integrator;
  double dt, kT, gamma, inv_mass;
  uint64_t seed;
  int64_t step;  // global step index of THIS update
  int64_t n;
  double* x;
  double* v;
  const double* g;  // gradient (= -force) at x
  const double* eterms;  // AMD: the MMM_NUM_TERMS per-term energies at x
  double amd_alpha, amd_e;
};

__global__ void __launch_bounds__(256) k_md_step(const MdArgs A) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.n) return;
  double nrm[3] = {0.0, 0.0, 0.0};
  if (A.integrator == MMM_MD_LANGEVIN || A.integrator == MMM_MD_BROWNIAN) normals3(A.seed, i, A.step, 1u, nrm);
  double boost = 1.0;
  if (A.integrator == MMM_MD_AMD) {
    double pot = 0.0;
    for (int t = 0; t < MMM_NUM_TERMS; ++t) pot += A.eterms[t];  // same order as the host's total
    if (A.amd_e - pot >= 0.0) {
      const double q = A.amd_alpha / (A.amd_alpha + A.amd_e - pot);
      boost = q * q;
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double f = -A.g[3 * i + d];
    double x = A.x[3 * i + d], v = A.v[3 * i + d];
    if (A.integrator == MMM_MD_LANGEVIN) {
      const double a = exp(-A.gamma * A.dt);
      const double fscale = A.gamma > 0.0 ? (1.0 - a) / A.gamma : A.dt;
      v = a * v + fscale * A.inv_mass * f + sqrt(A.kT * (1.0 - a * a) * A.inv_mass) * nrm[d];
      x += A.dt * v;
    } else if (A.integrator == MMM_MD_VERLET) {
      v += A.dt * A.inv_mass * f;
      x += A.dt * v;
    } else if (A.integrator == MMM_MD_AMD) {
      v += A.dt * (f * boost) * A.inv_mass;
      x += A.dt * v;
    } else {  // Brownian
      const double dx = A.dt * A.inv_mass / A.gamma * f + sqrt(2.0 * A.kT * A.dt * A.inv_mass / A.gamma) * nrm[d];
      x += dx;
      v = dx / A.dt;
    }
    A.x[3 * i + d] = x;
    A.v[3 * i + d] = v;
  }
}

// Maxwell-Boltzmann velocities (context.setVelocitiesToTemperature, model.py:878)
__global__ void __launch_bounds__(256) k_md_init_velocities(int64_t n, double sigma, uint64_t seed, double* v) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double nrm[3];
  normals3(seed, i, 0, 0u, nrm);
  v[3 * i] = sigma * nrm[0];
  v[3 * i + 1] = sigma * nrm[1];
  v[3 * i + 2] = sigma * nrm[2];
}

// sum of v^2 per block (kinetic energy = 1/2 m sum)
__global__ void __launch_bounds__(256) k_md_v2(int64_t n3, const double* __restrict__ v, double* __restrict__ part) {
  __shared__ double s[256];
  double acc = 0.0;
  for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < n3; e += (int64_t)gridDim.x * 256) acc += v[e] * v[e];
  s[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = s[0];
}

// velocities are zero until something sets them
int ensure_velocities(mmm_system* h) {
  if (h->d_v) return MMM_OK;
  int rc = mmm_reserve(h, h->d_v, 3 * (size_t)h->n, "velocities");
  if (rc) return rc;
  MMM_CUDA(h, cudaMemsetAsync(h->d_v, 0, sizeof(double) * 3 * (size_t)h->n, h->stream));
  return MMM_OK;
}

}  // namespace

extern "C" {

int mmm_md_configure(mmm_handle h, int integrator, double dt_ps, double temperature_k, double friction_per_ps,
                     double mass_amu, uint64_t seed) {
  if (!h) return MMM_ERR_ARG;
  if (integrator < MMM_MD_LANGEVIN || integrator > MMM_MD_AMD)
    return mmm_fail(h, MMM_ERR_ARG, "Unknown SIM_INTEGRATOR_TYPE (supported: langevin, verlet, brownian, amd)");
  if (!(dt_ps > 0.0) || !(mass_amu > 0.0) || temperature_k < 0.0 || friction_per_ps < 0.0)
    return mmm_fail(h, MMM_ERR_ARG, "mmm_md_configure: need dt > 0, mass > 0, temperature >= 0, friction >= 0");
  if (integrator == MMM_MD_BROWNIAN && !(friction_per_ps > 0.0))
    return mmm_fail(h, MMM_ERR_ARG, "mmm_md_configure: the Brownian integrator needs friction > 0");
  h->md_integrator = integrator;
  h->md_dt = dt_ps;
  h->md_temperature = temperature_k;
  h->md_gamma = friction_per_ps;
  h->md_mass = mass_amu;
  h->md_seed = seed;
  h->md_step = 0;
  h->md_configured = true;
  return MMM_OK;
}

int mmm_md_set_amd(mmm_handle h, double alpha_kj_mol, double e_boost_kj_mol) {
  if (!h) return MMM_ERR_ARG;
  // alpha = 0 makes the boost factor 0/0 at V = E; OpenMM leaves that to the user, a handle refuses it
  if (!isfinite(alpha_kj_mol) || !isfinite(e_boost_kj_mol) || !(alpha_kj_mol > 0.0))
    return mmm_fail(h, MMM_ERR_ARG, "mmm_md_set_amd: need alpha > 0 and a finite E");
  h->md_amd_alpha = alpha_kj_mol;
  h->md_amd_e = e_boost_kj_mol;
  return MMM_OK;
}

int mmm_set_velocities_to_temperature(mmm_handle h, double temperature_k, uint64_t seed) {
  if (!h) return MMM_ERR_ARG;
  if (temperature_k < 0.0) return mmm_fail(h, MMM_ERR_ARG, "temperature must be >= 0");
  cudaSetDevice(h->device);
  int rc = ensure_velocities(h);
  if (rc) return rc;
  const double mass = h->md_configured ? h->md_mass : 16427.889;
  const double sigma = sqrt(kBoltz * temperature_k / mass);
  k_md_init_velocities<<<(unsigned)((h->n + 255) / 256), 256, 0, h->stream>>>(h->n, sigma, seed, h->d_v);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_set_velocities(mmm_handle h, const double* v) {
  if (!h || !v) return MMM_ERR_ARG;
  cudaSetDevice(h->device);
  int rc = ensure_velocities(h);
  if (rc) return rc;
  MMM_CUDA(h, cudaMemcpyAsync(h->d_v, v, sizeof(double) * 3 * h->n, cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_get_velocities(mmm_handle h, double* v_out) {
  if (!h || !v_out) return MMM_ERR_ARG;
  cudaSetDevice(h->device);
  int rc = ensure_velocities(h);
  if (rc) return rc;
  MMM_CUDA(h, cudaMemcpyAsync(v_out, h->d_v, sizeof(double) * 3 * h->n, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_md_run(mmm_handle h, int64_t n_steps, mmm_md_report* out) {
  if (!h) return MMM_ERR_ARG;
  if (!h->md_configured) return mmm_fail(h, MMM_ERR_STATE, "mmm_md_run: call mmm_md_configure first");
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  if (n_steps < 0) return mmm_fail(h, MMM_ERR_ARG, "mmm_md_run: n_steps must be >= 0");
  cudaSetDevice(h->device);
  int rc = ensure_velocities(h);
  if (rc) return rc;
  h->have_result = false;  // the integrator reuses d_g / d_eterms
  MdArgs A;
  A.integrator = h->md_integrator;
  A.dt = h->md_dt;
  A.kT = kBoltz * h->md_temperature;
  A.gamma = h->md_gamma;
  A.inv_mass = 1.0 / h->md_mass;
  A.seed = h->md_seed;
  A.n = h->n;
  A.x = h->d_x;
  A.v = h->d_v;
  A.g = h->d_g;
  A.eterms = h->d_eterms;
  A.amd_alpha = h->md_amd_alpha;
  A.amd_e = h->md_amd_e;
  const unsigned blocks = (unsigned)((h->n + 255) / 256);
  for (int64_t s = 0; s < n_steps; ++s) {
    if ((rc = mmm_evaluate(h, nullptr))) return rc;  // forces at x(t)
    if (A.integrator == MMM_MD_AMD && (rc = mmm_launch_finalize_energy(h))) return rc;  // V(x(t)) for the boost
    A.step = h->md_step++;
    k_md_step<<<blocks, 256, 0, h->stream>>>(A);
    h->launches++;
  }
  if (!out) {  // no report wanted: the steps stay enqueued, nothing is evaluated or read back for it
    MMM_CUDA(h, cudaGetLastError());
    return MMM_OK;
  }
  // energies at the final positions (potential) and velocities (kinetic)
  if ((rc = mmm_evaluate(h, nullptr))) return rc;
  if ((rc = mmm_launch_finalize_energy(h))) return rc;
  const int nb = h->n_dot_blocks;
  k_md_v2<<<nb, 256, 0, h->stream>>>(3 * h->n, h->d_v, h->d_dpart);
  h->launches++;
  double e[MMM_NUM_TERMS];
  std::vector<double> part((size_t)nb);
  MMM_CUDA(h, cudaMemcpyAsync(e, h->d_eterms, sizeof(e), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(part.data(), h->d_dpart, sizeof(double) * nb, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  MMM_CUDA(h, cudaGetLastError());
  double pot = 0.0, v2 = 0.0;
  for (int t = 0; t < MMM_NUM_TERMS; ++t) pot += e[t];
  for (double p : part) v2 += p;
  if (out) {
    out->step = h->md_step;
    out->potential = pot;
    out->kinetic = 0.5 * h->md_mass * v2;
    out->temperature = 2.0 * out->kinetic / (3.0 * (double)h->n * kBoltz);
  }
  if (!isfinite(pot) || !isfinite(v2)) return mmm_fail(h, MMM_ERR_NUMERIC, "non-finite energy during MD (time step too large?)");
  return MMM_OK;
}

}  // extern "C"
