// mmm_api.cu — the extern "C" surface declared in include/multimm_b200.h, plus handle
// bookkeeping.  Host code only; every kernel lives in the sibling .cu files.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <new>

#include "mmm_internal.cuh"

int mmm_launch_dots_decide(mmm_system* h);  // mmm_lbfgs.cu

static thread_local std::string g_create_error;
static void free_scratch(mmm_system* h);

int mmm_fail(mmm_system* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  else g_create_error = msg;
  return code;
}

#define REQUIRE(h, cond, msg) \
  do { if (!(cond)) return mmm_fail((h), MMM_ERR_ARG, (msg)); } while (0)

static void derive_pair_params(mmm_system* h) {
  PairParams& p = h->pp;
  p.ev_pref = p.ev_form == MMM_EV_POWERLAW ? p.ev_eps * powf(p.ev_sigma, p.ev_power) : 0.0f;
  const float rc = p.scb_form >= 0 ? p.scb_rc : p.cob_rc;
  if (rc > 0.0f) {
    p.g_c = -1.4426950408889634f / (2.0f * rc * rc);
    p.g_inv_rc2 = 1.0f / (rc * rc);
    // exp(-rg^2 / 2rc^2) = 2^-26: beyond rg a Gaussian term is < 1.5e-8 of its prefactor; the part of
    // the term's total energy that lies beyond rg is < 1e-7 at chromatin density (DESIGN.md 4.1)
    p.rg2 = 2.0f * rc * rc * 26.0f * 0.6931471805599453f;
  } else {
    p.g_c = 0.0f; p.g_inv_rc2 = 0.0f; p.rg2 = 0.0f;
  }
  p.cutoff2 = (float)h->cutoff * (float)h->cutoff;
}

extern "C" {

int mmm_abi_version(void) { return MMM_ABI_VERSION; }

const char* mmm_last_error(mmm_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int mmm_create(int device, int64_t n_beads, mmm_handle* out) {
  if (!out) return mmm_fail(nullptr, MMM_ERR_ARG, "mmm_create: out is NULL");
  *out = nullptr;
  // 2^24 = the number of points of the order-8 Hilbert curve the reference starts from
  // (initial_structure_tools.py:157-166); it also keeps the work-item tables within 32-bit counts
  if (n_beads < 2 || n_beads > (int64_t)1 << 24)
    return mmm_fail(nullptr, MMM_ERR_ARG, "mmm_create: n_beads must be in [2, 2^24]");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return mmm_fail(nullptr, MMM_ERR_CUDA,
                    std::string("CUDA error: no usable device (") + cudaGetErrorString(e) +
                        "); this engine has no CPU fallback");
  if (device < 0 || device >= ndev) return mmm_fail(nullptr, MMM_ERR_ARG, "mmm_create: device index out of range");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return mmm_fail(nullptr, MMM_ERR_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e));
  if (prop.major != 10)
    return mmm_fail(nullptr, MMM_ERR_CUDA,
                    "CUDA error: device is not sm_100 (B200); the kernels are built for sm_100a only");
  mmm_system* h = new (std::nothrow) mmm_system();
  if (!h) return mmm_fail(nullptr, MMM_ERR_NOMEM, "out of host memory");
  h->device = device;
  h->n = n_beads;
  h->npad = (n_beads + MMM_PAD_TO - 1) / MMM_PAD_TO * MMM_PAD_TO;
  h->ntiles = h->npad / MMM_TILE;
  h->sm_count = prop.multiProcessorCount;
  h->pp.ev_form = h->pp.cob_form = h->pp.scb_form = h->pp.chb_form = MMM_FORM_OFF;
  h->ep.sc_form = h->ep.lam_form = h->ep.cf_form = MMM_FORM_OFF;
  h->n_red_blocks = (int)((n_beads + MMM_ASM_BLOCK - 1) / MMM_ASM_BLOCK);
  h->n_dot_blocks = std::min(h->n_red_blocks, 2 * h->sm_count);
  int rc = MMM_OK;
  auto fail = [&](int code) { g_create_error = h->err; mmm_destroy(h); return code; };
  if (cudaSetDevice(device) != cudaSuccess) return fail(mmm_fail(h, MMM_ERR_CUDA, "CUDA error: cudaSetDevice"));
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
    return fail(mmm_fail(h, MMM_ERR_CUDA, "CUDA error: cudaStreamCreate"));
  cudaEventCreate(&h->ev_a);
  cudaEventCreate(&h->ev_b);
  const size_t n3 = 3 * (size_t)n_beads;
  if ((rc = mmm_reserve(h, h->d_type, (size_t)h->npad, "bead types")) ||
      (rc = mmm_reserve(h, h->d_cstr, (size_t)n_beads, "chromosome strengths")) ||
      (rc = mmm_reserve(h, h->d_s, (size_t)n_beads, "compartment labels")) ||
      (rc = mmm_reserve(h, h->d_x, n3, "positions")) ||
      (rc = mmm_reserve(h, h->d_center, 3, "centre")) ||
      (rc = mmm_reserve(h, h->d_pos4, (size_t)h->npad, "FP32 positions")) ||
      (rc = mmm_reserve(h, h->d_soa, 3 * (size_t)h->npad, "FP32 coordinate planes")) ||
      (rc = mmm_reserve(h, h->d_tiles, (size_t)h->ntiles, "tile boxes")) ||
      (rc = mmm_reserve(h, h->d_g, n3, "gradient")) ||
      (rc = mmm_reserve(h, h->d_counter, 4, "work counters")) ||
      (rc = mmm_reserve(h, h->d_epart, (size_t)h->n_red_blocks * 6, "energy partials")) ||
      (rc = mmm_reserve(h, h->d_dpart, (size_t)h->n_red_blocks * MMM_NDOT, "dot partials")) ||
      (rc = mmm_reserve(h, h->d_eterms, MMM_NUM_TERMS, "energy terms")) ||
      (rc = mmm_reserve(h, h->d_lb, 1, "L-BFGS state")))
    return fail(rc);
  if (cudaMallocHost((void**)&h->h_done, 64) != cudaSuccess)
    return fail(mmm_fail(h, MMM_ERR_NOMEM, "CUDA error: cudaMallocHost"));
  cudaMemsetAsync(h->d_cstr, 0, sizeof(double) * n_beads, h->stream);
  cudaMemsetAsync(h->d_s, 0, n_beads, h->stream);
  cudaMemsetAsync(h->d_lb, 0, sizeof(LbfgsState), h->stream);
  std::vector<int> ty((size_t)h->npad);
  for (int64_t i = 0; i < h->npad; ++i)
    ty[i] = i < n_beads ? mmm_pack_type(0, 0) : mmm_pack_type(0, MMM_PAD_CHROM + (int)(i - n_beads));
  cudaMemcpyAsync(h->d_type, ty.data(), sizeof(int) * ty.size(), cudaMemcpyHostToDevice, h->stream);
  if (cudaStreamSynchronize(h->stream) != cudaSuccess)
    return fail(mmm_fail(h, MMM_ERR_CUDA, "CUDA error: initialisation copies failed"));
  h->types_dirty = false;
  *out = h;
  return MMM_OK;
}

int mmm_destroy(mmm_handle h) {
  if (!h) return MMM_OK;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  mmm_dist_destroy(h);
  if (h->h_done) cudaFreeHost(h->h_done);
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  for (cudaEvent_t e : {h->ev_a, h->ev_b, h->ev_c0, h->ev_c1, h->ct_ev0, h->ct_ev1, h->dm_ev0, h->dm_ev1,
                        h->sp_ev0, h->sp_ev1, h->lp_ev0, h->lp_ev1, h->tp_ev0, h->tp_ev1})
    if (e) cudaEventDestroy(e);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;  // the device buffers free themselves
  return MMM_OK;
}

// ---- topology --------------------------------------------------------------------------
static int check_pairs(mmm_system* h, const int32_t* i, const int32_t* j, int64_t cnt, const char* what) {
  for (int64_t q = 0; q < cnt; ++q)
    if (i[q] < 0 || j[q] < 0 || i[q] >= h->n || j[q] >= h->n || i[q] == j[q])
      return mmm_fail(h, MMM_ERR_ARG, std::string(what) + ": bead index out of range or degenerate");
  return MMM_OK;
}

int mmm_set_bonds(mmm_handle h, const int32_t* i, const int32_t* j, const double* r0, const double* k,
                  int64_t n_bonds) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, n_bonds >= 0 && (n_bonds == 0 || (i && j && r0 && k)), "mmm_set_bonds: NULL array");
  int rc = check_pairs(h, i, j, n_bonds, "mmm_set_bonds");
  if (rc) return rc;
  h->h_bond_i.assign(i, i + n_bonds); h->h_bond_j.assign(j, j + n_bonds);
  h->h_bond_r0.assign(r0, r0 + n_bonds); h->h_bond_k.assign(k, k + n_bonds);
  h->n_bonds = n_bonds;
  h->topo_dirty = true;
  return MMM_OK;
}

int mmm_set_loops(mmm_handle h, const int32_t* i, const int32_t* j, const double* r0, const double* k,
                  int64_t n_loops, int form) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, form >= MMM_LOOP_HARMONIC && form <= MMM_LOOP_GAUSSIAN_TETHER, "Unknown loop force type");
  REQUIRE(h, n_loops >= 0 && (n_loops == 0 || (i && j && r0 && k)), "mmm_set_loops: NULL array");
  int rc = check_pairs(h, i, j, n_loops, "mmm_set_loops");
  if (rc) return rc;
  h->h_loop_i.assign(i, i + n_loops); h->h_loop_j.assign(j, j + n_loops);
  h->h_loop_r0.assign(r0, r0 + n_loops); h->h_loop_k.assign(k, k + n_loops);
  h->n_loops = n_loops;
  h->loop_form = form;
  h->topo_dirty = true;
  return MMM_OK;
}

int mmm_set_angles(mmm_handle h, const int32_t* i, const int32_t* j, const int32_t* k, const double* theta0,
                   const double* k_theta, int64_t n_angles) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, n_angles >= 0 && (n_angles == 0 || (i && j && k && theta0 && k_theta)), "mmm_set_angles: NULL array");
  for (int64_t q = 0; q < n_angles; ++q)
    if (i[q] < 0 || j[q] < 0 || k[q] < 0 || i[q] >= h->n || j[q] >= h->n || k[q] >= h->n)
      return mmm_fail(h, MMM_ERR_ARG, "mmm_set_angles: bead index out of range");
  cudaSetDevice(h->device);
  return mmm_upload_angles(h, i, j, k, theta0, k_theta, n_angles);
}

int mmm_set_bead_params(mmm_handle h, const int8_t* s, const int32_t* chrom, const double* chrom_strength) {
  if (!h) return MMM_ERR_ARG;
  cudaSetDevice(h->device);
  std::vector<int> ty((size_t)h->npad);
  for (int64_t i = h->n; i < h->npad; ++i) ty[i] = mmm_pack_type(0, MMM_PAD_CHROM + (int)(i - h->n));
  std::vector<signed char> sv((size_t)h->n, 0);
  for (int64_t i = 0; i < h->n; ++i) {
    const int si = s ? (int)s[i] : 0;
    const int ci = chrom ? chrom[i] : 0;
    if (si < -2 || si > 2) return mmm_fail(h, MMM_ERR_ARG, "mmm_set_bead_params: compartment label outside [-2, 2]");
    if (ci < 0 || ci >= MMM_PAD_CHROM) return mmm_fail(h, MMM_ERR_ARG, "mmm_set_bead_params: chromosome id outside [0, 64511]");
    ty[i] = mmm_pack_type(si, ci);
    sv[i] = (signed char)si;
  }
  if (chrom) h->h_chrom.assign(chrom, chrom + h->n);
  else h->h_chrom.clear();
  if (h->scratch_sig >= 0) free_scratch(h);  // the CHB-only item list depends on the chromosome ids
  MMM_CUDA(h, cudaMemcpyAsync(h->d_type, ty.data(), sizeof(int) * ty.size(), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaMemcpyAsync(h->d_s, sv.data(), sv.size(), cudaMemcpyHostToDevice, h->stream));
  if (chrom_strength)
    MMM_CUDA(h, cudaMemcpyAsync(h->d_cstr, chrom_strength, sizeof(double) * h->n, cudaMemcpyHostToDevice, h->stream));
  else
    MMM_CUDA(h, cudaMemsetAsync(h->d_cstr, 0, sizeof(double) * h->n, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_set_pair_term(mmm_handle h, int term, int form, const double* g, int ng) {
  if (!h) return MMM_ERR_ARG;
  PairParams& p = h->pp;
  REQUIRE(h, form == MMM_FORM_OFF || g, "mmm_set_pair_term: globals is NULL");
  switch (term) {
    case MMM_TERM_EV:
      REQUIRE(h, form >= -1 && form <= MMM_EV_GAUSSIAN_CORE, "Unknown EV_FORCE_TYPE");
      p.ev_form = form;
      if (form >= 0) {
        REQUIRE(h, ng >= 4, "EV needs {epsilon, r_small, sigma, power}");
        p.ev_eps = (float)g[0]; p.ev_rs = (float)g[1]; p.ev_sigma = (float)g[2]; p.ev_power = (float)g[3];
        memcpy(p.d_ev, g, 4 * sizeof(double));
      }
      break;
    case MMM_TERM_COB:
      REQUIRE(h, form >= -1 && form <= MMM_BLOCK_THETA, "Unknown COB_FORCE_TYPE");
      p.cob_form = form;
      if (form >= 0) {
        REQUIRE(h, ng >= 3, "COB needs {rc, Ea, Eb}");
        p.cob_rc = (float)g[0]; p.cob_ea = (float)g[1]; p.cob_eb = (float)g[2];
        memcpy(p.d_cob, g, 3 * sizeof(double));
      }
      break;
    case MMM_TERM_SCB:
      REQUIRE(h, form >= -1 && form <= MMM_BLOCK_THETA, "Unknown SCB_FORCE_TYPE");
      p.scb_form = form;
      if (form >= 0) {
        REQUIRE(h, ng >= 5, "SCB needs {rsc, Ea1, Ea2, Eb1, Eb2}");
        p.scb_rc = (float)g[0];
        for (int q = 0; q < 4; ++q) p.scb_e[q] = (float)g[1 + q];
        memcpy(p.d_scb, g, 5 * sizeof(double));
      }
      break;
    case MMM_TERM_CHB:
      REQUIRE(h, form >= -1 && form <= MMM_CHB_SATURATING, "Unknown CHB_FORCE_TYPE");
      p.chb_form = form;
      if (form >= 0) {
        REQUIRE(h, ng >= 2, "CHB needs {k_C, dE}");
        p.chb_kc = (float)g[0]; p.chb_de = (float)g[1];
        memcpy(p.d_chb, g, 2 * sizeof(double));
      }
      break;
    default:
      return mmm_fail(h, MMM_ERR_ARG, "mmm_set_pair_term: term is not a pair term");
  }
  derive_pair_params(h);
  return MMM_OK;
}

int mmm_set_external_term(mmm_handle h, int term, int form, const double* g, int ng) {
  if (!h) return MMM_ERR_ARG;
  ExternalParams& p = h->ep;
  REQUIRE(h, form == MMM_FORM_OFF || g, "mmm_set_external_term: globals is NULL");
  switch (term) {
    case MMM_TERM_SC:
      REQUIRE(h, form >= -1 && form <= MMM_SC_DOUBLE_WALL, "Unknown spherical container form");
      p.sc_form = form;
      if (form >= 0) { REQUIRE(h, ng >= 6, "SC needs {C, R1, R2, x0, y0, z0}"); memcpy(p.sc, g, 6 * sizeof(double)); }
      break;
    case MMM_TERM_LAM:
      REQUIRE(h, form >= -1 && form <= MMM_LAM_LOGISTIC_SHELL, "Unknown BLAMINA_FORCE_TYPE");
      p.lam_form = form;
      if (form >= 0) { REQUIRE(h, ng >= 6, "LAM needs {B, R1, R2, x0, y0, z0}"); memcpy(p.lam, g, 6 * sizeof(double)); }
      break;
    case MMM_TERM_CF:
      REQUIRE(h, form >= -1 && form <= MMM_CF_LOGISTIC, "Unknown CENTRAL_FORCE_TYPE");
      p.cf_form = form;
      if (form >= 0) { REQUIRE(h, ng >= 5, "CF needs {G, R1, x0, y0, z0}"); memcpy(p.cf, g, 5 * sizeof(double)); }
      break;
    default:
      return mmm_fail(h, MMM_ERR_ARG, "mmm_set_external_term: term is not an external term");
  }
  return MMM_OK;
}

int mmm_set_cutoff(mmm_handle h, double rc_nm) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, rc_nm >= 0.0 && isfinite(rc_nm), "mmm_set_cutoff: cutoff must be >= 0");
  h->cutoff = rc_nm;
  h->sort_age = 0;
  derive_pair_params(h);
  return MMM_OK;
}

// ---- state -----------------------------------------------------------------------------
static int set_center_from_host(mmm_system* h, const double* x) {
  // arithmetic mean in index order: identical on the oracle side, so the FP32 copies agree bit for bit.
  // The same pass is the finiteness check: a NaN or an infinity anywhere leaves a non-finite sum.
  double c0 = 0, c1 = 0, c2 = 0;
  for (int64_t i = 0; i < h->n; ++i) {
    c0 += x[3 * i];
    c1 += x[3 * i + 1];
    c2 += x[3 * i + 2];
  }
  if (!isfinite(c0) || !isfinite(c1) || !isfinite(c2)) {
    cudaStreamSynchronize(h->stream);  // the caller's buffer may still be in flight
    return mmm_fail(h, MMM_ERR_NUMERIC, "non-finite coordinate");
  }
  double c[3] = {c0 / (double)h->n, c1 / (double)h->n, c2 / (double)h->n};
  MMM_CUDA(h, cudaMemcpyAsync(h->d_center, c, sizeof(c), cudaMemcpyHostToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_set_positions(mmm_handle h, const double* xyz) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, xyz, "mmm_set_positions: NULL");
  cudaSetDevice(h->device);
  // the copy (asynchronous from pinned memory) overlaps the host's one pass over the coordinates
  MMM_CUDA(h, cudaMemcpyAsync(h->d_x, xyz, sizeof(double) * 3 * h->n, cudaMemcpyHostToDevice, h->stream));
  int rc = set_center_from_host(h, xyz);
  if (rc) {
    h->positions_set = false;  // d_x holds the rejected coordinates
    return rc;
  }
  h->positions_set = true;
  h->sort_age = 0;  // cut-off mode: new positions from outside, rebuild the Morton order
  return MMM_OK;
}

int mmm_get_positions(mmm_handle h, double* out) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, out, "mmm_get_positions: NULL");
  REQUIRE(h, h->positions_set, "mmm_get_positions: positions were never set");
  cudaSetDevice(h->device);
  MMM_CUDA(h, cudaMemcpyAsync(out, h->d_x, sizeof(double) * 3 * h->n, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

static int refresh_center_from_device(mmm_system* h) {
  std::vector<double> x(3 * (size_t)h->n);
  MMM_CUDA(h, cudaMemcpyAsync(x.data(), h->d_x, sizeof(double) * x.size(), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return set_center_from_host(h, x.data());
}

int mmm_set_positions_device(mmm_handle h, const double* d_xyz) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, d_xyz, "mmm_set_positions_device: NULL");
  cudaSetDevice(h->device);
  MMM_CUDA(h, cudaMemcpyAsync(h->d_x, d_xyz, sizeof(double) * 3 * h->n, cudaMemcpyDeviceToDevice, h->stream));
  int rc = refresh_center_from_device(h);
  if (rc) return rc;
  h->positions_set = true;
  h->sort_age = 0;
  return MMM_OK;
}

int mmm_get_positions_device(mmm_handle h, double* d_out) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, d_out, "mmm_get_positions_device: NULL");
  REQUIRE(h, h->positions_set, "mmm_get_positions_device: positions were never set");
  cudaSetDevice(h->device);
  MMM_CUDA(h, cudaMemcpyAsync(d_out, h->d_x, sizeof(double) * 3 * h->n, cudaMemcpyDeviceToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_hilbert_init(mmm_handle h, int p, double spacing_nm) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, p >= 1 && p <= 10, "mmm_hilbert_init: order p must be in [1, 10]");
  REQUIRE(h, h->n <= ((int64_t)1 << (3 * p)), "mmm_hilbert_init: N exceeds the 2^(3p) points of the curve");
  cudaSetDevice(h->device);
  int rc = mmm_launch_hilbert(h, p, spacing_nm, nullptr);
  if (rc) return rc;
  if ((rc = refresh_center_from_device(h))) return rc;
  h->positions_set = true;
  h->sort_age = 0;
  return MMM_OK;
}

int mmm_hilbert_points(mmm_handle h, int p, int32_t* ijk_out) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, ijk_out, "mmm_hilbert_points: NULL");
  REQUIRE(h, p >= 1 && p <= 10, "mmm_hilbert_points: order p must be in [1, 10]");
  REQUIRE(h, h->n <= ((int64_t)1 << (3 * p)), "mmm_hilbert_points: N exceeds the 2^(3p) points of the curve");
  cudaSetDevice(h->device);
  DevBuf<int32_t> d_ijk;
  int rc;
  if ((rc = mmm_reserve(h, d_ijk, 3 * (size_t)h->n, "Hilbert points")) || (rc = mmm_launch_hilbert(h, p, 0.0, d_ijk)))
    return rc;
  MMM_CUDA(h, cudaMemcpyAsync(ijk_out, d_ijk, sizeof(int32_t) * 3 * h->n, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

}  // extern "C"

// ---- evaluation --------------------------------------------------------------------------
static bool any_pair_term(const mmm_system* h) {
  return h->pp.ev_form >= 0 || h->pp.cob_form >= 0 || h->pp.scb_form >= 0 || h->pp.chb_form >= 0;
}

// Which pair kernel serves the current parameters.
static int wanted_pair_mode(const mmm_system* h) {
  if (!any_pair_term(h)) return 0;
  if (h->cutoff > 0.0) return 3;
  if (h->pair_kernel_pref != 1 && (mmm_pair_n3_eligible(h) || mmm_pair_n3_generic(h))) return 2;
  return 1;
}

static void free_scratch(mmm_system* h) {
  cudaStreamSynchronize(h->stream);
  h->d_fpair.reset();
  h->d_epair_buf.reset();
  h->d_epair = nullptr;
  h->d_facc.reset();
  h->d_items.reset();
  h->d_items_cut.reset();
  h->d_cut_npairs.reset();
  h->d_cut_eacc.reset();
  h->scratch_sig = -1;
}

// Size the pair-kernel work decomposition and its scratch for the kernel that will run.
static int ensure_scratch(mmm_system* h) {
  const int mode = wanted_pair_mode(h);
  // cut-off mode: the default forms run on the Newton-3 machinery over Morton-sorted tiles
  // (mmm_cutoff.cu), every other form on the cell-list gather kernel (mmm_cells.cu)
  const bool cut_n3 = mode == 3 && h->pair_kernel_pref != 1 && mmm_pair_n3_eligible(h);
  // coarse-stage surrogate: CHB on cluster centroids instead of the exact same-chromosome pass
  // (and the EV tail beyond the cut-off); default forms only
  const bool chb_cl = mode == 3 && h->chb_surrogate && cut_n3;
  // pair_kernel_pref 2: the CTA-level CUT variant instead of the one-warp-per-item kernel (A/B timing)
  const bool cut_warp = cut_n3 && h->pair_kernel_pref != 2;
  const int sig = mode * 4 + (mode == 3 ? h->pp.chb_form + 1 : 0) + (cut_n3 ? 64 : 0) + (chb_cl ? 128 : 0) +
                  (cut_warp ? 256 : 0);
  if (h->scratch_sig == sig) return MMM_OK;
  free_scratch(h);
  h->pair_mode = mode;
  h->cut_n3 = cut_n3;
  h->cut_warp = cut_warp;
  h->chb_clusters = chb_cl;
  h->sort_age = 0;
  int rc;
  if (chb_cl && h->nccl_comm) return mmm_fail(h, MMM_ERR_STATE, "the CHB cluster surrogate is single-GPU (coarse stage of the two-stage minimisation)");
  // cut-off mode with CHB on: an exact CHB-only pass runs beside the cell-list pass — the Newton-3
  // kernel over same-chromosome tile pairs for the polynomial form, the generic gather kernel else
  const bool chb_n3 = mode == 3 && h->pp.chb_form == MMM_CHB_POLYNOMIAL && !chb_cl;
  const bool chb_gather = mode == 3 && h->pp.chb_form >= 0 && !chb_n3 && !chb_cl;
  h->n_items = 0;
  h->n3_items = 0;
  h->n_planes = 0;
  h->nchunk = 1;
  std::vector<int2> items_cut;
  if (cut_warp) mmm_cut_warp_build_items(h, items_cut);
  else if (cut_n3) mmm_n3_build_items(h, items_cut, false);
  // energy slots of the cut-off pass: one per item (CTA-level kernel) or one per rank (warp kernel)
  h->n_cut_slots = cut_warp ? h->dist_world : (int)items_cut.size();
  if (mode == 2 || chb_n3) {
    // Newton-3: fixed-point force planes + work-item table
    std::vector<int2> items;
    mmm_n3_build_items(h, items, chb_n3);
    h->n3_items = (int)items.size();
    h->n3_chb_only = chb_n3;
    h->n_items = h->n3_items;
    if ((rc = mmm_upload(h, h->d_items, items, "Newton-3 work items"))) return rc;
  }
  if (mode == 2 || chb_n3 || cut_n3) {
    // several GPUs: the per-item energy slots live behind the force planes in the same allocation,
    // so that ONE all-reduce (uint64 sum) covers both (mmm_dist.cu)
    const size_t tail = h->nccl_comm ? 4 * ((size_t)h->n3_items + (size_t)h->n_cut_slots) : 0;
    if ((rc = mmm_reserve(h, h->d_facc, 3 * (size_t)h->npad + tail, "force accumulator"))) return rc;
    MMM_CUDA(h, cudaMemsetAsync(h->d_facc, 0, sizeof(unsigned long long) * (3 * (size_t)h->npad + tail), h->stream));
  }
  if (mode == 1 || chb_gather) {
    // gather kernel: items = i-blocks x j-chunks, enough of them that the dynamic scheduler keeps
    // every SM busy to the end; one partial-force plane per chunk
    const int64_t niblk = h->npad / MMM_IBLOCK;
    const int64_t stages = h->ntiles / (MMM_STAGE / MMM_TILE);
    const int64_t target = (int64_t)h->sm_count * 4 * 6;  // ~6 items per resident CTA
    int64_t nchunk = (target + niblk - 1) / niblk;
    nchunk = std::max<int64_t>(1, std::min<int64_t>(nchunk, std::min<int64_t>(stages, 64)));
    // chunks are whole stages; recompute the count so that no chunk is empty
    const int64_t chunk_stages = (stages + nchunk - 1) / nchunk;
    nchunk = (stages + chunk_stages - 1) / chunk_stages;
    h->nchunk = (int)nchunk;
    h->chunk_tiles = (int)((stages + nchunk - 1) / nchunk) * (MMM_STAGE / MMM_TILE);
    h->n_items = niblk * nchunk;
    h->n_planes = (int)nchunk;
  }
  if (cut_n3) {
    const std::vector<int2>& items = items_cut;
    h->n_items_cut = (int)items.size();
    h->h_cut_iblk.resize(items.size());
    for (size_t q = 0; q < items.size(); ++q) h->h_cut_iblk[q] = items[q].x;
    if ((rc = mmm_upload(h, h->d_items_cut, items, "cut-off work items"))) return rc;
    if ((rc = mmm_reserve(h, h->d_cut_npairs, (size_t)h->n_cut_slots, "cut-off pair counts"))) return rc;
    MMM_CUDA(h, cudaMemsetAsync(h->d_cut_npairs, 0, sizeof(double) * (size_t)h->n_cut_slots, h->stream));
    if (cut_warp) {
      if ((rc = mmm_reserve(h, h->d_cut_eacc, 4, "cut-off energy accumulator"))) return rc;
      MMM_CUDA(h, cudaMemsetAsync(h->d_cut_eacc, 0, sizeof(unsigned long long) * 4, h->stream));
    }
    h->cells_item0 = h->n_items;
    h->n_items += h->n_cut_slots;
  } else if (mode == 3) {
    h->cells_plane = h->n_planes;
    h->cells_item0 = h->n_items;
    h->n_planes += 1;
    h->n_items += mmm_cells_energy_slots(h);
  }
  if (chb_cl) {
    if ((rc = mmm_chb_clusters_build(h))) return rc;
    h->cl_item0 = h->n_items;
    h->n_items += mmm_chb_clusters_blocks(h);
  }
  if (h->n_items == 0) h->n_items = 1;
  if (h->n_planes > 0) {
    const size_t cnt = (size_t)h->n_planes * 3 * (size_t)h->npad;
    if ((rc = mmm_reserve(h, h->d_fpair, cnt, "force planes"))) return rc;
    MMM_CUDA(h, cudaMemsetAsync(h->d_fpair, 0, sizeof(double) * cnt, h->stream));
  }
  if (h->nccl_comm) {
    const bool chb_ok = h->pp.chb_form < 0 || h->pp.chb_form == MMM_CHB_POLYNOMIAL;
    if (!(mode == 2 || (cut_n3 && chb_ok)))
      return mmm_fail(h, MMM_ERR_STATE, "the multi-GPU path needs the Newton-3 kernel (in cut-off mode: default functional forms, EV on)");
    h->d_epair = reinterpret_cast<double*>(h->d_facc + 3 * (size_t)h->npad);
  } else {
    if ((rc = mmm_reserve(h, h->d_epair_buf, (size_t)h->n_items * 4, "energy slots"))) return rc;
    h->d_epair = h->d_epair_buf;
    MMM_CUDA(h, cudaMemsetAsync(h->d_epair, 0, sizeof(double) * (size_t)h->n_items * 4, h->stream));
  }
  h->scratch_sig = sig;
  return MMM_OK;
}

int mmm_evaluate(mmm_system* h, const int* d_skip) {
  int rc;
  if (h->topo_dirty && (rc = mmm_upload_topology(h))) return rc;
  if ((rc = ensure_scratch(h))) return rc;
  if ((rc = mmm_launch_prepare(h, d_skip))) return rc;
  // several GPUs: the energy slots of the other ranks' items must enter the all-reduce as zero bits
  if (h->nccl_comm) MMM_CUDA(h, cudaMemsetAsync(h->d_epair, 0, sizeof(double) * 4 * (size_t)h->n_items, h->stream));
  if (h->pair_mode == 3) {
    if (h->chb_clusters) {
      if ((rc = mmm_launch_chb_clusters(h, d_skip))) return rc;
    } else if (h->pp.chb_form == MMM_CHB_POLYNOMIAL) {
      if ((rc = mmm_launch_pair_n3(h, d_skip, true))) return rc;
    } else if (h->pp.chb_form >= 0) {
      PairParams only_chb = h->pp;
      only_chb.ev_form = only_chb.cob_form = only_chb.scb_form = MMM_FORM_OFF;
      only_chb.cutoff2 = 0.0f;
      if ((rc = mmm_launch_pair_exact(h, d_skip, &only_chb))) return rc;
    }
    rc = h->cut_n3 ? mmm_launch_pair_cutoff_n3(h, d_skip) : mmm_launch_pair_cutoff(h, d_skip);
    if (!rc && h->nccl_comm) rc = mmm_dist_allreduce(h);
  } else if (h->pair_mode == 2) {
    rc = mmm_launch_pair_n3(h, d_skip);
    // the one exchange step per evaluation (every rank enqueues it, converged or not, so that
    // the collective can never be entered by some ranks only)
    if (!rc && h->nccl_comm) rc = mmm_dist_allreduce(h);
  }
  else if (h->pair_mode == 1) rc = mmm_launch_pair_exact(h, d_skip);
  if (rc) return rc;
  return mmm_launch_assemble(h, d_skip);
}

static __global__ void __launch_bounds__(256) k_negate(int64_t n3, const double* __restrict__ g, double* __restrict__ f) {
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e < n3) f[e] = -g[e];
}

static int check_ready(mmm_system* h) {
  if (!h->positions_set) return mmm_fail(h, MMM_ERR_STATE, "positions were never set");
  return MMM_OK;
}

extern "C" {

int mmm_energy_forces_device(mmm_handle h, double* e_terms, double* d_forces) {
  if (!h) return MMM_ERR_ARG;
  int rc = check_ready(h);
  if (rc) return rc;
  cudaSetDevice(h->device);
  if ((rc = mmm_evaluate(h, nullptr))) return rc;
  if ((rc = mmm_launch_finalize_energy(h))) return rc;
  double e[MMM_NUM_TERMS];
  MMM_CUDA(h, cudaMemcpyAsync(e, h->d_eterms, sizeof(e), cudaMemcpyDeviceToHost, h->stream));
  if (d_forces)
    MMM_CUDA(h, cudaMemcpyAsync(d_forces, h->d_g, sizeof(double) * 3 * h->n, cudaMemcpyDeviceToDevice, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->pair_mode != 0) cudaEventElapsedTime(&h->last_pair_ms, h->ev_a, h->ev_b);
  double tot = 0;
  for (int t = 0; t < MMM_NUM_TERMS; ++t) tot += e[t];
  if (e_terms) memcpy(e_terms, e, sizeof(e));
  if (!isfinite(tot)) return mmm_fail(h, MMM_ERR_NUMERIC, "non-finite energy");
  return MMM_OK;
}

// d_g holds the gradient: negated on the device, not by a host pass over 24 N bytes
static int copy_forces_to_host(mmm_system* h, double* forces) {
  int rc = mmm_reserve(h, h->d_fout, 3 * (size_t)h->n, "force copy");
  if (rc) return rc;
  k_negate<<<(unsigned)((3 * h->n + 255) / 256), 256, 0, h->stream>>>(3 * h->n, h->d_g, h->d_fout);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  MMM_CUDA(h, cudaMemcpyAsync(forces, h->d_fout, sizeof(double) * 3 * h->n, cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  return MMM_OK;
}

int mmm_energy_forces(mmm_handle h, double* e_terms, double* forces) {
  if (!h) return MMM_ERR_ARG;
  int rc = mmm_energy_forces_device(h, e_terms, nullptr);
  if (rc) return rc;
  return forces ? copy_forces_to_host(h, forces) : MMM_OK;
}

int mmm_last_result(mmm_handle h, double* e_terms, double* forces) {
  if (!h) return MMM_ERR_ARG;
  if (!h->have_result) return mmm_fail(h, MMM_ERR_STATE, "mmm_last_result: no result to read (nothing evaluated since creation, mmm_minimize or mmm_md_run)");
  cudaSetDevice(h->device);
  if (e_terms) {
    MMM_CUDA(h, cudaMemcpyAsync(e_terms, h->d_eterms, sizeof(double) * MMM_NUM_TERMS, cudaMemcpyDeviceToHost, h->stream));
    MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return forces ? copy_forces_to_host(h, forces) : MMM_OK;
}

int mmm_evaluate_n(mmm_handle h, int n) {
  if (!h) return MMM_ERR_ARG;
  int rc = check_ready(h);
  if (rc) return rc;
  cudaSetDevice(h->device);
  for (int q = 0; q < n; ++q) {
    if ((rc = mmm_evaluate(h, nullptr))) return rc;
    if ((rc = mmm_launch_finalize_energy(h))) return rc;
  }
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->pair_mode != 0) cudaEventElapsedTime(&h->last_pair_ms, h->ev_a, h->ev_b);
  return MMM_OK;
}

int mmm_evaluate_timed(mmm_handle h, int n, int flush_l2, float* total_ms, float* pair_ms) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, n >= 1 && n <= 100000, "mmm_evaluate_timed: n must be in [1, 100000]");
  int rc = check_ready(h);
  if (rc) return rc;
  cudaSetDevice(h->device);
  const size_t flush_bytes = (size_t)256 << 20;
  if (flush_l2 && (rc = mmm_reserve(h, h->d_flush, flush_bytes, "L2-flush scratch"))) return rc;
  while (h->ev_pool.size() < (size_t)2 * n + 2) {
    cudaEvent_t e;
    MMM_CUDA(h, cudaEventCreate(&e));
    h->ev_pool.push_back(e);
  }
  // the last two pool events bracket the whole batch
  cudaEvent_t t0 = h->ev_pool[h->ev_pool.size() - 2], t1 = h->ev_pool[h->ev_pool.size() - 1];
  h->ev_cursor = any_pair_term(h) ? 0 : -1;
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  MMM_CUDA(h, cudaEventRecord(t0, h->stream));
  for (int q = 0; q < n; ++q) {
    if (flush_l2) MMM_CUDA(h, cudaMemsetAsync(h->d_flush, q & 0xff, flush_bytes, h->stream));
    if ((rc = mmm_evaluate(h, nullptr))) { h->ev_cursor = -1; return rc; }
    if ((rc = mmm_launch_finalize_energy(h))) { h->ev_cursor = -1; return rc; }
  }
  MMM_CUDA(h, cudaEventRecord(t1, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  const int collected = h->ev_cursor;
  h->ev_cursor = -1;
  float tot = 0.f, pair = 0.f;
  cudaEventElapsedTime(&tot, t0, t1);
  for (int q = 0; q < collected; ++q) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev_pool[2 * q], h->ev_pool[2 * q + 1]);
    pair += ms;
  }
  if (collected > 0) h->last_pair_ms = pair / collected;
  if (total_ms) *total_ms = tot;
  if (pair_ms) *pair_ms = pair;
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}

int mmm_minimize(mmm_handle h, double tol, int64_t max_iter, mmm_min_report* out) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, tol > 0.0 && max_iter >= 0, "mmm_minimize: tolerance must be > 0 and max_iter >= 0");
  int rc = check_ready(h);
  if (rc) return rc;
  cudaSetDevice(h->device);
  const size_t n3 = 3 * (size_t)h->n;
  if ((rc = mmm_reserve(h, h->d_xp, n3, "L-BFGS x")) || (rc = mmm_reserve(h, h->d_gp, n3, "L-BFGS g")) ||
      (rc = mmm_reserve(h, h->d_d, n3, "L-BFGS direction")) ||
      (rc = mmm_reserve(h, h->d_S, n3 * MMM_LBFGS_M, "L-BFGS s history")) ||
      (rc = mmm_reserve(h, h->d_Y, n3 * MMM_LBFGS_M, "L-BFGS y history")))
    return rc;
  h->have_result = false;  // the line search leaves trial-point state in d_g / d_eterms
  return mmm_run_minimize(h, tol, max_iter, out);
}

int64_t mmm_launch_count(mmm_handle h) { return h ? h->launches : 0; }

int mmm_set_pair_kernel(mmm_handle h, int which) {
  if (!h) return MMM_ERR_ARG;
  REQUIRE(h, which >= 0 && which <= 2, "mmm_set_pair_kernel: 0 = automatic, 1 = gather kernels, 2 = CTA-level cut-off kernel");
  h->pair_kernel_pref = which;
  return MMM_OK;
}

int mmm_pair_kernel_in_use(mmm_handle h) { return h ? h->pair_mode : 0; }

int mmm_set_chb_surrogate(mmm_handle h, int on) {
  if (!h) return MMM_ERR_ARG;
  h->chb_surrogate = on != 0;
  return MMM_OK;
}

int mmm_set_graph(mmm_handle h, int on) {
  if (!h) return MMM_ERR_ARG;
  h->no_graph = on == 0;
  return MMM_OK;
}

int mmm_last_pair_kernel_ms(mmm_handle h, float* ms_out) {
  if (!h || !ms_out) return MMM_ERR_ARG;
  *ms_out = h->last_pair_ms;
  return MMM_OK;
}

}  // extern "C"
