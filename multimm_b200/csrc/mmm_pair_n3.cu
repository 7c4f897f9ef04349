// mmm_pair_n3.cu — exact all-pairs ("NoCutoff") pair kernel, Newton's-third-law formulation,
// for sm_100a.  Default path for the reference's default functional forms: power-law EV with an
// integer power (model.py:199), Gaussian COB/SCB (model.py:246-250, 322-328), polynomial CHB
// (model.py:416-419).  Every unordered pair is evaluated ONCE (the gather kernel in mmm_pair.cu
// visits it from both sides), and the result is still bit-reproducible.
//
// Decomposition
//   i-block  = 512 consecutive beads, stationary in registers for a whole work item:
//              warp w owns 64 of them, lane (a = lane >> 2, b = lane & 3) holds the 8 beads
//              64 w + 8 a + {0..7}; the four b-lanes of a group hold the same beads.
//   j-stage  = 256 consecutive beads in shared memory (float4 xyz + type bits, and a negated,
//              duplicated copy for the packed path), double buffered.
//   step     = one tile of 32 j-beads: register ii of lane (a, b) meets j-bead 4 (jj ^ a) + b,
//              jj = 0..7, so a lane evaluates an 8 x 8 rectangle = 64 pairs and a warp 64 x 32.
//   item     = (i-block, run of <= cj j-stages), handed out by an atomic counter; only j-stages at
//              or above the diagonal exist.  The two stages that overlap the i-block itself are
//              evaluated in "diagonal" mode: ordered pairs, i-side only, energy halved, self masked.
//
// Accumulation (all in units of U = p eps sigma^p, the EV force prefactor)
//   i side : 24 FP32 registers per lane for the whole item, butterfly over the 4 b-lanes at the
//            end, then 64-bit fixed-point RED.ADD to facc[3][npad].
//   j side : 24 FP32 registers per step.  The XOR mapping above makes the reduce-scatter over
//            the 8 a-lanes select-free: 12 + 6 + 3 SHFL.BFLY/FADD pairs leave lane l holding the
//            total for j-bead 32 step + l, which it adds to its warp's private shared-memory
//            column.  After the stage, thread t sums the 8 warp columns of j-bead t in fixed
//            order and issues 3 fixed-point REDs.
//   Integer addition is associative, so the force is independent of which CTA ran which item
//   and in which order: deterministic per-bead accumulation without a partial-sum buffer per
//   chunk.  Resolution 2^-24 kJ/mol/nm, range +-5.5e11.
//   energies: FP32 within a stage, FP64 across stages, one slot per item (fixed order).
//
// Tile classification is warp-uniform, from the 32-bead bounding boxes / chromosome ranges of
// k_prepare (lane s classifies tile s of the stage, the steps fetch their class by shuffle): far
// tiles skip the Gaussians (< 2^-26 of their prefactor), CHB only where the chromosome ranges
// overlap, per-pair chromosome compare only when a tile is not single-chromosome.
//
// The hot variant (far, no CHB) per unordered pair: 3 add (dx,dy,dz), mul + 2 fma (r^2),
// MUFU.SQRT, fma (q = r^2 + r_s r), MUFU.RCP (w/r), mul (w), 3 mul (w^6), add (energy), mul
// (w^6 w/r), 6 fma (both force accumulators) = 19 FMA-pipe operations + 2 MUFU.  They are issued as
// packed f32x2 instructions on two i-beads at a time (FFMA2 / FMUL2 / FADD2: 9.5 issue slots per
// pair), which moves the bound from instruction issue to the FMA pipe: 19 cycles per warp-pair per
// scheduler.  The 64 pairs of a step run as a rolled loop over 16-pair groups, unrolled by 2 (a
// fully unrolled body was instruction-fetch bound); the stationary beads are loaded from
// coordinate planes (d_soa) so that they arrive as aligned register pairs.
// Measured (profiles/r01_pair_n3_*): the hot loop runs at ~78 % of that floor, the kernel at
// 0.58-0.60 of the measured FFMA peak on SURVEY 8(d)'s algorithmic flops (28 flop per EV pair).
#include <algorithm>

#include "mmm_internal.cuh"
#include "mmm_pairmath.cuh"

namespace {

constexpr int N3_THREADS = 256;
constexpr int N3_WARPS = N3_THREADS / 32;
constexpr int N3_IB = 512;                 // i-beads per block
constexpr int N3_JB = 256;                 // j-beads per stage
constexpr int N3_STEPS = N3_JB / MMM_TILE; // 8
constexpr double N3_FIXED = 16777216.0;    // 2^24
#ifndef N3_GROUP_UNROLL
#define N3_GROUP_UNROLL 2
#endif
constexpr int kGroupUnroll = N3_GROUP_UNROLL;
#ifndef N3_USE_F32X2
#define N3_USE_F32X2 1
#endif
#ifndef N3_PACKED_NEAR
#define N3_PACKED_NEAR 1  // tiles within the Gaussian range: packed f32x2 body (0: the scalar one)
#endif
#ifndef N3_MIN_BLOCKS
#define N3_MIN_BLOCKS 2  // resident CTAs per SM the register budget is set for (2: 128 registers; 3: 80)
#endif

static_assert(N3_IB == MMM_PAD_TO, "npad must be a multiple of the i-block");
static_assert(N3_IB == N3_WARPS * 64, "a warp owns 64 i-beads");

__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_sqrt(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int P>
__device__ __forceinline__ float powi(float w) {
  if constexpr (P == 1) {
    return w;
  } else if constexpr (P % 2 == 0) {
    const float hf = powi<P / 2>(w);
    return hf * hf;
  } else {
    return w * powi<P - 1>(w);
  }
}

struct N3Consts {
  float ev_rs;
  float g_c;       // -log2(e) / (2 rc^2)
  float rg2;       // Gaussian range^2 (box test)
  float chb_kc;
  float chb_c;     // dE / U
  float a_scb[5];  // eps(s) / (rc^2 U), indexed by s + 2
  float a_cob[4];  // by class bits: [1] = A, [2] = B, others 0
  int gk;          // bit 0: SCB on, bit 1: COB on
  float cut2;      // cut-off^2 (CUT variants): pairs with r^2 >= cut2 contribute nothing
};

struct N3Args {
  const float4* pos4;
  const float* soa;          // [3][npad] coordinate planes
  const TileInfo* tiles;
  unsigned long long* facc;  // [3][npad] fixed-point force, units 2^-24 kJ/mol/nm
  double* epair;             // [n_items][4]
  const int2* items;         // (i-block, first j-stage | number of stages << 24)
  int* counter;
  const int* skip;
  int64_t npad;
  int n_items;
  int item_first, item_stride;  // this launch handles items item_first + k * item_stride
  int sys_counter;              // the counter lives in another GPU's memory: system-scope atomics (NVLink)
  double fscale;             // U * 2^24
  double e_ev, e_gauss, e_chb;  // energy prefactors: eps sigma^p; -rc^2 U; dE
  // CUT variants (mmm_cutoff.cu): the arrays above are in Morton-sorted order
  const TileInfo* stage_boxes;  // [npad / 256] bounding box of every j-stage
  const int* perm;              // sorted slot -> bead id (force emission)
  double* npairs;               // [n_items] pairs inside the cut-off, per item
  N3Consts c;
  PairParams pp;                // generic variant (EVP < 0) only: every functional form, FP64 body
};


typedef unsigned long long u64;

// Packed FP32 pairs (sm_100 f32x2 arithmetic: FFMA2 / FMUL2 / FADD2).  One issue slot does two
// FP32 operations, so the hot loop is bound by the FMA pipe (19 lane-ops per pair) instead of
// by instruction issue (21 per pair); MUFU works on the halves of a pair in place, ptxas
// coalesces the pack/unpack moves away.
__device__ __forceinline__ u64 pk2(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpk2(u64 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
// Positions live as packed register pairs (beads 2m, 2m+1) so that the f32x2 path reads them
// without moves; the scalar variants address the halves.
struct IBeads {
  u64 x2[4], y2[4], z2[4];
  float fx[8], fy[8], fz[8];
  __device__ __forceinline__ float x(int ii) const { float lo, hi; unpk2(x2[ii >> 1], lo, hi); return (ii & 1) ? hi : lo; }
  __device__ __forceinline__ float y(int ii) const { float lo, hi; unpk2(y2[ii >> 1], lo, hi); return (ii & 1) ? hi : lo; }
  __device__ __forceinline__ float z(int ii) const { float lo, hi; unpk2(z2[ii >> 1], lo, hi); return (ii & 1) ? hi : lo; }
};

__device__ __forceinline__ u64 fma2(u64 x, u64 y, u64 z) {
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(x), "l"(y), "l"(z));
  return d;
}
__device__ __forceinline__ u64 mul2(u64 x, u64 y) {
  u64 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(x), "l"(y));
  return d;
}
__device__ __forceinline__ u64 add2(u64 x, u64 y) {
  u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(x), "l"(y));
  return d;
}

template <int P>
__device__ __forceinline__ u64 powi2(u64 w) {
  if constexpr (P == 1) {
    return w;
  } else if constexpr (P % 2 == 0) {
    const u64 hf = powi2<P / 2>(w);
    return mul2(hf, hf);
  } else {
    return mul2(w, powi2<P - 1>(w));
  }
}

struct EAcc {
  float ev, scb, cob, chb;
  u64 ev2, chb2;  // packed partial sums of the f32x2 path
  float cnt;      // CUT: pairs inside the cut-off (reported through the CHB slot, which a CUT pass never uses)
  u64 cnt2;
  u64 scb2, cob2;  // packed partial sums of the Gaussian-range packed path
  double gen[4];   // generic variant: EV, COB, SCB, CHB in kJ/mol (all prefactors applied)
};

// j-beads of a stage, laid out for the packed path: xy[j] = {-x, -x, -y, -y}, z[j] = {-z, -z}
struct JDup {
  const float4* xy;
  const float2* z;
};

// Packed variant of pairs16 for the hot cases (no Gaussians, no self pairs; CHBM 0 or 1): the 8
// i-beads are processed as 4 register pairs.
template <int EVP, int CHBM, bool CUT>
__device__ __forceinline__ void pairs16_packed(const JDup sjd, const int a, const int b, const int jj0,
                                               IBeads& I, float (&cx)[2], float (&cy)[2], float (&cz)[2],
                                               EAcc& E, const N3Consts& c) {
  const u64 rs2 = pk2(c.ev_rs, c.ev_rs);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int jl = (((jj0 + k) ^ a) << 2) | b;
    const float4 nxy = sjd.xy[jl];
    const float2 nz = sjd.z[jl];
    const u64 njx = pk2(nxy.x, nxy.y), njy = pk2(nxy.z, nxy.w), njz = pk2(nz.x, nz.y);
    u64 ax = pk2(0.0f, 0.0f), ay = ax, az = ax;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const u64 dx = add2(I.x2[m], njx);
      const u64 dy = add2(I.y2[m], njy);
      const u64 dz = add2(I.z2[m], njz);
      const u64 r2 = fma2(dz, dz, fma2(dy, dy, mul2(dx, dx)));
      float r2a, r2b;
      unpk2(r2, r2a, r2b);
      const u64 r = pk2(fast_sqrt(r2a), fast_sqrt(r2b));
      u64 fs = pk2(0.0f, 0.0f);
      if constexpr (EVP > 0) {
        const u64 q = fma2(rs2, r, r2);
        float qa, qb;
        unpk2(q, qa, qb);
        const u64 wr = pk2(fast_rcp(qa), fast_rcp(qb));  // w / r
        const u64 w = mul2(r, wr);
        u64 wp = powi2<EVP>(w);
        if (CUT) {  // plain truncation: the oracle's pair_in_cut on the same FP32 r^2
          const u64 in2 = pk2(r2a < c.cut2 ? 1.0f : 0.0f, r2b < c.cut2 ? 1.0f : 0.0f);
          wp = mul2(wp, in2);
          E.cnt2 = add2(E.cnt2, in2);
        }
        E.ev2 = add2(E.ev2, wp);
        fs = mul2(wp, wr);
      }
      if (CHBM == 1) {
        const u64 kc2 = pk2(c.chb_kc, c.chb_kc), one2 = pk2(1.0f, 1.0f), mone2 = pk2(-1.0f, -1.0f);
        const u64 t = fma2(kc2, r2, fma2(mone2, r, one2));  // kC r^2 + 1 - r
        E.chb2 = fma2(r2, t, E.chb2);
        const u64 kc4 = pk2(4.0f * c.chb_kc, 4.0f * c.chb_kc), two2 = pk2(2.0f, 2.0f), m3 = pk2(-3.0f, -3.0f);
        const u64 bb = fma2(m3, r, fma2(kc4, r2, two2));
        const u64 nc = pk2(-c.chb_c, -c.chb_c);
        fs = fma2(nc, bb, fs);
      }
      u64 t;
      t = fma2(fs, dx, pk2(I.fx[2 * m], I.fx[2 * m + 1])); unpk2(t, I.fx[2 * m], I.fx[2 * m + 1]);
      t = fma2(fs, dy, pk2(I.fy[2 * m], I.fy[2 * m + 1])); unpk2(t, I.fy[2 * m], I.fy[2 * m + 1]);
      t = fma2(fs, dz, pk2(I.fz[2 * m], I.fz[2 * m + 1])); unpk2(t, I.fz[2 * m], I.fz[2 * m + 1]);
      ax = fma2(fs, dx, ax);
      ay = fma2(fs, dy, ay);
      az = fma2(fs, dz, az);
    }
    float lo, hi;
    unpk2(ax, lo, hi); cx[k] = lo + hi;
    unpk2(ay, lo, hi); cy[k] = lo + hi;
    unpk2(az, lo, hi); cz[k] = lo + hi;
  }
}

// Packed variant for tiles within the Gaussian range (and for every tile of a cut-off pass whose
// cut-off is shorter than that range): EV + Gaussian block terms, optional same-chromosome CHB
// (CHBM 1), optional truncation.  The label match of a block term is integer work on the ALU pipe
// (2 LOP3 + 2 FSEL per term and register pair), everything else is packed; 3 MUFU per pair.
template <int EVP, int GK, int CHBM, bool CUT>
__device__ __forceinline__ void pairs16_packed_near(const float4* __restrict__ sj, const JDup sjd, const int a,
                                                    const int b, const int jj0, IBeads& I, float (&cx)[2],
                                                    float (&cy)[2], float (&cz)[2], EAcc& E, const N3Consts& c,
                                                    const int* __restrict__ si4) {
  const u64 rs2 = pk2(c.ev_rs, c.ev_rs), gc2 = pk2(c.g_c, c.g_c), mone2 = pk2(-1.0f, -1.0f);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int jl = (((jj0 + k) ^ a) << 2) | b;
    const float4 nxy = sjd.xy[jl];
    const float2 nz = sjd.z[jl];
    const int tj = __float_as_int(sj[jl].w);
    const float aj_scb = (GK & 1) ? c.a_scb[tj & 7] : 0.0f;
    const float aj_cob = (GK & 2) ? c.a_cob[(tj >> 3) & 3] : 0.0f;
    const u64 njx = pk2(nxy.x, nxy.y), njy = pk2(nxy.z, nxy.w), njz = pk2(nz.x, nz.y);
    u64 ax = pk2(0.0f, 0.0f), ay = ax, az = ax;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const u64 dx = add2(I.x2[m], njx);
      const u64 dy = add2(I.y2[m], njy);
      const u64 dz = add2(I.z2[m], njz);
      const u64 r2 = fma2(dz, dz, fma2(dy, dy, mul2(dx, dx)));
      float r2a, r2b;
      unpk2(r2, r2a, r2b);
      const u64 r = pk2(fast_sqrt(r2a), fast_sqrt(r2b));
      const u64 q = fma2(rs2, r, r2);
      float qa, qb;
      unpk2(q, qa, qb);
      const u64 wr = pk2(fast_rcp(qa), fast_rcp(qb));  // w / r
      const u64 w = mul2(r, wr);
      u64 wp = powi2<EVP>(w);
      const u64 ge = mul2(r2, gc2);
      float ga, gb;
      unpk2(ge, ga, gb);
      u64 g = pk2(fast_ex2(ga), fast_ex2(gb));
      if (CUT) {
        const u64 in2 = pk2(r2a < c.cut2 ? 1.0f : 0.0f, r2b < c.cut2 ? 1.0f : 0.0f);
        wp = mul2(wp, in2);
        g = mul2(g, in2);
        E.cnt2 = add2(E.cnt2, in2);
      }
      E.ev2 = add2(E.ev2, wp);
      u64 fs = mul2(wp, wr);
      const int2 ti = *reinterpret_cast<const int2*>(si4 + 2 * m);  // labels of i-beads 2m, 2m + 1
      const int xa = ti.x ^ tj, xb = ti.y ^ tj;
      if (GK & 1) {
        const u64 t = mul2(pk2((xa & 0x7) == 0 ? aj_scb : 0.0f, (xb & 0x7) == 0 ? aj_scb : 0.0f), g);
        E.scb2 = add2(E.scb2, t);
        fs = fma2(mone2, t, fs);
      }
      if (GK & 2) {
        const u64 t = mul2(pk2((xa & 0x18) == 0 ? aj_cob : 0.0f, (xb & 0x18) == 0 ? aj_cob : 0.0f), g);
        E.cob2 = add2(E.cob2, t);
        fs = fma2(mone2, t, fs);
      }
      if (CHBM == 1) {
        const u64 kc2 = pk2(c.chb_kc, c.chb_kc), one2 = pk2(1.0f, 1.0f);
        const u64 t = fma2(kc2, r2, fma2(mone2, r, one2));  // kC r^2 + 1 - r
        E.chb2 = fma2(r2, t, E.chb2);
        const u64 kc4 = pk2(4.0f * c.chb_kc, 4.0f * c.chb_kc), two2 = pk2(2.0f, 2.0f), m3 = pk2(-3.0f, -3.0f);
        const u64 bb = fma2(m3, r, fma2(kc4, r2, two2));
        fs = fma2(pk2(-c.chb_c, -c.chb_c), bb, fs);
      }
      u64 t;
      t = fma2(fs, dx, pk2(I.fx[2 * m], I.fx[2 * m + 1])); unpk2(t, I.fx[2 * m], I.fx[2 * m + 1]);
      t = fma2(fs, dy, pk2(I.fy[2 * m], I.fy[2 * m + 1])); unpk2(t, I.fy[2 * m], I.fy[2 * m + 1]);
      t = fma2(fs, dz, pk2(I.fz[2 * m], I.fz[2 * m + 1])); unpk2(t, I.fz[2 * m], I.fz[2 * m + 1]);
      ax = fma2(fs, dx, ax);
      ay = fma2(fs, dy, ay);
      az = fma2(fs, dz, az);
    }
    float lo, hi;
    unpk2(ax, lo, hi); cx[k] = lo + hi;
    unpk2(ay, lo, hi); cy[k] = lo + hi;
    unpk2(az, lo, hi); cz[k] = lo + hi;
  }
}

// Two j-beads (registers jj0, jj0 + 1 of the XOR mapping) against this lane's 8 i-beads: 16 pairs.
// GAUSS: evaluate the Gaussian block terms (runtime c.gk says which); CHBM: 0 none, 1 every pair
// is same-chromosome, 2 compare per pair; SELF: mask i == j (diagonal stages).
// si4: this lane's i-beads in shared memory (type bits for the slow variants).
template <int EVP, int GK, int CHBM, bool SELF, bool CUT>
__device__ __forceinline__ void pairs16(const float4* __restrict__ sj, const int a, const int b, const int jj0,
                                        IBeads& I, float (&cx)[2], float (&cy)[2], float (&cz)[2],
                                        EAcc& E, const N3Consts& c, const int* __restrict__ si4,
                                        const int self_d) {
  constexpr bool GAUSS = GK != 0;
  constexpr bool kTypes = GAUSS || CHBM == 2;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int jl = (((jj0 + k) ^ a) << 2) | b;
    const float4 pj = sj[jl];
    const int tj = __float_as_int(pj.w);
    // a Gaussian term is non-zero only for equal labels / classes, so its prefactor can be looked
    // up from the j-bead once per 8 pairs
    float aj_scb = 0.0f, aj_cob = 0.0f;
    if (GK & 1) aj_scb = c.a_scb[tj & 7];
    if (GK & 2) aj_cob = c.a_cob[(tj >> 3) & 3];
    float ax = 0.0f, ay = 0.0f, az = 0.0f;
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      const float dx = I.x(ii) - pj.x, dy = I.y(ii) - pj.y, dz = I.z(ii) - pj.z;
      float r2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
      bool self = false;
      bool in = true;
      if (CUT) in = r2 < c.cut2;  // the oracle's pair_in_cut on the same FP32 r^2
      if (SELF) {
        self = (jl - ii) == self_d;
        r2 = self ? 1.0f : r2;
      }
      if (CUT) {
        if (SELF) in = in && !self;
        E.cnt += in ? 1.0f : 0.0f;
      }
      const float r = fast_sqrt(r2);
      float fs = 0.0f;
      if constexpr (EVP > 0) {
        const float q = fmaf(c.ev_rs, r, r2);
        const float wr = fast_rcp(q);  // w / r with w = 1 / (r + r_s)
        const float w = r * wr;
        float wp = powi<EVP>(w);
        if (SELF) wp = self ? 0.0f : wp;
        if (CUT) wp = in ? wp : 0.0f;
        E.ev += wp;
        fs = wp * wr;  // -(dE_ev/dr) / r in units of U
      }
      if (kTypes) {
        const int ti = si4[ii];
        const int xr = ti ^ tj;
        if (GAUSS) {
          float g = fast_ex2(r2 * c.g_c);
          if (SELF) g = self ? 0.0f : g;
          if (CUT) g = in ? g : 0.0f;
          if (GK & 1) {
            const float t = ((xr & 0x7) == 0) ? aj_scb * g : 0.0f;
            E.scb += t;
            fs -= t;
          }
          if (GK & 2) {
            const float t = ((xr & 0x18) == 0) ? aj_cob * g : 0.0f;
            E.cob += t;
            fs -= t;
          }
        }
        if (CHBM == 2) {
          // E = dE (kC r^4 - r^3 + r^2);  -(dE/dr)/r = -dE (4 kC r^2 - 3 r + 2)
          bool same = (xr & 0xFFFF00) == 0;
          if (SELF) same = same && !self;
          const float e = r2 * fmaf(c.chb_kc, r2, 1.0f - r);
          const float bb = fmaf(-3.0f, r, fmaf(4.0f * c.chb_kc, r2, 2.0f));
          E.chb += same ? e : 0.0f;
          fs = fmaf(-c.chb_c, same ? bb : 0.0f, fs);
        }
      }
      if (CHBM == 1) {
        E.chb = fmaf(r2, fmaf(c.chb_kc, r2, 1.0f - r), E.chb);
        fs = fmaf(-c.chb_c, fmaf(-3.0f, r, fmaf(4.0f * c.chb_kc, r2, 2.0f)), fs);
      }
      I.fx[ii] = fmaf(fs, dx, I.fx[ii]);
      I.fy[ii] = fmaf(fs, dy, I.fy[ii]);
      I.fz[ii] = fmaf(fs, dz, I.fz[ii]);
      ax = fmaf(fs, dx, ax);
      ay = fmaf(fs, dy, ay);
      az = fmaf(fs, dz, az);
    }
    cx[k] = ax; cy[k] = ay; cz[k] = az;
  }
}

// Generic variant (EVP < 0): any functional form of any pair term (model.py:205-211, 258-288, 338-378,
// 424-445) and non-integer EV powers, through pairmath::pair_generic — FP32 deltas, FP64 after that — on
// the Newton-3 machinery: every unordered pair once instead of the gather kernel's twice.  The slow path:
// rolled loops, the i-beads indexed at run time (local memory), forces in kJ/mol/nm (U = 1).
// "Particle 1" of the reference's s1-only Yukawa COB (model.py:262-266) is the lower index [OpenMM]: the
// i side everywhere except in the diagonal stages, where ordered pairs are compared by index.
template <bool SELF>
__device__ __forceinline__ void pairs16_generic(const float4* __restrict__ sj, const int a, const int b, const int jj0,
                                                IBeads& I, float (&cx)[2], float (&cy)[2], float (&cz)[2], EAcc& E,
                                                const PairParams& pp, const int* __restrict__ si4, const int self_d) {
#pragma unroll 1
  for (int k = 0; k < 2; ++k) {
    const int jl = (((jj0 + k) ^ a) << 2) | b;
    const float4 pj = sj[jl];
    float ax = 0.0f, ay = 0.0f, az = 0.0f;
#pragma unroll 1
    for (int ii = 0; ii < 8; ++ii) {
      pairmath::IBead ib;
      ib.x = I.x(ii); ib.y = I.y(ii); ib.z = I.z(ii);
      ib.w = si4[ii];
      ib.a_scb = ib.a_cob = 0.0f;
      bool live = true, i_lower = true;
      if (SELF) {
        live = (jl - ii) != self_d;
        i_lower = (jl - ii) > self_d;  // j - i > 0
      }
      double px = 0.0, py = 0.0, pz = 0.0;
      pairmath::pair_generic(pj, ib, (ib.w & 7) - 2, i_lower, pp, live, px, py, pz, E.gen);
      const float fx = (float)px, fy = (float)py, fz = (float)pz;
      I.fx[ii] += fx; I.fy[ii] += fy; I.fz[ii] += fz;
      ax += fx; ay += fy; az += fz;
    }
    cx[k] = ax; cy[k] = ay; cz[k] = az;
  }
}

#define N3_SHFL3(dst, src, m)                                  \
  dst##x = __shfl_xor_sync(0xffffffffu, src##x, m);            \
  dst##y = __shfl_xor_sync(0xffffffffu, src##y, m);            \
  dst##z = __shfl_xor_sync(0xffffffffu, src##z, m);

// One step: this lane's 8 i-beads against its 8 j-beads of the tile at sj[0..31], as a ROLLED loop
// over four groups of two j-registers (the body is 16 pairs, ~5 KB of SASS, so that it stays in the
// instruction cache), with the reduce-scatter over the 8 a-lanes folded in between the groups.
// Register jj of lane (a, b) holds j-bead 4 (jj ^ a) + b, so lanes L and L ^ 8 (a bit 1) hold the
// same beads in registers r and r ^ 2, L and L ^ 16 in r and r ^ 4, L and L ^ 4 in r and r ^ 1:
// partners exchange matching beads without selects.  12 + 6 + 3 SHFL.BFLY/FADD pairs leave lane l
// with the warp's total for j-bead l of the tile (returned in out[3]).  WANT_J false (diagonal
// stages, ordered pairs): the j side is dropped.
template <int EVP, int GK, int CHBM, bool SELF, bool WANT_J, bool CUT>
__device__ __forceinline__ void step64(const float4* __restrict__ sj, const JDup sjd, const int a,
                                       const int b, IBeads& I, float (&out)[3], EAcc& E, const N3Consts& c,
                                       const int* __restrict__ si4, const int self_d, const PairParams* pp = nullptr) {
  constexpr bool kPacked = N3_USE_F32X2 && GK == 0 && !SELF && (EVP > 0 ? CHBM <= 1 : CHBM == 1);
  constexpr bool kPackedNear = N3_USE_F32X2 && N3_PACKED_NEAR && GK != 0 && !SELF && EVP > 0 && CHBM <= 1;
  float s0x = 0.f, s0y = 0.f, s0z = 0.f, s1x = 0.f, s1y = 0.f, s1z = 0.f;  // saved group (g even)
  float p0x = 0.f, p0y = 0.f, p0z = 0.f, p1x = 0.f, p1y = 0.f, p1z = 0.f;  // registers 0,1 after level "2"
#pragma unroll kGroupUnroll
  for (int g = 0; g < 4; ++g) {
    float cx[2], cy[2], cz[2];
    if constexpr (EVP < 0) pairs16_generic<SELF>(sj, a, b, 2 * g, I, cx, cy, cz, E, *pp, si4, self_d);
    else if constexpr (kPacked) pairs16_packed<EVP, CHBM, CUT>(sjd, a, b, 2 * g, I, cx, cy, cz, E, c);
    else if constexpr (kPackedNear) pairs16_packed_near<EVP, GK, CHBM, CUT>(sj, sjd, a, b, 2 * g, I, cx, cy, cz, E, c, si4);
    else pairs16<EVP, GK, CHBM, SELF, CUT>(sj, a, b, 2 * g, I, cx, cy, cz, E, c, si4, self_d);
    if (!WANT_J) continue;
    if ((g & 1) == 0) {
      s0x = cx[0]; s0y = cy[0]; s0z = cz[0];
      s1x = cx[1]; s1y = cy[1]; s1z = cz[1];
    } else {
      float t0x, t0y, t0z, t1x, t1y, t1z;
      const float c0x = cx[0], c0y = cy[0], c0z = cz[0], c1x = cx[1], c1y = cy[1], c1z = cz[1];
      N3_SHFL3(t0, c0, 8)
      N3_SHFL3(t1, c1, 8)
      t0x += s0x; t0y += s0y; t0z += s0z;
      t1x += s1x; t1y += s1y; t1z += s1z;
      if (g == 1) {
        p0x = t0x; p0y = t0y; p0z = t0z;
        p1x = t1x; p1y = t1y; p1z = t1z;
      } else {
        float u0x, u0y, u0z, u1x, u1y, u1z;
        N3_SHFL3(u0, t0, 16)
        N3_SHFL3(u1, t1, 16)
        p0x += u0x; p0y += u0y; p0z += u0z;
        p1x += u1x; p1y += u1y; p1z += u1z;
      }
    }
  }
  if (WANT_J) {
    float vx, vy, vz;
    N3_SHFL3(v, p1, 4)
    out[0] = p0x + vx; out[1] = p0y + vy; out[2] = p0z + vz;
  }
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void red_fixed(unsigned long long* p, float v, double fscale, double& poison) {
  if (!(fabsf(v) <= 3.0e38f)) poison = __longlong_as_double(0x7ff8000000000000LL);  // NaN/Inf force
  const long long q = __double2ll_rn((double)v * fscale);
  atomicAdd(p, (unsigned long long)q);
}

__device__ __forceinline__ float box_dist2(const TileInfo& p, const TileInfo& q) {
  const float ddx = fmaxf(0.0f, fmaxf(p.lox - q.hix, q.lox - p.hix));
  const float ddy = fmaxf(0.0f, fmaxf(p.loy - q.hiy, q.loy - p.hiy));
  const float ddz = fmaxf(0.0f, fmaxf(p.loz - q.hiz, q.loz - p.hiz));
  return fmaf(ddz, ddz, fmaf(ddy, ddy, ddx * ddx));
}

// CUT (cut-off mode, mmm_cutoff.cu): the bead arrays are Morton sorted; stages whose box lies beyond
// the cut-off from the i-block are dropped by one ballot per item, tiles by the classification, pairs
// by the r^2 < rc^2 mask; forces are emitted through the sort permutation; the number of pairs inside
// the cut-off is reported in the item's CHB energy slot (a CUT pass never evaluates CHB).
template <int EVP, int GK, bool CHB, bool CUT>
__global__ void __launch_bounds__(N3_THREADS, N3_MIN_BLOCKS) k_pair_n3(const N3Args A) {
  __shared__ __align__(16) float4 s_j[2][N3_JB];
  __shared__ __align__(16) float4 s_jxy[2][N3_JB];
  __shared__ __align__(8) float2 s_jz[2][N3_JB];
  __shared__ __align__(16) TileInfo s_jt[2][N3_STEPS];
  __shared__ int s_it[N3_IB];  // type bits of the i-block (slow variants)
  __shared__ float s_acc[N3_WARPS][3][N3_JB];
  __shared__ __align__(16) double s_red[4][N3_WARPS];
  // CUT: per-warp i boxes for the stage cull live in s_red's bytes (used at the start of an item,
  // s_red at its end, barriers in between) — the static 48 KB are otherwise full
  TileInfo* const s_ibox = reinterpret_cast<TileInfo*>(&s_red[0][0]);
  static_assert(sizeof(TileInfo) * N3_WARPS <= sizeof(double) * 4 * N3_WARPS, "s_ibox must fit in s_red");
  __shared__ int s_item;
  __shared__ unsigned s_mask;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int a = lane >> 2, b = lane & 3;
  const N3Consts& c = A.c;
  if (A.skip && *A.skip) return;

#pragma unroll
  for (int w = 0; w < N3_WARPS; ++w)
#pragma unroll
    for (int d = 0; d < 3; ++d) s_acc[w][d][tid] = 0.0f;

  for (;;) {
    __syncthreads();  // protects s_item, s_i, s_j, s_red across items
    if (tid == 0) s_item = A.sys_counter ? atomicAdd_system(A.counter, 1) : atomicAdd(A.counter, 1);
    __syncthreads();
    const int item = A.item_first + s_item * A.item_stride;
    if (item >= A.n_items) break;
    const int2 it = A.items[item];
    const int iblk = it.x, js0 = it.y & 0xFFFFFF, cnt = it.y >> 24;
    const int64_t ibase = (int64_t)iblk * N3_IB;
    const int iw = warp * 64 + a * 8;  // first of this lane's i-beads within the block

    // the i-block: registers (positions) and shared memory (type bits for the slow variants)
    IBeads I;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int64_t i0 = ibase + iw + 2 * m;  // even: the 8-byte loads are aligned
      I.x2[m] = *reinterpret_cast<const u64*>(A.soa + i0);
      I.y2[m] = *reinterpret_cast<const u64*>(A.soa + A.npad + i0);
      I.z2[m] = *reinterpret_cast<const u64*>(A.soa + 2 * A.npad + i0);
      I.fx[2 * m] = I.fy[2 * m] = I.fz[2 * m] = 0.0f;
      I.fx[2 * m + 1] = I.fy[2 * m + 1] = I.fz[2 * m + 1] = 0.0f;
      if (m == b) {
        s_it[iw + 2 * m] = __float_as_int(A.pos4[i0].w);
        s_it[iw + 2 * m + 1] = __float_as_int(A.pos4[i0 + 1].w);
      }
    }
    // bounding box / chromosome range of the warp's 64 i-beads (two tiles); a padding-only tile
    // does not widen the box
    TileInfo ib = A.tiles[(ibase >> 5) + warp * 2];
    {
      const TileInfo ib2 = A.tiles[(ibase >> 5) + warp * 2 + 1];
      if (ib.cmin >= MMM_PAD_CHROM) {
        ib = ib2;
      } else if (ib2.cmin < MMM_PAD_CHROM) {
        ib.lox = fminf(ib.lox, ib2.lox); ib.loy = fminf(ib.loy, ib2.loy); ib.loz = fminf(ib.loz, ib2.loz);
        ib.hix = fmaxf(ib.hix, ib2.hix); ib.hiy = fmaxf(ib.hiy, ib2.hiy); ib.hiz = fmaxf(ib.hiz, ib2.hiz);
        ib.cmin = min(ib.cmin, ib2.cmin); ib.cmax = max(ib.cmax, ib2.cmax);
      }
    }
    const bool i_all_pad = ib.cmin >= MMM_PAD_CHROM;

    // which stages of the item are visited: all of them, or (CUT) those whose box is within the
    // cut-off of some warp's i-beads — thread t of warp 0 tests stage js0 + t, one ballot
    unsigned todo = cnt >= 32 ? 0xffffffffu : ((1u << cnt) - 1u);
    if (CUT) {
      if (lane == 0) s_ibox[warp] = ib;
      __syncthreads();
      if (warp == 0) {
        bool keep = false;
        if (lane < cnt) {
          const TileInfo sb = A.stage_boxes[js0 + lane];
          if (sb.cmin < MMM_PAD_CHROM) {
#pragma unroll
            for (int w = 0; w < N3_WARPS; ++w) {
              const TileInfo wb = s_ibox[w];
              keep = keep || (wb.cmin < MMM_PAD_CHROM && box_dist2(wb, sb) < c.cut2);
            }
          }
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_mask = m;
      }
      __syncthreads();
      todo = s_mask;
    }

    double de0 = 0.0, de1 = 0.0, de2 = 0.0, de3 = 0.0, poison = 0.0;

    if (todo != 0u) {
      int js = js0 + __ffs(todo) - 1;
      todo &= todo - 1u;
      // first stage
      {
        const float4 p0 = A.pos4[(int64_t)js * N3_JB + tid];
        s_j[0][tid] = p0;
        s_jxy[0][tid] = make_float4(-p0.x, -p0.x, -p0.y, -p0.y);
        s_jz[0][tid] = make_float2(-p0.z, -p0.z);
      }
      if (tid < 2 * N3_STEPS)
        reinterpret_cast<float4*>(s_jt[0])[tid] = reinterpret_cast<const float4*>(A.tiles + (int64_t)js * N3_STEPS)[tid];
      __syncthreads();

      for (int buf = 0;; buf ^= 1) {
        const bool more = todo != 0u;
        const int js_next = more ? js0 + __ffs(todo) - 1 : 0;
        todo &= todo - 1u;
        float4 nxt = make_float4(0.f, 0.f, 0.f, 0.f), nxt_t = nxt;
        if (more) {
          nxt = A.pos4[(int64_t)js_next * N3_JB + tid];
          if (tid < 2 * N3_STEPS)
            nxt_t = reinterpret_cast<const float4*>(A.tiles + (int64_t)js_next * N3_STEPS)[tid];
        }
        const bool diag = (js >> 1) == iblk;
        // global j index minus global i index of (jl = 0, ii = 0): self pair when jl - ii == -that
        const int self_base = (int)(ibase + iw - (int64_t)js * N3_JB);
        EAcc E;
        E.ev = E.scb = E.cob = E.chb = E.cnt = 0.0f;
        E.ev2 = E.chb2 = E.cnt2 = E.scb2 = E.cob2 = pk2(0.0f, 0.0f);
        E.gen[0] = E.gen[1] = E.gen[2] = E.gen[3] = 0.0;

        if (!i_all_pad) {
          // Classify the stage's 8 tiles at once: lane s < 8 classifies tile s against this warp's
          // i-beads, the steps fetch their class with one shuffle.  Class: -1 nothing to do;
          // bits 0-1 CHB mode (0 none, 1 every pair same-chromosome, 2 compare per pair); bit 2
          // within the Gaussian range.
          int my_class = -1;
          if (lane < N3_STEPS) {
            const TileInfo jt = s_jt[buf][lane];
            if (jt.cmin < MMM_PAD_CHROM) {  // not padding only
              int chb_mode = 0;
              if (CHB) {
                const bool overlap = !(ib.cmax < jt.cmin || jt.cmax < ib.cmin);
                const bool uniform = (ib.cmin == ib.cmax) && (jt.cmin == jt.cmax);
                chb_mode = overlap ? (uniform ? 1 : 2) : 0;
              }
              bool near = false;
              float d2 = 0.0f;
              if (GK != 0 || CUT) d2 = box_dist2(ib, jt);
              if (GK != 0) near = d2 < c.rg2;
              my_class = chb_mode | (near ? 4 : 0);
              if (EVP == 0 && chb_mode == 0) my_class = -1;  // CHB-only pass: nothing to do for this tile pair
              if (CUT && !(d2 < c.cut2)) my_class = -1;      // every pair of the tile pair is beyond the cut-off
            }
          }
          for (int step = 0; step < N3_STEPS; ++step) {
            const int cls = __shfl_sync(0xffffffffu, my_class, step);
            if (cls < 0) continue;
            const float4* sj = s_j[buf] + step * MMM_TILE;
            const JDup sjd = {s_jxy[buf] + step * MMM_TILE, s_jz[buf] + step * MMM_TILE};
            float fj[3];
            if (diag) {
              const int self_d = self_base - step * MMM_TILE;
              step64<EVP, GK, CHB ? 2 : 0, true, false, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, self_d, &A.pp);
              continue;  // ordered pairs: the j side is somebody's i side in this same stage pair
            }
            const int chb_mode = cls & 3;
            if (cls & 4) {
              if (!CHB || chb_mode == 0) step64<EVP, GK, 0, false, true, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, 0, &A.pp);
              else if (chb_mode == 1) step64<EVP, GK, CHB ? 1 : 0, false, true, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, 0, &A.pp);
              else step64<EVP, GK, CHB ? 2 : 0, false, true, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, 0, &A.pp);
            } else if (!CHB || chb_mode == 0) {
              step64<EVP, 0, 0, false, true, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, 0, &A.pp);
            } else if (chb_mode == 1) {
              step64<EVP, 0, CHB ? 1 : 0, false, true, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, 0, &A.pp);
            } else {
              step64<EVP, 0, CHB ? 2 : 0, false, true, CUT>(sj, sjd, a, b, I, fj, E, c, s_it + iw, 0, &A.pp);
            }
            // lane (a, b) now holds j-bead 4 a + b = lane of this step; force on j is -sum.  A warp writes a
            // column at most once per stage and the emission below leaves it zero: a plain store, no read
            const int col = step * MMM_TILE + lane;
            s_acc[warp][0][col] = -fj[0];
            s_acc[warp][1][col] = -fj[1];
            s_acc[warp][2][col] = -fj[2];
          }
        }
        {
          float lo, hi;
          unpk2(E.ev2, lo, hi); E.ev += lo + hi;
          unpk2(E.chb2, lo, hi); E.chb += lo + hi;
          if (GK & 1) { unpk2(E.scb2, lo, hi); E.scb += lo + hi; }
          if (GK & 2) { unpk2(E.cob2, lo, hi); E.cob += lo + hi; }
          if (CUT) { unpk2(E.cnt2, lo, hi); E.chb = E.cnt + lo + hi; }
        }
        const double wgt = diag ? 0.5 : 1.0;
        if constexpr (EVP < 0) {
          de0 += wgt * E.gen[0]; de1 += wgt * E.gen[1]; de2 += wgt * E.gen[2]; de3 += wgt * E.gen[3];
        } else {
          de0 += wgt * (double)E.ev;
          de1 += wgt * (double)E.cob;
          de2 += wgt * (double)E.scb;
          de3 += wgt * (double)E.chb;
        }

        if (more) {
          s_j[buf ^ 1][tid] = nxt;
          s_jxy[buf ^ 1][tid] = make_float4(-nxt.x, -nxt.x, -nxt.y, -nxt.y);
          s_jz[buf ^ 1][tid] = make_float2(-nxt.z, -nxt.z);
          if (tid < 2 * N3_STEPS) reinterpret_cast<float4*>(s_jt[buf ^ 1])[tid] = nxt_t;
        }
        __syncthreads();
        if (!diag) {
          // j-side emission: thread t owns j-bead t of the stage
          float sx = 0.0f, sy = 0.0f, sz = 0.0f;
#pragma unroll
          for (int w = 0; w < N3_WARPS; ++w) {
            sx += s_acc[w][0][tid]; sy += s_acc[w][1][tid]; sz += s_acc[w][2][tid];
            s_acc[w][0][tid] = 0.0f; s_acc[w][1][tid] = 0.0f; s_acc[w][2][tid] = 0.0f;
          }
          if (sx != 0.0f || sy != 0.0f || sz != 0.0f) {
            int64_t j = (int64_t)js * N3_JB + tid;
            if (CUT) j = A.perm[j];
            red_fixed(A.facc + j, sx, A.fscale, poison);
            red_fixed(A.facc + A.npad + j, sy, A.fscale, poison);
            red_fixed(A.facc + 2 * A.npad + j, sz, A.fscale, poison);
          }
        }
        __syncthreads();
        if (!more) break;
        js = js_next;
      }
    }

    // i-side emission: butterfly over the 4 b-lanes, then lane b emits beads 2b and 2b + 1
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      I.fx[ii] += __shfl_xor_sync(0xffffffffu, I.fx[ii], 1);
      I.fy[ii] += __shfl_xor_sync(0xffffffffu, I.fy[ii], 1);
      I.fz[ii] += __shfl_xor_sync(0xffffffffu, I.fz[ii], 1);
      I.fx[ii] += __shfl_xor_sync(0xffffffffu, I.fx[ii], 2);
      I.fy[ii] += __shfl_xor_sync(0xffffffffu, I.fy[ii], 2);
      I.fz[ii] += __shfl_xor_sync(0xffffffffu, I.fz[ii], 2);
    }
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      if ((ii >> 1) == b) {
        int64_t i = ibase + iw + ii;
        if (CUT) {
          if (I.fx[ii] == 0.0f && I.fy[ii] == 0.0f && I.fz[ii] == 0.0f) continue;  // most i-beads of a culled item
          i = A.perm[i];
        }
        red_fixed(A.facc + i, I.fx[ii], A.fscale, poison);
        red_fixed(A.facc + A.npad + i, I.fy[ii], A.fscale, poison);
        red_fixed(A.facc + 2 * A.npad + i, I.fz[ii], A.fscale, poison);
      }
    }

    // energies of the item, fixed order
    de0 = de0 * A.e_ev + poison;
    de1 *= A.e_gauss;
    de2 *= A.e_gauss;
    if (!CUT) de3 *= A.e_chb;  // CUT: the slot carries the number of pairs inside the cut-off
    de0 = warp_sum_d(de0); de1 = warp_sum_d(de1); de2 = warp_sum_d(de2); de3 = warp_sum_d(de3);
    if (lane == 0) { s_red[0][warp] = de0; s_red[1][warp] = de1; s_red[2][warp] = de2; s_red[3][warp] = de3; }
    __syncthreads();
    if (tid < 4) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < N3_WARPS; ++w) s += s_red[tid][w];
      if (CUT && tid == 3) {
        A.npairs[item] = s;
        s = 0.0;
      }
      A.epair[(size_t)item * 4 + tid] = s;
    }
  }
}

// ---- cut-off mode, one warp per work item -------------------------------------------------
// In cut-off mode the surviving work is sparse: of the (512-bead i-block) x (256-bead stage) rectangles
// the CTA-level kernel above visits, only a fraction of the (warp, tile) combinations lies within the
// cut-off, and the other warps wait at the stage barriers.  Here every warp works alone: an item is
// (64 consecutive sorted i-beads) x (a chunk of 32 stages); lane t tests stage t of the chunk against
// the warp's i-box (one ballot), lanes 0-7 the tiles of a surviving stage (one ballot), and each
// surviving 32-bead tile is staged in the warp's own slice of shared memory and evaluated by the same
// step64 bodies (r^2 < rc^2 mask).  No block barrier anywhere.  j-side forces leave per tile, i-side
// forces per item, both as 64-bit fixed point through the sort permutation; energies and the pair
// count leave as 64-bit fixed point too (2^-20 kJ/mol), so that every sum is associative and the
// result does not depend on which warp ran which item.
// (Measured and dropped, profiles/r02_cutoff_mode.md: testing all 64 tiles of a chunk with two ballots and
// fetching the next surviving tile while the current one is evaluated — 0.811 against 0.805 ms, the pass is
// bound by the arithmetic of its candidate pairs, not by these round trips; 128-thread CTAs at 96 registers
// (5 per SM instead of 2 x 256 threads at 128): 0.871 ms.)
constexpr double CW_EFIXED = 1048576.0;  // 2^20
constexpr int CW_CHUNK = 8;              // stages per item: fine enough that the items near the diagonal (where the work is) spread over all warps

struct CutWArgs {
  const float4* pos4;
  const float* soa;
  const TileInfo* tiles;
  const TileInfo* stage_boxes;
  const int* perm;
  unsigned long long* facc;
  long long* eacc;   // [4] EV, COB, SCB energies and the pair count, fixed point
  const int2* items; // (i-group, first stage of the chunk)
  int* counter;
  const int* skip;
  int64_t npad;
  int nstages, item_begin, item_end;
  double fscale, e_ev, e_gauss;
  N3Consts c;
};

template <int EVP, int GK>
__global__ void __launch_bounds__(N3_THREADS, N3_MIN_BLOCKS) k_pair_cut_warp(const CutWArgs A) {
  __shared__ __align__(16) float4 s_j[N3_WARPS][MMM_TILE];
  __shared__ __align__(16) float4 s_jxy[N3_WARPS][MMM_TILE];
  __shared__ __align__(8) float2 s_jz[N3_WARPS][MMM_TILE];
  __shared__ int s_it[N3_WARPS][64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int a = lane >> 2, b = lane & 3;
  const N3Consts& c = A.c;
  if (A.skip && *A.skip) return;

  for (;;) {
    int item = 0;
    if (lane == 0) item = A.item_begin + atomicAdd(A.counter, 1);
    item = __shfl_sync(0xffffffffu, item, 0);
    if (item >= A.item_end) break;
    const int2 it = A.items[item];
    const int g = it.x, s0 = it.y, s1 = min(s0 + CW_CHUNK, A.nstages);
    const int64_t ibase = (int64_t)g * 64;
    IBeads I;
    __syncwarp();  // the previous item's readers of s_it are done
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int64_t i0 = ibase + 8 * a + 2 * m;
      I.x2[m] = *reinterpret_cast<const u64*>(A.soa + i0);
      I.y2[m] = *reinterpret_cast<const u64*>(A.soa + A.npad + i0);
      I.z2[m] = *reinterpret_cast<const u64*>(A.soa + 2 * A.npad + i0);
      I.fx[2 * m] = I.fy[2 * m] = I.fz[2 * m] = 0.0f;
      I.fx[2 * m + 1] = I.fy[2 * m + 1] = I.fz[2 * m + 1] = 0.0f;
      if (m == b) {
        s_it[warp][8 * a + 2 * m] = __float_as_int(A.pos4[i0].w);
        s_it[warp][8 * a + 2 * m + 1] = __float_as_int(A.pos4[i0 + 1].w);
      }
    }
    TileInfo ib = A.tiles[2 * g];
    {
      const TileInfo ib2 = A.tiles[2 * g + 1];
      if (ib.cmin >= MMM_PAD_CHROM) {
        ib = ib2;
      } else if (ib2.cmin < MMM_PAD_CHROM) {
        ib.lox = fminf(ib.lox, ib2.lox); ib.loy = fminf(ib.loy, ib2.loy); ib.loz = fminf(ib.loz, ib2.loz);
        ib.hix = fmaxf(ib.hix, ib2.hix); ib.hiy = fmaxf(ib.hiy, ib2.hiy); ib.hiz = fmaxf(ib.hiz, ib2.hiz);
      }
    }
    if (ib.cmin >= MMM_PAD_CHROM) continue;  // padding only
    __syncwarp();

    bool keep = false;
    if (s0 + lane < s1) {
      const TileInfo sb = A.stage_boxes[s0 + lane];
      keep = sb.cmin < MMM_PAD_CHROM && box_dist2(ib, sb) < c.cut2;
    }
    unsigned smask = __ballot_sync(0xffffffffu, keep);
    double de0 = 0.0, de1 = 0.0, de2 = 0.0, de3 = 0.0, poison = 0.0;

    while (smask) {
      const int s = s0 + __ffs(smask) - 1;
      smask &= smask - 1u;
      int cls = -1;
      if (lane < N3_STEPS) {
        const int t = s * N3_STEPS + lane;
        if (t >= 2 * g) {  // tiles below the group's own belong to the groups before it
          const TileInfo jt = A.tiles[t];
          if (jt.cmin < MMM_PAD_CHROM) {
            const float d2 = box_dist2(ib, jt);
            if (d2 < c.cut2) cls = (GK != 0 && d2 < c.rg2) ? 4 : 0;
          }
        }
      }
      unsigned tmask = __ballot_sync(0xffffffffu, cls >= 0);
      const unsigned nearmask = __ballot_sync(0xffffffffu, cls == 4);
      while (tmask) {
        const int q = __ffs(tmask) - 1;
        tmask &= tmask - 1u;
        const int t = s * N3_STEPS + q;
        const float4 p = A.pos4[(int64_t)t * MMM_TILE + lane];
        s_j[warp][lane] = p;
        s_jxy[warp][lane] = make_float4(-p.x, -p.x, -p.y, -p.y);
        s_jz[warp][lane] = make_float2(-p.z, -p.z);
        __syncwarp();
        const JDup sjd = {s_jxy[warp], s_jz[warp]};
        EAcc E;
        E.ev = E.scb = E.cob = E.chb = E.cnt = 0.0f;
        E.ev2 = E.chb2 = E.cnt2 = E.scb2 = E.cob2 = pk2(0.0f, 0.0f);
        float fj[3] = {0.0f, 0.0f, 0.0f};
        double wgt = 1.0;
        if (t < 2 * g + 2) {  // the group's own two tiles: ordered pairs, i side only, self masked, halved
          const int self_d = (int)(ibase + 8 * a - (int64_t)t * MMM_TILE);
          step64<EVP, GK, 0, true, false, true>(s_j[warp], sjd, a, b, I, fj, E, c, s_it[warp] + 8 * a, self_d);
          wgt = 0.5;
        } else {
          if (GK != 0 && ((nearmask >> q) & 1u))
            step64<EVP, GK, 0, false, true, true>(s_j[warp], sjd, a, b, I, fj, E, c, s_it[warp] + 8 * a, 0);
          else
            step64<EVP, 0, 0, false, true, true>(s_j[warp], sjd, a, b, I, fj, E, c, s_it[warp] + 8 * a, 0);
          if (fj[0] != 0.0f || fj[1] != 0.0f || fj[2] != 0.0f) {  // lane l holds j-bead l of the tile
            const int64_t j = A.perm[(int64_t)t * MMM_TILE + lane];
            red_fixed(A.facc + j, -fj[0], A.fscale, poison);
            red_fixed(A.facc + A.npad + j, -fj[1], A.fscale, poison);
            red_fixed(A.facc + 2 * A.npad + j, -fj[2], A.fscale, poison);
          }
        }
        {
          float lo, hi;
          unpk2(E.ev2, lo, hi); E.ev += lo + hi;
          if (GK & 1) { unpk2(E.scb2, lo, hi); E.scb += lo + hi; }
          if (GK & 2) { unpk2(E.cob2, lo, hi); E.cob += lo + hi; }
          unpk2(E.cnt2, lo, hi); E.cnt += lo + hi;
        }
        de0 += wgt * (double)E.ev;
        de1 += wgt * (double)E.cob;
        de2 += wgt * (double)E.scb;
        de3 += wgt * (double)E.cnt;
        __syncwarp();  // everybody has read the tile before the next one overwrites it
      }
    }

    // i-side emission: butterfly over the 4 b-lanes, then lane b emits beads 2b and 2b + 1
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      I.fx[ii] += __shfl_xor_sync(0xffffffffu, I.fx[ii], 1);
      I.fy[ii] += __shfl_xor_sync(0xffffffffu, I.fy[ii], 1);
      I.fz[ii] += __shfl_xor_sync(0xffffffffu, I.fz[ii], 1);
      I.fx[ii] += __shfl_xor_sync(0xffffffffu, I.fx[ii], 2);
      I.fy[ii] += __shfl_xor_sync(0xffffffffu, I.fy[ii], 2);
      I.fz[ii] += __shfl_xor_sync(0xffffffffu, I.fz[ii], 2);
    }
#pragma unroll
    for (int ii = 0; ii < 8; ++ii) {
      if ((ii >> 1) == b && (I.fx[ii] != 0.0f || I.fy[ii] != 0.0f || I.fz[ii] != 0.0f)) {
        const int64_t i = A.perm[ibase + 8 * a + ii];
        red_fixed(A.facc + i, I.fx[ii], A.fscale, poison);
        red_fixed(A.facc + A.npad + i, I.fy[ii], A.fscale, poison);
        red_fixed(A.facc + 2 * A.npad + i, I.fz[ii], A.fscale, poison);
      }
    }
    // energies and pair count of the item: fixed point, so that the total is the same in any order
    de0 = warp_sum_d(de0 * A.e_ev + poison);
    de1 = warp_sum_d(de1 * A.e_gauss);
    de2 = warp_sum_d(de2 * A.e_gauss);
    de3 = warp_sum_d(de3);
    if (lane < 4) {
      const double v = lane == 0 ? de0 : (lane == 1 ? de1 : (lane == 2 ? de2 : de3));
      // a NaN / Inf force poisons the EV energy: keep it visible (the largest magnitude) instead of wrapping
      const long long fx = isfinite(v) ? __double2ll_rn(v * CW_EFIXED) : 0x7fffffffffffffffLL;
      if (fx != 0) atomicAdd(reinterpret_cast<unsigned long long*>(A.eacc + lane), (unsigned long long)fx);
    }
  }
}

// fixed-point totals -> the energy slot of this rank's cut-off pass, and the pair count; re-arm
__global__ void k_cut_finish(long long* __restrict__ eacc, double* __restrict__ epair_slot, double* __restrict__ npairs,
                             const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int t = threadIdx.x;
  if (t < 4) {
    const long long v = eacc[t];
    eacc[t] = 0;
    const double d = v == 0x7fffffffffffffffLL ? __longlong_as_double(0x7ff8000000000000LL) : (double)v / CW_EFIXED;
    if (t < 3) epair_slot[t] = d;
    else { npairs[0] = d; epair_slot[3] = 0.0; }
  }
}

template <int EVP, int GK>
int launch_cut_warp(mmm_system* h, const CutWArgs& A) {
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pair_cut_warp<EVP, GK>, N3_THREADS, 0);
  if (occ < 1) occ = 1;
  int grid = h->sm_count * occ;
  const int n_local = A.item_end - A.item_begin;
  if (grid * N3_WARPS > n_local) grid = (n_local + N3_WARPS - 1) / N3_WARPS;
  if (grid < 1) grid = 1;
  k_pair_cut_warp<EVP, GK><<<grid, N3_THREADS, 0, h->stream>>>(A);
  return 0;
}

template <int EVP>
int launch_cut_warp_gk(mmm_system* h, const CutWArgs& A, int gk) {
  switch (gk) {
    case 0: return launch_cut_warp<EVP, 0>(h, A);
    case 1: return launch_cut_warp<EVP, 1>(h, A);
    case 2: return launch_cut_warp<EVP, 2>(h, A);
    default: return launch_cut_warp<EVP, 3>(h, A);
  }
}

template <int EVP, int GK, bool CHB, bool CUT>
int launch_n3(mmm_system* h, const N3Args& A) {
  int occ = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_pair_n3<EVP, GK, CHB, CUT>, N3_THREADS, 0);
  if (occ < 1) occ = 1;
  int grid = h->sm_count * occ;
  const int n_local = (A.n_items - A.item_first + A.item_stride - 1) / A.item_stride;
  if (grid > n_local) grid = n_local > 0 ? n_local : 1;
  k_pair_n3<EVP, GK, CHB, CUT><<<grid, N3_THREADS, 0, h->stream>>>(A);
  return 0;
}

template <int EVP>
int launch_n3_evp(mmm_system* h, const N3Args& A, int gk, bool chb) {
  switch (gk * 2 + (chb ? 1 : 0)) {
    case 0: return launch_n3<EVP, 0, false, false>(h, A);
    case 1: return launch_n3<EVP, 0, true, false>(h, A);
    case 2: return launch_n3<EVP, 1, false, false>(h, A);
    case 3: return launch_n3<EVP, 1, true, false>(h, A);
    case 4: return launch_n3<EVP, 2, false, false>(h, A);
    case 5: return launch_n3<EVP, 2, true, false>(h, A);
    case 6: return launch_n3<EVP, 3, false, false>(h, A);
    default: return launch_n3<EVP, 3, true, false>(h, A);
  }
}

template <int EVP>
int launch_n3_cut(mmm_system* h, const N3Args& A, int gk) {
  switch (gk) {
    case 0: return launch_n3<EVP, 0, false, true>(h, A);
    case 1: return launch_n3<EVP, 1, false, true>(h, A);
    case 2: return launch_n3<EVP, 2, false, true>(h, A);
    default: return launch_n3<EVP, 3, false, true>(h, A);
  }
}

// constants shared by the exact and the cut-off launch
void fill_consts(const PairParams& p, bool chb_only, bool with_chb, N3Args& A) {
  // U = p eps sigma^p in double, from the float parameters the gather kernel uses too (1 in the
  // CHB-only pass, where EV is not evaluated)
  const double U = chb_only ? 1.0 : (double)p.ev_power * (double)p.ev_eps * pow((double)p.ev_sigma, (double)p.ev_power);
  A.pp = p;
  A.fscale = U * N3_FIXED;
  A.e_ev = chb_only ? 0.0 : (double)p.ev_eps * pow((double)p.ev_sigma, (double)p.ev_power);
  N3Consts& c = A.c;
  c.ev_rs = p.ev_rs;
  c.g_c = p.g_c;
  c.rg2 = p.rg2;
  c.chb_kc = p.chb_kc;
  c.chb_c = (with_chb && p.chb_form >= 0) ? (float)((double)p.chb_de / U) : 0.0f;
  c.gk = chb_only ? 0 : ((p.scb_form >= 0 ? 1 : 0) | (p.cob_form >= 0 ? 2 : 0));
  c.cut2 = p.cutoff2;
  const double rc = p.scb_form >= 0 ? p.scb_rc : p.cob_rc;
  const double inv = rc > 0.0 ? 1.0 / (rc * rc * U) : 0.0;
  // s + 2 = 0..4 <-> s = -2..2 ; scb_e = {Ea1 (s=2), Ea2 (s=1), Eb1 (s=-1), Eb2 (s=-2)}
  c.a_scb[0] = (float)(p.scb_e[3] * inv);
  c.a_scb[1] = (float)(p.scb_e[2] * inv);
  c.a_scb[2] = 0.0f;
  c.a_scb[3] = (float)(p.scb_e[1] * inv);
  c.a_scb[4] = (float)(p.scb_e[0] * inv);
  c.a_cob[0] = 0.0f;
  c.a_cob[1] = (float)(p.cob_ea * inv);
  c.a_cob[2] = (float)(p.cob_eb * inv);
  c.a_cob[3] = 0.0f;
  A.e_gauss = -(rc * rc) * U;
  A.e_chb = (double)p.chb_de;
}

}  // namespace

// Newton-3 path: the fast-path forms of mmm_pair.cu plus EV switched on (its prefactor is the
// unit of the accumulators).
bool mmm_pair_n3_eligible(const mmm_system* h) {
  if (!mmm_pair_fast_path(h)) return false;
  if (h->pp.ev_form != MMM_EV_POWERLAW) return false;
  if (!(h->pp.ev_eps > 0.0f) || !(h->pp.ev_sigma > 0.0f)) return false;
  return true;
}

// Every other combination of functional forms (and non-integer EV powers) takes the same machinery with
// the generic FP64 body (k_pair_n3<-1, 0, false, false>): exact mode only.
bool mmm_pair_n3_generic(const mmm_system* h) {
  const PairParams& p = h->pp;
  const bool any = p.ev_form >= 0 || p.cob_form >= 0 || p.scb_form >= 0 || p.chb_form >= 0;
  return any && !mmm_pair_fast_path(h);
}

// Work items: for every i-block, runs of at most cj j-stages starting at the diagonal.
// chb_only (cut-off mode's exact CHB pass): only stages whose chromosome range overlaps the
// i-block's are visited; chromosome ids are static, so the list is built once on the host.
int mmm_n3_build_items(mmm_system* h, std::vector<int2>& items, bool chb_only) {
  const int64_t nib = h->npad / N3_IB, njs = h->npad / N3_JB;
  // chromosome range of every j-stage (real beads only)
  std::vector<int> lo((size_t)njs, 0x7fffffff), hi((size_t)njs, -1);
  if (chb_only) {
    for (int64_t i = 0; i < h->n; ++i) {
      const int c = h->h_chrom.empty() ? 0 : h->h_chrom[(size_t)i];
      const int64_t s = i / N3_JB;
      lo[s] = std::min(lo[s], c);
      hi[s] = std::max(hi[s], c);
    }
  }
  auto wanted = [&](int64_t ib, int64_t js) {
    if (!chb_only) return true;
    if ((js >> 1) == ib) return hi[js] >= 0;  // diagonal stages (unless padding only)
    const int ilo = std::min(lo[2 * ib], lo[2 * ib + 1]), ihi = std::max(hi[2 * ib], hi[2 * ib + 1]);
    return hi[js] >= 0 && ihi >= 0 && !(ihi < lo[js] || hi[js] < ilo);
  };
  int64_t pairs = 0;
  for (int64_t i = 0; i < nib; ++i)
    for (int64_t js = 2 * i; js < njs; ++js) pairs += wanted(i, js) ? 1 : 0;
  const int64_t target_items = (int64_t)h->sm_count * 2 * 48;
  int64_t cj = pairs / target_items;
  cj = cj < 1 ? 1 : (cj > 16 ? 16 : cj);
  // (Measured and dropped: half-stage items for small systems — S1 has 420 stage pairs for 296 resident
  // CTAs — cost 108.7 against 101 us per evaluation: the per-item i-side emission and energy reduction
  // outweigh the shorter last wave.)
  items.clear();
  for (int64_t i = 0; i < nib; ++i) {
    int64_t js = 2 * i;
    while (js < njs) {
      if (!wanted(i, js)) { ++js; continue; }
      int64_t cnt = 1;
      while (cnt < cj && js + cnt < njs && wanted(i, js + cnt)) ++cnt;
      items.push_back(make_int2((int)i, (int)(js | (cnt << 24))));
      js += cnt;
    }
  }
  if (items.empty()) items.push_back(make_int2(0, 0));  // zero stages: the kernel writes a zero energy slot
  return MMM_OK;
}

int mmm_launch_pair_n3(mmm_system* h, const int* d_skip, bool chb_only) {
  const PairParams& p = h->pp;
  N3Args A;
  A.pos4 = h->d_pos4;
  A.soa = h->d_soa;
  A.tiles = h->d_tiles;
  A.facc = h->d_facc;
  A.epair = h->d_epair;
  A.items = h->d_items;
  A.counter = h->d_counter;
  A.skip = d_skip;
  A.npad = h->npad;
  A.n_items = h->n3_items;
  A.stage_boxes = nullptr;
  A.perm = nullptr;
  A.npairs = nullptr;
  A.sys_counter = 0;
  fill_consts(p, chb_only, true, A);
  const bool generic = !chb_only && !mmm_pair_n3_eligible(h);
  if (generic) {  // forces and energies leave the generic body with every prefactor applied
    A.fscale = N3_FIXED;
    A.e_ev = A.e_gauss = A.e_chb = 1.0;
  }
  const N3Consts& c = A.c;

  const bool timed = !chb_only;  // the CHB-only pass is timed with the cell-list pass
  const bool collect = timed && h->ev_cursor >= 0 && (size_t)(2 * h->ev_cursor + 1) < h->ev_pool.size();
  cudaEvent_t ea = collect ? h->ev_pool[2 * h->ev_cursor] : h->ev_a;
  cudaEvent_t eb = collect ? h->ev_pool[2 * h->ev_cursor + 1] : h->ev_b;
  if (collect) h->ev_cursor++;
  if (timed && !h->capturing) MMM_CUDA(h, cudaEventRecord(ea, h->stream));
  const bool chb = p.chb_form >= 0;
  // one launch for this rank's share of the items; in emulation every rank's share in turn
  const int r0 = h->dist_emulate ? 0 : h->dist_rank, r1 = h->dist_emulate ? h->dist_world : h->dist_rank + 1;
  for (int r = r0; r < r1; ++r) {
    A.item_first = r;
    A.item_stride = h->dist_world;
    if (h->d_gqueue && !h->dist_emulate && !chb_only) {
      // (exact mode only: there the all-reduce of every evaluation separates the two counters' uses)
      // one queue for all GPUs: every rank draws from counter (k & 1) of evaluation k; rank 0 re-arms
      // the other counter, which nobody touches until the all-reduce of this evaluation has passed
      const int which = (int)(h->gqueue_eval & 1);
      if (h->gqueue_owner) MMM_CUDA(h, cudaMemsetAsync(h->d_gqueue + (which ^ 1), 0, sizeof(int), h->stream));
      A.counter = h->d_gqueue + which;
      A.sys_counter = 1;
      A.item_first = 0;
      A.item_stride = 1;
      h->gqueue_eval++;
    } else {
      MMM_CUDA(h, cudaMemsetAsync(h->d_counter, 0, sizeof(int), h->stream));
    }
    if (chb_only) launch_n3<0, 0, true, false>(h, A);
    else if (generic) launch_n3<-1, 0, false, false>(h, A);
    else if (p.ev_power == 6.0f) launch_n3_evp<6>(h, A, c.gk, chb);
    else launch_n3_evp<3>(h, A, c.gk, chb);
    h->launches++;
  }
  MMM_CUDA(h, cudaGetLastError());
  if (timed && !h->capturing) MMM_CUDA(h, cudaEventRecord(eb, h->stream));
  return MMM_OK;
}

// Items of the one-warp-per-item cut-off kernel: (group of 64 sorted beads, chunk of 32 stages from the
// group's own stage on), groups in ascending order (the sharded mode cuts this list into slabs).
int mmm_cut_warp_build_items(mmm_system* h, std::vector<int2>& items) {
  const int ngroups = (int)((h->n + 63) / 64), nstages = (int)(h->npad / N3_JB);
  items.clear();
  for (int g = 0; g < ngroups; ++g)
    for (int s = g / 4; s < nstages; s += CW_CHUNK) items.push_back(make_int2(g, s));
  return MMM_OK;
}

int mmm_launch_pair_cut_warp(mmm_system* h, const int* d_skip) {
  const PairParams& p = h->pp;
  N3Args tmp;
  fill_consts(p, false, false, tmp);
  CutWArgs A;
  A.pos4 = h->d_pos4_sorted;
  A.soa = h->d_soa_sorted;
  A.tiles = h->d_tiles_sorted;
  A.stage_boxes = h->d_stage_boxes;
  A.perm = h->d_order;
  A.facc = h->d_facc;
  A.eacc = reinterpret_cast<long long*>(h->d_cut_eacc.get());
  A.items = h->d_items_cut;
  A.counter = h->d_counter + 1;
  A.skip = d_skip;
  A.npad = h->npad;
  A.nstages = (int)(h->npad / N3_JB);
  A.fscale = tmp.fscale;
  A.e_ev = tmp.e_ev;
  A.e_gauss = tmp.e_gauss;
  A.c = tmp.c;
  // Several GPUs: contiguous slabs of 64-bead groups of the Morton order, one slab per rank
  const int ngroups = (int)((h->n + 63) / 64);
  const int r0 = h->dist_emulate ? 0 : h->dist_rank, r1 = h->dist_emulate ? h->dist_world : h->dist_rank + 1;
  for (int r = r0; r < r1; ++r) {
    const int g0 = (int)((int64_t)ngroups * r / h->dist_world), g1 = (int)((int64_t)ngroups * (r + 1) / h->dist_world);
    const auto& ig = h->h_cut_iblk;  // group of every item
    A.item_begin = (int)(std::lower_bound(ig.begin(), ig.end(), g0) - ig.begin());
    A.item_end = (int)(std::lower_bound(ig.begin(), ig.end(), g1) - ig.begin());
    MMM_CUDA(h, cudaMemsetAsync(h->d_counter + 1, 0, sizeof(int), h->stream));
    if (A.item_end > A.item_begin) {
      if (p.ev_power == 6.0f) launch_cut_warp_gk<6>(h, A, A.c.gk);
      else launch_cut_warp_gk<3>(h, A, A.c.gk);
      h->launches++;
    }
    // this rank's slot (one writer per slot: the sharded sum stays exact)
    k_cut_finish<<<1, 32, 0, h->stream>>>(A.eacc, h->d_epair + 4 * ((size_t)h->cells_item0 + r), h->d_cut_npairs + r, d_skip);
    h->launches++;
  }
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}

// Cut-off mode (mmm_cutoff.cu): EV / COB / SCB truncated at rc over the Morton-sorted arrays; the
// item table is the all-pairs one, the kernel culls.  Energy slots follow those of the CHB-only pass.
int mmm_launch_pair_n3_cut(mmm_system* h, const int* d_skip) {
  if (h->cut_warp) return mmm_launch_pair_cut_warp(h, d_skip);
  const PairParams& p = h->pp;
  N3Args A;
  A.pos4 = h->d_pos4_sorted;
  A.soa = h->d_soa_sorted;
  A.tiles = h->d_tiles_sorted;
  A.facc = h->d_facc;
  A.epair = h->d_epair + 4 * (size_t)h->cells_item0;
  A.items = h->d_items_cut;
  A.counter = h->d_counter + 1;
  A.skip = d_skip;
  A.npad = h->npad;
  A.n_items = h->n_items_cut;
  A.item_first = 0;
  A.item_stride = 1;
  A.stage_boxes = h->d_stage_boxes;
  A.perm = h->d_order;
  A.npairs = h->d_cut_npairs;
  A.sys_counter = 0;
  fill_consts(p, false, false, A);
  // Several GPUs: the sorted order is cut into contiguous slabs of i-blocks — spatial slabs along
  // the Morton curve — and rank r evaluates the items of its slab (pairs with the stages at or above
  // its diagonal, i.e. its own beads and the halo towards the higher slabs within the cut-off); the
  // j-side forces that land on other slabs' beads travel in the all-reduce of the force planes.
  const int nib = (int)(h->npad / N3_IB);
  const int r0 = h->dist_emulate ? 0 : h->dist_rank, r1 = h->dist_emulate ? h->dist_world : h->dist_rank + 1;
  for (int r = r0; r < r1; ++r) {
    const int b0 = (int)((int64_t)nib * r / h->dist_world), b1 = (int)((int64_t)nib * (r + 1) / h->dist_world);
    const auto& ib = h->h_cut_iblk;
    A.item_first = (int)(std::lower_bound(ib.begin(), ib.end(), b0) - ib.begin());
    A.n_items = (int)(std::lower_bound(ib.begin(), ib.end(), b1) - ib.begin());
    A.item_stride = 1;
    if (h->dist_world == 1) { A.item_first = 0; A.n_items = h->n_items_cut; }
    if (A.n_items <= A.item_first) continue;
    MMM_CUDA(h, cudaMemsetAsync(h->d_counter + 1, 0, sizeof(int), h->stream));
    if (p.ev_power == 6.0f) launch_n3_cut<6>(h, A, A.c.gk);
    else launch_n3_cut<3>(h, A, A.c.gk);
    h->launches++;
  }
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}
