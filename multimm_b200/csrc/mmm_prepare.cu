// mmm_prepare.cu — HBM-bound O(N) kernels that produce the pair kernel's inputs:
//   k_prepare : FP64 master positions -> centred FP32 float4 (xyz + type bits) and the
//               per-tile (32 beads) bounding boxes / chromosome ranges;
//   k_hilbert : on-device Hilbert start, replaces generate_hilbert_curve
//               (initial_structure_tools.py:157-166; HilbertCurve(8,3).points_from_distances).
#include "mmm_internal.cuh"

// ---------------------------------------------------------------------------------------
// prepare: one warp per tile. 24 B read + 28 B written per bead (+ 32 B per tile).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_prepare(const double* __restrict__ x,
                                                 const double* __restrict__ center,
                                                 const int* __restrict__ type, int64_t n,
                                                 int64_t npad, float4* __restrict__ pos4,
                                                 float* __restrict__ soa, TileInfo* __restrict__ tiles,
                                                 const int* __restrict__ skip) {
  if (skip && *skip) return;
  const int lane = threadIdx.x & 31;
  const int64_t tile = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t i = tile * MMM_TILE + lane;
  if (i >= npad) return;
  const bool real = i < n;
  float px, py, pz;
  const int ty = type[i];  // pads carry their own unique chromosome id (mmm_internal.cuh)
  if (real) {
    px = (float)(x[3 * i] - center[0]);
    py = (float)(x[3 * i + 1] - center[1]);
    pz = (float)(x[3 * i + 2] - center[2]);
  } else {
    px = py = pz = MMM_PAD_COORD + MMM_PAD_STEP * (float)(i - n);
  }
  pos4[i] = make_float4(px, py, pz, __int_as_float(ty));
  // plane copy x[], y[], z[]: the Newton-3 kernel loads its stationary beads as aligned register
  // pairs (LDG.64 of two consecutive beads) for the f32x2 path
  soa[i] = px;
  soa[npad + i] = py;
  soa[2 * npad + i] = pz;

  // bounding box over the real beads of the tile; an all-padding tile sits at the pad point
  const float big = 3.0e38f;
  float lox = real ? px : big, loy = real ? py : big, loz = real ? pz : big;
  float hix = real ? px : -big, hiy = real ? py : -big, hiz = real ? pz : -big;
  int ch = (ty >> 8) & 0xFFFF;
  int cmin = real ? ch : 0x7fffffff, cmax = real ? ch : -1;
  // bounding box and chromosome range cover the REAL beads only; a tile that mixes real and
  // padding beads gets cmax = a pad id, so it is never treated as single-chromosome
  const bool mixed = __any_sync(0xffffffffu, real) && !__all_sync(0xffffffffu, real);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lox = fminf(lox, __shfl_xor_sync(0xffffffffu, lox, o));
    loy = fminf(loy, __shfl_xor_sync(0xffffffffu, loy, o));
    loz = fminf(loz, __shfl_xor_sync(0xffffffffu, loz, o));
    hix = fmaxf(hix, __shfl_xor_sync(0xffffffffu, hix, o));
    hiy = fmaxf(hiy, __shfl_xor_sync(0xffffffffu, hiy, o));
    hiz = fmaxf(hiz, __shfl_xor_sync(0xffffffffu, hiz, o));
    cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
    cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
  }
  if (lane == 0) {
    TileInfo t;
    if (cmax < 0) {  // padding only
      t.lox = t.loy = t.loz = t.hix = t.hiy = t.hiz = MMM_PAD_COORD;
      t.cmin = MMM_PAD_CHROM;
      t.cmax = MMM_PAD_CHROM;
    } else {
      t.lox = lox; t.loy = loy; t.loz = loz;
      t.hix = hix; t.hiy = hiy; t.hiz = hiz;
      t.cmin = cmin; t.cmax = mixed ? MMM_PAD_CHROM : cmax;
    }
    tiles[tile] = t;
  }
}

int mmm_launch_prepare(mmm_system* h, const int* d_skip) {
  const int warps_per_block = 8;
  const int64_t blocks = (h->ntiles + warps_per_block - 1) / warps_per_block;
  k_prepare<<<(unsigned)blocks, 256, 0, h->stream>>>(h->d_x, h->d_center, h->d_type, h->n, h->npad,
                                                     h->d_pos4, h->d_soa, h->d_tiles, d_skip);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}

// ---------------------------------------------------------------------------------------
// Hilbert curve: Skilling's transpose -> axes decode, one thread per bead.
// The distance h is written as a 3p-bit string, MSB first; axis a takes bits a, a+3, ...
// (hilbertcurve 2.0.5 _hilbert_integer_to_transpose); then Gray decode and the
// "undo excess work" loop.  Integer-exact.  16 B (ijk) + 24 B (x) written per bead.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void hilbert_decode(uint64_t hdist, int p, uint32_t X[3]) {
  X[0] = X[1] = X[2] = 0;
  for (int b = 0; b < 3 * p; ++b) {
    const uint32_t bit = (uint32_t)((hdist >> (3 * p - 1 - b)) & 1ull);
    const int a = b % 3;
    X[a] = (X[a] << 1) | bit;
  }
  const uint32_t z = 2u << (p - 1);
  uint32_t t = X[2] >> 1;
  X[2] ^= X[1];
  X[1] ^= X[0];
  X[0] ^= t;
  for (uint32_t q = 2; q != z; q <<= 1) {
    const uint32_t pm = q - 1;
#pragma unroll
    for (int i = 2; i >= 0; --i) {
      if (X[i] & q) {
        X[0] ^= pm;
      } else {
        t = (X[0] ^ X[i]) & pm;
        X[0] ^= t;
        X[i] ^= t;
      }
    }
  }
}

__global__ void __launch_bounds__(256) k_hilbert(int64_t n, int p, double spacing,
                                                 double* __restrict__ x, int32_t* __restrict__ ijk) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t X[3];
  hilbert_decode((uint64_t)i, p, X);
  if (x) {
    x[3 * i] = spacing * (double)X[0];
    x[3 * i + 1] = spacing * (double)X[1];
    x[3 * i + 2] = spacing * (double)X[2];
  }
  if (ijk) {
    ijk[3 * i] = (int32_t)X[0];
    ijk[3 * i + 1] = (int32_t)X[1];
    ijk[3 * i + 2] = (int32_t)X[2];
  }
}

int mmm_launch_hilbert(mmm_system* h, int p, double spacing, int32_t* d_ijk) {
  const int64_t blocks = (h->n + 255) / 256;
  k_hilbert<<<(unsigned)blocks, 256, 0, h->stream>>>(h->n, p, spacing, d_ijk ? nullptr : h->d_x.get(), d_ijk);
  h->launches++;
  MMM_CUDA(h, cudaGetLastError());
  return MMM_OK;
}
