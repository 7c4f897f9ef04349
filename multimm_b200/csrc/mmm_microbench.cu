// mmm_microbench.cu — measures the two roofline denominators of the pair kernel on the GPU it
// runs on: FP32 FMA throughput (FFMA, 2 flop each) and MUFU throughput (rsqrt.approx).
// MEASURED_PEAKS.json only carries HBM bandwidth and bf16 tensor throughput, neither of which
// bounds an FP32/SFU kernel.
#include <stdio.h>

#include "mmm_internal.cuh"

namespace {

constexpr int kIters = 4096;

__global__ void __launch_bounds__(256) k_ffma_peak(float* out, float a, float b) {
  float v0 = threadIdx.x, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3, v4 = v0 + 4, v5 = v0 + 5, v6 = v0 + 6, v7 = v0 + 7;
#pragma unroll 1
  for (int it = 0; it < kIters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      v0 = fmaf(v0, a, b); v1 = fmaf(v1, a, b); v2 = fmaf(v2, a, b); v3 = fmaf(v3, a, b);
      v4 = fmaf(v4, a, b); v5 = fmaf(v5, a, b); v6 = fmaf(v6, a, b); v7 = fmaf(v7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = v0 + v1 + v2 + v3 + v4 + v5 + v6 + v7;
}

__global__ void __launch_bounds__(256) k_mufu_peak(float* out, float a) {
  float v0 = threadIdx.x + 1.0f, v1 = v0 + 1, v2 = v0 + 2, v3 = v0 + 3;
#pragma unroll 1
  for (int it = 0; it < kIters; ++it) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      asm volatile("rsqrt.approx.ftz.f32 %0, %0;" : "+f"(v0));
      asm volatile("rsqrt.approx.ftz.f32 %0, %0;" : "+f"(v1));
      asm volatile("rsqrt.approx.ftz.f32 %0, %0;" : "+f"(v2));
      asm volatile("rsqrt.approx.ftz.f32 %0, %0;" : "+f"(v3));
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = (v0 + v1 + v2 + v3) * a;
}

}  // namespace

extern "C" int mmm_measure_fp32_peak(int device, double* tflops_out, double* mufu_tops_out) {
  if (cudaSetDevice(device) != cudaSuccess) return MMM_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MMM_ERR_CUDA;
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  DevBuf<float> d_out;
  int rc = mmm_reserve(nullptr, d_out, (size_t)blocks * threads, "peak-rate output");
  if (rc) return rc;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  double best_f = 0.0, best_m = 0.0;
  for (int rep = 0; rep < 6; ++rep) {
    float ms = 0.f;
    cudaEventRecord(a);
    k_ffma_peak<<<blocks, threads>>>(d_out, 1.0000001f, 1e-9f);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    cudaEventElapsedTime(&ms, a, b);
    const double flop = 2.0 * 64.0 * kIters * (double)blocks * threads;
    if (rep > 0 && ms > 0.f) best_f = fmax(best_f, flop / (ms * 1e-3) / 1e12);
    cudaEventRecord(a);
    k_mufu_peak<<<blocks, threads>>>(d_out, 1.0f);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    cudaEventElapsedTime(&ms, a, b);
    const double ops = 16.0 * kIters * (double)blocks * threads;
    if (rep > 0 && ms > 0.f) best_m = fmax(best_m, ops / (ms * 1e-3) / 1e12);
  }
  cudaError_t e = cudaGetLastError();
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  if (e != cudaSuccess) return MMM_ERR_CUDA;
  if (tflops_out) *tflops_out = best_f;
  if (mufu_tops_out) *mufu_tops_out = best_m;
  return MMM_OK;
}
