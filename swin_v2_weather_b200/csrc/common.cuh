// Shared helpers for the swinb200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#include "../../include/swinb200.h"
#include "../../include/swinb200_debug.h"

namespace swinb200 {

// ---- error plumbing: C-ABI entry points return an int, message kept per thread -----------------
void set_error(const char* fmt, ...);

#define SWB_CHECK_ARG(cond, ...)                                   \
  do {                                                              \
    if (!(cond)) {                                                  \
      ::swinb200::set_error(__VA_ARGS__);                           \
      return SWINB200_ERR_INVALID_ARG;                              \
    }                                                               \
  } while (0)

#define SWB_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::swinb200::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),       \
                            __FILE__, __LINE__);                                          \
      return SWINB200_ERR_CUDA;                                                           \
    }                                                                                     \
  } while (0)

#define SWB_LAUNCH_CHECK() SWB_CUDA(cudaGetLastError())

inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// out[i] (+)= sum_{p < n_part} sum_{j < inner} part[p * stride + i * inner + j], summed in exactly that order and added once
// into out: the second stage of every deterministic-mode reduction (determinism.cu)
int ordered_reduce(const float* part, int n_part, long long stride, long long n, int inner, float* out, int accumulate,
                   cudaStream_t stream);

// LayerNorm + DropPath scale + residual operands of the fused proj / fc2 epilogue (SWINB200_EPI_BIAS_LN, gemm_tc.cu)
struct GemmLnFuse {
  const float* x_in;
  const float* gamma;
  const float* beta;
  const float* sample_scale;   // may be null
  float* x_out;
  void* xb_out;
  float* stats;
  int* counters;
  int n_counters;
  int rows_per_sample;
  float eps;
};

// ---- activation storage type helpers ------------------------------------------------------------
template <typename T> struct Act;
template <> struct Act<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
  static __device__ __forceinline__ float round(float v) { return v; }
};
template <> struct Act<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};

// 8-element vector load/store in activation type (16 B for bf16, 32 B for fp32)
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld8(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 r = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ void st8(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void st8(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]);
  r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]);
  r.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = r;
}

// ---- math ---------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
__device__ __forceinline__ float gelu_erf_grad(float x) {
  // d/dx [x * Phi(x)] = Phi(x) + x * phi(x)
  const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
  const float pdf = 0.39894228040143267794f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Region label used by the shifted-window mask (reference swinv2_global.py:410-420):
// label 1 iff the *rolled* row index is >= H - shift_h (every row if only the W shift is active).
__host__ __device__ __forceinline__ int shift_region_label(int rolled_row, int H, int shift_h) {
  return (shift_h > 0) ? (rolled_row >= H - shift_h ? 1 : 0) : 1;
}

}  // namespace swinb200
