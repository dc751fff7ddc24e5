// Latitude-weighted reductions beside the L2 training loss (SURVEY 8(f) rank 4): the L1 loss family
// (utils/losses.py:116-124 with GeometricLpLoss p = 1, :188-232) and the anomaly-correlation sums of the validation loop
// (utils/weighted_acc_rmse.py:89-105).  Same structure as latw_l2_*: one streaming pass, 128-bit loads, warp-shuffle ->
// shared-memory -> one fp32 atomic per (plane, CTA).
#include "common.cuh"

namespace swinb200 {

// NACC accumulators per plane:  MODE 0 (L1): {sum q|p-t|, sum q|t|};  MODE 1 (ACC): {sum q p t, sum q p p, sum q t t}
// DET: acc_out is a [gridDim.y, planes, NACC] scratch, one row per row block
template <int MODE, bool DET = false>
__global__ void __launch_bounds__(256) latw_reduce_kernel(const float* __restrict__ prd, const float* __restrict__ tar,
                                                          const float* __restrict__ qw, float* __restrict__ acc_out, int H, int W,
                                                          int rows_per_block) {
  constexpr int NACC = MODE == 0 ? 2 : 3;
  __shared__ float red[NACC][8];
  const int plane = blockIdx.x;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(H, r0 + rows_per_block);
  const int w4 = W / 4;
  const float4* p4 = reinterpret_cast<const float4*>(prd + (size_t)plane * H * W);
  const float4* t4 = reinterpret_cast<const float4*>(tar + (size_t)plane * H * W);
  float a[NACC];
#pragma unroll
  for (int k = 0; k < NACC; ++k) a[k] = 0.f;
  const int n4 = (r1 - r0) * w4;
  const size_t base = (size_t)r0 * w4;
  for (int i = threadIdx.x; i < n4; i += blockDim.x * 4) {
    float4 p[4], t[4];
    float q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int ii = i + u * blockDim.x;
      if (ii < n4) {
        p[u] = __ldg(p4 + base + ii);
        t[u] = __ldg(t4 + base + ii);
        q[u] = __ldg(qw + r0 + ii / w4);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int ii = i + u * blockDim.x;
      if (ii < n4) {
        if (MODE == 0) {
          a[0] += q[u] * ((fabsf(p[u].x - t[u].x) + fabsf(p[u].y - t[u].y)) + (fabsf(p[u].z - t[u].z) + fabsf(p[u].w - t[u].w)));
          a[1] += q[u] * ((fabsf(t[u].x) + fabsf(t[u].y)) + (fabsf(t[u].z) + fabsf(t[u].w)));
        } else {
          a[0] += q[u] * ((p[u].x * t[u].x + p[u].y * t[u].y) + (p[u].z * t[u].z + p[u].w * t[u].w));
          a[1] += q[u] * ((p[u].x * p[u].x + p[u].y * p[u].y) + (p[u].z * p[u].z + p[u].w * p[u].w));
          a[NACC - 1] += q[u] * ((t[u].x * t[u].x + t[u].y * t[u].y) + (t[u].z * t[u].z + t[u].w * t[u].w));
        }
      }
    }
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    a[k] = warp_sum(a[k]);
    if (lane == 0) red[k][wid] = a[k];
  }
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
      float v = lane < (int)(blockDim.x >> 5) ? red[k][lane] : 0.f;
      v = warp_sum(v);
      if constexpr (DET) {
        if (lane == 0) acc_out[((size_t)blockIdx.y * gridDim.x + plane) * NACC + k] = v;
      } else {
        if (lane == 0) atomicAdd(acc_out + (size_t)plane * NACC + k, v);
      }
    }
  }
}

// L1: loss = sum_bc chw[c] * (relative ? num/den : num)
__global__ void latw_l1_finish_kernel(const float* __restrict__ sums, const float* __restrict__ chw, int relative,
                                      float* __restrict__ loss, int BC, int C) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < BC; i += blockDim.x) acc += chw[i % C] * (relative ? sums[2 * i] / sums[2 * i + 1] : sums[2 * i]);
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    acc = warp_sum(acc);
    if (threadIdx.x == 0) *loss = acc;
  }
}

// acc[b,c] = S_pt / sqrt(S_pp * S_tt)
__global__ void latw_acc_finish_kernel(const float* __restrict__ sums, float* __restrict__ acc, int BC) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < BC) acc[i] = sums[3 * i] / sqrtf(sums[3 * i + 1] * sums[3 * i + 2]);
}

// d|p-t|/dp = sign(p-t) (0 at 0, as torch.abs' backward)
__global__ void __launch_bounds__(256) latw_l1_bwd_kernel(const float* __restrict__ prd, const float* __restrict__ tar,
                                                          const float* __restrict__ qw, const float* __restrict__ chw,
                                                          const float* __restrict__ sums, const float* __restrict__ gloss,
                                                          int relative, float* __restrict__ dprd, int C, int H, int W,
                                                          int rows_per_block) {
  const int plane = blockIdx.x;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(H, r0 + rows_per_block);
  const int w4 = W / 4;
  const float coef = gloss[0] * chw[plane % C] / (relative ? sums[2 * plane + 1] : 1.0f);
  const float4* p4 = reinterpret_cast<const float4*>(prd + (size_t)plane * H * W);
  const float4* t4 = reinterpret_cast<const float4*>(tar + (size_t)plane * H * W);
  float4* d4 = reinterpret_cast<float4*>(dprd + (size_t)plane * H * W);
  const int n4 = (r1 - r0) * w4;
  const size_t base = (size_t)r0 * w4;
  auto sgn = [](float d) { return d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f); };
  for (int i = threadIdx.x; i < n4; i += blockDim.x) {
    const float4 p = __ldg(p4 + base + i), t = __ldg(t4 + base + i);
    const float s = coef * __ldg(qw + r0 + i / w4);
    d4[base + i] = make_float4(s * sgn(p.x - t.x), s * sgn(p.y - t.y), s * sgn(p.z - t.z), s * sgn(p.w - t.w));
  }
}

static void plane_split(int planes, int H, int& split, int& rpb) {
  split = max(1, (sm_count() * 8 + planes - 1) / planes);
  rpb = max(1, (H + split - 1) / split);
  split = (H + rpb - 1) / rpb;
}

}  // namespace swinb200

using namespace swinb200;

extern "C" int swinb200_latw_l1_fwd(const float* prd, const float* tar, const float* qw, const float* chw, int relative,
                                    float* sums, float* loss, int B, int C, int H, int W, void* stream) {
  SWB_CHECK_ARG(prd && tar && qw && chw && sums && loss, "latw_l1_fwd: null pointer");
  SWB_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && W % 4 == 0, "latw_l1_fwd: bad shape (W must be a multiple of 4)");
  cudaStream_t s = (cudaStream_t)stream;
  const int planes = B * C;
  SWB_CUDA(cudaMemsetAsync(sums, 0, sizeof(float) * 2 * planes, s));
  int split, rpb;
  plane_split(planes, H, split, rpb);
  latw_reduce_kernel<0><<<dim3(planes, split), 256, 0, s>>>(prd, tar, qw, sums, H, W, rpb);
  SWB_LAUNCH_CHECK();
  latw_l1_finish_kernel<<<1, 256, 0, s>>>(sums, chw, relative, loss, planes, C);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

extern "C" int swinb200_latw_l1_bwd(const float* prd, const float* tar, const float* qw, const float* chw, const float* sums,
                                    const float* gloss, int relative, float* dprd, int B, int C, int H, int W, void* stream) {
  SWB_CHECK_ARG(prd && tar && qw && chw && gloss && dprd && (sums || !relative), "latw_l1_bwd: null pointer");
  SWB_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && W % 4 == 0, "latw_l1_bwd: bad shape");
  const int planes = B * C;
  int split, rpb;
  plane_split(planes, H, split, rpb);
  latw_l1_bwd_kernel<<<dim3(planes, split), 256, 0, (cudaStream_t)stream>>>(prd, tar, qw, chw, sums, gloss, relative, dprd, C, H, W, rpb);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

extern "C" int swinb200_latw_acc(const float* prd, const float* tar, const float* qw, float* sums, float* acc, int B, int C, int H,
                                 int W, void* stream) {
  SWB_CHECK_ARG(prd && tar && qw && sums && acc, "latw_acc: null pointer");
  SWB_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && W % 4 == 0, "latw_acc: bad shape (W must be a multiple of 4)");
  cudaStream_t s = (cudaStream_t)stream;
  const int planes = B * C;
  SWB_CUDA(cudaMemsetAsync(sums, 0, sizeof(float) * 3 * planes, s));
  int split, rpb;
  plane_split(planes, H, split, rpb);
  latw_reduce_kernel<1><<<dim3(planes, split), 256, 0, s>>>(prd, tar, qw, sums, H, W, rpb);
  SWB_LAUNCH_CHECK();
  latw_acc_finish_kernel<<<(planes + 255) / 256, 256, 0, s>>>(sums, acc, planes);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

// ---- deterministic mode: row-block partials, summed in row-block order by swinb200_ordered_reduce ------------------------
template <int MODE>
static int latw_sums_det(const float* prd, const float* tar, const float* qw, float* sums, int B, int C, int H, int W, float* part,
                         long long part_floats, cudaStream_t s) {
  constexpr int NACC = MODE == 0 ? 2 : 3;
  SWB_CHECK_ARG(part != nullptr && part_floats >= (long long)NACC * B * C * H, "latw (deterministic): scratch of %d*B*C*H = %lld floats "
                "required, got %lld", NACC, (long long)NACC * B * C * H, part_floats);
  const int planes = B * C;
  int split, rpb;
  plane_split(planes, H, split, rpb);
  latw_reduce_kernel<MODE, true><<<dim3(planes, split), 256, 0, s>>>(prd, tar, qw, part, H, W, rpb);
  SWB_LAUNCH_CHECK();
  return ordered_reduce(part, split, (long long)planes * NACC, (long long)planes * NACC, 1, sums, 0, s);
}

extern "C" int swinb200_latw_l1_fwd_det(const float* prd, const float* tar, const float* qw, const float* chw, int relative, float* sums,
                                        float* loss, int B, int C, int H, int W, float* part, long long part_floats, void* stream) {
  SWB_CHECK_ARG(prd && tar && qw && chw && sums && loss, "latw_l1_fwd_det: null pointer");
  SWB_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && W % 4 == 0, "latw_l1_fwd_det: bad shape (W must be a multiple of 4)");
  cudaStream_t s = (cudaStream_t)stream;
  if (int e = latw_sums_det<0>(prd, tar, qw, sums, B, C, H, W, part, part_floats, s)) return e;
  latw_l1_finish_kernel<<<1, 256, 0, s>>>(sums, chw, relative, loss, B * C, C);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

extern "C" int swinb200_latw_acc_det(const float* prd, const float* tar, const float* qw, float* sums, float* acc, int B, int C, int H,
                                     int W, float* part, long long part_floats, void* stream) {
  SWB_CHECK_ARG(prd && tar && qw && sums && acc, "latw_acc_det: null pointer");
  SWB_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && W % 4 == 0, "latw_acc_det: bad shape (W must be a multiple of 4)");
  cudaStream_t s = (cudaStream_t)stream;
  if (int e = latw_sums_det<1>(prd, tar, qw, sums, B, C, H, W, part, part_floats, s)) return e;
  latw_acc_finish_kernel<<<(B * C + 255) / 256, 256, 0, s>>>(sums, acc, B * C);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}
