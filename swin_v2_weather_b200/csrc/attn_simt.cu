// CUDA-core windowed cosine attention (forward + backward), one CTA per (sample, window, head).
// fp32 validation back end and bring-up stand-in for the tcgen05 kernel.  The cyclic shift, window
// partition and window reverse of the reference (swinv2_global.py:89-119, 446-478) are pure index
// arithmetic here: slot n = a*Ww + c of window (wh, ww) is token ((wh*Wh+a+s0) % H, (ww*Ww+c+s1) % W).
#include "common.cuh"

namespace swinb200 {

struct WinGeom {
  int B, H, W, C, heads, Wh, Ww, s0, s1;
  __host__ __device__ int L() const { return Wh * Ww; }
  __host__ __device__ int nWw() const { return W / Ww; }
  __host__ __device__ int nW() const { return (H / Wh) * (W / Ww); }
  __host__ __device__ int d() const { return C / heads; }
};

__device__ __forceinline__ void window_slot(const WinGeom& g, int b, int w, int n, int& token, int& label) {
  const int wh = w / g.nWw(), ww = w % g.nWw();
  const int a = n / g.Ww, c = n % g.Ww;
  const int rr = wh * g.Wh + a;
  const int i = (rr + g.s0) % g.H;
  const int j = (ww * g.Ww + c + g.s1) % g.W;
  token = (b * g.H + i) * g.W + j;
  label = shift_region_label(rr, g.H, g.s0);
}

constexpr int kAttnWarps = 8;
constexpr int kMaxHeadDim = 256;

// GLOBAL_KV: the per-window operand tiles (2 x L rows of d + 1 fp32 / d + 2 bf16 values) do not fit in shared memory -- fp32 at
// head_dim 256 needs 333 KB for 9x18 windows -- so the dot products read their rows in place from global memory (L2).
// This back end is the validation / bring-up path; the layout of the loops is the same either way.

template <typename T>
__device__ __forceinline__ int pad_d(int d) { return sizeof(T) == 4 ? d + 1 : d + 2; }

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// LSE = false: forward-only launches (lse == NULL).  A compile-time flag rather than a runtime test: the test pushed the
// fp32 global-K/V kernel into a spill.
template <typename T, bool GLOBAL_KV, bool LSE = true>
__global__ void __launch_bounds__(kAttnWarps * 32) attn_simt_fwd_kernel(const T* __restrict__ qkv, const float* __restrict__ scale_p,
                                                                        const float* __restrict__ bias, T* __restrict__ o,
                                                                        float* __restrict__ lse, WinGeom g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int L = g.L(), d = g.d(), dp = pad_d<T>(d);
  const int head = blockIdx.x % g.heads;
  const int w = (blockIdx.x / g.heads) % g.nW();
  const int b = blockIdx.x / (g.heads * g.nW());
  const bool masked = (g.s0 > 0 || g.s1 > 0);
  T* Ks = reinterpret_cast<T*>(smem_raw);
  T* Vs = Ks + (GLOBAL_KV ? 0 : (size_t)L * dp);
  float* fbase = reinterpret_cast<float*>(Vs + (GLOBAL_KV ? 0 : (size_t)L * dp));  // 2*L*dp*sizeof(T) is a multiple of 4
  float* qs = fbase;                          // [warps][d]
  float* ps = qs + kAttnWarps * d;            // [warps][L]
  int* tok = reinterpret_cast<int*>(ps + kAttnWarps * L);  // [L]
  int* lab = tok + L;                                       // [L]
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int C3 = 3 * g.C;

  for (int n = threadIdx.x; n < L; n += blockDim.x) {
    int t, l;
    window_slot(g, b, w, n, t, l);
    tok[n] = t;
    lab[n] = l;
  }
  __syncthreads();
  if (!GLOBAL_KV) {
    for (int it = threadIdx.x; it < L * d; it += blockDim.x) {
      const int n = it / d, c = it % d;
      const T* row = qkv + (size_t)tok[n] * C3 + head * d + c;
      Ks[n * dp + c] = row[g.C];
      Vs[n * dp + c] = row[2 * g.C];
    }
    __syncthreads();
  }
  auto k_row = [&](int j) -> const T* { return GLOBAL_KV ? qkv + (size_t)tok[j] * C3 + g.C + head * d : Ks + j * dp; };
  auto v_row = [&](int j) -> const T* { return GLOBAL_KV ? qkv + (size_t)tok[j] * C3 + 2 * g.C + head * d : Vs + j * dp; };

  const float scale = scale_p[head];
  float* myq = qs + wid * d;
  float* myp = ps + wid * L;
  for (int i = wid; i < L; i += kAttnWarps) {
    const T* qrow = qkv + (size_t)tok[i] * C3 + head * d;
    for (int c = lane; c < d; c += 32) myq[c] = Act<T>::ld(qrow + c);
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < L; j += 32) {
      float acc = 0.f;
      const T* kr = k_row(j);
      for (int c = 0; c < d; ++c) acc = fmaf(myq[c], Act<T>::ld(kr + c), acc);
      float s = acc * scale;
      if (bias) s += bias[((size_t)head * L + i) * L + j];
      if (masked && lab[i] != lab[j]) s += -100.0f;
      myp[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < L; j += 32) {
      const float p = expf(myp[j] - mx);
      myp[j] = p;
      sum += p;
    }
    sum = warp_sum(sum);
    __syncwarp();
    const float inv = 1.0f / sum;
    T* orow = o + (size_t)tok[i] * g.C + head * d;
    for (int c = lane; c < d; c += 32) {
      float acc = 0.f;
      for (int j = 0; j < L; ++j) acc = fmaf(myp[j], Act<T>::ld(v_row(j) + c), acc);
      Act<T>::st(orow + c, acc * inv);
    }
    if (LSE && lane == 0) lse[(((size_t)b * g.nW() + w) * g.heads + head) * L + i] = mx + logf(sum);
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------
// DET (deterministic mode): dscale is a (B*nW*heads) scratch receiving the CTA's d(scale) at its item index, dbias a
// (B*nW*heads, L, L) scratch receiving the item's slice (each (i, j) is visited by exactly one lane of the CTA)
template <typename T, bool GLOBAL_KV, bool DET = false>
__global__ void __launch_bounds__(kAttnWarps * 32) attn_simt_bwd_kernel(const T* __restrict__ qkv, const float* __restrict__ inv_norm,
                                                                        const float* __restrict__ scale_p, const float* __restrict__ bias,
                                                                        const T* __restrict__ o, const T* __restrict__ d_o,
                                                                        const float* __restrict__ lse, T* __restrict__ dqkv,
                                                                        float* __restrict__ dscale, float* __restrict__ dbias,
                                                                        WinGeom g) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int L = g.L(), d = g.d(), dp = pad_d<T>(d);
  const int head = blockIdx.x % g.heads;
  const int w = (blockIdx.x / g.heads) % g.nW();
  const int b = blockIdx.x / (g.heads * g.nW());
  const bool masked = (g.s0 > 0 || g.s1 > 0);
  T* M0 = reinterpret_cast<T*>(smem_raw);   // phase 1: Khat ; phase 2: Qhat
  T* M1 = M0 + (GLOBAL_KV ? 0 : (size_t)L * dp);              // phase 1: V    ; phase 2: dO
  float* fbase = reinterpret_cast<float*>(M1 + (GLOBAL_KV ? 0 : (size_t)L * dp));
  float* va = fbase;                         // [warps][d]  phase 1: qhat_i ; phase 2: khat_j
  float* vb = va + kAttnWarps * d;           // [warps][d]  phase 1: dO_i   ; phase 2: v_j
  float* ps = vb + kAttnWarps * d;           // [warps][L]  dS
  float* pp = ps + kAttnWarps * L;           // [warps][L]  P (phase 2)
  float* Ds = pp + kAttnWarps * L;           // [L]  rowsum(dO * O)
  float* lses = Ds + L;                      // [L]
  float* redsc = lses + L;                   // [warps]
  int* tok = reinterpret_cast<int*>(redsc + kAttnWarps);
  int* lab = tok + L;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int C3 = 3 * g.C;
  const int nvt = 2 * g.heads;

  for (int n = threadIdx.x; n < L; n += blockDim.x) {
    int t, l;
    window_slot(g, b, w, n, t, l);
    tok[n] = t;
    lab[n] = l;
    lses[n] = lse[(((size_t)b * g.nW() + w) * g.heads + head) * L + n];
  }
  __syncthreads();
  if (!GLOBAL_KV) {
    for (int it = threadIdx.x; it < L * d; it += blockDim.x) {
      const int n = it / d, c = it % d;
      const T* row = qkv + (size_t)tok[n] * C3 + head * d + c;
      M0[n * dp + c] = row[g.C];
      M1[n * dp + c] = row[2 * g.C];
    }
    __syncthreads();
  }
  int phase = 1;
  auto m0_row = [&](int n) -> const T* {
    if (!GLOBAL_KV) return M0 + n * dp;
    return qkv + (size_t)tok[n] * C3 + (phase == 1 ? g.C : 0) + head * d;
  };
  auto m1_row = [&](int n) -> const T* {
    if (!GLOBAL_KV) return M1 + n * dp;
    return phase == 1 ? qkv + (size_t)tok[n] * C3 + 2 * g.C + head * d : d_o + (size_t)tok[n] * g.C + head * d;
  };

  const float scale = scale_p[head];
  float dsc_acc = 0.f;
  float* mya = va + wid * d;
  float* myb = vb + wid * d;
  float* myds = ps + wid * L;
  float* myp = pp + wid * L;

  // ---- phase 1: one query row per warp-iteration -> dq --------------------------------------------
  for (int i = wid; i < L; i += kAttnWarps) {
    const size_t t = tok[i];
    float dsum = 0.f;
    for (int c = lane; c < d; c += 32) {
      mya[c] = Act<T>::ld(qkv + t * C3 + head * d + c);
      const float go = Act<T>::ld(d_o + t * g.C + head * d + c);
      myb[c] = go;
      dsum += go * Act<T>::ld(o + t * g.C + head * d + c);
    }
    dsum = warp_sum(dsum);
    if (lane == 0) Ds[i] = dsum;
    __syncwarp();
    const float lse_i = lses[i];
    for (int j = lane; j < L; j += 32) {
      float cs = 0.f, dpv = 0.f;
      const T* kr = m0_row(j);
      const T* vr = m1_row(j);
      for (int c = 0; c < d; ++c) {
        cs = fmaf(mya[c], Act<T>::ld(kr + c), cs);
        dpv = fmaf(myb[c], Act<T>::ld(vr + c), dpv);
      }
      float s = cs * scale;
      if (bias) s += bias[((size_t)head * L + i) * L + j];
      if (masked && lab[i] != lab[j]) s += -100.0f;
      const float p = expf(s - lse_i);
      const float ds = p * (dpv - dsum);
      myds[j] = ds;
      dsc_acc += ds * cs;
      if constexpr (DET) {
        if (dbias) dbias[((size_t)blockIdx.x * L + i) * L + j] = ds;
      } else {
        if (dbias) atomicAdd(dbias + ((size_t)head * L + i) * L + j, ds);
      }
    }
    __syncwarp();
    // dqhat, then back through the normalisation: dq = inv_norm * (dqhat - qhat * <qhat, dqhat>)
    float dq[kMaxHeadDim / 32];
    float dot = 0.f;
    int cc = 0;
    for (int c = lane; c < d; c += 32, ++cc) {
      float acc = 0.f;
      for (int j = 0; j < L; ++j) acc = fmaf(myds[j], Act<T>::ld(m0_row(j) + c), acc);
      dq[cc] = acc * scale;
      dot += dq[cc] * mya[c];
    }
    dot = warp_sum(dot);
    const float inq = inv_norm[t * nvt + head];
    cc = 0;
    for (int c = lane; c < d; c += 32, ++cc)
      Act<T>::st(dqkv + t * C3 + head * d + c, inq * (dq[cc] - mya[c] * dot));
    __syncwarp();
  }
  __syncthreads();

  // ---- phase 2: reload with Qhat / dO; one key row per warp-iteration -> dk, dv ------------------
  phase = 2;
  if (!GLOBAL_KV) {
    for (int it = threadIdx.x; it < L * d; it += blockDim.x) {
      const int n = it / d, c = it % d;
      M0[n * dp + c] = qkv[(size_t)tok[n] * C3 + head * d + c];
      M1[n * dp + c] = d_o[(size_t)tok[n] * g.C + head * d + c];
    }
    __syncthreads();
  }
  for (int j = wid; j < L; j += kAttnWarps) {
    const size_t t = tok[j];
    for (int c = lane; c < d; c += 32) {
      mya[c] = Act<T>::ld(qkv + t * C3 + g.C + head * d + c);
      myb[c] = Act<T>::ld(qkv + t * C3 + 2 * g.C + head * d + c);
    }
    __syncwarp();
    for (int i = lane; i < L; i += 32) {
      float cs = 0.f, dpv = 0.f;
      const T* qr = m0_row(i);
      const T* gr = m1_row(i);
      for (int c = 0; c < d; ++c) {
        cs = fmaf(mya[c], Act<T>::ld(qr + c), cs);
        dpv = fmaf(myb[c], Act<T>::ld(gr + c), dpv);
      }
      float s = cs * scale;
      if (bias) s += bias[((size_t)head * L + i) * L + j];
      if (masked && lab[i] != lab[j]) s += -100.0f;
      const float p = expf(s - lses[i]);
      myp[i] = p;
      myds[i] = p * (dpv - Ds[i]);
    }
    __syncwarp();
    float dk[kMaxHeadDim / 32];
    float dot = 0.f;
    int cc = 0;
    for (int c = lane; c < d; c += 32, ++cc) {
      float ak = 0.f, av = 0.f;
      for (int i = 0; i < L; ++i) {
        ak = fmaf(myds[i], Act<T>::ld(m0_row(i) + c), ak);
        av = fmaf(myp[i], Act<T>::ld(m1_row(i) + c), av);
      }
      dk[cc] = ak * scale;
      dot += dk[cc] * mya[c];
      Act<T>::st(dqkv + t * C3 + 2 * g.C + head * d + c, av);
    }
    dot = warp_sum(dot);
    const float ink = inv_norm[t * nvt + g.heads + head];
    cc = 0;
    for (int c = lane; c < d; c += 32, ++cc)
      Act<T>::st(dqkv + t * C3 + g.C + head * d + c, ink * (dk[cc] - mya[c] * dot));
    __syncwarp();
  }

  dsc_acc = warp_sum(dsc_acc);
  if (lane == 0) redsc[wid] = dsc_acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < kAttnWarps; ++i) s += redsc[i];
    if constexpr (DET) dscale[blockIdx.x] = s;
    else atomicAdd(dscale + head, s);
  }
}

template <typename T>
static size_t attn_smem_bytes(const WinGeom& g, bool bwd, bool global_kv) {
  const int L = g.L(), d = g.d();
  const int dp = sizeof(T) == 4 ? d + 1 : d + 2;
  size_t b = global_kv ? 0 : 2 * (size_t)L * dp * sizeof(T);
  b = (b + 3) / 4 * 4;
  if (!bwd)
    b += (size_t)(kAttnWarps * d + kAttnWarps * L) * 4 + 2 * (size_t)L * 4;
  else
    b += (size_t)(2 * kAttnWarps * d + 2 * kAttnWarps * L + 2 * L + kAttnWarps) * 4 + 2 * (size_t)L * 4;
  return b + 16;
}

template <typename T>
static int launch_fwd(const T* qkv, const float* scale, const float* bias, T* o, float* lse, const WinGeom& g, cudaStream_t s) {
  const bool global_kv = attn_smem_bytes<T>(g, false, false) > 227 * 1024;
  const size_t smem = attn_smem_bytes<T>(g, false, global_kv);
  if (smem > 227 * 1024) {
    set_error("window_attn_fwd (CUDA-core back end): window %dx%d, head_dim %d needs %zu B of shared memory", g.Wh, g.Ww, g.d(), smem);
    return SWINB200_ERR_UNSUPPORTED;
  }
  auto kernel = global_kv ? (lse ? attn_simt_fwd_kernel<T, true> : attn_simt_fwd_kernel<T, true, false>)
                          : (lse ? attn_simt_fwd_kernel<T, false> : attn_simt_fwd_kernel<T, false, false>);
  SWB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<g.B * g.nW() * g.heads, kAttnWarps * 32, smem, s>>>(qkv, scale, bias, o, lse, g);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

template <typename T>
static int launch_bwd(const T* qkv, const float* inv_norm, const float* scale, const float* bias, const T* o, const T* d_o,
                      const float* lse, T* dqkv, float* dscale, float* dbias, const WinGeom& g, cudaStream_t s,
                      float* det_part = nullptr) {
  const bool global_kv = attn_smem_bytes<T>(g, true, false) > 227 * 1024;
  const size_t smem = attn_smem_bytes<T>(g, true, global_kv);
  if (smem > 227 * 1024) {
    set_error("window_attn_bwd (CUDA-core back end): window %dx%d, head_dim %d needs %zu B of shared memory", g.Wh, g.Ww, g.d(), smem);
    return SWINB200_ERR_UNSUPPORTED;
  }
  if (det_part != nullptr) {
    const int bw = g.B * g.nW(), L = g.L();
    const long long dbias_n = (long long)g.heads * L * L;
    // same slot layout as the tcgen05 back ends: the d(scale) slots first, then the per-item d(bias) slices
    float* dbias_part = (dbias != nullptr) ? det_part + (long long)bw * g.heads * 4 * ((L + 127) / 128) : nullptr;
    auto kernel = global_kv ? attn_simt_bwd_kernel<T, true, true> : attn_simt_bwd_kernel<T, false, true>;
    SWB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<bw * g.heads, kAttnWarps * 32, smem, s>>>(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, det_part, dbias_part, g);
    SWB_LAUNCH_CHECK();
    if (int e = ordered_reduce(det_part, bw, g.heads, g.heads, 1, dscale, 1, s)) return e;
    if (dbias != nullptr) return ordered_reduce(dbias_part, bw, dbias_n, dbias_n, 1, dbias, 1, s);
    return SWINB200_OK;
  }
  auto kernel = global_kv ? attn_simt_bwd_kernel<T, true> : attn_simt_bwd_kernel<T, false>;
  SWB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<g.B * g.nW() * g.heads, kAttnWarps * 32, smem, s>>>(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, g);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

int attn_tcgen05_fwd(const void* qkv, const float* scale, const float* bias, void* o, float* lse, int B, int H, int W, int C,
                     int heads, int Wh, int Ww, int s0, int s1, cudaStream_t stream);
int attn_tcgen05_bwd(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o,
                     const void* d_o, const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, int B, int H, int W,
                     int C, int heads, int Wh, int Ww, int s0, int s1, cudaStream_t stream, float* det_part = nullptr);

static int check_geom(const char* who, int B, int H, int W, int C, int heads, int Wh, int Ww, int s0, int s1) {
  SWB_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && heads > 0, "%s: bad shape", who);
  SWB_CHECK_ARG(Wh > 0 && Ww > 0 && H % Wh == 0 && W % Ww == 0, "%s: window (%d,%d) does not tile the (%d,%d) grid", who, Wh, Ww, H, W);
  SWB_CHECK_ARG(C % heads == 0 && (C / heads) % 8 == 0 && C / heads <= kMaxHeadDim, "%s: head_dim %d unsupported", who, C / heads);
  SWB_CHECK_ARG(s0 >= 0 && s0 < Wh && s1 >= 0 && s1 < Ww, "%s: shift (%d,%d) must be smaller than the window", who, s0, s1);
  return SWINB200_OK;
}

}  // namespace swinb200

using namespace swinb200;

extern "C" int swinb200_window_attn_fwd(int backend, const void* qkv, int act_dtype, const float* scale, const float* bias,
                                        void* o, float* lse, int B, int H, int W, int C, int heads, int Wh, int Ww, int s0,
                                        int s1, void* stream) {
  SWB_CHECK_ARG(qkv && scale && o, "window_attn_fwd: null pointer");     // lse may be null (forward-only)
  if (int e = check_geom("window_attn_fwd", B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  const WinGeom g{B, H, W, C, heads, Wh, Ww, s0, s1};
  cudaStream_t s = (cudaStream_t)stream;
  if (backend == SWINB200_GEMM_TCGEN05) {
    SWB_CHECK_ARG(act_dtype == SWINB200_BF16, "window_attn_fwd: the tcgen05 back end needs bf16 activations");
    return attn_tcgen05_fwd(qkv, scale, bias, o, lse, B, H, W, C, heads, Wh, Ww, s0, s1, s);
  }
  SWB_CHECK_ARG(backend == SWINB200_GEMM_SIMT, "window_attn_fwd: unknown backend %d", backend);
  // second plane of `lse` (softmax-weighted mean cosine): not used by this back end's backward, defined as zero
  if (lse != nullptr)
    SWB_CUDA(cudaMemsetAsync(lse + (size_t)B * g.nW() * heads * Wh * Ww, 0, sizeof(float) * (size_t)B * g.nW() * heads * Wh * Ww, s));
  if (act_dtype == SWINB200_BF16) return launch_fwd<__nv_bfloat16>((const __nv_bfloat16*)qkv, scale, bias, (__nv_bfloat16*)o, lse, g, s);
  if (act_dtype == SWINB200_F32) return launch_fwd<float>((const float*)qkv, scale, bias, (float*)o, lse, g, s);
  SWB_CHECK_ARG(false, "window_attn_fwd: bad act_dtype %d", act_dtype);
}

extern "C" int swinb200_window_attn_bwd(int backend, const void* qkv, int act_dtype, const float* inv_norm, const float* scale,
                                        const float* bias, const void* o, const void* d_o, const float* lse, void* dqkv,
                                        float* dscale, float* dbias, float* ws, int B, int H, int W, int C, int heads, int Wh,
                                        int Ww, int s0, int s1, void* stream) {
  SWB_CHECK_ARG(qkv && inv_norm && scale && o && d_o && lse && dqkv && dscale, "window_attn_bwd: null pointer");
  if (int e = check_geom("window_attn_bwd", B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  const WinGeom g{B, H, W, C, heads, Wh, Ww, s0, s1};
  cudaStream_t s = (cudaStream_t)stream;
  if (backend == SWINB200_GEMM_TCGEN05) {
    SWB_CHECK_ARG(act_dtype == SWINB200_BF16, "window_attn_bwd: the tcgen05 back end needs bf16 activations");
    return attn_tcgen05_bwd(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, ws, B, H, W, C, heads, Wh, Ww, s0, s1, s);
  }
  SWB_CHECK_ARG(backend == SWINB200_GEMM_SIMT, "window_attn_bwd: unknown backend %d", backend);
  if (act_dtype == SWINB200_BF16)
    return launch_bwd<__nv_bfloat16>((const __nv_bfloat16*)qkv, inv_norm, scale, bias, (const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o, lse, (__nv_bfloat16*)dqkv, dscale, dbias, g, s);
  if (act_dtype == SWINB200_F32)
    return launch_bwd<float>((const float*)qkv, inv_norm, scale, bias, (const float*)o, (const float*)d_o, lse, (float*)dqkv, dscale, dbias, g, s);
  SWB_CHECK_ARG(false, "window_attn_bwd: bad act_dtype %d", act_dtype);
}

extern "C" int swinb200_window_attn_bwd_det(int backend, const void* qkv, int act_dtype, const float* inv_norm, const float* scale,
                                            const float* bias, const void* o, const void* d_o, const float* lse, void* dqkv,
                                            float* dscale, float* dbias, float* ws, int B, int H, int W, int C, int heads, int Wh,
                                            int Ww, int s0, int s1, float* part, long long part_floats, void* stream) {
  SWB_CHECK_ARG(qkv && inv_norm && scale && o && d_o && lse && dqkv && dscale, "window_attn_bwd_det: null pointer");
  SWB_CHECK_ARG(dbias == nullptr || bias != nullptr, "window_attn_bwd_det: dbias needs the bias table");
  if (int e = check_geom("window_attn_bwd_det", B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  const WinGeom g{B, H, W, C, heads, Wh, Ww, s0, s1};
  const long long items = (long long)B * g.nW() * heads, L = g.L();
  const long long need = items * (4 * ((L + 127) / 128) + (dbias != nullptr ? L * L : 0));
  SWB_CHECK_ARG(part != nullptr && part_floats >= need, "window_attn_bwd_det: scratch of %lld floats required, got %lld", need, part_floats);
  cudaStream_t s = (cudaStream_t)stream;
  if (backend == SWINB200_GEMM_TCGEN05) {
    SWB_CHECK_ARG(act_dtype == SWINB200_BF16, "window_attn_bwd_det: the tcgen05 back end needs bf16 activations");
    return attn_tcgen05_bwd(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, ws, B, H, W, C, heads, Wh, Ww, s0, s1, s, part);
  }
  SWB_CHECK_ARG(backend == SWINB200_GEMM_SIMT, "window_attn_bwd_det: unknown backend %d", backend);
  if (act_dtype == SWINB200_BF16)
    return launch_bwd<__nv_bfloat16>((const __nv_bfloat16*)qkv, inv_norm, scale, bias, (const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o,
                                     lse, (__nv_bfloat16*)dqkv, dscale, dbias, g, s, part);
  if (act_dtype == SWINB200_F32)
    return launch_bwd<float>((const float*)qkv, inv_norm, scale, bias, (const float*)o, (const float*)d_o, lse, (float*)dqkv, dscale, dbias,
                             g, s, part);
  SWB_CHECK_ARG(false, "window_attn_bwd_det: bad act_dtype %d", act_dtype);
}
