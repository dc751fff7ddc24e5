// CUDA-core GEMM: D = epilogue(A * B^T) with arbitrary operand majors.
// This is the fp32 validation back end (fp32 storage, fp32 FMA accumulation -> parity <= 1e-5 against
// the fp32 oracle) and the bring-up stand-in for the tcgen05 GEMM in bf16 mode.  It is correct for any
// shape; it is not the performance path.
#include "common.cuh"

namespace swinb200 {

constexpr int SBM = 64, SBN = 64, SBK = 16;

template <typename T, int EPI>
__global__ void __launch_bounds__(256) gemm_simt_kernel(int M, int N, int K, const T* __restrict__ A, long long sam,
                                                        long long sak, const T* __restrict__ B, long long sbn, long long sbk,
                                                        const float* __restrict__ bias, void* __restrict__ Dv, int ldd,
                                                        void* __restrict__ D2v, const void* __restrict__ auxv, int ld_aux,
                                                        int accumulate) {
  __shared__ float As[SBK][SBM + 4];
  __shared__ float Bs[SBK][SBN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * SBM, n0 = blockIdx.x * SBN;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const bool a_kfast = (sak == 1);
  const bool b_kfast = (sbk == 1);
  for (int k0 = 0; k0 < K; k0 += SBK) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = tid + r * 256;
      {
        const int kk = a_kfast ? (i & 15) : (i >> 6);
        const int mm = a_kfast ? (i >> 4) : (i & 63);
        const int gm = m0 + mm, gk = k0 + kk;
        As[kk][mm] = (gm < M && gk < K) ? Act<T>::ld(A + gm * sam + gk * sak) : 0.f;
      }
      {
        const int kk = b_kfast ? (i & 15) : (i >> 6);
        const int nn = b_kfast ? (i >> 4) : (i & 63);
        const int gn = n0 + nn, gk = k0 + kk;
        Bs[kk][nn] = (gn < N && gk < K) ? Act<T>::ld(B + gn * sbn + gk * sbk) : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SBK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w};
      const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }

#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j];
      const size_t o = (size_t)m * ldd + n;
      if (EPI == SWINB200_EPI_BIAS) {
        if (bias) v += bias[n];
        Act<T>::st(reinterpret_cast<T*>(Dv) + o, v);
      } else if (EPI == SWINB200_EPI_BIAS_GELU) {
        if (bias) v += bias[n];
        Act<T>::st(reinterpret_cast<T*>(D2v) + o, v);
        // GELU is evaluated on the stored (rounded) pre-activation so forward and backward agree
        Act<T>::st(reinterpret_cast<T*>(Dv) + o, gelu_erf(Act<T>::round(v)));
      } else if (EPI == SWINB200_EPI_BIAS_GELU_FWD) {
        if (bias) v += bias[n];
        Act<T>::st(reinterpret_cast<T*>(Dv) + o, gelu_erf(Act<T>::round(v)));   // BIAS_GELU's D without D2
      } else if (EPI == SWINB200_EPI_DGELU) {
        const float h = Act<T>::ld(reinterpret_cast<const T*>(auxv) + (size_t)m * ld_aux + n);
        Act<T>::st(reinterpret_cast<T*>(Dv) + o, v * gelu_erf_grad(h));
      } else if (EPI == SWINB200_EPI_ADD_F32) {
        const float r = reinterpret_cast<const float*>(auxv)[(size_t)m * ld_aux + n];
        reinterpret_cast<float*>(Dv)[o] = v + r;
      } else {
        float* d = reinterpret_cast<float*>(Dv) + o;
        *d = accumulate ? (*d + v) : v;
      }
    }
  }
}

template <typename T>
static int launch_simt(int M, int N, int K, const T* A, int a_major, int lda, const T* B, int b_major, int ldb, int epi,
                       const float* bias, void* D, int ldd, void* D2, const void* aux, int ld_aux, int accumulate,
                       cudaStream_t s) {
  const long long sam = a_major ? 1 : lda, sak = a_major ? lda : 1;
  const long long sbn = b_major ? 1 : ldb, sbk = b_major ? ldb : 1;
  dim3 grid((N + SBN - 1) / SBN, (M + SBM - 1) / SBM);
#define SWB_SIMT(E) gemm_simt_kernel<T, E><<<grid, 256, 0, s>>>(M, N, K, A, sam, sak, B, sbn, sbk, bias, D, ldd, D2, aux, ld_aux, accumulate)
  switch (epi) {
    case SWINB200_EPI_BIAS: SWB_SIMT(SWINB200_EPI_BIAS); break;
    case SWINB200_EPI_BIAS_GELU: SWB_SIMT(SWINB200_EPI_BIAS_GELU); break;
    case SWINB200_EPI_BIAS_GELU_FWD: SWB_SIMT(SWINB200_EPI_BIAS_GELU_FWD); break;
    case SWINB200_EPI_DGELU: SWB_SIMT(SWINB200_EPI_DGELU); break;
    case SWINB200_EPI_ADD_F32: SWB_SIMT(SWINB200_EPI_ADD_F32); break;
    case SWINB200_EPI_F32: SWB_SIMT(SWINB200_EPI_F32); break;
    default: set_error("gemm: unknown epilogue %d", epi); return SWINB200_ERR_INVALID_ARG;
  }
#undef SWB_SIMT
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

int gemm_tcgen05(int M, int N, int K, const void* A, int a_major, int lda, const void* B, int b_major, int ldb, int epilogue,
                 const float* bias, void* D, int ldd, void* D2, const void* aux, int ld_aux, int accumulate, int split_k,
                 cudaStream_t stream, const GemmLnFuse* ln = nullptr, float* colsum_out = nullptr, float* part = nullptr);

}  // namespace swinb200

using namespace swinb200;

extern "C" int swinb200_gemm(int backend, int M, int N, int K, const void* A, int a_major, int lda, const void* B, int b_major,
                             int ldb, int in_dtype, int epilogue, const float* bias, void* D, int ldd, void* D2,
                             const void* aux, int ld_aux, int out_dtype, int accumulate, int split_k, void* stream) {
  SWB_CHECK_ARG(M > 0 && N > 0 && K > 0, "gemm: bad shape M=%d N=%d K=%d", M, N, K);
  SWB_CHECK_ARG(A && B && D, "gemm: null operand");
  SWB_CHECK_ARG(a_major == 0 || a_major == 1, "gemm: a_major must be 0/1");
  SWB_CHECK_ARG(b_major == 0 || b_major == 1, "gemm: b_major must be 0/1");
  SWB_CHECK_ARG(lda >= (a_major ? M : K) && ldb >= (b_major ? N : K) && ldd >= N, "gemm: leading dimension too small");
  SWB_CHECK_ARG((epilogue >= SWINB200_EPI_BIAS && epilogue <= SWINB200_EPI_BIAS_QKNORM) || epilogue == SWINB200_EPI_BIAS_GELU_FWD,
                "gemm: unknown epilogue %d", epilogue);
  if (epilogue == SWINB200_EPI_BIAS_QKNORM) {
    SWB_CHECK_ARG(backend == SWINB200_GEMM_TCGEN05 && in_dtype == SWINB200_BF16 && out_dtype == SWINB200_BF16,
                  "gemm: BIAS_QKNORM is a tcgen05 / bf16 epilogue (use BIAS + swinb200_qk_normalize elsewhere)");
    SWB_CHECK_ARG(ld_aux == 96 && N % 288 == 0 && a_major == 0 && b_major == 0,
                  "gemm: BIAS_QKNORM needs head_dim 96 and N = 3*C with C a multiple of 96");
    return gemm_tcgen05(M, N, K, A, a_major, lda, B, b_major, ldb, epilogue, bias, D, ldd, D2, aux, ld_aux, accumulate, 1, (cudaStream_t)stream);
  }
  const bool f32_out = (epilogue == SWINB200_EPI_ADD_F32 || epilogue == SWINB200_EPI_F32);
  SWB_CHECK_ARG(out_dtype == (f32_out ? SWINB200_F32 : in_dtype), "gemm: out_dtype %d does not match epilogue %d", out_dtype, epilogue);
  SWB_CHECK_ARG(epilogue != SWINB200_EPI_BIAS_GELU || D2, "gemm: BIAS_GELU needs D2");
  SWB_CHECK_ARG((epilogue != SWINB200_EPI_DGELU && epilogue != SWINB200_EPI_ADD_F32) || (aux && ld_aux >= N), "gemm: epilogue %d needs aux", epilogue);
  SWB_CHECK_ARG(split_k >= 1, "gemm: split_k must be >= 1");
  SWB_CHECK_ARG(split_k == 1 || (epilogue == SWINB200_EPI_F32 && accumulate), "gemm: split_k > 1 needs EPI_F32 with accumulate");
  cudaStream_t s = (cudaStream_t)stream;
  if (backend == SWINB200_GEMM_TCGEN05) {
    SWB_CHECK_ARG(in_dtype == SWINB200_BF16, "gemm: the tcgen05 back end needs bf16 operands");
    return gemm_tcgen05(M, N, K, A, a_major, lda, B, b_major, ldb, epilogue, bias, D, ldd, D2, aux, ld_aux, accumulate, split_k, s);
  }
  SWB_CHECK_ARG(backend == SWINB200_GEMM_SIMT, "gemm: unknown backend %d", backend);
  if (in_dtype == SWINB200_BF16)
    return launch_simt<__nv_bfloat16>(M, N, K, (const __nv_bfloat16*)A, a_major, lda, (const __nv_bfloat16*)B, b_major, ldb, epilogue, bias, D, ldd, D2, aux, ld_aux, accumulate, s);
  if (in_dtype == SWINB200_F32)
    return launch_simt<float>(M, N, K, (const float*)A, a_major, lda, (const float*)B, b_major, ldb, epilogue, bias, D, ldd, D2, aux, ld_aux, accumulate, s);
  SWB_CHECK_ARG(false, "gemm: bad in_dtype %d", in_dtype);
}

extern "C" int swinb200_linear_wgrad(int backend, int n_out, int n_in, int T, const void* dY, int ldy, const void* X, int ldx,
                                     float* dW, int lddw, float* dbias, int split_k, void* stream) {
  SWB_CHECK_ARG(n_out > 0 && n_in > 0 && T > 0, "linear_wgrad: bad shape n_out=%d n_in=%d T=%d", n_out, n_in, T);
  SWB_CHECK_ARG(dY && X && dW, "linear_wgrad: null pointer");
  SWB_CHECK_ARG(ldy >= n_out && ldx >= n_in && lddw >= n_in && split_k >= 1, "linear_wgrad: leading dimension too small");
  if (backend != SWINB200_GEMM_TCGEN05 || n_out % 256 != 0 || n_in < 256) {
    set_error("linear_wgrad: the fused weight + bias gradient is a tcgen05 / bf16 kernel for n_out a multiple of 256 and "
              "n_in >= 256; run swinb200_gemm(a1, b1, EPI_F32, accumulate) + swinb200_colsum for backend %d, n_out = %d, n_in = %d",
              backend, n_out, n_in);
    return SWINB200_ERR_UNSUPPORTED;
  }
  return gemm_tcgen05(n_out, n_in, T, dY, 1, ldy, X, 1, ldx, SWINB200_EPI_F32, nullptr, dW, lddw, nullptr, nullptr, 0, 1, split_k,
                      (cudaStream_t)stream, nullptr, dbias);
}

extern "C" int swinb200_linear_ln_residual(int backend, int M, int N, int K, const void* A, int lda, const void* W, int ldw,
                                           const float* bias, void* z, int ldz, const float* x_in, const float* gamma,
                                           const float* beta, const float* sample_scale, float* x_out, void* xb_out, float* stats,
                                           int rows_per_sample, float eps, int* counters, int n_counters, void* stream) {
  SWB_CHECK_ARG(M > 0 && N > 0 && K > 0, "linear_ln_residual: bad shape M=%d N=%d K=%d", M, N, K);
  SWB_CHECK_ARG(A && W && z && x_in && gamma && beta && x_out && xb_out && stats && counters, "linear_ln_residual: null pointer");
  SWB_CHECK_ARG(lda >= K && ldw >= K && ldz >= N && rows_per_sample > 0, "linear_ln_residual: leading dimension too small");
  if (backend != SWINB200_GEMM_TCGEN05 || N != 768) {
    set_error("linear_ln_residual: the fused epilogue is a tcgen05 / bf16 kernel for 768 output channels; "
              "run swinb200_gemm(EPI_BIAS) + swinb200_ln_residual_fwd for backend %d, N = %d", backend, N);
    return SWINB200_ERR_UNSUPPORTED;
  }
  GemmLnFuse ln{x_in, gamma, beta, sample_scale, x_out, xb_out, stats, counters, n_counters, rows_per_sample, eps};
  return gemm_tcgen05(M, N, K, A, 0, lda, W, 0, ldw, SWINB200_EPI_BIAS_LN, bias, z, ldz, nullptr, nullptr, 0, 0, 1, (cudaStream_t)stream, &ln);
}

extern "C" int swinb200_gemm_wgrad_det(int backend, int M, int N, int K, const void* A, int lda, const void* B, int ldb, int in_dtype,
                                       float* D, int split_k, float* part, long long part_floats, void* stream) {
  SWB_CHECK_ARG(M > 0 && N > 0 && K > 0 && split_k >= 1, "gemm_wgrad_det: bad shape M=%d N=%d K=%d split_k=%d", M, N, K, split_k);
  SWB_CHECK_ARG(A && B && D, "gemm_wgrad_det: null operand");
  SWB_CHECK_ARG(lda >= M && ldb >= N, "gemm_wgrad_det: leading dimension too small");
  cudaStream_t s = (cudaStream_t)stream;
  if (backend == SWINB200_GEMM_TCGEN05) {
    SWB_CHECK_ARG(in_dtype == SWINB200_BF16, "gemm_wgrad_det: the tcgen05 back end needs bf16 operands");
    SWB_CHECK_ARG(part != nullptr && part_floats >= (long long)split_k * M * N,
                  "gemm_wgrad_det: scratch of split_k*M*N = %lld floats required, got %lld", (long long)split_k * M * N, part_floats);
    return gemm_tcgen05(M, N, K, A, 1, lda, B, 1, ldb, SWINB200_EPI_F32, nullptr, D, N, nullptr, nullptr, 0, 1, split_k, s, nullptr,
                        nullptr, part);
  }
  // the CUDA-core GEMM does not split K: one thread adds each element once, in a fixed k order
  SWB_CHECK_ARG(backend == SWINB200_GEMM_SIMT, "gemm_wgrad_det: unknown backend %d", backend);
  if (in_dtype == SWINB200_BF16)
    return launch_simt<__nv_bfloat16>(M, N, K, (const __nv_bfloat16*)A, 1, lda, (const __nv_bfloat16*)B, 1, ldb, SWINB200_EPI_F32, nullptr, D, N,
                                      nullptr, nullptr, 0, 1, s);
  if (in_dtype == SWINB200_F32)
    return launch_simt<float>(M, N, K, (const float*)A, 1, lda, (const float*)B, 1, ldb, SWINB200_EPI_F32, nullptr, D, N, nullptr, nullptr, 0, 1, s);
  SWB_CHECK_ARG(false, "gemm_wgrad_det: bad in_dtype %d", in_dtype);
}

extern "C" int swinb200_linear_wgrad_det(int backend, int n_out, int n_in, int T, const void* dY, int ldy, const void* X, int ldx,
                                         float* dW, float* dbias, int split_k, float* part, long long part_floats, void* stream) {
  SWB_CHECK_ARG(n_out > 0 && n_in > 0 && T > 0, "linear_wgrad_det: bad shape n_out=%d n_in=%d T=%d", n_out, n_in, T);
  SWB_CHECK_ARG(dY && X && dW, "linear_wgrad_det: null pointer");
  SWB_CHECK_ARG(ldy >= n_out && ldx >= n_in && split_k >= 1, "linear_wgrad_det: leading dimension too small");
  const long long need = (long long)split_k * ((long long)n_out * n_in + n_out);
  SWB_CHECK_ARG(part != nullptr && part_floats >= need, "linear_wgrad_det: scratch of split_k*(n_out*n_in + n_out) = %lld floats required, got %lld",
                need, part_floats);
  if (backend != SWINB200_GEMM_TCGEN05 || n_out % 256 != 0 || n_in < 256) {
    set_error("linear_wgrad_det: tcgen05 / bf16 only, n_out a multiple of 256 and n_in >= 256 (backend %d, n_out = %d, n_in = %d)",
              backend, n_out, n_in);
    return SWINB200_ERR_UNSUPPORTED;
  }
  return gemm_tcgen05(n_out, n_in, T, dY, 1, ldy, X, 1, ldx, SWINB200_EPI_F32, nullptr, dW, n_in, nullptr, nullptr, 0, 1, split_k,
                      (cudaStream_t)stream, nullptr, dbias, part);
}
