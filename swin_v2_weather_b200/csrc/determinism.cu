// Fixed-order second stage of the deterministic-mode reductions.  In deterministic mode every kernel that would sum floats
// with atomics (split-K weight gradients, bias / LayerNorm parameter gradients, loss and metric sums, attention d(scale)
// and d(bias)) instead writes each partial with a plain store to a slot whose index is fixed by the problem -- a split, a
// statically assigned CTA, a (sample, window, head) item, a row block -- and this kernel adds the slots in index order.
// The result depends only on the inputs and the launch geometry, never on which CTA or warp finished first.
#include <algorithm>

#include "common.cuh"

namespace swinb200 {

__global__ void __launch_bounds__(256) ordered_reduce_kernel(const float* __restrict__ part, int n_part, long long stride, long long n,
                                                             int inner, float* __restrict__ out, int accumulate) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int p = 0; p < n_part; ++p) {
      const float* src = part + p * stride + i * inner;
      for (int j = 0; j < inner; ++j) s += __ldg(src + j);
    }
    out[i] = accumulate ? out[i] + s : s;
  }
}

int ordered_reduce(const float* part, int n_part, long long stride, long long n, int inner, float* out, int accumulate,
                   cudaStream_t stream) {
  SWB_CHECK_ARG(part && out && n_part > 0 && n > 0 && inner > 0 && stride >= n * inner,
                "ordered_reduce: bad arguments n_part=%d stride=%lld n=%lld inner=%d", n_part, stride, n, inner);
  const long long blocks = std::min<long long>((n + 255) / 256, (long long)sm_count() * 16);
  ordered_reduce_kernel<<<(unsigned)blocks, 256, 0, stream>>>(part, n_part, stride, n, inner, out, accumulate);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

}  // namespace swinb200

extern "C" int swinb200_ordered_reduce(const float* part, int n_part, long long stride, long long n, int inner, float* out,
                                       int accumulate, void* stream) {
  return swinb200::ordered_reduce(part, n_part, stride, n, inner, out, accumulate, (cudaStream_t)stream);
}
