// tcgen05 windowed cosine attention for sm_100a: dispatch to the kernels and the pieces they share.
//
// Two kernel families: the tuned 9x18 / head_dim-96 kernels (attn_tc_fwd4.cu, attn_tc_bwd3.cu) and the generic ones for every
// other geometry (attn_tc_gen.cu).  The cyclic shift, window partition and window reverse of the reference
// (swinv2_global.py:89-119, 446-478) are folded into their gather / scatter addressing (win_token, attn_make_window_tmap), so no
// rolled or permuted copy ever reaches HBM.
#include "attn_tc.cuh"

namespace swinb200 {

int attn_set_phase_buffer3(long long* buf);

int attn_make_geom(AttnGeom& g, int B, int H, int W, int C, int heads, int Wh, int Ww, int s0, int s1) {
  g.B = B; g.H = H; g.W = W; g.C = C; g.heads = heads; g.Wh = Wh; g.Ww = Ww; g.s0 = s0; g.s1 = s1;
  g.L = Wh * Ww;
  g.LP = (g.L + 15) / 16 * 16;
  g.nWw = W / Ww;
  g.nW = (H / Wh) * g.nWw;
  if (!attn_gen_supports(C / heads)) {
    set_error("window_attn (tcgen05): head_dim %d is not instantiated (48, 64, 96, 128, 192, 256)", C / heads);
    return SWINB200_ERR_UNSUPPORTED;
  }
  return SWINB200_OK;
}
// the tuned kernels: head_dim 96 and windows of up to 176 (padded) tokens -- the shipped 9x18 configuration
static bool attn_is_specialised(const AttnGeom& g) { return g.C / g.heads == 96 && g.LP <= kMaxLP && g.LP >= 16; }

// The tcgen05 kernels move qkv / o / d_o / dqkv rows in 16-byte pieces (TMA boxes, cp.async, uint4 loads and stores); row
// strides are multiples of 8 elements, so an aligned base keeps every piece aligned.
static bool aligned16(const void* p) { return (uintptr_t)p % 16 == 0; }

int attn_tcgen05_fwd(const void* qkv, const float* scale, const float* bias, void* o, float* lse, int B, int H, int W, int C,
                     int heads, int Wh, int Ww, int s0, int s1, cudaStream_t stream) {
  SWB_CHECK_ARG(aligned16(qkv) && aligned16(o), "window_attn_fwd (tcgen05): qkv and o must be 16-byte aligned");
  AttnGeom g;
  if (int e = attn_make_geom(g, B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  // with a bias table the tiled kernel is the faster forward on every geometry (434 vs 660 us at 9x18 / 8 heads): its table
  // values are prefetched and reach their rows through a shared-memory slab; the persistent kernel reads them row by row
  if (attn_is_specialised(g) && bias == nullptr) return attn_tcgen05_fwd4(qkv, scale, bias, o, lse, g, stream);
  return attn_tcgen05_gen_fwd(qkv, scale, bias, o, lse, g, stream);
}

// D[t, h] = <dO[t, h, :], O[t, h, :]>  (the softmax-backward row term), four lanes per (token, head)
__global__ void __launch_bounds__(256) attn_rowdot_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o,
                                                          float* __restrict__ out, long long n_pairs, int d) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long pair = gid >> 2;
  const int q = (int)(gid & 3);
  float acc = 0.f;
  if (pair < n_pairs) {
    const __nv_bfloat16* a = o + pair * d;
    const __nv_bfloat16* b = d_o + pair * d;
    for (int c = q * 8; c < d; c += 32) {
      float a8[8], b8[8];
      ld8(a + c, a8);
      ld8(b + c, b8);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc = fmaf(a8[e], b8[e], acc);
    }
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  if (q == 0 && pair < n_pairs) out[pair] = acc;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_tiled();

// (B, H, W, channels) bf16 activation seen as [32 | channels/32 | W | H | B]; one box = a 32-channel (64-byte) column of a
// window, written 64B-swizzled
int attn_make_window_tmap(CUtensorMap* m, const void* base, int B, int H, int W, int channels, int Wh, int Ww) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return SWINB200_ERR_CUDA;
  }
  const cuuint64_t row = (cuuint64_t)channels * 2;
  cuuint64_t dims[5] = {32, (cuuint64_t)channels / 32, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[4] = {64, row, row * W, row * W * H};
  cuuint32_t box[5] = {32, 1, (cuuint32_t)Ww, (cuuint32_t)Wh, 1};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (window map) failed (%d)", (int)r);
    return SWINB200_ERR_CUDA;
  }
  return SWINB200_OK;
}

// ws: workspace of B*H*W*heads floats for D = <dO, O>, formed by a streaming pre-pass (attn_rowdot_kernel)
int attn_tcgen05_bwd(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o,
                     const void* d_o, const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, int B, int H, int W,
                     int C, int heads, int Wh, int Ww, int s0, int s1, cudaStream_t stream, float* det_part) {
  SWB_CHECK_ARG(ws != nullptr, "window_attn_bwd (tcgen05): a workspace of B*H*W*heads floats is required");
  SWB_CHECK_ARG(aligned16(qkv) && aligned16(o) && aligned16(d_o) && aligned16(dqkv),
                "window_attn_bwd (tcgen05): qkv, o, d_o and dqkv must be 16-byte aligned");
  AttnGeom g;
  if (int e = attn_make_geom(g, B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  if (attn_is_specialised(g))
    return attn_tcgen05_bwd3(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, ws, g, stream, det_part);
  return attn_tcgen05_gen_bwd(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, ws, g, stream, det_part);
}

}  // namespace swinb200

extern "C" int swinb200_debug_attn_phase_buffer(void* buf) { return swinb200::attn_set_phase_buffer3((long long*)buf); }
