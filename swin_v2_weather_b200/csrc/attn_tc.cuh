// Shared pieces of the tcgen05 window-attention kernels: attn_tc_fwd4.cu and attn_tc_bwd3.cu (9x18 windows, head_dim 96),
// attn_tc_gen.cu (every other geometry) and the dispatch in attn_tc.cu.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace swinb200 {
using namespace ptx;

constexpr int kMaxLP = 176;  // padded keys per window (multiple of 16); 9x18 = 162 -> 176


__host__ __device__ constexpr uint64_t umma_desc_nosw(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

struct AttnGeom {
  int B, H, W, C, heads, Wh, Ww, s0, s1;
  int L, LP, nW, nWw;
};

__device__ __forceinline__ int win_token(const AttnGeom& g, int b, int w, int n, int& rolled_row) {
  const int wh = w / g.nWw, ww = w - wh * g.nWw;
  const int a = n / g.Ww, c = n - a * g.Ww;
  rolled_row = wh * g.Wh + a;
  int i = rolled_row + g.s0;
  if (i >= g.H) i -= g.H;
  int j = ww * g.Ww + c + g.s1;
  if (j >= g.W) j -= g.W;
  return (b * g.H + i) * g.W + j;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float as_f(uint32_t u) { return __uint_as_float(u); }
__device__ __forceinline__ uint4 pack8(const float (&v)[16], int o) {
  uint4 r;
  r.x = pack_bf16x2(v[o + 0], v[o + 1]); r.y = pack_bf16x2(v[o + 2], v[o + 3]);
  r.z = pack_bf16x2(v[o + 4], v[o + 5]); r.w = pack_bf16x2(v[o + 6], v[o + 7]);
  return r;
}


__device__ __forceinline__ void tmem_st_32x4(uint32_t taddr, const uint4& v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint4& a, const uint4& b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(a.x), "r"(a.y),
               "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}


constexpr int kCS64 = kMaxLP * 64;          // chunk stride: 11,264 B = 22 x 512
__host__ __device__ constexpr uint64_t umma_desc_sw64(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (4ull << 61) /* SWIZZLE_64B */;
}
__device__ __forceinline__ uint64_t opnd_kmajor(uint32_t base, int k, int row0) {   // k-th 16-wide k step, rows from row0
  return umma_desc_sw64(base + (uint32_t)((k >> 1) * kCS64 + (k & 1) * 32 + row0 * 64), 16, 512);
}
__device__ __forceinline__ uint64_t opnd_mnmajor(uint32_t base, int k) {             // k-th group of 16 rows (= k dimension)
  return umma_desc_sw64(base + (uint32_t)(k * 1024), kCS64, 512);
}
// byte offset of the 16-byte piece `piece` (0..11) of row `row` inside an operand tile
__device__ __forceinline__ uint32_t opnd_off(int row, int piece) {
  return (uint32_t)((piece >> 2) * kCS64 + row * 64 + (((piece & 3) ^ ((row >> 1) & 3)) << 4));
}

__device__ __forceinline__ void tma_load_5d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}


bool attn_gen_supports(int head_dim);
int attn_tcgen05_gen_fwd(const void* qkv, const float* scale, const float* bias, void* o, float* lse, const AttnGeom& g, cudaStream_t stream);
// det_part (deterministic mode, see swinb200_window_attn_bwd_det): attn_det_dscale_slots(g) d(scale) slots, followed (with a
// bias table) by the (B*nW*heads, L, L) per-item d(bias) slices
int attn_tcgen05_gen_bwd(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o, const void* d_o,
                         const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, const AttnGeom& g, cudaStream_t stream,
                         float* det_part = nullptr);
int attn_make_geom(AttnGeom& g, int B, int H, int W, int C, int heads, int Wh, int Ww, int s0, int s1);
int attn_make_window_tmap(CUtensorMap* m, const void* base, int B, int H, int W, int channels, int Wh, int Ww);
int attn_tcgen05_fwd4(const void* qkv, const float* scale, const float* bias, void* o, float* lse, const AttnGeom& g, cudaStream_t stream);
int attn_tcgen05_bwd3(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o, const void* d_o,
                      const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, const AttnGeom& g, cudaStream_t stream,
                      float* det_part = nullptr);
// D[t, h] = <dO[t, h, :], O[t, h, :]> over n_pairs (token, head) rows of d elements: the backward's pre-pass into ws
__global__ void attn_rowdot_kernel(const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o, float* __restrict__ out,
                                   long long n_pairs, int d);
// one slot per (item, 128-row tile, warp of attn_tc_gen.cu) -- enough for every back end
inline long long attn_det_dscale_slots(const AttnGeom& g) { return (long long)g.B * g.nW * g.heads * 4 * ((g.L + 127) / 128); }

}  // namespace swinb200
