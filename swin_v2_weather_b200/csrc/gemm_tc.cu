// tcgen05 GEMM for sm_100a:  D[M,N] = epilogue( sum_k A(m,k) * B(n,k) ),  bf16 operands, fp32 accumulation in TMEM.
//
// Persistent, warp-specialised, one CTA per SM (576 threads):
//   warps 0..15 epilogue       (four groups of 4 warps; group g owns every fourth 64-byte column chunk of the tile:
//                               tcgen05.ld -> fused epilogue in registers -> swizzled smem staging -> TMA store /
//                               TMA reduce-add, so global writes are whole 64-byte row pieces issued by the copy engine)
//   warp 16     TMA producer   (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier complete_tx)
//   warp 17     MMA issuer     (tcgen05.mma 128 x BN x 16 by one elected lane, accumulators double-buffered in TMEM)
// The two single-lane roles sit in the HIGHEST warp ids of their scheduler partitions: the issue arbiter favours the
// highest warp id, and the MMA loop is latency-critical (its ~40 instructions per k-block must not queue behind the
// epilogue warps' arithmetic, which is what capped the GELU GEMMs at 54 % tensor-pipe activity).  Both loops run
// warp-convergent with the issuing lane elected per instruction, so descriptors live in uniform registers.
// Tile scheduling (CTA pairs): the grid has one cluster per output tile; the 74 resident clusters keep their TMEM,
// barriers and pipeline state and obtain further tiles by cancelling pending clusters (clusterlaunchcontrol.try_cancel),
// one query ahead of the producer.  SMs that are busy with another kernel (NCCL's all-reduce CTAs during the backward of
// a data-parallel step) simply take no tiles, instead of stalling a static round-robin schedule until they are free.
// Operand majors: K-major (row = m/n, 64 k per 128-byte row) or MN-major (row = k, 64 m/n per 128-byte row),
// so nn.Linear forward (A k-major, B k-major), dgrad (B = weight read n-major) and wgrad (both operands
// token-major, reduction over tokens, split-K with fp32 TMA reduce-add) all run without transposed copies.
// Side work of the epilogue warps: (i) weight gradients -- the bias gradient (column sums of the m-major A operand) is taken
// from the staged A tiles while the main loop runs (GemmTcParams::colsum_out, entry point swinb200_linear_wgrad);
// (ii) BIAS_LN -- LayerNorm + DropPath scale + residual of every finished 128-row block (swinb200_linear_ln_residual; opt-in,
// measured slower than the stand-alone LayerNorm kernel).
#include <cuda.h>
#include <stdlib.h>
#include "common.cuh"
#include "ptx.cuh"

namespace swinb200 {

using namespace ptx;

constexpr int GBM = 128;  // UMMA M (cta_group::1)
constexpr int GBK = 64;   // k per pipeline stage (one 128-byte swizzle row of bf16)
constexpr int kEpiGroups = 4;             // epilogue groups of 4 warps (one warp per TMEM lane quarter)
constexpr int kGemmThreads = 64 + kEpiGroups * 128;
constexpr int kProducerWarp = kEpiGroups * 4, kMmaWarp = kEpiGroups * 4 + 1;
constexpr int kStagingBytes = 32 * 64;     // one [32 rows x 64 B] output piece per epilogue WARP
constexpr int kStagingBufs = 2;            // staging buffers per warp: a store only waits for the one before the previous one
constexpr int kBiasBytes = 2048;           // per-group bias slices (<= 64 floats per group), double-buffered by tile parity

struct GemmTcParams {
  int M, N, K;
  const float* bias;
  const void* aux;
  float* inv_norm;   // BIAS_QKNORM: (M, 2*N/(3*96)) reciprocal L2 norms of the q / k head vectors, or null (not stored)
  int ld_aux;
  int pair;        // 1 = CTA-pair (cta_group::2) launch: 256 x 256 tiles over two SMs
  int debug;       // bring-up timing experiments (SWINB200_GEMM_DEBUG): 1 = no staging wait, 2 = no store, 4 = no tmem ld wait
  int atomic_out;  // EPI_F32: 1 = TMA reduce-add (split-K / accumulate), 0 = plain TMA store
  int num_m_tiles, num_n_tiles, split_k, kb_total, kb_per_split;
  // BIAS_LN: post-norm LayerNorm + DropPath scale + residual add of finished 128-row blocks, inside the epilogue
  const float* ln_x_in;           // (M, N) fp32 residual stream
  const float* ln_gamma;          // (N)
  const float* ln_beta;           // (N)
  const float* ln_sample_scale;   // (M / rows_per_sample) DropPath multipliers or null
  float* ln_x_out;                // (M, N) fp32
  __nv_bfloat16* ln_xb_out;       // (M, N) bf16 shadow
  float* ln_stats;                // (M, 2) mean, rstd
  const __nv_bfloat16* ln_z;      // D as the epilogue warps re-read it (ldd pitch)
  int ln_ldz;
  int* ln_counters;               // one per 128-row block, zero on entry and on exit
  int ln_rows_per_sample;
  float ln_eps;
  int ln_slices;                  // 32-row LayerNorm slices a CTA may run per tile boundary
  float* colsum_out;              // weight-gradient GEMMs (A m-major): column sums of A (= bias gradient) += here, or null
};

// PAIR: two CTAs of a cluster (two SMs) share one 256 x BN tile: tcgen05.mma.cta_group::2 reads the A rows and one half
// of the B columns from each CTA's shared memory, so every SM stages (and the tensor core re-reads) a third less operand
// data per k-step and the smem ring gets deeper.
template <int BN, bool PAIR = false, bool LN = false>
struct GemmCfg {
  static constexpr int kStageA = GBM * GBK * 2;
  static constexpr int kStageB = (PAIR ? BN / 2 : BN) * GBK * 2;
  static constexpr int kStage = kStageA + kStageB;
  static constexpr int kStages = LN ? (PAIR ? 4 : 3) : (PAIR ? 5 : ((BN >= 192) ? 3 : 5));   // 5 x 32 KB stages + 64 KB of staging fill the SM; BIAS_LN: 4 stages, so that 60 KB of L1 remain for the row loads of the LayerNorm pass
  static constexpr int kTmemCols = (2 * BN <= 256) ? 256 : 512;
  // BIAS_LN keeps gamma / beta (up to 1024 channels each) in shared memory and pays for them with the second staging buffer
  static constexpr int kSB = LN ? 1 : kStagingBufs;
  static constexpr int kOffStaging = kStages * kStage;
  static constexpr int kOffBars = kOffStaging + kEpiGroups * 4 * kSB * kStagingBytes;
  static constexpr int kOffBias = kOffBars + 256;
  static constexpr int kOffSsq = kOffBias + kBiasBytes;               // BIAS_QKNORM: [2 tile parities][BN/32 pieces][128 rows] partial sums of squares
  static constexpr int kOffLn = kOffSsq + ((BN == 192) ? 2 * (BN / 32) * GBM * 4 : 0);   // BIAS_LN: gamma[1024], beta[1024], flag
  static constexpr int kOffLnX = kOffLn + 2 * 1024 * 4 + 64;                          // BIAS_LN: one fp32 row of x_in per epilogue warp (prefetch)
  static constexpr int kSmem = LN ? kOffLnX + kEpiGroups * 4 * 768 * 4 : kOffLn;
  static_assert(kSmem <= 227 * 1024, "shared memory budget");
};

// GELU in the epilogue has an instruction budget: a 128x256 tile with K = 768 keeps the tensor pipe busy for ~6.1k
// cycles, in which 8 epilogue warps must process 32k elements -> <= ~19 issue slots per element.  erff()/expf() cost
// ~30, so the normal CDF is evaluated as  Phi(x) = 0.5 + xc * P(xc^2),  xc = clamp(x, -4, 4),  with a degree-7 minimax
// polynomial in x^2 (|Phi error| <= 7.5e-5 on the clamp range, 3.2e-5 beyond it; the exact-erf CUDA-core kernels remain
// the reference used by the fp32 validation mode).
__device__ __forceinline__ float normal_cdf_fast(float x) {
  const float xc = fminf(fmaxf(x, -4.0f), 4.0f);
  const float u = xc * xc;
  float p = -1.5809101805430714e-09f;
  p = fmaf(p, u, 1.21718073842203e-07f);
  p = fmaf(p, u, -4.101022113900399e-06f);
  p = fmaf(p, u, 8.066916052484885e-05f);
  p = fmaf(p, u, -0.001048215082846582f);
  p = fmaf(p, u, 0.009664907120168209f);
  p = fmaf(p, u, -0.0661754235625267f);
  p = fmaf(p, u, 0.3988475203514099f);
  return fmaf(xc, p, 0.5f);
}
// The multiplier is max(x, -4), not x: below the clamp Phi_fast stays at Phi(-4) = 3.2e-5 instead of decaying, and x * Phi_fast
// would grow linearly with |x|; max(x, -4) * Phi_fast(-4) = -1.3e-4 bounds the tail error (the exact value tends to 0-).
__device__ __forceinline__ float gelu_fast(float x) { return fmaxf(x, -4.0f) * normal_cdf_fast(x); }

// Packed fp32 arithmetic (Blackwell FFMA2 / FMUL2 / FADD2: two fp32 lanes per instruction, operands in 64-bit register
// pairs).  The epilogues are issue-slot bound, so evaluating the polynomial two columns at a time halves their cost.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 splat2(float c) { return pack2(c, c); }
// normal_cdf_fast on two values (same polynomial, same rounding: fma.rn per lane)
__device__ __forceinline__ f32x2 normal_cdf_fast2(float x0, float x1) {
  const f32x2 xc = pack2(fminf(fmaxf(x0, -4.0f), 4.0f), fminf(fmaxf(x1, -4.0f), 4.0f));
  const f32x2 u = mul2(xc, xc);
  f32x2 q = splat2(-1.5809101805430714e-09f);
  q = fma2(q, u, splat2(1.21718073842203e-07f));
  q = fma2(q, u, splat2(-4.101022113900399e-06f));
  q = fma2(q, u, splat2(8.066916052484885e-05f));
  q = fma2(q, u, splat2(-0.001048215082846582f));
  q = fma2(q, u, splat2(0.009664907120168209f));
  q = fma2(q, u, splat2(-0.0661754235625267f));
  q = fma2(q, u, splat2(0.3988475203514099f));
  return fma2(xc, q, splat2(0.5f));
}
__device__ __forceinline__ void gelu_fast2(float x0, float x1, float& g0, float& g1) {
  unpack2(mul2(pack2(fmaxf(x0, -4.0f), fmaxf(x1, -4.0f)), normal_cdf_fast2(x0, x1)), g0, g1);
}
// v{0,1} *= d/dx[x Phi(x)] at h{0,1}
__device__ __forceinline__ void gelu_grad_mul2(float h0, float h1, float& v0, float& v1) {
  const f32x2 x = pack2(h0, h1);
  float a0, a1, e0, e1;
  unpack2(mul2(mul2(x, x), splat2(-0.72134752044448170368f)), a0, a1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(a0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(a1));
  const f32x2 d = fma2(mul2(x, splat2(0.39894228040143267794f)), pack2(e0, e1), normal_cdf_fast2(h0, h1));
  unpack2(mul2(pack2(v0, v1), d), v0, v1);
}
// d/dx [x Phi(x)] = Phi(x) + x phi(x),  phi(x) = exp(-x^2/2) / sqrt(2 pi)
__device__ __forceinline__ float gelu_grad_fast(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752044448170368f));
  return fmaf(x * 0.39894228040143267794f, e, normal_cdf_fast(x));
}
__device__ __forceinline__ void unpack_bf16x2(uint32_t w, float& lo, float& hi) {
  lo = __uint_as_float(w << 16);
  hi = __uint_as_float(w & 0xffff0000u);
}

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// 3-D map [S, M, N]: box depth 1, so the copy engine clips a ragged tile's rows at M inside its own slice
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void group_bar(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }
// one lane of a converged warp (the same lane every time)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ---- cta_group::2 (CTA pair) forms.  Shared-window addresses of the two CTAs of a pair differ in bit 24; clearing it
// addresses the leader (even) CTA's copy of the same variable (CUTLASS: Sm100MmaPeerBitMask).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all MMAs issued so far -> one arrival on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_result, uint32_t ncols) {  // one warp in each CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// ---- cluster launch control: a running cluster cancels a not-yet-launched cluster of the same grid and takes over its
// block index.  The 16-byte response is multicast to the same shared-memory offset of every CTA of the cluster and
// completes 16 bytes on the mbarrier at the same offset in each of them.
__device__ __forceinline__ void clc_try_cancel(void* resp, uint64_t* bar) {
  asm volatile(
      "clusterlaunchcontrol.try_cancel.async.shared::cta.mbarrier::complete_tx::bytes.multicast::cluster::all.b128 [%0], [%1];"
      ::"r"(smem_u32(resp)), "r"(smem_u32(bar))
      : "memory");
}
// -> blockIdx.x of the first CTA of the cancelled cluster, or -1 when nothing was left to cancel
__device__ __forceinline__ int clc_decode(const void* resp) {
  uint32_t ok = 0, x = 0;
  asm volatile(
      "{\n\t.reg .pred p1;\n\t.reg .b128 r;\n\t"
      "ld.shared.b128 r, [%2];\n\t"
      "clusterlaunchcontrol.query_cancel.is_canceled.pred.b128 p1, r;\n\t"
      "selp.u32 %1, 1, 0, p1;\n\t"
      "@p1 clusterlaunchcontrol.query_cancel.get_first_ctaid.v4.b32.b128 {%0, _, _, _}, r;\n\t}"
      : "+r"(x), "=r"(ok)
      : "r"(smem_u32(resp))
      : "memory");
  return ok ? (int)x : -1;
}

// 16-byte chunk `c` (0..3) of the 64-byte staging row `r`, 64B-swizzled exactly as the TMA store expects
// (address bits [4,6) ^= bits [7,9)); eight consecutive rows land in eight distinct 16-byte bank groups.
__device__ __forceinline__ unsigned char* staging_chunk(unsigned char* buf, int r, int c) {
  return buf + r * 64 + ((c ^ ((r >> 1) & 3)) << 4);
}

// DET (split-K weight gradients in deterministic mode): split ks stores its fp32 tile into slice ks of a [S, M, N] scratch
// (tmD is then a 3-D map) and its column sums into row ks of an [S, M] scratch; swinb200_ordered_reduce adds them up.
template <int BN, bool A_MN, bool B_MN, int EPI, bool PAIR, bool DET = false>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmD2, const GemmTcParams p) {
  constexpr bool kLn = (EPI == SWINB200_EPI_BIAS_LN);
  using Cfg = GemmCfg<BN, PAIR, kLn>;
  constexpr int kSB = Cfg::kSB;                        // staging buffers per epilogue warp
  constexpr int BNL = PAIR ? BN / 2 : BN;              // B columns staged by this CTA
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u; // 0 = leader (issues the MMAs), 1 = peer
  const int cta_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;   // persistent stride in tiles
  const int cta_first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  constexpr bool kF32Out = (EPI == SWINB200_EPI_ADD_F32 || EPI == SWINB200_EPI_F32);
  constexpr int kChunkCols = kF32Out ? 16 : 32;          // 64 bytes of output per row per chunk
  constexpr int kNumChunks = BN / kChunkCols;
  constexpr bool kHasAux = (EPI == SWINB200_EPI_DGELU || EPI == SWINB200_EPI_ADD_F32);
  extern __shared__ __align__(1024) unsigned char smem[];   // 128B-swizzled stages need 1024-byte alignment
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBars);
  uint64_t* full_bar = bars;                       // [kStages]
  uint64_t* empty_bar = bars + Cfg::kStages;       // [kStages]
  uint64_t* tfull_bar = bars + 2 * Cfg::kStages;   // [2]
  uint64_t* tempty_bar = tfull_bar + 2;            // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  static_assert((2 * Cfg::kStages + 4) * 8 + 4 <= 128, "pipeline barriers overflow their 128 bytes");
  constexpr int kSched = 4;                                                           // tile-id ring (CLC responses)
  unsigned char* clc_resp = smem + Cfg::kOffBars + 128;                               // [kSched] x 16 bytes
  uint64_t* sfull = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBars + 192);          // [kSched] response has landed
  uint64_t* sempty = sfull + kSched;                                                  // [kSched] every role has read it (leader's copy)

  // Weight gradients (A = dY read m-major): the bias gradient is the column sum of dY, i.e. the sum over k of the very A tiles
  // this kernel stages.  The epilogue warps, idle during the main loop, add up every stage after its MMAs have completed and
  // before the producer refills it (tiles of the first column block only), so dY is not read a third time from HBM by a
  // separate column-sum kernel.  cs_bar[stage]: the 16 epilogue warps are done with the stage.
  constexpr bool kCanCs = A_MN && B_MN && PAIR && (EPI == SWINB200_EPI_F32) && (BN == 256);
  const bool cs_on = kCanCs && p.colsum_out != nullptr;
  uint64_t* cs_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kOffBias);     // the bias table is unused by this epilogue

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == kProducerWarp && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmD);
    if (EPI == SWINB200_EPI_BIAS_GELU) prefetch_tmap(&tmD2);
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], (PAIR ? 2 : 1) * 4 * kEpiGroups);   // PAIR: both CTAs' epilogue warps report to the leader
    }
    if (kCanCs) {
      for (int s = 0; s < Cfg::kStages; ++s) mbar_init(&cs_bar[s], 4 * kEpiGroups);
    }
    if (PAIR) {
      for (int q = 0; q < kSched; ++q) {
        mbar_init(&sfull[q], 1);
        mbar_init(&sempty[q], 2 * (1 + 4 * kEpiGroups) + 1);       // producer + epilogue warps of both CTAs, MMA warp
      }
    }
    fence_barrier_init();
    if (PAIR)
      for (int q = 0; q < kSched; ++q) mbar_arrive_expect_tx(&sfull[q], 16);   // armed for the first kSched responses
  }
  if (warp == kMmaWarp) {
    if (PAIR) tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
    else tmem_alloc(tmem_slot, Cfg::kTmemCols);
  }
  if (kLn) {
    float* sg = reinterpret_cast<float*>(smem + Cfg::kOffLn);
    for (int i = threadIdx.x; i < p.N; i += kGemmThreads) {
      sg[i] = __ldg(p.ln_gamma + i);
      sg[1024 + i] = __ldg(p.ln_beta + i);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();     // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int num_tiles = p.num_m_tiles * p.num_n_tiles * p.split_k;
  // tile after the i-th one this role has processed (-1: none).  Called by whole, converged warps.
  auto next_tile = [&](int tile, int i, bool rearm) -> int {
    if (!PAIR) {
      const int t = tile + cta_stride;
      return t < num_tiles ? t : -1;
    }
    const int q = i & (kSched - 1);
    mbar_wait(&sfull[q], (uint32_t)((i / kSched) & 1), 700 + q);
    const int bid = clc_decode(clc_resp + q * 16);
    fence_proxy_async_smem();                       // the read is ordered before the next asynchronous overwrite
    if (rearm && elect_one()) mbar_arrive_expect_tx(&sfull[q], 16);   // this CTA's barrier, for response i + kSched
    __syncwarp();
    if (lane == 0) mbar_arrive_leader(&sempty[q]);
    return bid < 0 ? -1 : (bid >> 1);
  };

  if (warp == kProducerWarp) {
    // =============================== TMA producer (warp-convergent, one elected lane issues) ====================
    int stage = 0;
    uint32_t phase = 0;
    int local = 0;
    for (int tile = cta_first; tile >= 0; tile = next_tile(tile, local, true), ++local) {
      if (PAIR && crank == 0) {
        // scheduler: ask for the tile after this one while this one's loads are issued
        const int q = local & (kSched - 1);
        if (local >= kSched) mbar_wait(&sempty[q], (uint32_t)((local / kSched - 1) & 1), 720 + q);
        if (elect_one()) clc_try_cancel(clc_resp + q * 16, &sfull[q]);
        __syncwarp();
      }
      const int ks = tile % p.split_k;
      const int rest = tile / p.split_k;
      const int n0 = (rest % p.num_n_tiles) * BN + (int)crank * BNL;            // PAIR: this CTA's half of the B columns
      const int m0 = (rest / p.num_n_tiles) * (PAIR ? 2 * GBM : GBM) + (int)crank * GBM;
      const int kb0 = ks * p.kb_per_split;
      const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1, 100 + stage);
        if (kCanCs && cs_on) mbar_wait(&cs_bar[stage], phase ^ 1, 110 + stage);
        if (elect_one()) {
          unsigned char* sa = smem + stage * Cfg::kStage;
          unsigned char* sb = sa + Cfg::kStageA;
          // PAIR: every load of both CTAs completes on the leader's barrier, which expects both CTAs' bytes
          if (!PAIR) mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStage);
          else if (crank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::kStage);
          const int k0 = kb * GBK;
          auto load = [&](void* dst, const CUtensorMap* tm, int c0, int c1) {
            if (PAIR) tma_load_2d_pair(dst, tm, &full_bar[stage], c0, c1);
            else tma_load_2d(dst, tm, &full_bar[stage], c0, c1);
          };
          if (!A_MN) {
            load(sa, &tmA, k0, m0);  // box {64 k, 128 m}
          } else {
#pragma unroll
            for (int c = 0; c < GBM / 64; ++c)  // box {64 m, 64 k}
              load(sa + c * (64 * GBK * 2), &tmA, m0 + c * 64, k0);
          }
          if (!B_MN) {
            load(sb, &tmB, k0, n0);  // box {64 k, BNL n}
          } else {
#pragma unroll
            for (int c = 0; c < BNL / 64; ++c)  // box {64 n, 64 k}
              load(sb + c * (64 * GBK * 2), &tmB, n0 + c * 64, k0);
          }
        }
        __syncwarp();
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == kMmaWarp) {
    if (crank == 0) {
      // =============================== MMA issuer (leader CTA only in PAIR mode) =================================
      constexpr uint32_t idesc = umma_idesc_bf16(PAIR ? 2 * GBM : GBM, BN, A_MN, B_MN);
      // K-major: 8-row groups 1024 B apart, k advances 32 B inside the swizzle row.
      // MN-major: 8-k groups 1024 B apart, 64-wide m/n chunks 64*128 B apart, k advances 16 rows = 2048 B.
      // Descriptors are built once; stage and k only move the 16-byte-unit start address in the low word.
      constexpr uint32_t kLboMn = 64 * GBK * 2;
      const uint32_t smem0 = smem_u32(smem);
      const uint64_t adesc0 = A_MN ? umma_smem_desc_sw128(smem0, kLboMn, 1024) : umma_smem_desc_sw128(smem0, 16, 1024);
      const uint64_t bdesc0 = B_MN ? umma_smem_desc_sw128(smem0 + Cfg::kStageA, kLboMn, 1024)
                                   : umma_smem_desc_sw128(smem0 + Cfg::kStageA, 16, 1024);
      constexpr uint32_t kAStep = (A_MN ? 2048 : 32) >> 4, kBStep = (B_MN ? 2048 : 32) >> 4;
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      for (int tile = cta_first; tile >= 0; tile = next_tile(tile, local, false), ++local) {
        const int ks = tile % p.split_k;
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        const int buf = local & 1;
        const uint32_t use = (uint32_t)(local >> 1);
        mbar_wait(&tempty_bar[buf], (use & 1) ^ 1, 200 + buf);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(buf * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase, 300 + stage);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t ad = adesc0 + (uint64_t)(stage * (Cfg::kStage >> 4));
            const uint64_t bd = bdesc0 + (uint64_t)(stage * (Cfg::kStage >> 4));
#pragma unroll
            for (int k = 0; k < GBK / 16; ++k) {
              if (PAIR) umma_bf16_ss_pair(tmem_d, ad + k * kAStep, bd + k * kBStep, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
              else umma_bf16_ss(tmem_d, ad + k * kAStep, bd + k * kBStep, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            }
            // frees the smem stage (in both CTAs of a pair) once these MMAs have read it
            if (PAIR) umma_commit_pair(&empty_bar[stage]); else umma_commit(&empty_bar[stage]);
            // accumulator complete -> epilogue (of both CTAs)
            if (kb == kb1 - 1) { if (PAIR) umma_commit_pair(&tfull_bar[buf]); else umma_commit(&tfull_bar[buf]); }
          }
          __syncwarp();
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ================================= epilogue ===================================
    const int ew = warp;                   // 0 .. 4*kEpiGroups-1
    const int grp = ew >> 2;               // epilogue group: owns chunks grp, grp + kEpiGroups, ...
    const int quarter = warp & 3;          // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;     // row inside the tile
    const int gt = threadIdx.x & 127;      // thread index inside the group (group g = warps 4g .. 4g+3)
    unsigned char* stg_base = smem + Cfg::kOffStaging + ew * kSB * kStagingBytes;
    uint32_t stg_sel = 0;                  // staging buffer of the next piece
    // Each warp stages and stores its own 32 rows: no cross-warp barrier sits between tcgen05.ld and the TMA store.
    constexpr bool kBiasEpi = (EPI == SWINB200_EPI_BIAS || EPI == SWINB200_EPI_BIAS_GELU || EPI == SWINB200_EPI_BIAS_GELU_FWD ||
                               EPI == SWINB200_EPI_BIAS_QKNORM || kLn);
    constexpr int kChunksPerGroup = (kNumChunks + kEpiGroups - 1) / kEpiGroups;
    constexpr int kBiasSlots = kChunksPerGroup * kChunkCols;
    static_assert(!kBiasEpi || kBiasSlots <= 64, "bias slices must fit");
    float* sbias_grp = reinterpret_cast<float*>(smem + Cfg::kOffBias) + grp * 64;   // + 256 floats for odd tiles
    const bool has_bias = kBiasEpi && p.bias != nullptr;
    const int mrow0 = quarter * 32;        // first tile row of this warp
    int qk_tiles = 0;                      // BIAS_QKNORM: tiles that exchanged norms so far
    int cs_stage = 0;                      // column sums of A: the stage / phase the main loop is at (all tiles, all k blocks)
    uint32_t cs_phase = 0;
    // ---- BIAS_LN: x_out = x_in + s * (LN(z) gamma + beta) for a 128-row block whose last column tile has just landed ----------
    // Every CTA counts the tiles it has *completely* written (all 16 warps' TMA stores finished) per 128-row block; the CTA
    // that brings a block's count to num_n_tiles re-reads the block's bf16 rows of z (L2-hot, written by up to three SMs)
    // and runs the row routine of ln_residual_fwd_kernel, warp per row, while the MMA warp is already filling the next
    // accumulators.  The bookkeeping runs one tile behind so that no warp ever waits for its own stores to drain.
    int ln_prev_blk = -1;
    volatile int* ln_flag = reinterpret_cast<volatile int*>(smem + Cfg::kOffLn + 2 * 1024 * 4);
    auto ln_rows = [&](int blk, int r_begin, int r_end) {
      constexpr int NK = 6;                  // 768 channels: lane owns 4 channels at lane*4 + 128*k (host checks N == 768), so
                                             // every fp32 access is one whole 512-byte line per warp and every bf16 access 256 bytes
      const float* sg = reinterpret_cast<const float*>(smem + Cfg::kOffLn);
      const float invC = 1.0f / (float)p.N;
      // Two rows are in flight per warp: while row i is normalised, row i+1's x_in streams into the warp's shared-memory
      // row (cp.async: no registers) and its z sits in 12 registers.  Every lane reads back exactly the bytes it copied.
      float* xrow = reinterpret_cast<float*>(smem + Cfg::kOffLnX) + ew * 768;
      auto fetch = [&](int row, uint2 (&zn)[NK]) {
        if (row < p.M) {
#pragma unroll
          for (int k = 0; k < NK; ++k) {
            const int c = lane * 4 + k * 128;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(xrow + c)), "l"(p.ln_x_in + (size_t)row * p.N + c) : "memory");
            zn[k] = __ldcg(reinterpret_cast<const uint2*>(p.ln_z + (size_t)row * p.ln_ldz + c));
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      uint2 zn[NK];
      fetch(blk * GBM + r_begin + ew, zn);
      for (int rr = r_begin + ew; rr < r_end; rr += 4 * kEpiGroups) {
        const int row = blk * GBM + rr;
        if (row >= p.M) break;
        uint2 zq[NK];
        float4 xi[NK];
        asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          zq[k] = zn[k];
          xi[k] = *reinterpret_cast<const float4*>(xrow + lane * 4 + k * 128);
        }
        if (rr + 4 * kEpiGroups < r_end) fetch(row + 4 * kEpiGroups, zn);
        float v[NK][4];
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          unpack_bf16x2(zq[k].x, v[k][0], v[k][1]);
          unpack_bf16x2(zq[k].y, v[k][2], v[k][3]);
          sum += (v[k][0] + v[k][1]) + (v[k][2] + v[k][3]);
        }
        const float mean = warp_sum(sum) * invC;
        float sq = 0.f;
#pragma unroll
        for (int k = 0; k < NK; ++k)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float d = v[k][e] - mean;
            sq = fmaf(d, d, sq);
          }
        const float rstd = rsqrtf(warp_sum(sq) * invC + p.ln_eps);
        const float sc = p.ln_sample_scale ? __ldg(p.ln_sample_scale + row / p.ln_rows_per_sample) : 1.0f;
#pragma unroll
        for (int k = 0; k < NK; ++k) {
          const int c = lane * 4 + k * 128;
          const float4 g4 = *reinterpret_cast<const float4*>(sg + c);
          const float4 b4 = *reinterpret_cast<const float4*>(sg + 1024 + c);
          float4 r;
          r.x = fmaf((v[k][0] - mean) * rstd, g4.x, b4.x) * sc + xi[k].x;
          r.y = fmaf((v[k][1] - mean) * rstd, g4.y, b4.y) * sc + xi[k].y;
          r.z = fmaf((v[k][2] - mean) * rstd, g4.z, b4.z) * sc + xi[k].z;
          r.w = fmaf((v[k][3] - mean) * rstd, g4.w, b4.w) * sc + xi[k].w;
          if (!(p.debug & 16)) {
            *reinterpret_cast<float4*>(p.ln_x_out + (size_t)row * p.N + c) = r;
            uint2 pk;
            pk.x = pack_bf16x2(r.x, r.y);
            pk.y = pack_bf16x2(r.z, r.w);
            *reinterpret_cast<uint2*>(p.ln_xb_out + (size_t)row * p.N + c) = pk;
          }
        }
        if (lane == 0) {
          p.ln_stats[2 * (size_t)row] = mean;
          p.ln_stats[2 * (size_t)row + 1] = rstd;
        }
      }
    };
    // Finished blocks wait in a small queue and are normalised in slices of 32 rows, at most p.ln_slices per tile boundary:
    // the LayerNorm's HBM traffic is spread over the whole kernel instead of arriving in bursts that outlast the two tiles
    // the MMA warp can run ahead.  Queue indices are replicated in every warp (all warps see the same flags); only the
    // block ids live in shared memory.
    constexpr int kLnSliceRows = 32, kLnSlicesPerBlock = GBM / kLnSliceRows, kLnQueue = 8;
    volatile int* ln_q = ln_flag + 1;          // [kLnQueue]
    int q_head = 0, q_tail = 0, q_slice = 0;
    long long ln_cyc = 0, ln_wait_cyc = 0, ln_t0 = clock64();
    int ln_nslices = 0;
    auto ln_run_slices = [&](int max_slices) {
      for (int s_ = 0; s_ < max_slices && q_head != q_tail; ++s_) {
        const long long t0_ = clock64();
        if (!(p.debug & 8)) ln_rows(ln_q[q_head & (kLnQueue - 1)], q_slice * kLnSliceRows, (q_slice + 1) * kLnSliceRows);
        ln_cyc += clock64() - t0_;
        ++ln_nslices;
        if (++q_slice == kLnSlicesPerBlock) { q_slice = 0; ++q_head; }
      }
    };
    auto ln_finish_block = [&](int blk, bool wait_all) {
      if (q_tail - q_head >= kLnQueue - 1) ln_run_slices(kLnSlicesPerBlock);   // never overflows: make room first
      if (lane == 0) {
        // this warp's stores of block `blk`: everything except the groups committed since (two per tile)
        if (wait_all) bulk_wait0();
        else asm volatile("cp.async.bulk.wait_group 2;" ::: "memory");
        asm volatile("fence.proxy.async;" ::: "memory");
        __threadfence();
      }
      __syncwarp();
      asm volatile("bar.sync 6, %0;" ::"r"(kEpiGroups * 128) : "memory");
      if (threadIdx.x == 0) {
        __threadfence();
        const int old = atomicAdd(p.ln_counters + blk, 1);
        const int last = (old == p.num_n_tiles - 1) ? 1 : 0;
        if (last) {
          p.ln_counters[blk] = 0;              // ready for the next launch
          ln_q[q_tail & (kLnQueue - 1)] = blk;
        }
        __threadfence();
        *ln_flag = last;
      }
      asm volatile("bar.sync 6, %0;" ::"r"(kEpiGroups * 128) : "memory");
      if (*ln_flag) ++q_tail;
    };
    int local = 0;
    for (int tile = cta_first; tile >= 0; tile = next_tile(tile, local, false), ++local) {
      const int rest = tile / p.split_k;
      const int n0 = (rest % p.num_n_tiles) * BN;
      const int m0 = (rest / p.num_n_tiles) * (PAIR ? 2 * GBM : GBM) + (int)crank * GBM;
      const int buf = local & 1;
      const uint32_t use = (uint32_t)(local >> 1);
      if (kCanCs && cs_on) {
        // follow the main loop of this tile: stage `cs_stage` is ours between the completion of its MMAs (empty_bar, which
        // the commit multicasts to both CTAs of the pair) and the producer's refill (which waits for cs_bar)
        const int ks_ = tile % p.split_k;
        const int kb0_ = ks_ * p.kb_per_split, kb1_ = min(p.kb_total, kb0_ + p.kb_per_split);
        const bool sum_tile = (n0 == 0);
        // thread <-> (64-column box, 8-row k group, 4-byte word of the 128-byte swizzled row = two columns)
        const int cs_box = ew >> 3, cs_kg = ew & 7;
        float cs0 = 0.f, cs1 = 0.f;
        for (int kb = kb0_; kb < kb1_; ++kb) {
          mbar_wait(&empty_bar[cs_stage], cs_phase, 120 + cs_stage);
          if (sum_tile) {
            const unsigned char* box = smem + cs_stage * Cfg::kStage + cs_box * (64 * GBK * 2);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int k = cs_kg * 8 + j;
              const uint32_t w2 = *reinterpret_cast<const uint32_t*>(box + k * 128 + ((((lane >> 2) ^ (k & 7))) << 4) + (lane & 3) * 4);
              cs0 += __uint_as_float(w2 << 16);
              cs1 += __uint_as_float(w2 & 0xffff0000u);
            }
          }
          fence_proxy_async_smem();            // these generic-proxy reads are ordered before the async-proxy refill
          __syncwarp();
          if (lane == 0) mbar_arrive(&cs_bar[cs_stage]);
          if (++cs_stage == Cfg::kStages) { cs_stage = 0; cs_phase ^= 1; }
        }
        if (sum_tile) {
          // fold the 8 k groups of each box through the (idle) staging buffers, then one atomic per column
          // (every warp parks its partial sums in its OWN staging buffer: only it knows when its stores have drained)
          constexpr int kWarpStg = kSB * kStagingBytes / 4;                       // floats per warp
          float* xch = reinterpret_cast<float*>(smem + Cfg::kOffStaging);
          if (lane == 0) bulk_wait_read0();      // this warp's output pieces of the previous tile have left its staging buffers
          __syncwarp();
          xch[ew * kWarpStg + lane * 2] = cs0;
          xch[ew * kWarpStg + lane * 2 + 1] = cs1;
          asm volatile("bar.sync 7, %0;" ::"r"(kEpiGroups * 128) : "memory");
          const int t_ = threadIdx.x;            // 0 .. 511: threads 0..127 own one column each
          if (t_ < GBM) {
            const int bx = t_ >> 6, wd = (t_ & 63) >> 1, hf = t_ & 1;
            float tot = 0.f;
#pragma unroll
            for (int g8 = 0; g8 < 8; ++g8) tot += xch[(bx * 8 + g8) * kWarpStg + wd * 2 + hf];
            const int col = m0 + t_;
            if constexpr (DET) {
              if (col < p.M) p.colsum_out[(size_t)ks_ * p.M + col] = tot;
            } else {
              if (col < p.M) atomicAdd(p.colsum_out + col, tot);
            }
          }
          asm volatile("bar.sync 7, %0;" ::"r"(kEpiGroups * 128) : "memory");   // before the staging buffers take output pieces
        }
      }
      // this group's slice of the bias vector goes through shared memory (there is no L1 left beside the 225 KB of
      // operand stages, so a per-chunk __ldg would expose an L2 round trip): fetched before the accumulator wait
      float bias_v = 0.f;
      if (kBiasEpi && has_bias && gt < kBiasSlots) {
        const int chb = grp + (gt / kChunkCols) * kEpiGroups;
        const int col = n0 + chb * kChunkCols + (gt % kChunkCols);
        if (chb < kNumChunks && col < p.N) bias_v = __ldg(p.bias + col);
      }
      const long long tw0_ = kLn ? clock64() : 0;
      mbar_wait(&tfull_bar[buf], use & 1, 400 + buf);
      if (kLn) ln_wait_cyc += clock64() - tw0_;
      tc_fence_after();
      // double-buffered by tile parity: a warp can only be one barrier ahead of the slowest warp of its group, so the
      // slice being overwritten (two tiles old) has no readers left
      float* sbias = sbias_grp + (local & 1) * 256;
      if (kBiasEpi && has_bias) {
        if (gt < kBiasSlots) sbias[gt] = bias_v;
        group_bar(1 + grp);
      }
      const int m = m0 + r;
      const bool row_ok = m < p.M;
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * BN);
      // epilogue operand (h for DGELU, the fp32 residual gradient for ADD_F32): 64 bytes per row per chunk, fetched one
      // chunk ahead into registers so its latency hides behind the previous chunk's arithmetic
      if (EPI == SWINB200_EPI_BIAS_QKNORM) {
        // BN = 192 = two heads of 96 columns = six 32-column pieces.  Piece p belongs to group p % 4 (groups 0 and 1 own
        // two pieces, groups 2 and 3 one), so at most 64 accumulator columns are live per thread (the one-head-per-group
        // version held 96 and spilled under the 96-register cap).  The squared norm of a head is the sum of three pieces
        // held by three different groups: partials go through shared memory, one named barrier per tile.
        constexpr int kPiecesPerTile = BN / 32;                      // 6
        const bool normalise = n0 < (p.N / 3) * 2;                    // q and k thirds only (a tile is two whole heads: it never straddles)
        // [piece][row], double-buffered over the tiles that exchange norms: a warp can be at most one barrier ahead
        float* ssq = reinterpret_cast<float*>(smem + Cfg::kOffSsq) + (qk_tiles & 1) * kPiecesPerTile * GBM;
        if (normalise) ++qk_tiles;
        // pass 1: squared-norm partials of this group's pieces (accumulator + bias, nothing kept in registers)
        if (normalise) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int pc = grp + j * kEpiGroups;
            if (pc < kPiecesPerTile && n0 + pc * 32 < p.N) {             // uniform across the group
              uint32_t rr[32];
              tmem_ld_32x32(t_row + pc * 32, rr);
              tmem_ld_wait();
              float ss = 0.f;
#pragma unroll
              for (int g4 = 0; g4 < 8; ++g4) {
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_bias) b4 = *reinterpret_cast<const float4*>(sbias + j * 32 + g4 * 4);
                const float a0 = __uint_as_float(rr[g4 * 4 + 0]) + b4.x, a1 = __uint_as_float(rr[g4 * 4 + 1]) + b4.y;
                const float a2 = __uint_as_float(rr[g4 * 4 + 2]) + b4.z, a3 = __uint_as_float(rr[g4 * 4 + 3]) + b4.w;
                ss = fmaf(a0, a0, ss); ss = fmaf(a1, a1, ss); ss = fmaf(a2, a2, ss); ss = fmaf(a3, a3, ss);
              }
              ssq[pc * GBM + r] = ss;
            }
          }
          asm volatile("bar.sync 5, %0;" ::"r"(kEpiGroups * 128) : "memory");   // all epilogue warps (uniform per tile)
        }
        // pass 2: accumulator again (tensor memory is cheap to re-read, 64 live fp32 values are not under a 96-register
        // cap) + bias, scaled by the head's reciprocal norm, staged and stored
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int pc = grp + j * kEpiGroups;
          const int nb = n0 + pc * 32;
          if (pc < kPiecesPerTile && nb < p.N) {
            uint32_t rr[32];
            tmem_ld_32x32(t_row + pc * 32, rr);
            float inv = 1.0f;
            if (normalise) {
              const int hp = (pc / 3) * 3;                              // first piece of this piece's head
              const float tot = ssq[hp * GBM + r] + ssq[(hp + 1) * GBM + r] + ssq[(hp + 2) * GBM + r];
              inv = 1.0f / fmaxf(sqrtf(tot), 1e-12f);
              if (pc == hp && row_ok && p.inv_norm != nullptr) p.inv_norm[(size_t)m * ((p.N / 3) * 2 / 96) + nb / 96] = inv;
            }
            unsigned char* stg0 = stg_base + (stg_sel & (kSB - 1)) * kStagingBytes;
            stg_sel ^= 1;
            if (lane == 0) { if (kSB == 2) bulk_wait_read1(); else bulk_wait_read0(); }
            __syncwarp();
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              float o8[8];
#pragma unroll
              for (int h2 = 0; h2 < 2; ++h2) {
                float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_bias) b4 = *reinterpret_cast<const float4*>(sbias + j * 32 + c * 8 + h2 * 4);
                o8[h2 * 4 + 0] = (__uint_as_float(rr[c * 8 + h2 * 4 + 0]) + b4.x) * inv;
                o8[h2 * 4 + 1] = (__uint_as_float(rr[c * 8 + h2 * 4 + 1]) + b4.y) * inv;
                o8[h2 * 4 + 2] = (__uint_as_float(rr[c * 8 + h2 * 4 + 2]) + b4.z) * inv;
                o8[h2 * 4 + 3] = (__uint_as_float(rr[c * 8 + h2 * 4 + 3]) + b4.w) * inv;
              }
              uint4 pk;
              pk.x = pack_bf16x2(o8[0], o8[1]); pk.y = pack_bf16x2(o8[2], o8[3]);
              pk.z = pack_bf16x2(o8[4], o8[5]); pk.w = pack_bf16x2(o8[6], o8[7]);
              *reinterpret_cast<uint4*>(staging_chunk(stg0, lane, c)) = pk;
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&tmD, stg0, nb, m0 + mrow0);
              bulk_commit();
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if (PAIR) mbar_arrive_leader(&tempty_bar[buf]); else mbar_arrive(&tempty_bar[buf]); }
        continue;
      }
      // The operand is fetched with lane l on the 16-byte piece (l & 3) of rows (l >> 2) + 8 i: one load instruction covers
      // 8 rows x 64 contiguous bytes.  (Lane = row, four pieces each, is 32 different rows per instruction = 32 L1 tag
      // cycles, 4096 per tile for the 16 warps against 6144 cycles of tensor time.)  The pieces reach the thread that owns
      // their row through the staging buffer this chunk's output will use next.
      uint4 aux_nxt[4];
      auto aux_fetch = [&](int chn) {
        if (kHasAux) {
          const int nbn = n0 + chn * kChunkCols;
          const int piece = lane & 3;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int mr = m0 + mrow0 + i * 8 + (lane >> 2);
            const unsigned char* src = reinterpret_cast<const unsigned char*>(p.aux) + ((size_t)mr * p.ld_aux + nbn) * (kF32Out ? 4 : 2);
            aux_nxt[i] = (mr < p.M && chn < kNumChunks && nbn + piece * (kChunkCols / 4) < p.N)
                             ? __ldg(reinterpret_cast<const uint4*>(src) + piece) : make_uint4(0, 0, 0, 0);
          }
        }
      };
      aux_fetch(grp);
#pragma unroll 1
      for (int ch = grp; ch < kNumChunks; ch += kEpiGroups) {
        const int nb = n0 + ch * kChunkCols;
        if (nb >= p.N) break;                       // whole chunk beyond N (uniform across the group)
        uint4 aux_cur[4];
        if (kHasAux) {
          unsigned char* xb = stg_base + (stg_sel & (kSB - 1)) * kStagingBytes;
          if (lane == 0 && !(p.debug & 1)) { if (kSB == 2) bulk_wait_read1(); else bulk_wait_read0(); }
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(staging_chunk(xb, i * 8 + (lane >> 2), lane & 3)) = aux_nxt[i];
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 4; ++q) aux_cur[q] = *reinterpret_cast<const uint4*>(staging_chunk(xb, lane, q));
          __syncwarp();                             // everyone has its row before the output pieces overwrite the buffer
          aux_fetch(ch + kEpiGroups);
        }
        float v[kChunkCols];
        if (kChunkCols == 32) {
          uint32_t rr[32];
          tmem_ld_32x32(t_row + ch * kChunkCols, rr);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(rr[i]);
        } else {
          uint32_t rr[16];
          tmem_ld_32x16(t_row + ch * kChunkCols, rr);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rr[i]);
        }
        if (kBiasEpi) {
          if (has_bias) {
            const float4* b4p = reinterpret_cast<const float4*>(sbias + ((ch - grp) / kEpiGroups) * kChunkCols);
#pragma unroll
            for (int g = 0; g < kChunkCols / 4; ++g) {
              const float4 b4 = b4p[g];
              unpack2(add2(pack2(v[g * 4 + 0], v[g * 4 + 1]), pack2(b4.x, b4.y)), v[g * 4 + 0], v[g * 4 + 1]);
              unpack2(add2(pack2(v[g * 4 + 2], v[g * 4 + 3]), pack2(b4.z, b4.w)), v[g * 4 + 2], v[g * 4 + 3]);
            }
          }
        } else if (EPI == SWINB200_EPI_DGELU) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {           // 4 x (8 bf16 of h)
            float h8[8];
            unpack_bf16x2(aux_cur[g].x, h8[0], h8[1]); unpack_bf16x2(aux_cur[g].y, h8[2], h8[3]);
            unpack_bf16x2(aux_cur[g].z, h8[4], h8[5]); unpack_bf16x2(aux_cur[g].w, h8[6], h8[7]);
#pragma unroll
            for (int e = 0; e < 8; e += 2) gelu_grad_mul2(h8[e], h8[e + 1], v[g * 8 + e], v[g * 8 + e + 1]);
          }
        } else if (EPI == SWINB200_EPI_ADD_F32) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {           // 4 x (4 fp32)
            v[g * 4 + 0] += __uint_as_float(aux_cur[g].x); v[g * 4 + 1] += __uint_as_float(aux_cur[g].y);
            v[g * 4 + 2] += __uint_as_float(aux_cur[g].z); v[g * 4 + 3] += __uint_as_float(aux_cur[g].w);
          }
        }
        if constexpr (EPI == SWINB200_EPI_BIAS_GELU_FWD) {
          // forward-only fc1: the activation of BIAS_GELU's second pass -- GELU of the bf16-rounded pre-activation, same
          // rounding, same polynomial, so the bits equal BIAS_GELU's D -- in one pass, the pre-activation is never stored
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float h8[8];
            unpack_bf16x2(pack_bf16x2(v[c * 8 + 0], v[c * 8 + 1]), h8[0], h8[1]);
            unpack_bf16x2(pack_bf16x2(v[c * 8 + 2], v[c * 8 + 3]), h8[2], h8[3]);
            unpack_bf16x2(pack_bf16x2(v[c * 8 + 4], v[c * 8 + 5]), h8[4], h8[5]);
            unpack_bf16x2(pack_bf16x2(v[c * 8 + 6], v[c * 8 + 7]), h8[6], h8[7]);
#pragma unroll
            for (int e = 0; e < 8; e += 2) gelu_fast2(h8[e], h8[e + 1], v[c * 8 + e], v[c * 8 + e + 1]);
          }
        }
        // ---- stage this warp's 32 rows of the chunk and hand them to the copy engine; the warp's previous store must
        //      have finished *reading* the buffer.  GELU stores the pre-activation first and evaluates the activation
        //      while the copy engine drains the buffer.
        constexpr int kPasses = (EPI == SWINB200_EPI_BIAS_GELU) ? 2 : 1;
#pragma unroll
        for (int pass = 0; pass < kPasses; ++pass) {
          unsigned char* stg0 = stg_base + (stg_sel & (kSB - 1)) * kStagingBytes;
          stg_sel ^= 1;
          if (lane == 0 && !(p.debug & 1)) { if (kSB == 2) bulk_wait_read1(); else bulk_wait_read0(); }
          __syncwarp();
          uint4 pk[4];
          if (kF32Out) {
#pragma unroll
            for (int c = 0; c < 4; ++c)
              *reinterpret_cast<float4*>(staging_chunk(stg0, lane, c)) = make_float4(v[c * 4], v[c * 4 + 1], v[c * 4 + 2], v[c * 4 + 3]);
          } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              pk[c].x = pack_bf16x2(v[c * 8 + 0], v[c * 8 + 1]); pk[c].y = pack_bf16x2(v[c * 8 + 2], v[c * 8 + 3]);
              pk[c].z = pack_bf16x2(v[c * 8 + 4], v[c * 8 + 5]); pk[c].w = pack_bf16x2(v[c * 8 + 6], v[c * 8 + 7]);
              *reinterpret_cast<uint4*>(staging_chunk(stg0, lane, c)) = pk[c];
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && !(p.debug & 2)) {
            if constexpr (DET) tma_store_3d(&tmD, stg0, nb, m0 + mrow0, tile % p.split_k);
            else if (EPI == SWINB200_EPI_F32 && p.atomic_out) tma_reduce_add_2d(&tmD, stg0, nb, m0 + mrow0);
            else if (EPI == SWINB200_EPI_BIAS_GELU && pass == 0) tma_store_2d(&tmD2, stg0, nb, m0 + mrow0);
            else tma_store_2d(&tmD, stg0, nb, m0 + mrow0);
            bulk_commit();
          }
          if (EPI == SWINB200_EPI_BIAS_GELU && pass == 0) {
            // GELU of the stored (bf16-rounded) pre-activation, so forward and backward see the same h;
            // v[] is overwritten with the activation for the second pass
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              float h8[8];
              unpack_bf16x2(pk[c].x, h8[0], h8[1]); unpack_bf16x2(pk[c].y, h8[2], h8[3]);
              unpack_bf16x2(pk[c].z, h8[4], h8[5]); unpack_bf16x2(pk[c].w, h8[6], h8[7]);
#pragma unroll
              for (int e = 0; e < 8; e += 2) gelu_fast2(h8[e], h8[e + 1], v[c * 8 + e], v[c * 8 + e + 1]);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if (PAIR) mbar_arrive_leader(&tempty_bar[buf]); else mbar_arrive(&tempty_bar[buf]); }
      if (kLn) {
        if (ln_prev_blk >= 0) ln_finish_block(ln_prev_blk, false);
        ln_prev_blk = m0 / GBM;
        ln_run_slices(p.ln_slices);
      }
    }
    if (kLn) {
      const long long tl0_ = clock64();
      if (ln_prev_blk >= 0) ln_finish_block(ln_prev_blk, true);
      ln_run_slices(1 << 20);
      if ((p.debug & 32) && threadIdx.x == 0) {      // probe: per-CTA cycle counts into the head of the stats buffer
        float* o_ = p.ln_stats + (size_t)blockIdx.x * 8;
        o_[0] = (float)(clock64() - ln_t0); o_[1] = (float)ln_cyc; o_[2] = (float)ln_wait_cyc; o_[3] = (float)ln_nslices;
        o_[4] = (float)local; o_[5] = (float)(clock64() - tl0_);
      }
    }
    if (lane == 0) bulk_wait0();   // all global writes of this warp have completed before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();     // neither CTA leaves (or frees tensor memory) while its peer can still touch it
  if (warp == kMmaWarp) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
    else tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---- host side ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && p) fn = (EncodeTiledFn)p;
  }
  return fn;
}

// 2-D tensor map: `inner` contiguous elements, `outer` rows of pitch `ld` elements, 128B swizzle
int make_tmap_2d(CUtensorMap* m, bool f32, const void* base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_inner,
                 uint32_t box_outer, bool swizzle64 = false) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return SWINB200_ERR_CUDA;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims,
                   strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): base=%p inner=%llu outer=%llu ld=%llu box=%ux%u", (int)r, base,
              (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld, box_inner, box_outer);
    return SWINB200_ERR_CUDA;
  }
  return SWINB200_OK;
}

// 3-D fp32 map over `depth` slices of `outer` x `inner` (row pitch `inner`): the partial-sum scratch of DET launches
static int make_tmap_3d_f32(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t depth, uint32_t box_inner,
                            uint32_t box_outer) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return SWINB200_ERR_CUDA;
  }
  cuuint64_t dims[3] = {inner, outer, depth};
  cuuint64_t strides[2] = {inner * 4, inner * outer * 4};
  cuuint32_t box[3] = {box_inner, box_outer, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (3-D) failed (%d): base=%p dims=%llux%llux%llu", (int)r, base, (unsigned long long)inner,
              (unsigned long long)outer, (unsigned long long)depth);
    return SWINB200_ERR_CUDA;
  }
  return SWINB200_OK;
}

template <int BN, bool A_MN, bool B_MN, int EPI, bool PAIR, bool DET = false>
static int launch_tc_impl(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, const CUtensorMap& tmD2,
                          const GemmTcParams& p, cudaStream_t s) {
  using Cfg = GemmCfg<BN, PAIR, EPI == SWINB200_EPI_BIAS_LN>;
  auto kern = gemm_tc_kernel<BN, A_MN, B_MN, EPI, PAIR, DET>;
  static bool configured = false;
  if (!configured) {
    SWB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
    configured = true;
  }
  const int tiles = p.num_m_tiles * p.num_n_tiles * p.split_k;
  if (!PAIR) {
    const int grid = min(tiles, sm_count());
    kern<<<grid, kGemmThreads, Cfg::kSmem, s>>>(tmA, tmB, tmD, tmD2, p);
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * tiles);      // one cluster per tile; resident clusters cancel and absorb the pending ones
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = Cfg::kSmem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SWB_CUDA(cudaLaunchKernelEx(&cfg, kern, tmA, tmB, tmD, tmD2, p));
  }
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

// BN 256 runs as CTA pairs, BN 128 (N <= 128) as single CTAs; p.num_m_tiles counts 256-row pair tiles or 128-row tiles to match
template <int BN, bool A_MN, bool B_MN, int EPI, bool DET = false>
static int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, const CUtensorMap& tmD2,
                     const GemmTcParams& p, cudaStream_t s) {
  return launch_tc_impl<BN, A_MN, B_MN, EPI, BN == 256, DET>(tmA, tmB, tmD, tmD2, p, s);
}

// Only the operand-major / epilogue pairs the model uses are instantiated:
//   forward  (A k-major, B k-major) : BIAS, BIAS_GELU, BIAS_GELU_FWD (forward-only fc1), F32
//   dgrad    (A k-major, B n-major) : BIAS (no bias pointer), DGELU, ADD_F32, F32
//   wgrad    (A m-major, B n-major) : F32 (plain or split-K reduce-add)
template <int BN>
static int dispatch(int epi, int a_major, int b_major, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD,
                    const CUtensorMap& tmD2, const GemmTcParams& p, cudaStream_t s) {
  if (!a_major && !b_major) {
    if (epi == SWINB200_EPI_BIAS) return launch_tc<BN, false, false, SWINB200_EPI_BIAS>(tmA, tmB, tmD, tmD2, p, s);
    if (epi == SWINB200_EPI_BIAS_GELU) return launch_tc<BN, false, false, SWINB200_EPI_BIAS_GELU>(tmA, tmB, tmD, tmD2, p, s);
    if (epi == SWINB200_EPI_BIAS_GELU_FWD) return launch_tc<BN, false, false, SWINB200_EPI_BIAS_GELU_FWD>(tmA, tmB, tmD, tmD2, p, s);
    if (epi == SWINB200_EPI_F32) return launch_tc<BN, false, false, SWINB200_EPI_F32>(tmA, tmB, tmD, tmD2, p, s);
  } else if (!a_major && b_major) {
    if (epi == SWINB200_EPI_BIAS) return launch_tc<BN, false, true, SWINB200_EPI_BIAS>(tmA, tmB, tmD, tmD2, p, s);
    if (epi == SWINB200_EPI_DGELU) return launch_tc<BN, false, true, SWINB200_EPI_DGELU>(tmA, tmB, tmD, tmD2, p, s);
    if (epi == SWINB200_EPI_ADD_F32) return launch_tc<BN, false, true, SWINB200_EPI_ADD_F32>(tmA, tmB, tmD, tmD2, p, s);
    if (epi == SWINB200_EPI_F32) return launch_tc<BN, false, true, SWINB200_EPI_F32>(tmA, tmB, tmD, tmD2, p, s);
  } else if (a_major && b_major) {
    if (epi == SWINB200_EPI_F32) return launch_tc<BN, true, true, SWINB200_EPI_F32>(tmA, tmB, tmD, tmD2, p, s);
  }
  set_error("gemm(tcgen05): combination a_major=%d b_major=%d epilogue=%d is not instantiated", a_major, b_major, epi);
  return SWINB200_ERR_UNSUPPORTED;
}

int gemm_tcgen05(int M, int N, int K, const void* A, int a_major, int lda, const void* B, int b_major, int ldb, int epilogue,
                 const float* bias, void* D, int ldd, void* D2, const void* aux, int ld_aux, int accumulate, int split_k,
                 cudaStream_t stream, const GemmLnFuse* ln, float* colsum_out, float* part) {
  const bool qknorm = (epilogue == SWINB200_EPI_BIAS_QKNORM);
  if (epilogue == SWINB200_EPI_BIAS_LN) {
    SWB_CHECK_ARG(ln != nullptr && ln->x_in && ln->gamma && ln->beta && ln->x_out && ln->xb_out && ln->stats && ln->counters,
                  "gemm(tcgen05): BIAS_LN needs the LayerNorm operands");
    SWB_CHECK_ARG(N == 768 && a_major == 0 && b_major == 0, "gemm(tcgen05): BIAS_LN is instantiated for 768 output channels, forward operand order");
    SWB_CHECK_ARG(ln->n_counters >= (M + GBM - 1) / GBM, "gemm(tcgen05): BIAS_LN needs one counter per 128-row block (%d < %d)",
                  ln->n_counters, (M + GBM - 1) / GBM);
    SWB_CHECK_ARG(((uintptr_t)ln->x_in % 16 == 0) && ((uintptr_t)ln->x_out % 16 == 0) && ((uintptr_t)ln->xb_out % 16 == 0),
                  "gemm(tcgen05): BIAS_LN operands must be 16-byte aligned");
  }
  SWB_CHECK_ARG(lda % 8 == 0 && ldb % 8 == 0, "gemm(tcgen05): lda/ldb must be multiples of 8 elements (16 bytes)");
  SWB_CHECK_ARG(N % 8 == 0 && ldd % 8 == 0, "gemm(tcgen05): N and ldd must be multiples of 8");
  SWB_CHECK_ARG(((uintptr_t)A % 16 == 0) && ((uintptr_t)B % 16 == 0) && ((uintptr_t)D % 16 == 0), "gemm(tcgen05): operands must be 16-byte aligned");
  SWB_CHECK_ARG(aux == nullptr || (((uintptr_t)aux % 16 == 0) && ld_aux % 8 == 0), "gemm(tcgen05): aux must be 16-byte aligned with ld_aux %% 8 == 0");
  SWB_CHECK_ARG(D2 == nullptr || ((uintptr_t)D2 % 16 == 0), "gemm(tcgen05): D2 must be 16-byte aligned");
  SWB_CHECK_ARG(bias == nullptr || ((uintptr_t)bias % 16 == 0), "gemm(tcgen05): bias must be 16-byte aligned");
  SWB_CHECK_ARG(part == nullptr || (epilogue == SWINB200_EPI_F32 && a_major == 1 && b_major == 1 && ((uintptr_t)part % 16 == 0)),
                "gemm(tcgen05): split partials are a weight-gradient (a1, b1, EPI_F32) option and need 16-byte alignment");

  const int BN = qknorm ? 192 : ((N > 128) ? 256 : 128);   // QKNORM: two 96-wide heads per tile
  const bool f32_out = (epilogue == SWINB200_EPI_ADD_F32 || epilogue == SWINB200_EPI_F32);
  GemmTcParams p;
  p.M = M; p.N = N; p.K = K;
  p.bias = bias; p.aux = aux; p.ld_aux = ld_aux;
  {
    static int dbg = -1;
    if (dbg < 0) { const char* e = getenv("SWINB200_GEMM_DEBUG"); dbg = e ? atoi(e) : 0; }
    p.debug = dbg;
  }
  p.inv_norm = qknorm ? reinterpret_cast<float*>(D2) : nullptr;
  p.ln_x_in = nullptr; p.ln_gamma = nullptr; p.ln_beta = nullptr; p.ln_sample_scale = nullptr; p.ln_x_out = nullptr;
  p.ln_xb_out = nullptr; p.ln_stats = nullptr; p.ln_z = nullptr; p.ln_ldz = 0; p.ln_counters = nullptr;
  p.ln_rows_per_sample = 1; p.ln_eps = 0.f; p.ln_slices = 0; p.colsum_out = colsum_out;
  if (part != nullptr) SWB_CHECK_ARG(ldd == N, "gemm(tcgen05): split partials need a dense D (ldd == N)");
  if (epilogue == SWINB200_EPI_BIAS_LN) {
    p.ln_x_in = ln->x_in; p.ln_gamma = ln->gamma; p.ln_beta = ln->beta; p.ln_sample_scale = ln->sample_scale;
    p.ln_x_out = ln->x_out; p.ln_xb_out = reinterpret_cast<__nv_bfloat16*>(ln->xb_out); p.ln_stats = ln->stats;
    p.ln_z = reinterpret_cast<const __nv_bfloat16*>(D); p.ln_ldz = ldd; p.ln_counters = ln->counters;
    p.ln_rows_per_sample = ln->rows_per_sample; p.ln_eps = ln->eps;
    {
      static int sl = -1;
      if (sl < 0) { const char* e = getenv("SWINB200_LN_SLICES"); sl = e ? atoi(e) : 4; }
      p.ln_slices = max(1, sl);
    }
  }
  p.atomic_out = (epilogue == SWINB200_EPI_F32 && (accumulate || split_k > 1)) ? 1 : 0;
  p.pair = (BN == 256 || BN == 192) ? 1 : 0;
  p.num_m_tiles = p.pair ? (M + 2 * GBM - 1) / (2 * GBM) : (M + GBM - 1) / GBM;
  p.num_n_tiles = (N + BN - 1) / BN;
  p.kb_total = (K + GBK - 1) / GBK;
  split_k = max(1, min(split_k, p.kb_total));
  p.kb_per_split = (p.kb_total + split_k - 1) / split_k;
  p.split_k = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;  // no empty splits
  if (part != nullptr && colsum_out != nullptr) p.colsum_out = part + (size_t)p.split_k * M * N;   // [S, M] after the [S, M, N] slices

  CUtensorMap tmA, tmB, tmD, tmD2;
  int e;
  if (!a_major) e = make_tmap_2d(&tmA, false, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, GBK, GBM);
  else e = make_tmap_2d(&tmA, false, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, 64, GBK);
  if (e) return e;
  if (!b_major) e = make_tmap_2d(&tmB, false, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb, GBK, (uint32_t)(p.pair ? BN / 2 : BN));
  else e = make_tmap_2d(&tmB, false, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb, 64, GBK);
  if (e) return e;
  // output maps: one [32 rows x 64 bytes] box per staged piece; the copy engine clips rows >= M and columns >= N
  if (part != nullptr) e = make_tmap_3d_f32(&tmD, part, (uint64_t)N, (uint64_t)M, (uint64_t)p.split_k, 16, 32);
  else e = make_tmap_2d(&tmD, f32_out, D, (uint64_t)N, (uint64_t)M, (uint64_t)ldd, f32_out ? 16 : 32, 32, true);
  if (e) return e;
  tmD2 = tmD;
  if (epilogue == SWINB200_EPI_BIAS_GELU) {
    e = make_tmap_2d(&tmD2, false, D2, (uint64_t)N, (uint64_t)M, (uint64_t)ldd, 32, 32, true);
    if (e) return e;
  }

  if (qknorm) return launch_tc_impl<192, false, false, SWINB200_EPI_BIAS_QKNORM, true>(tmA, tmB, tmD, tmD2, p, stream);
  if (epilogue == SWINB200_EPI_BIAS_LN) return launch_tc_impl<256, false, false, SWINB200_EPI_BIAS_LN, true>(tmA, tmB, tmD, tmD2, p, stream);
  if (part != nullptr) {
    // every split writes its own slice with plain stores; the slices (and the column-sum rows) are then added in split order
    e = (BN == 256) ? launch_tc<256, true, true, SWINB200_EPI_F32, true>(tmA, tmB, tmD, tmD2, p, stream)
                    : launch_tc<128, true, true, SWINB200_EPI_F32, true>(tmA, tmB, tmD, tmD2, p, stream);
    if (e) return e;
    const long long mn = (long long)M * N;
    if ((e = ordered_reduce(part, p.split_k, mn, mn, 1, reinterpret_cast<float*>(D), accumulate, stream))) return e;
    if (colsum_out != nullptr) return ordered_reduce(p.colsum_out, p.split_k, M, M, 1, colsum_out, 1, stream);
    return SWINB200_OK;
  }
  if (BN == 256) return dispatch<256>(epilogue, a_major, b_major, tmA, tmB, tmD, tmD2, p, stream);
  return dispatch<128>(epilogue, a_major, b_major, tmA, tmB, tmD, tmD2, p, stream);
}

}  // namespace swinb200
