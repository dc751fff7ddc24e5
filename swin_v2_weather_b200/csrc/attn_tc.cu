// tcgen05 windowed cosine attention for sm_100a (bf16 storage, fp32 accumulation in tensor memory).
//
// One CTA per (sample, window, head).  The cyclic shift, window partition and window reverse of the reference
// (swinv2_global.py:89-119, 446-478) are folded into the gather / scatter addressing: slot n = a*Ww + c of window
// (wh, ww) is token ((wh*Wh + a + s0) % H, (ww*Ww + c + s1) % W), so no rolled or permuted copy ever reaches HBM.
//
// Shared-memory operand layout (un-swizzled UMMA core matrices), for a [rows x cols] bf16 tile:
//     byte(row, col) = (col / 8) * chunk_stride + row * 16 + (col % 8) * 2
// i.e. "[16-byte column chunk][row][8 elements]".  One 16-byte cp.async (or st.shared) per (row, chunk); consecutive
// rows are consecutive 16-byte words -> conflict-free stores.  The same bytes serve as a K-major operand
// (rows = m/n, cols = k: LBO = chunk_stride, SBO = 128) and as an MN-major operand (rows = k, cols = m/n:
// LBO = 128, SBO = chunk_stride), which is what lets K^ feed S = Q^ K^T and dQ = dS K^ without a transpose.
//
// forward:   S = Q^ K^T (tcgen05, TMEM) -> thread-per-row softmax(scale*S + bias + mask) -> P (bf16, smem)
//            -> O = P V (tcgen05, accumulator aliases S) -> O / rowsum -> scatter to (T, C); row LSE saved.
#include <stdlib.h>
#include "attn_tc.cuh"

namespace swinb200 {

// optional per-phase cycle stamps (bring-up aid): when non-null, CTA b writes clock64() deltas to g_phase[b*16 + i]
__device__ long long* g_phase_buf = nullptr;
#define SWB_STAMP(i)                                                                 \
  do {                                                                               \
    if (g_phase_buf != nullptr && threadIdx.x == 0 && blockIdx.x < 4096) g_phase_buf[blockIdx.x * 16 + (i)] = clock64(); \
  } while (0)

// ------------------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------------------
template <int D>
struct FwdSmem {
  static constexpr int kChunks = D / 8;
  static constexpr int kCS = kMaxLP * 16 + 16;                  // chunk stride of the Q / K / V tiles (bank de-phasing pad)
  static constexpr int kTile = kChunks * kCS;                   // one operand
  static constexpr int kPCS = 128 * 16;                         // chunk stride of a P tile (128 query rows)
  static constexpr int kPTile = (kMaxLP / 8) * kPCS;            // 22 key chunks
  static constexpr int kOffQ = 0, kOffK = kTile, kOffV = 2 * kTile, kOffP = 3 * kTile;   // Q first: its M-tile over-read lands in K/V
  static constexpr int kOffTok = kOffP + 2 * kPTile;
  static constexpr int kOffBar = kOffTok + kMaxLP * 4;
  static constexpr int kBytes = kOffBar + 64;
  static_assert(256 * kRowPitch <= 2 * kPTile, "output staging must fit in the P tiles");
};

template <int D>
__global__ void __launch_bounds__(256, 1)
attn_tc_fwd_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ scale_p, const float* __restrict__ bias,
                   __nv_bfloat16* __restrict__ o, float* __restrict__ lse, const AttnGeom g) {
  using SM = FwdSmem<D>;
  constexpr float kLog2e = 1.4426950408889634f;
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* sQ = smem + SM::kOffQ;
  unsigned char* sK = smem + SM::kOffK;
  unsigned char* sV = smem + SM::kOffV;
  unsigned char* sP = smem + SM::kOffP;
  int* tok = reinterpret_cast<int*>(smem + SM::kOffTok);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::kOffBar);   // [0] S ready, [1] O ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  SWB_STAMP(0);
  const int head = blockIdx.x % g.heads;
  const int w = (blockIdx.x / g.heads) % g.nW;
  const int b = blockIdx.x / (g.heads * g.nW);
  const int L = g.L, LP = g.LP;
  const int ntiles = (L > 128) ? 2 : 1;
  const bool shifted = (g.s0 > 0) || (g.s1 > 0);

  // ---- prologue: token table, barriers, tensor memory ---------------------------------------------------------
  int label_split = LP;   // first slot whose region label is 1 (keys >= label_split are "label 1")
  if (shifted) {
    // label(n) = (rolled_row >= H - s0) with rolled_row = wh*Wh + n / Ww  (every row if only the W shift is active)
    const int wh = w / g.nWw;
    if (g.s0 > 0) {
      const int first_row = g.H - g.s0 - wh * g.Wh;     // window-local row where label 1 starts
      label_split = first_row <= 0 ? 0 : (first_row >= g.Wh ? LP : first_row * g.Ww);
    } else {
      label_split = 0;
    }
  }
  // "plain" windows: no position bias and a single region label -> logits are just scale * cos
  const bool plain = (bias == nullptr) && !(label_split > 0 && label_split < L);
  for (int n = tid; n < LP; n += 256) {
    int rr;
    tok[n] = (n < L) ? win_token(g, b, w, n, rr) : -1;
  }
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  // zero the pad rows [L, LP) of Q, K and V (V pad rows must be finite: P is exactly 0 there)
  for (int i = tid; i < (LP - L) * SM::kChunks * 3; i += 256) {
    const int op = i / ((LP - L) * SM::kChunks);
    const int rem = i - op * (LP - L) * SM::kChunks;
    const int c = rem / (LP - L), r = L + rem % (LP - L);
    *reinterpret_cast<uint4*>(smem + op * SM::kTile + c * SM::kCS + r * 16) = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
  SWB_STAMP(1);

  // ---- gather Q^, K^, V of this (window, head): one 16-byte cp.async per (token, 8 channels) ----------------------
  {
    const int C3 = 3 * g.C;
    const int per_op = L * SM::kChunks;
    for (int i = tid; i < 3 * per_op; i += 256) {
      const int op = i / per_op;
      const int rem = i - op * per_op;
      const int n = rem / SM::kChunks, c = rem - n * SM::kChunks;
      const __nv_bfloat16* src = qkv + (size_t)tok[n] * C3 + op * g.C + head * D + c * 8;
      cp_async16(smem + op * SM::kTile + c * SM::kCS + n * 16, src);
    }
    cp_async_wait_all();
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  SWB_STAMP(2);
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // ---- S_t = Q^_t K^T ----------------------------------------------------------------------------------------------
  if (tid == 0) {
    const uint32_t idesc = umma_idesc_bf16(128, LP, false, false);
    const uint32_t q0 = smem_u32(sQ), k0 = smem_u32(sK);
    for (int t = 0; t < ntiles; ++t)
#pragma unroll
      for (int k = 0; k < D / 16; ++k)
        umma_bf16_ss(tmem_base + t * kMaxLP, umma_desc_nosw(q0 + 2 * k * SM::kCS + t * 128 * 16, SM::kCS, 128),
                     umma_desc_nosw(k0 + 2 * k * SM::kCS, SM::kCS, 128), idesc, k > 0);
    umma_commit(&bars[0]);
  }

  // ---- softmax: thread = one query row of tile t ---------------------------------------------------------------------
  const int t = warp >> 2;                       // warpgroup -> query tile
  const int r = (warp & 3) * 32 + lane;          // row inside the tile == TMEM lane
  const int n = t * 128 + r;                     // slot (query) index inside the window
  const bool row_ok = (t < ntiles) && (n < L);
  const float scale_l2 = scale_p[head] * kLog2e;  // work in the log2 domain
  const uint32_t t_s = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(t * kMaxLP);
  float row_sum = 0.f, row_max = -INFINITY;

  mbar_wait(&bars[0], 0, 500);
  SWB_STAMP(3);
  tc_fence_after();
  if (t < ntiles) {
    unsigned char* myP = sP + t * SM::kPTile + r * 16;
    if (plain) {
      // pass 1: max of the raw cosines (scale > 0); TMEM loads run one chunk ahead of the arithmetic.
      // Pad keys hold exact zeros (zeroed K^ rows): including them can only raise the max, which is harmless.
      uint32_t va[16], vb[16];
      float mx = -INFINITY;
      tmem_ld_32x16(t_s, va);
      for (int c0 = 0; c0 < LP; c0 += 32) {
        tmem_ld_wait();
        const bool has_b = c0 + 16 < LP;
        if (has_b) tmem_ld_32x16(t_s + c0 + 16, vb);
#pragma unroll
        for (int j = 0; j < 16; ++j) mx = fmaxf(mx, as_f(va[j]));
        if (has_b) {
          tmem_ld_wait();
          if (c0 + 32 < LP) tmem_ld_32x16(t_s + c0 + 32, va);
#pragma unroll
          for (int j = 0; j < 16; ++j) mx = fmaxf(mx, as_f(vb[j]));
        }
      }
      row_max = mx * scale_l2;
      const float neg_m = -row_max;
      // pass 2: p = 2^(scale*cos - max) -> bf16 P tile; fp32 row sum
      tmem_ld_32x16(t_s, va);
      for (int c0 = 0; c0 < LP; c0 += 32) {
        tmem_ld_wait();
        const bool has_b = c0 + 16 < LP;
        if (has_b) tmem_ld_32x16(t_s + c0 + 16, vb);
        {
          float p[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) p[j] = ex2_approx(fmaf(as_f(va[j]), scale_l2, neg_m));
          if (c0 + 16 > L) {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (c0 + j >= L) p[j] = 0.f;
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) row_sum += p[j];
          *reinterpret_cast<uint4*>(myP + (c0 / 8) * SM::kPCS) = pack8(p, 0);
          *reinterpret_cast<uint4*>(myP + (c0 / 8 + 1) * SM::kPCS) = pack8(p, 8);
        }
        if (has_b) {
          tmem_ld_wait();
          if (c0 + 32 < LP) tmem_ld_32x16(t_s + c0 + 32, va);
          const int c1 = c0 + 16;
          float p[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) p[j] = ex2_approx(fmaf(as_f(vb[j]), scale_l2, neg_m));
          if (c1 + 16 > L) {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (c1 + j >= L) p[j] = 0.f;
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) row_sum += p[j];
          *reinterpret_cast<uint4*>(myP + (c1 / 8) * SM::kPCS) = pack8(p, 0);
          *reinterpret_cast<uint4*>(myP + (c1 / 8 + 1) * SM::kPCS) = pack8(p, 8);
        }
      }
    } else {
      // general path: continuous position bias and / or the shifted-window mask (-100 across region labels)
      const float* brow = (bias != nullptr && row_ok) ? bias + ((size_t)head * L + n) * L : nullptr;
      const int my_label = (n >= label_split) ? 1 : 0;
      for (int c0 = 0; c0 < LP; c0 += 16) {
        uint32_t v[16];
        tmem_ld_32x16(t_s + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int key = c0 + j;
          float s = as_f(v[j]) * scale_l2;
          if (brow != nullptr && key < L) s += brow[key] * kLog2e;
          if (((key >= label_split) ? 1 : 0) != my_label) s += -100.0f * kLog2e;
          if (key < L) row_max = fmaxf(row_max, s);
        }
      }
      for (int c0 = 0; c0 < LP; c0 += 16) {
        uint32_t v[16];
        tmem_ld_32x16(t_s + c0, v);
        tmem_ld_wait();
        float p[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int key = c0 + j;
          float s = as_f(v[j]) * scale_l2;
          if (brow != nullptr && key < L) s += brow[key] * kLog2e;
          if (((key >= label_split) ? 1 : 0) != my_label) s += -100.0f * kLog2e;
          p[j] = (key < L && row_ok) ? ex2_approx(s - row_max) : 0.f;
          row_sum += p[j];
        }
        *reinterpret_cast<uint4*>(myP + (c0 / 8) * SM::kPCS) = pack8(p, 0);
        *reinterpret_cast<uint4*>(myP + (c0 / 8 + 1) * SM::kPCS) = pack8(p, 8);
      }
    }
    if (row_ok)
      lse[(((size_t)b * g.nW + w) * g.heads + head) * L + n] = (row_max + log2f(row_sum)) * 0.6931471805599453f;
  }
  fence_proxy_async_smem();   // P (generic-proxy stores) -> visible to the tensor core's async-proxy reads
  tc_fence_before();
  __syncthreads();            // every thread has finished reading S: O may overwrite its columns
  SWB_STAMP(4);

  // ---- O_t = P_t V  (accumulator aliases S_t) ----------------------------------------------------------------------------
  if (tid == 0) {
    tc_fence_after();
    const uint32_t idesc = umma_idesc_bf16(128, D, false, true);
    const uint32_t p0 = smem_u32(sP), v0 = smem_u32(sV);
    for (int tt = 0; tt < ntiles; ++tt)
      for (int k = 0; k < LP / 16; ++k)
        umma_bf16_ss(tmem_base + tt * kMaxLP, umma_desc_nosw(p0 + tt * SM::kPTile + 2 * k * SM::kPCS, SM::kPCS, 128),
                     umma_desc_nosw(v0 + k * 256, 128, SM::kCS), idesc, k > 0);
    umma_commit(&bars[1]);
  }
  mbar_wait(&bars[1], 0, 501);
  SWB_STAMP(5);
  tc_fence_after();
  // the P tiles are dead once the MMAs have completed: reuse them to stage the output rows
  if (t < ntiles) {
    const float inv = 1.0f / row_sum;
    float ov[D];
#pragma unroll
    for (int c0 = 0; c0 < D; c0 += 32) {
      uint32_t v[32];
      tmem_ld_32x32(t_s + c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) ov[c0 + j] = as_f(v[j]) * inv;
    }
    if (row_ok) park_row<D>(sP, n, ov);
  }
  tc_fence_before();
  __syncthreads();
  scatter_rows<D>(sP, L, tok, 0, o, g.C, head * D, tid, 256);
  SWB_STAMP(6);
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------
// forward, version 2: two CTAs per SM, operands that are only ever the A side of an MMA live in tensor memory
// ------------------------------------------------------------------------------------------------------------
// One 128-thread CTA per (sample, window, head); the block scheduler keeps two of them resident per SM so one CTA's
// gather overlaps the other's softmax / MMAs.  Shared memory holds only K^ and V (B operands) plus one row-major
// staging tile: Q^ rows land there (coalesced cp.async), are copied by their owning thread into tensor memory
// (tcgen05.st, thread = row = TMEM lane) and S = Q^ K^T runs with A from TMEM.  P overwrites S in place as packed
// bf16 (the thread that reads a row's S is the one that writes its P), O = P V again takes A from TMEM, and the
// staging tile is reused to park the output rows for whole-row global stores.
//   TMEM columns (256 allocated):  Q^ [0,48)   S [48,224)   P [48,136) in place   O [136,232) over the tail of S
template <int D>
struct Fwd2Smem {
  static constexpr int kChunks = D / 8;
  static constexpr int kCS = kMaxLP * 16 + 16;
  static constexpr int kTile = kChunks * kCS;
  static constexpr int kOffK = 0, kOffV = kTile;
  static constexpr int kOffStage = 2 * kTile;                    // [128 rows][kRowPitch]
  static constexpr int kOffTok = kOffStage + 128 * kRowPitch;
  static constexpr int kOffBar = kOffTok + kMaxLP * 4;
  static constexpr int kBytes = kOffBar + 64;
};

template <int D>
__global__ void __launch_bounds__(128, 2)
attn_tc_fwd2_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ scale_p, const float* __restrict__ bias,
                    __nv_bfloat16* __restrict__ o, float* __restrict__ lse, const AttnGeom g) {
  using SM = Fwd2Smem<D>;
  constexpr float kLog2e = 1.4426950408889634f;
  constexpr uint32_t kColQ = 0, kColS = 48, kColO = 136;
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* sK = smem + SM::kOffK;
  unsigned char* sV = smem + SM::kOffV;
  unsigned char* sStage = smem + SM::kOffStage;
  int* tok = reinterpret_cast<int*>(smem + SM::kOffTok);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + SM::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  SWB_STAMP(0);
  const int head = blockIdx.x % g.heads;
  const int w = (blockIdx.x / g.heads) % g.nW;
  const int b = blockIdx.x / (g.heads * g.nW);
  const int L = g.L, LP = g.LP;
  const int ntiles = (L > 128) ? 2 : 1;
  int label_split = LP;
  if ((g.s0 > 0) || (g.s1 > 0)) {
    const int wh = w / g.nWw;
    if (g.s0 > 0) {
      const int first_row = g.H - g.s0 - wh * g.Wh;
      label_split = first_row <= 0 ? 0 : (first_row >= g.Wh ? LP : first_row * g.Ww);
    } else {
      label_split = 0;
    }
  }
  const bool plain = (bias == nullptr) && !(label_split > 0 && label_split < L);

  for (int n = tid; n < LP; n += 128) {
    int rr;
    tok[n] = (n < L) ? win_token(g, b, w, n, rr) : -1;
  }
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  for (int i = tid; i < (LP - L) * SM::kChunks * 2; i += 128) {          // zero pad rows [L, LP) of K^ and V
    const int op = i / ((LP - L) * SM::kChunks);
    const int rem = i - op * (LP - L) * SM::kChunks;
    const int c = rem / (LP - L), r = L + rem % (LP - L);
    *reinterpret_cast<uint4*>(smem + op * SM::kTile + c * SM::kCS + r * 16) = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
  SWB_STAMP(1);

  const int C3 = 3 * g.C;
  auto gather_q_tile = [&](int t) {          // Q^ rows of tile t -> staging, row-major, coalesced
    const int rows = min(128, L - t * 128);
    for (int i = tid; i < rows * SM::kChunks; i += 128) {
      const int rr = i / SM::kChunks, c = i - rr * SM::kChunks;
      cp_async16(sStage + rr * kRowPitch + c * 16, qkv + (size_t)tok[t * 128 + rr] * C3 + head * D + c * 8);
    }
  };
  {
    const int per_op = L * SM::kChunks;
    for (int i = tid; i < 2 * per_op; i += 128) {                          // K^ and V -> chunked operand layout
      const int op = i / per_op;
      const int rem = i - op * per_op;
      const int n = rem / SM::kChunks, c = rem - n * SM::kChunks;
      cp_async16(smem + op * SM::kTile + c * SM::kCS + n * 16, qkv + (size_t)tok[n] * C3 + (op + 1) * g.C + head * D + c * 8);
    }
    gather_q_tile(0);
    cp_async_wait_all();
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  SWB_STAMP(2);
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t t_lane = tmem_base + ((uint32_t)(warp * 32) << 16);
  const float scale_l2 = scale_p[head] * kLog2e;
  const uint32_t k0 = smem_u32(sK), v0 = smem_u32(sV);
  const uint32_t idesc_s = umma_idesc_bf16(128, LP, false, false);
  const uint32_t idesc_o = umma_idesc_bf16(128, D, false, true);
  uint32_t parity = 0;

  for (int t = 0; t < ntiles; ++t) {
    const int n = t * 128 + tid;                  // this thread's query slot; TMEM lane = tid
    const bool row_ok = n < L;
    // ---- Q^ row: staging -> tensor memory (packed bf16, 4 columns per 16-byte chunk) ---------------------------------
    if (t > 0) {
      gather_q_tile(t);
      cp_async_wait_all();
      __syncthreads();
    }
#pragma unroll
    for (int c = 0; c < SM::kChunks; ++c) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (row_ok) v = *reinterpret_cast<const uint4*>(sStage + tid * kRowPitch + c * 16);
      tmem_st_32x4(t_lane + kColQ + c * 4, v);
    }
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    // ---- S = Q^ K^T (A from TMEM) -----------------------------------------------------------------------------------------
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < D / 16; ++k)
        umma_bf16_ts(tmem_base + kColS, tmem_base + kColQ + k * 8, umma_desc_nosw(k0 + 2 * k * SM::kCS, SM::kCS, 128), idesc_s, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 700 + t);
    parity ^= 1;
    SWB_STAMP(3);
    tc_fence_after();
    // ---- softmax, P written over S in place --------------------------------------------------------------------------------
    float row_sum = 0.f, row_max = -INFINITY;
    const uint32_t t_s = t_lane + kColS;
    if (plain) {
      uint32_t va[16], vb[16];
      float mx = -INFINITY;
      tmem_ld_32x16(t_s, va);
      for (int c0 = 0; c0 < LP; c0 += 32) {
        tmem_ld_wait();
        const bool has_b = c0 + 16 < LP;
        if (has_b) tmem_ld_32x16(t_s + c0 + 16, vb);
#pragma unroll
        for (int j = 0; j < 16; ++j) mx = fmaxf(mx, as_f(va[j]));
        if (has_b) {
          tmem_ld_wait();
          if (c0 + 32 < LP) tmem_ld_32x16(t_s + c0 + 32, va);
#pragma unroll
          for (int j = 0; j < 16; ++j) mx = fmaxf(mx, as_f(vb[j]));
        }
      }
      row_max = mx * scale_l2;
      const float neg_m = -row_max;
      for (int c0 = 0; c0 < LP; c0 += 16) {
        uint32_t v[16];
        tmem_ld_32x16(t_s + c0, v);
        tmem_ld_wait();
        float p[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) p[j] = ex2_approx(fmaf(as_f(v[j]), scale_l2, neg_m));
        if (c0 + 16 > L) {
#pragma unroll
          for (int j = 0; j < 16; ++j) if (c0 + j >= L) p[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) row_sum += p[j];
        tmem_st_32x8(t_s + c0 / 2, pack8(p, 0), pack8(p, 8));      // keys [c0, c0+16) -> 8 packed columns, already consumed
      }
    } else {
      const float* brow = (bias != nullptr && row_ok) ? bias + ((size_t)head * L + n) * L : nullptr;
      const int my_label = (n >= label_split) ? 1 : 0;
      for (int c0 = 0; c0 < LP; c0 += 16) {
        uint32_t v[16];
        tmem_ld_32x16(t_s + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int key = c0 + j;
          float sv = as_f(v[j]) * scale_l2;
          if (brow != nullptr && key < L) sv += brow[key] * kLog2e;
          if (((key >= label_split) ? 1 : 0) != my_label) sv += -100.0f * kLog2e;
          if (key < L) row_max = fmaxf(row_max, sv);
        }
      }
      for (int c0 = 0; c0 < LP; c0 += 16) {
        uint32_t v[16];
        tmem_ld_32x16(t_s + c0, v);
        tmem_ld_wait();
        float p[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int key = c0 + j;
          float sv = as_f(v[j]) * scale_l2;
          if (brow != nullptr && key < L) sv += brow[key] * kLog2e;
          if (((key >= label_split) ? 1 : 0) != my_label) sv += -100.0f * kLog2e;
          p[j] = (key < L && row_ok) ? ex2_approx(sv - row_max) : 0.f;
          row_sum += p[j];
        }
        tmem_st_32x8(t_s + c0 / 2, pack8(p, 0), pack8(p, 8));
      }
    }
    if (row_ok)
      lse[(((size_t)b * g.nW + w) * g.heads + head) * L + n] = (row_max + log2f(row_sum)) * 0.6931471805599453f;
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    SWB_STAMP(4);
    // ---- O = P V (A = P from TMEM, B = V read n-major) ------------------------------------------------------------------------
    if (tid == 0) {
      tc_fence_after();
      for (int k = 0; k < LP / 16; ++k)
        umma_bf16_ts(tmem_base + kColO, tmem_base + kColS + k * 8, umma_desc_nosw(v0 + k * 256, 128, SM::kCS), idesc_o, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 710 + t);
    parity ^= 1;
    SWB_STAMP(5);
    tc_fence_after();
    {
      const float inv = 1.0f / row_sum;
      float ov[D];
#pragma unroll
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_lane + kColO + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) ov[c0 + j] = as_f(v[j]) * inv;
      }
      if (row_ok) park_row<D>(sStage, tid, ov);     // the staging tile is free again: Q^ went to TMEM long ago
    }
    tc_fence_before();
    __syncthreads();
    scatter_rows<D>(sStage, min(128, L - t * 128), tok, t * 128, o, g.C, head * D, tid, 128);
    __syncthreads();
    SWB_STAMP(6);
  }
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

int attn_set_phase_buffer3(long long* buf);
int attn_set_phase_buffer_f3(long long* buf);
int attn_set_phase_buffer(long long* buf) {
  SWB_CUDA(cudaMemcpyToSymbol(g_phase_buf, &buf, sizeof(buf)));
  if (int e = attn_set_phase_buffer_f3(buf)) return e;
  return attn_set_phase_buffer3(buf);
}

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

int attn_tcgen05_fwd(const void* qkv, const float* scale, const float* bias, void* o, float* lse, int B, int H, int W, int C,
                     int heads, int Wh, int Ww, int s0, int s1, cudaStream_t stream) {
  AttnGeom g;
  if (int e = attn_make_geom(g, B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  static int variant = -1;
  if (variant < 0) {
    const char* e = getenv("SWINB200_ATTN_FWD");
    variant = e ? atoi(e) : 5;   // 1 = first SS-mode kernel; 2 = two CTAs per SM, cp.async gather; 3 = persistent, TMA boxes, double-buffered; 4 = tiled (attn_tc_gen.cu); 5 = two items in flight per SM (attn_tc_fwd4.cu)
  }
  // with a bias table the tiled kernel is the faster forward on every geometry (434 vs 660 us at 9x18 / 8 heads): its table
  // values are prefetched and reach their rows through a shared-memory slab; the persistent kernel reads them row by row
  if (!attn_is_specialised(g) || variant == 4 || (bias != nullptr && variant >= 3)) return attn_tcgen05_gen_fwd(qkv, scale, bias, o, lse, g, stream);
  if (variant == 5 && ((uintptr_t)qkv % 16 == 0)) return attn_tcgen05_fwd4(qkv, scale, bias, o, lse, g, stream);   // two items in flight per SM
  if (variant == 3 && ((uintptr_t)qkv % 16 == 0) && g.L * kRowPitch <= (96 / 32) * kCS64)
    return attn_tcgen05_fwd3(qkv, scale, bias, o, lse, g, stream);
  // the earlier generations do not produce the mean-cosine plane: define it as zero (= un-centred d(scale) in backward)
  SWB_CUDA(cudaMemsetAsync(lse + (size_t)g.B * g.nW * g.heads * g.L, 0, sizeof(float) * (size_t)g.B * g.nW * g.heads * g.L, stream));
  if (variant == 1) {
    using SM = FwdSmem<96>;
    static bool configured = false;
    if (!configured) {
      SWB_CUDA(cudaFuncSetAttribute(attn_tc_fwd_kernel<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
      configured = true;
    }
    attn_tc_fwd_kernel<96><<<B * g.nW * heads, 256, SM::kBytes, stream>>>((const __nv_bfloat16*)qkv, scale, bias,
                                                                          (__nv_bfloat16*)o, lse, g);
  } else {
    using SM = Fwd2Smem<96>;
    static bool configured = false;
    if (!configured) {
      SWB_CUDA(cudaFuncSetAttribute(attn_tc_fwd2_kernel<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
      configured = true;
    }
    attn_tc_fwd2_kernel<96><<<B * g.nW * heads, 128, SM::kBytes, stream>>>((const __nv_bfloat16*)qkv, scale, bias,
                                                                           (__nv_bfloat16*)o, lse, g);
  }
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

// ------------------------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------------------------
// Two sweeps over the same resident operands (Q^, K^, V, dO in shared memory):
//   A (query-major, per 128-query tile):  S = Q^ K^T, dP = dO V^T  ->  dS = P o (dP - D)  ->  dQ^ = dS K^  -> dq
//   B (key-major,   per 128-key tile):    S^T = K^ Q^T, dP^T = V dO^T -> P^T, dS^T -> dV = P^T dO, dK^ = dS^T Q^ -> dk
// S and dP are recomputed for the transposed sweep instead of transposing P / dS through shared memory; the tensor
// pipe has the headroom (the kernel is bound by the softmax arithmetic and HBM, not by the MMAs).
template <int D>
struct BwdSmem {
  static constexpr int kChunks = D / 8;
  static constexpr int kCS = kMaxLP * 16 + 16;
  static constexpr int kTile = kChunks * kCS;
  static constexpr int kPCS = 128 * 16;
  static constexpr int kPTile = (kMaxLP / 8) * kPCS;
  static constexpr int kOffQ = 0, kOffK = kTile, kOffV = 2 * kTile, kOffG = 3 * kTile;   // G = dO
  static constexpr int kOffP = 4 * kTile, kOffDS = kOffP + kPTile;
  static constexpr int kOffTok = kOffDS + kPTile;
  static constexpr int kOffLse = kOffTok + kMaxLP * 4;
  static constexpr int kOffDv = kOffLse + kMaxLP * 4;
  static constexpr int kOffRed = kOffDv + kMaxLP * 4;
  static constexpr int kOffBar = kOffRed + 64;
  static constexpr int kOffTok2 = kOffBar + 64;                  // persistent kernel: next item's token table
  static constexpr int kOffDsc = kOffTok2 + kMaxLP * 4;          // persistent kernel: per-head d(scale) partials
  static constexpr int kBytes = kOffDsc + 128;
};

template <int D>
__global__ void __launch_bounds__(256, 1)
attn_tc_bwd_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ inv_norm, const float* __restrict__ scale_p,
                   const float* __restrict__ bias, const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o,
                   const float* __restrict__ lse, __nv_bfloat16* __restrict__ dqkv, float* __restrict__ dscale,
                   float* __restrict__ dbias, const AttnGeom g) {
  using SM = BwdSmem<D>;
  constexpr float kLog2e = 1.4426950408889634f;
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* sQ = smem + SM::kOffQ;
  unsigned char* sK = smem + SM::kOffK;
  unsigned char* sV = smem + SM::kOffV;
  unsigned char* sG = smem + SM::kOffG;
  unsigned char* sP = smem + SM::kOffP;
  unsigned char* sDS = smem + SM::kOffDS;
  int* tok = reinterpret_cast<int*>(smem + SM::kOffTok);
  float* lse2 = reinterpret_cast<float*>(smem + SM::kOffLse);   // log2-domain LSE per query (+inf for pad queries)
  float* Dv = reinterpret_cast<float*>(smem + SM::kOffDv);      // rowsum(dO o O) per query
  float* red = reinterpret_cast<float*>(smem + SM::kOffRed);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + SM::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  SWB_STAMP(0);
  const int head = blockIdx.x % g.heads;
  const int w = (blockIdx.x / g.heads) % g.nW;
  const int b = blockIdx.x / (g.heads * g.nW);
  const int L = g.L, LP = g.LP, C = g.C, C3 = 3 * g.C;
  const int ntiles = (L > 128) ? 2 : 1;
  const bool shifted = (g.s0 > 0) || (g.s1 > 0);
  int label_split = LP;
  if (shifted) {
    const int wh = w / g.nWw;
    if (g.s0 > 0) {
      const int first_row = g.H - g.s0 - wh * g.Wh;
      label_split = first_row <= 0 ? 0 : (first_row >= g.Wh ? LP : first_row * g.Ww);
    } else {
      label_split = 0;
    }
  }

  // ---- prologue --------------------------------------------------------------------------------------------------
  for (int n = tid; n < LP; n += 256) {
    int rr;
    tok[n] = (n < L) ? win_token(g, b, w, n, rr) : -1;
    lse2[n] = (n < L) ? lse[(((size_t)b * g.nW + w) * g.heads + head) * L + n] * kLog2e : INFINITY;
  }
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  for (int i = tid; i < (LP - L) * SM::kChunks * 4; i += 256) {      // zero pad rows [L, LP) of Q^, K^, V, dO
    const int op = i / ((LP - L) * SM::kChunks);
    const int rem = i - op * (LP - L) * SM::kChunks;
    const int c = rem / (LP - L), r = L + rem % (LP - L);
    *reinterpret_cast<uint4*>(smem + op * SM::kTile + c * SM::kCS + r * 16) = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
  SWB_STAMP(1);
  {
    const int per_op = L * SM::kChunks;
    for (int i = tid; i < 4 * per_op; i += 256) {
      const int op = i / per_op;
      const int rem = i - op * per_op;
      const int n = rem / SM::kChunks, c = rem - n * SM::kChunks;
      const __nv_bfloat16* src = (op < 3) ? qkv + (size_t)tok[n] * C3 + op * C + head * D + c * 8
                                          : d_o + (size_t)tok[n] * C + head * D + c * 8;
      cp_async16(smem + op * SM::kTile + c * SM::kCS + n * 16, src);
    }
    // D_n = <dO_n, O_n> while the copies are in flight
    for (int n = tid; n < LP; n += 256) {
      float acc = 0.f;
      if (n < L) {
        const __nv_bfloat16* go = d_o + (size_t)tok[n] * C + head * D;
        const __nv_bfloat16* oo = o + (size_t)tok[n] * C + head * D;
#pragma unroll
        for (int c = 0; c < D; c += 8) {
          float a8[8], b8[8];
          ld8(go + c, a8);
          ld8(oo + c, b8);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc = fmaf(a8[e], b8[e], acc);
        }
      }
      Dv[n] = acc;
    }
    cp_async_wait_all();
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  SWB_STAMP(2);
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t q0 = smem_u32(sQ), k0 = smem_u32(sK), v0 = smem_u32(sV), g0 = smem_u32(sG), p0 = smem_u32(sP), ds0 = smem_u32(sDS);
  const uint32_t idesc_s = umma_idesc_bf16(128, LP, false, false);      // [128 x LP] = A(k-major) * B(k-major)^T
  const uint32_t idesc_o = umma_idesc_bf16(128, D, false, true);        // [128 x D]  = A(k-major) * B(n-major)
  const float scale = scale_p[head];
  const float scale_l2 = scale * kLog2e;
  uint32_t parity = 0;
  const bool plain = (bias == nullptr) && !(label_split > 0 && label_split < L);

  const int r = (warp & 3) * 32 + lane;                 // row inside the current 128-row tile == TMEM lane
  const int half = warp >> 2;                           // which part of the LP columns this thread handles
  const int c_split = ((LP + 31) / 32) * 16;            // both parts are multiples of 16 columns (176 -> 96 + 80)
  const int c_begin = half ? c_split : 0, c_end = half ? LP : c_split;
  const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
  float dsc_acc = 0.f;

  // ================================ sweep A: query-major -> dq ================================
  for (int t = 0; t < ntiles; ++t) {
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // S = Q^_t K^T
        umma_bf16_ss(tmem_base, umma_desc_nosw(q0 + 2 * k * SM::kCS + t * 2048, SM::kCS, 128),
                     umma_desc_nosw(k0 + 2 * k * SM::kCS, SM::kCS, 128), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // dP = dO_t V^T
        umma_bf16_ss(tmem_base + kMaxLP, umma_desc_nosw(g0 + 2 * k * SM::kCS + t * 2048, SM::kCS, 128),
                     umma_desc_nosw(v0 + 2 * k * SM::kCS, SM::kCS, 128), idesc_s, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 600 + t);
    SWB_STAMP(3);
    parity ^= 1;
    tc_fence_after();
    {
      const int n = t * 128 + r;                        // query slot of this thread
      const bool row_ok = n < L;
      const float my_lse = row_ok ? lse2[n] : INFINITY;  // pad rows: p = 2^(-inf) = 0
      const float my_D = row_ok ? Dv[n] : 0.f;
      unsigned char* myDS = sDS + r * 16;
      float dsc_tile = 0.f;
      if (plain) {
        // dS = P o (dP - D), P = 2^(scale*cos - lse); loads of the next 16 columns overlap this chunk's arithmetic
        uint32_t sa[16], pa[16], sb[16], pb[16];
        tmem_ld_32x16(t_lane + c_begin, sa);
        tmem_ld_32x16(t_lane + kMaxLP + c_begin, pa);
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
          tmem_ld_wait();
          const bool has_b = c0 + 16 < c_end;
          if (has_b) {
            tmem_ld_32x16(t_lane + c0 + 16, sb);
            tmem_ld_32x16(t_lane + kMaxLP + c0 + 16, pb);
          }
          {
            float ds[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float cosv = as_f(sa[j]);
              const float p = ex2_approx(fmaf(cosv, scale_l2, -my_lse));
              ds[j] = p * (as_f(pa[j]) - my_D);
              if (c0 + 16 > L && c0 + j >= L) ds[j] = 0.f;
              dsc_tile = fmaf(ds[j], cosv, dsc_tile);
            }
            *reinterpret_cast<uint4*>(myDS + (c0 / 8) * SM::kPCS) = pack8(ds, 0);
            *reinterpret_cast<uint4*>(myDS + (c0 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
          }
          if (has_b) {
            tmem_ld_wait();
            if (c0 + 32 < c_end) {
              tmem_ld_32x16(t_lane + c0 + 32, sa);
              tmem_ld_32x16(t_lane + kMaxLP + c0 + 32, pa);
            }
            const int c1 = c0 + 16;
            float ds[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float cosv = as_f(sb[j]);
              const float p = ex2_approx(fmaf(cosv, scale_l2, -my_lse));
              ds[j] = p * (as_f(pb[j]) - my_D);
              if (c1 + 16 > L && c1 + j >= L) ds[j] = 0.f;
              dsc_tile = fmaf(ds[j], cosv, dsc_tile);
            }
            *reinterpret_cast<uint4*>(myDS + (c1 / 8) * SM::kPCS) = pack8(ds, 0);
            *reinterpret_cast<uint4*>(myDS + (c1 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
          }
        }
      } else {
        const int my_label = (n >= label_split) ? 1 : 0;
        const float* brow = (bias != nullptr && row_ok) ? bias + ((size_t)head * L + n) * L : nullptr;
        float* dbrow = (dbias != nullptr && row_ok) ? dbias + ((size_t)head * L + n) * L : nullptr;
        for (int c0 = c_begin; c0 < c_end; c0 += 16) {
          uint32_t sv[16], pv[16];
          tmem_ld_32x16(t_lane + c0, sv);
          tmem_ld_32x16(t_lane + kMaxLP + c0, pv);
          tmem_ld_wait();
          float ds[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int key = c0 + j;
            const float cosv = as_f(sv[j]);
            float s = cosv * scale_l2;
            if (brow != nullptr && key < L) s += brow[key] * kLog2e;
            if (((key >= label_split) ? 1 : 0) != my_label) s += -100.0f * kLog2e;
            const float p = (key < L && row_ok) ? ex2_approx(s - my_lse) : 0.f;
            // pad rows / pad keys read whatever follows the real rows in shared memory: keep them exactly zero
            ds[j] = (key < L && row_ok) ? p * (as_f(pv[j]) - my_D) : 0.f;
            if (key < L && row_ok) dsc_tile = fmaf(ds[j], cosv, dsc_tile);
            if (dbrow != nullptr && key < L) atomicAdd(dbrow + key, ds[j]);
          }
          *reinterpret_cast<uint4*>(myDS + (c0 / 8) * SM::kPCS) = pack8(ds, 0);
          *reinterpret_cast<uint4*>(myDS + (c0 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
        }
      }
      if (row_ok) dsc_acc += dsc_tile;   // pad rows carry garbage cosines (their P is 0, but 0 * NaN would poison the sum)
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    SWB_STAMP(4);
    if (tid == 0) {
      tc_fence_after();
      for (int k = 0; k < LP / 16; ++k)     // dQ^_t = dS K^   (K^ read n-major: rows = keys = k-dimension)
        umma_bf16_ss(tmem_base, umma_desc_nosw(ds0 + 2 * k * SM::kPCS, SM::kPCS, 128),
                     umma_desc_nosw(k0 + k * 256, 128, SM::kCS), idesc_o, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 610 + t);
    SWB_STAMP(5);
    parity ^= 1;
    tc_fence_after();
    const int rows_here = min(128, L - t * 128);
    if (half == 0) {
      // dq = inv_norm * (dq^ - q^ <q^, dq^>),  dq^ = scale * (dS K^);  the dS tile is dead: stage the rows there
      const int n = t * 128 + r;
      const bool row_ok = n < L;
      float dq[D];
      float dot = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_lane + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) dq[c0 + j] = as_f(v[j]) * scale;
      }
      if (row_ok) {
        float qh[D];
#pragma unroll
        for (int c = 0; c < D / 8; ++c) {
          float t8[8];
          ld8(reinterpret_cast<const __nv_bfloat16*>(sQ + c * SM::kCS + n * 16), t8);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            qh[c * 8 + e] = t8[e];
            dot = fmaf(t8[e], dq[c * 8 + e], dot);
          }
        }
        const float inq = inv_norm[(size_t)tok[n] * 2 * g.heads + head];
#pragma unroll
        for (int c = 0; c < D; ++c) dq[c] = inq * (dq[c] - qh[c] * dot);
        park_row<D>(sDS, r, dq);
      }
    }
    tc_fence_before();
    __syncthreads();      // dQ^ has been read (the next S may overwrite it) and the staged rows are complete
    scatter_rows<D>(sDS, rows_here, tok, t * 128, dqkv, C3, head * D, tid, 256);
    __syncthreads();      // staging drained before the next tile's dS lands in the same buffer
    SWB_STAMP(6);
  }

  // ================================ sweep B: key-major -> dk, dv ================================
  for (int u = 0; u < ntiles; ++u) {
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // S^T = K^_u Q^T
        umma_bf16_ss(tmem_base, umma_desc_nosw(k0 + 2 * k * SM::kCS + u * 2048, SM::kCS, 128),
                     umma_desc_nosw(q0 + 2 * k * SM::kCS, SM::kCS, 128), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // dP^T = V_u dO^T
        umma_bf16_ss(tmem_base + kMaxLP, umma_desc_nosw(v0 + 2 * k * SM::kCS + u * 2048, SM::kCS, 128),
                     umma_desc_nosw(g0 + 2 * k * SM::kCS, SM::kCS, 128), idesc_s, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 620 + u);
    SWB_STAMP(7);
    parity ^= 1;
    tc_fence_after();
    {
      const int jk = u * 128 + r;                       // key slot of this thread
      const bool key_ok = jk < L;
      const int key_label = (jk >= label_split) ? 1 : 0;
      unsigned char* myP = sP + r * 16;
      unsigned char* myDS = sDS + r * 16;
      // columns = queries; lse2[q] = +inf for pad queries -> P = 0 there.  Pad key rows only feed discarded output rows,
      // but they are zeroed so that no NaN ever enters the tensor pipe.
      for (int c0 = c_begin; c0 < c_end; c0 += 16) {
        uint32_t sv[16], pv[16];
        tmem_ld_32x16(t_lane + c0, sv);
        tmem_ld_32x16(t_lane + kMaxLP + c0, pv);
        float ls[16], dd[16];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          *reinterpret_cast<float4*>(&ls[j]) = *reinterpret_cast<const float4*>(&lse2[c0 + j]);
          *reinterpret_cast<float4*>(&dd[j]) = *reinterpret_cast<const float4*>(&Dv[c0 + j]);
        }
        tmem_ld_wait();
        float pp[16], ds[16];
        if (plain) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float p = ex2_approx(fmaf(as_f(sv[j]), scale_l2, -ls[j]));
            pp[j] = key_ok ? p : 0.f;
            ds[j] = key_ok ? p * (as_f(pv[j]) - dd[j]) : 0.f;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int qi = c0 + j;
            float s = as_f(sv[j]) * scale_l2;
            if (bias != nullptr && key_ok && qi < L) s += bias[((size_t)head * L + qi) * L + jk] * kLog2e;
            if (((qi >= label_split) ? 1 : 0) != key_label) s += -100.0f * kLog2e;
            const float p = key_ok ? ex2_approx(s - ls[j]) : 0.f;
            pp[j] = p;
            ds[j] = (key_ok && qi < L) ? p * (as_f(pv[j]) - dd[j]) : 0.f;
          }
        }
        *reinterpret_cast<uint4*>(myP + (c0 / 8) * SM::kPCS) = pack8(pp, 0);
        *reinterpret_cast<uint4*>(myP + (c0 / 8 + 1) * SM::kPCS) = pack8(pp, 8);
        *reinterpret_cast<uint4*>(myDS + (c0 / 8) * SM::kPCS) = pack8(ds, 0);
        *reinterpret_cast<uint4*>(myDS + (c0 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    SWB_STAMP(8);
    if (tid == 0) {
      tc_fence_after();
      for (int k = 0; k < LP / 16; ++k)     // dV_u = P^T dO   (dO read n-major: rows = queries = k-dimension)
        umma_bf16_ss(tmem_base, umma_desc_nosw(p0 + 2 * k * SM::kPCS, SM::kPCS, 128),
                     umma_desc_nosw(g0 + k * 256, 128, SM::kCS), idesc_o, k > 0);
      for (int k = 0; k < LP / 16; ++k)     // dK^_u = dS^T Q^
        umma_bf16_ss(tmem_base + kMaxLP, umma_desc_nosw(ds0 + 2 * k * SM::kPCS, SM::kPCS, 128),
                     umma_desc_nosw(q0 + k * 256, 128, SM::kCS), idesc_o, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 630 + u);
    SWB_STAMP(9);
    parity ^= 1;
    tc_fence_after();
    const int rows_here = min(128, L - u * 128);
    {
      // warps 0-3: dv rows (staged in the P tile); warps 4-7: dk rows (staged in the dS tile)
      const int jk = u * 128 + r;
      const bool key_ok = jk < L;
      float acc[D];
#pragma unroll
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_lane + half * kMaxLP + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[c0 + j] = as_f(v[j]);
      }
      if (key_ok) {
        if (half == 0) {
          park_row<D>(sP, r, acc);
        } else {                                         // dk = inv_norm * (dk^ - k^ <k^, dk^>), dk^ = scale * (dS^T Q^)
          float dot = 0.f;
          float kh[D];
#pragma unroll
          for (int c = 0; c < D / 8; ++c) {
            float t8[8];
            ld8(reinterpret_cast<const __nv_bfloat16*>(sK + c * SM::kCS + jk * 16), t8);
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              kh[c * 8 + e] = t8[e];
              acc[c * 8 + e] *= scale;
              dot = fmaf(t8[e], acc[c * 8 + e], dot);
            }
          }
          const float ink = inv_norm[(size_t)tok[jk] * 2 * g.heads + g.heads + head];
#pragma unroll
          for (int c = 0; c < D; ++c) acc[c] = ink * (acc[c] - kh[c] * dot);
          park_row<D>(sDS, r, acc);
        }
      }
    }
    tc_fence_before();
    __syncthreads();
    // 128 threads drain each staging tile with whole-row stores
    if (half == 0) scatter_rows<D>(sP, rows_here, tok, u * 128, dqkv, C3, 2 * C + head * D, tid, 128);
    else scatter_rows<D>(sDS, rows_here, tok, u * 128, dqkv, C3, C + head * D, tid - 128, 128);
    __syncthreads();
    SWB_STAMP(10);
  }

  // ---- d(scale) = sum dS o cos -----------------------------------------------------------------------------------------
  dsc_acc = warp_sum(dsc_acc);
  if (lane == 0) red[warp] = dsc_acc;
  __syncthreads();
  if (tid == 0) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i];
    atomicAdd(dscale + head, s);
  }
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// Persistent variant.  Operand tiles (Q^, K^, V, dO) use 64-byte rows with the 64B swizzle: a [rows x 96] bf16 tile is
// three 32-column chunks of [176 rows x 64 B], and one chunk of a window is ONE TMA box [32 elements x Ww x Wh] of the
// (B, H, W, channels) activation tensor (64-byte rows move four times faster through the copy engine than the 16-byte
// rows of the un-swizzled layout).  The same bytes serve as K-major operands (rows = m/n, k along the row: 8-row groups
// 512 B apart, k advances 32 B inside the row, 32-k chunks a chunk stride apart) and as MN-major operands (rows = k:
// 8-k groups 512 B apart, 32-wide n chunks a chunk stride apart, k advances 16 rows = 1024 B).
template <int D>
struct Bwd2Smem {
  static constexpr int kChunks = D / 8;
  static constexpr int kCS = kMaxLP * 16;                        // 2816 = 22 * 128
  static constexpr int kTile = kChunks * kCS;
  static constexpr int kPCS = 128 * 16;
  static constexpr int kPTile = (kMaxLP / 8) * kPCS;
  static constexpr int kOffQ = 0, kOffK = kTile, kOffV = 2 * kTile, kOffG = 3 * kTile;   // G = dO
  static constexpr int kOffP = 4 * kTile, kOffDS = kOffP + kPTile;
  static constexpr int kOffTok = kOffDS + kPTile;
  static constexpr int kOffLse = kOffTok + kMaxLP * 4;
  static constexpr int kOffDv = kOffLse + kMaxLP * 4;
  static constexpr int kOffRed = kOffDv + kMaxLP * 4;
  static constexpr int kOffBar = kOffRed + 64;
  static constexpr int kOffTok2 = kOffBar + 64;                  // next item's token table
  static constexpr int kOffDsc = kOffTok2 + kMaxLP * 4;          // per-head d(scale) partials
  static constexpr int kBytes = kOffDsc + 128;
  static_assert(kBytes <= 227 * 1024, "shared memory budget");
};

template <int D>
__global__ void __launch_bounds__(256, 1)
attn_tc_bwd2_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_do,
                   const float* __restrict__ Dpre,
                   const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ inv_norm, const float* __restrict__ scale_p,
                   const float* __restrict__ bias, const __nv_bfloat16* __restrict__ o, const __nv_bfloat16* __restrict__ d_o,
                   const float* __restrict__ lse, __nv_bfloat16* __restrict__ dqkv, float* __restrict__ dscale,
                   float* __restrict__ dbias, const AttnGeom g) {
  using SM = Bwd2Smem<D>;
  constexpr float kLog2e = 1.4426950408889634f;
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* sQ = smem + SM::kOffQ;
  unsigned char* sK = smem + SM::kOffK;
  unsigned char* sV = smem + SM::kOffV;
  unsigned char* sG = smem + SM::kOffG;
  unsigned char* sP = smem + SM::kOffP;
  unsigned char* sDS = smem + SM::kOffDS;
  int* tok = reinterpret_cast<int*>(smem + SM::kOffTok);   // token table of the current item (double-buffered)
  float* lse2 = reinterpret_cast<float*>(smem + SM::kOffLse);   // log2-domain LSE per query (+inf for pad queries)
  float* Dv = reinterpret_cast<float*>(smem + SM::kOffDv);      // rowsum(dO o O) per query
  float* red = reinterpret_cast<float*>(smem + SM::kOffRed);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + SM::kOffBar);     // MMA completion
  uint64_t* ld_bar = bar + 1;                                          // operand boxes of the next item have landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long ph_acc[12];
  for (int i = 0; i < 12; ++i) ph_acc[i] = 0;
  long long ph_t = clock64();
#define SWB_ACC(i) do { if (tid == 0) { const long long now_ = clock64(); ph_acc[i] += now_ - ph_t; ph_t = now_; } } while (0)
  const int L = g.L, LP = g.LP, C = g.C, C3 = 3 * g.C;
  const int ntiles = (L > 128) ? 2 : 1;
  const bool shifted = (g.s0 > 0) || (g.s1 > 0);
  const int nitems = g.B * g.nW * g.heads;
  int* tokbuf[2] = {tok, reinterpret_cast<int*>(smem + SM::kOffTok2)};
  float* dsc_heads = reinterpret_cast<float*>(smem + SM::kOffDsc);     // per-head d(scale) partial sums of this CTA

  // ---- one-time set-up: barrier, tensor memory, zero pad rows (gathers only ever write rows < L) -------------------
  if (tid == 0) {
    prefetch_tmap(&tm_qkv);
    prefetch_tmap(&tm_do);
    mbar_init(bar, 1);
    mbar_init(ld_bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  for (int i = tid; i < (LP - L) * SM::kChunks * 4; i += 256) {
    const int op = i / ((LP - L) * SM::kChunks);
    const int rem = i - op * (LP - L) * SM::kChunks;
    const int c = rem / (LP - L), r = L + rem % (LP - L);
    *reinterpret_cast<uint4*>(smem + op * SM::kTile + opnd_off(r, c)) = make_uint4(0, 0, 0, 0);
  }
  if (tid < 32) dsc_heads[tid] = 0.f;
  // operands op_lo..op_hi-1 (0 Q^, 1 K^, 2 V, 3 dO) of the (window, head) whose token table is `tk`
  auto gather = [&](int op_lo, int op_hi, const int* tk, int hd) {
    const int per_op = L * SM::kChunks;
    for (int i = tid; i < (op_hi - op_lo) * per_op; i += 256) {
      const int op = op_lo + i / per_op;
      const int rem = i % per_op;
      const int n = rem / SM::kChunks, c = rem - n * SM::kChunks;
      const __nv_bfloat16* src = (op < 3) ? qkv + (size_t)tk[n] * C3 + op * C + hd * D + c * 8
                                          : d_o + (size_t)tk[n] * C + hd * D + c * 8;
      cp_async16(smem + op * SM::kTile + opnd_off(n, c), src);
    }
  };
  auto fill_tok = [&](int item, int* tk) {
    const int hd = item % g.heads;
    const int ww = (item / g.heads) % g.nW;
    const int bb = item / (g.heads * g.nW);
    for (int n = tid; n < LP; n += 256) {
      int rr;
      tk[n] = (n < L) ? win_token(g, bb, ww, n, rr) : -1;
    }
    return hd;
  };
  // A window whose rows or columns wrap around the cyclic shift is not one box of the tensor: those items (the last
  // window row / column of the shifted blocks, ~10 % of them) keep the per-thread cp.async gather.
  auto item_is_box = [&](int item) {
    const int ww_all = (item / g.heads) % g.nW;
    const int wh = ww_all / g.nWw, ww = ww_all - wh * g.nWw;
    return !((g.s0 > 0 && (wh + 1) * g.Wh + g.s0 > g.H) || (g.s1 > 0 && (ww + 1) * g.Ww + g.s1 > g.W));
  };
  constexpr uint32_t kBoxBytes = 64;   // x L rows, per (operand, 32-column chunk)
  constexpr int kBoxes = D / 32;
  // one thread: boxes of operands [op_lo, op_hi) of `item`; `first` registers the item's total byte count
  auto issue_boxes = [&](int op_lo, int op_hi, int item, bool first) {
    const int hd = item % g.heads;
    const int ww_all = (item / g.heads) % g.nW;
    const int bb = item / (g.heads * g.nW);
    const int wh = ww_all / g.nWw, ww = ww_all - wh * g.nWw;
    fence_proxy_async_smem();    // earlier generic-proxy reads of these tiles are ordered before the async-proxy writes
    if (first) mbar_arrive_expect_tx(ld_bar, 4u * kBoxes * kBoxBytes * (uint32_t)L);
    for (int op = op_lo; op < op_hi; ++op) {
      const CUtensorMap* tm = (op < 3) ? &tm_qkv : &tm_do;
      const int chunk0 = ((op < 3) ? op * C + hd * D : hd * D) / 32;
#pragma unroll
      for (int c = 0; c < kBoxes; ++c)
        tma_load_5d(smem + op * SM::kTile + c * kCS64, tm, ld_bar, 0, chunk0 + c, ww * g.Ww + g.s1, wh * g.Wh + g.s0, bb);
    }
  };
  bool cur_box = false;
  uint32_t ld_parity = 0;
  if ((int)blockIdx.x < nitems) {
    fill_tok(blockIdx.x, tokbuf[0]);
    cur_box = item_is_box(blockIdx.x);
  }
  __syncthreads();
  if ((int)blockIdx.x < nitems) {
    if (cur_box) { if (tid == 0) issue_boxes(0, 4, blockIdx.x, true); }
    else gather(0, 4, tokbuf[0], (int)blockIdx.x % g.heads);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t q0 = smem_u32(sQ), k0 = smem_u32(sK), v0 = smem_u32(sV), g0 = smem_u32(sG), p0 = smem_u32(sP), ds0 = smem_u32(sDS);
  const uint32_t idesc_s = umma_idesc_bf16(128, LP, false, false);      // [128 x LP] = A(k-major) * B(k-major)^T
  const uint32_t idesc_o = umma_idesc_bf16(128, D, false, true);        // [128 x D]  = A(k-major) * B(n-major)
  uint32_t parity = 0;
  SWB_ACC(1);

  int it = 0;
  for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
  tok = tokbuf[it & 1];
  int* tok_next = tokbuf[(it & 1) ^ 1];
  const int head = item % g.heads;
  const int w = (item / g.heads) % g.nW;
  const int b = item / (g.heads * g.nW);
  const int item_next = item + gridDim.x;
  const bool has_next = item_next < nitems;
  const int head_next = has_next ? fill_tok(item_next, tok_next) : 0;    // visible after the next barrier
  const bool next_box = has_next && item_is_box(item_next);
  int label_split = LP;
  if (shifted) {
    const int wh = w / g.nWw;
    if (g.s0 > 0) {
      const int first_row = g.H - g.s0 - wh * g.Wh;
      label_split = first_row <= 0 ? 0 : (first_row >= g.Wh ? LP : first_row * g.Ww);
    } else {
      label_split = 0;
    }
  }
  for (int n = tid; n < LP; n += 256) {
    lse2[n] = (n < L) ? lse[(((size_t)b * g.nW + w) * g.heads + head) * L + n] * kLog2e : INFINITY;
    Dv[n] = (n < L) ? Dpre[(size_t)tok[n] * g.heads + head] : 0.f;      // D_n = <dO_n, O_n> (pre-pass kernel)
  }
  const float scale = scale_p[head];
  const float scale_l2 = scale * kLog2e;
  // this item's operands: TMA boxes issued during the previous item (or just above), or the cp.async gather
  if (cur_box) {
    mbar_wait(ld_bar, ld_parity, 640);
    ld_parity ^= 1;
  } else {
    cp_async_wait_all();
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  SWB_ACC(2);
  tc_fence_after();
  const bool plain = (bias == nullptr) && !(label_split > 0 && label_split < L);

  const int r = (warp & 3) * 32 + lane;                 // row inside the current 128-row tile == TMEM lane
  const int half = warp >> 2;                           // which part of the LP columns this thread handles
  const int c_split = ((LP + 31) / 32) * 16;            // both parts are multiples of 16 columns (176 -> 96 + 80)
  const int c_begin = half ? c_split : 0, c_end = half ? LP : c_split;
  const uint32_t t_lane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
  float dsc_acc = 0.f;

  // ================================ sweep A: query-major -> dq ================================
  for (int t = 0; t < ntiles; ++t) {
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // S = Q^_t K^T
        umma_bf16_ss(tmem_base, opnd_kmajor(q0, k, t * 128), opnd_kmajor(k0, k, 0), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // dP = dO_t V^T
        umma_bf16_ss(tmem_base + kMaxLP, opnd_kmajor(g0, k, t * 128), opnd_kmajor(v0, k, 0), idesc_s, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 600 + t);
    SWB_ACC(3);
    parity ^= 1;
    tc_fence_after();
    {
      const int n = t * 128 + r;                        // query slot of this thread
      const bool row_ok = n < L;
      const float my_lse = row_ok ? lse2[n] : INFINITY;  // pad rows: p = 2^(-inf) = 0
      const float my_D = row_ok ? Dv[n] : 0.f;
      unsigned char* myDS = sDS + r * 16;
      float dsc_tile = 0.f;
      if (plain) {
        // dS = P o (dP - D), P = 2^(scale*cos - lse); loads of the next 16 columns overlap this chunk's arithmetic
        uint32_t sa[16], pa[16], sb[16], pb[16];
        tmem_ld_32x16(t_lane + c_begin, sa);
        tmem_ld_32x16(t_lane + kMaxLP + c_begin, pa);
        for (int c0 = c_begin; c0 < c_end; c0 += 32) {
          tmem_ld_wait();
          const bool has_b = c0 + 16 < c_end;
          if (has_b) {
            tmem_ld_32x16(t_lane + c0 + 16, sb);
            tmem_ld_32x16(t_lane + kMaxLP + c0 + 16, pb);
          }
          {
            float ds[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float cosv = as_f(sa[j]);
              const float p = ex2_approx(fmaf(cosv, scale_l2, -my_lse));
              ds[j] = p * (as_f(pa[j]) - my_D);
              if (c0 + 16 > L && c0 + j >= L) ds[j] = 0.f;
              dsc_tile = fmaf(ds[j], cosv, dsc_tile);
            }
            *reinterpret_cast<uint4*>(myDS + (c0 / 8) * SM::kPCS) = pack8(ds, 0);
            *reinterpret_cast<uint4*>(myDS + (c0 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
          }
          if (has_b) {
            tmem_ld_wait();
            if (c0 + 32 < c_end) {
              tmem_ld_32x16(t_lane + c0 + 32, sa);
              tmem_ld_32x16(t_lane + kMaxLP + c0 + 32, pa);
            }
            const int c1 = c0 + 16;
            float ds[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const float cosv = as_f(sb[j]);
              const float p = ex2_approx(fmaf(cosv, scale_l2, -my_lse));
              ds[j] = p * (as_f(pb[j]) - my_D);
              if (c1 + 16 > L && c1 + j >= L) ds[j] = 0.f;
              dsc_tile = fmaf(ds[j], cosv, dsc_tile);
            }
            *reinterpret_cast<uint4*>(myDS + (c1 / 8) * SM::kPCS) = pack8(ds, 0);
            *reinterpret_cast<uint4*>(myDS + (c1 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
          }
        }
      } else {
        const int my_label = (n >= label_split) ? 1 : 0;
        const float* brow = (bias != nullptr && row_ok) ? bias + ((size_t)head * L + n) * L : nullptr;
        float* dbrow = (dbias != nullptr && row_ok) ? dbias + ((size_t)head * L + n) * L : nullptr;
        for (int c0 = c_begin; c0 < c_end; c0 += 16) {
          uint32_t sv[16], pv[16];
          tmem_ld_32x16(t_lane + c0, sv);
          tmem_ld_32x16(t_lane + kMaxLP + c0, pv);
          tmem_ld_wait();
          float ds[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int key = c0 + j;
            const float cosv = as_f(sv[j]);
            float s = cosv * scale_l2;
            if (brow != nullptr && key < L) s += brow[key] * kLog2e;
            if (((key >= label_split) ? 1 : 0) != my_label) s += -100.0f * kLog2e;
            const float p = (key < L && row_ok) ? ex2_approx(s - my_lse) : 0.f;
            // pad rows / pad keys read whatever follows the real rows in shared memory: keep them exactly zero
            ds[j] = (key < L && row_ok) ? p * (as_f(pv[j]) - my_D) : 0.f;
            if (key < L && row_ok) dsc_tile = fmaf(ds[j], cosv, dsc_tile);
            if (dbrow != nullptr && key < L) atomicAdd(dbrow + key, ds[j]);
          }
          *reinterpret_cast<uint4*>(myDS + (c0 / 8) * SM::kPCS) = pack8(ds, 0);
          *reinterpret_cast<uint4*>(myDS + (c0 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
        }
      }
      if (row_ok) dsc_acc += dsc_tile;   // pad rows carry garbage cosines (their P is 0, but 0 * NaN would poison the sum)
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    SWB_ACC(4);
    if (tid == 0) {
      tc_fence_after();
      for (int k = 0; k < LP / 16; ++k)     // dQ^_t = dS K^   (K^ read n-major: rows = keys = k-dimension)
        umma_bf16_ss(tmem_base, umma_desc_nosw(ds0 + 2 * k * SM::kPCS, SM::kPCS, 128),
                     opnd_mnmajor(k0, k), idesc_o, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 610 + t);
    SWB_ACC(5);
    parity ^= 1;
    tc_fence_after();
    const int rows_here = min(128, L - t * 128);
    if (half == 0) {
      // dq = inv_norm * (dq^ - q^ <q^, dq^>),  dq^ = scale * (dS K^);  the dS tile is dead: stage the rows there
      const int n = t * 128 + r;
      const bool row_ok = n < L;
      float dq[D];
      float dot = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_lane + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) dq[c0 + j] = as_f(v[j]) * scale;
      }
      if (row_ok) {
        float qh[D];
#pragma unroll
        for (int c = 0; c < D / 8; ++c) {
          float t8[8];
          ld8(reinterpret_cast<const __nv_bfloat16*>(sQ + opnd_off(n, c)), t8);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            qh[c * 8 + e] = t8[e];
            dot = fmaf(t8[e], dq[c * 8 + e], dot);
          }
        }
        const float inq = inv_norm[(size_t)tok[n] * 2 * g.heads + head];
#pragma unroll
        for (int c = 0; c < D; ++c) dq[c] = inq * (dq[c] - qh[c] * dot);
        park_row<D>(sDS, r, dq);
      }
    }
    tc_fence_before();
    __syncthreads();      // dQ^ has been read (the next S may overwrite it) and the staged rows are complete
    scatter_rows<D>(sDS, rows_here, tok, t * 128, dqkv, C3, head * D, tid, 256);
    __syncthreads();      // staging drained before the next tile's dS lands in the same buffer
    SWB_ACC(6);
  }

  // ================================ sweep B: key-major -> dk, dv ================================
  for (int u = 0; u < ntiles; ++u) {
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // S^T = K^_u Q^T
        umma_bf16_ss(tmem_base, opnd_kmajor(k0, k, u * 128), opnd_kmajor(q0, k, 0), idesc_s, k > 0);
#pragma unroll
      for (int k = 0; k < D / 16; ++k)      // dP^T = V_u dO^T
        umma_bf16_ss(tmem_base + kMaxLP, opnd_kmajor(v0, k, u * 128), opnd_kmajor(g0, k, 0), idesc_s, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 620 + u);
    SWB_ACC(7);
    parity ^= 1;
    tc_fence_after();
    // K^ and V have served their last MMA of this item: start gathering the next item's K^ / V into them
    if (u == ntiles - 1 && has_next) {
      if (next_box) { if (tid == 0) issue_boxes(1, 3, item_next, true); }
      else gather(1, 3, tok_next, head_next);
    }
    {
      const int jk = u * 128 + r;                       // key slot of this thread
      const bool key_ok = jk < L;
      const int key_label = (jk >= label_split) ? 1 : 0;
      unsigned char* myP = sP + r * 16;
      unsigned char* myDS = sDS + r * 16;
      // columns = queries; lse2[q] = +inf for pad queries -> P = 0 there.  Pad key rows only feed discarded output rows,
      // but they are zeroed so that no NaN ever enters the tensor pipe.
      for (int c0 = c_begin; c0 < c_end; c0 += 16) {
        uint32_t sv[16], pv[16];
        tmem_ld_32x16(t_lane + c0, sv);
        tmem_ld_32x16(t_lane + kMaxLP + c0, pv);
        float ls[16], dd[16];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          *reinterpret_cast<float4*>(&ls[j]) = *reinterpret_cast<const float4*>(&lse2[c0 + j]);
          *reinterpret_cast<float4*>(&dd[j]) = *reinterpret_cast<const float4*>(&Dv[c0 + j]);
        }
        tmem_ld_wait();
        float pp[16], ds[16];
        if (plain) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float p = ex2_approx(fmaf(as_f(sv[j]), scale_l2, -ls[j]));
            pp[j] = key_ok ? p : 0.f;
            ds[j] = key_ok ? p * (as_f(pv[j]) - dd[j]) : 0.f;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int qi = c0 + j;
            float s = as_f(sv[j]) * scale_l2;
            if (bias != nullptr && key_ok && qi < L) s += bias[((size_t)head * L + qi) * L + jk] * kLog2e;
            if (((qi >= label_split) ? 1 : 0) != key_label) s += -100.0f * kLog2e;
            const float p = key_ok ? ex2_approx(s - ls[j]) : 0.f;
            pp[j] = p;
            ds[j] = (key_ok && qi < L) ? p * (as_f(pv[j]) - dd[j]) : 0.f;
          }
        }
        *reinterpret_cast<uint4*>(myP + (c0 / 8) * SM::kPCS) = pack8(pp, 0);
        *reinterpret_cast<uint4*>(myP + (c0 / 8 + 1) * SM::kPCS) = pack8(pp, 8);
        *reinterpret_cast<uint4*>(myDS + (c0 / 8) * SM::kPCS) = pack8(ds, 0);
        *reinterpret_cast<uint4*>(myDS + (c0 / 8 + 1) * SM::kPCS) = pack8(ds, 8);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    SWB_ACC(8);
    if (tid == 0) {
      tc_fence_after();
      for (int k = 0; k < LP / 16; ++k)     // dV_u = P^T dO   (dO read n-major: rows = queries = k-dimension)
        umma_bf16_ss(tmem_base, umma_desc_nosw(p0 + 2 * k * SM::kPCS, SM::kPCS, 128),
                     opnd_mnmajor(g0, k), idesc_o, k > 0);
      for (int k = 0; k < LP / 16; ++k)     // dK^_u = dS^T Q^
        umma_bf16_ss(tmem_base + kMaxLP, umma_desc_nosw(ds0 + 2 * k * SM::kPCS, SM::kPCS, 128),
                     opnd_mnmajor(q0, k), idesc_o, k > 0);
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 630 + u);
    SWB_ACC(9);
    parity ^= 1;
    tc_fence_after();
    // ... and Q^ / dO after the last dV / dK^ MMAs
    if (u == ntiles - 1 && has_next) {
      if (next_box) {
        if (tid == 0) { issue_boxes(0, 1, item_next, false); issue_boxes(3, 4, item_next, false); }
      } else {
        gather(0, 1, tok_next, head_next);
        gather(3, 4, tok_next, head_next);
      }
    }
    const int rows_here = min(128, L - u * 128);
    {
      // warps 0-3: dv rows (staged in the P tile); warps 4-7: dk rows (staged in the dS tile)
      const int jk = u * 128 + r;
      const bool key_ok = jk < L;
      float acc[D];
#pragma unroll
      for (int c0 = 0; c0 < D; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_lane + half * kMaxLP + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[c0 + j] = as_f(v[j]);
      }
      if (key_ok) {
        if (half == 0) {
          park_row<D>(sP, r, acc);
        } else {                                         // dk = inv_norm * (dk^ - k^ <k^, dk^>), dk^ = scale * (dS^T Q^)
          float dot = 0.f;
          float kh[D];
#pragma unroll
          for (int c = 0; c < D / 8; ++c) {
            float t8[8];
            ld8(qkv + (size_t)tok[jk] * C3 + C + head * D + c * 8, t8);   // L2-resident; sK may already hold the next item
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              kh[c * 8 + e] = t8[e];
              acc[c * 8 + e] *= scale;
              dot = fmaf(t8[e], acc[c * 8 + e], dot);
            }
          }
          const float ink = inv_norm[(size_t)tok[jk] * 2 * g.heads + g.heads + head];
#pragma unroll
          for (int c = 0; c < D; ++c) acc[c] = ink * (acc[c] - kh[c] * dot);
          park_row<D>(sDS, r, acc);
        }
      }
    }
    tc_fence_before();
    __syncthreads();
    // 128 threads drain each staging tile with whole-row stores
    if (half == 0) scatter_rows<D>(sP, rows_here, tok, u * 128, dqkv, C3, 2 * C + head * D, tid, 128);
    else scatter_rows<D>(sDS, rows_here, tok, u * 128, dqkv, C3, C + head * D, tid - 128, 128);
    __syncthreads();
    SWB_ACC(10);
  }

  // ---- d(scale) = sum dS o cos: per-warp partial -> per-head slot of this CTA ------------------------------------------
  dsc_acc = warp_sum(dsc_acc);
  if (lane == 0) atomicAdd(&dsc_heads[head], dsc_acc);
  cur_box = next_box;
  }   // item loop
  __syncthreads();
  if (tid < g.heads) {
    const float v = dsc_heads[tid];
    if (v != 0.f) atomicAdd(dscale + tid, v);
  }
  if (g_phase_buf != nullptr && tid == 0 && blockIdx.x < 4096)
    for (int i = 0; i < 12; ++i) g_phase_buf[blockIdx.x * 16 + i] = ph_acc[i];
#undef SWB_ACC
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
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

// ws: optional workspace of B*H*W*heads floats.  With it the persistent kernel runs (operands arrive as TMA boxes while the
// previous window is still being processed, D = <dO, O> comes from a streaming pre-pass); without it the one-CTA-per-window
// kernel does everything in place.
int attn_tcgen05_bwd(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o,
                     const void* d_o, const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, int B, int H, int W,
                     int C, int heads, int Wh, int Ww, int s0, int s1, cudaStream_t stream, float* det_part) {
  AttnGeom g;
  if (int e = attn_make_geom(g, B, H, W, C, heads, Wh, Ww, s0, s1)) return e;
  static int variant = -1;
  if (variant < 0) {
    const char* e = getenv("SWINB200_ATTN_BWD");
    variant = e ? atoi(e) : 3;   // 1 = one CTA per (window, head);  2 = persistent two-sweep kernel;  3 = single-pass warp-specialised;  4 = generic
  }
  if (!attn_is_specialised(g) || variant == 4)
    return attn_tcgen05_gen_bwd(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, ws, g, stream, det_part);
  const bool aligned = ((uintptr_t)qkv % 16 == 0) && ((uintptr_t)d_o % 16 == 0);
  if (variant == 3 && ws != nullptr && aligned)
    return attn_tcgen05_bwd3(qkv, inv_norm, scale, bias, o, d_o, lse, dqkv, dscale, dbias, ws, g, stream, det_part);
  if (det_part != nullptr) {
    set_error("window_attn_bwd: the one-CTA-per-window and two-sweep kernels (SWINB200_ATTN_BWD=1/2, no workspace or unaligned "
              "operands) have no deterministic version");
    return SWINB200_ERR_UNSUPPORTED;
  }
  if (variant == 1 || ws == nullptr || !aligned) {
    using SM = BwdSmem<96>;
    static bool configured = false;
    if (!configured) {
      SWB_CUDA(cudaFuncSetAttribute(attn_tc_bwd_kernel<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
      configured = true;
    }
    attn_tc_bwd_kernel<96><<<B * g.nW * heads, 256, SM::kBytes, stream>>>(
        (const __nv_bfloat16*)qkv, inv_norm, scale, bias, (const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o, lse,
        (__nv_bfloat16*)dqkv, dscale, dbias, g);
  } else {
    using SM = Bwd2Smem<96>;
    static bool configured2 = false;
    if (!configured2) {
      SWB_CUDA(cudaFuncSetAttribute(attn_tc_bwd2_kernel<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
      configured2 = true;
    }
    CUtensorMap tm_qkv, tm_do;
    if (int e = attn_make_window_tmap(&tm_qkv, qkv, B, H, W, 3 * C, Wh, Ww)) return e;
    if (int e = attn_make_window_tmap(&tm_do, d_o, B, H, W, C, Wh, Ww)) return e;
    const long long n_pairs = (long long)B * H * W * heads;
    attn_rowdot_kernel<<<(unsigned)((n_pairs * 4 + 255) / 256), 256, 0, stream>>>((const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o,
                                                                                  ws, n_pairs, C / heads);
    SWB_LAUNCH_CHECK();
    const int grid = min(B * g.nW * heads, sm_count());
    attn_tc_bwd2_kernel<96><<<grid, 256, SM::kBytes, stream>>>(
        tm_qkv, tm_do, ws, (const __nv_bfloat16*)qkv, inv_norm, scale, bias, (const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o, lse,
        (__nv_bfloat16*)dqkv, dscale, dbias, g);
  }
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

}  // namespace swinb200

extern "C" int swinb200_debug_attn_phase_buffer(void* buf) { return swinb200::attn_set_phase_buffer((long long*)buf); }
