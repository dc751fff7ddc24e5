// tcgen05 window attention for every geometry the specialised 9x18 / head_dim-96 kernels (attn_tc_fwd4.cu,
// attn_tc_bwd3.cu) are not instantiated for: head_dim 48 / 64 / 96 / 128 / 192 / 256 and windows of any size (BASELINE
// config 5: 6x12, 12x24, 18x36 ...).  Restates WindowMultiHeadAttention.forward (reference networks/swinv2_global.py:300-319)
// and its backward as three flash-style kernels of one shape:
//
//   a CTA owns one 128-row "stationary" tile X of a (sample, window, head) item and streams 64-row tiles Y past it
//
//   forward      X = Q^ rows          Y = (K^, V) rows     S = X Y0^T -> P -> O += P Y1                  (thread = query)
//   backward A   X = (Q^, dO) rows    Y = (K^, V) rows     S, dP = X1 Y1^T -> dS -> dQ^ += dS Y0         (thread = query)
//   backward B   X = (K^, V) rows     Y = (Q^, dO) rows    S^T, dP^T -> P^T, dS^T -> dV += P^T Y1, dK^ += dS^T Y0   (thread = key)
//
// head_dim 256 (the e2048 / 8-head config) does not fit that shape everywhere: backward A streams 32-row tiles (two 128 x 256
// stationary operands leave no room for 64-row double buffers), and backward B -- two 256-column fp32 accumulators plus the
// S^T / dP^T tiles exceed the 512 tensor-memory columns at any tile height -- runs as two passes over the same items:
//   backward V   X = K^ rows          Y = (Q^, dO) rows    S^T -> P^T -> dV += P^T Y1                                  (thread = key)
//   backward K   X = (K^, V) rows     Y = (Q^, dO) rows    S^T, dP^T -> dS^T -> dK^ += dS^T Y0, d(bias)              (thread = key)
// d(scale) is summed by backward A only and d(bias) by backward B / K only, so the split counts neither twice.
//
// S-type products take both operands from shared memory (un-swizzled core-matrix layout [16-byte chunk][row][8 elements]: the
// same bytes serve K-major and MN-major descriptors, so no transposed copy exists anywhere); P / dS are packed to bf16 in place
// in tensor memory and feed the second product as the TS-mode A operand.  The logits of cosine attention are bounded: without
// a bias table (and scale*log2e < 60) the forward's softmax offset is the bound scale*1 and no maximum is ever taken;
// otherwise a running maximum is kept per row and the accumulator rows are rescaled in tensor memory only when it grows by more
// than 2^8 (rare: the tiles of one window see similar logits).  Bias values reach the thread that owns their row through a
// per-warp shared-memory slab and are fetched one 16-column chunk ahead.  Y tiles are double-buffered with cp.async groups; two
// to four CTAs per SM overlap one CTA's softmax with another's gathers.  The roll / window partition is the address
// computation of the gather (win_token), the shift mask the label predicate of the specialised kernels.
#include "attn_tc.cuh"

namespace swinb200 {
namespace {

constexpr int kModeFwd = 0, kModeBwdQ = 1, kModeBwdKV = 2, kModeBwdV = 3, kModeBwdK = 4;
__host__ __device__ constexpr bool key_mode(int mode) { return mode >= kModeBwdKV; }     // thread = key, Y = (Q^, dO)

__host__ __device__ constexpr int pow2_cols(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : n <= 256 ? 256 : 512; }

template <int D, int KT, int MODE, bool HAS_BIAS>
struct GenCfg {
  static constexpr int kChunks = D / 8;
  static constexpr int kNX = (MODE == kModeFwd || MODE == kModeBwdV) ? 1 : 2;
  static constexpr int kCSX = 128 * 16 + 16;                 // chunk stride of the stationary tile (+16: spreads the gather over banks)
  static constexpr int kTileX = kChunks * kCSX;
  static constexpr int kCSY = KT * 16 + 16;
  static constexpr int kTileY = kChunks * kCSY;
  static constexpr int kOffX = 0;
  static constexpr int kOffY = kNX * kTileX;                  // [buffer][operand]
  static constexpr int kOffTokX = kOffY + 4 * kTileY;
  static constexpr int kOffColA = kOffTokX + 128 * 4;         // [2][KT]  log2-domain LSE of the streamed query rows (backward B)
  static constexpr int kOffColB = kOffColA + 2 * KT * 4;      // [2][KT]  D = <dO, O> of the streamed query rows
  static constexpr int kOffBias = kOffColB + 2 * KT * 4;      // [4 warps][32 rows][20] bias pieces on their way to their rows (fwd / A)
  static constexpr int kOffBar = kOffBias + ((key_mode(MODE) || !HAS_BIAS) ? 0 : 4 * 32 * 20 * 4);
  static constexpr int kBytes = kOffBar + 64;
  static constexpr int kStagePitch = D * 2 + 16;              // output rows parked in the (dead) Y buffers
  static constexpr int kColS = 0, kColDP = KT;
  static constexpr int kColAcc0 = (kNX == 1) ? KT : 2 * KT;     // one stationary operand: no dP tile
  static constexpr int kColAcc1 = kColAcc0 + D;
  static constexpr int kColAdd = kColAcc0 + D;               // forward: log2-domain addend (bias + mask) of the current tile
  static constexpr int kColsUsed = kColAcc0 + ((MODE == kModeBwdKV) ? 2 : 1) * D + ((MODE == kModeFwd && HAS_BIAS) ? KT : 0);
  static constexpr int kTmemCols = pow2_cols(kColsUsed);
  static_assert(D % 16 == 0 && D >= 16 && D <= 256, "head_dim");
  static_assert(KT % 16 == 0 && KT <= 128, "streamed tile");
  static_assert(128 * kStagePitch <= 4 * kTileY, "staging fits the Y buffers");
  static_assert(kColsUsed <= 512, "tensor memory");
  static_assert(kBytes <= 227 * 1024, "shared memory");
};

struct GenArgs {
  const __nv_bfloat16* qkv;      // (T, 3C): q^ | k^ | v, q^ / k^ already L2-normalised per head
  const __nv_bfloat16* d_o;      // (T, C)                                   (backward)
  const float* inv_norm;         // (T, 2 heads) reciprocal norms of q, k      (backward)
  const float* scale;            // (heads) exp(min(logit_scale, ln 100))
  const float* bias;             // (heads, L, L) or null
  const float* Dpre;             // (T, heads) <dO, O>                         (backward)
  float* lse;                    // (2, B, nW, heads, L): LSE | E_P[cos];  written by forward (unless null), read by backward
  __nv_bfloat16* out;            // forward: o (T, C);  backward: dqkv (T, 3C)
  float* dscale;                 // (heads)
  float* dbias;                  // (heads, L, L) or null
};

__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]),
      "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
      : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// DET (deterministic mode): a.dscale holds one slot per (item, X tile, warp) and a.dbias one (L, L) slice per item, all
// written with plain stores (every (query, key) of an item is visited by exactly one thread of the K pass)
template <int D, int KT, int MODE, bool HAS_BIAS, bool DET = false>
__global__ void __launch_bounds__(128) attn_gen_kernel(const GenArgs a, const AttnGeom g) {
  using CF = GenCfg<D, KT, MODE, HAS_BIAS>;
  constexpr float kLog2e = 1.4426950408889634f;
  constexpr float kLn2 = 0.6931471805599453f;
  constexpr float kMaskL2 = -100.0f * kLog2e;
  extern __shared__ __align__(128) unsigned char smem[];
  int* tokX = reinterpret_cast<int*>(smem + CF::kOffTokX);
  float* colA = reinterpret_cast<float*>(smem + CF::kOffColA);
  float* colB = reinterpret_cast<float*>(smem + CF::kOffColB);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + CF::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = g.L, C = g.C, C3 = 3 * g.C;
  const int nX = (L + 127) / 128, nY = (L + KT - 1) / KT;
  const int xt = blockIdx.x % nX;
  const int item = blockIdx.x / nX;
  const int head = item % g.heads;
  const int w = (item / g.heads) % g.nW;
  const int b = item / (g.heads * g.nW);

  // shifted-window mask: slots >= label_split belong to the rows that wrapped around (reference :410-420)
  int label_split = L;
  if (g.s0 > 0) {
    const int first_row = g.H - g.s0 - (w / g.nWw) * g.Wh;
    label_split = first_row <= 0 ? 0 : (first_row >= g.Wh ? L : first_row * g.Ww);
  }
  const bool use_mask = label_split > 0 && label_split < L;
  const bool plain = !HAS_BIAS && !use_mask;

  const int nx = xt * 128 + tid;                 // this thread's stationary slot (query for fwd / A, key for B) == TMEM lane
  const bool row_ok = nx < L;
  const int x_label = (nx >= label_split) ? 1 : 0;
  const size_t row_base = (((size_t)b * g.nW + w) * g.heads + head) * L;     // index of slot 0 in the per-row planes

  // ---- set-up -------------------------------------------------------------------------------------------------------------
  {
    int rr;
    tokX[tid] = row_ok ? win_token(g, b, w, nx, rr) : -1;
  }
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, CF::kTmemCols);
  {
    const int rows_x = min(128, L - xt * 128);
    if (rows_x < 128) {                          // pad rows of the stationary tile: exact zeros (they meet P = 0, and 0 * NaN = NaN)
      const int pad = 128 - rows_x;
      for (int i = tid; i < CF::kNX * CF::kChunks * pad; i += 128) {
        const int r = rows_x + i % pad, oc = i / pad;
        *reinterpret_cast<uint4*>(smem + CF::kOffX + (oc / CF::kChunks) * CF::kTileX + (oc % CF::kChunks) * CF::kCSX + r * 16) =
            make_uint4(0, 0, 0, 0);
      }
    }
    if (L % KT != 0)                             // the last streamed tile is ragged: its pad rows must never be NaN bit patterns
      for (int i = tid; i < 4 * CF::kTileY / 16; i += 128) *reinterpret_cast<uint4*>(smem + CF::kOffY + i * 16) = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();

  // stationary operands
  {
    const int rows_x = min(128, L - xt * 128);
    for (int i = tid; i < CF::kNX * rows_x * CF::kChunks; i += 128) {
      const int op = i / (rows_x * CF::kChunks);
      const int rem = i - op * rows_x * CF::kChunks;
      const int r = rem / CF::kChunks, c = rem - r * CF::kChunks;
      const __nv_bfloat16* src;
      if (MODE == kModeFwd) src = a.qkv + (size_t)tokX[r] * C3 + head * D + c * 8;
      else if (MODE == kModeBwdQ) src = (op == 0) ? a.qkv + (size_t)tokX[r] * C3 + head * D + c * 8 : a.d_o + (size_t)tokX[r] * C + head * D + c * 8;
      else src = a.qkv + (size_t)tokX[r] * C3 + (op + 1) * C + head * D + c * 8;
      cp_async16(smem + CF::kOffX + op * CF::kTileX + c * CF::kCSX + r * 16, src);
    }
  }
  // streamed tile t of the item -> buffer `buf`; op_mask bit 0 / 1 selects the operands
  auto gather_y = [&](int t, int buf, int op_mask) {
    const int rows = min(KT, L - t * KT);
    unsigned char* base = smem + CF::kOffY + buf * 2 * CF::kTileY;
    for (int i = tid; i < rows * CF::kChunks; i += 128) {
      const int r = i / CF::kChunks, c = i - r * CF::kChunks;
      int rr;
      const size_t tk = (size_t)win_token(g, b, w, t * KT + r, rr);
      if (key_mode(MODE)) {
        if (op_mask & 1) cp_async16(base + c * CF::kCSY + r * 16, a.qkv + tk * C3 + head * D + c * 8);
        if (op_mask & 2) cp_async16(base + CF::kTileY + c * CF::kCSY + r * 16, a.d_o + tk * C + head * D + c * 8);
      } else {
        if (op_mask & 1) cp_async16(base + c * CF::kCSY + r * 16, a.qkv + tk * C3 + C + head * D + c * 8);
        if (op_mask & 2) cp_async16(base + CF::kTileY + c * CF::kCSY + r * 16, a.qkv + tk * C3 + 2 * C + head * D + c * 8);
      }
    }
    if (key_mode(MODE) && tid < KT) {            // per-column (= streamed query) terms
      if (tid < rows) {
        int rr;
        const size_t tk = (size_t)win_token(g, b, w, t * KT + tid, rr);
        cp_async4(colA + buf * KT + tid, a.lse + row_base + t * KT + tid);
        cp_async4(colB + buf * KT + tid, a.Dpre + tk * g.heads + head);
      } else {
        colA[buf * KT + tid] = INFINITY;         // pad queries: P = 2^(-inf) = 0
        colB[buf * KT + tid] = 0.f;
      }
    }
  };

  const float scale = a.scale[head];
  const float scale_l2 = scale * kLog2e;
  // forward: the bound scale*1 on the logits replaces the row maximum when nothing is added to them; otherwise a running
  // maximum, re-based (accumulator rows rescaled in tensor memory) only when it grows by more than 2^8
  const bool bounded = !HAS_BIAS && scale_l2 < 60.f;
  const int total = nY;

  gather_y(0, 0, 3);
  cp_async_commit();

  // per-row terms of backward A
  float my_lse2 = INFINITY, my_D = 0.f, my_mc = 0.f;
  if (MODE == kModeBwdQ && row_ok) {
    my_lse2 = a.lse[row_base + nx] * kLog2e;
    my_mc = a.lse[(size_t)g.B * g.nW * g.heads * L + row_base + nx];
    my_D = a.Dpre[(size_t)tokX[tid] * g.heads + head];
  }
  // bias[query][key .. key+15] for this thread's query: a warp instruction reading 32 different rows costs 32 L1 tag
  // cycles, so the warp fetches the 32 x 16 block as 16 loads of two 64-byte row pieces each and redistributes it through
  // a 2.5 KB slab (row pitch 80 B: the 16-byte reads are conflict-free)
  // Values are fetched one 16-column chunk ahead (across tile boundaries too), so the L2 latency hides behind the arithmetic
  // of the current chunk and the waits between tiles.  Backward B (thread = key) reads bias[query][key] with consecutive
  // lanes on consecutive keys: coalesced as it is, prefetched the same way.
  float* sbias = reinterpret_cast<float*>(smem + CF::kOffBias) + warp * (32 * 20);
  float nb[16];
  auto bias_fetch = [&](int y0_) {               // y0_ = first streamed slot of the chunk; out-of-range chunks fetch nothing
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (key_mode(MODE)) {
        const int qi = y0_ + i;
        nb[i] = (row_ok && qi < L) ? __ldg(a.bias + ((size_t)head * L + qi) * L + nx) : 0.f;
      } else {
        const int row = 2 * i + (lane >> 4), col = lane & 15;
        const int q = xt * 128 + warp * 32 + row, key = y0_ + col;
        nb[i] = (q < L && key < L) ? __ldg(a.bias + ((size_t)head * L + q) * L + key) : 0.f;
      }
    }
  };
  auto bias_take = [&](float (&bv)[16]) {        // the chunk fetched last, as log2-domain addends of this thread's 16 columns
    if (key_mode(MODE)) {
#pragma unroll
      for (int j = 0; j < 16; ++j) bv[j] = nb[j] * kLog2e;
    } else {
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 16; ++i) sbias[(2 * i + (lane >> 4)) * 20 + (lane & 15)] = nb[i] * kLog2e;
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 16; j += 4) *reinterpret_cast<float4*>(&bv[j]) = *reinterpret_cast<const float4*>(sbias + lane * 20 + j);
    }
  };
  // first slot of the chunk after (tile u, column c0) in processing order
  auto next_chunk = [&](int u, int c0) {
    if (c0 + 16 < KT) return u * KT + c0 + 16;
    return (u + 1 >= total) ? L : (u + 1) * KT;
  };
  if (HAS_BIAS) bias_fetch(0);

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t t_lane = tmem_base + ((uint32_t)(warp * 32) << 16);
  const uint32_t x0 = smem_u32(smem + CF::kOffX);
  const uint32_t y0 = smem_u32(smem + CF::kOffY);
  const uint32_t idesc_s = umma_idesc_bf16(128, KT, false, false);      // [128 x KT] = X(k-major) Y(k-major)^T
  const uint32_t idesc_o = umma_idesc_bf16(128, D, false, true);        // [128 x D]  = A(tensor memory) Y(n-major)
  uint32_t parity = 0;

  float row_max = -INFINITY, row_sum = 0.f, cos_sum = 0.f, dsc_acc = 0.f;

  for (int u = 0; u < total; ++u) {
    const int t = u;
    const int buf = u & 1;
    if (u + 1 < total) gather_y(u + 1, buf ^ 1, 3);
    cp_async_commit();
    cp_async_wait_1();                           // everything but the group just committed: tile u (and X) have landed
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    const uint32_t yb = y0 + buf * 2 * CF::kTileY;
    if (tid == 0) {
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < D / 16; ++k)
        umma_bf16_ss(tmem_base + CF::kColS, umma_desc_nosw(x0 + 2 * k * CF::kCSX, CF::kCSX, 128),
                     umma_desc_nosw(yb + 2 * k * CF::kCSY, CF::kCSY, 128), idesc_s, k > 0);
      if (CF::kNX == 2) {
#pragma unroll
        for (int k = 0; k < D / 16; ++k)
          umma_bf16_ss(tmem_base + CF::kColDP, umma_desc_nosw(x0 + CF::kTileX + 2 * k * CF::kCSX, CF::kCSX, 128),
                       umma_desc_nosw(yb + CF::kTileY + 2 * k * CF::kCSY, CF::kCSY, 128), idesc_s, k > 0);
      }
      umma_commit(bar);
    }
    mbar_wait(bar, parity, 800 + MODE);
    parity ^= 1;
    tc_fence_after();

    const int y_base = t * KT;                   // first streamed slot of this tile
    const bool ragged = y_base + KT > L;
    if (MODE == kModeFwd) {
      if (!bounded) {
        // sub-pass 1: the addend (bias + mask, -inf for pad keys) of every column goes to scratch columns, tile maximum on the way
        float tile_max = -INFINITY;
#pragma unroll 1
        for (int c0 = 0; c0 < KT; c0 += 16) {
          uint32_t v[16];
          tmem_ld_32x16(t_lane + CF::kColS + c0, v);
          float bv[16];
          if (HAS_BIAS) {
            bias_take(bv);
            bias_fetch(next_chunk(u, c0));
          }
          tmem_ld_wait();
          float add[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int key = y_base + c0 + j;
            float ad = HAS_BIAS ? bv[j] : 0.f;
            if (use_mask && ((key >= label_split) ? 1 : 0) != x_label) ad += kMaskL2;
            if (ragged && key >= L) ad = -INFINITY;
            add[j] = ad;
            tile_max = fmaxf(tile_max, fmaf(as_f(v[j]), scale_l2, ad));
          }
          if (HAS_BIAS) tmem_st_32x16(t_lane + CF::kColAdd + c0, add);      // without a table the addend is recomputed below
        }
        if (HAS_BIAS) tmem_st_wait();
        const bool grow = tile_max > row_max + 8.f;            // first tile: row_max = -inf
        if (__any_sync(0xffffffffu, grow)) {
          const float f = grow ? ex2_approx(row_max - tile_max) : 1.f;
          if (t > 0) {
#pragma unroll 1
            for (int c0 = 0; c0 < D; c0 += 16) {
              uint32_t v[16];
              tmem_ld_32x16(t_lane + CF::kColAcc0 + c0, v);
              tmem_ld_wait();
              float r16[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) r16[j] = as_f(v[j]) * f;
              tmem_st_32x16(t_lane + CF::kColAcc0 + c0, r16);
            }
          }
          row_sum *= f;
          cos_sum *= f;
          if (grow) row_max = tile_max;
        }
      }
      const float off = bounded ? scale_l2 : row_max;
#pragma unroll 1
      for (int c0 = 0; c0 < KT; c0 += 16) {
        uint32_t v[16], ad[16];
        tmem_ld_32x16(t_lane + CF::kColS + c0, v);
        if (HAS_BIAS) tmem_ld_32x16(t_lane + CF::kColAdd + c0, ad);
        tmem_ld_wait();
        float p[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int key = y_base + c0 + j;
          float s = as_f(v[j]) * scale_l2;
          if (HAS_BIAS) s += as_f(ad[j]);                       // bias + mask, -inf for pad keys
          else if (use_mask && ((key >= label_split) ? 1 : 0) != x_label) s += kMaskL2;
          p[j] = ex2_approx(s - off);
          if (!HAS_BIAS && ragged && key >= L) p[j] = 0.f;
          row_sum += p[j];
          cos_sum = fmaf(p[j], as_f(v[j]), cos_sum);
        }
        tmem_st_32x8(t_lane + CF::kColS + c0 / 2, pack8(p, 0), pack8(p, 8));     // keys [c0, c0+16) -> 8 packed columns, already consumed
      }
    } else if (MODE == kModeBwdQ) {
      float dsc_tile = 0.f;
#pragma unroll 1
      for (int c0 = 0; c0 < KT; c0 += 16) {
        uint32_t v[16], dp[16];
        tmem_ld_32x16(t_lane + CF::kColS + c0, v);
        tmem_ld_32x16(t_lane + CF::kColDP + c0, dp);
        float bv[16];
        if (HAS_BIAS) {
          bias_take(bv);
          bias_fetch(next_chunk(u, c0));
        }
        tmem_ld_wait();
        float ds[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int key = y_base + c0 + j;
          const float cosv = as_f(v[j]);
          float s = cosv * scale_l2;
          if (!plain) {
            if (HAS_BIAS) s += bv[j];
            if (use_mask && ((key >= label_split) ? 1 : 0) != x_label) s += kMaskL2;
          }
          const float p = ex2_approx(s - my_lse2);               // pad query rows: lse = +inf -> 0
          float d = p * (as_f(dp[j]) - my_D);
          if (ragged && key >= L) d = 0.f;
          ds[j] = d;
          dsc_tile = fmaf(d, cosv - my_mc, dsc_tile);
        }
        tmem_st_32x8(t_lane + CF::kColDP + c0 / 2, pack8(ds, 0), pack8(ds, 8));
      }
      if (row_ok) dsc_acc += dsc_tile;
    } else {
      const float* cA = colA + buf * KT;
      const float* cB = colB + buf * KT;
#pragma unroll 1
      for (int c0 = 0; c0 < KT; c0 += 16) {
        uint32_t v[16], dp[16];
        tmem_ld_32x16(t_lane + CF::kColS + c0, v);
        if (MODE != kModeBwdV) tmem_ld_32x16(t_lane + CF::kColDP + c0, dp);
        float ls[16], dd[16];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          *reinterpret_cast<float4*>(&ls[j]) = *reinterpret_cast<const float4*>(cA + c0 + j);
          *reinterpret_cast<float4*>(&dd[j]) = *reinterpret_cast<const float4*>(cB + c0 + j);
        }
        float bv[16];
        if (HAS_BIAS) {
          bias_take(bv);
          bias_fetch(next_chunk(u, c0));
        }
        tmem_ld_wait();
        float pp[16], ds[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int qi = y_base + c0 + j;
          float s = as_f(v[j]) * scale_l2;
          if (!plain) {
            if (HAS_BIAS) s += bv[j];
            if (use_mask && ((qi >= label_split) ? 1 : 0) != x_label) s += kMaskL2;
          }
          const float p = row_ok ? ex2_approx(fmaf(-ls[j], kLog2e, s)) : 0.f;     // pad queries: lse = +inf -> 0
          pp[j] = p;
          if (MODE != kModeBwdV) {
            const float d = (qi < L) ? p * (as_f(dp[j]) - dd[j]) : 0.f;
            ds[j] = d;
            if constexpr (DET) {
              if (a.dbias != nullptr && row_ok && qi < L) a.dbias[((size_t)item * L + qi) * L + nx] = d;
            } else {
              if (a.dbias != nullptr && row_ok && qi < L) atomicAdd(a.dbias + ((size_t)head * L + qi) * L + nx, d);
            }
          }
        }
        if (MODE != kModeBwdK) tmem_st_32x8(t_lane + CF::kColS + c0 / 2, pack8(pp, 0), pack8(pp, 8));
        if (MODE != kModeBwdV) tmem_st_32x8(t_lane + CF::kColDP + c0 / 2, pack8(ds, 0), pack8(ds, 8));
      }
    }
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t acc = (t > 0) ? 1u : 0u;
      if (MODE == kModeFwd) {
#pragma unroll
        for (int k = 0; k < KT / 16; ++k)        // O += P V
          umma_bf16_ts(tmem_base + CF::kColAcc0, tmem_base + CF::kColS + k * 8, umma_desc_nosw(yb + CF::kTileY + k * 256, 128, CF::kCSY),
                       idesc_o, acc | (uint32_t)(k > 0));
      } else if (MODE == kModeBwdQ) {
#pragma unroll
        for (int k = 0; k < KT / 16; ++k)        // dQ^ += dS K^
          umma_bf16_ts(tmem_base + CF::kColAcc0, tmem_base + CF::kColDP + k * 8, umma_desc_nosw(yb + k * 256, 128, CF::kCSY), idesc_o,
                       acc | (uint32_t)(k > 0));
      } else {
        if (MODE != kModeBwdK) {
#pragma unroll
          for (int k = 0; k < KT / 16; ++k)      // dV += P^T dO
            umma_bf16_ts(tmem_base + CF::kColAcc0, tmem_base + CF::kColS + k * 8, umma_desc_nosw(yb + CF::kTileY + k * 256, 128, CF::kCSY),
                         idesc_o, acc | (uint32_t)(k > 0));
        }
        if (MODE != kModeBwdV) {
          const uint32_t col_dk = (MODE == kModeBwdKV) ? CF::kColAcc1 : CF::kColAcc0;
#pragma unroll
          for (int k = 0; k < KT / 16; ++k)      // dK^ += dS^T Q^
            umma_bf16_ts(tmem_base + col_dk, tmem_base + CF::kColDP + k * 8, umma_desc_nosw(yb + k * 256, 128, CF::kCSY), idesc_o,
                         acc | (uint32_t)(k > 0));
        }
      }
      umma_commit(bar);
    }
    // the products above read buffer `buf`, which the next iteration's gather (tile u+2) overwrites: wait here
    mbar_wait(bar, parity, 810 + MODE);
    parity ^= 1;
    tc_fence_after();
  }

  // ---- epilogue: accumulator rows -> bf16 -> staging (the Y buffers are dead) -> whole-row global stores -------------------
  unsigned char* stage = smem + CF::kOffY;
  const int rows_x = min(128, L - xt * 128);
  auto scatter = [&](int ld, int col0) {
    for (int i = tid; i < rows_x * CF::kChunks; i += 128) {
      const int r = i / CF::kChunks, c = i - r * CF::kChunks;
      *reinterpret_cast<uint4*>(a.out + (size_t)tokX[r] * ld + col0 + c * 8) =
          *reinterpret_cast<const uint4*>(stage + r * CF::kStagePitch + c * 16);
    }
  };
  // (acc columns [col, col + D) * mul - [use_x] xhat * sub) * post  ->  staging row (xhat = this row of stationary operand 0)
  auto park = [&](uint32_t col, float mul, bool use_x, float sub, float post) {
#pragma unroll 1
    for (int c0 = 0; c0 < D; c0 += 16) {
      uint32_t v[16];
      tmem_ld_32x16(t_lane + col + c0, v);
      tmem_ld_wait();
      float r16[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) r16[j] = as_f(v[j]) * mul;
      if (use_x) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float x8[8];
          ld8(reinterpret_cast<const __nv_bfloat16*>(smem + CF::kOffX + (c0 / 8 + h) * CF::kCSX + tid * 16), x8);
#pragma unroll
          for (int e = 0; e < 8; ++e) r16[h * 8 + e] = fmaf(-x8[e], sub, r16[h * 8 + e]);
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) r16[j] *= post;
      if (row_ok) {
        *reinterpret_cast<uint4*>(stage + tid * CF::kStagePitch + c0 * 2) = pack8(r16, 0);
        *reinterpret_cast<uint4*>(stage + tid * CF::kStagePitch + c0 * 2 + 16) = pack8(r16, 8);
      }
    }
  };
  // <xhat, acc * mul> over the row
  auto row_dot = [&](uint32_t col, float mul) {
    float dot = 0.f;
#pragma unroll 1
    for (int c0 = 0; c0 < D; c0 += 16) {
      uint32_t v[16];
      tmem_ld_32x16(t_lane + col + c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float x8[8];
        ld8(reinterpret_cast<const __nv_bfloat16*>(smem + CF::kOffX + (c0 / 8 + h) * CF::kCSX + tid * 16), x8);
#pragma unroll
        for (int e = 0; e < 8; ++e) dot = fmaf(x8[e], as_f(v[h * 8 + e]) * mul, dot);
      }
    }
    return dot;
  };

  if (MODE == kModeFwd) {
    if (row_ok && a.lse != nullptr) {       // null: forward-only run
      const float off = bounded ? scale_l2 : row_max;
      a.lse[row_base + nx] = (off + log2f(row_sum)) * kLn2;
      a.lse[(size_t)g.B * g.nW * g.heads * L + row_base + nx] = cos_sum / row_sum;
    }
    park(CF::kColAcc0, 1.0f / row_sum, false, 0.f, 1.f);
    __syncthreads();
    scatter(C, head * D);
  } else if (MODE == kModeBwdQ) {
    // dq = inv_norm * (dq^ - q^ <q^, dq^>),  dq^ = scale * (dS K^)
    const float dot = row_dot(CF::kColAcc0, scale);
    const float inq = row_ok ? a.inv_norm[(size_t)tokX[tid] * 2 * g.heads + head] : 0.f;
    park(CF::kColAcc0, scale, true, dot, inq);
    __syncthreads();
    scatter(C3, head * D);
    dsc_acc = warp_sum(dsc_acc);
    if constexpr (DET) {
      if (lane == 0) a.dscale[((size_t)item * nX + xt) * 4 + warp] = dsc_acc;
    } else {
      if (lane == 0 && dsc_acc != 0.f) atomicAdd(a.dscale + head, dsc_acc);
    }
  } else {
    if (MODE != kModeBwdK) {
      park(CF::kColAcc0, 1.f, false, 0.f, 1.f);  // dv
      __syncthreads();
      scatter(C3, 2 * C + head * D);
      __syncthreads();
    }
    if (MODE != kModeBwdV) {
      const uint32_t col_dk = (MODE == kModeBwdKV) ? CF::kColAcc1 : CF::kColAcc0;
      const float dot = row_dot(col_dk, scale);
      const float ink = row_ok ? a.inv_norm[(size_t)tokX[tid] * 2 * g.heads + g.heads + head] : 0.f;
      park(col_dk, scale, true, dot, ink);
      __syncthreads();
      scatter(C3, C + head * D);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, CF::kTmemCols);
  }
}

template <int D, int KT, int MODE, bool HAS_BIAS, bool DET = false>
int launch_gen_b(const GenArgs& a, const AttnGeom& g, cudaStream_t stream) {
  using CF = GenCfg<D, KT, MODE, HAS_BIAS>;
  static bool configured = false;
  if (!configured) {
    SWB_CUDA(cudaFuncSetAttribute(attn_gen_kernel<D, KT, MODE, HAS_BIAS, DET>, cudaFuncAttributeMaxDynamicSharedMemorySize, CF::kBytes));
    configured = true;
  }
  const long long ctas = (long long)g.B * g.nW * g.heads * ((g.L + 127) / 128);
  if (ctas > 0x7fffffffLL) {
    set_error("window_attn (tcgen05): %lld CTAs exceed the grid limit", ctas);
    return SWINB200_ERR_UNSUPPORTED;
  }
  attn_gen_kernel<D, KT, MODE, HAS_BIAS, DET><<<(unsigned)ctas, 128, CF::kBytes, stream>>>(a, g);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}
// det: only the backward modes have a deterministic instantiation (the forward sums nothing across CTAs)
template <int D, int KT, int MODE>
int launch_gen(const GenArgs& a, const AttnGeom& g, cudaStream_t stream, bool det = false) {
  if constexpr (MODE != kModeFwd) {
    if (det) return a.bias != nullptr ? launch_gen_b<D, KT, MODE, true, true>(a, g, stream) : launch_gen_b<D, KT, MODE, false, true>(a, g, stream);
  }
  return a.bias != nullptr ? launch_gen_b<D, KT, MODE, true>(a, g, stream) : launch_gen_b<D, KT, MODE, false>(a, g, stream);
}

// head_dim 256: 206 KB of shared memory for the forward at KT = 64 and for backward A at KT = 32; backward B as the V pass
// (KT = 64) followed by the K pass (KT = 32), 196 KB each; every one of them allocates 512 tensor-memory columns
template <int MODE>
int launch_gen_256(const GenArgs& a, const AttnGeom& g, cudaStream_t stream, bool det) {
  if constexpr (MODE == kModeFwd) return launch_gen<256, 64, kModeFwd>(a, g, stream);
  if constexpr (MODE == kModeBwdQ) return launch_gen<256, 32, kModeBwdQ>(a, g, stream, det);
  if constexpr (MODE == kModeBwdKV) {
    if (int e = launch_gen<256, 64, kModeBwdV>(a, g, stream, det)) return e;
    return launch_gen<256, 32, kModeBwdK>(a, g, stream, det);
  }
}

template <int MODE>
int dispatch_gen(const GenArgs& a, const AttnGeom& g, cudaStream_t stream, bool det = false) {
  switch (g.C / g.heads) {
    case 48: return launch_gen<48, 64, MODE>(a, g, stream, det);
    case 64: return launch_gen<64, 64, MODE>(a, g, stream, det);
    case 96: return launch_gen<96, 64, MODE>(a, g, stream, det);
    case 128: return launch_gen<128, 64, MODE>(a, g, stream, det);
    case 192: return launch_gen<192, 64, MODE>(a, g, stream, det);
    case 256: return launch_gen_256<MODE>(a, g, stream, det);
    default:
      set_error("window_attn (tcgen05): head_dim %d is not instantiated (48, 64, 96, 128, 192, 256)", g.C / g.heads);
      return SWINB200_ERR_UNSUPPORTED;
  }
}

}  // namespace

bool attn_gen_supports(int head_dim) {
  return head_dim == 48 || head_dim == 64 || head_dim == 96 || head_dim == 128 || head_dim == 192 || head_dim == 256;
}

int attn_tcgen05_gen_fwd(const void* qkv, const float* scale, const float* bias, void* o, float* lse, const AttnGeom& g, cudaStream_t stream) {
  GenArgs a{};
  a.qkv = (const __nv_bfloat16*)qkv; a.scale = scale; a.bias = bias; a.out = (__nv_bfloat16*)o; a.lse = lse;
  return dispatch_gen<kModeFwd>(a, g, stream);
}

int attn_tcgen05_gen_bwd(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o, const void* d_o,
                         const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, const AttnGeom& g, cudaStream_t stream,
                         float* det_part) {
  const long long n_pairs = (long long)g.B * g.H * g.W * g.heads;
  attn_rowdot_kernel<<<(unsigned)((n_pairs * 4 + 255) / 256), 256, 0, stream>>>((const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o, ws,
                                                                                n_pairs, g.C / g.heads);
  SWB_LAUNCH_CHECK();
  GenArgs a{};
  a.qkv = (const __nv_bfloat16*)qkv; a.d_o = (const __nv_bfloat16*)d_o; a.inv_norm = inv_norm; a.scale = scale; a.bias = bias;
  a.Dpre = ws; a.lse = const_cast<float*>(lse); a.out = (__nv_bfloat16*)dqkv; a.dscale = dscale; a.dbias = dbias;
  if (det_part == nullptr) {
    if (int e = dispatch_gen<kModeBwdQ>(a, g, stream)) return e;
    return dispatch_gen<kModeBwdKV>(a, g, stream);
  }
  const int bw = g.B * g.nW, slots = 4 * ((g.L + 127) / 128);
  const long long dbias_n = (long long)g.heads * g.L * g.L;
  a.dscale = det_part;
  a.dbias = (dbias != nullptr) ? det_part + attn_det_dscale_slots(g) : nullptr;
  if (int e = dispatch_gen<kModeBwdQ>(a, g, stream, true)) return e;
  if (int e = dispatch_gen<kModeBwdKV>(a, g, stream, true)) return e;
  if (int e = ordered_reduce(det_part, bw, (long long)g.heads * slots, g.heads, slots, dscale, 1, stream)) return e;
  if (dbias != nullptr) return ordered_reduce(a.dbias, bw, dbias_n, dbias_n, 1, dbias, 1, stream);
  return SWINB200_OK;
}

}  // namespace swinb200
