// tcgen05 windowed cosine attention, forward, 9x18 windows at head_dim 96: TWO (window, head) items in flight per SM.
//
// Reference math: swinv2_global.py:300-318 -- S = scale * q^ k^T (+ CPB bias) (+ shift mask), P = softmax(S), O = P v; the
// roll / window_partition / window_reverse copies (:89-119, 446-478) are folded into the TMA box coordinates and the scatter.
// Operands arrive as TMA window boxes: per 32-channel chunk, one [32 channels x Ww x Wh] box of a 5-D tensor map over the
// (B, H, W, 3C) activation (attn_make_window_tmap), 64B-swizzled; windows that wrap around the cyclic shift are gathered with
// cp.async instead.  K^ / V pad rows [L, 176) are zeroed once and never written again, so padded keys contribute exact zeros.
//
// With one item per SM at a time every phase of that item waits for the previous one (DESIGN.md 5.0: no unit is busy more
// than 25 %).  Here a CTA is two independent halves, each with four compute warps (thread = query row = TMEM lane), its own
// control warp (one elected lane issues the TMA boxes and every tcgen05.mma), its own (Q^, K^, V) stage in shared memory, its
// own 256 tensor-memory columns and its own barriers; half g takes the CTA's items g, g+2, g+4, ...  While one half waits for an MMA, a TMA box or its row
// stores, the other half's softmax owns the issue slots.
//   per item and half:  for each 128-query tile t:  S_t = Q^_t K^T (SS) -> softmax in tensor memory, P packed in place ->
//                       O_t = P_t V (TS) -> O_t / rowsum into registers (tensor memory is free for S_{t+1}) -> rows parked
//                       in the dead Q^ rows of the stage (same swizzled layout, so tile 1's Q^ rows are never touched)
//                       then: all 162 rows stored as whole 192-byte rows, stage released, next item's boxes requested
//   TMEM columns of half g (base 256 g):  S [0,176)   P bf16 in place [0,88)   O [88,184)
#include <stdlib.h>
#include "attn_tc.cuh"

namespace swinb200 {

constexpr int kF4Halves = 2;
constexpr int kF4Compute = kF4Halves * 128;            // 8 compute warps
constexpr int kF4Threads = kF4Compute + kF4Halves * 32; // + one control warp per half

template <int D>
struct Fwd4Smem {
  static constexpr int kTile = (D / 32) * kCS64;            // one operand: 3 x [176 rows x 64 B]
  static constexpr int kStage = 3 * kTile;                  // Q^, K^, V
  static constexpr int kOffTok = kF4Halves * kStage;        // [2][176] token indices (one table per half)
  static constexpr int kOffBar = kOffTok + kF4Halves * kMaxLP * 4;
  static constexpr int kBytes = kOffBar + 128;
  static_assert(kTile % 512 == 0, "64B-swizzled operand tiles need 512-byte alignment");
  static_assert(kBytes <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ bool elect_one_f4() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void named_bar_f4(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

template <int D>
__global__ void __launch_bounds__(kF4Threads, 1)
attn_tc_fwd4_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __nv_bfloat16* __restrict__ qkv,
                    const float* __restrict__ scale_p, const float* __restrict__ bias, __nv_bfloat16* __restrict__ o,
                    float* __restrict__ lse, const AttnGeom g) {
  using SM = Fwd4Smem<D>;
  constexpr float kLog2e = 1.4426950408889634f;
  constexpr int kPieces = D / 8;
  constexpr int kBoxes = D / 32;
  extern __shared__ __align__(1024) unsigned char smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::kOffBar);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = g.L, LP = g.LP, C = g.C, C3 = 3 * g.C;
  const int ntiles = (L > 128) ? 2 : 1;
  const int nitems = g.B * g.nW * g.heads;
  const bool is_compute = warp < kF4Compute / 32;
  const int half = is_compute ? (warp >> 2) : (warp - kF4Compute / 32);        // which half of the CTA this warp serves
  // this half's items: the CTA's items (blockIdx.x, + gridDim.x, ...) of parity `half`
  const int first = blockIdx.x + half * gridDim.x, stride = 2 * gridDim.x;

  uint64_t* full = bars + half * 6 + 0;     // the stage's three operands have landed
  uint64_t* sbar = bars + half * 6 + 1;     // S_t is in tensor memory
  uint64_t* pbar = bars + half * 6 + 2;     // P_t written back by the four compute warps
  uint64_t* obar = bars + half * 6 + 3;     // O_t is complete
  uint64_t* tbar = bars + half * 6 + 4;     // O_t sits in registers: tensor memory may take the next S           (4 warps)
  uint64_t* ebar = bars + half * 6 + 5;     // rows stored, stage released                                         (4 warps)
  unsigned char* stage = smem + half * SM::kStage;
  int* tok = reinterpret_cast<int*>(smem + SM::kOffTok) + half * kMaxLP;
  auto op_ptr = [&](int op) { return stage + op * SM::kTile; };                 // op: 0 Q^, 1 K^, 2 V

  auto item_is_box = [&](int item) {
    const int ww_all = (item / g.heads) % g.nW;
    const int wh = ww_all / g.nWw, ww = ww_all - wh * g.nWw;
    return !((g.s0 > 0 && (wh + 1) * g.Wh + g.s0 > g.H) || (g.s1 > 0 && (ww + 1) * g.Ww + g.s1 > g.W));
  };

  // ---- one-time set-up -----------------------------------------------------------------------------------------------
  if (tid == 0) {
    prefetch_tmap(&tm_qkv);
    for (int h = 0; h < kF4Halves; ++h) {
      mbar_init(bars + h * 6 + 0, 1);
      mbar_init(bars + h * 6 + 1, 1);
      mbar_init(bars + h * 6 + 2, 4);
      mbar_init(bars + h * 6 + 3, 1);
      mbar_init(bars + h * 6 + 4, 4);
      mbar_init(bars + h * 6 + 5, 4);
    }
    fence_barrier_init();
  }
  if (warp == kF4Compute / 32) tmem_alloc(tmem_slot, 512);
  for (int i = tid; i < (LP - L) * kPieces * 3 * kF4Halves; i += kF4Threads) {   // zero pad rows [L, LP) of every operand buffer
    const int buf = i / ((LP - L) * kPieces);
    const int rem = i - buf * (LP - L) * kPieces;
    const int c = rem / (LP - L), r = L + rem % (LP - L);
    *reinterpret_cast<uint4*>(smem + (buf / 3) * SM::kStage + (buf % 3) * SM::kTile + opnd_off(r, c)) = make_uint4(0, 0, 0, 0);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot + (uint32_t)(half * 256);
  const uint32_t idesc_s = umma_idesc_bf16(128, LP, false, false);   // [128 queries x LP keys] = A(k-major) B(k-major)^T
  const uint32_t idesc_o = umma_idesc_bf16(128, D, false, true);     // [128 x D] = A(TMEM) B(n-major)

  if (!is_compute) {
    // =========================================== control warp of this half ===========================================
    // operands [op_lo, op_hi) of `item` (0 Q^, 1 K^, 2 V); `arm` registers the item's total byte count.  Whole warp; one lane issues.
    auto tma_ops = [&](int item, int op_lo, int op_hi, bool arm) {
      const int hd = item % g.heads;
      const int ww_all = (item / g.heads) % g.nW;
      const int bb = item / (g.heads * g.nW);
      const int wh = ww_all / g.nWw, ww = ww_all - wh * g.nWw;
      if (elect_one_f4()) {
        if (arm) mbar_arrive_expect_tx(full, 3u * kBoxes * 64u * (uint32_t)L);
        for (int op = op_lo; op < op_hi; ++op)
#pragma unroll
          for (int c = 0; c < kBoxes; ++c)
            tma_load_5d(op_ptr(op) + c * kCS64, &tm_qkv, full, 0, (op * C + hd * D) / 32 + c, ww * g.Ww + g.s1, wh * g.Wh + g.s0, bb);
      }
      __syncwarp();
    };
    auto tma_item = [&](int item) { tma_ops(item, 0, 3, true); };
    if (first < nitems && item_is_box(first)) tma_item(first);
    const int nk = LP / 16;
    const uint32_t q0 = smem_u32(op_ptr(0)), k0 = smem_u32(op_ptr(1)), v0 = smem_u32(op_ptr(2));
    uint32_t ph_f = 0, ph_p = 0, ph_t = 0, ph_e = 0, ph_o = 0;
    bool first_s = true;
    for (int item = first; item < nitems; item += stride) {
      const int item_next = item + stride;
      const bool next_box = item_next < nitems && item_is_box(item_next);
      mbar_wait(full, ph_f, 951); ph_f ^= 1;
      tc_fence_after();
      for (int t = 0; t < ntiles; ++t) {
        const bool last_tile = (t == ntiles - 1);
        if (!first_s) { mbar_wait(tbar, ph_t, 952); ph_t ^= 1; }     // the previous O is in registers: its columns are free
        first_s = false;
        tc_fence_after();
        if (elect_one_f4()) {
#pragma unroll
          for (int k = 0; k < D / 16; ++k)
            umma_bf16_ss(tmem_base, opnd_kmajor(q0, k, t * 128), opnd_kmajor(k0, k, 0), idesc_s, k > 0);
          umma_commit(sbar);
        }
        __syncwarp();
        mbar_wait(pbar, ph_p, 953); ph_p ^= 1;
        tc_fence_after();
        // the item's last S has been consumed: K^ is dead, the next item's K^ boxes may land on it (they carry the byte count)
        if (last_tile && next_box) tma_ops(item_next, 1, 2, true);
        if (elect_one_f4()) {
          const uint64_t bv = opnd_mnmajor(v0, 0);
#pragma unroll
          for (int k = 0; k < kMaxLP / 16; ++k)       // O_t = P_t V   (A = P from tensor memory, V read n-major: rows = keys = k)
            if (k < nk) umma_bf16_ts(tmem_base + 88, tmem_base + k * 8, bv + (uint64_t)(k * 64), idesc_o, k > 0);
          umma_commit(obar);
        }
        __syncwarp();
        // ... and V after the last P V (the compute warps wait on the same barrier)
        mbar_wait(obar, ph_o, 955); ph_o ^= 1;
        if (last_tile && next_box) tma_ops(item_next, 2, 3, false);
      }
      mbar_wait(ebar, ph_e, 954); ph_e ^= 1;           // rows stored: the Q^ buffer (where they were parked) is free
      if (next_box) tma_ops(item_next, 0, 1, false);
    }
  } else {
    // ============================================ compute warps of this half ============================================
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int ht = tid & 127;                         // thread index inside the half
    const uint32_t t_s = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int bar_id = 1 + half;
    auto fill_tok = [&](int item) {
      const int ww = (item / g.heads) % g.nW;
      const int bb = item / (g.heads * g.nW);
      for (int n = ht; n < LP; n += 128) {
        int rr;
        tok[n] = (n < L) ? win_token(g, bb, ww, n, rr) : -1;
      }
    };
    // all three operands of `item` -> this half's stage, per-thread 16-byte copies (windows that wrap around the cyclic shift)
    auto gather_item = [&](int item) {
      const int hd = item % g.heads;
      for (int i = ht; i < 3 * L * kPieces; i += 128) {
        const int op = i / (L * kPieces);
        const int rem = i - op * L * kPieces;
        const int n = rem / kPieces, c = rem - n * kPieces;
        cp_async16(op_ptr(op) + opnd_off(n, c), qkv + (size_t)tok[n] * C3 + op * C + hd * D + c * 8);
      }
      cp_async_wait_all();
      fence_proxy_async_smem();
      named_bar_f4(bar_id, 128);
      if (ht == 0) mbar_arrive(full);
    };
    if (first < nitems) {
      fill_tok(first);
      named_bar_f4(bar_id, 128);
      if (!item_is_box(first)) gather_item(first);
    }
    uint32_t ph_s = 0, ph_o = 0;
    for (int item = first; item < nitems; item += stride) {
      const int head = item % g.heads;
      const int w = (item / g.heads) % g.nW;
      const int b = item / (g.heads * g.nW);
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
      const float scale_l2 = scale_p[head] * kLog2e;
      unsigned char* rows_buf = op_ptr(0);            // output rows go where the (dead) Q^ rows were
      for (int t = 0; t < ntiles; ++t) {
        const int n = t * 128 + r;                    // this thread's query slot
        const bool row_ok = n < L;
        const bool warp_rows = t * 128 + quarter * 32 < L;      // warp-uniform: the warp has real query rows
        mbar_wait(sbar, ph_s, 960); ph_s ^= 1;
        tc_fence_after();
        float row_sum = 0.f, row_max = -INFINITY, cos_sum = 0.f;
        if (warp_rows) {
          if (plain) {
            float mx = 1.0f;                          // cosines are bounded by 1: scale*1 is a safe offset for scale*log2e < 60
            if (scale_l2 >= 60.0f) {
              mx = -INFINITY;
              for (int c0 = 0; c0 < LP; c0 += 16) {
                uint32_t v[16];
                tmem_ld_32x16(t_s + c0, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) mx = fmaxf(mx, as_f(v[j]));
              }
            }
            row_max = mx * scale_l2;
            const float neg_m = -row_max;
            auto softmax16 = [&](const uint32_t (&v)[16], int c0) {
              float p[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) p[j] = ex2_approx(fmaf(as_f(v[j]), scale_l2, neg_m));
              if (c0 + 16 > L) {
#pragma unroll
                for (int j = 0; j < 16; ++j) if (c0 + j >= L) p[j] = 0.f;
              }
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                row_sum += p[j];
                cos_sum = fmaf(p[j], as_f(v[j]), cos_sum);
              }
              tmem_st_32x8(t_s + c0 / 2, pack8(p, 0), pack8(p, 8));
            };
            uint32_t va[16], vb[16];
            tmem_ld_32x16(t_s, va);
            for (int c0 = 0; c0 < LP; c0 += 32) {
              tmem_ld_wait();
              const bool has_b = c0 + 16 < LP;
              if (has_b) tmem_ld_32x16(t_s + c0 + 16, vb);
              softmax16(va, c0);
              if (has_b) {
                tmem_ld_wait();
                if (c0 + 32 < LP) tmem_ld_32x16(t_s + c0 + 32, va);
                softmax16(vb, c0 + 16);
              }
            }
          } else {
            // continuous position bias and / or the shifted-window mask (-100 across region labels)
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
                if (key < L && row_ok) cos_sum = fmaf(p[j], as_f(v[j]), cos_sum);
              }
              tmem_st_32x8(t_s + c0 / 2, pack8(p, 0), pack8(p, 8));
            }
          }
          if (row_ok && lse != nullptr) {       // null: forward-only run
            const size_t ri = (((size_t)b * g.nW + w) * g.heads + head) * L + n;
            lse[ri] = (row_max + log2f(row_sum)) * 0.6931471805599453f;
            // second plane: E_P[cos] of the row.  The backward accumulates d(scale) = sum dS (cos - E_P[cos]); the row sum of dS
            // is zero in exact arithmetic, so this changes nothing but removes the first-order sensitivity to D = <dO, O>
            // being formed from the bf16-rounded O.
            lse[(size_t)g.B * g.nW * g.heads * L + ri] = cos_sum / row_sum;
          }
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pbar);

        // ---- O_t / rowsum -> registers -> parked where this row's Q^ was ----------------------------------------------------
        mbar_wait(obar, ph_o, 961); ph_o ^= 1;
        tc_fence_after();
        if (warp_rows) {
          const float inv = 1.0f / row_sum;
          float ov[D];
#pragma unroll
          for (int c0 = 0; c0 < D; c0 += 32) {
            uint32_t v[32];
            tmem_ld_32x32(t_s + 88 + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) ov[c0 + j] = as_f(v[j]) * inv;
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tbar);
          if (row_ok) {
#pragma unroll
            for (int c = 0; c < kPieces; ++c) {
              uint4 pk;
              pk.x = pack_bf16x2(ov[c * 8 + 0], ov[c * 8 + 1]); pk.y = pack_bf16x2(ov[c * 8 + 2], ov[c * 8 + 3]);
              pk.z = pack_bf16x2(ov[c * 8 + 4], ov[c * 8 + 5]); pk.w = pack_bf16x2(ov[c * 8 + 6], ov[c * 8 + 7]);
              *reinterpret_cast<uint4*>(rows_buf + opnd_off(n, c)) = pk;
            }
          }
        } else {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(tbar);
        }
      }
      // ---- all rows of the item parked: whole-row stores, then the stage goes back to the loads ------------------------------
      named_bar_f4(bar_id, 128);
      for (int i = ht; i < L * kPieces; i += 128) {
        const int row = i / kPieces, c = i - row * kPieces;
        *reinterpret_cast<uint4*>(o + (size_t)tok[row] * C + head * D + c * 8) = *reinterpret_cast<const uint4*>(rows_buf + opnd_off(row, c));
      }
      named_bar_f4(bar_id, 128);                      // parked rows and the token table have been read by everyone
      const int item_next = item + stride;
      if (item_next < nitems) fill_tok(item_next);
      fence_proxy_async_smem();                       // generic-proxy accesses of the stage before the async-proxy refill
      __syncwarp();
      if (lane == 0) mbar_arrive(ebar);
      if (item_next < nitems) {
        named_bar_f4(bar_id, 128);                    // token table of the next item is complete
        if (!item_is_box(item_next)) gather_item(item_next);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kF4Compute / 32) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(*tmem_slot, 512);
  }
}

int attn_tcgen05_fwd4(const void* qkv, const float* scale, const float* bias, void* o, float* lse, const AttnGeom& g, cudaStream_t stream) {
  using SM = Fwd4Smem<96>;
  static bool configured = false;
  if (!configured) {
    SWB_CUDA(cudaFuncSetAttribute(attn_tc_fwd4_kernel<96>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
    configured = true;
  }
  CUtensorMap tm_qkv;
  if (int e = attn_make_window_tmap(&tm_qkv, qkv, g.B, g.H, g.W, 3 * g.C, g.Wh, g.Ww)) return e;
  const int grid = max(1, min((g.B * g.nW * g.heads + 1) / 2, sm_count()));
  attn_tc_fwd4_kernel<96><<<grid, kF4Threads, SM::kBytes, stream>>>(tm_qkv, (const __nv_bfloat16*)qkv, scale, bias, (__nv_bfloat16*)o, lse, g);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

}  // namespace swinb200
