// tcgen05 windowed cosine attention, backward, third generation: ONE pass over the logits, warp-specialised.
//
// Reference math: swinv2_global.py:300-318 (cosine logits, clamped scale, CPB bias, shift mask, softmax, PV) differentiated.
//
// Work item = (sample, window, head), persistent CTAs (one per SM) loop over items.  13 warps:
//   warps 0..11  compute (3 column groups x 4 TMEM lane quarters): thread-per-key-row softmax gradient, output epilogues
//   warp 12      control: one lane issues every TMA load and every tcgen05.mma of the CTA and sequences them with mbarriers.
//                (tcgen05.mma issue is nearly synchronous with execution -- measured ~110 cycles per instruction -- so it must
//                not sit inside a warp that the epilogue barriers wait for; 13 warps keep 4 warps per scheduler = 128 registers.)
// Key-major orientation, so that each product is computed once (5 MMA chains per 128-key tile instead of the 7 of the
// two-sweep kernel, and one exp per logit instead of two):
//   S^T_u = K^_u Q^T , dP^T_u = V_u dO^T            (keys on TMEM lanes, queries on columns; fp32)
//   P^T_u = 2^(scale*S^T - lse_q) ; dS^T_u = P^T_u o (dP^T_u - D_q)           [compute warps; D = <dO, O> from the pre-pass]
//   dV_u  = P^T_u dO      A = P^T_u packed bf16 in TENSOR MEMORY (TS mode, never touches shared memory)
//   dK^_u = dS^T_u Q^     A = dS^T_u from shared memory, K-major
//   dQ^_t = dS_t K^       A = the SAME dS^T bytes read MN-major (rows = keys = k dimension): no transposed copy, no recompute
// The L2-normalisation Jacobians need <k^_j, dk^_j> = scale * sum_i dS_ij cos_ij -- exactly the per-thread partial sums the
// softmax phase already forms for d(logit_scale) -- so the dk epilogue needs no extra reduction; <q^_i, dq^_i> is reduced
// over the three column groups of a row through shared memory.
// Global traffic of the epilogues goes through a 2 KB per-warp slab: a thread owns 32 columns (64 B) of its row, but a warp
// instruction that touches 32 different rows costs 32 L1 tag cycles, so rows are exchanged through the slab and every
// global load / store instruction covers 8 rows x 64 contiguous bytes.
//
// TMEM columns (512):  S^T [0,176)  dP^T [176,352)  P^T bf16 [416,504);  once a tile's softmax is done its dV / dK^ accumulators
// reuse [192,288) / [288,384) and, after the last tile, dQ^_0 / dQ^_1 reuse [0,96) / [96,192).  S^T of the next key tile is issued
// while the compute warps are still draining dV / dK^ of the current one.
// Shared memory: dS^T 60.5 KB + four operand buffers (Q^, K^, V, dO; 33 KB each, 64B-swizzled TMA boxes as in the second
// generation).  Buffers are released by MMA completion, in the order V, (Q^, dO), K^; the next item's K^ is loaded into the
// buffer V just left (K^/V swap buffers every item), so its operands arrive while this item's tail is still computing.
#include <stdlib.h>
#include "attn_tc.cuh"

namespace swinb200 {

__device__ long long* g_phase_buf3 = nullptr;

constexpr int kB3Groups = 3;                         // column groups of compute warps
constexpr int kB3Compute = kB3Groups * 128;          // 12 compute warps
constexpr int kB3Threads = kB3Compute + 32;          // + the control warp
constexpr int kB3CtrlWarp = kB3Compute / 32;
constexpr uint32_t kColST = 0, kColDPT = 176, kColDV = 192, kColDK = 288, kColDQ = 0, kColP = 416;

template <int D>
struct Bwd3Smem {
  static constexpr int kDSCS = kMaxLP * 16;                 // dS^T tile: [22 chunks of 8 queries][176 key rows][16 B]
  static constexpr int kDS = (kMaxLP / 8) * kDSCS;          // 61,952
  static constexpr int kTile = (D / 32) * kCS64;            // one operand: 3 x [176 rows x 64 B]
  static constexpr int kOffDS = 0;                          // first: MMA over-reads past its end land in the operand buffers
  static constexpr int kOffOp = kDS;
  static constexpr int kOffSlab = kOffOp + 4 * kTile;       // [12 warps][32 rows x 64 B] row-exchange slabs
  static constexpr int kOffTok = kOffSlab + (kB3Compute / 32) * 2048;   // [2][176] token indices (current / next item)
  static constexpr int kOffLse = kOffTok + 2 * kMaxLP * 4;  // log2-domain LSE per query (+inf for pad queries)
  static constexpr int kOffDv = kOffLse + kMaxLP * 4;       // D = <dO, O> per query
  static constexpr int kOffInq = kOffDv + kMaxLP * 4;       // 1 / ||q|| per query slot
  static constexpr int kOffInk = kOffInq + kMaxLP * 4;      // 1 / ||k|| per key slot
  static constexpr int kOffEc = kOffInk + kMaxLP * 4;       // E_P[cos] per query (second plane of the forward's lse output)
  static constexpr int kOffDot = kOffEc + kMaxLP * 4;       // [2 tile parities][groups][128 rows]: sum_i dS_ij cos_ij partials
  static constexpr int kOffRed = kOffDot;                   // <q^, dQ^> partials of the dQ^ epilogue share the buffer: tile t uses
                                                            // parity (t + ntiles) & 1, never the one the last dK^ epilogue reads
  static constexpr int kOffDsc = kOffDot + 2 * kB3Groups * 128 * 4;     // per-head d(scale) partial sums of this CTA
  static constexpr int kOffBar = kOffDsc + 128;
  static constexpr int kBytes = kOffBar + 128;
  static_assert(kDS % 512 == 0 && kTile % 512 == 0, "64B-swizzled operand tiles need 512-byte alignment");
  static_assert(kBytes <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// one lane of a converged warp (the same lane every time): keeps descriptors of the issuing code in uniform registers
__device__ __forceinline__ bool elect_one3() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint4 pack8f(const float* v) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]); r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]); r.w = pack_bf16x2(v[6], v[7]);
  return r;
}
__device__ __forceinline__ void unpack8(const uint4& w, float* v) {
  v[0] = __uint_as_float(w.x << 16); v[1] = __uint_as_float(w.x & 0xffff0000u);
  v[2] = __uint_as_float(w.y << 16); v[3] = __uint_as_float(w.y & 0xffff0000u);
  v[4] = __uint_as_float(w.z << 16); v[5] = __uint_as_float(w.z & 0xffff0000u);
  v[6] = __uint_as_float(w.w << 16); v[7] = __uint_as_float(w.w & 0xffff0000u);
}
// 16-byte piece p (0..3) of row rr (0..31) inside a warp's slab; the XOR keeps both access patterns conflict-free:
// lane = row (4 pieces of one row per thread) and lane = (row % 8) * 4 + piece (8 rows x 64 B per warp instruction)
__device__ __forceinline__ unsigned char* slab_at(unsigned char* slab, int rr, int p) {
  return slab + rr * 64 + ((p ^ ((rr >> 1) & 3)) << 4);
}

// DET (deterministic mode): dscale is a (B*nW*heads) scratch that receives each item's d(scale), folded over the 12 compute
// warps in warp order (two 16-slot buffers in the per-head area, alternating per item); dbias is a (B*nW*heads, L, L)
// scratch in which each item writes its own slice with plain stores.  Items are statically assigned (item += gridDim.x).
template <int D, bool kProf, bool DET = false>
__global__ void __launch_bounds__(kB3Threads, 1)
attn_tc_bwd3_kernel(const __grid_constant__ CUtensorMap tm_qkv, const __grid_constant__ CUtensorMap tm_do,
                    const float* __restrict__ Dpre, const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ inv_norm,
                    const float* __restrict__ scale_p, const float* __restrict__ bias, const __nv_bfloat16* __restrict__ d_o,
                    const float* __restrict__ lse, __nv_bfloat16* __restrict__ dqkv, float* __restrict__ dscale,
                    float* __restrict__ dbias, const AttnGeom g, const int dbg) {
  using SM = Bwd3Smem<D>;
  static_assert(D == 96 && kB3Groups == 3, "the epilogues give each of the 3 column groups 32 of the 96 head channels");
  constexpr float kLog2e = 1.4426950408889634f;
  constexpr int kPieces = D / 8;                 // 16-byte pieces per operand row
  constexpr int kBoxes = D / 32;                 // TMA boxes (32-channel chunks) per operand
  constexpr int kEpiCols = D / kB3Groups;        // output columns per thread in the epilogues (32 = 64 bytes)
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* sDS = smem + SM::kOffDS;
  int* tokbuf0 = reinterpret_cast<int*>(smem + SM::kOffTok);
  float* lse2 = reinterpret_cast<float*>(smem + SM::kOffLse);
  float* Dv = reinterpret_cast<float*>(smem + SM::kOffDv);
  float* s_inq = reinterpret_cast<float*>(smem + SM::kOffInq);
  float* s_ink = reinterpret_cast<float*>(smem + SM::kOffInk);
  float* s_ec = reinterpret_cast<float*>(smem + SM::kOffEc);
  float* dotk = reinterpret_cast<float*>(smem + SM::kOffDot);
  float* red = reinterpret_cast<float*>(smem + SM::kOffRed);
  float* dsc_heads = reinterpret_cast<float*>(smem + SM::kOffDsc);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::kOffBar);
  uint64_t* full = bars;            // [4] operand (0 Q^, 1 K^, 2 V, 3 dO) of the next item to start has landed
  uint64_t* sbar = bars + 4;        // S^T / dP^T of a key tile are in tensor memory
  uint64_t* pbar = bars + 5;        // P^T (TMEM) and dS^T (smem) of the tile are written              (12 warps)
  uint64_t* obar = bars + 6;        // dV / dK^ accumulators of the tile are complete
  uint64_t* ebar = bars + 7;        // ... and have been read by the epilogue                            (12 warps)
  uint64_t* qbar = bars + 8;        // dQ^ accumulators are complete
  uint64_t* eqbar = bars + 9;       // ... and have been read                                            (12 warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int L = g.L, LP = g.LP, C = g.C, C3 = 3 * g.C;
  const int ntiles = (LP > 128) ? 2 : 1;
  const bool shifted = (g.s0 > 0) || (g.s1 > 0);
  const int nitems = g.B * g.nW * g.heads;
  const int first = blockIdx.x;
  const bool is_compute = warp < kB3CtrlWarp;

  auto op_ptr = [&](int buf) { return smem + SM::kOffOp + buf * SM::kTile; };
  auto item_is_box = [&](int item) {   // a window that wraps around the cyclic shift is not one box of the tensor
    const int ww_all = (item / g.heads) % g.nW;
    const int wh = ww_all / g.nWw, ww = ww_all - wh * g.nWw;
    return !((g.s0 > 0 && (wh + 1) * g.Wh + g.s0 > g.H) || (g.s1 > 0 && (ww + 1) * g.Ww + g.s1 > g.W));
  };

  // ---- one-time set-up -----------------------------------------------------------------------------------------------
  if (tid == 0) {
    prefetch_tmap(&tm_qkv);
    prefetch_tmap(&tm_do);
    for (int i = 0; i < 4; ++i) mbar_init(&full[i], 1);
    mbar_init(sbar, 1);
    mbar_init(pbar, kB3Compute / 32);
    mbar_init(obar, 1);
    mbar_init(ebar, kB3Compute / 32);
    mbar_init(qbar, 1);
    mbar_init(eqbar, kB3Compute / 32);
    fence_barrier_init();
  }
  if (warp == kB3CtrlWarp) tmem_alloc(tmem_slot, 512);
  // pad rows [L, LP) of the four operand buffers stay zero for the whole kernel (loads only ever write rows < L)
  for (int i = tid; i < (LP - L) * kPieces * 4; i += kB3Threads) {
    const int op = i / ((LP - L) * kPieces);
    const int rem = i - op * (LP - L) * kPieces;
    const int c = rem / (LP - L), r = L + rem % (LP - L);
    *reinterpret_cast<uint4*>(op_ptr(op) + opnd_off(r, c)) = make_uint4(0, 0, 0, 0);
  }
  if (tid < 32) dsc_heads[tid] = 0.f;
  for (int n = L + tid; n < LP; n += kB3Threads) {      // pad slots never change: p = 2^(-inf) = 0 for pad queries
    lse2[n] = INFINITY;
    Dv[n] = 0.f;
    s_inq[n] = 0.f;
    s_ink[n] = 0.f;
    s_ec[n] = 0.f;
  }
  auto fill_tok = [&](int item, int* tk) {          // compute threads
    const int ww = (item / g.heads) % g.nW;
    const int bb = item / (g.heads * g.nW);
    for (int n = tid; n < LP; n += kB3Compute) {
      int rr;
      tk[n] = (n < L) ? win_token(g, bb, ww, n, rr) : -1;
    }
  };
  // per-slot row data of `item` (natural-log LSE, D = <dO, O>, reciprocal q / k norms) -> shared memory with 4-byte
  // cp.async, so that nobody waits for these dependent L2 round trips; rows_ready() completes them (thread n owns slot n)
  auto fill_rows = [&](int item, const int* tk) {
    const int hd = item % g.heads;
    const int ww = (item / g.heads) % g.nW;
    const int bb = item / (g.heads * g.nW);
    for (int n = tid; n < L; n += kB3Compute) {
      const int t = tk[n];
      const size_t ri = (((size_t)bb * g.nW + ww) * g.heads + hd) * L + n;
      cp_async4(&lse2[n], lse + ri);
      cp_async4(&s_ec[n], lse + (size_t)g.B * g.nW * g.heads * L + ri);
      cp_async4(&Dv[n], Dpre + (size_t)t * g.heads + hd);
      cp_async4(&s_inq[n], inv_norm + (size_t)t * 2 * g.heads + hd);
      cp_async4(&s_ink[n], inv_norm + (size_t)t * 2 * g.heads + g.heads + hd);
    }
  };
  auto rows_ready = [&]() {       // before the item's first barrier: my copies have landed; LSE goes to the log2 domain
    cp_async_wait_all();
    for (int n = tid; n < L; n += kB3Compute) lse2[n] *= kLog2e;
  };
  // operand `role` (0 Q^, 1 K^, 2 V, 3 dO) of the (window, head) with token table `tk` -> buffer `buf`, by the compute threads
  auto gather = [&](int role, int buf, const int* tk, int hd) {
    unsigned char* dst = op_ptr(buf);
    for (int i = tid; i < L * kPieces; i += kB3Compute) {
      const int n = i / kPieces, c = i - n * kPieces;
      const __nv_bfloat16* src = (role < 3) ? qkv + (size_t)tk[n] * C3 + role * C + hd * D + c * 8
                                            : d_o + (size_t)tk[n] * C + hd * D + c * 8;
      cp_async16(dst + opnd_off(n, c), src);
    }
  };
  if (is_compute && first < nitems) fill_tok(first, tokbuf0);
  __syncthreads();
  if (is_compute && first < nitems) {
    fill_rows(first, tokbuf0);
    rows_ready();
    if (!item_is_box(first)) {
      const int hd = first % g.heads;
      gather(0, 0, tokbuf0, hd);
      gather(1, 1, tokbuf0, hd);
      gather(2, 2, tokbuf0, hd);
      gather(3, 3, tokbuf0, hd);
      cp_async_wait_all();
      fence_proxy_async_smem();
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (tid == 0 && first < nitems && !item_is_box(first))
    for (int i = 0; i < 4; ++i) mbar_arrive(&full[i]);

  const uint32_t idesc_s = umma_idesc_bf16(128, LP, false, false);   // [128 keys x LP queries] = A(k-major) B(k-major)^T
  const uint32_t idesc_o = umma_idesc_bf16(128, D, false, true);     // [128 x D] = A(k-major or TMEM) B(n-major)
  const uint32_t idesc_q = umma_idesc_bf16(128, D, true, true);      // [128 x D] = A(m-major) B(n-major)
  const uint32_t ds0 = smem_u32(sDS);

  if (!is_compute) {
    // =========================================== control: TMA + MMA issue ===========================================
    // The whole warp runs this loop convergently and one elected lane issues: descriptors then live in uniform registers
    // (a single diverged lane makes the compiler wrap every UTCHMMA in a warp-uniformisation loop, ~100 cycles per MMA --
    // twice the 48 cycles the tensor pipe needs for one).
    {
      uint32_t ph_full = 0, ph_s = 0, ph_p = 0, ph_o = 0, ph_e = 0, ph_q = 0, ph_eq = 0;
      int kb = 1, vb = 2;
      const int nk = LP / 16;
      auto tma_operand = [&](int role, int buf, int item) {    // role: 0 Q^, 1 K^, 2 V, 3 dO   (whole warp; one lane issues)
        const int hd = item % g.heads;
        const int ww_all = (item / g.heads) % g.nW;
        const int bb = item / (g.heads * g.nW);
        const int wh = ww_all / g.nWw, ww = ww_all - wh * g.nWw;
        const CUtensorMap* tm = (role < 3) ? &tm_qkv : &tm_do;
        const int chunk0 = ((role < 3) ? role * C + hd * D : hd * D) / 32;
        if (elect_one3()) {
          mbar_arrive_expect_tx(&full[role], (uint32_t)kBoxes * 64u * (uint32_t)L);
#pragma unroll
          for (int c = 0; c < kBoxes; ++c)
            tma_load_5d(op_ptr(buf) + c * kCS64, tm, &full[role], 0, chunk0 + c, ww * g.Ww + g.s1, wh * g.Wh + g.s0, bb);
        }
        __syncwarp();
      };
      if (first < nitems && item_is_box(first)) {
        tma_operand(1, 1, first);
        tma_operand(0, 0, first);
        tma_operand(2, 2, first);
        tma_operand(3, 3, first);
      }
      int it = 0;
      for (int item = first; item < nitems; item += gridDim.x, ++it) {
        const int item_next = item + gridDim.x;
        const bool next_box = item_next < nitems && item_is_box(item_next);
        const uint32_t q0 = smem_u32(op_ptr(0)), k0 = smem_u32(op_ptr(kb)), v0 = smem_u32(op_ptr(vb)), g0 = smem_u32(op_ptr(3));
        auto issue_st = [&](int u) {
          if (elect_one3()) {
#pragma unroll
            for (int k = 0; k < D / 16; ++k)
              umma_bf16_ss(tmem_base + kColST, opnd_kmajor(k0, k, u * 128), opnd_kmajor(q0, k, 0), idesc_s, k > 0);
          }
          __syncwarp();
        };
        auto issue_dpt = [&](int u) {
          if (elect_one3()) {
#pragma unroll
            for (int k = 0; k < D / 16; ++k)
              umma_bf16_ss(tmem_base + kColDPT, opnd_kmajor(v0, k, u * 128), opnd_kmajor(g0, k, 0), idesc_s, k > 0);
            umma_commit(sbar);
          }
          __syncwarp();
        };
        mbar_wait(&full[1], ph_full, 800);
        mbar_wait(&full[0], ph_full, 801);
        if (it > 0) { mbar_wait(eqbar, ph_eq, 802); ph_eq ^= 1; }      // dQ^ columns [0,192) of the previous item drained
        tc_fence_after();
        issue_st(0);
        mbar_wait(&full[2], ph_full, 803);
        mbar_wait(&full[3], ph_full, 804);
        ph_full ^= 1;
        if (it > 0) { mbar_wait(ebar, ph_e, 805); ph_e ^= 1; }          // dV / dK^ columns of the previous item's last tile drained
        tc_fence_after();
        issue_dpt(0);
        for (int u = 0; u < ntiles; ++u) {
          const bool last = (u == ntiles - 1);
          if (u > 0) {
            mbar_wait(ebar, ph_e, 806); ph_e ^= 1;                      // dV_{u-1} / dK^_{u-1} drained: dP^T may overwrite them
            tc_fence_after();
            issue_dpt(u);
          }
          if (last) {
            mbar_wait(sbar, ph_s, 807);                                 // last MMA that reads V is complete: its buffer is free
            if (next_box) tma_operand(1, vb, item_next);                // the next item's K^ goes where V was
          }
          ph_s ^= 1;
          mbar_wait(pbar, ph_p, 808); ph_p ^= 1;
          tc_fence_after();
          if (elect_one3()) {
            // descriptors advance by constants per 16-wide k step (16-byte units): dO / Q^ / K^ n-major +1024 B, dS^T k-major
            // +2 chunks, dS^T m-major +256 B, P^T +8 columns
            const uint64_t bg = opnd_mnmajor(g0, 0), bq = opnd_mnmajor(q0, 0);
            const uint64_t ads = umma_desc_nosw(ds0 + u * 128 * 16, SM::kDSCS, 128);
#pragma unroll
            for (int k = 0; k < kMaxLP / 16; ++k)       // dV_u = P^T_u dO   (A from tensor memory; dO read n-major: rows = queries = k)
              if (k < nk) umma_bf16_ts(tmem_base + kColDV, tmem_base + kColP + k * 8, bg + (uint64_t)(k * 64), idesc_o, k > 0);
#pragma unroll
            for (int k = 0; k < kMaxLP / 16; ++k)       // dK^_u = dS^T_u Q^
              if (k < nk) umma_bf16_ss(tmem_base + kColDK, ads + (uint64_t)(k * (2 * SM::kDSCS / 16)), bq + (uint64_t)(k * 64), idesc_o, k > 0);
            umma_commit(obar);
            if (!last) {
#pragma unroll
              for (int k = 0; k < D / 16; ++k)          // S^T of the next key tile runs while the compute warps drain dV_u / dK^_u
                umma_bf16_ss(tmem_base + kColST, opnd_kmajor(k0, k, (u + 1) * 128), opnd_kmajor(q0, k, 0), idesc_s, k > 0);
            } else {
              const uint64_t bk = opnd_mnmajor(k0, 0);
              for (int t = 0; t < ntiles; ++t) {        // dQ^_t = dS_t K^   (A = dS^T read m-major, K^ read n-major; k = keys)
                const uint64_t adq = umma_desc_nosw(ds0 + t * 16 * SM::kDSCS, 128, SM::kDSCS);
#pragma unroll
                for (int k = 0; k < kMaxLP / 16; ++k)
                  if (k < nk) umma_bf16_ss(tmem_base + kColDQ + t * D, adq + (uint64_t)(k * 16), bk + (uint64_t)(k * 64), idesc_q, k > 0);
              }
              umma_commit(qbar);
            }
          }
          __syncwarp();
          if (!last) ph_o ^= 1;                     // (only the last tile's completion is waited on below)
        }
        mbar_wait(obar, ph_o, 809); ph_o ^= 1;                          // Q^ and dO have served their last MMA
        if (next_box) { tma_operand(0, 0, item_next); tma_operand(3, 3, item_next); }
        mbar_wait(qbar, ph_q, 810); ph_q ^= 1;                          // ... and K^
        if (next_box) tma_operand(2, kb, item_next);                    // the next item's V goes where K^ was
        const int tmp = kb; kb = vb; vb = tmp;
      }
    }
  } else {
    // ================================================ compute warps ================================================
    const int grp = warp >> 2, quarter = warp & 3;
    const int r = quarter * 32 + lane;                    // row inside the current 128-row tile == TMEM lane
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int nchunks = LP / 16;
    const int c_begin = (nchunks * grp / kB3Groups) * 16, c_end = (nchunks * (grp + 1) / kB3Groups) * 16;   // this group's query columns
    const int ecol = grp * kEpiCols;                      // this group's output columns in the epilogues
    unsigned char* slab = smem + SM::kOffSlab + warp * 2048;
    const int xrow = lane >> 2, xpiece = lane & 3;        // row-exchange role: row 8*i + xrow, 16-byte piece xpiece
    uint32_t ph_s = 0, ph_o = 0, ph_q = 0;
    int kb = 1, vb = 2;
    // per-phase cycle accounting of thread 0 (bring-up aid; the kProf = false instantiation carries none of it)
    long long ph_acc[kProf ? 16 : 1];
#pragma unroll
    for (int i = 0; i < (kProf ? 16 : 1); ++i) ph_acc[i] = 0;
    long long ph_t = kProf ? clock64() : 0;
#define SWB_ACC(i) do { if (kProf && tid == 0) { const long long now_ = clock64(); ph_acc[kProf ? (i) : 0] += now_ - ph_t; ph_t = now_; } } while (0)

    // this thread's 64 bytes -> slab -> 8 rows x 64 contiguous bytes per global store instruction.
    // `base` = dqkv + column offset of this (part, head, group); slot0 = window slot of the warp's row 0; rows < nvalid are real.
    auto store_rows = [&](const uint4 (&mine)[4], __nv_bfloat16* base, const int* tok, int slot0, int nvalid) {
      __syncwarp();
#pragma unroll
      for (int p = 0; p < 4; ++p) *reinterpret_cast<uint4*>(slab_at(slab, lane, p)) = mine[p];
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rr = i * 8 + xrow;
        if (rr < nvalid && !(dbg & 1)) {
          const uint4 v = *reinterpret_cast<const uint4*>(slab_at(slab, rr, xpiece));
          *reinterpret_cast<uint4*>(base + (size_t)tok[slot0 + rr] * C3 + xpiece * 8) = v;
        }
      }
    };
    // the reverse, in two steps so that the L2 round trip can sit under a barrier wait: fetch_rows issues 8 rows x 64 bytes
    // per global load instruction into registers, exchange_rows passes them through the slab -> this thread's 64 bytes
    auto fetch_rows = [&](uint4 (&tmp)[4], const __nv_bfloat16* base, const int* tok, int slot0, int nvalid) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rr = i * 8 + xrow;
        tmp[i] = (rr < nvalid && !(dbg & 2)) ? __ldg(reinterpret_cast<const uint4*>(base + (size_t)tok[slot0 + rr] * C3 + xpiece * 8))
                               : make_uint4(0, 0, 0, 0);
      }
    };
    auto exchange_rows = [&](uint4 (&mine)[4], const uint4 (&tmp)[4]) {
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) *reinterpret_cast<uint4*>(slab_at(slab, i * 8 + xrow, xpiece)) = tmp[i];
      __syncwarp();
#pragma unroll
      for (int p = 0; p < 4; ++p) mine[p] = *reinterpret_cast<const uint4*>(slab_at(slab, lane, p));
    };

    int it = 0;
    for (int item = first; item < nitems; item += gridDim.x, ++it) {
      int* tok = tokbuf0 + (it & 1) * kMaxLP;
      int* tok_next = tokbuf0 + ((it & 1) ^ 1) * kMaxLP;
      const int head = item % g.heads;
      const int w = (item / g.heads) % g.nW;
      const int item_next = item + gridDim.x;
      const bool has_next = item_next < nitems;
      const bool next_gather = has_next && !item_is_box(item_next);
      const int head_next = item_next % g.heads;
      if (has_next) fill_tok(item_next, tok_next);
      if (it > 0) rows_ready();
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
      const bool plain = (bias == nullptr) && !(label_split > 0 && label_split < L);
      const float scale = scale_p[head];
      const float scale_l2 = scale * kLog2e;
      named_bar_sync(1, kB3Compute);      // this item's per-slot rows / tok (written during the previous item) are visible
      if constexpr (DET) {
        if (tid == 0 && it > 0) {           // the previous item's warp sums are complete
          float v = 0.f;
          for (int w8 = 0; w8 < kB3Compute / 32; ++w8) v += dsc_heads[((it - 1) & 1) * 16 + w8];
          dscale[item - gridDim.x] = v;
        }
      }
      // reciprocal norms of this thread's rows, taken now: the per-slot arrays are refilled for the next item before the
      // last epilogues of this one run
      float my_ink[2], my_inq[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int n = t * 128 + r;
        my_ink[t] = (n < L) ? s_ink[n] : 0.f;
        my_inq[t] = (n < L) ? s_inq[n] : 0.f;
      }
      SWB_ACC(0);
      float dsc_acc = 0.f;

      for (int u = 0; u < ntiles; ++u) {
        const bool last = (u == ntiles - 1);
        const int jk = u * 128 + r;                         // key slot of this thread
        const bool key_ok = jk < L;
        const bool warp_rows = u * 128 + quarter * 32 < LP;   // warp-uniform: this warp's lanes hold rows of the padded window
        mbar_wait(sbar, ph_s, 820 + u); ph_s ^= 1;
        tc_fence_after();
        SWB_ACC(1);
        if (last && next_gather) gather(1, vb, tok_next, head_next);   // V served its last MMA: the next item's K^ goes there
        // ---- P^T, dS^T of this thread's key row over the group's query columns ------------------------------------------
        float part = 0.f;                                   // sum_i dS_ij cos_ij
        float partc = 0.f;                                  // sum_i dS_ij E_P[cos]_i  (d(scale) uses part - partc)
        if (warp_rows && !(dbg & 4)) {
          const int key_label = (jk >= label_split) ? 1 : 0;
          const bool row_exists = jk < LP;
          if (plain) {
            // logits are scale * cos: P^T -> tensor memory, dS^T -> shared memory, partial sum of dS o cos
#pragma unroll 1
            for (int c0 = c_begin; c0 < c_end; c0 += 16) {
              uint32_t sv[16], pv[16];
              tmem_ld_32x16(t_lane + kColST + c0, sv);
              tmem_ld_32x16(t_lane + kColDPT + c0, pv);
              tmem_ld_wait();
#pragma unroll
              for (int hh = 0; hh < 2; ++hh) {          // two halves of 8 queries keep the live set small
                const int cb = c0 + hh * 8;
                float ls[8], dd[8];
                *reinterpret_cast<float4*>(&ls[0]) = *reinterpret_cast<const float4*>(&lse2[cb]);
                *reinterpret_cast<float4*>(&ls[4]) = *reinterpret_cast<const float4*>(&lse2[cb + 4]);
                *reinterpret_cast<float4*>(&dd[0]) = *reinterpret_cast<const float4*>(&Dv[cb]);
                *reinterpret_cast<float4*>(&dd[4]) = *reinterpret_cast<const float4*>(&Dv[cb + 4]);
                float pp[8], ds[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float cosv = as_f(sv[hh * 8 + j]);
                  const float p = ex2_approx(fmaf(cosv, scale_l2, -ls[j]));     // pad queries: lse2 = +inf -> p = 0
                  pp[j] = key_ok ? p : 0.f;                                     // pad keys: cos = 0 but p != 0 -> force zero
                  ds[j] = key_ok ? p * (as_f(pv[hh * 8 + j]) - dd[j]) : 0.f;
                  part = fmaf(ds[j], cosv, part);
                }
                {
                  const float4 e0 = *reinterpret_cast<const float4*>(&s_ec[cb]), e1 = *reinterpret_cast<const float4*>(&s_ec[cb + 4]);
                  partc = fmaf(ds[0], e0.x, partc); partc = fmaf(ds[1], e0.y, partc); partc = fmaf(ds[2], e0.z, partc); partc = fmaf(ds[3], e0.w, partc);
                  partc = fmaf(ds[4], e1.x, partc); partc = fmaf(ds[5], e1.y, partc); partc = fmaf(ds[6], e1.z, partc); partc = fmaf(ds[7], e1.w, partc);
                }
                tmem_st_32x4(t_lane + kColP + cb / 2, pack8f(pp));             // 8 queries = 4 packed columns of P^T
                if (row_exists) *reinterpret_cast<uint4*>(sDS + (cb / 8) * SM::kDSCS + jk * 16) = pack8f(ds);
              }
            }
          } else {
            // continuous position bias and / or the shifted-window mask (-100 across region labels)
#pragma unroll 1
            for (int cb = c_begin; cb < c_end; cb += 8) {
              uint32_t sv[8], pv[8];
              tmem_ld_32x8(t_lane + kColST + cb, sv);
              tmem_ld_32x8(t_lane + kColDPT + cb, pv);
              tmem_ld_wait();
              float pp[8], ds[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const int qi = cb + j;
                const float cosv = as_f(sv[j]);
                float sl = cosv * scale_l2;
                if (bias != nullptr && key_ok && qi < L) sl += __ldg(bias + ((size_t)head * L + qi) * L + jk) * kLog2e;
                if (((qi >= label_split) ? 1 : 0) != key_label) sl += -100.0f * kLog2e;
                const float p = key_ok ? ex2_approx(sl - lse2[qi]) : 0.f;
                pp[j] = p;
                ds[j] = (key_ok && qi < L) ? p * (as_f(pv[j]) - Dv[qi]) : 0.f;
                part = fmaf(ds[j], cosv, part);
                partc = fmaf(ds[j], s_ec[qi], partc);
                if constexpr (DET) {
                  if (dbias != nullptr && key_ok && qi < L) dbias[((size_t)item * L + qi) * L + jk] = ds[j];
                } else {
                  if (dbias != nullptr && key_ok && qi < L) atomicAdd(dbias + ((size_t)head * L + qi) * L + jk, ds[j]);
                }
              }
              tmem_st_32x4(t_lane + kColP + cb / 2, pack8f(pp));
              if (row_exists) *reinterpret_cast<uint4*>(sDS + (cb / 8) * SM::kDSCS + jk * 16) = pack8f(ds);
            }
          }
          tmem_st_wait();
        }
        dotk[((u & 1) * kB3Groups + grp) * 128 + r] = part;
        if (key_ok) dsc_acc += part - partc;   // rows beyond the window read garbage cosines (0 * NaN would poison the sum)
        fence_proxy_async_smem();       // dS^T (generic-proxy stores) -> visible to the tensor core's async-proxy reads
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pbar);
        SWB_ACC(2);

        // ---- dV_u / dK^_u epilogue: this thread owns 32 of the 96 columns of its key row ----------------------------------
        const int slot0 = u * 128 + quarter * 32;           // window slot of this warp's first row
        const int nvalid = min(32, L - slot0);
        uint4 kfetch[4];
        if (last && slot0 < L) fetch_rows(kfetch, qkv + C + head * D + ecol, tok, slot0, nvalid);   // L2 round trip under the wait
        mbar_wait(obar, ph_o, 830 + u); ph_o ^= 1;
        tc_fence_after();
        SWB_ACC(3);
        if (last && has_next) {
          fill_rows(item_next, tok_next);                   // every warp is past its last read of the per-slot rows
          if (next_gather) { gather(0, 0, tok_next, head_next); gather(3, 3, tok_next, head_next); }   // Q^ / dO served their last MMA
        }
        if (slot0 < L && !(dbg & 8)) {                      // warp-uniform: the warp has real key rows
          // k^ rows: from shared memory while the K^ buffer is live, from L2 once it is being recycled (last tile)
          uint4 kraw[4];
          if (!last) {
#pragma unroll
            for (int p = 0; p < 4; ++p)
              kraw[p] = *reinterpret_cast<const uint4*>(op_ptr(kb) + opnd_off(min(jk, LP - 1), grp * 4 + p));
          } else {
            exchange_rows(kraw, kfetch);
          }
          uint4 outv[4];
          {
            uint32_t av[kEpiCols];
            tmem_ld_32x32(t_lane + kColDV + ecol, av);
            tmem_ld_wait();
#pragma unroll
            for (int p = 0; p < 4; ++p) outv[p] = pack8f(reinterpret_cast<const float*>(&av[p * 8]));
          }
          store_rows(outv, dqkv + 2 * C + head * D + ecol, tok, slot0, nvalid);
          {
            uint32_t ak[kEpiCols];
            tmem_ld_32x32(t_lane + kColDK + ecol, ak);
            const float* dk4 = dotk + (u & 1) * kB3Groups * 128 + r;
            const float dot = dk4[0] + dk4[128] + dk4[256];                 // sum_i dS_ij cos_ij = <k^_j, dK^_j>
            const float ks = my_ink[u] * scale;
            tmem_ld_wait();
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              float kh[8], ok[8];
              unpack8(kraw[p], kh);
#pragma unroll
              for (int e = 0; e < 8; ++e) ok[e] = ks * fmaf(-kh[e], dot, as_f(ak[p * 8 + e]));   // dk = inv_norm scale (dK^ - k^ <k^, dK^>)
              outv[p] = pack8f(ok);
            }
          }
          store_rows(outv, dqkv + C + head * D + ecol, tok, slot0, nvalid);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ebar);
        SWB_ACC(4);
      }

      // ---- dQ^ epilogue ------------------------------------------------------------------------------------------------------
      uint4 qfetch[4];
      if (quarter * 32 < L) fetch_rows(qfetch, qkv + head * D + ecol, tok, quarter * 32, min(32, L - quarter * 32));
      mbar_wait(qbar, ph_q, 840); ph_q ^= 1;
      tc_fence_after();
      SWB_ACC(5);
      if (next_gather) gather(2, kb, tok_next, head_next);        // K^ served its last MMA: the next item's V goes there
      for (int t = 0; t < ntiles; ++t) {
        const int n = t * 128 + r;
        const bool row_ok = n < L;
        const int slot0 = t * 128 + quarter * 32;
        const bool warp_has = slot0 < L && !(dbg & 16);
        const int nvalid = min(32, L - slot0);
        uint32_t aq[kEpiCols];
        float partq = 0.f;
        if (warp_has) {
          tmem_ld_32x32(t_lane + kColDQ + t * D + ecol, aq);
          uint4 qraw[4];
          exchange_rows(qraw, qfetch);
          tmem_ld_wait();
          if (row_ok) {
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              float qh[8];
              unpack8(qraw[p], qh);
#pragma unroll
              for (int e = 0; e < 8; ++e) partq = fmaf(qh[e], as_f(aq[p * 8 + e]), partq);
            }
          }
        }
        red[(((t + ntiles) & 1) * kB3Groups + grp) * 128 + r] = partq;
        if (t + 1 < ntiles && slot0 + 128 < L)               // next tile's q^ rows: their L2 round trip runs under the barrier
          fetch_rows(qfetch, qkv + head * D + ecol, tok, slot0 + 128, min(32, L - slot0 - 128));
        named_bar_sync(2, kB3Compute);
        if (warp_has) {
          const float* rq = red + ((t + ntiles) & 1) * kB3Groups * 128 + r;
          const float dot = rq[0] + rq[128] + rq[256];                      // <q^_i, dQ^_i>
          const float qs = my_inq[t] * scale;
          uint4 outq[4];
#pragma unroll
          for (int p = 0; p < 4; ++p) {
            float qh[8], oq[8];
            unpack8(*reinterpret_cast<const uint4*>(slab_at(slab, lane, p)), qh);    // q^ row again: still in the slab
#pragma unroll
            for (int e = 0; e < 8; ++e) oq[e] = qs * fmaf(-qh[e], dot, as_f(aq[p * 8 + e]));     // dq = inv_norm scale (dQ^ - q^ <q^, dQ^>)
            outq[p] = pack8f(oq);
          }
          store_rows(outq, dqkv + head * D + ecol, tok, slot0, nvalid);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(eqbar);
      SWB_ACC(6);
      if (next_gather) {                                     // the gathered operands of the next item are complete
        cp_async_wait_all();
        fence_proxy_async_smem();
        named_bar_sync(3, kB3Compute);
        if (tid == 0)
          for (int i = 0; i < 4; ++i) mbar_arrive(&full[i]);
      }
      dsc_acc = warp_sum(dsc_acc);
      if constexpr (DET) {
        if (lane == 0) dsc_heads[(it & 1) * 16 + warp] = dsc_acc;
      } else {
        if (lane == 0) atomicAdd(&dsc_heads[head], dsc_acc);
      }
      const int tmp = kb; kb = vb; vb = tmp;
      SWB_ACC(7);
    }
    named_bar_sync(1, kB3Compute);
    if constexpr (DET) {
      if (tid == 0 && it > 0) {
        float v = 0.f;
        for (int w8 = 0; w8 < kB3Compute / 32; ++w8) v += dsc_heads[((it - 1) & 1) * 16 + w8];
        dscale[first + (it - 1) * gridDim.x] = v;
      }
    } else {
      if (tid < g.heads) {
        const float v = dsc_heads[tid];
        if (v != 0.f) atomicAdd(dscale + tid, v);
      }
    }
    if (kProf && g_phase_buf3 != nullptr && tid == 0 && blockIdx.x < 4096)
      for (int i = 0; i < 16; ++i) g_phase_buf3[blockIdx.x * 16 + i] = ph_acc[i];
#undef SWB_ACC
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kB3CtrlWarp) {
    __syncwarp();
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

static bool g_prof3 = false;
int attn_set_phase_buffer3(long long* buf) {
  SWB_CUDA(cudaMemcpyToSymbol(g_phase_buf3, &buf, sizeof(buf)));
  g_prof3 = buf != nullptr;
  return SWINB200_OK;
}

int attn_tcgen05_bwd3(const void* qkv, const float* inv_norm, const float* scale, const float* bias, const void* o, const void* d_o,
                      const float* lse, void* dqkv, float* dscale, float* dbias, float* ws, const AttnGeom& g, cudaStream_t stream,
                      float* det_part) {
  using SM = Bwd3Smem<96>;
  static bool configured = false;
  if (!configured) {
    SWB_CUDA(cudaFuncSetAttribute(attn_tc_bwd3_kernel<96, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
    SWB_CUDA(cudaFuncSetAttribute(attn_tc_bwd3_kernel<96, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
    SWB_CUDA(cudaFuncSetAttribute(attn_tc_bwd3_kernel<96, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM::kBytes));
    configured = true;
  }
  CUtensorMap tm_qkv, tm_do;
  if (int e = attn_make_window_tmap(&tm_qkv, qkv, g.B, g.H, g.W, 3 * g.C, g.Wh, g.Ww)) return e;
  if (int e = attn_make_window_tmap(&tm_do, d_o, g.B, g.H, g.W, g.C, g.Wh, g.Ww)) return e;
  const long long n_pairs = (long long)g.B * g.H * g.W * g.heads;
  attn_rowdot_kernel<<<(unsigned)((n_pairs * 4 + 255) / 256), 256, 0, stream>>>((const __nv_bfloat16*)o, (const __nv_bfloat16*)d_o, ws,
                                                                                n_pairs, g.C / g.heads);
  SWB_LAUNCH_CHECK();
  const int grid = min(g.B * g.nW * g.heads, sm_count());
  static int dbg_env = -1;   // bring-up timing experiments (wrong results): SWINB200_BWD3_DEBUG bit mask, see the kernel
  if (dbg_env < 0) { const char* e = getenv("SWINB200_BWD3_DEBUG"); dbg_env = e ? atoi(e) : 0; }
  if (det_part != nullptr) {
    const int bw = g.B * g.nW;
    float* dbias_part = (dbias != nullptr) ? det_part + attn_det_dscale_slots(g) : nullptr;
    attn_tc_bwd3_kernel<96, false, true><<<grid, kB3Threads, SM::kBytes, stream>>>(tm_qkv, tm_do, ws, (const __nv_bfloat16*)qkv, inv_norm,
                                                                                   scale, bias, (const __nv_bfloat16*)d_o, lse,
                                                                                   (__nv_bfloat16*)dqkv, det_part, dbias_part, g, dbg_env);
    SWB_LAUNCH_CHECK();
    if (int e = ordered_reduce(det_part, bw, g.heads, g.heads, 1, dscale, 1, stream)) return e;
    if (dbias != nullptr) return ordered_reduce(dbias_part, bw, (long long)g.heads * g.L * g.L, (long long)g.heads * g.L * g.L, 1, dbias, 1, stream);
    return SWINB200_OK;
  }
  if (g_prof3)
    attn_tc_bwd3_kernel<96, true><<<grid, kB3Threads, SM::kBytes, stream>>>(tm_qkv, tm_do, ws, (const __nv_bfloat16*)qkv, inv_norm, scale,
                                                                            bias, (const __nv_bfloat16*)d_o, lse, (__nv_bfloat16*)dqkv,
                                                                            dscale, dbias, g, dbg_env);
  else
    attn_tc_bwd3_kernel<96, false><<<grid, kB3Threads, SM::kBytes, stream>>>(tm_qkv, tm_do, ws, (const __nv_bfloat16*)qkv, inv_norm, scale,
                                                                             bias, (const __nv_bfloat16*)d_o, lse, (__nv_bfloat16*)dqkv,
                                                                             dscale, dbias, g, dbg_env);
  SWB_LAUNCH_CHECK();
  return SWINB200_OK;
}

}  // namespace swinb200
