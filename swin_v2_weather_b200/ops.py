"""Tensor-level wrappers over the C ABI (include/swinb200.h).

PyTorch is used here for device memory, streams and shape bookkeeping only: every arithmetic
operation below is one of our CUDA kernels, launched on torch's current stream.  Arguments are
validated (device, dtype, contiguity) before their raw pointers cross the ABI.

Deterministic mode: while torch.use_deterministic_algorithms(True) is in force, every reduction whose float sums would depend on
the order in which CTAs finish (split-K weight gradients, bias / LayerNorm parameter gradients, loss and metric sums, attention
d(scale) / d(bias)) runs through the fixed-order `swinb200_*_det` entry points, with scratch from the torch allocator
(DESIGN.md section 10).  With the flag off nothing changes.

Forward-only runs: `need_stats=False` (ln_residual_fwd, linear_ln_residual, qkv_projection, window_attn_fwd) allocates none of
the row statistics that only a backward reads and passes NULL for them; every other output is bit-identical.
"""
from __future__ import annotations

import os

from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import (BACKEND_SIMT, BACKEND_TCGEN05, BF16, EPI_ADD_F32, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_GELU_FWD, EPI_BIAS_QKNORM,
                   EPI_DGELU, EPI_F32, F32, SwinB200Error)

LN_EPS = 1e-5


@dataclass(frozen=True)
class ComputeMode:
    """How the hot path computes.

    bf16 : activations stored in bf16, fp32 residual stream / statistics / accumulators, tcgen05 GEMMs.
    fp32 : fp32 storage and CUDA-core fp32 arithmetic everywhere (validation mode, parity <= 1e-5).
    `gemm_backend` / `attn_backend` select CUDA-core or tcgen05 kernels (tcgen05 needs bf16).
    """
    name: str
    act_dtype: torch.dtype
    gemm_backend: int
    attn_backend: int

    @property
    def act_code(self) -> int:
        return BF16 if self.act_dtype == torch.bfloat16 else F32


MODE_BF16 = ComputeMode("bf16", torch.bfloat16, BACKEND_TCGEN05, BACKEND_TCGEN05)
MODE_BF16_SIMT = ComputeMode("bf16_simt", torch.bfloat16, BACKEND_SIMT, BACKEND_SIMT)
MODE_FP32 = ComputeMode("fp32", torch.float32, BACKEND_SIMT, BACKEND_SIMT)
MODES = {m.name: m for m in (MODE_BF16, MODE_BF16_SIMT, MODE_FP32)}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def deterministic() -> bool:
    """Read at every call: torch.use_deterministic_algorithms(True) selects the fixed-order reductions."""
    return torch.are_deterministic_algorithms_enabled()


def _scratch(n_floats: int, device) -> torch.Tensor:
    """Partial-sum scratch of a deterministic entry point (every slot is written before it is read)."""
    return torch.empty((max(1, int(n_floats)),), dtype=torch.float32, device=device)


def _chk(t: Optional[torch.Tensor], name: str, dtype=None, allow_none=False) -> int:
    if t is None:
        if allow_none:
            return 0
        raise SwinB200Error(f"{name}: tensor is required")
    if not t.is_cuda:
        raise SwinB200Error(f"{name}: expected a CUDA tensor, got {t.device}")
    if not t.is_contiguous():
        raise SwinB200Error(f"{name}: tensor must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise SwinB200Error(f"{name}: expected dtype {dtype}, got {t.dtype}")
    return t.data_ptr()


def _code(dtype: torch.dtype) -> int:
    if dtype == torch.bfloat16:
        return BF16
    if dtype == torch.float32:
        return F32
    raise SwinB200Error(f"unsupported storage dtype {dtype}")


# ---- parameter staging -------------------------------------------------------------------------------
def cast_bf16(src: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    _lib.call("swinb200_cast_f32_to_bf16", _chk(src, "src", torch.float32), _chk(out, "out", torch.bfloat16), src.numel(), _stream())
    return out


def to_act(x: torch.Tensor, mode: ComputeMode) -> torch.Tensor:
    """fp32 tensor -> activation storage type (alias in fp32 mode)."""
    return x if mode.act_dtype == torch.float32 else cast_bf16(x)


# ---- patchify / unpatchify ---------------------------------------------------------------------------
def patchify(img: torch.Tensor, patch: int, order: int, mode: ComputeMode) -> torch.Tensor:
    B, C, Hi, Wi = img.shape
    T = B * (Hi // patch) * (Wi // patch)
    out = torch.empty((T, C * patch * patch), dtype=mode.act_dtype, device=img.device)
    _lib.call("swinb200_patchify", _chk(img, "img", torch.float32), out.data_ptr(), mode.act_code, B, C, Hi, Wi, patch, order, _stream())
    return out


def patchify_cat(parts, patch: int, mode: ComputeMode, mean: Optional[torch.Tensor] = None,
                 std: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Order-0 im2col of the channel-wise concatenation of `parts` without materialising it.  Every part is a contiguous
    fp32 (B or 1, C_s, Hi, Wi) CUDA tensor; a leading dimension of 1 is shared by the whole batch (static features).
    `mean` / `std`: optional (C,) fp32 per-channel statistics -- values enter the im2col as (x - mean) / std."""
    import ctypes
    B = max(p.shape[0] for p in parts)
    Hi, Wi = parts[0].shape[-2:]
    ptrs, chans, strides = [], [], []
    for i, p in enumerate(parts):
        if p.dim() != 4 or tuple(p.shape[-2:]) != (Hi, Wi) or p.shape[0] not in (1, B):
            raise SwinB200Error(f"patchify_cat: part {i} has shape {tuple(p.shape)}, expected ({B} or 1, C, {Hi}, {Wi})")
        ptrs.append(_chk(p, f"part {i}", torch.float32))
        chans.append(p.shape[1])
        strides.append(0 if (p.shape[0] == 1 and B > 1) else p.shape[1] * Hi * Wi)
    n, C = len(parts), sum(chans)
    T = B * (Hi // patch) * (Wi // patch)
    out = torch.empty((T, C * patch * patch), dtype=mode.act_dtype, device=parts[0].device)
    if mean is not None and (mean.numel() != C or std is None or std.numel() != C):
        raise SwinB200Error(f"patchify_cat: mean / std must have {C} entries")
    _lib.call("swinb200_patchify_cat_norm", n, (ctypes.c_void_p * n)(*ptrs), (ctypes.c_int * n)(*chans), (ctypes.c_longlong * n)(*strides),
              _chk(mean, "mean", torch.float32, True), _chk(std, "std", torch.float32, True), out.data_ptr(), mode.act_code, B, Hi, Wi,
              patch, _stream())
    return out


def unpatchify(y: torch.Tensor, skip: Optional[torch.Tensor], B: int, Co: int, Hi: int, Wi: int, patch: int,
               order: int = 1, skip_mean: Optional[torch.Tensor] = None, skip_std: Optional[torch.Tensor] = None) -> torch.Tensor:
    out = torch.empty((B, Co, Hi, Wi), dtype=torch.float32, device=y.device)
    skip_ch = 0 if skip is None else skip.shape[1]
    if skip_mean is not None and (skip_mean.numel() < Co or skip_std is None or skip_std.numel() < Co):
        raise SwinB200Error(f"unpatchify: skip mean / std need at least {Co} entries")
    _lib.call("swinb200_unpatchify_norm", _chk(y, "y"), _code(y.dtype), _chk(skip, "skip", torch.float32, True), skip_ch,
              _chk(skip_mean, "skip_mean", torch.float32, True), _chk(skip_std, "skip_std", torch.float32, True), out.data_ptr(),
              B, Co, Hi, Wi, patch, order, _stream())
    return out


# ---- GEMM ------------------------------------------------------------------------------------------
def gemm(mode: ComputeMode, A: torch.Tensor, a_major: int, B: torch.Tensor, b_major: int, epilogue: int, *,
         bias: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
         out2: Optional[torch.Tensor] = None, accumulate: bool = False, split_k: int = 1, backend: Optional[int] = None):
    """D[M,N] = epi(sum_k A(m,k) B(n,k)); see swinb200_gemm.  A/B are 2-D contiguous tensors.
    Returns D, or (D, D2) for EPI_BIAS_GELU (activation, pre-activation); EPI_BIAS_GELU_FWD returns the activation alone."""
    if a_major == 0:
        M, K = A.shape
    else:
        K, M = A.shape
    if b_major == 0:
        N, Kb = B.shape
    else:
        Kb, N = B.shape
    if K != Kb:
        raise SwinB200Error(f"gemm: reduction sizes differ ({K} vs {Kb})")
    if A.dtype != B.dtype:
        raise SwinB200Error("gemm: A and B must share a storage dtype")
    f32_out = epilogue in (EPI_ADD_F32, EPI_F32)
    out_dtype = torch.float32 if f32_out else A.dtype
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=A.device)
    if epilogue == EPI_BIAS_GELU and out2 is None:
        out2 = torch.empty((M, N), dtype=out_dtype, device=A.device)
    be = mode.gemm_backend if backend is None else backend
    if split_k > 1 and be == BACKEND_TCGEN05 and deterministic():
        # split-K reduce-adds arrive in scheduling order: every split stores its own slice, the slices are summed in order
        if not (epilogue == EPI_F32 and accumulate and a_major == 1 and b_major == 1):
            raise SwinB200Error("gemm: split_k > 1 is a weight-gradient option (a_major 1, b_major 1, EPI_F32, accumulate)")
        part = _scratch(split_k * M * N, A.device)
        _lib.call("swinb200_gemm_wgrad_det", be, M, N, K, _chk(A, "A"), A.shape[1], _chk(B, "B"), B.shape[1], _code(A.dtype),
                  _chk(out, "out", torch.float32), int(split_k), part.data_ptr(), part.numel(), _stream())
        return out
    _lib.call("swinb200_gemm", be, M, N, K, _chk(A, "A"), a_major, A.shape[1], _chk(B, "B"), b_major, B.shape[1], _code(A.dtype),
              epilogue, _chk(bias, "bias", torch.float32, True), _chk(out, "out", out_dtype), out.shape[1],
              _chk(out2, "out2", out_dtype, True), _chk(aux, "aux", None, True), 0 if aux is None else aux.shape[1],
              _code(out_dtype), int(accumulate), int(split_k), _stream())
    return (out, out2) if epilogue == EPI_BIAS_GELU else out


def qkv_projection(mode: ComputeMode, xb: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, C: int, heads: int,
                   need_stats: bool = True):
    """qkv = xb @ W^T + b with q and k L2-normalised per head; returns (qkv, inv_norm (T, 2, heads)), inv_norm None when
    not `need_stats`.
    tcgen05 / head_dim 96: the normalisation runs in the GEMM epilogue (accumulators never leave fp32 before it);
    otherwise the GEMM is followed by the stand-alone normalisation kernel."""
    T = xb.shape[0]
    if mode.gemm_backend == BACKEND_TCGEN05 and C // heads == 96:
        qkv = torch.empty((T, 3 * C), dtype=xb.dtype, device=xb.device)
        inv_norm = torch.empty((T, 2, heads), dtype=torch.float32, device=xb.device) if need_stats else None
        _lib.call("swinb200_gemm", BACKEND_TCGEN05, T, 3 * C, C, _chk(xb, "xb", torch.bfloat16), 0, C, _chk(w, "w", torch.bfloat16), 0, C,
                  BF16, EPI_BIAS_QKNORM, _chk(bias, "bias", torch.float32), qkv.data_ptr(), 3 * C,
                  0 if inv_norm is None else inv_norm.data_ptr(), 0, 96, BF16, 0, 1, _stream())
        return qkv, inv_norm
    qkv = gemm(mode, xb, 0, w, 0, EPI_BIAS, bias=bias)
    return qkv, qk_normalize_(qkv, C, heads, need_stats)


def wgrad_split_k(M: int, N: int, K: int) -> int:
    """Split-K factor for a weight-gradient GEMM (few 128x256 output tiles, K = tokens): the smallest split in
    [2, 16] whose tile x split count fills whole waves of the persistent grid best (>= 95 % of the last wave),
    so the 148 SMs neither idle in a ragged tail nor pay for more fp32 reduce-add traffic than needed."""
    tiles = ((M + 127) // 128) * ((N + 255) // 256 if N > 128 else 1)
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    kb = (K + 63) // 64
    best, best_eff = 1, 0.0
    for s in range(1, min(16, kb) + 1):
        items = tiles * s
        eff = items / (((items + sms - 1) // sms) * sms)
        if items >= sms and eff >= 0.95:
            return s
        if eff > best_eff + 1e-9:
            best, best_eff = s, eff
    return best


# ---- LayerNorm + residual ------------------------------------------------------------------------------
def ln_residual_fwd(z, x_in, gamma, beta, sample_scale, pos, rows_per_sample: int, mode: ComputeMode, need_stats: bool = True):
    """-> (x_out, xb_out, stats (rows, 2) or None when not `need_stats`)"""
    rows, C = z.shape
    x_out = torch.empty((rows, C), dtype=torch.float32, device=z.device)
    xb = x_out if mode.act_dtype == torch.float32 else torch.empty((rows, C), dtype=mode.act_dtype, device=z.device)
    stats = torch.empty((rows, 2), dtype=torch.float32, device=z.device) if need_stats else None
    _lib.call("swinb200_ln_residual_fwd", _chk(z, "z", mode.act_dtype), mode.act_code, _chk(x_in, "x_in", torch.float32, True),
              _chk(gamma, "gamma", torch.float32), _chk(beta, "beta", torch.float32),
              _chk(sample_scale, "sample_scale", torch.float32, True), _chk(pos, "pos", torch.float32, True),
              x_out.data_ptr(), xb.data_ptr(), 0 if stats is None else stats.data_ptr(), rows, C, rows_per_sample, LN_EPS, _stream())
    return x_out, xb, stats


def linear_wgrad(mode: ComputeMode, dy: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, dbias: Optional[torch.Tensor],
                 split_k: int, fuse: bool = True):
    """dw (n_out, n_in) fp32 += dy^T x ;  dbias (n_out) fp32 += column sums of dy  (both pre-zeroed accumulators).
    tcgen05, n_out a multiple of 256: ONE kernel -- the epilogue warps of the weight-gradient GEMM sum the dy tiles the main
    loop stages in shared memory (swinb200_linear_wgrad), so dy is not read again by a column-sum pass.  Otherwise (and with
    fuse=False): the split-K GEMM followed by swinb200_colsum."""
    T, n_out = dy.shape
    n_in = x.shape[1]
    if fuse and dbias is not None and mode.gemm_backend == BACKEND_TCGEN05 and n_out % 256 == 0 and n_in >= 256:
        if deterministic():
            part = _scratch(split_k * (n_out * n_in + n_out), dy.device)
            _lib.call("swinb200_linear_wgrad_det", BACKEND_TCGEN05, n_out, n_in, T, _chk(dy, "dy", torch.bfloat16), n_out,
                      _chk(x, "x", torch.bfloat16), n_in, _chk(dw, "dw", torch.float32), _chk(dbias, "dbias", torch.float32),
                      int(split_k), part.data_ptr(), part.numel(), _stream())
            return dw, dbias
        _lib.call("swinb200_linear_wgrad", BACKEND_TCGEN05, n_out, n_in, T, _chk(dy, "dy", torch.bfloat16), n_out,
                  _chk(x, "x", torch.bfloat16), n_in, _chk(dw, "dw", torch.float32), n_in, _chk(dbias, "dbias", torch.float32),
                  int(split_k), _stream())
        return dw, dbias
    gemm(mode, dy, 1, x, 1, EPI_F32, out=dw, accumulate=True, split_k=split_k)
    if dbias is not None:
        colsum(dy, out=dbias)
    return dw, dbias


_LN_COUNTERS = {}


def linear_ln_residual(mode: ComputeMode, a, w, bias, x_in, gamma, beta, sample_scale, rows_per_sample: int,
                       fuse: Optional[bool] = None, need_stats: bool = True):
    """z = a @ w^T + bias ; x_out = x_in + sample_scale * (LN(z) gamma + beta)  ->  (z, x_out, xb_out, stats).

    Two implementations with identical results (tests/test_kernels_gpu.py::test_linear_ln_residual_fused_epilogue):
    * the GEMM followed by the stand-alone LayerNorm kernel (default);
    * `fuse=True` / SWINB200_FUSE_LN=1, tcgen05 / 768 channels: ONE kernel, the LayerNorm + DropPath scale + residual run
      inside the GEMM epilogue (swinb200_linear_ln_residual).  Measured on the B200 it is not faster -- fc2: 323 us against
      216 + 105 us, proj: 225 us against 65 + 105 us -- because the LayerNorm's 600 MB of HBM traffic raises the latency of
      the operand loads beyond what the 4-stage ring covers (DESIGN.md section 5.2), so the model keeps the two kernels.
    `need_stats=False` drops the statistics of the two-kernel path (None is returned); the fused kernel always stores them."""
    M, K = a.shape
    N = w.shape[0]
    if fuse is None:
        env = os.environ.get("SWINB200_FUSE_LN", "0")          # 1: every eligible GEMM; 2: only the long-K ones (fc2)
        fuse = env == "1" or (env == "2" and K >= 2048)
    if not (fuse and mode.gemm_backend == BACKEND_TCGEN05 and N == 768):
        z = gemm(mode, a, 0, w, 0, EPI_BIAS, bias=bias)
        return (z,) + ln_residual_fwd(z, x_in, gamma, beta, sample_scale, None, rows_per_sample, mode, need_stats)
    dev = a.device
    counters = _LN_COUNTERS.get(dev)
    n_blocks = (M + 127) // 128
    if counters is None or counters.numel() < n_blocks:
        counters = _LN_COUNTERS[dev] = torch.zeros((max(4096, n_blocks),), dtype=torch.int32, device=dev)
    z = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
    x_out = torch.empty((M, N), dtype=torch.float32, device=dev)
    xb = torch.empty((M, N), dtype=torch.bfloat16, device=dev)
    stats = torch.empty((M, 2), dtype=torch.float32, device=dev)
    _lib.call("swinb200_linear_ln_residual", BACKEND_TCGEN05, M, N, K, _chk(a, "a", torch.bfloat16), K, _chk(w, "w", torch.bfloat16), K,
              _chk(bias, "bias", torch.float32, True), z.data_ptr(), N, _chk(x_in, "x_in", torch.float32),
              _chk(gamma, "gamma", torch.float32), _chk(beta, "beta", torch.float32),
              _chk(sample_scale, "sample_scale", torch.float32, True), x_out.data_ptr(), xb.data_ptr(), stats.data_ptr(),
              rows_per_sample, LN_EPS, counters.data_ptr(), counters.numel(), _stream())
    return z, x_out, xb, stats


def ln_residual_bwd(dx, z, stats, gamma, sample_scale, rows_per_sample: int, mode: ComputeMode, want_dbias_prev=True,
                    acc: Optional[torch.Tensor] = None):
    """`acc`: optional pre-zeroed (3, C) fp32 accumulator (dgamma, dbeta, dbias_prev)."""
    rows, C = z.shape
    dz = torch.empty((rows, C), dtype=mode.act_dtype, device=z.device)
    if acc is None:
        acc = torch.zeros((3, C), dtype=torch.float32, device=z.device)
    if deterministic():
        part = _scratch(3 * C * 256 * max(1, 2048 // C), z.device)
        _lib.call("swinb200_ln_residual_bwd_det", _chk(dx, "dx", torch.float32), _chk(z, "z", mode.act_dtype), mode.act_code,
                  _chk(stats, "stats", torch.float32), _chk(gamma, "gamma", torch.float32),
                  _chk(sample_scale, "sample_scale", torch.float32, True), dz.data_ptr(), acc[0].data_ptr(), acc[1].data_ptr(),
                  acc[2].data_ptr() if want_dbias_prev else 0, rows, C, rows_per_sample, part.data_ptr(), part.numel(), _stream())
        return dz, acc[0], acc[1], acc[2]
    _lib.call("swinb200_ln_residual_bwd", _chk(dx, "dx", torch.float32), _chk(z, "z", mode.act_dtype), mode.act_code,
              _chk(stats, "stats", torch.float32), _chk(gamma, "gamma", torch.float32),
              _chk(sample_scale, "sample_scale", torch.float32, True), dz.data_ptr(), acc[0].data_ptr(), acc[1].data_ptr(),
              acc[2].data_ptr() if want_dbias_prev else 0, rows, C, rows_per_sample, _stream())
    return dz, acc[0], acc[1], acc[2]


def transpose_f32(src: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    R, Cc = src.shape
    dst = torch.empty((Cc, R), dtype=torch.float32, device=src.device) if out is None else out
    if tuple(dst.shape) != (Cc, R):
        raise SwinB200Error(f"transpose_f32: out has shape {tuple(dst.shape)}, expected {(Cc, R)}")
    _chk(dst, "out", torch.float32)
    _lib.call("swinb200_transpose_f32", _chk(src, "src", torch.float32), dst.data_ptr(), R, Cc, _stream())
    return dst


def pos_embed_grad(dx: torch.Tensor, B: int, rows_per_sample: int, C: int) -> torch.Tensor:
    dpos = torch.empty((C, rows_per_sample), dtype=torch.float32, device=dx.device)
    _lib.call("swinb200_pos_embed_grad", _chk(dx, "dx", torch.float32), dpos.data_ptr(), B, rows_per_sample, C, _stream())
    return dpos


def colsum(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`out`: optional pre-zeroed (cols,) fp32 accumulator."""
    rows, cols = x.shape
    if out is None:
        out = torch.zeros((cols,), dtype=torch.float32, device=x.device)
    if deterministic():
        part = _scratch(cols * min((rows + 63) // 64, 256), x.device)
        _lib.call("swinb200_colsum_det", _chk(x, "x"), _code(x.dtype), out.data_ptr(), rows, cols, cols, part.data_ptr(), part.numel(),
                  _stream())
        return out
    _lib.call("swinb200_colsum", _chk(x, "x"), _code(x.dtype), out.data_ptr(), rows, cols, cols, _stream())
    return out


# ---- attention --------------------------------------------------------------------------------------------
def qk_normalize_(qkv: torch.Tensor, C: int, heads: int, need_stats: bool = True) -> Optional[torch.Tensor]:
    T = qkv.shape[0]
    inv_norm = torch.empty((T, 2, heads), dtype=torch.float32, device=qkv.device) if need_stats else None
    _lib.call("swinb200_qk_normalize", _chk(qkv, "qkv"), _code(qkv.dtype), 0 if inv_norm is None else inv_norm.data_ptr(), T, C,
              heads, _stream())
    return inv_norm


def shift_mask(H, W, Wh, Ww, s0, s1, device) -> torch.Tensor:
    nW, L = (H // Wh) * (W // Ww), Wh * Ww
    mask = torch.empty((nW, L, L), dtype=torch.float32, device=device)
    _lib.call("swinb200_shift_mask", mask.data_ptr(), H, W, Wh, Ww, s0, s1, _stream())
    return mask


TCGEN05_HEAD_DIMS = (48, 64, 96, 128, 192, 256)


def attn_backend_for(mode: ComputeMode, C: int, heads: int, Wh: int, Ww: int) -> int:
    """bf16 mode runs window attention on the tcgen05 kernels for head_dim 48 / 64 / 96 / 128 / 192 / 256 and any window
    size: the tuned persistent kernels for head_dim 96 with up to 176 (padded) tokens per window -- the 9x18 = 162 headline
    config -- and the tiled flash-style kernels (csrc/attn_tc_gen.cu) for everything else (BASELINE config 5, the e2048 /
    head_dim-256 config).  Other head dims and the fp32 validation mode run on the CUDA-core kernels; this is a dispatch on
    the problem shape decided up front, not an error fallback."""
    if mode.attn_backend == BACKEND_TCGEN05 and C // heads in TCGEN05_HEAD_DIMS:
        return BACKEND_TCGEN05
    return BACKEND_SIMT


def window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, Wh, Ww, s0, s1, mode: ComputeMode, backend=None, need_stats: bool = True):
    """-> (o, lse (2, B, nW, heads, L) or None when not `need_stats`)"""
    T = B * H * W
    if backend is None:
        backend = attn_backend_for(mode, C, heads, Wh, Ww)
    nW, L = (H // Wh) * (W // Ww), Wh * Ww
    o = torch.empty((T, C), dtype=qkv.dtype, device=qkv.device)
    lse = None
    if need_stats:
        lse = torch.empty((2, B, nW, heads, L), dtype=torch.float32, device=qkv.device)   # plane 0: LSE, plane 1: mean cosine
    _lib.call("swinb200_window_attn_fwd", backend, _chk(qkv, "qkv"), _code(qkv.dtype),
              _chk(scale, "scale", torch.float32), _chk(bias, "bias", torch.float32, True), o.data_ptr(),
              0 if lse is None else lse.data_ptr(),
              B, H, W, C, heads, Wh, Ww, s0, s1, _stream())
    return o, lse


def window_attn_bwd(qkv, inv_norm, scale, bias, o, d_o, lse, B, H, W, C, heads, Wh, Ww, s0, s1, mode: ComputeMode,
                    backend=None, dscale: Optional[torch.Tensor] = None):
    L = Wh * Ww
    if backend is None:
        backend = attn_backend_for(mode, C, heads, Wh, Ww)
    dqkv = torch.empty_like(qkv)
    if dscale is None:
        dscale = torch.zeros((heads,), dtype=torch.float32, device=qkv.device)
    dbias = torch.zeros((heads, L, L), dtype=torch.float32, device=qkv.device) if bias is not None else None
    # scratch for the row term D = <dO, O> (required by the tcgen05 back end)
    ws = torch.empty((qkv.shape[0] * heads,), dtype=torch.float32, device=qkv.device) if backend == BACKEND_TCGEN05 else None
    if deterministic():
        items = B * (H // Wh) * (W // Ww) * heads
        part = _scratch(items * (4 * ((L + 127) // 128) + (L * L if dbias is not None else 0)), qkv.device)
        _lib.call("swinb200_window_attn_bwd_det", backend, _chk(qkv, "qkv"), _code(qkv.dtype),
                  _chk(inv_norm, "inv_norm", torch.float32), _chk(scale, "scale", torch.float32),
                  _chk(bias, "bias", torch.float32, True), _chk(o, "o", qkv.dtype), _chk(d_o, "d_o", qkv.dtype),
                  _chk(lse, "lse", torch.float32), dqkv.data_ptr(), dscale.data_ptr(), 0 if dbias is None else dbias.data_ptr(),
                  0 if ws is None else ws.data_ptr(), B, H, W, C, heads, Wh, Ww, s0, s1, part.data_ptr(), part.numel(), _stream())
        return dqkv, dscale, dbias
    _lib.call("swinb200_window_attn_bwd", backend, _chk(qkv, "qkv"), _code(qkv.dtype),
              _chk(inv_norm, "inv_norm", torch.float32), _chk(scale, "scale", torch.float32),
              _chk(bias, "bias", torch.float32, True), _chk(o, "o", qkv.dtype), _chk(d_o, "d_o", qkv.dtype),
              _chk(lse, "lse", torch.float32), dqkv.data_ptr(), dscale.data_ptr(), 0 if dbias is None else dbias.data_ptr(),
              0 if ws is None else ws.data_ptr(), B, H, W, C, heads, Wh, Ww, s0, s1, _stream())
    return dqkv, dscale, dbias


# ---- loss ---------------------------------------------------------------------------------------------------
def latw_l2_fwd(prd, tar, qw, chw, relative: bool, squared: bool = True):
    _check_loss_args(prd, tar, qw, chw)
    B, C, H, W = prd.shape
    num = torch.empty((B * C,), dtype=torch.float32, device=prd.device)
    den = torch.empty((B * C,), dtype=torch.float32, device=prd.device)
    loss = torch.empty((1,), dtype=torch.float32, device=prd.device)
    if deterministic():
        part = _scratch(2 * B * C * H, prd.device)
        _lib.call("swinb200_latw_l2_fwd_det", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32),
                  _chk(qw, "qw", torch.float32), _chk(chw, "chw", torch.float32), int(relative), int(squared), num.data_ptr(),
                  den.data_ptr(), loss.data_ptr(), B, C, H, W, part.data_ptr(), part.numel(), _stream())
        return loss, num, den
    _lib.call("swinb200_latw_l2_fwd", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32), _chk(qw, "qw", torch.float32),
              _chk(chw, "chw", torch.float32), int(relative), int(squared), num.data_ptr(), den.data_ptr(), loss.data_ptr(), B, C, H, W, _stream())
    return loss, num, den


def latw_l2_bwd(prd, tar, qw, chw, num, den, gloss, relative: bool, squared: bool = True):
    _check_loss_args(prd, tar, qw, chw)
    B, C, H, W = prd.shape
    dprd = torch.empty_like(prd)
    _lib.call("swinb200_latw_l2_bwd", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32), _chk(qw, "qw", torch.float32),
              _chk(chw, "chw", torch.float32), _chk(num, "num", torch.float32), _chk(den, "den", torch.float32),
              _chk(gloss, "gloss", torch.float32), int(relative), int(squared), dprd.data_ptr(), B, C, H, W, _stream())
    return dprd


def _check_loss_args(prd, tar, qw, chw=None):
    if prd.dim() != 4 or prd.shape != tar.shape:
        raise SwinB200Error(f"loss: prediction {tuple(prd.shape)} and target {tuple(tar.shape)} must be equal (B, C, H, W) shapes")
    if qw.numel() != prd.shape[2]:
        raise SwinB200Error(f"loss: {qw.numel()} quadrature row weights for {prd.shape[2]} rows")
    if chw is not None and chw.numel() != prd.shape[1]:
        raise SwinB200Error(f"loss: {chw.numel()} channel weights for {prd.shape[1]} channels")


def latw_l1_fwd(prd, tar, qw, chw, relative: bool):
    _check_loss_args(prd, tar, qw, chw)
    B, C, H, W = prd.shape
    sums = torch.empty((B * C, 2), dtype=torch.float32, device=prd.device)
    loss = torch.empty((1,), dtype=torch.float32, device=prd.device)
    if deterministic():
        part = _scratch(2 * B * C * H, prd.device)
        _lib.call("swinb200_latw_l1_fwd_det", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32),
                  _chk(qw, "qw", torch.float32), _chk(chw, "chw", torch.float32), int(relative), sums.data_ptr(), loss.data_ptr(),
                  B, C, H, W, part.data_ptr(), part.numel(), _stream())
        return loss, sums
    _lib.call("swinb200_latw_l1_fwd", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32), _chk(qw, "qw", torch.float32),
              _chk(chw, "chw", torch.float32), int(relative), sums.data_ptr(), loss.data_ptr(), B, C, H, W, _stream())
    return loss, sums


def latw_l1_bwd(prd, tar, qw, chw, sums, gloss, relative: bool):
    _check_loss_args(prd, tar, qw, chw)
    B, C, H, W = prd.shape
    dprd = torch.empty_like(prd)
    _lib.call("swinb200_latw_l1_bwd", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32), _chk(qw, "qw", torch.float32),
              _chk(chw, "chw", torch.float32), _chk(sums, "sums", torch.float32), _chk(gloss, "gloss", torch.float32), int(relative),
              dprd.data_ptr(), B, C, H, W, _stream())
    return dprd


def latw_acc(prd, tar, qw):
    """(B, C) anomaly correlation sum(q p t) / sqrt(sum(q p p) sum(q t t)) in one pass over prd and tar."""
    _check_loss_args(prd, tar, qw)
    B, C, H, W = prd.shape
    sums = torch.empty((B * C, 3), dtype=torch.float32, device=prd.device)
    acc = torch.empty((B, C), dtype=torch.float32, device=prd.device)
    if deterministic():
        part = _scratch(3 * B * C * H, prd.device)
        _lib.call("swinb200_latw_acc_det", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32),
                  _chk(qw, "qw", torch.float32), sums.data_ptr(), acc.data_ptr(), B, C, H, W, part.data_ptr(), part.numel(), _stream())
        return acc
    _lib.call("swinb200_latw_acc", _chk(prd, "prd", torch.float32), _chk(tar, "tar", torch.float32), _chk(qw, "qw", torch.float32),
              sums.data_ptr(), acc.data_ptr(), B, C, H, W, _stream())
    return acc
