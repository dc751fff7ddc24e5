"""Autograd wiring of the hot path: each Function's forward/backward is a fixed sequence of our CUDA
kernels (swin_v2_weather_b200/ops.py).  Nothing here computes with PyTorch ops except trivial views.

Saved-for-backward per block (bf16 mode, per token): xb, qkv (q^,k^,v), o, z1, xb_mid, h, g, z2 in
activation storage + fp32 row statistics -- ~24.6 KB/token, 1.6 GB per block per 64,800-token sample.

Forward-only runs (no gradient will be taken): `patch_embed_forward_only`, `block_forward_only` and `head_forward_only` issue
the C-ABI sequence of the three Functions' forwards with fc1 on the single-output BIAS_GELU_FWD epilogue (the pre-activation
h is never written) and NULL row statistics, and save nothing.  Every output is bit-identical to the training forward's.
"""
from __future__ import annotations

import weakref
from typing import Dict, Optional, Tuple

import torch

from . import ops
from .ops import ComputeMode, EPI_ADD_F32, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_GELU_FWD, EPI_DGELU, EPI_F32


# ---- bf16 weight shadows ------------------------------------------------------------------------------
class _ShadowCache:
    """bf16 copies of fp32 master weights, refreshed when the parameter's version counter moves
    (optimizer.step() bumps it).  Parameters themselves are never replaced (optimizer / DDP hold them).
    Entries are validated by object identity (weak reference), version and storage pointer: `id()` values and
    allocator blocks are both recycled once a model is freed, so neither alone identifies a parameter.
    The same entries hold the token-major fp32 copy of pos_embed that forward-only runs read (`pos_tokens`)."""

    def __init__(self):
        self._store: Dict[object, Tuple[weakref.ref, int, int, torch.Tensor]] = {}

    def _cached(self, key, w: torch.Tensor, shape, make) -> torch.Tensor:
        """The entry `key` derived from `w` (expected `shape`), rebuilt by make(old buffer or None) when `w` has changed."""
        ent = self._store.get(key)
        ver, ptr = w._version, w.data_ptr()
        if ent is not None and ent[0]() is w and ent[1] == ver and ent[2] == ptr and ent[3].shape == shape:
            return ent[3]
        reuse = ent is not None and ent[0]() is w and ent[3].shape == shape and ent[3].device == w.device
        sh = make(ent[3] if reuse else None)
        if ent is None:     # a new parameter: drop the shadows of parameters that have been freed since (discarded models)
            self._store = {k: v for k, v in self._store.items() if v[0]() is not None}
        self._store[key] = (weakref.ref(w), ver, ptr, sh)
        return sh

    def get(self, w: torch.Tensor, mode: ComputeMode) -> torch.Tensor:
        if mode.act_dtype == torch.float32:
            return w.detach()
        return self._cached(id(w), w, w.shape, lambda old: ops.cast_bf16(w.detach().contiguous(), old))

    def pos_tokens(self, pos_embed: torch.Tensor) -> torch.Tensor:
        """(H*W, E) fp32 token-major copy of the (1, E, H, W) pos_embed parameter, rewritten only when the parameter has changed
        (forward-only runs; the training forward transposes it every call, as it always has)."""
        E = pos_embed.shape[1]
        rows = pos_embed.numel() // E
        return self._cached(("pos_tokens", id(pos_embed)), pos_embed, (rows, E),
                            lambda old: ops.transpose_f32(pos_embed.detach().reshape(E, rows), old))

    def peek(self, w: torch.Tensor):
        """The live shadow of `w` (possibly stale), or None -- lets the fused optimizer rewrite it in its own pass."""
        ent = self._store.get(id(w))
        if ent is not None and ent[0]() is w and ent[2] == w.data_ptr() and ent[3].shape == w.shape:
            return ent[3]
        return None

    def mark_fresh(self, w: torch.Tensor) -> None:
        """The shadow of `w` has just been rewritten from its current value by someone else (optim.Adam)."""
        ent = self._store.get(id(w))
        if ent is not None and ent[0]() is w:
            self._store[id(w)] = (ent[0], w._version, w.data_ptr(), ent[3])

    def clear(self):
        self._store.clear()


SHADOWS = _ShadowCache()


def _flat2(w: torch.Tensor) -> torch.Tensor:
    return w.reshape(w.shape[0], -1)


# ---- PatchEmbed (+ LayerNorm + pos_embed) --------------------------------------------------------------
class PatchEmbedFn(torch.autograd.Function):
    """reference: PatchEmbed.forward + `x + pos_embed` (swinv2_global.py:540-546, 779-780).
    Returns the fp32 token stream (B, H, W, C) and its activation-type shadow."""

    @staticmethod
    def forward(ctx, img, proj_w, proj_b, norm_w, norm_b, pos_embed, patch: int, mode: ComputeMode, in_mean, in_std, *more_channels):
        """`more_channels`: further (B or 1, C_s, Hi, Wi) tensors whose channels follow those of `img` (zenith angle, static
        land-mask / orography features): the im2col reads all of them in place, torch.cat never runs.
        `in_mean` / `in_std`: optional (Cin,) per-channel statistics; the im2col then reads (x - mean) / std -- the loaders'
        z-score (data_loader_era5_dali.py:77-90) without a normalised copy of the field."""
        ctx.set_materialize_grads(False)   # no zero-filled gradient for the (non-differentiable) bf16 shadow output
        B, C0, Hi, Wi = img.shape
        Cin = C0 + sum(t.shape[1] for t in more_channels)
        E = proj_w.shape[0]
        H, W = Hi // patch, Wi // patch
        if more_channels or in_mean is not None:
            patches = ops.patchify_cat([img.contiguous()] + [t.detach().float().contiguous() for t in more_channels], patch, mode,
                                       in_mean, in_std)
        else:
            patches = ops.patchify(img.contiguous(), patch, 0, mode)                   # (T, Cin*P*P)
        w2 = SHADOWS.get(proj_w, mode).reshape(E, -1)
        if w2.shape[1] != patches.shape[1]:
            raise ValueError(f"PatchEmbed: input has {Cin} channels, the projection expects {w2.shape[1] // (patch * patch)}")
        z0 = ops.gemm(mode, patches, 0, w2, 0, EPI_BIAS, bias=proj_b.detach())        # (T, E)
        pos_tok = None
        if pos_embed is not None:
            pos_tok = ops.transpose_f32(pos_embed.detach().reshape(E, H * W))          # (H*W, E) token-major
        x, xb, stats = ops.ln_residual_fwd(z0, None, norm_w.detach(), norm_b.detach(), None, pos_tok, H * W, mode)
        ctx.save_for_backward(patches, z0, stats, norm_w, proj_w)
        ctx.meta = (B, C0, Cin, Hi, Wi, E, H, W, patch, mode, pos_embed is not None, tuple(proj_w.shape), len(more_channels))
        ctx.in_std = in_std
        shadow = xb if mode.act_dtype != torch.float32 else x.new_empty(0)   # fp32 mode: the stream is its own shadow
        ctx.mark_non_differentiable(shadow)
        return x.view(B, H, W, E), shadow

    @staticmethod
    def backward(ctx, dx, _dxb):
        patches, z0, stats, norm_w, proj_w = ctx.saved_tensors
        B, C0, Cin, Hi, Wi, E, H, W, patch, mode, has_pos, wshape, n_more = ctx.meta
        dx = dx.contiguous().view(B * H * W, E)
        dpos = ops.pos_embed_grad(dx, B, H * W, E).view(1, E, H, W) if has_pos else None
        dz0, dgamma, dbeta, dbias = ops.ln_residual_bwd(dx, z0, stats, norm_w.detach(), None, H * W, mode)
        K = patches.shape[1]
        dw = torch.zeros((E, K), dtype=torch.float32, device=dx.device)
        ops.gemm(mode, dz0, 1, patches, 1, EPI_F32, out=dw, accumulate=True, split_k=ops.wgrad_split_k(E, K, dz0.shape[0]))
        dimg = None
        if ctx.needs_input_grad[0]:
            # multi-step rollouts (networks/helpers.py:26-41) back-propagate into the previous step's prediction:
            # d patches = dz0 @ W (dgrad GEMM, weight read n-major), scattered back by the im2col adjoint.  Only the
            # channels of `img` itself carry a gradient (the appended zenith / static channels are data).
            w2 = SHADOWS.get(proj_w, mode).reshape(E, -1)
            if C0 != Cin:
                w2 = w2[:, :C0 * patch * patch].contiguous()
            dpatch = ops.gemm(mode, dz0, 0, w2, 1, EPI_BIAS)                          # (T, C0*P*P), columns (c, p, q)
            dimg = ops.unpatchify(dpatch, None, B, C0, Hi, Wi, patch, order=0)
            if ctx.in_std is not None:      # d/dx (x - m)/s = 1/s
                dimg = dimg / ctx.in_std[:C0].view(1, C0, 1, 1)
        return (dimg, dw.view(wshape), dbias, dgamma, dbeta, dpos, None, None, None, None) + (None,) * n_more


def patch_embed_forward_only(img, proj_w, proj_b, norm_w, norm_b, pos_embed, patch: int, mode: ComputeMode, in_mean, in_std,
                             *more_channels):
    """PatchEmbedFn.forward without saving anything: the LayerNorm statistics are not stored and the token-major pos_embed
    comes from the shadow cache instead of a fresh transpose.  Returns (x (B, H, W, E), shadow) as the Function does."""
    B, C0, Hi, Wi = img.shape
    E = proj_w.shape[0]
    H, W = Hi // patch, Wi // patch
    if more_channels or in_mean is not None:
        patches = ops.patchify_cat([img.contiguous()] + [t.detach().float().contiguous() for t in more_channels], patch, mode,
                                   in_mean, in_std)
    else:
        patches = ops.patchify(img.contiguous(), patch, 0, mode)
    w2 = SHADOWS.get(proj_w, mode).reshape(E, -1)
    if w2.shape[1] != patches.shape[1]:
        Cin = C0 + sum(t.shape[1] for t in more_channels)
        raise ValueError(f"PatchEmbed: input has {Cin} channels, the projection expects {w2.shape[1] // (patch * patch)}")
    z0 = ops.gemm(mode, patches, 0, w2, 0, EPI_BIAS, bias=proj_b.detach())
    del patches
    pos_tok = SHADOWS.pos_tokens(pos_embed) if pos_embed is not None else None
    x, xb, _ = ops.ln_residual_fwd(z0, None, norm_w.detach(), norm_b.detach(), None, pos_tok, H * W, mode, need_stats=False)
    shadow = xb if mode.act_dtype != torch.float32 else x.new_empty(0)
    return x.view(B, H, W, E), shadow


# ---- one SwinV2 block ------------------------------------------------------------------------------------
class SwinBlockFn(torch.autograd.Function):
    """reference: SwinTransformerV2CrBlock.forward (swinv2_global.py:480-497) with the attention module
    (:170-201 / :289-321), shift/partition/reverse (:446-478) and timm Mlp folded in.

    Inputs: x fp32 (B,H,W,C) residual stream, xb its activation-type shadow, `scale` =
    exp(min(logit_scale, ln 100)) (heads,), `bias` = CPB table (heads, L, L) or None, and
    `dp1`/`dp2` = per-sample DropPath multipliers (B,) or None."""

    @staticmethod
    def forward(ctx, x, xb, scale, bias, qkv_w, qkv_b, proj_w, proj_b, n1_w, n1_b, fc1_w, fc1_b, fc2_w, fc2_b, n2_w, n2_b,
                dp1, dp2, geom, mode: ComputeMode):
        ctx.set_materialize_grads(False)
        B, H, W, C = x.shape
        heads, Wh, Ww, s0, s1 = geom
        T = B * H * W
        x2 = x.contiguous().view(T, C)
        if mode.act_dtype == torch.float32:
            xb = x2
        wq, wp = SHADOWS.get(qkv_w, mode), SHADOWS.get(proj_w, mode)
        w1, w2 = SHADOWS.get(fc1_w, mode), SHADOWS.get(fc2_w, mode)
        scale_c = scale.detach().contiguous()
        bias_c = None if bias is None else bias.detach().contiguous()
        # attention branch
        qkv, inv_norm = ops.qkv_projection(mode, xb, wq, qkv_b.detach(), C, heads)              # (T, 3C): q^, k^, v
        o, lse = ops.window_attn_fwd(qkv, scale_c, bias_c, B, H, W, C, heads, Wh, Ww, s0, s1, mode)
        # proj + LayerNorm + DropPath + residual: one kernel on the tcgen05 path (LN in the GEMM epilogue)
        z1, x_mid, xb_mid, st1 = ops.linear_ln_residual(mode, o, wp, proj_b.detach(), x2, n1_w.detach(), n1_b.detach(), dp1, H * W)
        # MLP branch
        g, h = ops.gemm(mode, xb_mid, 0, w1, 0, EPI_BIAS_GELU, bias=fc1_b.detach())             # (T, hidden) x2
        z2, x_out, xb_out, st2 = ops.linear_ln_residual(mode, g, w2, fc2_b.detach(), x_mid, n2_w.detach(), n2_b.detach(), dp2, H * W)
        ctx.save_for_backward(xb, qkv, inv_norm, lse, o, z1, st1, xb_mid, h, g, z2, st2, scale_c, bias_c, qkv_w, proj_w,
                              fc1_w, fc2_w, n1_w, n2_w, dp1, dp2)
        ctx.meta = (B, H, W, C, geom, mode)
        shadow = xb_out if mode.act_dtype != torch.float32 else x_out.new_empty(0)
        ctx.mark_non_differentiable(shadow)
        return x_out.view(B, H, W, C), shadow

    @staticmethod
    def backward(ctx, dx_out, _dxb):
        (xb, qkv, inv_norm, lse, o, z1, st1, xb_mid, h, g, z2, st2, scale_c, bias_c, qkv_w, proj_w, fc1_w, fc2_w, n1_w, n2_w,
         dp1, dp2) = ctx.saved_tensors
        B, H, W, C, geom, mode = ctx.meta
        heads, Wh, Ww, s0, s1 = geom
        T = B * H * W
        hid = h.shape[1]
        dev = dx_out.device
        wq, wp = SHADOWS.get(qkv_w, mode), SHADOWS.get(proj_w, mode)
        w1, w2 = SHADOWS.get(fc1_w, mode), SHADOWS.get(fc2_w, mode)
        dx_out = dx_out.contiguous().view(T, C)

        # every fp32 accumulator of this block's backward (split-K weight gradients, column sums, d logit-scale) lives in
        # one buffer cleared by a single fill instead of ~10 small ones
        sizes = dict(w_qkv=3 * C * C, w_proj=C * C, w_fc1=hid * C, w_fc2=C * hid, ln2=3 * C, ln1=3 * C, b_fc1=hid,
                     b_qkv=3 * C, dscale=heads)
        flat = torch.zeros((sum(-(-v // 64) * 64 for v in sizes.values()),), dtype=torch.float32, device=dev)
        acc, off = {}, 0
        for k, v in sizes.items():
            acc[k] = flat[off:off + v]
            off += -(-v // 64) * 64          # 256-byte aligned slices (TMA reduce-add needs 16 B)

        def wgrad(dy, act_in, n_out, n_in, key):
            dw = acc[key].view(n_out, n_in)
            ops.gemm(mode, dy, 1, act_in, 1, EPI_F32, out=dw, accumulate=True, split_k=ops.wgrad_split_k(n_out, n_in, T))
            return dw

        # ---- MLP branch: x_out = x_mid + dp2 * LN2(fc2(gelu(fc1(xb_mid))))
        dz2, dg2, db2, dbias_fc2 = ops.ln_residual_bwd(dx_out, z2, st2, n2_w.detach(), dp2, H * W, mode, acc=acc["ln2"].view(3, C))
        # Order: every tensor is consumed right after it was produced, and consecutive kernels alternate their direction over
        # the token rows (GEMMs ascend, the row-wise kernels descend), so each one starts on the ~100 MB its predecessor left
        # in L2.  The two weight gradients that do not touch the fresh tensor (fc2: dz2, g; proj: dz1, o) run last.
        dh = ops.gemm(mode, dz2, 0, w2, 1, EPI_DGELU, aux=h)                                     # (T, hidden)
        dx_mid = ops.gemm(mode, dh, 0, w1, 1, EPI_ADD_F32, aux=dx_out)                           # fp32 (T, C)
        # weight + bias gradient of fc1 in one kernel (the bias gradient is the column sum of the dh tiles the GEMM stages)
        dw_fc1, dbias_fc1 = ops.linear_wgrad(mode, dh, xb_mid, acc["w_fc1"].view(hid, C), acc["b_fc1"], ops.wgrad_split_k(hid, C, T))
        del dh
        dw_fc2 = wgrad(dz2, g, C, hid, "w_fc2")
        # ---- attention branch: x_mid = x + dp1 * LN1(proj(attn(qkv(xb))))
        dz1, dg1, db1, dbias_proj = ops.ln_residual_bwd(dx_mid, z1, st1, n1_w.detach(), dp1, H * W, mode, acc=acc["ln1"].view(3, C))
        d_o = ops.gemm(mode, dz1, 0, wp, 1, EPI_BIAS)                                            # (T, C)
        dqkv, dscale, dbias_tab = ops.window_attn_bwd(qkv, inv_norm, scale_c, bias_c, o, d_o, lse, B, H, W, C, heads, Wh, Ww,
                                                       s0, s1, mode, dscale=acc["dscale"])
        dx_in = ops.gemm(mode, dqkv, 0, wq, 1, EPI_ADD_F32, aux=dx_mid)                          # fp32 (T, C)
        dw_qkv, dbias_qkv = ops.linear_wgrad(mode, dqkv, xb, acc["w_qkv"].view(3 * C, C), acc["b_qkv"], ops.wgrad_split_k(3 * C, C, T))
        dw_proj = wgrad(dz1, o, C, C, "w_proj")
        return (dx_in.view(B, H, W, C), None, dscale, dbias_tab, dw_qkv, dbias_qkv, dw_proj, dbias_proj, dg1, db1, dw_fc1,
                dbias_fc1, dw_fc2, dbias_fc2, dg2, db2, None, None, None, None)


def block_forward_only(x, xb, scale, bias, qkv_w, qkv_b, proj_w, proj_b, n1_w, n1_b, fc1_w, fc1_b, fc2_w, fc2_b, n2_w, n2_b,
                       dp1, dp2, geom, mode: ComputeMode):
    """SwinBlockFn.forward without saving anything (same arguments, same (x_out, shadow) result, same bits): fc1 runs the
    single-output BIAS_GELU_FWD epilogue and the LayerNorm / q-k norm / softmax statistics are not stored.  Intermediates are
    released as soon as they are consumed, so the peak is the fc1 output plus the residual stream."""
    B, H, W, C = x.shape
    heads, Wh, Ww, s0, s1 = geom
    T = B * H * W
    x2 = x.contiguous().view(T, C)
    if mode.act_dtype == torch.float32:
        xb = x2
    wq, wp = SHADOWS.get(qkv_w, mode), SHADOWS.get(proj_w, mode)
    w1, w2 = SHADOWS.get(fc1_w, mode), SHADOWS.get(fc2_w, mode)
    scale_c = scale.detach().contiguous()
    bias_c = None if bias is None else bias.detach().contiguous()
    qkv, _ = ops.qkv_projection(mode, xb, wq, qkv_b.detach(), C, heads, need_stats=False)
    o, _ = ops.window_attn_fwd(qkv, scale_c, bias_c, B, H, W, C, heads, Wh, Ww, s0, s1, mode, need_stats=False)
    del qkv
    _, x_mid, xb_mid, _ = ops.linear_ln_residual(mode, o, wp, proj_b.detach(), x2, n1_w.detach(), n1_b.detach(), dp1, H * W,
                                                 need_stats=False)
    del o
    g = ops.gemm(mode, xb_mid, 0, w1, 0, EPI_BIAS_GELU_FWD, bias=fc1_b.detach())
    del xb_mid
    _, x_out, xb_out, _ = ops.linear_ln_residual(mode, g, w2, fc2_b.detach(), x_mid, n2_w.detach(), n2_b.detach(), dp2, H * W,
                                                 need_stats=False)
    shadow = xb_out if mode.act_dtype != torch.float32 else x_out.new_empty(0)
    return x_out.view(B, H, W, C), shadow


# ---- head + unpatchify (+ skip) ------------------------------------------------------------------------------
class HeadFn(torch.autograd.Function):
    """reference: forward_head + `x + skip[:, :out_chans]` (swinv2_global.py:784-803)."""

    @staticmethod
    def forward(ctx, x, xb, head_w, skip, out_chans: int, patch: int, mode: ComputeMode, skip_mean=None, skip_std=None):
        B, H, W, C = x.shape
        if mode.act_dtype == torch.float32:
            xb = x.contiguous().view(B * H * W, C)
        wh = SHADOWS.get(head_w, mode)
        y = ops.gemm(mode, xb, 0, wh, 0, EPI_BIAS)                                               # (T, P*P*Co), cols (p,q,c)
        out = ops.unpatchify(y, None if skip is None else skip.contiguous(), B, out_chans, H * patch, W * patch, patch,
                             skip_mean=skip_mean, skip_std=skip_std)
        ctx.save_for_backward(xb, head_w)
        ctx.skip_std = skip_std
        ctx.meta = (B, H, W, C, out_chans, patch, mode, skip is not None, None if skip is None else skip.shape[1])
        return out

    @staticmethod
    def backward(ctx, dout):
        xb, head_w = ctx.saved_tensors
        B, H, W, C, Co, patch, mode, has_skip, skip_ch = ctx.meta
        wh = SHADOWS.get(head_w, mode)
        dout = dout.contiguous()
        dy = ops.patchify(dout, patch, 1, mode)                                                  # (T, P*P*Co)
        dx = ops.gemm(mode, dy, 0, wh, 1, EPI_F32)                                               # fp32 (T, C)
        N = head_w.shape[0]
        dw = torch.zeros((N, C), dtype=torch.float32, device=dout.device)
        ops.gemm(mode, dy, 1, xb, 1, EPI_F32, out=dw, accumulate=True, split_k=ops.wgrad_split_k(N, C, dy.shape[0]))
        dskip = None
        if has_skip and ctx.needs_input_grad[3]:
            dskip = torch.zeros((B, skip_ch, H * patch, W * patch), dtype=torch.float32, device=dout.device)
            dskip[:, :Co] = dout if ctx.skip_std is None else dout / ctx.skip_std[:Co].view(1, Co, 1, 1)
        return dx.view(B, H, W, C), None, dw, dskip, None, None, None, None, None


def head_forward_only(x, xb, head_w, skip, out_chans: int, patch: int, mode: ComputeMode, skip_mean=None, skip_std=None):
    """HeadFn.forward without saving anything (the head saves no statistics: the launches are the same)."""
    B, H, W, C = x.shape
    if mode.act_dtype == torch.float32:
        xb = x.contiguous().view(B * H * W, C)
    y = ops.gemm(mode, xb, 0, SHADOWS.get(head_w, mode), 0, EPI_BIAS)
    return ops.unpatchify(y, None if skip is None else skip.contiguous(), B, out_chans, H * patch, W * patch, patch,
                          skip_mean=skip_mean, skip_std=skip_std)


# ---- loss ---------------------------------------------------------------------------------------------------------
class LatWeightedL2Fn(torch.autograd.Function):
    """reference: GeometricLpLoss.rel / .abs with p=2, squared (utils/losses.py:188-232) over
    GridQuadrature 'naive' weights (utils/grids.py:68-117).  Returns a 0-d loss (sum over batch and channel)."""

    @staticmethod
    def forward(ctx, prd, tar, qw, chw, relative: bool, squared: bool):
        prd, tar = prd.contiguous(), tar.contiguous()
        loss, num, den = ops.latw_l2_fwd(prd, tar, qw, chw, relative, squared)
        ctx.save_for_backward(prd, tar, qw, chw, num, den)
        ctx.flags = (relative, squared)
        return loss.view(())

    @staticmethod
    def backward(ctx, gloss):
        prd, tar, qw, chw, num, den = ctx.saved_tensors
        g = gloss.detach().to(torch.float32).reshape(1).contiguous()
        dprd = ops.latw_l2_bwd(prd, tar, qw, chw, num, den, g, *ctx.flags)
        return dprd, None, None, None, None, None


class LatWeightedL1Fn(torch.autograd.Function):
    """reference: GeometricLpLoss.rel / .abs with p=1 (utils/losses.py:116-124, 188-232)."""

    @staticmethod
    def forward(ctx, prd, tar, qw, chw, relative: bool):
        prd, tar = prd.contiguous(), tar.contiguous()
        loss, sums = ops.latw_l1_fwd(prd, tar, qw, chw, relative)
        ctx.save_for_backward(prd, tar, qw, chw, sums)
        ctx.relative = relative
        return loss.view(())

    @staticmethod
    def backward(ctx, gloss):
        prd, tar, qw, chw, sums = ctx.saved_tensors
        g = gloss.detach().to(torch.float32).reshape(1).contiguous()
        return ops.latw_l1_bwd(prd, tar, qw, chw, sums, g, ctx.relative), None, None, None, None
