"""GPU parity tests of the individual kernels, called through the C ABI (ctypes), against the CPU oracle
(`oracle/swinv2_oracle.py`) or an fp32 torch restatement of the same op on the same seeded inputs.

Tolerances: fp32 storage -> 1e-5 relative L2 (the north-star fp32 validation bound); bf16 storage ->
1e-2 relative L2 (the bf16 bound); integer / mask work -> bit-exact.
"""
import math

import pytest
import torch

from oracle import swinv2_oracle as O
from swin_v2_weather_b200 import ops
from swin_v2_weather_b200._lib import (BACKEND_SIMT, BACKEND_TCGEN05, EPI_ADD_F32, EPI_BIAS, EPI_BIAS_GELU, EPI_DGELU,
                                        EPI_F32)

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {torch.float32: 1e-5, torch.bfloat16: 1e-2}


def rel(a, b):
    return O.rel_l2(a.float(), b.float())


def mode_for(dtype, tc=False):
    if dtype == torch.float32:
        return ops.MODE_FP32
    return ops.MODE_BF16 if tc else ops.MODE_BF16_SIMT


def gen(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


# ---------------------------------------------------------------------------------------------------------
def test_cast_bf16():
    for n in (8, 1000, 12345, 1 << 20):
        x = gen(n, seed=n)
        assert torch.equal(ops.cast_bf16(x), x.to(torch.bfloat16))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("order", [0, 1])
def test_patchify(dtype, order):
    B, C, Hi, Wi, P = 2, 7, 72, 144, 4
    x = gen(B, C, Hi, Wi, seed=1)
    got = ops.patchify(x, P, order, mode_for(dtype))
    H, W = Hi // P, Wi // P
    v = x.view(B, C, H, P, W, P)
    if order == 0:   # columns (c, p, q): Conv2d im2col
        want = v.permute(0, 2, 4, 1, 3, 5).reshape(B * H * W, C * P * P)
    else:            # columns (p, q, c): inverse of the head's unpatchify
        want = v.permute(0, 2, 4, 3, 5, 1).reshape(B * H * W, C * P * P)
    assert torch.equal(got, want.to(dtype))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("with_skip", [False, True])
def test_unpatchify(dtype, with_skip):
    B, Co, Hi, Wi, P = 2, 5, 72, 144, 4
    H, W = Hi // P, Wi // P
    y = gen(B * H * W, P * P * Co, seed=2).to(dtype)
    skip = gen(B, 7, Hi, Wi, seed=3) if with_skip else None
    got = ops.unpatchify(y, skip, B, Co, Hi, Wi, P)
    want = y.float().view(B, H, W, P, P, Co).permute(0, 5, 1, 3, 2, 4).reshape(B, Co, Hi, Wi)
    if with_skip:
        want = want + skip[:, :Co]
    assert torch.equal(got, want)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_unpatchify_is_adjoint_of_patchify(dtype):
    """order 0 unpatchify inverts order 0 patchify (used for dL/d image in multi-step rollouts)."""
    B, C, Hi, Wi, P = 2, 7, 72, 144, 4
    x = gen(B, C, Hi, Wi, seed=1).to(dtype).float()
    cols = ops.patchify(x, P, 0, mode_for(dtype))
    back = ops.unpatchify(cols, None, B, C, Hi, Wi, P, order=0)
    assert torch.equal(back, x)


def test_transpose_and_pos_grad():
    for shape in ((650, 200), (652, 200), (64, 64), (1300, 772)):     # scalar kernel / 128-bit kernel with ragged tiles
        src = gen(*shape, seed=4)
        assert torch.equal(ops.transpose_f32(src), src.t().contiguous())
    dx = gen(3, 648, 96, seed=5)
    got = ops.pos_embed_grad(dx.view(3 * 648, 96), 3, 648, 96)
    assert rel(got, dx.sum(0).t()) < 1e-6


def test_ln_residual_bwd_ring_kernel():
    """C = 768 / bf16 takes the warp-per-row ring kernel: more tiles than CTAs x stages, and a ragged last tile."""
    C, B, rps = 768, 2, 8 * 148 * 2 + 3
    rows = B * rps
    z = gen(rows, C, seed=16).to(torch.bfloat16)
    gamma, beta = 1 + 0.1 * gen(C, seed=17), 0.1 * gen(C, seed=18)
    ss = torch.tensor([1.0 / 0.8, 0.0], device=DEV)
    dx = gen(rows, C, seed=19)
    for use_ss in (False, True):
        _, _, stats = ops.ln_residual_fwd(z, None, gamma, beta, ss if use_ss else None, None, rps, ops.MODE_BF16)
        dz, dg, db, dbp = ops.ln_residual_bwd(dx, z, stats, gamma, ss if use_ss else None, rps, ops.MODE_BF16)
        zf = z.float().clone().requires_grad_(True)
        gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
        u = torch.nn.functional.layer_norm(zf, (C,), gf, bf, 1e-5)
        if use_ss:
            u = u * ss.repeat_interleave(rps).view(-1, 1)
        u.backward(dx)
        assert rel(dz, zf.grad) < TOL[torch.bfloat16]
        assert rel(dg, gf.grad) < 1e-5 and rel(db, bf.grad) < 1e-5
        assert rel(dbp, zf.grad.sum(0)) < 1e-4      # sum of bf16-rounded dz vs fp32 reference rows


@pytest.mark.parametrize("T,n_out,n_in", [(1000, 512, 256), (5000, 768, 768), (64800, 3072, 768), (64800, 2304, 768)])
def test_linear_wgrad_with_bias_gradient_in_the_same_kernel(T, n_out, n_in):
    """Weight + bias gradient of nn.Linear (reference: autograd of swinv2_global.py:181/300 and timm Mlp.fc1): the column sums
    of dY taken inside the weight-gradient GEMM against the GEMM + column-sum kernels and against torch; ragged token
    counts (last k block partly out of range), accumulation into non-zero buffers."""
    dy = (0.5 * gen(T, n_out, seed=50)).to(torch.bfloat16)
    x = (0.5 * gen(T, n_in, seed=51)).to(torch.bfloat16)
    sk = ops.wgrad_split_k(n_out, n_in, T)
    dw0, db0 = gen(n_out, n_in, seed=52), gen(n_out, seed=53)
    dw, db = ops.linear_wgrad(ops.MODE_BF16, dy, x, dw0.clone(), db0.clone(), sk, fuse=True)
    dw_r, db_r = ops.linear_wgrad(ops.MODE_BF16, dy, x, dw0.clone(), db0.clone(), sk, fuse=False)
    want_w = dw0.double() + dy.double().t() @ x.double()
    want_b = db0.double() + dy.double().sum(0)
    assert rel(dw, want_w.float()) < 5e-5 and rel(dw_r, want_w.float()) < 5e-5      # fp32 accumulation over up to 64,800 tokens
    assert rel(dw, dw_r) < 1e-5
    assert rel(db, want_b.float()) < 1e-5 and rel(db_r, want_b.float()) < 1e-5
    assert float((db.double() - want_b).abs().max()) < 1e-3 * float(want_b.abs().max())


@pytest.mark.parametrize("M,K,B", [(300, 768, 1), (2 * 1296, 3072, 2), (64800, 768, 1), (64800, 3072, 1)])
def test_linear_ln_residual_fused_epilogue(M, K, B):
    """LayerNorm + DropPath scale + residual inside the proj / fc2 GEMM epilogue (north_star (2), reference
    swinv2_global.py:490,494) against the two-kernel path and against torch; ragged row blocks, reused counters."""
    C = 768
    rps = M // B
    a = (0.5 * gen(M, K, seed=40)).to(torch.bfloat16)
    w = (gen(C, K, seed=41) / K ** 0.5).to(torch.bfloat16)
    bias = 0.1 * gen(C, seed=42)
    x_in = gen(M, C, seed=43)
    gamma, beta = 1 + 0.1 * gen(C, seed=44), 0.1 * gen(C, seed=45)
    for ss in (None, torch.tensor([1.0 / 0.9, 0.0][:B], device=DEV)):
        for _ in range(2):        # second call: the block counters must have been left at zero
            z, x_out, xb, stats = ops.linear_ln_residual(ops.MODE_BF16, a, w, bias, x_in, gamma, beta, ss, rps, fuse=True)
        z_ref = ops.gemm(ops.MODE_BF16, a, 0, w, 0, EPI_BIAS, bias=bias)
        x_ref, xb_ref, st_ref = ops.ln_residual_fwd(z_ref, x_in, gamma, beta, ss, None, rps, ops.MODE_BF16)
        assert torch.equal(z, z_ref)
        assert rel(x_out, x_ref) < 1e-6 and float((x_out - x_ref).abs().max()) < 1e-4
        assert torch.equal(xb.float(), x_out.to(torch.bfloat16).float())
        assert rel(stats, st_ref) < 1e-6
        u = torch.nn.functional.layer_norm(z.float(), (C,), gamma, beta, 1e-5)
        if ss is not None:
            u = u * ss.repeat_interleave(rps).view(-1, 1)
        assert rel(x_out, x_in + u) < 1e-6
        assert int(ops._LN_COUNTERS[a.device].abs().sum()) == 0


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("C", [96, 192, 768])
def test_ln_residual_fwd_bwd(dtype, C):
    mode = mode_for(dtype)
    B, rps = 2, 300
    rows = B * rps
    z = gen(rows, C, seed=6).to(dtype)
    x_in = gen(rows, C, seed=7)
    gamma, beta = 1 + 0.1 * gen(C, seed=8), 0.1 * gen(C, seed=9)
    ss = torch.tensor([0.0, 1.0 / 0.9], device=DEV)
    pos = gen(rps, C, seed=10)
    for use_x, use_ss, use_pos in ((True, True, False), (False, False, True), (True, False, False)):
        x_out, xb, stats = ops.ln_residual_fwd(z, x_in if use_x else None, gamma, beta, ss if use_ss else None,
                                               pos if use_pos else None, rps, mode)
        zf = z.float().clone().requires_grad_(True)
        gf, bf = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
        u = torch.nn.functional.layer_norm(zf, (C,), gf, bf, 1e-5)
        if use_pos:
            u = u + pos.repeat(B, 1)
        if use_ss:
            u = u * ss.repeat_interleave(rps).view(-1, 1)
        want = (x_in if use_x else 0) + u
        assert rel(x_out, want) < 1e-6
        assert torch.equal(xb.float(), x_out.to(dtype).float())
        dx = gen(rows, C, seed=11)
        dz, dg, db, dbp = ops.ln_residual_bwd(dx, z, stats, gamma, ss if use_ss else None, rps, mode)
        want.backward(dx)
        assert rel(dz, zf.grad) < TOL[dtype]
        assert rel(dg, gf.grad) < 1e-5 and rel(db, bf.grad) < 1e-5
        assert rel(dbp, zf.grad.sum(0)) < 1e-5      # column sum of dz (bias gradient of the preceding Linear)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_colsum(dtype):
    for rows, cols in ((1000, 768), (333, 3072), (64, 8)):
        x = gen(rows, cols, seed=12).to(dtype)
        assert rel(ops.colsum(x), x.float().sum(0)) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("heads,C", [(8, 768), (2, 192), (4, 768), (12, 768), (16, 768)])
def test_qk_normalize(dtype, heads, C):
    T = 500
    qkv0 = gen(T, 3 * C, seed=13).to(dtype)
    qkv = qkv0.clone()
    inv = ops.qk_normalize_(qkv, C, heads)
    d = C // heads
    ref = qkv0.float().view(T, 3, heads, d)
    nrm = ref[:, :2].norm(dim=-1, keepdim=True).clamp_min(1e-12)
    want = ref.clone()
    want[:, :2] = ref[:, :2] / nrm
    assert rel(qkv.view(T, 3, heads, d)[:, :2], want[:, :2]) < (1e-6 if dtype == torch.float32 else 4e-3)
    assert torch.equal(qkv.view(T, 3, heads, d)[:, 2], qkv0.view(T, 3, heads, d)[:, 2])   # v untouched
    assert rel(inv, 1.0 / nrm.squeeze(-1)) < 1e-6


def test_shift_mask_bit_exact():
    for (H, W, Wh, Ww, s0, s1) in ((18, 36, 9, 18, 4, 9), (180, 360, 9, 18, 4, 9), (12, 24, 6, 12, 3, 6), (18, 36, 18, 18, 0, 9)):
        got = ops.shift_mask(H, W, Wh, Ww, s0, s1, DEV).cpu()
        want = O.shift_attention_mask((H, W), (Wh, Ww), (s0, s1))
        assert torch.equal(got, want), (H, W, Wh, Ww, s0, s1)


# ---- attention ----------------------------------------------------------------------------------------------
def oracle_attention(qkv_raw, scale, bias, B, H, W, C, heads, window, shift):
    """q/k/v (T, 3C) fp32 raw -> (o (T, C), grads fn) with the oracle's index arithmetic."""
    idx = O.window_token_index((H, W), window, shift).to(qkv_raw.device)
    nW, L = idx.shape
    d = C // heads
    tok = qkv_raw.view(B, H * W, 3, heads, d)
    w = tok[:, idx.reshape(-1)].view(B, nW, L, 3, heads, d).permute(3, 0, 1, 4, 2, 5)   # 3,B,nW,h,L,d
    q, k, v = w[0], w[1], w[2]
    qn = q / q.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    kn = k / k.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    s = (qn @ kn.transpose(-1, -2)) * scale.view(1, 1, heads, 1, 1)
    if bias is not None:
        s = s + bias.view(1, 1, heads, L, L)
    mask = O.shift_attention_mask((H, W), window, shift)
    if mask is not None:
        s = s + mask.to(s).view(1, nW, 1, L, L)
    p = torch.softmax(s, dim=-1)
    o = (p @ v).permute(0, 1, 3, 2, 4).reshape(B, nW * L, C)
    out = torch.empty(B, H * W, C, device=o.device, dtype=o.dtype)
    out[:, idx.reshape(-1)] = o
    lse = torch.logsumexp(s, dim=-1)
    return out.reshape(B * H * W, C), lse


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("cfg", [
    dict(B=2, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(0, 0), bias=False),
    dict(B=2, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(4, 9), bias=False),
    dict(B=1, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(4, 9), bias=True),
    dict(B=1, H=12, W=24, C=128, heads=2, window=(6, 12), shift=(3, 6), bias=True),
])
def test_window_attention_simt(dtype, cfg):
    B, H, W, C, heads = cfg["B"], cfg["H"], cfg["W"], cfg["C"], cfg["heads"]
    window, shift = cfg["window"], cfg["shift"]
    L = window[0] * window[1]
    mode = mode_for(dtype)
    T = B * H * W
    raw = gen(T, 3 * C, seed=20).to(dtype)
    scale = torch.tensor([10.0, 13.5][:heads], device=DEV)   # around the reference's init, exp(ln 10)
    bias = (0.5 * gen(heads, L, L, seed=21)) if cfg["bias"] else None
    # oracle (fp32, autograd) on the same stored values
    raw_f = raw.float().requires_grad_(True)
    sc_f = scale.clone().requires_grad_(True)
    b_f = bias.clone().requires_grad_(True) if bias is not None else None
    o_ref, lse_ref = oracle_attention(raw_f, sc_f, b_f, B, H, W, C, heads, window, shift)
    # ours
    qkv = raw.clone()
    inv = ops.qk_normalize_(qkv, C, heads)
    o, lse = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1], mode)
    tol = 2e-5 if dtype == torch.float32 else 1e-2
    assert rel(o, o_ref) < tol
    assert rel(lse[0].reshape(-1), lse_ref.reshape(-1)) < tol
    d_o = gen(T, C, seed=22).to(dtype)
    dqkv, dscale, dbias = ops.window_attn_bwd(qkv, inv, scale, bias, o, d_o, lse, B, H, W, C, heads, window[0], window[1],
                                              shift[0], shift[1], mode)
    o_ref.backward(d_o.float())
    assert rel(dqkv, raw_f.grad) < (5e-5 if dtype == torch.float32 else 2e-2)
    assert rel(dscale, sc_f.grad) < (5e-5 if dtype == torch.float32 else 6e-2)   # SURVEY F9: logit_scale is the noisiest grad
    if bias is not None:
        assert rel(dbias, b_f.grad) < (5e-5 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("cfg", [
    dict(B=2, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(0, 0), bias=False),
    dict(B=2, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(4, 9), bias=False),
    dict(B=1, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(4, 9), bias=True),
    dict(B=1, H=12, W=24, C=192, heads=2, window=(6, 12), shift=(3, 6), bias=True),
    dict(B=1, H=27, W=36, C=96, heads=1, window=(9, 18), shift=(4, 0), bias=False),
    dict(B=1, H=18, W=54, C=96, heads=1, window=(9, 18), shift=(0, 9), bias=False),
    dict(B=1, H=18, W=36, C=192, heads=2, window=(9, 18), shift=(0, 0), bias=False, scale=[8.0, 95.0]),   # exact-max softmax path
])
def test_window_attention_tcgen05(cfg):
    B, H, W, C, heads = cfg["B"], cfg["H"], cfg["W"], cfg["C"], cfg["heads"]
    window, shift = cfg["window"], cfg["shift"]
    L = window[0] * window[1]
    T = B * H * W
    raw = gen(T, 3 * C, seed=20).to(torch.bfloat16)
    scale = torch.tensor(cfg.get("scale", [10.0, 13.5])[:heads], device=DEV)
    bias = (0.5 * gen(heads, L, L, seed=21)) if cfg["bias"] else None
    o_ref, lse_ref = oracle_attention(raw.float(), scale, bias, B, H, W, C, heads, window, shift)
    qkv = raw.clone()
    ops.qk_normalize_(qkv, C, heads)
    o, lse = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1],
                                 ops.MODE_BF16, backend=BACKEND_TCGEN05)
    o2, lse2 = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1],
                                   ops.MODE_BF16, backend=BACKEND_SIMT)
    assert rel(o, o_ref) < 1e-2, (rel(o, o_ref), rel(o2, o_ref))
    assert rel(lse[0].reshape(-1), lse_ref.reshape(-1)) < 1e-2
    assert rel(o, o2) < 1e-2 and rel(lse[0], lse2[0]) < 2e-3     # the two back ends agree with each other
    # backward: tcgen05 vs fp32 autograd of the oracle on the same stored values
    raw_f = raw.float().requires_grad_(True)
    sc_f = scale.clone().requires_grad_(True)
    b_f = bias.clone().requires_grad_(True) if bias is not None else None
    o_r, _ = oracle_attention(raw_f, sc_f, b_f, B, H, W, C, heads, window, shift)
    d_o = gen(T, C, seed=22).to(torch.bfloat16)
    o_r.backward(d_o.float())
    inv = 1.0 / raw.float().view(T, 3, heads, C // heads)[:, :2].norm(dim=-1).clamp_min(1e-12)
    dqkv, dscale, dbias = ops.window_attn_bwd(qkv, inv.contiguous(), scale, bias, o, d_o, lse, B, H, W, C, heads, window[0],
                                              window[1], shift[0], shift[1], ops.MODE_BF16, backend=BACKEND_TCGEN05)
    dqkv2, dscale2, dbias2 = ops.window_attn_bwd(qkv, inv.contiguous(), scale, bias, o, d_o, lse, B, H, W, C, heads, window[0],
                                                 window[1], shift[0], shift[1], ops.MODE_BF16, backend=BACKEND_SIMT)
    Cq = C
    for name, sl in (("dq", slice(0, Cq)), ("dk", slice(Cq, 2 * Cq)), ("dv", slice(2 * Cq, 3 * Cq))):
        e = rel(dqkv[:, sl], raw_f.grad[:, sl])
        e2 = rel(dqkv2[:, sl], raw_f.grad[:, sl])
        assert e < 2e-2, (name, e, e2)
    assert rel(dscale, sc_f.grad) < 6e-2, (dscale, dscale2, sc_f.grad)
    if bias is not None:
        assert rel(dbias, b_f.grad) < 2e-2, (rel(dbias, b_f.grad), rel(dbias2, b_f.grad))


@pytest.mark.parametrize("shift,with_bias", [((0, 0), False), ((4, 9), False), ((4, 9), True)])
def test_window_attention_tcgen05_full_geometry(shift, with_bias):
    """BASELINE size: 180 x 360 tokens, C = 768, 8 heads of 96, 9 x 18 windows -> 3,200 (window, head) items, ~22 per
    persistent CTA.  Exercises what the small cases cannot: operand boxes of the next item arriving under the current
    one, wrap-around windows of the shifted blocks mixed in, per-head d(scale) partials across items."""
    B, H, W, C, heads, window = 1, 180, 360, 768, 8, (9, 18)
    L, T = window[0] * window[1], B * H * W
    raw = gen(T, 3 * C, seed=60).to(torch.bfloat16)
    scale = torch.linspace(8.0, 14.0, heads, device=DEV)
    bias = (0.5 * gen(heads, L, L, seed=61)) if with_bias else None
    raw_f = raw.float().requires_grad_(True)
    sc_f = scale.clone().requires_grad_(True)
    b_f = bias.clone().requires_grad_(True) if bias is not None else None
    o_ref, lse_ref = oracle_attention(raw_f, sc_f, b_f, B, H, W, C, heads, window, shift)
    qkv = raw.clone()
    inv = ops.qk_normalize_(qkv, C, heads)
    o, lse = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1],
                                 ops.MODE_BF16, backend=BACKEND_TCGEN05)
    assert rel(o, o_ref) < 1e-2
    assert rel(lse[0].reshape(-1), lse_ref.reshape(-1)) < 1e-2
    d_o = gen(T, C, seed=62).to(torch.bfloat16)
    o_ref.backward(d_o.float())
    dqkv, dscale, dbias = ops.window_attn_bwd(qkv, inv, scale, bias, o, d_o, lse, B, H, W, C, heads, window[0], window[1],
                                              shift[0], shift[1], ops.MODE_BF16, backend=BACKEND_TCGEN05)
    for name, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        assert rel(dqkv[:, sl], raw_f.grad[:, sl]) < 2e-2, name
    # per-token check as well: a single window gone wrong is invisible in a 64,800-token norm
    err_tok = (dqkv.float() - raw_f.grad).norm(dim=1) / raw_f.grad.norm(dim=1).clamp_min(1e-20)
    assert float(err_tok.max()) < 8e-2, float(err_tok.max())
    assert rel(dscale, sc_f.grad) < 3e-2
    if bias is not None:
        assert rel(dbias, b_f.grad) < 2e-2


@pytest.mark.parametrize("cfg", [
    dict(H=36, W=72, C=384, heads=2, window=(9, 18), shift=(4, 9)),       # d = 192
    dict(H=36, W=72, C=128, heads=2, window=(18, 36), shift=(9, 18)),     # d = 64, 648-token windows
    dict(H=36, W=72, C=192, heads=4, window=(6, 12), shift=(3, 6)),       # d = 48
    dict(H=36, W=72, C=192, heads=2, window=(12, 24), shift=(0, 0)),      # d = 96 but window > 176 tokens
    dict(H=36, W=72, C=384, heads=2, window=(12, 24), shift=(6, 12)),     # d = 192, 288 tokens (refused in round 1)
    dict(H=36, W=72, C=256, heads=2, window=(6, 12), shift=(3, 6)),       # d = 128
    dict(H=36, W=72, C=128, heads=2, window=(12, 24), shift=(6, 12), bias=False),   # no CPB table: bounded-logit single pass + mask
    dict(H=36, W=72, C=192, heads=4, window=(18, 36), shift=(0, 0), bias=False),    # d = 48, plain
    dict(H=36, W=72, C=128, heads=2, window=(9, 18), shift=(4, 9), bias=False, big_scale=True),   # scale 100: exact-max pass
])
def test_window_attention_geometry_sweep(cfg):
    """BASELINE config 5: other window sizes / head counts run on the tiled tcgen05 kernels (csrc/attn_tc_gen.cu)."""
    B, H, W, C, heads, window, shift = 2, cfg["H"], cfg["W"], cfg["C"], cfg["heads"], cfg["window"], cfg["shift"]
    L, T = window[0] * window[1], B * H * W
    raw = gen(T, 3 * C, seed=70).to(torch.bfloat16)
    scale = torch.linspace(9.0, 12.0, heads, device=DEV)
    if cfg.get("big_scale"):
        scale = torch.full((heads,), 100.0, device=DEV)
    bias = 0.5 * gen(heads, L, L, seed=71) if cfg.get("bias", True) else None
    raw_f = raw.float().requires_grad_(True)
    sc_f = scale.clone().requires_grad_(True)
    b_f = bias.clone().requires_grad_(True) if bias is not None else None
    o_ref, lse_ref = oracle_attention(raw_f, sc_f, b_f, B, H, W, C, heads, window, shift)
    qkv = raw.clone()
    inv = ops.qk_normalize_(qkv, C, heads)
    assert ops.attn_backend_for(ops.MODE_BF16, C, heads, *window) == BACKEND_TCGEN05
    o, lse = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1], ops.MODE_BF16)
    assert rel(o, o_ref) < 1e-2
    assert rel(lse[0].reshape(-1), lse_ref.reshape(-1)) < 1e-2
    d_o = gen(T, C, seed=72).to(torch.bfloat16)
    o_ref.backward(d_o.float())
    dqkv, dscale, dbias = ops.window_attn_bwd(qkv, inv, scale, bias, o, d_o, lse, B, H, W, C, heads, window[0], window[1],
                                              shift[0], shift[1], ops.MODE_BF16)
    for name, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        assert rel(dqkv[:, sl], raw_f.grad[:, sl]) < 2e-2, name
    if not cfg.get("big_scale"):     # at scale 100 the bf16 rounding of q^ / k^ alone moves single logits by ~0.4
        err_tok = (dqkv.float() - raw_f.grad).norm(dim=1) / raw_f.grad.norm(dim=1).clamp_min(1e-20)
        assert float(err_tok.max()) < 1e-1, float(err_tok.max())
    assert rel(dscale, sc_f.grad) < 6e-2
    if bias is not None:
        assert rel(dbias, b_f.grad) < 2e-2


def test_window_attention_unsupported_geometry_is_a_clean_error():
    """A head_dim the tcgen05 kernels are not instantiated for (80) is refused before any launch, with a message -- never a
    silent wrong answer or a CPU fallback; the shape dispatch sends it to the CUDA-core kernels instead."""
    B, H, W, C, heads, window = 1, 36, 72, 160, 2, (12, 24)
    qkv = gen(B * H * W, 3 * C, seed=80).to(torch.bfloat16)
    ops.qk_normalize_(qkv, C, heads)
    assert ops.attn_backend_for(ops.MODE_BF16, C, heads, *window) == BACKEND_SIMT
    with pytest.raises(Exception, match="not instantiated"):
        ops.window_attn_fwd(qkv, torch.ones(heads, device=DEV), None, B, H, W, C, heads, window[0], window[1], 0, 0,
                            ops.MODE_BF16, backend=BACKEND_TCGEN05)


# ---- loss ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("relative", [True, False])
@pytest.mark.parametrize("squared", [True, False])
def test_latw_l2(relative, squared):
    B, C, H, W = 2, 5, 72, 144
    prd = gen(B, C, H, W, seed=30).requires_grad_(True)
    tar = gen(B, C, H, W, seed=31)
    chw = torch.rand(C, generator=torch.Generator().manual_seed(32)).to(DEV)
    qw = O.quadrature_row_weights(H, W).to(DEV)
    loss, num, den = ops.latw_l2_fwd(prd.detach(), tar, qw, chw, relative, squared)
    want = O.geometric_l2(prd, tar, chw, relative, squared)
    assert abs(float(loss) - float(want)) / abs(float(want)) < 1e-5
    g = torch.tensor([0.7], device=DEV)
    dprd = ops.latw_l2_bwd(prd.detach(), tar, qw, chw, num, den, g, relative, squared)
    (want * 0.7).backward()
    assert rel(dprd, prd.grad) < 1e-5


# ---- GEMM ------------------------------------------------------------------------------------------------------
def gemm_reference(A, a_major, Bm, b_major, epi, bias, aux, dtype):
    Af = A.float() if a_major == 0 else A.float().t()
    Bf = Bm.float() if b_major == 0 else Bm.float().t()
    acc = (Af.double() @ Bf.double().t()).float()
    rnd = (lambda t: t.to(dtype).float())
    if epi == EPI_BIAS:
        return acc + (bias if bias is not None else 0)
    if epi == EPI_BIAS_GELU:
        h = acc + bias
        return torch.nn.functional.gelu(rnd(h)), h
    if epi == EPI_DGELU:
        h = aux.float().requires_grad_(True)
        torch.nn.functional.gelu(h).sum().backward()
        return acc * h.grad
    if epi == EPI_ADD_F32:
        return acc + aux
    return acc


GEMM_CASES = [
    # (M, N, K, a_major, b_major, epilogue)
    (300, 192, 96, 0, 0, EPI_BIAS),
    (1000, 2304, 768, 0, 0, EPI_BIAS),
    (777, 3072, 768, 0, 0, EPI_BIAS_GELU),
    (640, 768, 1168, 0, 0, EPI_BIAS),       # patch-embed shape: K tail
    (650, 1168, 768, 0, 0, EPI_BIAS),       # head shape: N tail
    (515, 768, 3072, 0, 1, EPI_DGELU),
    (515, 768, 2304, 0, 1, EPI_ADD_F32),
    (515, 768, 768, 0, 1, EPI_BIAS),
    (515, 768, 1168, 0, 1, EPI_F32),
    (768, 3072, 1000, 1, 1, EPI_F32),       # wgrad, K tail
    (2304, 768, 1300, 1, 1, EPI_F32),
    (1168, 768, 648, 1, 1, EPI_F32),        # head wgrad: M tail
    # N <= 128: single-CTA 128 x 128 tiles instead of CTA pairs, one row per instantiation, N tails included
    (300, 128, 768, 0, 0, EPI_BIAS),
    (333, 72, 520, 0, 0, EPI_BIAS_GELU),
    (300, 120, 768, 0, 0, EPI_F32),
    (515, 72, 768, 0, 1, EPI_BIAS),
    (515, 128, 3072, 0, 1, EPI_DGELU),
    (515, 96, 2304, 0, 1, EPI_ADD_F32),
    (515, 72, 1168, 0, 1, EPI_F32),
    (768, 72, 1000, 1, 1, EPI_F32),         # wgrad, N tail
]


def run_gemm_case(case, dtype, backend, split_k=1):
    M, N, K, a_major, b_major, epi = case
    mode = mode_for(dtype)
    A = gen(*((M, K) if a_major == 0 else (K, M)), seed=40, scale=0.5).to(dtype)
    Bm = gen(*((N, K) if b_major == 0 else (K, N)), seed=41, scale=0.5).to(dtype)
    bias = gen(N, seed=42) if epi in (EPI_BIAS, EPI_BIAS_GELU) else None
    aux = None
    if epi == EPI_DGELU:
        aux = gen(M, N, seed=43).to(dtype)
    elif epi == EPI_ADD_F32:
        aux = gen(M, N, seed=43)
    kw = {}
    if epi == EPI_F32 and split_k > 1:
        kw = dict(out=torch.zeros(M, N, device=DEV), accumulate=True, split_k=split_k)
    got = ops.gemm(mode, A, a_major, Bm, b_major, epi, bias=bias, aux=aux, backend=backend, **kw)
    want = gemm_reference(A, a_major, Bm, b_major, epi, bias, aux, dtype)
    tol = 1e-5 if dtype == torch.float32 else 6e-3
    if epi == EPI_BIAS_GELU:
        assert rel(got[0], want[0]) < tol and rel(got[1], want[1]) < tol
    else:
        assert rel(got, want) < (1e-5 if epi in (EPI_ADD_F32, EPI_F32) else tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("case", GEMM_CASES)
def test_gemm_simt(case, dtype):
    run_gemm_case(case, dtype, BACKEND_SIMT)


@pytest.mark.parametrize("case", GEMM_CASES)
def test_gemm_tcgen05(case):
    run_gemm_case(case, torch.bfloat16, BACKEND_TCGEN05)


@pytest.mark.parametrize("T,C,heads", [(700, 768, 8), (333, 192, 2), (260, 96, 1), (129, 288, 3)])
def test_gemm_tcgen05_qkv_projection_fused_normalise(T, C, heads):
    x = gen(T, C, seed=50, scale=0.5).to(torch.bfloat16)
    w = gen(3 * C, C, seed=51, scale=0.05).to(torch.bfloat16)
    b = gen(3 * C, seed=52)
    qkv, inv = ops.qkv_projection(ops.MODE_BF16, x, w, b, C, heads)
    d = C // heads
    ref = (x.float().double() @ w.float().double().t() + b.double()).float().view(T, 3, heads, d)
    nrm = ref[:, :2].norm(dim=-1, keepdim=True).clamp_min(1e-12)
    want = ref.clone()
    want[:, :2] = ref[:, :2] / nrm
    assert rel(qkv.view(T, 3, heads, d), want) < 4e-3          # bf16 storage of unit vectors / v
    assert rel(inv, 1.0 / nrm.squeeze(-1)) < 1e-5
    # and it agrees with the unfused path (GEMM + stand-alone normalisation kernel)
    qkv2, inv2 = ops.qkv_projection(ops.MODE_BF16_SIMT, x, w, b, C, heads)
    assert rel(qkv, qkv2) < 6e-3 and rel(inv, inv2) < 3e-3


@pytest.mark.parametrize("name", ["fc1_gelu", "fc2", "dgelu", "qkv_dgrad", "fc1_wgrad"])
def test_gemm_tcgen05_model_shapes(name):
    """The model's own shapes (T = 64,800 tokens): 3,042 output tiles per launch, i.e. ~40 tiles per resident CTA pair
    obtained through cluster-launch-control work stealing.  Reference: fp32 matmul of the same bf16 values."""
    T, C, HID = 64800, 768, 3072
    mode = ops.MODE_BF16
    f32mm = lambda a, b: a.float() @ b.float()
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        if name == "fc1_gelu":
            x, w, b = gen(T, C, seed=90, scale=0.5).bfloat16(), gen(HID, C, seed=91, scale=0.05).bfloat16(), gen(HID, seed=92)
            g, h = ops.gemm(mode, x, 0, w, 0, EPI_BIAS_GELU, bias=b)
            h_ref = f32mm(x, w.t()) + b
            assert rel(h, h_ref) < 6e-3
            assert rel(g, torch.nn.functional.gelu(h.float())) < 6e-3      # GELU of the stored pre-activation
        elif name == "fc2":
            x, w, b = gen(T, HID, seed=93, scale=0.5).bfloat16(), gen(C, HID, seed=94, scale=0.05).bfloat16(), gen(C, seed=95)
            assert rel(ops.gemm(mode, x, 0, w, 0, EPI_BIAS, bias=b), f32mm(x, w.t()) + b) < 6e-3
        elif name == "dgelu":
            dz, w, h = gen(T, C, seed=96, scale=0.5).bfloat16(), gen(C, HID, seed=97, scale=0.05).bfloat16(), gen(T, HID, seed=98).bfloat16()
            hf = h.float().requires_grad_(True)
            torch.nn.functional.gelu(hf).backward(f32mm(dz, w))
            assert rel(ops.gemm(mode, dz, 0, w, 1, EPI_DGELU, aux=h), hf.grad) < 6e-3
        elif name == "qkv_dgrad":
            dy, w, r = gen(T, 3 * C, seed=99, scale=0.5).bfloat16(), gen(3 * C, C, seed=100, scale=0.05).bfloat16(), gen(T, C, seed=101)
            assert rel(ops.gemm(mode, dy, 0, w, 1, EPI_ADD_F32, aux=r), f32mm(dy, w) + r) < 1e-5
        else:
            dy, x = gen(T, HID, seed=102, scale=0.5).bfloat16(), gen(T, C, seed=103, scale=0.5).bfloat16()
            dw = torch.zeros(HID, C, device=DEV)
            ops.gemm(mode, dy, 1, x, 1, EPI_F32, out=dw, accumulate=True, split_k=ops.wgrad_split_k(HID, C, T))
            # 64,800-term fp32 reductions: compare against fp64 on a slice of rows (the fp32 matmul reference carries
            # the same ~eps*sqrt(K) accumulation noise as the kernel) and against fp32 overall
            rows = torch.arange(0, HID, 48, device=DEV)
            ref64 = dy[:, rows].double().t() @ x.double()
            assert rel(dw[rows].double(), ref64) < 2e-5
            assert rel(dw, f32mm(dy.t(), x)) < 5e-5
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("split_k", [2, 5, 16])
def test_gemm_tcgen05_split_k(split_k):
    run_gemm_case((768, 3072, 4000, 1, 1, EPI_F32), torch.bfloat16, BACKEND_TCGEN05, split_k)


def test_gemm_tcgen05_persistent_many_tiles():
    # more tiles than SMs: exercises the TMEM double buffering and the smem ring wrap-around
    run_gemm_case((128 * 40, 2304, 768, 0, 0, EPI_BIAS), torch.bfloat16, BACKEND_TCGEN05)
    run_gemm_case((128 * 40 + 17, 3072, 768, 0, 0, EPI_BIAS_GELU), torch.bfloat16, BACKEND_TCGEN05)
    run_gemm_case((128 * 160 + 17, 96, 768, 0, 0, EPI_BIAS_GELU), torch.bfloat16, BACKEND_TCGEN05)   # single-CTA: 161 row tiles


# ---- optimizer (SURVEY 8(f) rank 1) --------------------------------------------------------------------------
@pytest.mark.parametrize("weight_decay", [0.0, 0.01])
def test_adam_matches_torch_fused(weight_decay):
    """swin_v2_weather_b200.optim.Adam vs torch.optim.Adam(fused=True) as the reference builds it (betas 0.9 / 0.95):
    ten steps on tensors of awkward sizes (chunk tails, one-element, 3 M elements), fp32 tolerance."""
    from swin_v2_weather_b200.optim import Adam
    shapes = [(1,), (7,), (768,), (2304, 768), (65536 + 3,), (3, 1000, 1000), (5, 13)]
    torch.manual_seed(0)
    ref_p = [torch.nn.Parameter(torch.randn(*s, device=DEV)) for s in shapes]
    our_p = [torch.nn.Parameter(p.detach().clone()) for p in ref_p]
    ref = torch.optim.Adam(ref_p, lr=3e-3, betas=(0.9, 0.95), weight_decay=weight_decay, fused=True)
    ours = Adam(our_p, lr=3e-3, betas=(0.9, 0.95), weight_decay=weight_decay, fused=True)
    for it in range(10):
        for a, b in zip(ref_p, our_p):
            g = torch.randn_like(a) * (10.0 ** (it % 3 - 1))
            a.grad, b.grad = g, g.clone()
        ref.step()
        ours.step()
    for a, b in zip(ref_p, our_p):
        assert rel(b, a) < 2e-6
    sd_ref, sd_ours = ref.state_dict(), ours.state_dict()
    assert sd_ref["state"].keys() == sd_ours["state"].keys()
    for k in sd_ref["state"]:
        assert set(sd_ref["state"][k]) == set(sd_ours["state"][k]) == {"step", "exp_avg", "exp_avg_sq"}
        assert float(sd_ref["state"][k]["step"]) == float(sd_ours["state"][k]["step"]) == 10
        assert rel(sd_ours["state"][k]["exp_avg"], sd_ref["state"][k]["exp_avg"]) < 2e-6
        assert rel(sd_ours["state"][k]["exp_avg_sq"], sd_ref["state"][k]["exp_avg_sq"]) < 2e-6
    # a torch Adam state_dict loads into ours and training continues identically
    ours2 = Adam([torch.nn.Parameter(p.detach().clone()) for p in ref_p], lr=3e-3, betas=(0.9, 0.95), weight_decay=weight_decay)
    import copy
    ours2.load_state_dict(copy.deepcopy(sd_ref))      # (load_state_dict aliases same-device tensors of the dict it is given)
    for a, b in zip(ref_p, ours2.param_groups[0]["params"]):
        g = torch.randn_like(a)
        a.grad, b.grad = g, g.clone()
    ref.step()
    ours2.step()
    for a, b in zip(ref_p, ours2.param_groups[0]["params"]):
        assert rel(b, a) < 2e-6


def test_adam_refreshes_bf16_shadows_and_honours_grad_scaler():
    from swin_v2_weather_b200.functional import SHADOWS
    from swin_v2_weather_b200.optim import Adam
    w = torch.nn.Parameter(gen(300, 96, seed=120))
    sh0 = SHADOWS.get(w, ops.MODE_BF16)
    assert torch.equal(sh0.float(), w.detach().bfloat16().float())
    opt = Adam([w], lr=1e-2, betas=(0.9, 0.95))
    w.grad = gen(300, 96, seed=121) * 1024.0                   # scaled gradient, GradScaler style
    opt.grad_scale = torch.tensor(1024.0, device=DEV)
    opt.found_inf = torch.tensor(0.0, device=DEV)
    before, v0 = w.detach().clone(), w._version
    opt.step()
    assert w._version > v0                                      # autograd sees the in-place update
    sh1 = SHADOWS.get(w, ops.MODE_BF16)
    assert sh1.data_ptr() == sh0.data_ptr()                     # same buffer, rewritten by the optimizer pass (no re-cast)
    assert torch.equal(sh1.float(), w.detach().bfloat16().float())
    ref = torch.nn.Parameter(before.clone())
    ropt = torch.optim.Adam([ref], lr=1e-2, betas=(0.9, 0.95), fused=True)
    ref.grad = gen(300, 96, seed=121)
    ropt.step()
    assert rel(w, ref) < 2e-6
    # overflow: the step is skipped on the device
    opt.found_inf = torch.tensor(1.0, device=DEV)
    snap = w.detach().clone()
    opt.step()
    assert torch.equal(w.detach(), snap)
    scaler = torch.amp.GradScaler("cuda", init_scale=256.0)
    loss = (w * gen(300, 96, seed=122)).sum()
    scaler.scale(loss).backward()
    scaler.step(opt)                                            # takes the _step_supports_amp_scaling path
    scaler.update()
    assert not torch.equal(w.detach(), snap)


def test_validation_weighted_rmse_matches_reference_formula():
    """utils/weighted_acc_rmse.py:59-87 restated with plain torch ops (the oracle here) vs the kernel-backed version."""
    from swin_v2_weather_b200.utils.weighted_acc_rmse import weighted_rmse_torch, weighted_rmse_torch_channels
    n, c, h, w = 2, 5, 72, 144
    pred, tar = gen(n, c, h, w, seed=130), gen(n, c, h, w, seed=131)
    lat_t = torch.arange(0, h, device=DEV)
    latv = 90. - lat_t * 180. / float(h - 1)
    s = torch.sum(torch.cos(3.1416 / 180. * latv))
    weight = (h * torch.cos(3.1416 / 180. * latv) / s).reshape(1, 1, -1, 1)
    want = torch.sqrt(torch.mean(weight * (pred - tar) ** 2., dim=(-1, -2)))
    assert rel(weighted_rmse_torch_channels(pred, tar), want) < 1e-6
    assert rel(weighted_rmse_torch(pred, tar), want.mean(0)) < 1e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_patchify_cat_equals_patchify_of_concatenation(dtype):
    mode = mode_for(dtype)
    B, H, W = 3, 24, 40
    parts = [gen(B, 5, H, W, seed=140), gen(B, 1, H, W, seed=141), gen(1, 3, H, W, seed=142)]
    cat = torch.cat([p.expand(B, -1, -1, -1) for p in parts], dim=1).contiguous()
    assert torch.equal(ops.patchify_cat(parts, 4, mode), ops.patchify(cat, 4, 0, mode))
    assert torch.equal(ops.patchify_cat([cat], 4, mode), ops.patchify(cat, 4, 0, mode))

