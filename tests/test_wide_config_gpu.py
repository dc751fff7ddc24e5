"""GPU parity of the widths the e2048 config (swin_73var_geo_depth24_e2048_mlp2_chweight_invar: embed_dim 2048, 8 heads of
256, mlp_ratio 2) adds: window attention at head_dim 256 on the tcgen05 kernels (forward, backward A at 32-row tiles,
backward B split into a dV pass and a dK^ pass) and on the CUDA-core kernels (fp32 validation and bf16_simt modes),
LayerNorm at C = 1280 / 2048, q / k normalisation at head_dim 256, and the whole model against the oracle.

Tolerances are those of tests/test_kernels_gpu.py and tests/test_model_gpu.py: fp32 1e-5 (2e-5 / 5e-5 for attention
outputs / gradients, 5e-5 for ill-conditioned model gradients), bf16 1e-2 (2e-2 for attention gradients, 6e-2 for
d(scale) at a few windows, 5e-2 for logit_scale / meta_mlp model gradients).
"""

import pytest
import torch

from oracle import swinv2_oracle as O
from swin_v2_weather_b200 import ops
from swin_v2_weather_b200._lib import BACKEND_SIMT, BACKEND_TCGEN05
from swin_v2_weather_b200.functional import LatWeightedL2Fn
from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    return O.rel_l2(a.float(), b.float())


def gen(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def oracle_attention(qkv_raw, scale, bias, B, H, W, C, heads, window, shift):
    """q/k/v (T, 3C) fp32 raw -> (o (T, C), lse) with the oracle's index arithmetic (as in test_kernels_gpu.py)."""
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


def attention_case(B, H, W, C, heads, window, shift, with_bias, scale, mode, backend, seed=20):
    """Ours (forward + backward through ops) and the fp32 autograd oracle on the same stored values."""
    L, T = window[0] * window[1], B * H * W
    raw = gen(T, 3 * C, seed=seed).to(mode.act_dtype)
    bias = (0.5 * gen(heads, L, L, seed=seed + 1)) if with_bias else None
    raw_f = raw.float().requires_grad_(True)
    sc_f = scale.clone().requires_grad_(True)
    b_f = bias.clone().requires_grad_(True) if bias is not None else None
    o_ref, lse_ref = oracle_attention(raw_f, sc_f, b_f, B, H, W, C, heads, window, shift)
    qkv = raw.clone()
    inv = ops.qk_normalize_(qkv, C, heads)
    o, lse = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, window[0], window[1], shift[0], shift[1], mode,
                                 backend=backend)
    d_o = gen(T, C, seed=seed + 2).to(mode.act_dtype)
    o_ref.backward(d_o.float())
    dqkv, dscale, dbias = ops.window_attn_bwd(qkv, inv, scale, bias, o, d_o, lse, B, H, W, C, heads, window[0], window[1],
                                              shift[0], shift[1], mode, backend=backend)
    return dict(o=o, lse=lse, dqkv=dqkv, dscale=dscale, dbias=dbias), dict(o=o_ref, lse=lse_ref, dqkv=raw_f.grad,
                                                                           dscale=sc_f.grad, dbias=None if b_f is None else b_f.grad)


def check_attention(got, want, C, tol_o, tol_g, tol_scale, tol_tok):
    assert rel(got["o"], want["o"]) < tol_o
    assert rel(got["lse"][0].reshape(-1), want["lse"].reshape(-1)) < tol_o
    for name, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        e = rel(got["dqkv"][:, sl], want["dqkv"][:, sl])
        assert e < tol_g, (name, e)
    if tol_tok is not None:       # a single window gone wrong is invisible in a whole-tensor norm
        g, r = got["dqkv"].float(), want["dqkv"]
        err_tok = (g - r).norm(dim=1) / r.norm(dim=1).clamp_min(1e-20)
        assert float(err_tok.max()) < tol_tok, float(err_tok.max())
    assert rel(got["dscale"], want["dscale"]) < tol_scale, (got["dscale"], want["dscale"])
    if want["dbias"] is not None:
        assert rel(got["dbias"], want["dbias"]) < tol_g


# windows 9x18 (L = 162: two stationary tiles, ragged 32- and 64-row streamed tiles), 6x12 (L = 72) and 12x24 (L = 288: three
# stationary tiles, nine 32-row streamed tiles) on a 36 x 72 grid (16 / 36 / 9 windows per sample, as in the geometry sweep of
# test_kernels_gpu.py: d(scale) is a cancelling sum whose bf16 noise only averages down over windows); head_dim 256 at two
# heads (C = 512)
CASES = [
    dict(window=(9, 18), shift=(0, 0), bias=False),
    dict(window=(9, 18), shift=(4, 9), bias=False),
    dict(window=(9, 18), shift=(4, 9), bias=True),
    dict(window=(9, 18), shift=(0, 0), bias=True),
    dict(window=(6, 12), shift=(3, 6), bias=True),
    dict(window=(6, 12), shift=(0, 0), bias=False),
    dict(window=(12, 24), shift=(6, 12), bias=True),
    dict(window=(12, 24), shift=(0, 0), bias=False),
    dict(window=(9, 18), shift=(4, 9), bias=False, big_scale=True),     # scale 100: the exact-max softmax path of tcgen05
]
GRID = (36, 72)


def case_id(c):
    return f"{c['window'][0]}x{c['window'][1]}-s{c['shift'][0]}-{'bias' if c['bias'] else 'nobias'}" + ("-scale100" if c.get("big_scale") else "")


def case_scale(c, heads):
    return torch.full((heads,), 100.0, device=DEV) if c.get("big_scale") else torch.linspace(9.0, 12.0, heads, device=DEV)


@pytest.mark.parametrize("cfg", CASES, ids=case_id)
def test_attention_head_dim_256_tcgen05(cfg):
    B, C, heads = 2, 512, 2
    assert ops.attn_backend_for(ops.MODE_BF16, C, heads, *cfg["window"]) == BACKEND_TCGEN05
    got, want = attention_case(B, *GRID, C, heads, cfg["window"], cfg["shift"], cfg["bias"], case_scale(cfg, heads),
                               ops.MODE_BF16, BACKEND_TCGEN05)
    # the tiled tcgen05 forward writes the softmax-weighted mean cosine into the second plane; the CUDA-core one zeroes it
    assert float(got["lse"][1].abs().max()) > 0, "the tcgen05 kernels did not run"
    check_attention(got, want, C, 1e-2, 2e-2, 6e-2, None if cfg.get("big_scale") else 1e-1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("cfg", [c for c in CASES if not c.get("big_scale")], ids=case_id)
def test_attention_head_dim_256_cuda_cores(cfg, dtype):
    """fp32: the K / V tiles of a window (333 KB at 9x18) exceed shared memory, the kernels read them from L2; bf16 fits
    (192 KB) up to 9x18 and reads from L2 at 12x24.  (These kernels always take the exact row maximum: the scale-100 case
    exercises a tcgen05 path only.)"""
    B, C, heads = 2, 512, 2
    mode = ops.MODE_FP32 if dtype == torch.float32 else ops.MODE_BF16_SIMT
    got, want = attention_case(B, *GRID, C, heads, cfg["window"], cfg["shift"], cfg["bias"], case_scale(cfg, heads),
                               mode, BACKEND_SIMT)
    if dtype == torch.float32:
        check_attention(got, want, C, 2e-5, 5e-5, 5e-5, None)
    else:
        check_attention(got, want, C, 1e-2, 2e-2, 6e-2, None)


def test_attention_head_dim_256_full_geometry():
    """73 x 720 x 1440 / 4 = 180 x 360 tokens, C = 2048, 8 heads of 256, shifted 9x18 windows with a bias table: 3,200
    (window, head) items per pass, wrap-around windows mixed in, d(scale) / d(bias) partials from every item."""
    B, H, W, C, heads, window, shift = 1, 180, 360, 2048, 8, (9, 18), (4, 9)
    assert ops.attn_backend_for(ops.MODE_BF16, C, heads, *window) == BACKEND_TCGEN05
    got, want = attention_case(B, H, W, C, heads, window, shift, True, torch.linspace(8.0, 14.0, heads, device=DEV),
                               ops.MODE_BF16, BACKEND_TCGEN05, seed=60)
    assert float(got["lse"][1].abs().max()) > 0
    check_attention(got, want, C, 1e-2, 2e-2, 3e-2, 8e-2)


# ---- LayerNorm / q,k normalisation at the new widths -------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("C", [1280, 2048])
def test_ln_residual_fwd_bwd_wide(dtype, C):
    mode = ops.MODE_FP32 if dtype == torch.float32 else ops.MODE_BF16_SIMT
    tol = 1e-5 if dtype == torch.float32 else 1e-2
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
        assert rel(dz, zf.grad) < tol
        assert rel(dg, gf.grad) < 1e-5 and rel(db, bf.grad) < 1e-5
        assert rel(dbp, zf.grad.sum(0)) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("heads,C", [(8, 2048), (2, 512)])
def test_qk_normalize_head_dim_256(dtype, heads, C):
    T = 500
    qkv0 = gen(T, 3 * C, seed=13).to(dtype)
    qkv = qkv0.clone()
    inv = ops.qk_normalize_(qkv, C, heads)
    d = C // heads
    ref = qkv0.float().view(T, 3, heads, d)
    nrm = ref[:, :2].norm(dim=-1, keepdim=True).clamp_min(1e-12)
    assert rel(qkv.view(T, 3, heads, d)[:, :2], ref[:, :2] / nrm) < (1e-6 if dtype == torch.float32 else 4e-3)
    assert torch.equal(qkv.view(T, 3, heads, d)[:, 2], qkv0.view(T, 3, heads, d)[:, 2])
    assert rel(inv, 1.0 / nrm.squeeze(-1)) < 1e-6


# ---- the model --------------------------------------------------------------------------------------------------------------
def wide_cfg(**kw):
    base = dict(img_size=(72, 144), depth=2, num_heads=8, in_chans=7, out_chans=5, embed_dim=2048, window_ratio=8, mlp_ratio=2.0,
                rel_pos=False)
    base.update(kw)
    return O.SwinConfig(**base)


def build(cfg: O.SwinConfig, sd, mode: str, **kw):
    m = SwinTransformerV2Cr(img_size=cfg.img_size, patch_size=cfg.patch_size, depths=(cfg.depth,), num_heads=(cfg.num_heads,),
                            in_chans=cfg.in_chans, out_chans=cfg.out_chans, embed_dim=cfg.embed_dim,
                            img_window_ratio=cfg.window_ratio, drop_path_rate=cfg.drop_path_rate,
                            full_pos_embed=cfg.full_pos_embed, rel_pos=cfg.rel_pos, mlp_ratio=cfg.mlp_ratio,
                            residual=cfg.residual, compute_mode=mode, **kw)
    m.load_state_dict(sd)
    return m.cuda().eval()


def inputs(cfg, batch, seed=1234):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, cfg.in_chans, *cfg.img_size, generator=g)
    tar = torch.randn(batch, cfg.out_chans, *cfg.img_size, generator=g)
    chw = torch.rand(cfg.out_chans, generator=g) + 0.5
    return x, tar, chw / chw.sum()


def run_ours(model, x, tar, chw, relative=True):
    qw = O.quadrature_row_weights(*x.shape[-2:]).to(DEV)
    model.zero_grad(set_to_none=True)
    pred = model(x.to(DEV))
    loss = LatWeightedL2Fn.apply(pred, tar.to(DEV), qw, chw.to(DEV), relative, True)
    loss.backward()
    torch.cuda.synchronize()
    return pred.detach().cpu(), float(loss), {k: p.grad.detach().cpu() for k, p in model.named_parameters()}


def model_errors(ours, ref):
    pred, loss, grads = ours
    pred_ref, loss_ref, grads_ref = ref
    rep = {"pred": O.rel_l2(pred, pred_ref), "loss": abs(loss - float(loss_ref)) / abs(float(loss_ref))}
    big = max(float(v.abs().max()) for v in grads_ref.values())
    for k, g_ref in grads_ref.items():
        if k.endswith("meta_mlp.fc2.bias"):      # analytically zero (softmax shift invariance): absolute check
            rep[k] = 0.0 if float(grads[k].abs().max()) <= 1e-3 * max(1.0, big) else float("inf")
            continue
        rep[k] = O.rel_l2(grads[k], g_ref.cpu())
    return rep


def assert_model(rep, tol, tol_scale):
    bad = [(k, v) for k, v in rep.items() if not v < (tol_scale if ("logit_scale" in k or "meta_mlp" in k) else tol)]
    assert not bad, sorted(bad, key=lambda t: -t[1])[:8]


@pytest.mark.parametrize("rel_pos", [False, True])
@pytest.mark.parametrize("mode", ["fp32", "bf16_simt", "bf16"])
def test_wide_model_parity_vs_oracle(mode, rel_pos):
    """72 x 144, depth 2, C = 2048, 8 heads of 256, mlp_ratio 2: output, loss and every parameter gradient."""
    cfg = wide_cfg(rel_pos=rel_pos)
    sd = O.init_state_dict(cfg, seed=3)
    x, tar, chw = inputs(cfg, 2)
    ref = O.loss_and_grads(x, tar, sd, cfg, chw, relative=True)
    ours = run_ours(build(cfg, sd, mode), x, tar, chw)
    tol, tol_scale = (1e-5, 5e-5) if mode == "fp32" else (1e-2, 5e-2)
    assert_model(model_errors(ours, ref), tol, tol_scale)


def test_wide_model_channel_groups_with_residual():
    """77 input channels as [field 73 | zenith 1 | static 3, shared by the batch] with the residual skip: identical to the
    concatenated input (same im2col values), in bf16 at the wide width."""
    B, H, W = 2, 72, 144
    model = SwinTransformerV2Cr(img_size=(H, W), patch_size=4, depths=(2,), num_heads=(8,), in_chans=77, out_chans=73,
                                embed_dim=2048, img_window_ratio=8, mlp_ratio=2.0, full_pos_embed=True, rel_pos=True,
                                residual=True, compute_mode="bf16").cuda().eval()
    g = torch.Generator().manual_seed(7)
    field, zen = torch.randn(B, 73, H, W, generator=g).to(DEV), torch.rand(B, 1, H, W, generator=g).to(DEV)
    static = torch.randn(1, 3, H, W, generator=g).to(DEV)
    cat = torch.cat([field, zen, static.expand(B, -1, -1, -1)], dim=1)

    def run(inp):
        model.zero_grad(set_to_none=True)
        out = model(inp)
        out.square().mean().backward()
        return out.detach(), {k: p.grad.detach().clone() for k, p in model.named_parameters()}

    o1, g1 = run([field, zen, static])
    o2, g2 = run(cat)
    assert torch.equal(o1, o2)
    for k in g1:
        assert O.rel_l2(g1[k].cpu(), g2[k].cpu()) < 1e-5, k


def test_wide_model_checkpoint_stages_equal_gradients():
    cfg = wide_cfg(rel_pos=True)
    sd = O.init_state_dict(cfg, seed=4)
    x, tar, chw = inputs(cfg, 2)
    outs = [run_ours(build(cfg, sd, "bf16", checkpoint_stages=ckpt), x, tar, chw) for ckpt in (False, True)]
    assert O.rel_l2(outs[1][0], outs[0][0]) < 1e-6
    assert abs(outs[0][1] - outs[1][1]) <= 1e-6 * abs(outs[0][1])
    for k in outs[0][2]:
        assert O.rel_l2(outs[1][2][k], outs[0][2][k]) < 5e-3, k     # fp32-atomic order can flip individual bf16 roundings


GEMM_WEIGHTS = ("attn.qkv.weight", "attn.proj.weight", "mlp.fc1.weight", "mlp.fc2.weight", "head.weight", "patch_embed.proj.weight")
NOISY = ("logit_scale", "meta_mlp")


def test_wide_full_resolution_vs_oracle():
    """73 x 720 x 1440 (64,800 tokens, 400 windows), depth 1, C = 2048, 8 heads of 256, bf16, against the fp32 oracle run
    on the GPU with TF32 off.  Bars as in test_parity_headline_gpu.py::test_full_resolution_vs_oracle: <= 1e-2 on the
    output and every gradient against the oracle at the bf16-rounded GEMM weights the tensor cores read and against the
    oracle at the fp32 weights; logit_scale gets the nearer of the two, and never more than 1.25x the distance rounding
    the weights alone puts between the oracles."""
    cfg = O.SwinConfig(depth=1, embed_dim=2048, num_heads=8, mlp_ratio=2.0, rel_pos=False)
    sd = O.init_state_dict(cfg, seed=2)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(1, cfg.in_chans, *cfg.img_size, generator=g)
    tar = torch.randn(1, cfg.out_chans, *cfg.img_size, generator=g)
    chw = torch.ones(73) / 73
    ours = run_ours(build(cfg, sd, "bf16"), x, tar, chw)
    torch.cuda.empty_cache()
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        refs = []
        for s in (sd, {k: (v.bfloat16().float() if k.endswith(GEMM_WEIGHTS) else v) for k, v in sd.items()}):
            p, l, gr = O.loss_and_grads(x.to(DEV), tar.to(DEV), {k: v.to(DEV) for k, v in s.items()}, cfg, chw.to(DEV))
            refs.append((p.cpu(), l.cpu(), {k: v.cpu() for k, v in gr.items()}))
            del p, l, gr
            torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    rep_ii, rep_i = model_errors(ours, refs[0]), model_errors(ours, refs[1])
    floor = max(O.rel_l2(refs[1][2][k], refs[0][2][k]) for k in refs[0][2] if any(t in k for t in NOISY))
    print("full-res e2048 worst (i):", sorted(((v, k) for k, v in rep_i.items()), reverse=True)[:4], "floor", floor)
    assert_model({k: v for k, v in rep_i.items() if not any(t in k for t in NOISY)}, 1e-2, 1e-2)
    assert_model({k: v for k, v in rep_ii.items() if not any(t in k for t in NOISY)}, 1e-2, 1e-2)
    assert_model({k: min(rep_i[k], rep_ii[k]) for k in rep_i if any(t in k for t in NOISY)}, 1e-2, 1e-2)
    assert_model({k: v for k, v in rep_ii.items() if any(t in k for t in NOISY)}, 1e-2, max(1e-2, 1.25 * floor))
