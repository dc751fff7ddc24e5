"""GPU: the forward-only path (no gradient will be taken) gives the same bits as the training forward, at the kernel level
and for the whole model, and does not hold the fc1 pre-activation."""
from types import SimpleNamespace

import pytest
import torch

from swin_v2_weather_b200 import ops
from swin_v2_weather_b200.networks import swinv2_global as SG
from swin_v2_weather_b200.networks.helpers import MultiStepWrapper
from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr, SwinTransformerV2CrBlock
from swin_v2_weather_b200.ops import EPI_BIAS_GELU, EPI_BIAS_GELU_FWD, MODES

pytestmark = pytest.mark.gpu
DEV = "cuda"


def both_paths(fn, *args):
    """fn(*args) on the training path (grad enabled, graph dropped) and under no_grad, from the same RNG state (CPB dropout
    and DropPath draw when the module is in training mode); outputs detached."""
    torch.manual_seed(11)
    with torch.enable_grad():
        ref = fn(*args)
        ref = tuple(t.detach() for t in ref) if isinstance(ref, tuple) else ref.detach()
    torch.manual_seed(11)
    with torch.no_grad():
        out = fn(*args)
    return ref, out


# ---- epilogue level ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [300, 64800, 129600])
@pytest.mark.parametrize("N", [3072, 4096, 512])
def test_bias_gelu_fwd_equals_bias_gelu(M, N):
    g = torch.Generator(device=DEV).manual_seed(M + N)
    K = 768 if N != 4096 else 2048
    a = torch.randn(M, K, device=DEV, generator=g).bfloat16()
    w = (torch.randn(N, K, device=DEV, generator=g) * K ** -0.5).bfloat16()
    b = torch.randn(N, device=DEV, generator=g)
    for mode in ("bf16", "bf16_simt"):
        if mode == "bf16_simt" and M > 300:
            continue
        m = MODES[mode]
        act, _ = ops.gemm(m, a, 0, w, 0, EPI_BIAS_GELU, bias=b)
        fwd = ops.gemm(m, a, 0, w, 0, EPI_BIAS_GELU_FWD, bias=b)
        assert torch.equal(act, fwd), (mode, M, N)
    m = MODES["fp32"]
    act, _ = ops.gemm(m, a[:300].float(), 0, w.float(), 0, EPI_BIAS_GELU, bias=b)
    assert torch.equal(act, ops.gemm(m, a[:300].float(), 0, w.float(), 0, EPI_BIAS_GELU_FWD, bias=b))


@pytest.mark.parametrize("N", [128, 64])
def test_bias_gelu_fwd_bn128(N):
    """N <= 128 runs the single-CTA BN 128 kernel (small test widths)."""
    g = torch.Generator(device=DEV).manual_seed(N)
    a = torch.randn(1000, 192, device=DEV, generator=g).bfloat16()
    w = torch.randn(N, 192, device=DEV, generator=g).bfloat16()
    b = torch.randn(N, device=DEV, generator=g)
    act, _ = ops.gemm(MODES["bf16"], a, 0, w, 0, EPI_BIAS_GELU, bias=b)
    assert torch.equal(act, ops.gemm(MODES["bf16"], a, 0, w, 0, EPI_BIAS_GELU_FWD, bias=b))


@pytest.mark.parametrize("mode", ["bf16", "bf16_simt", "fp32"])
@pytest.mark.parametrize("C,heads,H,W,shift,cpb", [(768, 8, 36, 72, (4, 9), False), (768, 8, 36, 72, (0, 0), True),
                                                    (512, 2, 18, 36, (4, 9), False), (2048, 8, 18, 36, (4, 9), True)])
def test_null_statistics_launches(mode, C, heads, H, W, shift, cpb):
    """qkv projection (GEMM epilogue or stand-alone normalisation), attention and LayerNorm: same outputs with NULL statistics."""
    if mode == "fp32" and C == 2048:
        pytest.skip("the fp32 validation mode is not run at embed_dim 2048")
    m = MODES[mode]
    g = torch.Generator(device=DEV).manual_seed(C + H)
    B, T = 2, 2 * H * W
    xb = torch.randn(T, C, device=DEV, generator=g).to(m.act_dtype)
    w = (torch.randn(3 * C, C, device=DEV, generator=g) * C ** -0.5).to(m.act_dtype)
    bq = torch.randn(3 * C, device=DEV, generator=g)
    qkv1, inv = ops.qkv_projection(m, xb, w, bq, C, heads)
    qkv2, none = ops.qkv_projection(m, xb, w, bq, C, heads, need_stats=False)
    assert none is None and inv is not None and torch.equal(qkv1, qkv2)
    scale = torch.rand(heads, device=DEV, generator=g) * 10 + 1
    L = 9 * 18
    bias = torch.randn(heads, L, L, device=DEV, generator=g) if cpb else None
    o1, lse = ops.window_attn_fwd(qkv1, scale, bias, B, H, W, C, heads, 9, 18, *shift, m)
    o2, none = ops.window_attn_fwd(qkv1, scale, bias, B, H, W, C, heads, 9, 18, *shift, m, need_stats=False)
    assert none is None and torch.equal(o1, o2)
    z = torch.randn(T, C, device=DEV, generator=g).to(m.act_dtype)
    x_in = torch.randn(T, C, device=DEV, generator=g)
    gam, bet = torch.randn(C, device=DEV, generator=g), torch.randn(C, device=DEV, generator=g)
    ss = torch.rand(B, device=DEV, generator=g)
    r1 = ops.ln_residual_fwd(z, x_in, gam, bet, ss, None, H * W, m)
    r2 = ops.ln_residual_fwd(z, x_in, gam, bet, ss, None, H * W, m, need_stats=False)
    assert r2[2] is None and torch.equal(r1[0], r2[0]) and torch.equal(r1[1], r2[1])


# ---- model level --------------------------------------------------------------------------------------------------
def small_model(mode, rel_pos, depth=2, drop_path=0.0, img=(72, 144), C=192, heads=2, in_chans=9):
    torch.manual_seed(0)
    m = SwinTransformerV2Cr(img_size=img, patch_size=4, depths=(depth,), num_heads=(heads,), in_chans=in_chans, out_chans=5,
                            embed_dim=C, img_window_ratio=8, drop_path_rate=drop_path, full_pos_embed=True, rel_pos=rel_pos,
                            residual=True, compute_mode=mode).to(DEV)
    with torch.no_grad():       # non-identity blocks (the reference zero-inits norm1/2.weight)
        for blk in m.stages[0].blocks:
            blk.norm1.weight.fill_(0.7)
            blk.norm2.weight.fill_(1.3)
    return m


@pytest.mark.parametrize("mode", ["bf16", "bf16_simt", "fp32"])
@pytest.mark.parametrize("rel_pos", [False, True], ids=["nopos", "cpb"])
@pytest.mark.parametrize("train", [False, True], ids=["eval", "train_droppath"])
def test_model_bitwise(mode, rel_pos, train):
    model = small_model(mode, rel_pos, drop_path=0.3 if train else 0.0)
    model.train(train)
    g = torch.Generator().manual_seed(3)
    B = 3
    groups = [torch.randn(B, 5, 72, 144, generator=g).to(DEV), torch.rand(B, 1, 72, 144, generator=g).to(DEV),
              torch.randn(1, 3, 72, 144, generator=g).to(DEV)]
    stats = (torch.rand(5, generator=g), torch.rand(5, generator=g) + 0.5)

    def run(*inp):
        torch.manual_seed(11)                        # CPB dropout and DropPath draws
        return model(list(inp), input_stats=stats)

    ref, out = both_paths(run, *groups)
    assert torch.equal(ref, out)
    with torch.inference_mode():
        torch.manual_seed(11)
        assert torch.equal(model(groups, input_stats=stats), ref)


def test_full_resolution_bitwise():
    """73 x 720 x 1440, depth 1, the headline widths (embed_dim 768, 8 heads of 96, 9 x 18 windows)."""
    torch.manual_seed(0)
    model = SwinTransformerV2Cr(img_size=(720, 1440), patch_size=4, depths=(1,), num_heads=(8,), in_chans=73, out_chans=73,
                                embed_dim=768, img_window_ratio=80, full_pos_embed=True, rel_pos=False, compute_mode="bf16").to(DEV)
    with torch.no_grad():
        model.stages[0].blocks[0].norm1.weight.fill_(0.7)
        model.stages[0].blocks[0].norm2.weight.fill_(1.3)
    x = torch.randn(1, 73, 720, 1440, generator=torch.Generator().manual_seed(5)).to(DEV)
    ref, out = both_paths(model, x)
    assert torch.equal(ref, out)


def test_e2048_block_bitwise():
    """embed_dim 2048, 8 heads of 256 (the tiled attention kernels), mlp_ratio 2 (hidden 4096), shifted windows + CPB with its
    hidden dropout active (training mode)."""
    torch.manual_seed(0)
    blk = SwinTransformerV2CrBlock(dim=2048, num_heads=8, feat_size=(36, 72), window_size=(9, 18), shift_size=(4, 9),
                                   mlp_ratio=2.0, init_values=1.0, rel_pos=True, compute_mode="bf16").to(DEV)
    x = torch.randn(2, 36, 72, 2048, generator=torch.Generator().manual_seed(5)).to(DEV)
    ref, out = both_paths(blk, x)
    assert torch.equal(ref, out)


def test_rollout_bitwise():
    model = small_model("bf16", True).eval()
    wrap = MultiStepWrapper(SimpleNamespace(n_future=2, add_orography=True, add_landmask=True), lambda p: model)
    g = torch.Generator().manual_seed(9)
    groups = [torch.randn(2, 5, 72, 144, generator=g).to(DEV), torch.rand(2, 1, 72, 144, generator=g).to(DEV),
              torch.randn(1, 3, 72, 144, generator=g).to(DEV)]
    coszen = torch.rand(2, 3, 72, 144, generator=g).to(DEV)
    ref, out = both_paths(wrap, groups, coszen)
    assert out.shape == (2, 15, 72, 144) and torch.equal(ref, out)


def _peak(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():
        out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    return out, peak


def test_peak_memory_drops_by_at_least_one_h(monkeypatch):
    """Depth 2 at full resolution under no_grad: the forward-only path against the training kernels with no graph (what
    no_grad ran before), peak allocation above what was allocated before the call."""
    torch.manual_seed(0)
    model = SwinTransformerV2Cr(img_size=(720, 1440), patch_size=4, depths=(2,), num_heads=(8,), in_chans=73, out_chans=73,
                                embed_dim=768, img_window_ratio=80, full_pos_embed=True, rel_pos=False, compute_mode="bf16").to(DEV)
    x = torch.randn(1, 73, 720, 1440, generator=torch.Generator().manual_seed(5)).to(DEV)
    model(x)                                   # shadows and the pos_embed copy exist before either measurement
    with torch.no_grad():
        model(x)
    out_fo, peak_fo = _peak(lambda: model(x))
    monkeypatch.setattr(SG, "_forward_only", lambda *t: False)
    out_tr, peak_tr = _peak(lambda: model(x))
    h_bytes = 180 * 360 * 3072 * 2
    print(f"peak no_grad forward: training kernels {peak_tr / 2**20:.0f} MiB, forward-only {peak_fo / 2**20:.0f} MiB")
    assert torch.equal(out_fo, out_tr)
    assert peak_tr - peak_fo >= h_bytes, (peak_tr, peak_fo)
