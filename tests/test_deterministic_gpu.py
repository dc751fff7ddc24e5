"""GPU: deterministic mode (torch.use_deterministic_algorithms(True)) gives the same bits on every run.

Every deterministic entry point runs three times and must return equal tensors each time; one of the runs happens while a
large torch.matmul occupies SMs on a second stream, which moves the persistent kernels' tile placement and the order in which
blocks arrive.  Each result is also compared with an fp64 torch reference where one is cheap to state, and with the default
(atomic) path within fp32 tolerance.  Whole training steps (forward, loss, backward) must be bitwise equal over three runs and
still meet the oracle bars of test_parity_headline_gpu.py.
"""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import swinv2_oracle as O
from swin_v2_weather_b200 import _lib, ops
from swin_v2_weather_b200.ops import EPI_F32, MODE_BF16, MODE_FP32

pytestmark = pytest.mark.gpu


@pytest.fixture
def det():
    """Deterministic mode for the test; CUBLAS_WORKSPACE_CONFIG for the torch-side CPB meta-MLP."""
    old_env = os.environ.get("CUBLAS_WORKSPACE_CONFIG")
    os.environ["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"
    old = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(old[0], warn_only=old[1])
    if old_env is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = old_env


def _flat(out):
    if isinstance(out, torch.Tensor):
        return [out]
    if isinstance(out, dict):
        return [v for k in sorted(out) for v in _flat(out[k])]
    return [v for o in out if o is not None for v in _flat(o)]


def thrice(fn):
    """fn() three times -- the second while a benign matmul keeps SMs busy on another stream -- all results bitwise equal."""
    runs = []
    for i in range(3):
        if i == 1:
            side = torch.cuda.Stream()
            a = torch.randn(8192, 8192, device="cuda")
            torch.cuda.synchronize()
            with torch.cuda.stream(side):
                for _ in range(4):
                    a = a @ a * 1e-4
            out = fn()
            torch.cuda.synchronize()
        else:
            out = fn()
            torch.cuda.synchronize()
        runs.append([t.detach().clone() for t in _flat(out)])
    for r in runs[1:]:
        assert len(r) == len(runs[0])
        for x, y in zip(runs[0], r):
            assert torch.equal(x, y), "deterministic mode gave different bits"
    return out


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def default_path(fn):
    torch.use_deterministic_algorithms(False)
    try:
        out = fn()
        torch.cuda.synchronize()
        return out
    finally:
        torch.use_deterministic_algorithms(True)


# ---- kernels -----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,T,S", [(2304, 768, 8192, 8), (1168, 768, 6000, 4), (768, 3072, 4096, 3)])
def test_splitk_wgrad(det, M, N, T, S):
    g = torch.Generator(device="cuda").manual_seed(M + S)
    dy = torch.randn(T, M, device="cuda", generator=g).bfloat16()
    x = torch.randn(T, N, device="cuda", generator=g).bfloat16()
    base = torch.randn(M, N, device="cuda", generator=g)

    def run():
        out = base.clone()
        return ops.gemm(MODE_BF16, dy, 1, x, 1, EPI_F32, out=out, accumulate=True, split_k=S)

    out = thrice(run)
    ref = base.double() + dy.double().t() @ x.double()
    assert rel(out, ref) < 1e-5
    assert rel(out, default_path(run)) < 1e-5


def test_fused_wgrad_colsum(det):
    g = torch.Generator(device="cuda").manual_seed(3)
    dy = torch.randn(9000, 2304, device="cuda", generator=g).bfloat16()
    x = torch.randn(9000, 768, device="cuda", generator=g).bfloat16()

    def run():
        dw = torch.zeros(2304, 768, device="cuda")
        db = torch.zeros(2304, device="cuda")
        return ops.linear_wgrad(MODE_BF16, dy, x, dw, db, 8)

    dw, db = thrice(run)
    assert rel(dw, dy.double().t() @ x.double()) < 1e-5
    assert rel(db, dy.double().sum(0)) < 1e-5
    dw0, db0 = default_path(run)
    assert rel(dw, dw0) < 1e-5 and rel(db, db0) < 1e-5


@pytest.mark.parametrize("C,dtype", [(768, torch.bfloat16), (768, torch.float32), (2048, torch.bfloat16), (2048, torch.float32),
                                     (192, torch.float32)])
def test_ln_residual_bwd(det, C, dtype):
    rows, rps = 5003, 2500
    mode = MODE_BF16 if dtype == torch.bfloat16 else MODE_FP32
    g = torch.Generator(device="cuda").manual_seed(C)
    dx = torch.randn(rows, C, device="cuda", generator=g)
    z = (torch.randn(rows, C, device="cuda", generator=g) * 2 + 0.5).to(dtype)
    zf = z.double()
    stats = torch.stack([zf.mean(1), (zf.var(1, unbiased=False) + 1e-5).rsqrt()], 1).float().contiguous()
    gamma = 1 + 0.1 * torch.randn(C, device="cuda", generator=g)
    sc = torch.rand(3, device="cuda", generator=g) + 0.5

    def run():
        return ops.ln_residual_bwd(dx, z, stats, gamma, sc, rps, mode)

    dz, dg, db, dbp = thrice(run)
    s = sc.double()[torch.arange(rows, device="cuda") // rps][:, None]
    xh = (zf - stats[:, :1].double()) * stats[:, 1:].double()
    gg = dx.double() * s * gamma.double()
    dz_ref = stats[:, 1:].double() * (gg - gg.mean(1, keepdim=True) - xh * (gg * xh).mean(1, keepdim=True))
    assert rel(dg, (dx.double() * s * xh).sum(0)) < 1e-4
    assert rel(db, (dx.double() * s).sum(0)) < 1e-4
    assert rel(dbp, dz_ref.sum(0)) < 1e-3
    ref = default_path(run)
    for a, b in zip((dg, db, dbp), ref[1:]):
        assert rel(a, b) < 1e-5
    assert torch.equal(dz, ref[0])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_colsum(det, dtype):
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(70001, 3072, device="cuda", generator=g).to(dtype)
    out = thrice(lambda: ops.colsum(x))
    assert rel(out, x.double().sum(0)) < 1e-5
    assert rel(out, default_path(lambda: ops.colsum(x))) < 1e-5


def test_losses_and_acc(det):
    g = torch.Generator(device="cuda").manual_seed(2)
    prd = torch.randn(2, 5, 720, 1440, device="cuda", generator=g)      # 10 planes: 119 row blocks per plane
    tar = torch.randn(2, 5, 720, 1440, device="cuda", generator=g)
    qw = O.quadrature_row_weights(720, 1440).cuda()
    chw = torch.rand(5, device="cuda", generator=g)
    l2 = thrice(lambda: ops.latw_l2_fwd(prd, tar, qw, chw, True))
    l1 = thrice(lambda: ops.latw_l1_fwd(prd, tar, qw, chw, True))
    acc = thrice(lambda: ops.latw_acc(prd, tar, qw))
    p, t, q = prd.double(), tar.double(), qw.double()[None, None, :, None]
    num, den = (q * (p - t) ** 2).sum((2, 3)), (q * t ** 2).sum((2, 3))
    assert rel(l2[0], ((num / den) * chw.double()).sum()) < 1e-5
    s0, s1 = (q * (p - t).abs()).sum((2, 3)), (q * t.abs()).sum((2, 3))
    assert rel(l1[0], ((s0 / s1) * chw.double()).sum()) < 1e-5
    assert rel(acc, (q * p * t).sum((2, 3)) / ((q * p * p).sum((2, 3)) * (q * t * t).sum((2, 3))).sqrt()) < 1e-5
    assert rel(l2[0], default_path(lambda: ops.latw_l2_fwd(prd, tar, qw, chw, True))[0]) < 1e-6
    assert rel(acc, default_path(lambda: ops.latw_acc(prd, tar, qw))) < 1e-6


ATTN_CASES = [
    # (mode, C, heads, H, W): d 96 on the full 180 x 360 token grid (persistent tcgen05 kernel), d 64 / d 256 (attn_tc_gen),
    # fp32 on the CUDA cores
    ("bf16", 768, 8, 180, 360),
    ("bf16", 512, 8, 36, 72),
    ("bf16", 512, 2, 36, 72),
    ("fp32", 192, 2, 36, 72),
]


@pytest.mark.parametrize("mode_name,C,heads,H,W", ATTN_CASES)
@pytest.mark.parametrize("shift", [False, True])
@pytest.mark.parametrize("with_bias", [False, True])
def test_attention_backward(det, mode_name, C, heads, H, W, shift, with_bias):
    mode = ops.MODES[mode_name]
    Wh, Ww = 9, 18
    s0, s1 = (Wh // 2, Ww // 2) if shift else (0, 0)
    B, L = 1, Wh * Ww
    g = torch.Generator(device="cuda").manual_seed(C + heads)
    qkv = torch.randn(B * H * W, 3 * C, device="cuda", generator=g).to(mode.act_dtype)
    inv_norm = ops.qk_normalize_(qkv, C, heads)
    scale = torch.rand(heads, device="cuda", generator=g) * 10 + 5
    bias = (torch.randn(heads, L, L, device="cuda", generator=g) * 0.5) if with_bias else None
    o, lse = ops.window_attn_fwd(qkv, scale, bias, B, H, W, C, heads, Wh, Ww, s0, s1, mode)
    d_o = torch.randn(B * H * W, C, device="cuda", generator=g).to(mode.act_dtype)

    def run():
        return ops.window_attn_bwd(qkv, inv_norm, scale, bias, o, d_o, lse, B, H, W, C, heads, Wh, Ww, s0, s1, mode)

    dqkv, dscale, dbias = thrice(run)
    dqkv0, dscale0, dbias0 = default_path(run)
    assert rel(dqkv.float(), dqkv0.float()) < 1e-6
    assert rel(dscale, dscale0) < 1e-4
    if with_bias:
        assert rel(dbias, dbias0) < 1e-5


# ---- whole training steps ------------------------------------------------------------------------------------------------------
def _model(cfg, sd, mode, **kw):
    from test_parity_headline_gpu import build
    return build(cfg, sd, mode, **kw)


def _step(model, x, tar, chw):
    from test_parity_headline_gpu import run_ours
    pred, loss, grads = run_ours(model, x, tar, chw, True)
    return pred, torch.tensor([loss], dtype=torch.float64), grads


def _model_thrice(model, x, tar, chw):
    out = thrice(lambda: _step(model, x, tar, chw))
    return out[0], float(out[1]), out[2]


@pytest.mark.parametrize("rel_pos", [False, True])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_training_step_small_image(det, mode, rel_pos):
    """C = 768, 8 heads, depth 2 on a 72 x 144 image: bitwise equal over three steps, and within the oracle bars."""
    from test_parity_headline_gpu import (BF16_TOL, FP32_TOL, FP32_TOL_SCALE, NOISY, assert_within, errors, inputs,
                                          round_gemm_weights)
    cfg = O.SwinConfig(img_size=(72, 144), depth=2, num_heads=8, in_chans=73, out_chans=73, embed_dim=768, window_ratio=8,
                       rel_pos=rel_pos)
    sd = O.init_state_dict(cfg, seed=11)
    x, tar = inputs(cfg, 2)
    chw = torch.ones(73) / 73
    ours = _model_thrice(_model(cfg, sd, mode), x, tar, chw)
    ref = O.loss_and_grads(x, tar, sd, cfg, chw, relative=True)
    name = f"deterministic_d2_{mode}_{'cpb' if rel_pos else 'nopos'}"
    if mode == "fp32":
        assert_within(errors(*ours, *ref), FP32_TOL, FP32_TOL_SCALE, name)
    else:
        # bars (i) and (ii) of test_parity_headline_gpu.py; logit_scale / meta_mlp.* within 2e-2 of the nearer oracle, the bar
        # that file uses for this 8-window image (there the weight rounding alone moves them by 1.3e-2)
        rep_i = errors(*ours, *O.loss_and_grads(x, tar, round_gemm_weights(sd), cfg, chw, relative=True))
        rep_ii = errors(*ours, *ref)
        noisy = lambda k: any(t in k for t in NOISY)       # noqa: E731
        assert_within({k: v for k, v in rep_i.items() if not noisy(k)}, BF16_TOL, None, name + " (i)")
        assert_within({k: v for k, v in rep_ii.items() if not noisy(k)}, BF16_TOL, None, name + " (ii)")
        assert_within({k: min(rep_i[k], rep_ii[k]) for k in rep_i if noisy(k)}, 2e-2, None, name + " (noisy)")


def test_training_step_full_resolution(det):
    """73 x 720 x 1440, depth 1, bf16: bitwise equal over three steps, and within the bf16 bar of the default path."""
    from test_parity_headline_gpu import inputs
    cfg = O.SwinConfig(depth=1)
    sd = O.init_state_dict(cfg, seed=2)
    x, tar = inputs(cfg, 1, seed=5)
    chw = torch.ones(73) / 73
    model = _model(cfg, sd, "bf16")
    pred, loss, grads = _model_thrice(model, x, tar, chw)
    pred0, loss0, grads0 = default_path(lambda: _step(model, x, tar, chw))
    assert rel(pred, pred0) < 1e-3 and abs(loss - float(loss0)) < 1e-4 * abs(loss)
    bad = [(k, rel(grads[k], grads0[k])) for k in grads if rel(grads[k], grads0[k]) > 1e-2]
    assert not bad, bad


def test_training_step_e2048_block(det):
    """The embed_dim 2048 / head_dim 256 / mlp_ratio 2 block on the small image (tcgen05 attention at d 256, C = 2048 LN)."""
    from test_parity_headline_gpu import inputs
    cfg = O.SwinConfig(img_size=(72, 144), depth=1, num_heads=8, in_chans=73, out_chans=73, embed_dim=2048, window_ratio=8,
                       mlp_ratio=2.0)
    sd = O.init_state_dict(cfg, seed=7)
    x, tar = inputs(cfg, 1)
    chw = torch.ones(73) / 73
    model = _model(cfg, sd, "bf16")
    pred, loss, grads = _model_thrice(model, x, tar, chw)
    pred0, _, grads0 = default_path(lambda: _step(model, x, tar, chw))
    assert rel(pred, pred0) < 1e-3
    bad = [(k, rel(grads[k], grads0[k])) for k in grads if rel(grads[k], grads0[k]) > 2e-2]
    assert not bad, bad


def test_training_step_config4(det, tmp_path):
    """BASELINE config 4 on the small image: 77 input channels as channel groups, residual skip, the 'weighted absolute
    temp-std squared geometric l2' LossHandler loss."""
    from swin_v2_weather_b200.utils.losses import LossHandler
    from test_parity_headline_gpu import inputs
    H, W = 72, 144
    cfg = O.SwinConfig(img_size=(H, W), depth=2, num_heads=8, in_chans=77, out_chans=73, embed_dim=768, window_ratio=8, residual=True)
    sd = O.init_state_dict(cfg, seed=4)
    x, tar = inputs(cfg, 2)
    rng = np.random.default_rng(7)
    np.save(tmp_path / "gs.npy", np.ones((1, 73, 1, 1), dtype=np.float32))
    np.save(tmp_path / "ts.npy", rng.uniform(0.2, 1.0, size=(1, 73, 1, 1)).astype(np.float32))
    lp = SimpleNamespace(n_future=0, img_shape_x=H, img_shape_y=W, loss='weighted absolute temp-std squared geometric l2',
                         channel_weights='auto', n_out_channels=73, channel_names=list(O.CHANNEL_NAMES_73), out_channels=list(range(73)),
                         dt=1, model_grid_type='equiangular', global_stds_path=str(tmp_path / "gs.npy"),
                         time_diff_stds_path=str(tmp_path / "ts.npy"))
    lossf = LossHandler(lp).cuda().train()
    model = _model(cfg, sd, "bf16")
    groups = (x[:, :73].cuda().contiguous(), x[:, 73:74].cuda().contiguous(), x[:1, 74:].cuda().contiguous())
    tar_d = tar.cuda()

    def run():
        model.zero_grad(set_to_none=True)
        pred = model(groups)
        loss = lossf(pred, tar_d, None)
        loss.backward()
        return pred.detach(), loss.detach(), {k: p.grad for k, p in model.named_parameters()}

    pred, loss, grads = thrice(run)
    pred0, loss0, grads0 = default_path(run)
    assert rel(pred, pred0) < 1e-3 and rel(loss, loss0) < 1e-4
    bad = [(k, rel(grads[k], grads0[k])) for k in grads if rel(grads[k], grads0[k]) > 1e-2]
    assert not bad, bad


def test_flag_is_read_at_each_call(det):
    """The same ops call switches path with the flag: no state is kept between calls."""
    x = torch.randn(4096, 768, device="cuda")
    calls = []
    real = _lib.call

    def spy(name, *args):
        calls.append(name)
        return real(name, *args)

    _lib.call = spy
    try:
        ops.colsum(x)
        default_path(lambda: ops.colsum(x))
        ops.colsum(x)
    finally:
        _lib.call = real
    assert calls == ["swinb200_colsum_det", "swinb200_colsum", "swinb200_colsum_det"]
