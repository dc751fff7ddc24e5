"""CPU: the oracle against the live, unmodified reference.  The reference is not part of this repository: these tests
run when SWIN_REFERENCE_ROOT names a checkout of it and are skipped otherwise -- then the committed fixtures of
tests/test_oracle_golden.py stand in for it."""
import pytest
import torch

from oracle import shim
from oracle import swinv2_oracle as O

pytestmark = pytest.mark.skipif(not shim.reference_available(), reason="reference tree not present (set SWIN_REFERENCE_ROOT)")


@pytest.mark.parametrize("rel_pos", [False, True])
@pytest.mark.parametrize("residual", [False, True])
def test_forward_backward_matches_reference(rel_pos, residual):
    swin, losses = shim.import_reference()
    cfg = O.SwinConfig(img_size=(72, 144), depth=3, num_heads=2, in_chans=7, out_chans=5, embed_dim=192, window_ratio=8,
                       rel_pos=rel_pos, residual=residual)
    m = swin.SwinTransformerV2Cr(img_size=cfg.img_size, patch_size=4, depths=(cfg.depth,), num_heads=(cfg.num_heads,),
                                 in_chans=cfg.in_chans, out_chans=cfg.out_chans, embed_dim=cfg.embed_dim,
                                 img_window_ratio=cfg.window_ratio, full_pos_embed=True, rel_pos=rel_pos,
                                 residual=residual).eval()
    sd = O.init_state_dict(cfg, seed=1)
    assert list(sd.keys()) == list(m.state_dict().keys())
    m.load_state_dict(sd)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, cfg.in_chans, 72, 144, generator=g)
    tar = torch.randn(2, cfg.out_chans, 72, 144, generator=g)
    chw = torch.ones(cfg.out_chans) / cfg.out_chans
    y_ref = m(x)
    for absolute in (False, True):
        lossf = losses.GeometricLpLoss((72, 144), (72, 144), (0, 0), p=2, absolute=absolute, squared=True)
        l_ref = lossf(y_ref, tar, chw.view(1, -1))
        g_ref = torch.autograd.grad(l_ref, list(m.parameters()), retain_graph=True)
        pred, loss, grads = O.loss_and_grads(x, tar, sd, cfg, chw, relative=not absolute)
        assert O.rel_l2(pred, y_ref) < 2e-6
        assert abs(float(loss) - float(l_ref)) / float(l_ref) < 2e-6
        for (k, _), gr in zip(m.named_parameters(), g_ref):
            if k.endswith("meta_mlp.fc2.bias"):
                continue
            assert O.rel_l2(grads[k], gr) < 2e-5, k
    for i, blk in enumerate(m.stages[0].blocks):
        mk = O.shift_attention_mask(cfg.grid, cfg.window, cfg.shift(i))
        assert (mk is None) == (blk.attn_mask is None)
        if mk is not None:
            assert torch.equal(mk, blk.attn_mask)
        if rel_pos:
            assert torch.equal(O.relative_coordinates_log(cfg.window), blk.attn.relative_coordinates_log)
            tbl = O.cpb_bias_table(sd, f"stages.0.blocks.{i}.attn.", cfg.window, cfg.num_heads)
            assert torch.equal(tbl, blk.attn._relative_positional_encodings()[0])


def test_seed_identical_initialisation():
    """Same torch seed -> the drop-in module and the reference hold identical parameters."""
    swin, _ = shim.import_reference()
    from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr
    for rel_pos in (False, True):
        kw = dict(img_size=(72, 144), patch_size=4, depths=(3,), num_heads=(2,), in_chans=7, out_chans=5, embed_dim=192,
                  img_window_ratio=8, full_pos_embed=True, rel_pos=rel_pos, drop_path_rate=0.1)
        torch.manual_seed(5)
        ref = swin.SwinTransformerV2Cr(**kw)
        torch.manual_seed(5)
        mine = SwinTransformerV2Cr(**kw)
        a, b = ref.state_dict(), mine.state_dict()
        assert list(a.keys()) == list(b.keys())
        for k in a:
            assert torch.equal(a[k], b[k]), k


def test_quadrature_and_loss_handler_weights():
    _, losses = shim.import_reference()
    from types import SimpleNamespace
    from swin_v2_weather_b200.utils.losses import LossHandler
    names = ['u10m', 't2m', 'z500', 'q850', 'tcwv', 'foo', '2d']
    p = SimpleNamespace(n_future=0, img_shape_x=72, img_shape_y=144, loss='weighted absolute squared geometric l2',
                        channel_weights='auto', n_out_channels=len(names), channel_names=names, out_channels=list(range(len(names))),
                        dt=1, model_grid_type='equiangular')
    ref, mine = losses.LossHandler(p), LossHandler(p)
    assert torch.equal(ref.channel_weights, mine.channel_weights)
    assert torch.equal(ref.loss_obj.quadrature.quad_weight, mine.loss_obj.quadrature.quad_weight.contiguous())
    assert torch.equal(ref.multistep_weight, mine.multistep_weight)


def _load_ref_metrics():
    import importlib.util
    import os
    import sys
    name = "_ref_weighted_acc_rmse"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(shim.REFERENCE_ROOT, "utils", "weighted_acc_rmse.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("loss", ["weighted absolute temp-std squared geometric l2", "weighted temp-std geometric l2",
                                  "weighted geometric l1", "absolute geometric l1", "l2", "absolute squared geometric l2"])
def test_loss_handler_variants_match_reference(loss, tmp_path):
    """Config-4 channel weights (`'auto'` table x temp-std ratio, utils/losses.py:56-99) and the L1 / non-squared loss
    variants (:101-124): oracle restatement vs the live reference LossHandler -- weights bit-exact, loss and dL/dprd 1e-6."""
    import numpy as np
    from types import SimpleNamespace
    _, losses = shim.import_reference()
    C = 73
    rng = np.random.default_rng(7)
    gstd = np.ones((1, C, 1, 1), dtype=np.float32)
    tstd = rng.uniform(0.2, 1.0, size=(1, C, 1, 1)).astype(np.float32)
    np.save(tmp_path / "global_stds.npy", gstd)
    np.save(tmp_path / "time_diff_stds.npy", tstd)
    p = SimpleNamespace(n_future=0, img_shape_x=36, img_shape_y=72, loss=loss, channel_weights='auto', n_out_channels=C,
                        channel_names=list(O.CHANNEL_NAMES_73), out_channels=list(range(C)), dt=1, model_grid_type='equiangular',
                        global_stds_path=str(tmp_path / "global_stds.npy"), time_diff_stds_path=str(tmp_path / "time_diff_stds.npy"))
    ref = losses.LossHandler(p).train()
    w = O.loss_handler_channel_weights(loss, 'auto', p.channel_names, C, p.out_channels, 1, gstd, tstd)
    assert torch.equal(ref.channel_weights.reshape(-1).float(), w)
    g = torch.Generator().manual_seed(2)
    prd = torch.randn(2, C, 36, 72, generator=g, requires_grad=True)
    tar = torch.randn(2, C, 36, 72, generator=g)
    l_ref = ref(prd, tar, None)
    g_ref, = torch.autograd.grad(l_ref, prd)
    prd2 = prd.detach().clone().requires_grad_(True)
    l_or = O.loss_handler(prd2, tar, loss, w, n_future=0, training=True)
    g_or, = torch.autograd.grad(l_or, prd2)
    assert abs(float(l_or) - float(l_ref)) <= 1e-6 * abs(float(l_ref))
    assert O.rel_l2(g_or, g_ref) < 1e-6


def test_validation_metrics_and_zscore_match_reference():
    m = _load_ref_metrics()
    g = torch.Generator().manual_seed(3)
    pred = torch.randn(3, 5, 37, 72, generator=g)
    tar = torch.randn(3, 5, 37, 72, generator=g)
    assert torch.allclose(O.weighted_rmse_channels(pred, tar), m.weighted_rmse_torch_channels(pred, tar), rtol=1e-6, atol=0)
    assert torch.allclose(O.weighted_acc_channels(pred, tar), m.weighted_acc_torch_channels(pred, tar), rtol=1e-5, atol=1e-7)
