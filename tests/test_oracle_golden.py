"""CPU: the oracle (our restatement) against fixtures produced by the unmodified reference
(`oracle/make_golden.py`, run with SWIN_REFERENCE_ROOT naming a checkout of the reference)."""
import os

import numpy as np
import pytest
import torch

from oracle import swinv2_oracle as O

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def inputs(cfg, batch, seed=1234):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, cfg.in_chans, *cfg.img_size, generator=g)
    tar = torch.randn(batch, cfg.out_chans, *cfg.img_size, generator=g)
    chw = torch.rand(cfg.out_chans, generator=g) + 0.5
    return x, tar, chw / chw.sum()


@pytest.mark.parametrize("case", ["nopos_rel", "cpb_abs_residual"])
def test_oracle_matches_reference_fixture(case):
    fix = torch.load(os.path.join(GOLDEN, f"model_{case}.pt"), weights_only=False)
    cfg = O.SwinConfig(**fix["config"])
    sd = O.init_state_dict(cfg, seed=1)
    x, tar, chw = inputs(cfg, fix["batch"])
    pred, loss, grads = O.loss_and_grads(x, tar, sd, cfg, chw, relative=fix["loss_kind"] == "rel")
    assert O.rel_l2(pred, fix["pred"]) < 1e-5
    assert abs(float(loss) - float(fix["loss"])) / float(fix["loss"]) < 1e-5
    for k, n in fix["grad_norm"].items():
        if k.endswith("meta_mlp.fc2.bias"):   # analytically zero (softmax shift invariance): pure rounding noise
            assert float(grads[k].abs().max()) < 1e-5
            continue
        g = grads[k]
        assert abs(float(g.double().norm()) - float(n)) / float(n) < 2e-5, k
        idx = torch.randint(0, g.numel(), (min(64, g.numel()),), generator=torch.Generator().manual_seed(g.numel()))
        got = g.reshape(-1)[idx]
        assert (got - fix["grad_sample"][k]).norm() <= 2e-5 * float(n) + 1e-5 * fix["grad_sample"][k].norm(), k


def test_bit_exact_buffers():
    buf = torch.load(os.path.join(GOLDEN, "buffers.pt"), weights_only=False)
    for tag, grid in (("small", (18, 36)), ("full", (180, 360))):
        mask = O.shift_attention_mask(grid, (9, 18), (4, 9))
        assert tuple(mask.shape) == tuple(buf[f"mask_shape_{tag}"])
        assert set(torch.unique(mask).tolist()) <= {0.0, -100.0}
        nWw = grid[1] // 18
        mrow = mask.view(grid[0] // 9, nWw, *mask.shape[1:])
        for j in range(nWw):
            assert torch.equal(mrow[:, 0], mrow[:, j])
        packed = torch.from_numpy(np.packbits((mrow[:, 0] != 0).numpy().reshape(-1)))
        assert torch.equal(packed, buf[f"mask_rows_packed_{tag}"])
    assert torch.equal(O.relative_coordinates_log((9, 18)), buf["relative_coordinates_log"])
    assert torch.equal(O.quadrature_row_weights(72, 144), buf["quad_rows_small"])
    assert torch.equal(O.quadrature_row_weights(720, 1440), buf["quad_rows_full"])


def test_mask_statistics_full_geometry():
    """SURVEY F6: only the last window row is masked; 2*90*72/162^2 of it; 2.47 % overall."""
    mask = O.shift_attention_mask((180, 360), (9, 18), (4, 9))
    nz = (mask != 0).float()
    assert float(nz[: 19 * 20].sum()) == 0.0
    assert abs(float(nz[19 * 20:].mean()) - 2 * 90 * 72 / 162 ** 2) < 1e-6
    assert abs(float(nz.mean()) - 0.0247) < 1e-4


def test_window_token_index_is_roll_then_partition():
    H, W, Wh, Ww, s0, s1 = 18, 36, 9, 18, 4, 9
    x = torch.arange(H * W).view(1, H, W, 1)
    rolled = torch.roll(x, shifts=(-s0, -s1), dims=(1, 2))
    win = rolled.view(1, H // Wh, Wh, W // Ww, Ww, 1).permute(0, 1, 3, 2, 4, 5).reshape(-1, Wh * Ww)
    assert torch.equal(O.window_token_index((H, W), (Wh, Ww), (s0, s1)), win)
    # every token appears exactly once
    assert torch.equal(torch.sort(O.window_token_index((H, W), (Wh, Ww), (s0, s1)).reshape(-1)).values, torch.arange(H * W))


def test_zero_init_norms_make_blocks_identity():
    """SURVEY F7: with the reference's init (norm weights 0) each block is the identity."""
    cfg = O.SwinConfig(img_size=(72, 144), depth=2, num_heads=1, in_chans=3, out_chans=3, embed_dim=96, window_ratio=8)
    sd = O.init_state_dict(cfg, seed=0, randomize_norms=False)
    t = O.patch_embed(torch.randn(1, 3, 72, 144), sd, cfg)
    assert torch.equal(O.block_forward(t, sd, cfg, 1), t)
