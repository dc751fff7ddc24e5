"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.pt by running the UNMODIFIED reference
(a checkout named by SWIN_REFERENCE_ROOT, imported through oracle/shim.py) on CPU in fp32.

Run:   SWIN_REFERENCE_ROOT=<reference checkout> python -m oracle.make_golden
The fixtures are small: inputs and weights are *not* stored -- they are regenerated from seeds with
`oracle.swinv2_oracle.init_state_dict` / CPU generators, which is deterministic for a given torch build.
Stored per case: prediction, loss, per-parameter gradient norms and 64 sampled gradient entries.
Also stored: the reference's bit-exact integer-derived buffers (shift masks, relative_coordinates_log,
quadrature weights) at the test geometry and at the full 180x360 / 720x1440 geometry.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import shim  # noqa: E402
from oracle import swinv2_oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

CASES = {
    # name: (SwinConfig kwargs, batch, loss kind)
    "nopos_rel": (dict(img_size=(72, 144), depth=2, num_heads=1, in_chans=7, out_chans=5, embed_dim=96, window_ratio=8,
                       rel_pos=False, residual=False), 2, "rel"),
    "cpb_abs_residual": (dict(img_size=(72, 144), depth=2, num_heads=2, in_chans=7, out_chans=5, embed_dim=192, window_ratio=8,
                              rel_pos=True, residual=True), 1, "abs"),
}


def case_inputs(cfg: O.SwinConfig, batch: int, seed: int = 1234):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, cfg.in_chans, *cfg.img_size, generator=g)
    tar = torch.randn(batch, cfg.out_chans, *cfg.img_size, generator=g)
    chw = torch.rand(cfg.out_chans, generator=g) + 0.5
    chw = chw / chw.sum()
    return x, tar, chw


def sample_index(numel: int, n: int = 64) -> torch.Tensor:
    g = torch.Generator().manual_seed(numel)
    return torch.randint(0, numel, (min(n, numel),), generator=g)


def build_reference_model(swin, cfg: O.SwinConfig, sd):
    m = swin.SwinTransformerV2Cr(img_size=cfg.img_size, patch_size=cfg.patch_size, depths=(cfg.depth,),
                                 num_heads=(cfg.num_heads,), in_chans=cfg.in_chans, out_chans=cfg.out_chans,
                                 embed_dim=cfg.embed_dim, img_window_ratio=cfg.window_ratio, drop_path_rate=0.0,
                                 full_pos_embed=cfg.full_pos_embed, rel_pos=cfg.rel_pos, mlp_ratio=cfg.mlp_ratio,
                                 residual=cfg.residual)
    m.load_state_dict(sd)
    return m.eval()


def main():
    os.makedirs(OUT, exist_ok=True)
    swin, losses = shim.import_reference()
    torch.manual_seed(0)
    for name, (kw, batch, kind) in CASES.items():
        cfg = O.SwinConfig(**kw)
        sd = O.init_state_dict(cfg, seed=1)
        x, tar, chw = case_inputs(cfg, batch)
        m = build_reference_model(swin, cfg, sd)
        pred = m(x)
        lossf = losses.GeometricLpLoss(cfg.img_size, cfg.img_size, (0, 0), p=2, absolute=(kind == "abs"), squared=True)
        loss = lossf(pred, tar, chw.view(1, -1))
        names = [k for k, _ in m.named_parameters()]
        grads = torch.autograd.grad(loss, list(m.parameters()))
        fix = {
            "config": kw, "batch": batch, "loss_kind": kind, "pred": pred.detach().clone(), "loss": loss.detach().double(),
            "grad_norm": {k: g.double().norm() for k, g in zip(names, grads)},
            "grad_sample": {k: g.reshape(-1)[sample_index(g.numel())].clone() for k, g in zip(names, grads)},
        }
        torch.save(fix, os.path.join(OUT, f"model_{name}.pt"))
        print(name, "loss", float(loss), "pred-norm", float(pred.norm()))

    # ---- bit-exact buffers -------------------------------------------------------------------------------
    buf = {}
    for tag, grid, ratio_window in (("small", (18, 36), (9, 18)), ("full", (180, 360), (9, 18))):
        blk = swin.SwinTransformerV2CrBlock(dim=96, num_heads=1, feat_size=grid, window_size=ratio_window,
                                            shift_size=(ratio_window[0] // 2, ratio_window[1] // 2), rel_pos=True)
        mask = blk.attn_mask                                   # (nW, L, L)
        nWw = grid[1] // ratio_window[1]
        mrow = mask.view(grid[0] // ratio_window[0], nWw, *mask.shape[1:])
        assert all(torch.equal(mrow[:, 0], mrow[:, j]) for j in range(nWw)), "mask varies along longitude?"
        vals = torch.unique(mask)
        assert set(vals.tolist()) <= {0.0, -100.0}
        buf[f"mask_rows_packed_{tag}"] = torch.from_numpy(np.packbits((mrow[:, 0] != 0).numpy().reshape(-1)))
        buf[f"mask_shape_{tag}"] = tuple(mask.shape)
        if tag == "small":
            buf["relative_coordinates_log"] = blk.attn.relative_coordinates_log.clone()
    for tag, shape in (("small", (72, 144)), ("full", (720, 1440))):
        q = losses.GeometricLpLoss(shape, shape, (0, 0), p=2).quadrature.quad_weight
        assert torch.equal(q[0, 0, :, :1].expand(-1, shape[1]), q[0, 0])
        buf[f"quad_rows_{tag}"] = q[0, 0, :, 0].clone()
    torch.save(buf, os.path.join(OUT, "buffers.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
