"""The fp64 attention reference (oracle/attention_exact.py) against autograd, on a machine without a GPU.

At fp64, with q^ / k^ exactly normalised and the passed o equal to the true output, the reference's explicit gradients must
be autograd through F.normalize of the oracle's forward (`oracle_attention` of tests/test_kernels_gpu.py, the same index
arithmetic) to rounding.  Plane 1 of the lse output, E_P[cos], is d lse / d scale, so it is checked through autograd as well.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle.attention_exact import attention_exact
from test_kernels_gpu import oracle_attention

TOL = 1e-10


def rel(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


@pytest.mark.parametrize("cfg", [
    dict(H=6, W=8, heads=2, d=8, window=(3, 4), shift=(0, 0), bias=False),
    dict(H=6, W=8, heads=2, d=8, window=(3, 4), shift=(1, 2), bias=True),
    dict(H=8, W=8, heads=1, d=16, window=(4, 4), shift=(2, 2), bias=False),
    dict(H=4, W=12, heads=3, d=12, window=(2, 6), shift=(0, 3), bias=True),   # column shift only: no mask
    dict(H=9, W=12, heads=2, d=16, window=(3, 6), shift=(1, 0), bias=True),
])
def test_attention_exact_matches_autograd(cfg):
    B, H, W, heads, d = 2, cfg["H"], cfg["W"], cfg["heads"], cfg["d"]
    Wh, Ww = cfg["window"]
    s0, s1 = cfg["shift"]
    C, L, T = heads * d, Wh * Ww, B * H * W
    g = torch.Generator().manual_seed(H * 100 + W + d)
    raw = torch.randn(T, 3 * C, generator=g, dtype=torch.float64)
    scale = (2.0 + 10.0 * torch.rand(heads, generator=g, dtype=torch.float64))
    bias = torch.randn(heads, L, L, generator=g, dtype=torch.float64) if cfg["bias"] else None
    d_o = torch.randn(T, C, generator=g, dtype=torch.float64)

    raw_a = raw.clone().requires_grad_(True)
    sc_a = scale.clone().requires_grad_(True)
    b_a = bias.clone().requires_grad_(True) if bias is not None else None
    o_ref, lse_ref = oracle_attention(raw_a, sc_a, b_a, B, H, W, C, heads, (Wh, Ww), (s0, s1))
    wl = torch.randn(lse_ref.shape, generator=g, dtype=torch.float64)
    ((o_ref * d_o).sum() + (lse_ref * wl).sum()).backward()
    # the lse term contributes to the scale gradient only through plane 1 (sum_i wl_i E_i) and to dq / dk / dbias too:
    # take it apart again with a second pass without it
    dscale_lse = sc_a.grad.clone()
    raw_b = raw.clone().requires_grad_(True)
    sc_b = scale.clone().requires_grad_(True)
    b_b = bias.clone().requires_grad_(True) if bias is not None else None
    o_b, _ = oracle_attention(raw_b, sc_b, b_b, B, H, W, C, heads, (Wh, Ww), (s0, s1))
    (o_b * d_o).sum().backward()
    dscale_lse -= sc_b.grad

    # the kernel's inputs: stored q^ / k^ (exactly normalised here), inv_norm, and the passed o
    x = raw.view(T, 3, heads, d)
    qkv = torch.cat([F.normalize(x[:, :2], dim=-1), x[:, 2:]], dim=1).reshape(T, 3 * C)
    inv = 1.0 / x[:, :2].norm(dim=-1)                                        # (T, 2, heads)
    got = attention_exact(qkv, scale, bias, o_ref.detach(), d_o, inv, B, H, W, C, heads, Wh, Ww, s0, s1)

    assert rel(got["o"], o_ref.detach()) < TOL
    assert rel(got["lse"][0], lse_ref.detach()) < TOL
    assert rel(got["D"], (o_ref.detach() * d_o).view(T, heads, d).sum(-1)) < TOL
    assert rel(got["dqkv"], raw_b.grad) < TOL
    for part in range(3):                                                    # dq, dk, dv one by one
        sl = slice(part * C, (part + 1) * C)
        assert rel(got["dqkv"][:, sl], raw_b.grad[:, sl]) < TOL, part
    assert rel(got["dscale"], sc_b.grad) < TOL
    assert rel(got["dscale_centred"], sc_b.grad) < TOL                      # o is exact here: the two forms agree
    if bias is not None:
        assert rel(got["dbias"], b_b.grad) < TOL
    else:
        assert got["dbias"] is None
    # plane 1: sum_i wl_i E_i per head == the lse term's share of d/d scale
    plane1 = (got["lse"][1] * wl).sum(dim=(0, 1, 3))
    assert rel(plane1, dscale_lse) < TOL


def test_attention_exact_uses_the_passed_o():
    """D = <dO, o> comes from the o handed in, as in the kernels: a perturbed o moves D and dS, not the forward."""
    B, H, W, heads, d, Wh, Ww = 1, 4, 8, 2, 8, 2, 4
    C, T = heads * d, B * H * W
    g = torch.Generator().manual_seed(5)
    x = torch.randn(T, 3, heads, d, generator=g, dtype=torch.float64)
    qkv = torch.cat([F.normalize(x[:, :2], dim=-1), x[:, 2:]], dim=1).reshape(T, 3 * C)
    inv = 1.0 / x[:, :2].norm(dim=-1)
    scale = torch.tensor([5.0, 9.0], dtype=torch.float64)
    d_o = torch.randn(T, C, generator=g, dtype=torch.float64)
    o = attention_exact(qkv, scale, None, None, None, None, B, H, W, C, heads, Wh, Ww, 0, 0)["o"]
    o2 = o + 0.01 * torch.randn(T, C, generator=g, dtype=torch.float64)
    a = attention_exact(qkv, scale, None, o, d_o, inv, B, H, W, C, heads, Wh, Ww, 0, 0)
    b = attention_exact(qkv, scale, None, o2, d_o, inv, B, H, W, C, heads, Wh, Ww, 0, 0)
    assert torch.equal(a["o"], b["o"]) and torch.equal(a["lse"], b["lse"])
    assert rel(b["D"], (o2 * d_o).view(T, heads, d).sum(-1)) < TOL
    assert not torch.allclose(a["dqkv"][:, :C], b["dqkv"][:, :C])
    assert torch.equal(a["dqkv"][:, 2 * C:], b["dqkv"][:, 2 * C:])           # dv does not depend on D
    # the centred d(scale) does not see the perturbation to first order; the plain one does
    assert abs(float(b["dscale_centred"][0] - a["dscale_centred"][0])) < 1e-3 * abs(float(b["dscale"][0] - a["dscale"][0]))
