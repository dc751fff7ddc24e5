"""TEST INFRASTRUCTURE ONLY -- fp64 window attention on exactly the inputs the C ABI takes.

`swinb200_window_attn_fwd` / `_bwd` (include/swinb200.h) read the *stored* q^ / k^ / v (qkv after the q / k normalisation,
bf16 in training mode), and the backward reads the `o`, `d_o` and `inv_norm` it is handed.  The parity tests of
tests/test_kernels_gpu.py compare with an fp32 autograd oracle fed the raw qkv instead, so their bars must absorb the
rounding of q^ / k^ (about scale * 2^-9 per logit in bf16).  This reference removes that: every quantity below is a
function of the kernel's own inputs, evaluated in fp64 on whatever device the inputs are on, so what is left between it and a
kernel is the kernel's own arithmetic.

Definitions (per sample b, window w, head h; i = query slot, j = key slot of the window; index arithmetic from
`swinv2_oracle.window_token_index` / `shift_attention_mask`):

    cos_ij = q^_i . k^_j ;  S_ij = scale_h cos_ij (+ bias[h, i, j]) (+ mask[w, i, j]) ;  lse_i = logsumexp_j S_ij
    P_ij = exp(S_ij - lse_i) ;  O_i = sum_j P_ij v_j ;  E_i = sum_j P_ij cos_ij          (lse planes 0 and 1)
    D_i = <dO_i, o_i>  with o the PASSED output (the kernels form it from what they are given)
    dS_ij = P_ij (dO_i . v_j - D_i)
    dq^_i = scale_h sum_j dS_ij k^_j ;  dq_i = inv_q_i (dq^_i - q^_i <q^_i, dq^_i>)      (dk alike, over i)
    dv_j = sum_i P_ij dO_i ;  dscale_h = sum dS_ij cos_ij ;  dbias[h] = sum over samples and windows of dS

d(scale) has two forms.  "dscale" is the sum above, what the CUDA-core backward computes.  The tcgen05 backward sums
dS_ij (cos_ij - E_i) instead (include/swinb200.h, DESIGN.md section 2): sum_j dS_ij is zero with the exact o and equals
delta_i = <dO_i, o_exact_i - o_i> with the passed one, so the centred sum is the exact-o gradient whatever rounding o carries,
and the two forms differ by sum_i delta_i E_i.  "dscale_centred" is that sum, with the exact E.

The work runs per head over chunks of windows, so the 180 x 360 grid at 8 heads (84 M logits per plane) needs a few hundred MB.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import swinv2_oracle as O

_CHUNK_LOGITS = 1 << 23          # logits per chunk (fp64: 64 MB per (B, windows, L, L) temporary)


def attention_exact(qkv: torch.Tensor, scale: torch.Tensor, bias: Optional[torch.Tensor], o: Optional[torch.Tensor],
                    d_o: Optional[torch.Tensor], inv_norm: Optional[torch.Tensor], B: int, H: int, W: int, C: int, heads: int,
                    Wh: int, Ww: int, s0: int, s1: int) -> Dict[str, torch.Tensor]:
    """qkv (T, 3C) stored q^ | k^ | v; scale (heads,); bias (heads, L, L) or None; o, d_o (T, C); inv_norm (T, 2, heads).

    Returns fp64 tensors on qkv's device: "o" (T, C), "lse" (2, B, nW, heads, L) (plane 0 LSE, plane 1 E_P[cos]) and, when
    d_o is given, "D" (T, heads), "dqkv" (T, 3C), "dscale" and "dscale_centred" (heads,) and "dbias" (heads, L, L) (None
    without a bias table).
    """
    dev = qkv.device
    f64 = torch.float64
    d = C // heads
    L = Wh * Ww
    T = B * H * W
    idx = O.window_token_index((H, W), (Wh, Ww), (s0, s1)).to(dev)               # (nW, L)
    nW = idx.shape[0]
    mask = O.shift_attention_mask((H, W), (Wh, Ww), (s0, s1))
    mask = None if mask is None else mask.to(device=dev, dtype=f64)
    x = qkv.view(B, H * W, 3, heads, d)
    backward = d_o is not None
    if backward and (o is None or inv_norm is None):
        raise ValueError("attention_exact: the backward needs o and inv_norm")
    if backward:
        go = d_o.view(B, H * W, heads, d)
        oo = o.view(B, H * W, heads, d)
        inv = inv_norm.view(B, H * W, 2, heads)

    out_o = torch.empty((B, H * W, heads, d), dtype=f64, device=dev)
    lse = torch.empty((2, B, nW, heads, L), dtype=f64, device=dev)
    if backward:
        out_D = torch.empty((B, H * W, heads), dtype=f64, device=dev)
        dqkv = torch.empty((B, H * W, 3, heads, d), dtype=f64, device=dev)
        dscale = torch.zeros((heads,), dtype=f64, device=dev)
        dscale_c = torch.zeros((heads,), dtype=f64, device=dev)
        dbias = torch.zeros((heads, L, L), dtype=f64, device=dev) if bias is not None else None

    cw = max(1, min(nW, _CHUNK_LOGITS // (B * L * L)))
    for h in range(heads):
        sc = float(scale[h])
        for w0 in range(0, nW, cw):
            ix = idx[w0:w0 + cw]                                                     # (cw, L)
            flat = ix.reshape(-1)

            def rows(t, *sel):                                                       # (B, cw, L, d) fp64
                return t[(slice(None), flat) + sel].to(f64).view(B, ix.shape[0], L, -1)

            q, k, v = rows(x, 0, h), rows(x, 1, h), rows(x, 2, h)
            cos = q @ k.transpose(-1, -2)                                            # (B, cw, L, L)
            s = sc * cos
            if bias is not None:
                s = s + bias[h].to(f64)
            if mask is not None:
                s = s + mask[w0:w0 + cw]
            m = torch.logsumexp(s, dim=-1, keepdim=True)
            p = torch.exp(s - m)
            out_o[:, flat, h] = (p @ v).reshape(B, -1, d)
            lse[0, :, w0:w0 + cw, h] = m.squeeze(-1)
            ec = (p * cos).sum(-1, keepdim=True)
            lse[1, :, w0:w0 + cw, h] = ec.squeeze(-1)
            if not backward:
                continue
            g = rows(go, h)
            Dv = (g * rows(oo, h)).sum(-1, keepdim=True)                            # (B, cw, L, 1)
            out_D[:, flat, h] = Dv.reshape(B, -1)
            ds = p * (g @ v.transpose(-1, -2) - Dv)
            dqh = sc * (ds @ k)
            dkh = sc * (ds.transpose(-1, -2) @ q)
            inq = rows(inv, 0, h)                                                    # (B, cw, L, 1)
            ink = rows(inv, 1, h)
            dqkv[:, flat, 0, h] = (inq * (dqh - q * (q * dqh).sum(-1, keepdim=True))).reshape(B, -1, d)
            dqkv[:, flat, 1, h] = (ink * (dkh - k * (k * dkh).sum(-1, keepdim=True))).reshape(B, -1, d)
            dqkv[:, flat, 2, h] = (p.transpose(-1, -2) @ g).reshape(B, -1, d)
            dscale[h] += (ds * cos).sum()
            dscale_c[h] += (ds * (cos - ec)).sum()
            if dbias is not None:
                dbias[h] += ds.sum(dim=(0, 1))

    res = {"o": out_o.view(T, C), "lse": lse}
    if backward:
        res.update(D=out_D.view(T, heads), dqkv=dqkv.view(T, 3 * C), dscale=dscale, dscale_centred=dscale_c, dbias=dbias)
    return res
