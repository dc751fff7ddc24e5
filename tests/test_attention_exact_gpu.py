"""Window attention kernels against the fp64 reference on their own stored inputs (oracle/attention_exact.py).

The parity tests of test_kernels_gpu.py feed their fp32 oracle the raw qkv, so their bars absorb the bf16 rounding of q^ / k^
(1e-2 .. 6e-2).  Here the reference reads exactly what the kernel reads -- the stored q^ / k^ / v, inv_norm, the o and d_o the
backward is handed -- so the bars below are set by the kernels' own arithmetic, a few times over what the B200 measured.

Each case calls the C ABI directly (as ops.py does) with buffers the test owns:
  * inputs (qkv, o, d_o, lse, inv_norm, bias) sit inside allocations with NaN margins of 4,096 elements on each side;
  * outputs (o, both lse planes, dqkv) are NaN inside and a sentinel in their margins: afterwards no NaN may be left inside
    (every element written) and the margins must be bitwise unchanged (nothing written outside);
  * the accumulators dscale / dbias start from a non-zero base (the ABI adds to them); the same margins guard them;
  * the backward workspace `ws` and the deterministic `part` scratch are NaN-filled (read before written would show).
Every tensor start is 256-byte aligned.

Metrics, per case:
  * o, dq, dk, dv: a per-window-row profile -- for each row slot i of the window, the largest error over (sample, window,
    head) of that row, divided by the RMS row norm of its (sample, window, head) item.  Asserted on its maximum; the
    failure message splits it into the first 128-row tile and the remainder tile.  In bf16 its floor is the rounding of
    the stored output itself, and it grows with the number of rows the maximum runs over.
  * o, dq, dk, dv (_l2): relative L2 error of the whole tensor, the metric of the parity tests (bars 1e-2 / 2e-2 there).
    A kernel that rounded its fp64-exact result to bf16 and nothing else would measure about 1.7e-3 here.
  * lse plane 0 (LSE) and plane 1 (E_P[cos]): absolute error.  The CUDA-core back end defines plane 1 as exactly zero.
  * dscale, dbias: relative error per head.  The tcgen05 back end is compared with the centred d(scale), the CUDA-core back
    end with the plain one (oracle/attention_exact.py explains the difference).
Cases that make a quantity zero by construction skip it (SKIP below).

Bars: about 3x the worst value measured over the case list on one NVIDIA B200 (1000 W power limit); the whole file took 9.3 s
there.  bf16 = the tcgen05 kernels and the CUDA-core kernels in bf16 storage; fp32 = the CUDA-core kernels in fp32 storage.

    metric   bf16 worst measured (case)            bar       fp32 worst measured (case)              bar
    o        1.49e-2 (full-e2048)                  4e-2      2.30e-6 (simt-f32-d256-162-globalkv)    6e-6
    dq       1.80e-2 (full-e768)                   5e-2      2.92e-6 (det-simt-f32)                  8e-6
    dk       1.92e-2 (full-e768)                   5e-2      2.55e-6 (simt-f32-d256-162-globalkv)    7e-6
    dv       1.51e-2 (full-e2048)                  4e-2      2.37e-6 (simt-f32-d256-162-globalkv)    7e-6
    o_l2     2.39e-3 (tiled-d64-72)                5e-3      3.83e-7 (simt-f32-d96-162)              1e-6
    dq_l2    2.38e-3 (bound-41-fwd4)               5e-3      5.13e-7 (simt-f32-d256-162-globalkv)    1.5e-6
    dk_l2    2.42e-3 (exact-42-fwd4)               5e-3      5.16e-7 (simt-f32-d256-162-globalkv)    1.5e-6
    dv_l2    2.38e-3 (tiled-d48-162)               5e-3      4.16e-7 (simt-f32-d96-162)              1.2e-6
    lse0     1.08e-5 (exact-100-fwd4)              3e-5      1.13e-6 (det-simt-f32)                  3e-6
    lse1     4.08e-6 (antiparallel-41-fwd4)        1.2e-5    0 (CUDA-core kernels, bf16 too)         0
    dscale   7.79e-5 (rescale-spike-d96)           2e-4      2.34e-6 (simt-f32-d96-162)              6e-6
    dbias    1.41e-6 (rescale-spike-d96)           4e-6      4.93e-7 (simt-f32-d256-162-globalkv)    1.4e-6
"""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import swinv2_oracle as O
from oracle.attention_exact import attention_exact
from swin_v2_weather_b200 import _lib
from swin_v2_weather_b200._lib import BACKEND_SIMT, BACKEND_TCGEN05, BF16, F32

pytestmark = pytest.mark.gpu
DEV = "cuda"
MARGIN = 4096

BARS = {
    torch.bfloat16: dict(o=4e-2, dq=5e-2, dk=5e-2, dv=4e-2, o_l2=5e-3, dq_l2=5e-3, dk_l2=5e-3, dv_l2=5e-3, lse0=3e-5, lse1=1.2e-5,
                         dscale=2e-4, dbias=4e-6),
    torch.float32: dict(o=6e-6, dq=8e-6, dk=7e-6, dv=7e-6, o_l2=1e-6, dq_l2=1.5e-6, dk_l2=1.5e-6, dv_l2=1.2e-6, lse0=3e-6,
                        lse1=0.0, dscale=6e-6, dbias=1.4e-6),
}


# ---- buffers the test owns ---------------------------------------------------------------------------------------------
class Guarded:
    """A tensor inside a larger allocation: `margin` fill on both sides of `inside`, start 256-byte aligned."""

    def __init__(self, shape, dtype, inside, margin):
        n = math.prod(shape)
        es = torch.empty((), dtype=dtype).element_size()
        self.base = torch.full((n + 2 * MARGIN + 256 // es,), margin, dtype=dtype, device=DEV)
        self.lo = MARGIN + (-(self.base.data_ptr() + MARGIN * es) % 256) // es
        self.hi = self.lo + n
        self.t = self.base[self.lo:self.hi].view(shape)
        if isinstance(inside, torch.Tensor):
            self.t.copy_(inside.reshape(shape))
        else:
            self.t.fill_(inside)
        assert self.t.data_ptr() % 256 == 0
        self.edges = self._edges().clone()

    def _edges(self):
        b = self.base.view(torch.int16 if self.base.element_size() == 2 else torch.int32)
        return torch.cat([b[:self.lo], b[self.hi:]])

    @property
    def ptr(self):
        return self.t.data_ptr()

    def check(self, name, written=False):
        assert torch.equal(self._edges(), self.edges), f"{name}: something was written outside the tensor"
        if written:
            bad = int(torch.isnan(self.t).sum())
            assert bad == 0, f"{name}: {bad} of {self.t.numel()} elements never written"


def guarded_in(x):
    return Guarded(tuple(x.shape), x.dtype, x, float("nan"))


def guarded_out(shape, dtype):
    return Guarded(shape, dtype, float("nan"), -1234.5)


# ---- cases -------------------------------------------------------------------------------------------------------------
def case(why, H, W, C, heads, window, shift=None, bias=False, B=2, dtype=torch.bfloat16, backend=BACKEND_TCGEN05,
         scale=None, det=False, kind="random", spike=False):
    if shift is None:
        shift = (window[0] // 2, window[1] // 2)
    return pytest.param(dict(H=H, W=W, C=C, heads=heads, window=window, shift=shift, bias=bias, B=B, dtype=dtype,
                             backend=backend, scale=scale, det=det, kind=kind, spike=spike), id=why)


CASES = [
    # tuned kernels (head_dim 96, LP <= 176): fwd4 without a bias table, bwd3 always
    case("tuned-162-box", 18, 36, 192, 2, (9, 18), shift=(0, 0)),
    case("tuned-162-shift", 18, 36, 192, 2, (9, 18), shift=(4, 9)),
    case("tuned-162-shift-bias", 18, 36, 192, 2, (9, 18), shift=(4, 9), bias=True),
    case("tuned-162-box-bias", 18, 36, 192, 2, (9, 18), shift=(0, 0), bias=True),
    case("tuned-72-fwd4", 12, 24, 192, 2, (6, 12)),
    case("tuned-128-one-tile", 16, 32, 192, 2, (8, 16)),
    case("tuned-176-maxLP", 22, 32, 192, 2, (11, 16), bias=True),
    # tiled kernels
    case("tiled-d96-180", 20, 36, 192, 2, (10, 18)),
    case("tiled-d48-72", 12, 24, 96, 2, (6, 12), bias=True),
    case("tiled-d48-162", 18, 36, 96, 2, (9, 18)),
    case("tiled-d48-288", 24, 48, 96, 2, (12, 24), shift=(0, 0), bias=True),
    case("tiled-d64-72", 12, 24, 128, 2, (6, 12), shift=(0, 0)),
    case("tiled-d64-162", 18, 36, 128, 2, (9, 18), bias=True),
    case("tiled-d64-288", 24, 48, 128, 2, (12, 24)),
    case("tiled-d128-72", 12, 24, 256, 2, (6, 12)),
    case("tiled-d128-162", 18, 36, 256, 2, (9, 18), shift=(0, 0), bias=True),
    case("tiled-d128-288", 24, 48, 256, 2, (12, 24), bias=True),
    case("tiled-d192-72", 12, 24, 384, 2, (6, 12), bias=True),
    case("tiled-d192-162", 18, 36, 384, 2, (9, 18)),
    case("tiled-d192-288", 24, 48, 384, 2, (12, 24), shift=(0, 0)),
    case("tiled-d64-648", 36, 72, 128, 2, (18, 36), bias=True),
    case("tiled-d256-162", 18, 36, 512, 2, (9, 18), bias=True),
    case("tiled-d256-72", 12, 24, 512, 2, (6, 12)),
    case("tiled-d256-288", 24, 48, 512, 2, (12, 24), bias=True),
    # softmax paths: the bound offset below scale*log2e = 60 (scale 41.59), the exact maximum above
    case("bound-41-fwd4", 18, 36, 192, 2, (9, 18), shift=(0, 0), scale=41.0),
    case("exact-42-fwd4", 18, 36, 192, 2, (9, 18), shift=(0, 0), scale=42.0),
    case("exact-100-fwd4", 18, 36, 192, 2, (9, 18), shift=(0, 0), scale=100.0),
    case("bound-41-tiled", 18, 36, 128, 2, (9, 18), shift=(0, 0), scale=41.0),
    case("exact-42-tiled", 18, 36, 128, 2, (9, 18), shift=(0, 0), scale=42.0),
    case("exact-100-tiled", 18, 36, 128, 2, (9, 18), shift=(4, 9), scale=100.0),
    case("rescale-spike-d96", 18, 36, 192, 2, (9, 18), shift=(4, 9), bias=True, spike=True),
    case("rescale-spike-d64-288", 24, 48, 128, 2, (12, 24), bias=True, spike=True),
    case("ties-fwd4", 18, 36, 192, 2, (9, 18), kind="ties"),
    case("ties-tiled", 18, 36, 128, 2, (9, 18), kind="ties"),
    case("antiparallel-41-fwd4", 18, 36, 192, 2, (9, 18), shift=(4, 9), scale=41.0, kind="antiparallel"),
    case("antiparallel-41-tiled", 18, 36, 128, 2, (9, 18), shift=(4, 9), scale=41.0, kind="antiparallel"),
    # CUDA-core kernels (GLOBAL_KV: the window's K / V rows do not fit in shared memory)
    case("simt-f32-d96-162", 18, 36, 192, 2, (9, 18), bias=True, dtype=torch.float32, backend=BACKEND_SIMT),
    case("simt-f32-d256-162-globalkv", 18, 36, 512, 2, (9, 18), bias=True, dtype=torch.float32, backend=BACKEND_SIMT),
    case("simt-bf16-d64-72", 12, 24, 128, 2, (6, 12), dtype=torch.bfloat16, backend=BACKEND_SIMT),
    case("simt-bf16-d256-288-globalkv", 24, 48, 512, 2, (12, 24), bias=True, backend=BACKEND_SIMT),
    # deterministic backward
    case("det-bwd3", 18, 36, 192, 2, (9, 18), shift=(4, 9), bias=True, det=True),
    case("det-tiled", 18, 36, 128, 2, (9, 18), bias=True, det=True),
    case("det-tiled-d256", 12, 24, 512, 2, (6, 12), bias=True, det=True),
    case("det-simt-f32", 12, 24, 128, 2, (6, 12), bias=True, dtype=torch.float32, backend=BACKEND_SIMT, det=True),
    # the two shipped configurations at full size
    case("full-e768", 180, 360, 768, 8, (9, 18), shift=(4, 9), bias=True, B=1),
    case("full-e768-nobias", 180, 360, 768, 8, (9, 18), shift=(4, 9), B=1),
    case("full-e2048", 180, 360, 2048, 8, (9, 18), shift=(4, 9), bias=True, B=1),
]


def make_inputs(cfg, seed):
    """Raw qkv -> stored (q^, k^, v) in the storage type, inv_norm, scale, bias, d_o."""
    B, H, W, C, heads = cfg["B"], cfg["H"], cfg["W"], cfg["C"], cfg["heads"]
    Wh, Ww = cfg["window"]
    d, L, T = C // heads, Wh * Ww, B * H * W
    g = torch.Generator().manual_seed(seed)
    raw = torch.randn(T, 3, heads, d, generator=g)
    if cfg["kind"] in ("ties", "antiparallel"):
        u = torch.randn(heads, d, generator=g)
        raw[:, 1] = u                                    # every k^ of every window equal: all logits of a row tie
        if cfg["kind"] == "antiparallel":
            raw[:, 0] = -u                               # every cosine -1, masked or not
    raw = raw.to(DEV)
    qk = raw[:, :2]
    inv = (1.0 / qk.norm(dim=-1).clamp_min(1e-12)).contiguous()                    # (T, 2, heads)
    qkv = torch.cat([F.normalize(qk, dim=-1), raw[:, 2:]], dim=1).reshape(T, 3 * C).to(cfg["dtype"])
    if cfg["scale"] is not None:
        scale = torch.full((heads,), float(cfg["scale"]), device=DEV)
    else:
        scale = torch.linspace(8.0, 14.0, heads, device=DEV)
    bias = None
    if cfg["bias"]:
        bias = torch.randn(heads, L, L, generator=g)
        if cfg["spike"]:
            # +30 on the keys of the last, ragged 64-key tile for every third query: the running maximum grows by far more than
            # 2^8 on that tile for some rows of a warp and not for others
            last = (L - 1) // 64 * 64
            bias[:, ::3, last:] += 30.0
        bias = bias.to(DEV)
    d_o = torch.randn(T, C, generator=g).to(DEV).to(cfg["dtype"])
    return qkv, inv, scale, bias, d_o


def window_rows(x, cfg):
    """(T, heads*d) -> (B, nW, heads, L, d) fp64, rows in window-slot order."""
    B, H, W, heads = cfg["B"], cfg["H"], cfg["W"], cfg["heads"]
    idx = O.window_token_index((H, W), cfg["window"], cfg["shift"]).to(x.device)
    nW, L = idx.shape
    t = x.double().view(B, H * W, heads, -1)[:, idx.reshape(-1)]
    return t.view(B, nW, L, heads, -1).permute(0, 1, 3, 2, 4)


def row_profile(got, ref, cfg):
    """max over (sample, window, head) of |row error| / RMS row norm of the item, per window slot -> (L,)"""
    g, r = window_rows(got, cfg), window_rows(ref, cfg)
    err = (g - r).norm(dim=-1)
    rms = r.norm(dim=-1).pow(2).mean(dim=-1, keepdim=True).sqrt()
    return (err / rms.clamp_min(1e-300)).amax(dim=(0, 1, 2))


def split(prof):
    head = f"[0,128) {float(prof[:128].max()):.2e}"
    return head if prof.numel() <= 128 else head + f"  [128,{prof.numel()}) {float(prof[128:].max()):.2e}"


def run_case(cfg):
    B, H, W, C, heads = cfg["B"], cfg["H"], cfg["W"], cfg["C"], cfg["heads"]
    Wh, Ww = cfg["window"]
    s0, s1 = cfg["shift"]
    dt, be = cfg["dtype"], cfg["backend"]
    act = BF16 if dt == torch.bfloat16 else F32
    L, T = Wh * Ww, B * H * W
    nW = (H // Wh) * (W // Ww)
    items = B * nW * heads
    geom = (B, H, W, C, heads, Wh, Ww, s0, s1)
    stream = torch.cuda.current_stream().cuda_stream
    qkv, inv, scale, bias, d_o = make_inputs(cfg, seed=hash(tuple(geom)) % 1000 + 7)

    # forward
    g_qkv = guarded_in(qkv)
    g_bias = guarded_in(bias) if bias is not None else None
    g_o = guarded_out((T, C), dt)
    g_lse = guarded_out((2, B, nW, heads, L), torch.float32)
    _lib.call("swinb200_window_attn_fwd", be, g_qkv.ptr, act, scale.data_ptr(), g_bias.ptr if g_bias else 0, g_o.ptr, g_lse.ptr,
              *geom, stream)
    torch.cuda.synchronize()
    g_o.check("o", written=True)
    g_lse.check("lse", written=True)

    # backward on the forward's own o and lse
    g_oin, g_lsein, g_do, g_inv = guarded_in(g_o.t), guarded_in(g_lse.t), guarded_in(d_o), guarded_in(inv)
    g_dqkv = guarded_out((T, 3 * C), dt)
    base_s = 0.0625 * torch.arange(1, heads + 1, dtype=torch.float32, device=DEV)
    base_b = torch.full((heads, L, L), 2.0 ** -6, device=DEV)
    g_dscale = Guarded((heads,), torch.float32, base_s, -1234.5)
    g_dbias = Guarded((heads, L, L), torch.float32, base_b, -1234.5) if bias is not None else None
    ws = torch.full((T * heads,), float("nan"), device=DEV)
    args = [be, g_qkv.ptr, act, g_inv.ptr, scale.data_ptr(), g_bias.ptr if g_bias else 0, g_oin.ptr, g_do.ptr, g_lsein.ptr,
            g_dqkv.ptr, g_dscale.ptr, g_dbias.ptr if g_dbias else 0, ws.data_ptr(), *geom]
    if cfg["det"]:
        part = torch.full((items * (4 * ((L + 127) // 128) + (L * L if bias is not None else 0)),), float("nan"), device=DEV)
        _lib.call("swinb200_window_attn_bwd_det", *args, part.data_ptr(), part.numel(), stream)
    else:
        _lib.call("swinb200_window_attn_bwd", *args, stream)
    torch.cuda.synchronize()
    g_dqkv.check("dqkv", written=True)
    g_dscale.check("dscale", written=True)
    if g_dbias is not None:
        g_dbias.check("dbias", written=True)
    for name, gi in (("qkv", g_qkv), ("bias", g_bias), ("o (in)", g_oin), ("lse (in)", g_lsein), ("d_o", g_do), ("inv_norm", g_inv)):
        if gi is not None:
            gi.check(name)

    ref = attention_exact(qkv, scale, bias, g_o.t, d_o, inv, *geom)
    got_lse = g_lse.t.double()
    m, info = {}, {}
    for name, got, want in (("o", g_o.t, ref["o"]), ("dq", g_dqkv.t[:, :C], ref["dqkv"][:, :C]),
                            ("dk", g_dqkv.t[:, C:2 * C], ref["dqkv"][:, C:2 * C]), ("dv", g_dqkv.t[:, 2 * C:], ref["dqkv"][:, 2 * C:])):
        prof = row_profile(got, want, cfg)
        m[name], info[name] = float(prof.max()), split(prof)
        m[name + "_l2"] = float((got.double() - want).norm() / want.norm())
    e0 = (got_lse[0] - ref["lse"][0]).abs().amax(dim=(0, 1, 2))
    m["lse0"], info["lse0"] = float(e0.max()), split(e0)
    if be == BACKEND_SIMT:
        m["lse1"] = float(got_lse[1].abs().max())                                   # defined as exactly zero
    else:
        e1 = (got_lse[1] - ref["lse"][1]).abs().amax(dim=(0, 1, 2))
        m["lse1"], info["lse1"] = float(e1.max()), split(e1)
    want_s = ref["dscale"] if be == BACKEND_SIMT else ref["dscale_centred"]
    m["dscale"] = float(((g_dscale.t.double() - base_s.double() - want_s).abs() / want_s.abs()).max())
    if bias is not None:
        db = g_dbias.t.double() - base_b.double() - ref["dbias"]
        m["dbias"] = float((db.flatten(1).norm(dim=1) / ref["dbias"].flatten(1).norm(dim=1)).max())
    return m, info


# In the constructed cases a quantity can be zero by construction, so that only rounding is left to compare; those are skipped:
# equal keys make every dq^ a multiple of the shared k^ scaled by sum_j dS_ij (zero up to the rounding of o), and d(scale) the
# constant cosine times the same sums; with q^ = -k^ as well, dk^ lies along k^ and the normalisation backward removes it.
SKIP = {"ties": ("dq", "dq_l2", "dscale"), "antiparallel": ("dq", "dq_l2", "dk", "dk_l2", "dscale")}


@pytest.mark.parametrize("cfg", CASES)
def test_attention_exact(cfg):
    m, info = run_case(cfg)
    bars = dict(BARS[cfg["dtype"]])
    if cfg["backend"] == BACKEND_SIMT:
        bars["lse1"] = 0.0
    skip = SKIP.get(cfg["kind"], ())
    line = "  ".join(f"{k} {v:.2e}" + (" (skipped)" if k in skip else "") for k, v in m.items())
    print(f"\nMEASURED {cfg['dtype']} {line}")
    for k, v in info.items():
        print(f"  {k:6s} {v}")
    bad = {k: v for k, v in m.items() if k not in skip and not v <= bars[k]}
    assert not bad, {k: (v, bars[k], info.get(k)) for k, v in bad.items()}
