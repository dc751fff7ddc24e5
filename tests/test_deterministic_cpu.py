"""CPU: the deterministic-mode entry points reject bad arguments and short scratch, and ops.py picks them exactly when
torch.use_deterministic_algorithms(True) is in force (the C ABI is replaced by a recorder: no kernel runs)."""
import ctypes

import pytest
import torch

from swin_v2_weather_b200 import _lib, ops
from swin_v2_weather_b200.ops import EPI_F32, MODE_BF16, MODE_FP32

P = ctypes.c_void_p(16)


def test_entry_points_reject_null_or_short_scratch():
    lib = _lib.load()
    cases = [
        (lambda part, n: lib.swinb200_gemm_wgrad_det(1, 256, 256, 1024, P, 256, P, 256, 1, P, 4, part, n, None), 4 * 256 * 256),
        (lambda part, n: lib.swinb200_linear_wgrad_det(1, 256, 256, 1024, P, 256, P, 256, P, P, 4, part, n, None), 4 * (256 * 256 + 256)),
        (lambda part, n: lib.swinb200_ln_residual_bwd_det(P, P, 1, P, P, None, P, P, P, P, 100, 768, 100, part, n, None),
         3 * 768 * 256 * 2),
        (lambda part, n: lib.swinb200_colsum_det(P, 1, P, 6400, 768, 768, part, n, None), 768 * 100),
        (lambda part, n: lib.swinb200_latw_l2_fwd_det(P, P, P, P, 1, 1, P, P, P, 2, 3, 720, 1440, part, n, None), 2 * 2 * 3 * 720),
        (lambda part, n: lib.swinb200_latw_l1_fwd_det(P, P, P, P, 1, P, P, 2, 3, 720, 1440, part, n, None), 2 * 2 * 3 * 720),
        (lambda part, n: lib.swinb200_latw_acc_det(P, P, P, P, P, 2, 3, 720, 1440, part, n, None), 3 * 2 * 3 * 720),
        (lambda part, n: lib.swinb200_window_attn_bwd_det(1, P, 1, P, P, P, P, P, P, P, P, P, P, 1, 180, 360, 768, 8, 9, 18, 0, 0,
                                                          part, n, None), 400 * 8 * (4 * 2 + 162 * 162)),
    ]
    for fn, need in cases:
        assert fn(None, need) == _lib.ERR_INVALID_ARG
        assert b"scratch" in lib.swinb200_last_error()
        assert fn(P, need - 1) == _lib.ERR_INVALID_ARG
        assert b"scratch" in lib.swinb200_last_error()


def test_ordered_reduce_rejects_bad_layout():
    lib = _lib.load()
    assert lib.swinb200_ordered_reduce(None, 4, 16, 16, 1, P, 0, None) == _lib.ERR_INVALID_ARG
    assert lib.swinb200_ordered_reduce(P, 4, 16, 16, 2, P, 0, None) == _lib.ERR_INVALID_ARG     # stride < n * inner
    assert lib.swinb200_ordered_reduce(P, 0, 16, 16, 1, P, 0, None) == _lib.ERR_INVALID_ARG
    assert b"ordered_reduce" in lib.swinb200_last_error()


def test_wgrad_det_rejects_what_it_is_not_built_for():
    lib = _lib.load()
    # the fused weight + bias gradient exists for n_out a multiple of 256 only, as the plain entry point
    assert lib.swinb200_linear_wgrad_det(1, 200, 256, 64, P, 200, P, 256, P, P, 2, P, 1 << 20, None) == _lib.ERR_UNSUPPORTED
    assert lib.swinb200_window_attn_bwd_det(1, P, 1, P, P, None, P, P, P, P, P, P, P, 1, 36, 72, 768, 8, 9, 18, 0, 0, P, 1 << 30,
                                            None) == _lib.ERR_INVALID_ARG        # dbias without the bias table
    assert b"bias table" in lib.swinb200_last_error()


def test_tcgen05_attention_rejects_missing_workspace_or_unaligned_operands():
    """The tcgen05 attention needs the D = <dO, O> workspace and 16-byte aligned operands at every geometry, in the plain and
    the deterministic entry points alike; here at the shipped 9x18 windows / head_dim 96."""
    lib = _lib.load()
    tc, bf16, geom = _lib.BACKEND_TCGEN05, _lib.BF16, (1, 36, 72, 768, 8, 9, 18, 0, 0)
    U = ctypes.c_void_p(18)

    def bwd(qkv, ws):
        return lib.swinb200_window_attn_bwd(tc, qkv, bf16, P, P, None, P, P, P, P, P, None, ws, *geom, None)

    def bwd_det(ws):
        return lib.swinb200_window_attn_bwd_det(tc, P, bf16, P, P, None, P, P, P, P, P, None, ws, *geom, P, 1 << 30, None)

    for call in (lambda: bwd(P, None), lambda: bwd_det(None)):
        assert call() == _lib.ERR_INVALID_ARG
        assert b"workspace" in lib.swinb200_last_error()
    for call in (lambda: lib.swinb200_window_attn_fwd(tc, U, bf16, P, None, P, P, *geom, None), lambda: bwd(U, P)):
        assert call() == _lib.ERR_INVALID_ARG
        assert b"16-byte aligned" in lib.swinb200_last_error()


@pytest.fixture
def recorder(monkeypatch):
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *args: calls.append(name))
    monkeypatch.setattr(ops, "_chk", lambda t, *a, **k: 0 if t is None else 16)
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    return calls


@pytest.fixture(params=[False, True], ids=["flag_off", "flag_on"])
def flag(request):
    old = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(request.param)
    yield request.param
    torch.use_deterministic_algorithms(old)


def _each_op():
    f, b = torch.float32, torch.bfloat16
    prd, tar = torch.zeros(1, 2, 8, 16), torch.zeros(1, 2, 8, 16)
    qw, chw = torch.ones(8), torch.ones(2)
    L = 162
    yield "swinb200_gemm", lambda: ops.gemm(MODE_BF16, torch.zeros(512, 256, dtype=b), 1, torch.zeros(512, 128, dtype=b), 1, EPI_F32,
                                            out=torch.zeros(256, 128), accumulate=True, split_k=4)
    yield "swinb200_linear_wgrad", lambda: ops.linear_wgrad(MODE_BF16, torch.zeros(512, 256, dtype=b), torch.zeros(512, 256, dtype=b),
                                                            torch.zeros(256, 256), torch.zeros(256), 4)
    yield "swinb200_ln_residual_bwd", lambda: ops.ln_residual_bwd(torch.zeros(64, 768), torch.zeros(64, 768, dtype=b),
                                                                  torch.zeros(64, 2), torch.ones(768), None, 64, MODE_BF16)
    yield "swinb200_colsum", lambda: ops.colsum(torch.zeros(64, 256))
    yield "swinb200_latw_l2_fwd", lambda: ops.latw_l2_fwd(prd, tar, qw, chw, True)
    yield "swinb200_latw_l1_fwd", lambda: ops.latw_l1_fwd(prd, tar, qw, chw, True)
    yield "swinb200_latw_acc", lambda: ops.latw_acc(prd, tar, qw)
    yield "swinb200_window_attn_bwd", lambda: ops.window_attn_bwd(
        torch.zeros(36 * 72, 3 * 192, dtype=f), torch.zeros(36 * 72, 4), torch.ones(2), torch.zeros(2, L, L), torch.zeros(36 * 72, 192),
        torch.zeros(36 * 72, 192), torch.zeros(2, 1, 16, 2, L), 1, 36, 72, 192, 2, 9, 18, 0, 0, MODE_FP32)


@pytest.mark.parametrize("entry,fn", list(_each_op()), ids=[e for e, _ in _each_op()])
def test_flag_selects_the_entry_point(recorder, flag, entry, fn):
    fn()
    det_entry = "swinb200_gemm_wgrad_det" if entry == "swinb200_gemm" else entry + "_det"
    assert recorder == [det_entry if flag else entry]


def test_split_k_one_keeps_the_plain_gemm(recorder, flag):
    """A single split adds each element of D once: the plain kernel is already deterministic."""
    b = torch.bfloat16
    ops.gemm(MODE_BF16, torch.zeros(512, 256, dtype=b), 1, torch.zeros(512, 128, dtype=b), 1, EPI_F32, out=torch.zeros(256, 128),
             accumulate=True, split_k=1)
    assert recorder == ["swinb200_gemm"]
