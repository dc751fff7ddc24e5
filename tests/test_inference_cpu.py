"""CPU: which C-ABI calls the model issues when no gradient will be taken (forward-only path) and when one will (training
path), with the library replaced by a recorder: no kernel runs."""
import ctypes
import os
import re

import pytest
import torch
from torch.utils.checkpoint import checkpoint

from swin_v2_weather_b200 import _lib, functional as Fn, ops
from swin_v2_weather_b200.networks.swinv2_global import SwinTransformerV2Cr, SwinTransformerV2CrBlock

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = ctypes.c_void_p(16)

# argument positions of the optional statistics outputs (include/swinb200.h)
STATS_ARG = {"swinb200_ln_residual_fwd": 9, "swinb200_qk_normalize": 2, "swinb200_window_attn_fwd": 6}
GEMM_EPI, GEMM_D2 = 11, 15


@pytest.fixture
def recorder(monkeypatch):
    """Every _lib.call as (name, args); tensors cross as their data_ptr (CPU tensors stand in for device memory)."""
    calls = []
    monkeypatch.setattr(_lib, "call", lambda name, *args: calls.append((name, args)))
    monkeypatch.setattr(ops, "_chk", lambda t, *a, **k: 0 if t is None else t.data_ptr())
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    Fn.SHADOWS.clear()
    yield calls
    Fn.SHADOWS.clear()


def summary(calls):
    """(entry point, epilogue or None, statistics pointer given?) per call, shadow casts left out."""
    out = []
    for name, args in calls:
        if name == "swinb200_cast_f32_to_bf16":
            continue
        if name == "swinb200_gemm":
            epi = args[GEMM_EPI]
            out.append((name, epi, bool(args[GEMM_D2]) if epi in (_lib.EPI_BIAS_GELU, _lib.EPI_BIAS_QKNORM) else None))
        elif name in STATS_ARG:
            out.append((name, None, bool(args[STATS_ARG[name]])))
        else:
            out.append((name, None, None))
    return out


def make_block(mode, C=192, heads=2, drop_path=0.0, rel_pos=False):
    torch.manual_seed(0)
    return SwinTransformerV2CrBlock(dim=C, num_heads=heads, feat_size=(18, 36), window_size=(9, 18), shift_size=(4, 9),
                                    mlp_ratio=4.0, drop_path=drop_path, rel_pos=rel_pos, compute_mode=mode)


G, B_, D2, QK = _lib.EPI_BIAS_GELU, _lib.EPI_BIAS, _lib.EPI_BIAS_QKNORM, _lib.EPI_BIAS_GELU_FWD

# the training forward of one block, as the parent revision issues it
TRAIN_TC96 = [("swinb200_gemm", D2, True), ("swinb200_window_attn_fwd", None, True), ("swinb200_gemm", B_, None),
              ("swinb200_ln_residual_fwd", None, True), ("swinb200_gemm", G, True), ("swinb200_gemm", B_, None),
              ("swinb200_ln_residual_fwd", None, True)]
TRAIN_SIMT = [("swinb200_gemm", B_, None), ("swinb200_qk_normalize", None, True)] + TRAIN_TC96[1:]


def forward_only_of(seq):
    """The forward-only sequence: the same calls, fc1 on BIAS_GELU_FWD, no statistics."""
    out = []
    for name, epi, st in seq:
        if epi == G:
            out.append((name, QK, None))
        else:
            out.append((name, epi, False if st is not None else None))
    return out


@pytest.mark.parametrize("mode,train_seq", [("bf16", TRAIN_TC96), ("bf16_simt", TRAIN_SIMT), ("fp32", TRAIN_SIMT)])
def test_block_sequences(recorder, mode, train_seq):
    blk = make_block(mode)
    x = torch.randn(1, 18, 36, 192)
    blk(x.requires_grad_())
    assert summary(recorder) == train_seq
    recorder.clear()
    with torch.no_grad():
        blk(x)
    fo = summary(recorder)
    assert fo == forward_only_of(train_seq)
    assert ("swinb200_gemm", QK, None) in fo and all(e != G for _, e, _ in fo)
    recorder.clear()
    with torch.inference_mode():
        blk(x.detach())
    assert summary(recorder) == fo


def test_block_without_any_grad_requirement_takes_the_forward_only_path(recorder):
    """Grad mode on, but neither the input nor a parameter requires grad: nothing can be differentiated."""
    blk = make_block("bf16").requires_grad_(False)
    blk(torch.randn(1, 18, 36, 192))
    assert summary(recorder) == forward_only_of(TRAIN_TC96)
    recorder.clear()
    blk.mlp.fc2.weight.requires_grad_(True)          # one trainable parameter is enough for the training path
    blk(torch.randn(1, 18, 36, 192))
    assert summary(recorder) == TRAIN_TC96


def test_dropout_draws_keep_their_order(recorder):
    """model.train() under no_grad: CPB hidden dropout and both DropPath masks are drawn exactly as on the training path."""
    blk = make_block("bf16", drop_path=0.3, rel_pos=True).train()
    x = torch.randn(4, 18, 36, 192)
    torch.manual_seed(7)
    blk(x.requires_grad_())
    state_train = torch.get_rng_state()
    dp_train = [a for n, a in recorder if n == "swinb200_ln_residual_fwd"]
    recorder.clear()
    torch.manual_seed(7)
    with torch.no_grad():
        blk(x)
    assert torch.equal(torch.get_rng_state(), state_train)
    dp_fo = [a for n, a in recorder if n == "swinb200_ln_residual_fwd"]
    assert [bool(a[5]) for a in dp_fo] == [bool(a[5]) for a in dp_train] == [True, True]     # sample_scale given


def test_checkpointed_training_keeps_the_training_path(recorder):
    blk = make_block("bf16")
    x = torch.randn(1, 18, 36, 192, requires_grad=True)
    checkpoint(blk, x, use_reentrant=False)
    assert summary(recorder) == TRAIN_TC96
    recorder.clear()
    with torch.no_grad():
        checkpoint(blk, x, use_reentrant=False)
    assert summary(recorder) == forward_only_of(TRAIN_TC96)


def small_model(checkpoint_stages=False):
    torch.manual_seed(0)
    return SwinTransformerV2Cr(img_size=(72, 144), patch_size=4, depths=(2,), num_heads=(2,), in_chans=7, out_chans=5,
                               embed_dim=192, img_window_ratio=8, full_pos_embed=True, rel_pos=False, residual=True,
                               checkpoint_stages=checkpoint_stages, compute_mode="bf16")


def test_model_forward_only(recorder):
    """PatchEmbed and head too: the LayerNorm after the patch projection stores no statistics, and pos_embed is transposed
    once and then taken from the shadow cache until the parameter changes."""
    model = small_model()
    x = torch.randn(1, 7, 72, 144)
    model(x)
    train = [n for n, _ in recorder if n != "swinb200_cast_f32_to_bf16"]
    recorder.clear()
    with torch.no_grad():
        model(x)
        first = [n for n, _ in recorder if n != "swinb200_cast_f32_to_bf16"]
        assert first == train                                    # the same entry points in the same order
        assert all(not a[9] for n, a in recorder if n == "swinb200_ln_residual_fwd")
        recorder.clear()
        model(x)
        second = [n for n, _ in recorder]
        assert "swinb200_transpose_f32" not in second and "swinb200_cast_f32_to_bf16" not in second
        assert second == [n for n in first if n != "swinb200_transpose_f32"]
        model.pos_embed.add_(1.0)                                # version moves: the copy is rewritten in place
        recorder.clear()
        model(x)
        assert [n for n, _ in recorder].count("swinb200_transpose_f32") == 1


def test_model_with_checkpointed_stages(recorder):
    model = small_model(checkpoint_stages=True)
    model(torch.randn(1, 7, 72, 144))
    epis = [a[GEMM_EPI] for n, a in recorder if n == "swinb200_gemm"]
    assert epis.count(G) == 2 and QK not in epis


def test_header_declares_the_forward_only_epilogue():
    text = open(os.path.join(ROOT, "include", "swinb200.h")).read()
    assert re.search(r"SWINB200_EPI_BIAS_GELU_FWD\s*=\s*7\b", text)
    assert _lib.EPI_BIAS_GELU_FWD == 7 and ops.EPI_BIAS_GELU_FWD == 7


def test_gemm_epilogue_range():
    """7 is accepted by the argument checks; 6 stays internal to swinb200_linear_ln_residual; 8 does not exist.  The calls
    fail on their arguments before any CUDA call."""
    lib = _lib.load()
    for epi in (6, 8):
        assert lib.swinb200_gemm(0, 64, 64, 64, P, 0, 64, P, 0, 64, 1, epi, None, P, 64, None, None, 0, 1, 0, 1, None) == 1
        assert b"unknown epilogue" in lib.swinb200_last_error()
    # epilogue 7 passes the epilogue check and fails on the bad split_k instead
    assert lib.swinb200_gemm(0, 64, 64, 64, P, 0, 64, P, 0, 64, 1, 7, None, P, 64, None, None, 0, 1, 0, 0, None) == 1
    assert b"split_k" in lib.swinb200_last_error()
