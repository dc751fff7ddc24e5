"""ctypes binding of libswinb200.so -- the C-ABI kernel library (include/swinb200.h).

There is no CPU or PyTorch fallback: if the library has not been built, importing the ops raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libswinb200.so")

# enums of include/swinb200.h
F32, BF16 = 0, 1
EPI_BIAS, EPI_BIAS_GELU, EPI_DGELU, EPI_ADD_F32, EPI_F32, EPI_BIAS_QKNORM = 0, 1, 2, 3, 4, 5
EPI_BIAS_GELU_FWD = 7     # BIAS_GELU's activation output alone (forward-only runs); 6 is internal to swinb200_linear_ln_residual
BACKEND_SIMT, BACKEND_TCGEN05 = 0, 1

_P = c_void_p
_I = c_int
_LL = ctypes.c_longlong

# name -> argtypes, exactly the prototypes of include/swinb200.h
PROTOTYPES = {
    "swinb200_cast_f32_to_bf16": [_P, _P, c_size_t, _P],
    "swinb200_patchify": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "swinb200_patchify_cat": [_I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "swinb200_unpatchify": [_P, _I, _P, _I, _P, _I, _I, _I, _I, _I, _I, _P],
    "swinb200_patchify_cat_norm": [_I, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "swinb200_unpatchify_norm": [_P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "swinb200_latw_l1_fwd": [_P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P],
    "swinb200_latw_l1_bwd": [_P, _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _P],
    "swinb200_latw_acc": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "swinb200_gemm": [_I, _I, _I, _I, _P, _I, _I, _P, _I, _I, _I, _I, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P],
    "swinb200_linear_wgrad": [_I, _I, _I, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P],
    "swinb200_linear_ln_residual": [_I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, c_float, _P, _I, _P],
    "swinb200_ln_residual_fwd": [_P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, c_float, _P],
    "swinb200_ln_residual_bwd": [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P],
    "swinb200_pos_embed_grad": [_P, _P, _I, _I, _I, _P],
    "swinb200_transpose_f32": [_P, _P, _I, _I, _P],
    "swinb200_colsum": [_P, _I, _P, _I, _I, _I, _P],
    "swinb200_qk_normalize": [_P, _I, _P, _I, _I, _I, _P],
    "swinb200_shift_mask": [_P, _I, _I, _I, _I, _I, _I, _P],
    "swinb200_window_attn_fwd": [_I, _P, _I, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "swinb200_window_attn_bwd": [_I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "swinb200_latw_l2_fwd": [_P, _P, _P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _I, _P],
    "swinb200_debug_attn_phase_buffer": [_P],
    "swinb200_debug_umma_probe": [_P, _P, _P, _I, _I, _I, _I, _I, _P],
    "swinb200_latw_l2_bwd": [_P, _P, _P, _P, _P, _P, _P, _I, _I, _P, _I, _I, _I, _I, _P],
    "swinb200_adam_step": [_I, _P, _P, _P, _P, _P, _P, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                           ctypes.c_double, ctypes.c_longlong, _P, _P, _P],
    # deterministic mode: caller-owned scratch (pointer, size in floats) before the stream
    "swinb200_ordered_reduce": [_P, _I, _LL, _LL, _I, _P, _I, _P],
    "swinb200_gemm_wgrad_det": [_I, _I, _I, _I, _P, _I, _P, _I, _I, _P, _I, _P, _LL, _P],
    "swinb200_linear_wgrad_det": [_I, _I, _I, _I, _P, _I, _P, _I, _P, _P, _I, _P, _LL, _P],
    "swinb200_ln_residual_bwd_det": [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _LL, _P],
    "swinb200_colsum_det": [_P, _I, _P, _I, _I, _I, _P, _LL, _P],
    "swinb200_latw_l2_fwd_det": [_P, _P, _P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _I, _P, _LL, _P],
    "swinb200_latw_l1_fwd_det": [_P, _P, _P, _P, _I, _P, _P, _I, _I, _I, _I, _P, _LL, _P],
    "swinb200_latw_acc_det": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P, _LL, _P],
    "swinb200_window_attn_bwd_det": [_I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _LL,
                                     _P],
}

_lib = None


ERR_INVALID_ARG, ERR_CUDA, ERR_UNSUPPORTED = 1, 2, 3


class SwinB200Error(RuntimeError):
    def __init__(self, msg: str, code: int = 0):
        super().__init__(msg)
        self.code = code        # SWINB200_ERR_* of a failed call, 0 for errors raised on the Python side


def load() -> ctypes.CDLL:
    """Loads the library (once).  Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SwinB200Error(
            f"{LIB_PATH} not found: build the CUDA kernels first "
            "(`python -m swin_v2_weather_b200.build` or `__graft_entry__.build()`); there is no fallback path."
        )
    lib = ctypes.CDLL(LIB_PATH)
    lib.swinb200_version.restype = c_int
    lib.swinb200_version.argtypes = []
    lib.swinb200_last_error.restype = c_char_p
    lib.swinb200_last_error.argtypes = []
    for name, argtypes in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = c_int
        fn.argtypes = argtypes
    _lib = lib
    return lib


# kernels launched per C-ABI call (everything else launches exactly one); used for the launch counter
# kernels launched per C-ABI call where it is not one (loss: reduce + finish; attention backward: <dO,O> pre-pass + main kernel)
_KERNELS_PER_CALL = {"swinb200_latw_l2_fwd": 2, "swinb200_window_attn_bwd": 2, "swinb200_latw_l1_fwd": 2, "swinb200_latw_acc": 2}
LAUNCH_COUNT = 0          # our kernels launched so far in this process
PROFILE_HOOK = None       # optional callable(name, args) -> context manager; set by bench.py to time kernels


def call(name: str, *args) -> None:
    global LAUNCH_COUNT
    lib = load()
    LAUNCH_COUNT += _KERNELS_PER_CALL.get(name, 1)
    if PROFILE_HOOK is not None:
        with PROFILE_HOOK(name, args):
            rc = getattr(lib, name)(*args)
    else:
        rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.swinb200_last_error().decode("utf-8", "replace")
        raise SwinB200Error(f"{name} failed (code {rc}): {msg}", rc)
