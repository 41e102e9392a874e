"""ctypes binding of libpm_emage.so (the C ABI in include/pm_emage.h).

There is no CPU fallback: if the library is missing or a kernel call fails, the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PM_EMAGE_LIB: an instrumented / tuning build of the same sources (pantomatrix_b200.build --variant), tools only
LIB_PATH = os.environ.get("PM_EMAGE_LIB") or os.path.join(_HERE, "libpm_emage.so")

_p = C.c_void_p
_i = C.c_int
_ll = C.c_longlong
_f = C.c_float

# name -> argument ctypes (all functions return int)
SIGNATURES = {
    "pm_abi_version": [],
    "pm_device_cc": [],
    "pm_tapgemm_f32": [_p, _ll, _i, _i, _i, _i, _p, _p, _i, _i, _i, _i, _i, _p, _ll, _i, _i, _f, _p, _ll, _i, _p],
    "pm_tapgemm_tc": [_p, _ll, _ll, _i, _i, _i, _i, _p, _ll, _i, _i, _i, _i, _i, _p, _i, _i, _p, _ll, _i,
                      _i, _i, _f, _f, _p, _ll, _i, _p, _ll, _ll, _i, _i, _p, _ll, _p],
    "pm_split_bf16": [_p, _ll, _i, _i, _i, _i, _p, _ll, _ll, _i, _i, _p],
    "pm_wav_stem_f32": [_p, _ll, _ll, _i, _i, _i, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p, _p, _p, _ll, _i, _i, _p],
    "pm_add_layernorm_f32": [_p, _p, _p, _p, _p, _ll, _i, _f, _p, _ll, _i, _i, _p],
    "pm_attention_f32": [_p, _i, _p, _i, _p, _i, _p, _i, _i, _i, _i, _i, _i, _p, _ll, _i, _i, _p],
    "pm_attention_tc": [_p, _ll, _ll, _i, _i, _i, _p, _ll, _ll, _i, _i, _i, _p, _ll, _ll, _i, _i, _i,
                        _p, _i, _i, _i, _i, _i, _i, _p, _ll, _i, _i, _p],
    "pm_add_rows_f32": [_p, _p, _p, _i, _i, _p, _i, _i, _i, _p, _ll, _i, _i, _p],
    "pm_add2_f32": [_p, _p, _p, _ll, _i, _p, _ll, _i, _i, _p],
    "pm_window_input_f32": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _ll, _p, _ll, _i, _i, _p],
    "pm_l2_argmin_f32": [_p, _ll, _i, _ll, _p, _p, _i, _i, _p, _p],
    "pm_row_argmax_f32": [_p, _ll, _i, _i, _i, _ll, _p, _p, _p],
    "pm_l2_argmin_tc": [_p, _ll, _i, _ll, _p, _p, _i, _i, _p, _i, _p],
    "pm_l2_argmin_simt_f32": [_p, _ll, _i, _ll, _p, _p, _i, _i, _p, _p],
    "pm_memset_async": [_p, _i, _ll, _p],
    "pm_gather_rows_f32": [_p, _ll, _p, _ll, _i, _p, _p, _ll, _i, _i, _p],
    "pm_row_sqnorm_f32": [_p, _i, _i, _p, _p],
    "pm_pose_compose_f32": [_p, _p, _p, _p, _p, _p, _p, _ll, _p],
    "pm_global_trans_f32": [_p, _i, _i, _p, _i, _f, _p, _i, _i, _p],
    "pm_lstm_bidir_f32": [_p, _ll, _i, _p, _p, _ll, _i, _p, _i, _i, _i, _p],
    "pm_rot6d_to_aa_f32": [_p, _ll, _i, _p, _p, _p],
    "pm_softmax2_mix_f32": [_p, _p, _p, _p, _ll, _i, _i, _p],
}
# ragged-batch twins: the entry point without `_rl` + per-clip limit arguments before the stream
for _rl, _name, _extra in (("pm_tapgemm_tc_rl", "pm_tapgemm_tc", [_p, _i]), ("pm_tapgemm_f32_rl", "pm_tapgemm_f32", [_p, _i]),
                           ("pm_wav_stem_rl", "pm_wav_stem_f32", [_p]), ("pm_attention_tc_rl", "pm_attention_tc", [_p, _p]),
                           ("pm_attention_f32_rl", "pm_attention_f32", [_p, _p]),
                           ("pm_window_input_rl", "pm_window_input_f32", [_p]),
                           ("pm_gather_rows_rl", "pm_gather_rows_f32", [_p, _i])):
    SIGNATURES[_rl] = SIGNATURES[_name][:-1] + _extra + [_p]

_lib = None


class PmError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built - never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PmError(
                f"{LIB_PATH} not found: build it with `python -m pantomatrix_b200.build` "
                "(there is no CPU or PyTorch fallback for the EMAGE hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here = header / library mismatch
            fn.argtypes = args
            fn.restype = C.c_int
        _lib = lib
    return _lib


def call(name: str, *args) -> None:
    rc = getattr(load(), name)(*args)
    if rc != 0:
        kind = "bad argument / unsupported shape" if rc < 0 else "cudaError"
        raise PmError(f"{name} failed: {kind} {rc}")
