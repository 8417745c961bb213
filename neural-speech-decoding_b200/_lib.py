"""ctypes binding of libneuroalpha_b200.so (the C ABI declared in include/neuroalpha.h).

There is no CPU fallback: if the shared object is missing or a call fails, a RuntimeError is
raised.  ``call(name, *args)`` converts a non-zero return code into
``RuntimeError(na_last_error())`` -- no exception crosses the ABI itself.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p
from pathlib import Path

from .build import LIB_PATH

P, I64, I32, F32 = c_void_p, c_int64, c_int, c_float

# name -> (restype, argtypes); mirrors include/neuroalpha.h one to one.
SIGNATURES = {
    "na_version": (c_int, []),
    "na_last_error": (c_char_p, []),
    "na_launch_count": (c_int64, []),
    "na_set_tuning": (c_int, [c_char_p, I64]),
    "na_ffma_probe": (c_int, [P, I64, I64, P]),
    "na_window_zscore": (c_int, [P, P, I64, I64, I64, I64, I32, I32, I64, I32, P]),
    "na_pack_lstm_layer": (c_int, [P, P, P, P, P, P, I64, I64, P]),
    "na_lstm_layer_fwd_f32": (c_int, [P, P, P, P, P, P, P, F32, P, I64, I64, I64, I64, P]),
    "na_lstm_layer_bwd_f32": (c_int, [P, P, P, P, P, P, P, P, F32, I64, I64, I64, I64, P]),
    "na_wgrad_partial_floats": (c_int64, [I64, I64]),
    "na_lstm_layer_wgrad_f32": (c_int, [P, P, P, P, P, P, P, I64, I64, I64, I64, P]),
    "na_head_fwd_f32": (c_int, [P] * 9 + [P, P, F32, P, P, P, P, I64, I64, I64, I64, I64, P]),
    "na_head_fwd_f32_ex": (c_int, [P] * 9 + [P, P, F32, P, P, P, P, P, P, P, I64, I64, I64, I64, I64, P]),
    "na_attention_softmax_f32": (c_int, [P, P, I64, I64, P]),
    "na_head_param_floats": (c_int64, [I64, I64]),
    "na_head_partial_floats": (c_int64, [I64, I64, I64]),
    "na_head_bwd_f32": (c_int, [P] * 12 + [P, P, F32, P, P, P, I64, I64, I64, I64, I64, P]),
    "na_decoder_packed_bf16_bytes": (c_int64, []),
    "na_decoder_pack_bf16": (c_int, [P] * 9 + [P]),
    "na_decoder_infer_bf16": (c_int, [P] * 12 + [I64, I64, I64, I64, P]),
    "na_decoder_infer_bf16_x32": (c_int, [P] * 12 + [I64, I64, I64, P]),
    "na_decoder_infer_bf16_ex": (c_int, [P] * 15 + [I64, I64, I64, I64, P]),
    "na_decoder_infer_bf16_x32_ex": (c_int, [P] * 15 + [I64, I64, I64, P]),
    "na_decoder_packed_x3_bytes": (c_int64, []),
    "na_decoder_pack_x3": (c_int, [P] * 9 + [P]),
    "na_decoder_infer_x3": (c_int, [P] * 12 + [I64, I64, I64, P]),
    "na_decoder_infer_x3_ex": (c_int, [P] * 15 + [I64, I64, I64, P]),
    "na_decoder_wide_packed_bytes": (c_int64, [I64]),
    "na_decoder_wide_state_bytes": (c_int64, [I64]),
    "na_decoder_pack_wide_bf16": (c_int, [P] * 11 + [I64, P]),
    "na_decoder_infer_wide_bf16": (c_int, [P] * 11 + [I64, I64, I64, I64, I64, P]),
    "na_decoder_infer_wide_bf16_ex": (c_int, [P] * 14 + [I64, I64, I64, I64, I64, P]),
    "na_train_bf16_partial_floats": (c_int64, []),
    "na_dropout_mask_u8": (c_int, [ctypes.c_uint64, I64, I64, I64, P, P]),
    "na_lstm2_fwd_train_bf16": (c_int, [P, P, P, ctypes.c_uint64, I64, F32, P, P, P, P, P, P, P, P, P, P, I64, I64, I64, I64, P]),
    "na_lstm_bwd_bf16": (c_int, [I64, P, P, P, P, P, P, P, P, P, ctypes.c_uint64, I64, F32, P, P, P, P, P,
                                 P, P, P, P, P, I64, P, I64, I64, I64, P]),
    "na_x3_split_input": (c_int, [P, P, I64, I64, I64, I64, P]),
    "na_lstm_fwd_train_x3": (c_int, [I64, P, P, P, P, P, ctypes.c_uint64, I64, F32, P, P, P, P, P, I64, I64, I64, I64, P]),
    "na_train_x3_scratch_floats": (c_int64, []),
    "na_train_x3_smem_bytes": (c_int64, [I64]),
    "na_lstm_bwd_x3": (c_int, [I64, P, P, P, P, P, P, P, ctypes.c_uint64, I64, F32, P, P, P, P, P, P, P, I64, P, P, I64, I64, I64, P]),
    "na_lstm_wgrad_x3": (c_int, [I64, P, P, P, P, P, P, P, P, I64, I64, I64, P]),
    "na_head_tail_fwd_f32": (c_int, [P] * 9 + [P, P, F32, P, P, I64, I64, I64, P]),
    "na_head_tail_bwd_f32": (c_int, [P] * 10 + [P, P, F32, P, P, P, I64, I64, I64, P]),
    "na_iir_chain": (c_int, [P, P, P, P, P, I64, I64, I64, I64, I32, I32, I32, I64, P]),
    "na_wide_train_ws_floats": (c_int64, [I64]),
    "na_lstm_wide_fwd_train": (c_int, [P, P, P, P, P, I64, I64, I64, P]),
    "na_lstm_wide_bwd": (c_int, [P, P, P, P, P, P, I64, I64, I64, P]),
    "na_phase_coupling_filter": (c_int, [P, P, P, ctypes.c_double, P, I64, I64, I64, P]),
    "na_csv_parse_f32": (c_int, [P, P, P, P, I64, I64, I64, P]),
    "na_adam_multi": (c_int, [P, I64, I64, F32, F32, F32, F32, F32, F32, F32, P, P]),
    "na_trial_mean_f32": (c_int, [P, P, I64, I64, P]),
}

_LIB = None


def load(path: str | Path | None = None):
    """Load (once) and return the shared library.  Raises RuntimeError if it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = Path(path or os.environ.get("NEUROALPHA_B200_LIB") or LIB_PATH)     # env override: A/B-timing a variant build
    if not p.exists():
        raise RuntimeError(
            f"{p} not found: the CUDA library is not built (run `python -c 'import __graft_entry__ as g; "
            "g.build()'`).  neural_speech_decoding_b200 has no CPU fallback.")
    lib = ctypes.CDLL(str(p))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)           # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    if lib.na_version() // 100 != 1:
        raise RuntimeError(f"libneuroalpha_b200 ABI version {lib.na_version()} is not 1xx")
    _LIB = lib
    return lib


def last_error() -> str:
    return load().na_last_error().decode("utf-8", "replace")


def call(name: str, *args):
    """Invoke an int-returning entry point; raise on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed (rc={rc}): {lib.na_last_error().decode('utf-8', 'replace')}")


def query(name: str, *args) -> int:
    """Invoke a size/count query (returns int64)."""
    return int(getattr(load(), name)(*args))
