"""The C-ABI library builds for sm_100a, loads, and exports every symbol include/neuroalpha.h
declares.  No compute call is made here (no GPU): only argument validation paths, which return
before any CUDA API is touched."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def lib(built_lib):
    from neural_speech_decoding_b200 import _lib
    return _lib.load()


def test_header_and_bindings_agree(lib):
    from neural_speech_decoding_b200 import _lib
    header = (ROOT / "include" / "neuroalpha.h").read_text()
    declared = set(re.findall(r"\b(na_[a-z0-9_]+)\s*\(", header))
    declared.discard("na_last_error")
    declared.add("na_last_error")
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name


def test_version_and_queries(lib):
    assert lib.na_version() == 100
    assert lib.na_launch_count() >= 0
    assert lib.na_head_param_floats(48, 3) == 48 + 1 + 48 + 48 + 32 * 48 + 32 + 32 * 3 + 3
    assert lib.na_wgrad_partial_floats(8, 48) > 0
    assert lib.na_head_partial_floats(100, 48, 3) > 100 * (64 + 3 * 48)


def test_error_codes_without_gpu(lib):
    # bad shapes / null / misaligned pointers are rejected before any CUDA call
    assert lib.na_trial_mean_f32(None, None, 0, 10, None) == -1
    assert b"bad shape" in lib.na_last_error()
    assert lib.na_trial_mean_f32(None, None, 10, 0, None) == 0           # empty input is a no-op
    assert lib.na_trial_mean_f32(None, None, 10, 5, None) == -1          # null pointer
    assert lib.na_trial_mean_f32(ctypes.c_void_p(8), ctypes.c_void_p(16), 10, 5, None) == -2   # alignment
    assert lib.na_window_zscore(None, None, 4, 625, 8, 0, 1, 0, 4, 0, None) == -1
    assert lib.na_window_zscore(None, None, 4, 625, 1000, 625, 1, 0, 4, 0, None) == -3
    assert lib.na_lstm_layer_fwd_f32(*([None] * 7), 1.0, None, 625, 33, 8, 48, None) == -1   # Bp % 32
    assert lib.na_lstm_layer_fwd_f32(*([None] * 7), 1.0, None, 625, 32, 8, 4096, None) == -3  # H too large
    assert lib.na_head_fwd_f32(*([None] * 11), 1.0, *([None] * 4), 625, 4, 32, 48, 99, None) == -3


def test_python_wrapper_raises_runtime_error(lib):
    from neural_speech_decoding_b200 import _lib
    with pytest.raises(RuntimeError, match="na_trial_mean_f32 failed"):
        _lib.call("na_trial_mean_f32", None, None, 0, 10, None)


def test_sass_is_sm100(built_lib):
    import subprocess
    from neural_speech_decoding_b200.build import find_nvcc
    cuobjdump = Path(find_nvcc()).resolve().parent / "cuobjdump"      # the toolkit that built the library, on PATH or not
    out = subprocess.run([str(cuobjdump), "-lelf", str(built_lib)], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out
