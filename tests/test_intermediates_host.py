"""Host-side checks of EEG_LSTM.decode_intermediates and of the argument validation of the intermediates entry points.
No GPU: the decoder runs on tests/fake_lib_intermediates.FakeLibIntermediates (the cpu_backend set-up with the
intermediates entry points added), the validation tests call the built library on paths that return before any CUDA
call."""
import ctypes

import numpy as np
import pytest
import torch

from oracle.torch_ref import RefEEGLSTM


@pytest.fixture
def cpu_backend_ex(cpu_backend, monkeypatch):
    """cpu_backend with a host stand-in that also implements na_head_fwd_f32_ex and na_attention_softmax_f32."""
    from neural_speech_decoding_b200 import _lib
    from tests.fake_lib_intermediates import FakeLibIntermediates
    fake = FakeLibIntermediates()
    monkeypatch.setattr(_lib, "load", lambda path=None: fake)
    return fake


def _model(checkpoint=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    m = EEG_LSTM(**kw)
    if checkpoint is not None:
        m.load_state_dict(checkpoint, strict=True)
    return m.eval()


def test_decode_intermediates_shapes_and_values(cpu_backend_ex, checkpoint, windows):
    from neural_speech_decoding_b200.lstm_eeg_model import DecoderOutputs
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:5, :40].copy())
    out = m.decode_intermediates(x)
    assert isinstance(out, DecoderOutputs)
    assert [tuple(t.shape) for t in out] == [(5, 3), (5, 3), (5, 40), (5, 48), (5, 48)]
    assert all(t.dtype == torch.float32 for t in out)
    lg, pr = m.decode(x)
    assert torch.equal(out.logits, lg) and torch.equal(out.probs, pr)
    # the hook idiom on the reference module gives the same quantities
    ref = RefEEGLSTM()
    ref.load_state_dict(checkpoint, strict=True)
    ref.eval()
    seen = {}
    ref.attn.register_forward_hook(lambda mod, i, o: seen.__setitem__("scores", o.squeeze(-1)))
    ref.ln.register_forward_hook(lambda mod, i, o: seen.update(pooled=i[0], emb=o))
    with torch.no_grad():
        ref(x)
    np.testing.assert_allclose(out.attention.numpy(), torch.softmax(seen["scores"], dim=1).numpy(), atol=1e-5)
    np.testing.assert_allclose(out.pooled.numpy(), seen["pooled"].numpy(), atol=1e-5)
    np.testing.assert_allclose(out.embedding.numpy(), seen["emb"].numpy(), atol=1e-4)
    np.testing.assert_allclose(out.attention.sum(1).numpy(), 1.0, atol=1e-6)


def test_decode_intermediates_empty_batch(cpu_backend_ex):
    m = _model(hidden_size=32, num_classes=5)
    out = m.decode_intermediates(torch.zeros(0, 17, 8))
    assert [tuple(t.shape) for t in out] == [(0, 5), (0, 5), (0, 17), (0, 32), (0, 32)]
    assert all(t.dtype == torch.float32 for t in out)


def test_decode_intermediates_rejects_cpu_tensor():
    m = _model()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.decode_intermediates(torch.zeros(2, 10, 8))


@pytest.fixture(scope="module")
def lib(built_lib):
    from neural_speech_decoding_b200 import _lib
    return _lib.load()


A, B16, MIS = ctypes.c_void_p(256), ctypes.c_void_p(512), ctypes.c_void_p(8)    # aligned / misaligned fake addresses


def test_attention_softmax_validation(lib):
    assert lib.na_attention_softmax_f32(A, B16, 0, 4, None) == -1
    assert b"bad shape" in lib.na_last_error()
    assert lib.na_attention_softmax_f32(A, B16, 10, 0, None) == -1
    assert lib.na_attention_softmax_f32(None, B16, 10, 4, None) == -1
    assert lib.na_attention_softmax_f32(A, None, 10, 4, None) == -1
    assert lib.na_attention_softmax_f32(MIS, B16, 10, 4, None) == -2
    assert lib.na_attention_softmax_f32(A, MIS, 10, 4, None) == -2


def test_head_fwd_ex_validation(lib):
    par = [A] * 8
    # misaligned extras are rejected; the shape rules of na_head_fwd_f32 still apply
    for k in range(3):
        ex = [None, None, None]
        ex[k] = MIS
        assert lib.na_head_fwd_f32_ex(A, *par, None, None, 1.0, A, None, *ex, None, None, 625, 4, 32, 48, 3, None) == -2
        assert b"not 16-byte aligned" in lib.na_last_error()
    assert lib.na_head_fwd_f32_ex(A, *par, None, None, 1.0, A, None, A, A, A, None, None, 625, 4, 32, 48, 99, None) == -3
    assert lib.na_head_fwd_f32_ex(A, *par, None, None, 1.0, A, None, A, A, A, None, None, 625, 0, 32, 48, 3, None) == -1


def test_decoder_ex_validation(lib):
    par = [A] * 8
    for k in range(3):
        ex = [None, None, None]
        ex[k] = MIS
        assert lib.na_decoder_infer_x3_ex(A, A, *par, A, A, *ex, 625, 4, 3, None) == -2
        assert lib.na_decoder_infer_bf16_x32_ex(A, A, *par, A, A, *ex, 625, 4, 3, None) == -2
        assert lib.na_decoder_infer_bf16_ex(A, A, *par, A, A, *ex, 625, 4, 128, 3, None) == -2
        assert lib.na_decoder_infer_wide_bf16_ex(A, A, *par[2:], A, A, A, *ex, 625, 4, 128, 96, 3, None) == -2
    assert lib.na_decoder_infer_x3_ex(A, A, *par, A, A, A, A, A, 625, 0, 3, None) == -1
    assert lib.na_decoder_infer_x3_ex(None, A, *par, A, A, A, A, A, 625, 4, 3, None) == -1
    assert lib.na_decoder_infer_x3_ex(A, A, *par, None, A, A, A, A, 625, 4, 3, None) == -1
    assert lib.na_decoder_infer_bf16_ex(A, A, *par, A, A, A, A, A, 625, 4, 100, 3, None) == -1      # Bp % 128
    assert lib.na_decoder_infer_wide_bf16_ex(A, A, *par[2:], A, A, A, A, A, A, 625, 4, 128, 64, 3, None) == -3
    assert lib.na_decoder_infer_x3_ex(A, A, *par, A, A, A, A, A, 625, 4, 17, None) == -3


def test_v1_kernel_rejects_intermediates(lib):
    assert lib.na_set_tuning(b"tc_infer_hs", 1) == 0
    try:
        assert lib.na_decoder_infer_bf16_ex(A, A, *([A] * 8), A, A, A, None, None, 625, 4, 128, 3, None) == -3
        assert b"v1 kernel" in lib.na_last_error()
    finally:
        assert lib.na_set_tuning(b"tc_infer_hs", 3) == 0
