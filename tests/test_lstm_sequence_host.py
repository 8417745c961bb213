"""Host-side checks of ``EEG_LSTM.lstm(x, hx)`` (nn.LSTM's contract): shapes, unbatched input, ``B == 0``, argument
errors against nn.LSTM's, the routing between the exact tensor-core kernel and the FFMA / generic kernels, and the
autograd wiring of ``ops.LSTMSequenceFunction`` against float64 nn.LSTM.  No GPU: the entry points run on
tests/fake_lib_sequence.FakeLibSequence (the cpu_backend set-up with the sequence entry points added)."""
import numpy as np
import pytest
import torch
import torch.nn as nn


@pytest.fixture
def fake(cpu_backend, monkeypatch):
    from neural_speech_decoding_b200 import _lib
    from tests.fake_lib_sequence import FakeLibSequence
    f = FakeLibSequence()
    monkeypatch.setattr(_lib, "load", lambda path=None: f)
    return f


def _model(checkpoint=None, seed=0, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(seed)
    m = EEG_LSTM(**kw)
    if checkpoint is not None:
        m.load_state_dict(checkpoint, strict=True)
    return m.eval()


def _ref_lstm(m, dtype=torch.float32):
    lstm = m.lstm
    ref = nn.LSTM(lstm.input_size, lstm.hidden_size, lstm.num_layers, batch_first=True, dropout=lstm.dropout)
    ref.load_state_dict({k: v.detach().float().cpu() for k, v in lstm.state_dict().items()}, strict=True)
    return ref.to(dtype).eval()


def _rand_hx(L, B, H, seed, unbatched=False):
    g = torch.Generator().manual_seed(seed)
    shape = (L, H) if unbatched else (L, B, H)
    return torch.rand(shape, generator=g) * 2 - 1, torch.randn(shape, generator=g)


def _close(a, b, tol=1e-5):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-30), np.abs(a - b).max()


@pytest.mark.parametrize("exact_tc", [True, False])
def test_shapes_values_and_unbatched(fake, monkeypatch, checkpoint, windows, exact_tc):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact_tc)
    m = _model(checkpoint)
    ref = _ref_lstm(m)
    x = torch.from_numpy(windows["X"][:5, :40].copy())
    hx = _rand_hx(2, 5, 48, 1)
    with torch.no_grad():
        for args in ((x,), (x, hx)):
            out, (h_n, c_n) = m.lstm(*args)
            assert (tuple(out.shape), tuple(h_n.shape), tuple(c_n.shape)) == ((5, 40, 48), (2, 5, 48), (2, 5, 48))
            assert out.dtype == h_n.dtype == c_n.dtype == torch.float32
            r_out, (r_h, r_c) = ref(*args)
            _close(out, r_out); _close(h_n, r_h); _close(c_n, r_c)
        # unbatched [T,C] with [L,H] state
        hu = _rand_hx(2, 1, 48, 2, unbatched=True)
        out, (h_n, c_n) = m.lstm(x[0], hu)
        r_out, (r_h, r_c) = ref(x[0], hu)
        assert (tuple(out.shape), tuple(h_n.shape), tuple(c_n.shape)) == ((40, 48), (2, 48), (2, 48))
        _close(out, r_out); _close(h_n, r_h); _close(c_n, r_c)
    assert ("na_decoder_lstm_x3" in fake.calls) == exact_tc


def test_empty_batch_launches_nothing(fake):
    m = _model(hidden_size=32, num_layers=3)
    n = fake.na_launch_count()
    out, (h_n, c_n) = m.lstm(torch.zeros(0, 17, 8))
    assert (tuple(out.shape), tuple(h_n.shape), tuple(c_n.shape)) == ((0, 17, 32), (3, 0, 32), (3, 0, 32))
    out, (h_n, c_n) = m.lstm(torch.zeros(0, 17, 8), (torch.zeros(3, 0, 32), torch.zeros(3, 0, 32)))
    assert tuple(out.shape) == (0, 17, 32)
    assert fake.na_launch_count() == n and fake.calls == []


def _bad_inputs():
    x = torch.zeros(3, 10, 8)
    z = lambda *s: torch.zeros(*s)
    return {
        "4d_input": (torch.zeros(1, 3, 10, 8), None),
        "1d_input": (torch.zeros(8), None),
        "input_size": (torch.zeros(3, 10, 7), None),
        "input_size_unbatched": (torch.zeros(10, 5), None),
        "dtype": (torch.zeros(3, 10, 8, dtype=torch.float64), None),
        "h0_batch": (x, (z(2, 4, 48), z(2, 3, 48))),
        "c0_batch": (x, (z(2, 3, 48), z(2, 3, 47))),
        "h0_layers": (x, (z(3, 3, 48), z(3, 3, 48))),
        "hx_2d_for_batched": (x, (z(2, 48), z(2, 48))),
        "hx_3d_for_unbatched": (x[0], (z(2, 1, 48), z(2, 1, 48))),
        "h0_unbatched_size": (x[0], (z(2, 47), z(2, 48))),
    }


@pytest.mark.parametrize("case", sorted(_bad_inputs()))
def test_errors_match_nn_lstm(case):
    m = _model()
    ref = _ref_lstm(m)
    inp, hx = _bad_inputs()[case]
    with pytest.raises(Exception) as want:
        ref(inp, hx)
    with pytest.raises(Exception) as got:
        m.lstm(inp, hx)
    assert type(got.value) is type(want.value)
    assert str(got.value) == str(want.value)


def test_cpu_tensor_raises():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _model().lstm(torch.zeros(2, 10, 8))


def _route(fake, m, x, hx=None, grad=False):
    fake.calls.clear()
    with torch.set_grad_enabled(grad):
        m.lstm(x, hx)
    return "x3" if "na_decoder_lstm_x3" in fake.calls else "generic"


def test_routing(fake, monkeypatch):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", True)
    x = torch.randn(4, 12, 8)
    hx = _rand_hx(2, 4, 48, 3)
    m = _model()
    assert _route(fake, m, x) == "x3"
    assert _route(fake, m, x, hx) == "x3"
    assert fake.calls == ["na_decoder_lstm_x3"]
    assert _route(fake, m, x, grad=True) == "generic"                      # parameters require grad
    assert _route(fake, m, x.requires_grad_(), grad=True) == "generic"
    x = x.detach()
    m.requires_grad_(False)
    assert _route(fake, m, x, grad=True) == "x3"                           # nothing needs a gradient
    assert _route(fake, m, x, (hx[0].requires_grad_(), hx[1]), grad=True) == "generic"
    m.train()
    assert _route(fake, m, x) == "generic"                                 # train-mode dropout (p = 0.6)
    assert _route(fake, _model(dropout=0.0).train(), x) == "x3"
    assert _route(fake, _model(hidden_size=32), x) == "generic"
    assert _route(fake, _model(num_layers=3), x) == "generic"
    mb = _model().bfloat16()
    assert _route(fake, mb, x.bfloat16()) == "generic"
    assert fake.calls[:1] == ["na_lstm_layer_fwd_f32_hx"]
    monkeypatch.setattr(ops, "EXACT_TC", False)
    assert _route(fake, _model(), x) == "generic"


def test_bf16_module_keeps_input_dtype(fake):
    m = _model().bfloat16()
    x = torch.randn(3, 9, 8).bfloat16()
    out, (h_n, c_n) = m.lstm(x)
    assert out.dtype == h_n.dtype == c_n.dtype == torch.bfloat16


def _ref64(m, x, hx, masks, p):
    """Layer-by-layer float64 nn.LSTM with the keep-masks applied between layers (nn.LSTM's own dropout).  Returns
    (out, h_n, c_n, {parameter name of m.lstm: the float64 parameter that stands for it})."""
    lstm = m.lstm
    inp, hn, cn, params = x, [], [], {}
    names = ("weight_ih", "weight_hh", "bias_ih", "bias_hh")
    for l in range(lstm.num_layers):
        cell = nn.LSTM(inp.shape[-1], lstm.hidden_size, 1, batch_first=True)
        cell.load_state_dict({f"{n}_l0": getattr(lstm, f"{n}_l{l}").detach().float().cpu() for n in names})
        cell.double()
        params.update({f"{n}_l{l}": getattr(cell, f"{n}_l0") for n in names})
        out, (h, c) = cell(inp, (hx[0][l:l + 1], hx[1][l:l + 1]))
        hn.append(h[0]); cn.append(c[0])
        inp = out * masks[l] / (1 - p) if (masks is not None and l < lstm.num_layers - 1) else out
    return inp, torch.stack(hn), torch.stack(cn), params


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("shape", [dict(), dict(hidden_size=32, num_layers=3)])
def test_autograd_against_float64(fake, train, shape):
    m = _model(seed=3, **shape)
    if train:
        m.train()
    L, H = m.lstm.num_layers, m.lstm.hidden_size
    B, T = 5, 7
    g = torch.Generator().manual_seed(4)
    x = (torch.randn(B, T, 8, generator=g) * 2).requires_grad_()
    h0, c0 = (t.requires_grad_() for t in _rand_hx(L, B, H, 5))
    R1, R2, R3 = torch.randn(B, T, H, generator=g), torch.randn(L, B, H, generator=g), torch.randn(L, B, H, generator=g)
    torch.manual_seed(99)
    out, (h_n, c_n) = m.lstm(x, (h0, c0))
    ((out * R1).sum() + (h_n * R2).sum() + (c_n * R3).sum()).backward()
    masks = None
    if train:
        torch.manual_seed(99)
        masks = [(torch.rand((B, T, H)) >= m.lstm.dropout).double() for _ in range(L - 1)]
    x64, h064, c064 = (t.detach().double().requires_grad_() for t in (x, h0, c0))
    r_out, r_h, r_c, sd = _ref64(m, x64, (h064, c064), masks, m.lstm.dropout)
    ((r_out * R1.double()).sum() + (r_h * R2.double()).sum() + (r_c * R3.double()).sum()).backward()
    _close(out.detach(), r_out.detach()); _close(h_n.detach(), r_h.detach()); _close(c_n.detach(), r_c.detach())
    _close(x.grad, x64.grad); _close(h0.grad, h064.grad); _close(c0.grad, c064.grad)
    for name, p in m.lstm.named_parameters():
        _close(p.grad, sd[name].grad)
    assert "na_lstm_layer_bwd_f32_hx" in fake.calls and "na_lstm_layer_wgrad_f32_hx" in fake.calls


@pytest.fixture(scope="module")
def lib(built_lib):
    from neural_speech_decoding_b200 import _lib
    return _lib.load()


def test_abi_validation(lib):
    import ctypes
    A, MIS = ctypes.c_void_p(256), ctypes.c_void_p(260)        # aligned / misaligned fake addresses
    for k in range(7):                                          # every pointer must be 16-byte aligned
        ptrs = [A] * 7
        ptrs[k] = MIS
        assert lib.na_decoder_lstm_x3(*ptrs, 625, 4, None) == -2, k
        assert b"not 16-byte aligned" in lib.na_last_error()
    assert lib.na_decoder_lstm_x3(A, A, A, None, A, A, A, 625, 4, None) == -1     # h_init without c_init
    assert b"given together" in lib.na_last_error()
    assert lib.na_decoder_lstm_x3(A, A, None, None, A, A, A, 625, 0, None) == -1  # B = 0
    assert lib.na_decoder_lstm_x3(A, A, None, None, A, A, A, 0, 4, None) == -1    # T = 0
    assert lib.na_decoder_lstm_x3(A, A, None, None, None, A, A, 625, 4, None) == -1
    assert lib.na_lstm_layer_fwd_f32_hx(*([A] * 7), 1.0, None, 625, 32, 8, 48, MIS, A, None) == -2
    assert lib.na_lstm_layer_fwd_f32_hx(*([A] * 7), 1.0, None, 625, 32, 8, 48, A, None, None) == -1
    assert lib.na_lstm_layer_bwd_f32_hx(*([A] * 8), 1.0, 625, 32, 8, 48, A, A, A, MIS, A, None) == -2
    assert lib.na_lstm_layer_wgrad_f32_hx(*([A] * 7), 625, 32, 8, 48, MIS, None) == -2
