"""``EEG_LSTM.lstm(x, hx)`` on the GPU: nn.LSTM(batch_first=True)'s contract on the exact tensor-core kernel
(``na_decoder_lstm_x3``) and on the FFMA / generic kernels (``ops.LSTMSequenceFunction``), against torch's own CPU
nn.LSTM loaded from the model's state_dict (float64).  Tolerance: rel = max|d| / max|ref| per tensor, 1e-5, except for
the fused kernel's per-step output over the 625 steps of the shipped windows (LONG_SEQ_TOL, see DESIGN section 10d)."""
import numpy as np
import pytest
import torch

from oracle.torch_ref import RefEEGLSTM
from tests.test_lstm_sequence_host import _rand_hx, _ref64

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
LONG_SEQ_TOL = 1e-4       # fused kernel, every h of 625 recurrent steps: measured 6.2e-5 against float64 nn.LSTM


def rel(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from neural_speech_decoding_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


@pytest.fixture
def exact_tc():
    """Yields a setter for ops.EXACT_TC and restores it."""
    from neural_speech_decoding_b200 import ops
    old = ops.EXACT_TC

    def set_(v):
        ops.EXACT_TC = v
    yield set_
    ops.EXACT_TC = old


@pytest.fixture
def fused_calls(monkeypatch):
    """Counts the calls of ops.decoder_lstm_x3 (the fused path)."""
    from neural_speech_decoding_b200 import ops
    n = [0]
    real = ops.decoder_lstm_x3

    def counted(*a, **k):
        n[0] += 1
        return real(*a, **k)
    monkeypatch.setattr(ops, "decoder_lstm_x3", counted)
    return n


def make_model(dev, sd=None, seed=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    if seed is not None:
        torch.manual_seed(seed)
    m = EEG_LSTM(**kw)
    if sd is not None:
        m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


def reference(m, x, hx=None):
    """torch's CPU nn.LSTM (RefEEGLSTM(...).lstm) with the model's weights, in float64."""
    lstm = m.lstm
    ref = RefEEGLSTM(lstm.input_size, lstm.hidden_size, lstm.num_layers, m.fc[3].out_features)
    ref.load_state_dict({k: v.detach().float().cpu() for k, v in m.state_dict().items()}, strict=True)
    ref.double().eval()
    with torch.no_grad():
        out, (h, c) = ref.lstm(x.cpu().double(), None if hx is None else tuple(t.cpu().double() for t in hx))
    return out, h, c


def check(got, want, tol=FP32_TOL, out_tol=None):
    for name, a, b in zip(("output", "h_n", "c_n"), got, want):
        r = rel(a.cpu(), b.cpu())
        print(f"{name}: rel {r:.2e}")
        assert r < (out_tol if name == "output" and out_tol else tol), (name, r)


def run(m, x, hx=None):
    with torch.no_grad():
        out, (h, c) = m.lstm(x, hx)
    return out, h, c


@pytest.mark.parametrize("fused", [True, False])
def test_shipped_checkpoint_all_windows(dev, checkpoint, windows, exact_tc, fused_calls, fused):
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"])
    got = run(m, x.to(dev))
    assert fused_calls[0] == (1 if fused else 0)
    assert [tuple(t.shape) for t in got] == [(324, 625, 48), (2, 324, 48), (2, 324, 48)]
    assert all(t.dtype == torch.float32 and t.is_cuda for t in got)
    check(got, reference(m, x), out_tol=LONG_SEQ_TOL if fused else None)


@pytest.mark.parametrize("fused", [True, False])
def test_random_initial_state(dev, checkpoint, windows, exact_tc, fused_calls, fused):
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:50, :100].copy())
    hx = _rand_hx(2, 50, 48, 7)
    got = run(m, x.to(dev), tuple(t.to(dev) for t in hx))
    assert fused_calls[0] == (1 if fused else 0)
    check(got, reference(m, x, hx))
    # unbatched
    with torch.no_grad():
        out, (h, c) = m.lstm(x[3].to(dev), (hx[0][:, 3].to(dev), hx[1][:, 3].to(dev)))
    assert [tuple(t.shape) for t in (out, h, c)] == [(100, 48), (2, 48), (2, 48)]
    r = reference(m, x[3:4], (hx[0][:, 3:4], hx[1][:, 3:4]))
    check((out, h, c), (r[0][0], r[1][:, 0], r[2][:, 0]))


@pytest.mark.parametrize("fused", [True, False])
def test_chunked_streaming(dev, checkpoint, windows, exact_tc, fused, fused_calls):
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:64].copy()).to(dev)
    whole = run(m, x)
    a = run(m, x[:, :200])
    b = run(m, x[:, 200:], (a[1], a[2]))
    assert fused_calls[0] == (3 if fused else 0)
    check((torch.cat([a[0], b[0]], dim=1), b[1], b[2]), whole)


def _raw(m, x, hx, pad):
    """na_decoder_lstm_x3 on NaN-filled buffers `pad` elements longer than needed: every element of the result is
    written, nothing past it."""
    from neural_speech_decoding_b200 import _lib, ops
    B, T = x.shape[0], x.shape[1]
    sizes = (B * T * 48, 2 * B * 48, 2 * B * 48)
    bufs = [torch.full((n + pad,), float("nan"), dtype=torch.float32, device=x.device) for n in sizes]
    h0, c0 = (None, None) if hx is None else (hx[0].contiguous(), hx[1].contiguous())
    _lib.call("na_decoder_lstm_x3", x.data_ptr(), m._packed_x3().data_ptr(), ops._ptr(h0), ops._ptr(c0),
              *[t.data_ptr() for t in bufs], T, B, ops._stream())
    for t, n in zip(bufs, sizes):
        assert bool(torch.isnan(t[n:]).all()), "write past B"
        assert bool(torch.isfinite(t[:n]).all()), "element not written"
    return bufs[0][:sizes[0]].view(B, T, 48), bufs[1][:sizes[1]].view(2, B, 48), bufs[2][:sizes[2]].view(2, B, 48)


@pytest.mark.parametrize("with_hx", [False, True])
def test_tile_layouts_against_ffma(dev, checkpoint, exact_tc, with_hx):
    m = make_model(dev, checkpoint)
    cases = [(B, 30) for B in (1, 31, 33, 64, 65, 97, 128, 129, 300)] + [(148 * 128 + 77, 3)]
    for B, T in cases:
        gen = torch.Generator().manual_seed(B + T)
        x = (torch.randn(B, T, 8, generator=gen) * 20.0).to(dev)
        hx = tuple(t.to(dev) for t in _rand_hx(2, B, 48, B)) if with_hx else None
        got = _raw(m, x, hx, pad=4096)
        api = run(m, x, hx)
        for a, b in zip(got, api):
            assert torch.equal(a, b), (B, T)
        exact_tc(False)
        try:
            ffma = run(m, x, hx)
        finally:
            exact_tc(True)
        check(got, ffma, tol=2 * FP32_TOL)        # two paths, each within FP32_TOL of the exact result


def test_misaligned_views(dev, checkpoint, exact_tc):
    """Contiguous views at an odd float offset (not 16-byte aligned) give the same result as aligned copies."""
    m = make_model(dev, checkpoint)
    B, T = 45, 40
    gen = torch.Generator().manual_seed(12)
    x = (torch.randn(B, T, 8, generator=gen) * 20.0).to(dev)
    hx = tuple(t.to(dev) for t in _rand_hx(2, B, 48, 12))
    views = []
    for t in (x, *hx):
        buf = torch.empty(t.numel() + 1, dtype=torch.float32, device=dev)
        v = buf[1:].view(t.shape)
        v.copy_(t)
        assert v.data_ptr() % 16 != 0
        views.append(v)
    for fused in (True, False):
        exact_tc(fused)
        want = run(m, x, hx)
        got = run(m, views[0], (views[1], views[2]))
        for a, b in zip(got, want):
            assert torch.equal(a, b), fused


def test_attention_pool_matches_decode_intermediates(dev, checkpoint, windows):
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:100].copy()).to(dev)
    with torch.no_grad():
        out, _ = m.lstm(x)
        w = torch.softmax(m.attn(out).squeeze(-1), dim=1)
        pooled = (out * w.unsqueeze(-1)).sum(dim=1)
        ref = m.decode_intermediates(x)
    assert rel(w.cpu(), ref.attention.cpu()) < FP32_TOL
    assert rel(pooled.cpu(), ref.pooled.cpu()) < FP32_TOL


@pytest.mark.parametrize("with_hx", [True, False])
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("shape", [dict(), dict(hidden_size=32, num_layers=3)])
def test_autograd_against_float64(dev, train, shape, with_hx):
    m = make_model(dev, seed=3, **shape)
    if train:
        m.train()
    L, H = m.lstm.num_layers, m.lstm.hidden_size
    B, T = 37, 23
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, T, 8, generator=g) * 5
    hx = _rand_hx(L, B, H, 5)
    R1, R2, R3 = torch.randn(B, T, H, generator=g), torch.randn(L, B, H, generator=g), torch.randn(L, B, H, generator=g)
    xd, h0, c0 = (t.to(dev).requires_grad_() for t in (x, *hx))
    torch.manual_seed(99)
    out, (h_n, c_n) = m.lstm(xd, (h0, c0) if with_hx else None)     # None: zero state, no hx gradients
    ((out * R1.to(dev)).sum() + (h_n * R2.to(dev)).sum() + (c_n * R3.to(dev)).sum()).backward()
    masks = None
    if train:
        torch.manual_seed(99)
        masks = [(torch.rand((B, T, H), device=dev) >= m.lstm.dropout).double().cpu() for _ in range(L - 1)]
    x64, h064, c064 = (t.double().requires_grad_() for t in (x, *(hx if with_hx else (torch.zeros(L, B, H),) * 2)))
    r_out, r_h, r_c, params = _ref64(m, x64, (h064, c064), masks, m.lstm.dropout)
    ((r_out * R1.double()).sum() + (r_h * R2.double()).sum() + (r_c * R3.double()).sum()).backward()
    if with_hx:
        assert h0.grad is not None and c0.grad is not None
    else:
        assert h0.grad is None and c0.grad is None
    for name, a, b in (("output", out, r_out), ("h_n", h_n, r_h), ("c_n", c_n, r_c), ("x", xd.grad, x64.grad),
                       *((("h_0", h0.grad, h064.grad), ("c_0", c0.grad, c064.grad)) if with_hx else ()),
                       *[(n, p.grad, params[n].grad) for n, p in m.lstm.named_parameters()]):
        assert rel(a.detach().cpu(), b.detach()) < FP32_TOL, (name, rel(a.detach().cpu(), b.detach()))
