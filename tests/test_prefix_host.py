"""Host-side checks of EEG_LSTM.decode_prefixes and of the argument validation of its two entry points.  No GPU: the
decoder runs on FakeLibPrefix below (tests/fake_lib.FakeLib plus numpy versions of the prefix entry points and of the
head tail), compared with a float64 restatement (one causal LSTM pass over the window, then a softmax pool per prefix);
the validation tests call the built library on paths that return before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch

from oracle.torch_ref import RefEEGLSTM
from tests.fake_lib import RRELU_EVAL, FakeLib, _arr, _sig

X3_PACKED_BYTES = 40 * 3072            # na_decoder_packed_x3_bytes()


def _lstm64(x, layers):
    """float64 nn.LSTM (zero state, eval) over x [B,T,K]; layers = [(w_ih, w_hh, b_ih, b_hh)] -> last layer's h [B,T,H]."""
    out = x
    for w_ih, w_hh, b_ih, b_hh in layers:
        B, T, _ = out.shape
        H = w_hh.shape[1]
        h, c = np.zeros((B, H)), np.zeros((B, H))
        pre = out @ w_ih.T + b_ih + b_hh
        hs = np.empty((B, T, H))
        for t in range(T):
            g = pre[:, t] + h @ w_hh.T
            i, f, gg, o = _sig(g[:, :H]), _sig(g[:, H:2 * H]), np.tanh(g[:, 2 * H:3 * H]), _sig(g[:, 3 * H:])
            c = f * c + i * gg
            h = o * np.tanh(c)
            hs[:, t] = h
        out = hs
    return out


def _pool_prefixes64(h, aw, ab, stride):
    """h [B,T,H] float64 -> pooled [B,P,H]: the softmax-over-time pool of h[:, :t_j] for every prefix end t_j."""
    T = h.shape[1]
    s = h @ aw + ab                                               # [B,T]
    ends = [min((j + 1) * stride, T) for j in range(-(-T // stride))]
    out = []
    for t in ends:
        e = np.exp(s[:, :t] - s[:, :t].max(axis=1, keepdims=True))
        out.append(np.einsum("bt,bth->bh", e, h[:, :t]) / e.sum(axis=1)[:, None])
    return np.stack(out, axis=1)


class FakeLibPrefix(FakeLib):
    """FakeLib with numpy versions of na_decoder_pack_x3 (the raw fp32 weights stand in for the fp16 image),
    na_decoder_prefix_pool_x3, na_attention_pool_prefix_f32 and na_head_tail_fwd_f32.  Records the entry points it runs."""

    def __init__(self):
        super().__init__()
        self.calls = []

    def na_decoder_packed_x3_bytes(self):
        return X3_PACKED_BYTES

    def na_decoder_pack_x3(self, w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1, packed, stream):
        shapes = [(192, 8), (192, 48), (192,), (192,), (192, 48), (192, 48), (192,), (192,)]
        flat = np.concatenate([_arr(p, s).ravel() for p, s in zip((w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1),
                                                                 shapes)])
        _arr(packed, (flat.size,))[...] = flat
        self.calls.append("na_decoder_pack_x3")
        self.launches += 1
        return 0

    def na_decoder_prefix_pool_x3(self, x, packed, aw, ab, pooled, T, B, stride, stream):
        if T < 1 or B < 1 or stride < 1:
            return self._fail("na_decoder_prefix_pool_x3: bad shape")
        flat = _arr(packed, (29952,)).astype(np.float64)
        sizes = [192 * 8, 192 * 48, 192, 192, 192 * 48, 192 * 48, 192, 192]
        parts = np.split(flat, np.cumsum(sizes)[:-1])
        layers = [(parts[0].reshape(192, 8), parts[1].reshape(192, 48), parts[2], parts[3]),
                  (parts[4].reshape(192, 48), parts[5].reshape(192, 48), parts[6], parts[7])]
        h = _lstm64(_arr(x, (B, T, 8)).astype(np.float64), layers)
        P = -(-T // stride)
        _arr(pooled, (B, P, 48))[...] = _pool_prefixes64(h, _arr(aw, (48,)).astype(np.float64), float(_arr(ab, (1,))[0]),
                                                         stride)
        self.calls.append("na_decoder_prefix_pool_x3")
        self.launches += 1
        return 0

    def na_attention_pool_prefix_f32(self, h, aw, ab, pooled, T, B, Bp, H, stride, stream):
        if T < 1 or B < 1 or Bp < B or stride < 1:
            return self._fail("na_attention_pool_prefix_f32: bad shape")
        hh = _arr(h, (T, Bp, H)).astype(np.float64)[:, :B].transpose(1, 0, 2)
        P = -(-T // stride)
        _arr(pooled, (B, P, H))[...] = _pool_prefixes64(hh, _arr(aw, (H,)).astype(np.float64), float(_arr(ab, (1,))[0]),
                                                        stride)
        self.calls.append("na_attention_pool_prefix_f32")
        self.launches += 1
        return 0

    def na_head_tail_fwd_f32(self, zpool, aw, ab, lw, lb, w0, b0, w3, b3, rrelu_slope, drop_mask, drop_scale,
                             logits, probs, B, H, NC, stream):
        assert rrelu_slope is None and drop_mask is None          # decode_prefixes: eval arithmetic
        P = self._head_params((aw, ab, lw, lb, w0, b0, w3, b3), H, NC)
        zp = _arr(zpool, (B, H)).astype(np.float64)
        a_post = self._tail(zp, P, float(RRELU_EVAL), 1.0)[4]
        lg = a_post @ P["w3"].T + P["b3"]
        _arr(logits, (B, NC))[...] = lg
        if probs is not None:
            e = np.exp(lg - lg.max(axis=1, keepdims=True))
            _arr(probs, (B, NC))[...] = e / e.sum(axis=1, keepdims=True)
        self.calls.append("na_head_tail_fwd_f32")
        self.launches += 1
        return 0


@pytest.fixture
def fake(cpu_backend, monkeypatch):
    from neural_speech_decoding_b200 import _lib
    f = FakeLibPrefix()
    monkeypatch.setattr(_lib, "load", lambda path=None: f)
    return f


def _model(checkpoint=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(0)
    m = EEG_LSTM(**kw)
    if checkpoint is not None:
        m.load_state_dict(checkpoint, strict=True)
    return m.eval()


def _ref(m):
    ref = RefEEGLSTM(input_size=m.lstm.input_size, hidden_size=m.lstm.hidden_size, num_layers=m.lstm.num_layers,
                     num_classes=m.fc[3].out_features)
    ref.load_state_dict({k: v.detach().float().cpu() for k, v in m.state_dict().items()}, strict=True)
    return ref.double().eval()


def prefix_reference(m, x, stride):
    """float64 restatement of decode_prefixes: the model's LSTM once over the whole window (torch nn.LSTM), then for
    every prefix end t_j the softmax pool of the scores over steps [0, t_j) and the eval head.  -> (lengths [P] long,
    logits [B,P,K] float64, pooled [B,P,H] float64)."""
    ref = _ref(m)
    T = x.shape[1]
    lengths = torch.clamp(torch.arange(1, -(-T // stride) + 1) * stride, max=T)
    with torch.no_grad():
        out, _ = ref.lstm(x.detach().cpu().double())
        s = ref.attn(out).squeeze(-1)                                         # [B,T]
        pooled = torch.stack([(out[:, :t] * torch.softmax(s[:, :t], dim=1).unsqueeze(-1)).sum(dim=1)
                              for t in lengths.tolist()], dim=1)
        logits = ref.fc(ref.ln(pooled))
    return lengths, logits, pooled


def truncated_reference(m, x, t):
    """RefEEGLSTM in float64 on the truncated windows x[:, :t] (the reference's own forward on the prefix)."""
    with torch.no_grad():
        return _ref(m)(x[:, :t].detach().cpu().double())


def rel_per_prefix(got, want):
    """max|d| / max|ref| over the batch, for each prefix: [B,P,K] -> [P]."""
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    return (got - want).abs().amax(dim=(0, 2)) / want.abs().amax(dim=(0, 2)).clamp_min(1e-30)


@pytest.mark.parametrize("T,stride", [(40, 7), (40, 8), (12, 50), (1, 1), (1, 3), (9, 1)])
@pytest.mark.parametrize("exact", [True, False])
def test_values_and_lengths(fake, monkeypatch, checkpoint, windows, T, stride, exact):
    """The lengths rule (T % stride != 0, stride > T, T = 1) and the logits of every prefix on both paths."""
    from neural_speech_decoding_b200 import ops
    from neural_speech_decoding_b200.lstm_eeg_model import PrefixOutputs
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:5, :T].copy())
    out = m.decode_prefixes(x, stride)
    assert isinstance(out, PrefixOutputs)
    P = -(-T // stride)
    want_len = [min((j + 1) * stride, T) for j in range(P)]
    assert out.lengths.dtype == torch.long and out.lengths.tolist() == want_len and want_len[-1] == T
    assert [tuple(t.shape) for t in out[1:]] == [(5, P, 3), (5, P, 3)]
    assert all(t.dtype == torch.float32 for t in out[1:])
    assert ("na_decoder_prefix_pool_x3" in fake.calls) == exact
    assert ("na_attention_pool_prefix_f32" in fake.calls) == (not exact)
    lengths, want, _ = prefix_reference(m, x, stride)
    assert torch.equal(lengths, out.lengths)
    assert float(rel_per_prefix(out.logits, want).max()) < 1e-5
    torch.testing.assert_close(out.probs.double(), torch.softmax(want, dim=2), atol=1e-6, rtol=0)
    for j, t in enumerate(want_len):                              # the reference's forward on each truncated window
        r = truncated_reference(m, x, t)
        assert float((out.logits[:, j].double() - r).abs().max() / r.abs().max()) < 1e-5, t
    # the last prefix is decode(x) (on the FFMA path: the fake has no na_decoder_infer_x3)
    monkeypatch.setattr(ops, "EXACT_TC", False)
    lg, _ = m.decode(x)
    torch.testing.assert_close(out.logits[:, -1], lg, atol=1e-5 * float(lg.abs().max()), rtol=0)


def test_restatement_is_the_reference_on_truncated_windows(checkpoint, windows):
    """The float64 restatement (one LSTM pass, pool per prefix) equals RefEEGLSTM on every truncated window."""
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:4, :30].copy())
    lengths, logits, _ = prefix_reference(m, x, 4)
    for j, t in enumerate(lengths.tolist()):
        torch.testing.assert_close(logits[:, j], truncated_reference(m, x, t), atol=1e-12, rtol=1e-12)


def test_other_shapes_take_the_ffma_path(fake, monkeypatch):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", True)
    m = _model(hidden_size=32, num_layers=3, num_classes=5)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(6, 23, 8, generator=g) * 3
    out = m.decode_prefixes(x, 5)
    assert fake.calls and "na_decoder_prefix_pool_x3" not in fake.calls
    assert [tuple(t.shape) for t in out[1:]] == [(6, 5, 5), (6, 5, 5)]
    lengths, want, _ = prefix_reference(m, x, 5)
    assert out.lengths.tolist() == [5, 10, 15, 20, 23]
    assert float(rel_per_prefix(out.logits, want).max()) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_inputs_and_compute_dtype(fake, monkeypatch, checkpoint, windows, dtype):
    """A 16-bit x is converted to fp32, and compute_dtype = bfloat16 still gets the fp32 (exact) path."""
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", True)
    m = _model(checkpoint)
    m.compute_dtype = torch.bfloat16
    x = torch.from_numpy(windows["X"][:3, :20].copy()).to(dtype)
    out = m.decode_prefixes(x, 6)
    assert "na_decoder_prefix_pool_x3" in fake.calls
    assert out.logits.dtype == torch.float32 and out.probs.dtype == torch.float32
    _, want, _ = prefix_reference(m, x.float(), 6)
    assert float(rel_per_prefix(out.logits, want).max()) < 1e-5


def test_train_mode_uses_eval_arithmetic(fake, checkpoint, windows):
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:3, :15].copy())
    a = m.decode_prefixes(x, 4)
    m.train()
    b = m.decode_prefixes(x, 4)
    assert m.training
    assert torch.equal(a.logits, b.logits) and torch.equal(a.probs, b.probs)


@pytest.mark.parametrize("exact", [True, False])
def test_empty_batch_launches_nothing(fake, monkeypatch, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(hidden_size=32, num_classes=5)
    n = fake.launches
    out = m.decode_prefixes(torch.zeros(0, 17, 8), 5)
    assert fake.launches == n
    assert out.lengths.tolist() == [5, 10, 15, 17]
    assert [tuple(t.shape) for t in out[1:]] == [(0, 4, 5), (0, 4, 5)]
    assert all(t.dtype == torch.float32 for t in out[1:])


def test_errors(fake, checkpoint, windows):
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:2, :20].copy())
    for bad in (0, -3):
        with pytest.raises(ValueError, match="stride"):
            m.decode_prefixes(x, bad)
    with pytest.raises(TypeError):
        m.decode_prefixes(x, 2.5)
    with pytest.raises(ValueError, match="shape"):
        m.decode_prefixes(x[0])
    with pytest.raises(ValueError, match="shape"):
        m.decode_prefixes(x[None])
    with pytest.raises(RuntimeError, match="input_size"):
        m.decode_prefixes(x[:, :, :7])
    with pytest.raises(ValueError, match="at least one step"):
        m.decode_prefixes(x[:, :0])
    m.zscore_input = True
    with pytest.raises(ValueError, match="zscore_input"):
        m.decode_prefixes(x)
    assert not fake.calls


def test_rejects_cpu_tensor(checkpoint):
    m = _model(checkpoint)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.decode_prefixes(torch.zeros(2, 10, 8))


def test_custom_ops_are_registered():
    from neural_speech_decoding_b200 import ops
    for op in (ops.decoder_prefix_pool_x3, ops.attention_pool_prefix):
        assert op in ops.all_custom_ops()
    with torch._subclasses.fake_tensor.FakeTensorMode():
        x = torch.empty(5, 31, 8)
        w, b = torch.empty(1, 48), torch.empty(1)
        assert tuple(ops.decoder_prefix_pool_x3(x, torch.empty(X3_PACKED_BYTES, dtype=torch.uint8), w, b, 10).shape) == (5, 4, 48)
        h = torch.empty(31, 32, 20)
        assert tuple(ops.attention_pool_prefix(h, 7, torch.empty(1, 20), b, 40).shape) == (7, 1, 20)


# ---- C ABI validation against the built library (paths that return before any CUDA call) -------------------------------
@pytest.fixture(scope="module")
def lib(built_lib):
    from neural_speech_decoding_b200 import _lib
    return _lib.load()


A, MIS = ctypes.c_void_p(256), ctypes.c_void_p(8)         # an aligned and a misaligned fake address


def test_prefix_pool_x3_validation(lib):
    f = lib.na_decoder_prefix_pool_x3
    assert f(A, A, A, A, A, 625, 4, 0, None) == -1
    assert b"stride" in lib.na_last_error()
    assert f(A, A, A, A, A, 625, 4, -5, None) == -1
    assert f(A, A, A, A, A, 0, 4, 25, None) == -1
    assert b"bad shape" in lib.na_last_error()
    assert f(A, A, A, A, A, 625, 0, 25, None) == -1
    assert f(A, A, A, A, A, 1 << 20, 4, 25, None) == -1
    for k in (0, 1, 4):                                     # x, packed, pooled: null, then misaligned
        args = [A] * 5
        args[k] = None
        assert f(*args, 625, 4, 25, None) == -1
        assert b"null pointer" in lib.na_last_error()
        args[k] = MIS
        assert f(*args, 625, 4, 25, None) == -2
        assert b"not 16-byte aligned" in lib.na_last_error()
    assert f(A, A, None, A, A, 625, 4, 25, None) == -1
    assert f(A, A, A, None, A, 625, 4, 25, None) == -1


def test_attention_pool_prefix_validation(lib):
    f = lib.na_attention_pool_prefix_f32
    assert f(A, A, A, A, 625, 4, 32, 48, 0, None) == -1
    assert b"stride" in lib.na_last_error()
    assert f(A, A, A, A, 0, 4, 32, 48, 25, None) == -1
    assert f(A, A, A, A, 625, 0, 32, 48, 25, None) == -1
    assert f(A, A, A, A, 625, 40, 32, 48, 25, None) == -1          # Bp < B
    assert f(A, A, A, A, 625, 4, 33, 48, 25, None) == -1           # Bp % 32
    for H in (0, 1025, -1):
        assert f(A, A, A, A, 625, 4, 32, H, 25, None) == -3
        assert b"outside [1,1024]" in lib.na_last_error()
    for k in (0, 3):                                              # h, pooled
        args = [A] * 4
        args[k] = None
        assert f(*args, 625, 4, 32, 48, 25, None) == -1
        args[k] = MIS
        assert f(*args, 625, 4, 32, 48, 25, None) == -2
    assert f(A, None, A, A, 625, 4, 32, 48, 25, None) == -1
    assert f(A, A, None, A, 625, 4, 32, 48, 25, None) == -1
