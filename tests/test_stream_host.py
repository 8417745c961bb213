"""Host-side checks of EEG_LSTM.decode_stream and of the argument validation of its two entry points.  No GPU: the decoder
runs on tests/fake_lib_stream.FakeLibStream (numpy, float64), compared with a float64 restatement (one causal LSTM pass
over everything streamed, the softmax pool of every prefix, the eval head); the validation tests call the built library
on paths that return before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch

from tests.fake_lib_stream import FakeLibStream, pool_steps
from tests.test_prefix_host import X3_PACKED_BYTES, _model, prefix_reference, rel_per_prefix

CHUNKINGS = [[40], [8] * 5, [1, 2, 17, 20], [1] * 6 + [34]]


@pytest.fixture
def fake(cpu_backend, monkeypatch):
    from neural_speech_decoding_b200 import _lib
    f = FakeLibStream()
    monkeypatch.setattr(_lib, "load", lambda path=None: f)
    return f


def stream(m, x, sizes, state=None):
    """decode_stream over x [B,T,C] in chunks of `sizes` steps -> (list of StreamOutputs, chunk ends)."""
    outs, ends, t = [], [], 0
    for n in sizes:
        out = m.decode_stream(x[:, t:t + n], state)
        state = out.state
        t += n
        outs.append(out)
        ends.append(t)
    assert t == x.shape[1]
    return outs, ends


def lstm_state_reference(m, x):
    """float64 nn.LSTM (the model's weights) over x -> (h_n, c_n) [L,B,H]."""
    lstm = torch.nn.LSTM(m.lstm.input_size, m.lstm.hidden_size, m.lstm.num_layers, batch_first=True).double()
    lstm.load_state_dict({k: v.detach().double() for k, v in m.lstm.state_dict().items()})
    with torch.no_grad():
        _, (h, c) = lstm(x.double())
    return h, c


@pytest.mark.parametrize("sizes", CHUNKINGS, ids=lambda s: "-".join(map(str, s[:4])))
@pytest.mark.parametrize("exact", [True, False])
def test_chunks_match_the_prefix_reference(fake, monkeypatch, checkpoint, windows, sizes, exact):
    """After every chunk the logits are the float64 forward of everything streamed; the final state is the float64 LSTM
    state and online-softmax state of the whole window; one chunk and many chunks agree."""
    from neural_speech_decoding_b200 import ops
    from neural_speech_decoding_b200.lstm_eeg_model import DecoderState, StreamOutputs
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:5, :40].copy())
    outs, ends = stream(m, x, sizes)
    assert all(isinstance(o, StreamOutputs) and isinstance(o.state, DecoderState) for o in outs)
    assert ("na_decoder_stream_x3" in fake.calls) == exact
    assert ("na_attention_pool_stream_f32" in fake.calls) == (not exact)
    _, want, pooled = prefix_reference(m, x, 1)
    got = torch.stack([o.logits for o in outs], dim=1)
    idx = [t - 1 for t in ends]
    assert float(rel_per_prefix(got, want[:, idx]).max()) < 1e-5
    probs = torch.stack([o.probs for o in outs], dim=1)
    torch.testing.assert_close(probs.double(), torch.softmax(want[:, idx], dim=2), atol=1e-6, rtol=0)
    st = outs[-1].state
    h64, c64 = lstm_state_reference(m, x)
    torch.testing.assert_close(st.h.double(), h64, atol=1e-6, rtol=0)
    torch.testing.assert_close(st.c.double(), c64, atol=1e-6, rtol=0)
    torch.testing.assert_close((st.pool_z / st.pool_sum[:, None]).double(), pooled[:, -1], atol=1e-6, rtol=0)
    one = m.decode_stream(x)
    torch.testing.assert_close(outs[-1].logits, one.logits, atol=1e-5, rtol=0)
    for a, b in zip(st, one.state):
        torch.testing.assert_close(a, b, atol=1e-5, rtol=1e-5)


def test_pool_restatement_is_the_softmax_pool():
    """pool_steps (the fakes' online softmax, chunked) equals the two-pass softmax pool."""
    g = np.random.default_rng(1)
    h, s = g.standard_normal((3, 30, 6)), 5 * g.standard_normal((3, 30))
    state = (np.full(3, -np.inf), np.zeros(3), np.zeros((3, 6)))
    for a, b in ((0, 11), (11, 12), (12, 30)):
        state = pool_steps(h[:, a:b], s[:, a:b], *state)
    m, l, z = state
    e = np.exp(s - s.max(axis=1, keepdims=True))
    np.testing.assert_allclose(z / l[:, None], np.einsum("bt,bth->bh", e, h) / e.sum(axis=1)[:, None], rtol=1e-12)
    np.testing.assert_array_equal(m, s.max(axis=1))


@pytest.mark.parametrize("exact", [True, False])
def test_initial_state_equals_none(fake, monkeypatch, checkpoint, windows, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:4, :12].copy())
    s0 = m.initial_stream_state(4)
    assert [tuple(t.shape) for t in s0] == [(2, 4, 48), (2, 4, 48), (4,), (4,), (4, 48)]
    assert all(t.dtype == torch.float32 for t in s0)
    assert torch.isneginf(s0.pool_max).all() and not any(t.any() for t in (s0.h, s0.c, s0.pool_sum, s0.pool_z))
    a, b = m.decode_stream(x), m.decode_stream(x, s0)
    assert torch.equal(a.logits, b.logits) and torch.equal(a.probs, b.probs)
    for u, v in zip(a.state, b.state):
        assert torch.equal(u, v)


@pytest.mark.parametrize("exact", [True, False])
def test_shapes_and_the_state_is_not_written(fake, monkeypatch, checkpoint, windows, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:3, :20].copy())
    s1 = m.decode_stream(x[:, :9]).state
    before = [t.clone() for t in s1]
    out = m.decode_stream(x[:, 9:], s1)
    assert [tuple(t.shape) for t in out[:2]] == [(3, 3), (3, 3)]
    assert [tuple(t.shape) for t in out.state] == [(2, 3, 48), (2, 3, 48), (3,), (3,), (3, 48)]
    assert all(t.dtype == torch.float32 for t in (*out[:2], *out.state))
    for t, u in zip(s1, before):
        assert torch.equal(t, u)
    assert all(t.data_ptr() != u.data_ptr() for t, u in zip(out.state, s1))


def test_other_shapes_take_the_ffma_path(fake, monkeypatch):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", True)
    m = _model(hidden_size=32, num_layers=3, num_classes=5)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(6, 23, 8, generator=g) * 3
    outs, ends = stream(m, x, [5, 1, 17])
    assert fake.calls and "na_decoder_stream_x3" not in fake.calls
    assert [tuple(t.shape) for t in outs[-1].state] == [(3, 6, 32), (3, 6, 32), (6,), (6,), (6, 32)]
    _, want, _ = prefix_reference(m, x, 1)
    got = torch.stack([o.logits for o in outs], dim=1)
    assert float(rel_per_prefix(got, want[:, [t - 1 for t in ends]]).max()) < 1e-5


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_half_inputs_and_compute_dtype(fake, monkeypatch, checkpoint, windows, dtype):
    """A 16-bit x is converted to fp32, and compute_dtype = bfloat16 still gets the fp32 (exact) path."""
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", True)
    m = _model(checkpoint)
    m.compute_dtype = torch.bfloat16
    x = torch.from_numpy(windows["X"][:3, :20].copy()).to(dtype)
    out = m.decode_stream(x)
    assert "na_decoder_stream_x3" in fake.calls
    assert out.logits.dtype == torch.float32
    _, want, _ = prefix_reference(m, x.float(), 20)
    assert float(rel_per_prefix(out.logits[:, None], want).max()) < 1e-5


def test_train_mode_uses_eval_arithmetic(fake, checkpoint, windows):
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:3, :15].copy())
    a = m.decode_stream(x)
    m.train()
    b = m.decode_stream(x)
    assert m.training
    assert torch.equal(a.logits, b.logits) and torch.equal(a.probs, b.probs)


@pytest.mark.parametrize("exact", [True, False])
def test_empty_batch_launches_nothing(fake, monkeypatch, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(hidden_size=32, num_classes=5)
    n = fake.launches
    out = m.decode_stream(torch.zeros(0, 17, 8))
    out2 = m.decode_stream(torch.zeros(0, 3, 8), out.state)
    assert fake.launches == n
    assert [tuple(t.shape) for t in out2[:2]] == [(0, 5), (0, 5)]
    assert [tuple(t.shape) for t in out2.state] == [(2, 0, 32), (2, 0, 32), (0,), (0,), (0, 32)]
    assert all(t.dtype == torch.float32 for t in (*out2[:2], *out2.state))


@pytest.mark.parametrize("exact", [True, False])
def test_misaligned_views_are_copied(fake, monkeypatch, checkpoint, windows, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:3, :20].copy())
    s = m.decode_stream(x[:, :8]).state
    xv = torch.empty(3 * 12 * 8 + 1)[1:].view(3, 12, 8)
    xv.copy_(x[:, 8:])
    sv = []
    for t in s:
        v = torch.empty(t.numel() + 1)[1:].view(t.shape)
        v.copy_(t)
        sv.append(v)
    assert xv.data_ptr() % 16 and all(v.data_ptr() % 16 for v in sv)
    a = m.decode_stream(x[:, 8:], s)
    b = m.decode_stream(xv, type(s)(*sv))
    assert torch.equal(a.logits, b.logits)


def test_errors(fake, checkpoint, windows):
    from neural_speech_decoding_b200.lstm_eeg_model import DecoderState
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:2, :20].copy())
    with pytest.raises(ValueError, match="shape"):
        m.decode_stream(x[0])
    with pytest.raises(ValueError, match="shape"):
        m.decode_stream(x[None])
    with pytest.raises(RuntimeError, match="input_size"):
        m.decode_stream(x[:, :, :7])
    with pytest.raises(ValueError, match="at least one step"):
        m.decode_stream(x[:, :0])
    s = m.initial_stream_state(2)
    with pytest.raises(ValueError, match="DecoderState"):
        m.decode_stream(x, tuple(s)[:4])
    for i, name in enumerate(DecoderState._fields):
        t = s[i]
        bad = list(s)
        bad[i] = t[..., :-1] if t.dim() > 1 else t[:1]                   # wrong shape
        with pytest.raises(RuntimeError, match=f"state.{name}"):
            m.decode_stream(x, DecoderState(*bad))
        bad[i] = t.double()
        with pytest.raises(ValueError, match=f"state.{name}"):
            m.decode_stream(x, DecoderState(*bad))
        bad[i] = torch.empty(t.shape, device="meta")
        with pytest.raises(RuntimeError, match=f"state.{name}"):
            m.decode_stream(x, DecoderState(*bad))
        bad[i] = None
        with pytest.raises(ValueError, match=f"state.{name}"):
            m.decode_stream(x, DecoderState(*bad))
    with pytest.raises(RuntimeError, match="state.h"):                     # a state for another batch size
        m.decode_stream(x, m.initial_stream_state(3))
    m.zscore_input = True
    with pytest.raises(ValueError, match="zscore_input"):
        m.decode_stream(x)
    assert not fake.calls


def test_rejects_cpu_tensor(checkpoint):
    m = _model(checkpoint)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.decode_stream(torch.zeros(2, 10, 8))


def test_custom_ops_are_registered():
    from neural_speech_decoding_b200 import ops
    for op in (ops.decoder_stream_x3, ops.attention_pool_stream):
        assert op in ops.all_custom_ops()
    with torch._subclasses.fake_tensor.FakeTensorMode():
        x = torch.empty(5, 31, 8)
        head = [torch.empty(1, 48), torch.empty(1), torch.empty(48), torch.empty(48), torch.empty(32, 48), torch.empty(32),
                torch.empty(4, 32), torch.empty(4)]
        packed = torch.empty(X3_PACKED_BYTES, dtype=torch.uint8)
        out = ops.decoder_stream_x3(x, packed, head, None, None, None, None, None)
        assert [tuple(t.shape) for t in out] == [(5, 4), (5, 4), (2, 5, 48), (2, 5, 48), (5,), (5,), (5, 48)]
        h = torch.empty(31, 32, 20)
        out = ops.attention_pool_stream(h, 7, torch.empty(1, 20), torch.empty(1), None, None, None)
        assert [tuple(t.shape) for t in out] == [(7, 20), (7,), (7,), (7, 20)]


# ---- C ABI validation against the built library (paths that return before any CUDA call) -------------------------------
@pytest.fixture(scope="module")
def lib(built_lib):
    from neural_speech_decoding_b200 import _lib
    return _lib.load()


MB = 1 << 20
MIS = ctypes.c_void_p(8)                                           # a misaligned fake address


def _addrs(n):
    """n distinct aligned fake addresses 1 MB apart (no two ranges of these sizes overlap)."""
    return [ctypes.c_void_p((k + 1) * MB) for k in range(n)]


def test_stream_x3_validation(lib):
    f = lib.na_decoder_stream_x3
    args = _addrs(22)                     # x, packed, 8 head parameters, 5 state inputs, 7 outputs
    ok = lambda a, T=625, B=4, NC=3: f(*a, T, B, NC, None)
    assert ok(args, T=0) == -1 and b"bad shape" in lib.na_last_error()
    assert ok(args, B=0) == -1
    assert ok(args, T=1 << 20) == -1
    assert ok(args, NC=0) == -3 and ok(args, NC=17) == -3
    for k in (0, 1, 15, 17, 18, 19, 20, 21):                       # x, packed, logits, h/c/m/l/z out: null, misaligned
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"null pointer" in lib.na_last_error()
        a[k] = MIS
        assert ok(a) == -2 and b"not 16-byte aligned" in lib.na_last_error()
    for k in range(2, 10):                                          # head parameters
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"null parameter pointer" in lib.na_last_error()
    for k in range(10, 15):                                         # the state inputs: all or none
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"given together" in lib.na_last_error()
        a[k] = MIS
        assert ok(a) == -2
    a = list(args)
    a[16] = MIS                                                     # probs is optional but must be aligned
    assert ok(a) == -2
    for i in range(15, 22):                                         # an output overlapping an input or another output
        for j in [0] + list(range(10, 15)) + list(range(15, i)):
            a = list(args)
            a[i] = args[j]
            assert ok(a) == -1, (i, j)
            assert b"overlaps" in lib.na_last_error()
    a = list(args)
    a[16] = ctypes.c_void_p(args[15].value + 16)                     # probs starts inside logits [4][3]
    assert ok(a) == -1 and b"probs overlaps logits" in lib.na_last_error()
    a = list(args)
    a[18] = ctypes.c_void_p(args[17].value + 2 * 4 * 48 * 4 - 16)    # c_out starts in the last row of h_out
    assert ok(a) == -1 and b"c_out overlaps h_out" in lib.na_last_error()


def test_attention_pool_stream_validation(lib):
    f = lib.na_attention_pool_stream_f32
    args = _addrs(10)                     # h, attn_w, attn_b, m_in, l_in, z_in, pooled, m_out, l_out, z_out
    ok = lambda a, T=25, B=4, Bp=32, H=48: f(*a, T, B, Bp, H, None)
    assert ok(args, T=0) == -1 and b"bad shape" in lib.na_last_error()
    assert ok(args, B=0) == -1
    assert ok(args, B=40) == -1                                     # Bp < B
    assert ok(args, Bp=33) == -1                                    # Bp % 32
    for H in (0, 1025, -1):
        assert ok(args, H=H) == -3 and b"outside [1,1024]" in lib.na_last_error()
    for k in (0, 6, 7, 8, 9):                                       # h and the outputs
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"null pointer" in lib.na_last_error()
        a[k] = MIS
        assert ok(a) == -2
    for k in (1, 2):
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"null parameter pointer" in lib.na_last_error()
    for k in (3, 4, 5):
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"given together" in lib.na_last_error()
        a[k] = MIS
        assert ok(a) == -2
