"""Host-side checks of ``decode`` / ``decode_stream`` with per-row ``lengths`` and of the argument validation of their two
entry points.  No GPU: the decoder runs on tests/fake_lib_ragged.FakeLibRagged (numpy, float64), compared with the
float64 restatement of tests/test_prefix_host.py (row b of a ragged call is the prefix x[b, :t_b] of its stream); the
validation tests call the built library on paths that return before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch

from tests.fake_lib_ragged import FakeLibRagged
from tests.test_prefix_host import X3_PACKED_BYTES, _model, prefix_reference

RAGGED_X3, RAGGED_POOL = "na_decoder_stream_ragged_x3", "na_attention_pool_stream_ragged_f32"


@pytest.fixture
def fake(cpu_backend, monkeypatch):
    from neural_speech_decoding_b200 import _lib
    f = FakeLibRagged()
    monkeypatch.setattr(_lib, "load", lambda path=None: f)
    return f


def padded(x, lengths):
    """x with every step past each row's length replaced by NaN."""
    x = x.clone()
    for b, n in enumerate(lengths):
        x[b, n:] = float("nan")
    return x


def at_lengths(want, lengths):
    """want [B,P,K] of every prefix (stride 1) -> [B,K] at prefix lengths[b]."""
    return torch.stack([want[b, n - 1] for b, n in enumerate(lengths)])


def rel(got, want):
    got, want = got.detach().double(), want.detach().double()
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("exact", [True, False])
def test_ragged_windows_match_the_prefix_reference(fake, monkeypatch, checkpoint, windows, exact):
    """Row b of decode(x, lengths) is the float64 forward of x[b, :lengths[b]]; NaN past a length changes nothing."""
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:6, :40].copy())
    lengths = [1, 2, 17, 39, 40, 25]
    logits, probs = m.decode(padded(x, lengths), lengths=lengths)
    assert (RAGGED_X3 in fake.calls) == exact and (RAGGED_POOL in fake.calls) == (not exact)
    assert "na_decoder_stream_x3" not in fake.calls and "na_attention_pool_stream_f32" not in fake.calls
    _, want, _ = prefix_reference(m, x, 1)
    w = at_lengths(want, lengths)
    assert rel(logits, w) < 1e-5
    torch.testing.assert_close(probs.double(), torch.softmax(w, dim=1), atol=1e-6, rtol=0)
    lg2, pr2 = m.decode(padded(x, lengths), want_probs=False, lengths=torch.tensor(lengths))
    assert torch.equal(lg2, logits) and pr2.numel() == 0


@pytest.mark.parametrize("exact", [True, False])
def test_ragged_stream_matches_the_prefix_reference(fake, monkeypatch, checkpoint, windows, exact):
    """Rows consume their 40 steps in different amounts per call (0 included): after every call row b's logits are the
    float64 forward of everything it received, a row given 0 steps keeps its state, and the last state is the one-chunk
    state."""
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    B, T = 5, 40
    x = torch.from_numpy(windows["X"][:B, :T].copy())
    _, want, _ = prefix_reference(m, x, 1)
    g = np.random.default_rng(7)
    done, state = np.zeros(B, dtype=np.int64), None
    while (done < T).any():
        n = np.minimum(g.integers(0, 12, size=B), T - done)
        Tc = max(int(n.max()), 1)
        chunk = torch.full((B, Tc, 8), float("nan"))
        for b in range(B):
            chunk[b, :n[b]] = x[b, done[b]:done[b] + n[b]]
        out = m.decode_stream(chunk, state, lengths=n.tolist())
        for b in np.flatnonzero(n == 0):
            if state is not None:
                for name, a, s in zip(out.state._fields, out.state, state):
                    k = (slice(None), b) if a.dim() == 3 else b
                    assert torch.equal(a[k], s[k]), name
        done += n
        live = np.flatnonzero(done > 0)
        got = out.logits[live]
        assert rel(got, torch.stack([want[b, done[b] - 1] for b in live])) < 1e-5
        state = out.state
    one = m.decode_stream(x)
    for name, a, b in zip(one.state._fields, state, one.state):
        torch.testing.assert_close(a, b, atol=1e-5, rtol=1e-5, msg=name)


@pytest.mark.parametrize("exact", [True, False])
def test_full_lengths_are_the_plain_call(fake, monkeypatch, checkpoint, windows, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:4, :20].copy())
    s = m.decode_stream(x[:, :7]).state
    a, b = m.decode_stream(x[:, 7:], s), m.decode_stream(x[:, 7:], s, lengths=[13] * 4)
    torch.testing.assert_close(a.logits, b.logits, atol=1e-6, rtol=0)
    for name, u, v in zip(a.state._fields, a.state, b.state):
        torch.testing.assert_close(u, v, atol=1e-6, rtol=1e-6, msg=name)


@pytest.mark.parametrize("exact", [True, False])
def test_fresh_stream_given_nothing_is_nan(fake, monkeypatch, checkpoint, windows, exact):
    """A fresh stream given 0 steps has the logits of an empty pool (0 / 0: NaN) and the fresh state."""
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:3, :10].copy())
    out = m.decode_stream(x, lengths=[10, 0, 4])
    assert bool(torch.isnan(out.logits[1]).all()) and bool(torch.isfinite(out.logits[[0, 2]]).all())
    fresh = m.initial_stream_state(1)
    for name, a, f in zip(out.state._fields, out.state, fresh):
        assert torch.equal(a[:, 1:2] if a.dim() == 3 else a[1:2], f), name


@pytest.mark.parametrize("form", ["list", "tuple", "numpy", "int64", "int32", "int16", "uint8"])
def test_lengths_forms(fake, checkpoint, windows, form):
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:3, :10].copy())
    n = [3, 10, 7]
    conv = {"list": list, "tuple": tuple, "numpy": np.array, "int64": torch.tensor,
            "int32": lambda v: torch.tensor(v, dtype=torch.int32), "int16": lambda v: torch.tensor(v, dtype=torch.int16),
            "uint8": lambda v: torch.tensor(v, dtype=torch.uint8)}[form]
    a = m.decode(x, lengths=n)[0]
    assert torch.equal(m.decode(x, lengths=conv(n))[0], a)


def test_other_shapes_take_the_ffma_path(fake, monkeypatch):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", True)
    m = _model(hidden_size=32, num_layers=3, num_classes=5)
    x = torch.randn(6, 23, 8, generator=torch.Generator().manual_seed(3)) * 3
    lengths = [23, 1, 5, 12, 22, 2]
    out = m.decode_stream(padded(x, lengths), lengths=lengths)
    assert RAGGED_POOL in fake.calls and RAGGED_X3 not in fake.calls
    assert [tuple(t.shape) for t in out.state] == [(3, 6, 32), (3, 6, 32), (6,), (6,), (6, 32)]
    _, want, _ = prefix_reference(m, x, 1)
    assert rel(out.logits, at_lengths(want, lengths)) < 1e-5


@pytest.mark.parametrize("exact", [True, False])
def test_empty_batch_launches_nothing(fake, monkeypatch, exact):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC", exact)
    m = _model(hidden_size=32, num_classes=5)
    n = fake.launches
    out = m.decode_stream(torch.zeros(0, 17, 8), lengths=[])
    lg, pr = m.decode(torch.zeros(0, 5, 8), lengths=torch.zeros(0, dtype=torch.int64))
    assert fake.launches == n and not fake.calls
    assert [tuple(t.shape) for t in out[:2]] == [(0, 5), (0, 5)] and tuple(lg.shape) == (0, 5) and tuple(pr.shape) == (0, 5)
    assert [tuple(t.shape) for t in out.state] == [(2, 0, 32), (2, 0, 32), (0,), (0,), (0, 32)]


def test_errors(fake, checkpoint, windows):
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:2, :20].copy())
    for call in (m.decode_stream, lambda x, lengths: m.decode(x, lengths=lengths)):
        for bad in ([[3, 4]], [3], [3, 4, 5], torch.tensor([[3, 4]])):
            with pytest.raises(ValueError, match="shape"):
                call(x, lengths=bad)
        for bad in ([3.0, 4.0], torch.tensor([3.0, 4.0]), torch.tensor([True, True])):
            with pytest.raises(ValueError, match="integers"):
                call(x, lengths=bad)
        for bad in ([-1, 4], [3, 21], torch.tensor([21, 3])):
            with pytest.raises(ValueError, match=r"lengths must lie in \["):
                call(x, lengths=bad)
    m.decode_stream(x, lengths=[0, 20])
    with pytest.raises(ValueError, match=r"in \[1, 20\]"):
        m.decode(x, lengths=[0, 20])
    with pytest.raises(RuntimeError, match="state.h"):                     # a state for another batch size
        m.decode_stream(x, m.initial_stream_state(3), lengths=[1, 2])
    with pytest.raises(ValueError, match="at least one step"):
        m.decode(x[:, :0], lengths=[0, 0])
    calls = list(fake.calls)
    m.zscore_input = True
    with pytest.raises(ValueError, match="zscore_input"):
        m.decode_stream(x, lengths=[1, 2])
    with pytest.raises(ValueError, match="zscore_input"):
        m.decode(x, lengths=[1, 2])
    assert fake.calls == calls


def test_rejects_cpu_tensor(checkpoint):
    m = _model(checkpoint)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.decode_stream(torch.zeros(2, 10, 8), lengths=[1, 2])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.decode(torch.zeros(2, 10, 8), lengths=[1, 2])


def test_custom_ops_are_registered():
    from neural_speech_decoding_b200 import ops
    for op in (ops.decoder_stream_ragged_x3, ops.attention_pool_stream_ragged):
        assert op in ops.all_custom_ops()
    with torch._subclasses.fake_tensor.FakeTensorMode():
        x = torch.empty(5, 31, 8)
        head = [torch.empty(1, 48), torch.empty(1), torch.empty(48), torch.empty(48), torch.empty(32, 48), torch.empty(32),
                torch.empty(4, 32), torch.empty(4)]
        packed = torch.empty(X3_PACKED_BYTES, dtype=torch.uint8)
        lengths = torch.empty(5, dtype=torch.int32)
        out = ops.decoder_stream_ragged_x3(x, packed, head, None, None, None, None, None, lengths)
        assert [tuple(t.shape) for t in out] == [(5, 4), (5, 4), (2, 5, 48), (2, 5, 48), (5,), (5,), (5, 48)]
        h = torch.empty(31, 32, 20)
        out = ops.attention_pool_stream_ragged(h, 7, torch.empty(1, 20), torch.empty(1), None, None, None,
                                               torch.empty(7, dtype=torch.int32))
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


def test_stream_ragged_x3_validation(lib):
    f = lib.na_decoder_stream_ragged_x3
    args = _addrs(23)                     # x, packed, 8 head parameters, 5 state inputs, lengths, 7 outputs
    ok = lambda a, T=625, B=4, NC=3: f(*a, T, B, NC, None)
    assert ok(args, T=0) == -1 and b"na_decoder_stream_ragged_x3: bad shape" in lib.na_last_error()
    assert ok(args, B=0) == -1
    assert ok(args, T=1 << 20) == -1
    assert ok(args, NC=0) == -3 and ok(args, NC=17) == -3
    for k in (0, 1, 15, 16, 18, 19, 20, 21, 22):                   # x, packed, lengths, logits, h/c/m/l/z out
        a = list(args)
        a[k] = None
        assert ok(a) == -1 and b"null pointer" in lib.na_last_error()
        a[k] = MIS
        assert ok(a) == -2 and b"not 16-byte aligned" in lib.na_last_error()
    a = list(args)
    a[15] = None
    assert ok(a) == -1 and b"null pointer lengths" in lib.na_last_error()
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
    a[17] = MIS                                                     # probs is optional but must be aligned
    assert ok(a) == -2
    for i in range(16, 23):                                         # an output overlapping an input or another output
        for j in [0] + list(range(10, 16)) + list(range(16, i)):
            a = list(args)
            a[i] = args[j]
            assert ok(a) == -1, (i, j)
            assert b"overlaps" in lib.na_last_error()
    a = list(args)
    a[20] = ctypes.c_void_p(args[15].value + 16)                     # m_out starts at lengths[4] of [8]
    assert ok(a, B=8) == -1 and b"m_out overlaps an input" in lib.na_last_error()


def test_attention_pool_stream_ragged_validation(lib):
    f = lib.na_attention_pool_stream_ragged_f32
    args = _addrs(11)                     # h, attn_w, attn_b, m_in, l_in, z_in, lengths, pooled, m_out, l_out, z_out
    ok = lambda a, T=25, B=4, Bp=32, H=48: f(*a, T, B, Bp, H, None)
    assert ok(args, T=0) == -1 and b"bad shape" in lib.na_last_error()
    assert ok(args, B=0) == -1
    assert ok(args, B=40) == -1                                     # Bp < B
    assert ok(args, Bp=33) == -1                                    # Bp % 32
    for H in (0, 1025, -1):
        assert ok(args, H=H) == -3 and b"outside [1,1024]" in lib.na_last_error()
    for k in (0, 6, 7, 8, 9, 10):                                   # h, lengths and the outputs
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
