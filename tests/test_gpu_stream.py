"""``EEG_LSTM.decode_stream`` on the GPU: the exact tensor-core kernel (``na_decoder_stream_x3``) bit for bit against
``decode`` and ``model.lstm`` on everything streamed so far, both paths against the float64 restatement of
tests/test_prefix_host.py, the FFMA path (``na_attention_pool_stream_f32``) at other shapes, every tile layout, streams of
different ages and a NaN stream in one batch.  Error of a chunk end: max|d| / max|ref| over the batch (DESIGN 10g)."""
import numpy as np
import pytest
import torch

from tests.test_prefix_host import prefix_reference, rel_per_prefix

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
# The exact path's logits after a chunk are decode(x[:, :t]) bit for bit, whose error in the middle of the shipped windows
# is up to 1.08e-5 at t = 175 (the fp16 hi + lo operand split of the per-step h; DESIGN 10d, 10f).
EXACT_TOL = 2e-5
CHUNKINGS = [[625], [125] * 5, [25] * 25, [1, 2, 17, 105, 500], [1] * 40 + [585]]


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
    """Counts the calls of ops.decoder_stream_x3 (the exact tensor-core path)."""
    from neural_speech_decoding_b200 import ops
    n = [0]
    real = ops.decoder_stream_x3

    def counted(*a, **k):
        n[0] += 1
        return real(*a, **k)
    monkeypatch.setattr(ops, "decoder_stream_x3", counted)
    return n


def make_model(dev, sd=None, seed=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    if seed is not None:
        torch.manual_seed(seed)
    m = EEG_LSTM(**kw)
    if sd is not None:
        m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


def stream(m, x, sizes, state=None):
    """decode_stream over x in chunks of `sizes` steps -> (list of StreamOutputs, chunk ends)."""
    outs, ends, t = [], [], 0
    for n in sizes:
        out = m.decode_stream(x[:, t:t + n], state)
        state = out.state
        t += n
        outs.append(out)
        ends.append(t)
    assert t == x.shape[1]
    return outs, ends


@pytest.mark.parametrize("sizes", CHUNKINGS, ids=["625", "125x5", "25x25", "1-2-17-105-500", "1x40-585"])
def test_exact_path_is_decode_bit_for_bit(dev, checkpoint, windows, exact_tc, fused_calls, sizes):
    """The 324 shipped windows: after every chunk, logits / probs are decode(x[:, :t]) bit for bit; the final h / c are
    model.lstm(x)'s h_n / c_n on the fused path bit for bit; the final state is the one-chunk state bit for bit."""
    exact_tc(True)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"]).to(dev)
    outs, ends = stream(m, x, sizes)
    assert fused_calls[0] == len(sizes)
    for out, t in zip(outs, ends):
        lg, pr = m.decode(x[:, :t], want_probs=True)
        assert torch.equal(out.logits, lg), t
        assert torch.equal(out.probs, pr), t
    with torch.no_grad():
        _, (h_n, c_n) = m.lstm(x)
    st = outs[-1].state
    assert torch.equal(st.h, h_n) and torch.equal(st.c, c_n)
    one = m.decode_stream(x).state
    for name, a, b in zip(st._fields, st, one):
        assert torch.equal(a, b), name


@pytest.mark.parametrize("fused", [True, False])
def test_shipped_windows_against_float64(dev, checkpoint, windows, exact_tc, fused_calls, fused):
    """Chunks of 25 steps: every chunk end within 1e-5 of the float64 restatement on the FFMA path (2e-5 on the exact
    path, see EXACT_TOL), argmax identical; the state's pool_z / pool_sum is the float64 pooled vector of the prefix."""
    exact_tc(fused)
    tol = EXACT_TOL if fused else FP32_TOL
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"])
    outs, ends = stream(m, x.to(dev), [25] * 25)
    assert fused_calls[0] == (25 if fused else 0)
    lengths, want, pooled = prefix_reference(m, x, 25)
    assert lengths.tolist() == ends
    got = torch.stack([o.logits for o in outs], dim=1).cpu()
    r = rel_per_prefix(got, want)
    print(f"fused={fused}: worst chunk end {float(r.max()):.2e} (t = {ends[int(r.argmax())]}), median {float(r.median()):.2e}")
    assert float(r.max()) < tol
    assert torch.equal(got.argmax(dim=2), want.argmax(dim=2))
    zs = torch.stack([(o.state.pool_z / o.state.pool_sum[:, None]) for o in outs], dim=1).cpu()
    rp = rel_per_prefix(zs, pooled)
    print(f"fused={fused}: pooled vector, worst chunk end {float(rp.max()):.2e}")
    assert float(rp.max()) < tol


@pytest.mark.parametrize("shape", [dict(hidden_size=32, num_layers=3, num_classes=5),
                                   dict(hidden_size=70, num_layers=1, num_classes=3)])
def test_ffma_shapes(dev, exact_tc, fused_calls, shape):
    """EXACT_TC = False, and shapes outside the tensor-core tier: chunked equals one chunk bit for bit, and both are
    within 1e-5 of float64."""
    m = make_model(dev, seed=3, **shape)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(37, 60, 8, generator=g) * 5
    for flag in (True, False):
        exact_tc(flag)
        outs, ends = stream(m, x.to(dev), [17, 1, 30, 12])
        one = m.decode_stream(x.to(dev))
        assert torch.equal(outs[-1].logits, one.logits) and torch.equal(outs[-1].probs, one.probs)
        for name, a, b in zip(one.state._fields, outs[-1].state, one.state):
            assert torch.equal(a, b), name
        _, want, _ = prefix_reference(m, x, 1)
        r = float(rel_per_prefix(torch.stack([o.logits for o in outs], dim=1).cpu(), want[:, [t - 1 for t in ends]]).max())
        print(f"{shape} EXACT_TC={flag}: {r:.2e}")
        assert r < FP32_TOL
    assert fused_calls[0] == 0


def test_flagship_ffma_chunked_is_one_chunk(dev, checkpoint, windows, exact_tc):
    exact_tc(False)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:50, :200].copy()).to(dev)
    outs, _ = stream(m, x, [3, 97, 100])
    one = m.decode_stream(x)
    assert torch.equal(outs[-1].logits, one.logits)
    for name, a, b in zip(one.state._fields, outs[-1].state, one.state):
        assert torch.equal(a, b), name


def _raw(m, x, state, pad):
    """na_decoder_stream_x3 on NaN-filled output buffers `pad` rows longer than B: every row below B is written, nothing
    past it."""
    from neural_speech_decoding_b200 import _lib, ops
    B, T = x.shape[0], x.shape[1]
    NC = m.fc[3].out_features
    nan = lambda *shape: torch.full(shape, float("nan"), dtype=torch.float32, device=x.device)
    logits, probs = nan(B + pad, NC), nan(B + pad, NC)
    h, c = nan(2 * B * 48 + pad), nan(2 * B * 48 + pad)            # [2][B][48], then padding
    mo, lo, zo = nan(B + pad), nan(B + pad), nan(B + pad, 48)
    head = [ops._f32c(t.detach()) for t in m._head_params()]
    ins = [None] * 5 if state is None else [t.contiguous() for t in state]
    _lib.call("na_decoder_stream_x3", x.data_ptr(), m._packed_x3().data_ptr(), *[t.data_ptr() for t in head],
              *[ops._ptr(t) for t in ins], logits.data_ptr(), probs.data_ptr(), h.data_ptr(), c.data_ptr(),
              mo.data_ptr(), lo.data_ptr(), zo.data_ptr(), T, B, NC, ops._stream())
    n = 2 * B * 48
    for name, t, k in (("logits", logits, B), ("probs", probs, B), ("m", mo, B), ("l", lo, B), ("z", zo, B), ("h", h, n),
                       ("c", c, n)):
        assert bool(torch.isnan(t[k:]).all()), f"{name}: write past B"
        assert bool(torch.isfinite(t[:k]).all()), f"{name}: row not written"
    return logits[:B], h[:n].view(2, B, 48), c[:n].view(2, B, 48), mo[:B], lo[:B], zo[:B]


def test_tile_layouts_against_ffma(dev, checkpoint, exact_tc):
    """Row-replicated short tiles (R = 4, 2), full tiles, several tiles per CTA, and a partial last quarter: the raw call
    writes exactly the rows b < B; the API's exact path agrees with the raw call bit for bit and with the FFMA path within
    2e-5 after each of two chunks."""
    m = make_model(dev, checkpoint)
    for B in (1, 31, 33, 64, 97, 128, 148 * 128 + 77, 2 * 148 * 128 + 5):
        gen = torch.Generator().manual_seed(B)
        x = (torch.randn(B, 20, 8, generator=gen) * 20.0).to(dev)
        exact_tc(True)
        a1 = m.decode_stream(x[:, :12])
        a2 = m.decode_stream(x[:, 12:], a1.state)
        r1 = _raw(m, x[:, :12].contiguous(), None, pad=64)
        r2 = _raw(m, x[:, 12:].contiguous(), r1[1:], pad=64)
        assert torch.equal(a2.logits, r2[0]), B
        for name, a, b in zip(a2.state._fields, a2.state, r2[1:]):
            assert torch.equal(a, b), (B, name)
        exact_tc(False)
        f1 = m.decode_stream(x[:, :12])
        f2 = m.decode_stream(x[:, 12:], f1.state)
        ra, rb = rel(a1.logits.cpu(), f1.logits.cpu()), rel(a2.logits.cpu(), f2.logits.cpu())
        print(f"B={B}: exact vs FFMA {ra:.2e} / {rb:.2e}")
        assert ra < 2 * FP32_TOL and rb < 2 * FP32_TOL, (B, ra, rb)


@pytest.mark.parametrize("fused", [True, False])
def test_streams_of_different_ages(dev, checkpoint, windows, exact_tc, fused):
    """Some rows are reset to initial_stream_state midway; each row's logits are decode of that row's own history (within
    1e-6, and the same argmax: the batches differ, and so do the tile layouts; on the FFMA path within 1e-5, since decode
    runs the H = 48 kernel from zeros and the stream the generic kernel from its state)."""
    exact_tc(fused)
    tol = 1e-6 if fused else FP32_TOL
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:64, :300].copy()).to(dev)
    reset, t_reset = torch.tensor([3, 10, 40, 63], device=dev), 100
    state, t = None, 0
    for n in (50, 50, 75, 125):
        if t == t_reset:
            fresh = m.initial_stream_state(len(reset), dev)
            state = type(state)(*[s.clone() for s in state])
            for s, f in zip(state, fresh):
                if s.dim() == 3:
                    s[:, reset] = f
                else:
                    s[reset] = f
        out = m.decode_stream(x[:, t:t + n], state)
        state, t = out.state, t + n
        if t > t_reset:
            old = torch.ones(64, dtype=torch.bool, device=dev)
            old[reset] = False
            want_old, _ = m.decode(x[old][:, :t])
            want_new, _ = m.decode(x[reset][:, t_reset:t])
            r = max(rel(out.logits[old].cpu(), want_old.cpu()), rel(out.logits[reset].cpu(), want_new.cpu()))
            print(f"fused={fused} t={t}: {r:.2e}")
            assert r < tol
            assert torch.equal(out.logits[reset].argmax(1), want_new.argmax(1))


@pytest.mark.parametrize("fused", [True, False])
def test_nan_stays_in_its_stream(dev, checkpoint, windows, exact_tc, fused):
    """A NaN sample in one stream's chunk makes that row NaN for every later call; every other row is bit-identical to a
    run without it."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:40, :150].copy()).to(dev)
    xn = x.clone()
    xn[7, 60, 3] = float("nan")
    a, _ = stream(m, x, [50, 50, 50])
    b, _ = stream(m, xn, [50, 50, 50])
    keep = torch.arange(40, device=dev) != 7
    assert torch.equal(a[0].logits, b[0].logits)
    for oa, ob in zip(a[1:], b[1:]):
        assert bool(torch.isnan(ob.logits[7]).all()) and bool(torch.isnan(ob.state.pool_z[7]).all())
        assert torch.equal(oa.logits[keep], ob.logits[keep])
        for name, sa, sb in zip(oa.state._fields, oa.state, ob.state):
            k = (slice(None), keep) if sa.dim() == 3 else keep
            assert torch.equal(sa[k], sb[k]), name


def test_every_rcp_knob_value(dev, checkpoint, windows):
    """The launcher runs every instantiation of the x3_rcp_fma knob; chunked equals decode bit for bit for each."""
    from neural_speech_decoding_b200 import _lib
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:70, :200].copy()).to(dev)
    try:
        for nr in (0, 1, 2, 3):
            _lib.call("na_set_tuning", b"x3_rcp_fma", nr)
            outs, ends = stream(m, x, [9, 91, 100])
            for out, t in zip(outs, ends):
                assert torch.equal(out.logits, m.decode(x[:, :t])[0]), (nr, t)
    finally:
        _lib.call("na_set_tuning", b"x3_rcp_fma", 0)


def test_misaligned_views(dev, checkpoint, windows, exact_tc):
    """Views of x and of the state at an odd float offset give the result of aligned copies on both paths."""
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:45, :60].copy()).to(dev)

    def odd(t):
        v = torch.empty(t.numel() + 1, dtype=torch.float32, device=dev)[1:].view(t.shape)
        v.copy_(t)
        assert v.data_ptr() % 16 != 0
        return v
    for fused in (True, False):
        exact_tc(fused)
        s = m.decode_stream(x[:, :20]).state
        a = m.decode_stream(x[:, 20:].contiguous(), s)
        b = m.decode_stream(odd(x[:, 20:]), type(s)(*[odd(t) for t in s]))
        assert torch.equal(a.logits, b.logits) and torch.equal(a.probs, b.probs), fused
        for name, u, v in zip(a.state._fields, a.state, b.state):
            assert torch.equal(u, v), (fused, name)
