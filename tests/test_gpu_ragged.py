"""``decode`` / ``decode_stream`` with per-row ``lengths`` on the GPU: the exact tensor-core kernel
(``na_decoder_stream_ragged_x3``) bit for bit against ``decode`` of each row's own prefix and against the plain stream,
the FFMA path (``na_attention_pool_stream_ragged_f32``) against the float64 restatement of tests/test_prefix_host.py,
streams fed different numbers of steps per call, every tile layout, shapes off the tensor-core tier and the raw call.
``x`` past every row's length is NaN throughout.  Error: max|d| / max|ref| over the rows compared (DESIGN 10h)."""
import numpy as np
import pytest
import torch

from tests.test_prefix_host import prefix_reference

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
# The exact path's logits of a row are decode(x[:, :len]) bit for bit, whose error in the middle of the shipped windows is
# up to 1.08e-5 (the fp16 hi + lo operand split of the per-step h; DESIGN 10d, 10f).
EXACT_TOL = 2e-5


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
def ragged_calls(monkeypatch):
    """Counts the calls of ops.decoder_stream_ragged_x3 (the exact tensor-core path)."""
    from neural_speech_decoding_b200 import ops
    n = [0]
    real = ops.decoder_stream_ragged_x3

    def counted(*a, **k):
        n[0] += 1
        return real(*a, **k)
    monkeypatch.setattr(ops, "decoder_stream_ragged_x3", counted)
    return n


@pytest.fixture(scope="module")
def reference(checkpoint, windows):
    """float64 logits of every prefix of the 324 shipped windows [B, 625, K]."""
    from tests.test_prefix_host import _model
    m = _model(checkpoint)
    return prefix_reference(m, torch.from_numpy(windows["X"]), 1)[1]


def make_model(dev, sd=None, seed=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    if seed is not None:
        torch.manual_seed(seed)
    m = EEG_LSTM(**kw)
    if sd is not None:
        m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


def padded(x, lengths):
    """x with every step past each row's length replaced by NaN."""
    x = x.clone()
    for b, n in enumerate(lengths.tolist()):
        x[b, n:] = float("nan")
    return x


def rows_at(want, t):
    """want [B,P,K] of every prefix -> [B,K] at prefix t[b] (t >= 1)."""
    return want[torch.arange(len(t)), torch.as_tensor(t) - 1]


def shipped_lengths(B, T=625):
    g = torch.Generator().manual_seed(11)
    n = torch.randint(1, T + 1, (B,), generator=g)
    n[:4] = torch.tensor([1, 2, T - 1, T])
    return n


@pytest.mark.parametrize("fused", [True, False])
def test_ragged_windows(dev, checkpoint, windows, reference, exact_tc, ragged_calls, fused):
    """The 324 shipped windows with lengths in [1, 625] (1, 2, 624 and 625 included), NaN past every length.  Exact path:
    row b is decode(x[:, :len_b])[b] bit for bit (same B, same tile layout).  Both paths against float64 (2e-5 exact,
    1e-5 FFMA), argmax identical."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"]).to(dev)
    n = shipped_lengths(x.shape[0])
    logits, probs = m.decode(padded(x, n), lengths=n)
    assert ragged_calls[0] == (1 if fused else 0)
    if fused:
        for t in torch.unique(n).tolist():
            rows = (n == t).nonzero().squeeze(1).to(dev)
            lg, pr = m.decode(x[:, :t])
            assert torch.equal(logits[rows], lg[rows]), t
            assert torch.equal(probs[rows], pr[rows]), t
    want = rows_at(reference, n)
    r = rel(logits.cpu(), want)
    print(f"fused={fused}: ragged windows vs float64 {r:.2e}")
    assert r < (EXACT_TOL if fused else FP32_TOL)
    assert torch.equal(logits.argmax(1).cpu(), want.argmax(1))


@pytest.mark.parametrize("fused", [True, False])
def test_full_lengths_are_the_plain_calls(dev, checkpoint, windows, exact_tc, fused):
    """lengths = T everywhere: decode_stream with lengths is decode_stream without them bit for bit, state included, on
    both paths.  decode with lengths is decode bit for bit on the exact path; on the FFMA path decode runs the H = 48
    kernel from zeros and the stream the generic kernel, so the two agree within 1e-5."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"]).to(dev)
    full = torch.full((x.shape[0],), x.shape[1])
    a, b = m.decode_stream(x), m.decode_stream(x, lengths=full)
    assert torch.equal(a.logits, b.logits) and torch.equal(a.probs, b.probs)
    for name, u, v in zip(a.state._fields, a.state, b.state):
        assert torch.equal(u, v), name
    lg, pr = m.decode(x, lengths=full)
    assert torch.equal(lg, b.logits) and torch.equal(pr, b.probs)
    d_lg, d_pr = m.decode(x)
    if fused:
        assert torch.equal(lg, d_lg) and torch.equal(pr, d_pr)
    else:
        assert rel(lg.cpu(), d_lg.cpu()) < FP32_TOL


def ragged_chunks(B, T, seed, most=40):
    """Per-call step counts [calls][B]: random in [0, most], capped at what each row has left, until every row is done."""
    g = np.random.default_rng(seed)
    done, calls = np.zeros(B, np.int64), []
    while (done < T).any():
        n = np.minimum(g.integers(0, most + 1, size=B), T - done)
        calls.append(n)
        done += n
    return calls


def run_ragged(m, x, calls, check):
    """decode_stream over the per-row step counts `calls`, each chunk built per row and padded with NaN; check(out, state
    before, n, t) after every call (t: the steps every row has received) -> the last state."""
    B, state, done = x.shape[0], None, np.zeros(x.shape[0], np.int64)
    for n in calls:
        chunk = torch.full((B, max(int(n.max()), 1), x.shape[2]), float("nan"), device=x.device)
        for b in range(B):
            chunk[b, :n[b]] = x[b, done[b]:done[b] + n[b]]
        out = m.decode_stream(chunk, state, lengths=torch.from_numpy(n))
        done = done + n
        check(out, state, n, done)
        state = out.state
    return state


@pytest.mark.parametrize("fused", [True, False])
def test_ragged_streams(dev, checkpoint, windows, reference, exact_tc, fused):
    """Every shipped window streamed in random per-row amounts of 0 to 40 steps per call.  Exact path: after every call row
    b's logits and probs are decode(x[:, :t_b])[b] bit for bit, rows given 0 steps return their state bit for bit, and
    the last state is the one-chunk state bit for bit.  FFMA path: within 1e-5 of float64 after every call, and the last
    state is the one-chunk state bit for bit."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"]).to(dev)
    B, T = x.shape[0], x.shape[1]
    worst = [0.0]

    def check(out, before, n, t):
        if before is not None:
            keep = torch.from_numpy(n == 0).to(dev)
            for name, a, s in zip(out.state._fields, out.state, before):
                k = (slice(None), keep) if a.dim() == 3 else keep
                assert torch.equal(a[k], s[k]), name
        live = t > 0
        if fused:
            for tt in np.unique(t[live]).tolist():
                rows = torch.from_numpy(t == tt).to(dev)
                lg, pr = m.decode(x[:, :tt])
                assert torch.equal(out.logits[rows], lg[rows]), tt
                assert torch.equal(out.probs[rows], pr[rows]), tt
        want = rows_at(reference[torch.from_numpy(live)], t[live])
        got = out.logits[torch.from_numpy(live).to(dev)].cpu()
        worst[0] = max(worst[0], rel(got, want))
        assert torch.equal(got.argmax(1), want.argmax(1))
    calls = ragged_chunks(B, T, seed=5)
    state = run_ragged(m, x, calls, check)
    print(f"fused={fused}: {len(calls)} calls, worst vs float64 {worst[0]:.2e}")
    assert worst[0] < (EXACT_TOL if fused else FP32_TOL)
    one = m.decode_stream(x).state
    for name, a, b in zip(one._fields, state, one):
        assert torch.equal(a, b), name


@pytest.mark.parametrize("fused", [True, False])
def test_fresh_stream_given_nothing(dev, checkpoint, windows, exact_tc, fused):
    """A fresh stream given 0 steps gets NaN logits (an empty pool, 0 / 0) and the fresh state; its neighbours are those
    of a call in which it took its steps, bit for bit."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:40, :100].copy()).to(dev)
    n = torch.full((40,), 100)
    a = m.decode_stream(x, lengths=n)
    n[[0, 17]] = 0
    b = m.decode_stream(padded(x, n), lengths=n)
    keep = n > 0
    assert bool(torch.isnan(b.logits[[0, 17]]).all())
    assert torch.equal(a.logits[keep.to(dev)], b.logits[keep.to(dev)])
    fresh = m.initial_stream_state(2, dev)
    for name, u, f in zip(b.state._fields, b.state, fresh):
        assert torch.equal(u[:, [0, 17]] if u.dim() == 3 else u[[0, 17]], f), name


def _raw(m, x, state, lengths, pad):
    """na_decoder_stream_ragged_x3 on NaN-filled output buffers `pad` rows longer than B: every row below B is written,
    nothing past it."""
    from neural_speech_decoding_b200 import _lib, ops
    B, T = x.shape[0], x.shape[1]
    NC = m.fc[3].out_features
    nan = lambda *shape: torch.full(shape, float("nan"), dtype=torch.float32, device=x.device)
    logits, probs = nan(B + pad, NC), nan(B + pad, NC)
    h, c = nan(2 * B * 48 + pad), nan(2 * B * 48 + pad)            # [2][B][48], then padding
    mo, lo, zo = nan(B + pad), nan(B + pad), nan(B + pad, 48)
    head = [ops._f32c(t.detach()) for t in m._head_params()]
    ins = [t.contiguous() for t in state]
    lens = lengths.to(device=x.device, dtype=torch.int32)
    _lib.call("na_decoder_stream_ragged_x3", x.data_ptr(), m._packed_x3().data_ptr(), *[t.data_ptr() for t in head],
              *[t.data_ptr() for t in ins], lens.data_ptr(), logits.data_ptr(), probs.data_ptr(), h.data_ptr(),
              c.data_ptr(), mo.data_ptr(), lo.data_ptr(), zo.data_ptr(), T, B, NC, ops._stream())
    n = 2 * B * 48
    for name, t, k in (("logits", logits, B), ("probs", probs, B), ("m", mo, B), ("l", lo, B), ("z", zo, B), ("h", h, n),
                       ("c", c, n)):
        assert bool(torch.isnan(t[k:]).all()), f"{name}: write past B"
        assert bool(torch.isfinite(t[:k]).all()), f"{name}: row not written"
    return logits[:B], h[:n].view(2, B, 48), c[:n].view(2, B, 48), mo[:B], lo[:B], zo[:B]


def test_tile_layouts_against_ffma(dev, checkpoint, exact_tc):
    """Row-replicated short tiles (R = 4, 2), full tiles, several tiles per CTA and a partial last quarter, two calls with
    random lengths (0 included in the second): the raw call writes exactly the rows b < B and equals the API bit for bit;
    the exact and FFMA paths agree within 2e-5."""
    m = make_model(dev, checkpoint)
    for B in (1, 31, 33, 97, 128, 148 * 128 + 77, 2 * 148 * 128 + 5):
        gen = torch.Generator().manual_seed(B)
        x = (torch.randn(B, 20, 8, generator=gen) * 20.0).to(dev)
        n1 = torch.randint(1, 13, (B,), generator=gen)
        n2 = torch.randint(0, 9, (B,), generator=gen)
        x1, x2 = padded(x[:, :12], n1), padded(x[:, 12:], n2)
        exact_tc(True)
        a1 = m.decode_stream(x1, lengths=n1)
        a2 = m.decode_stream(x2, a1.state, lengths=n2)
        r2 = _raw(m, x2.contiguous(), a1.state, n2, pad=64)
        assert torch.equal(a2.logits, r2[0]), B
        for name, a, b in zip(a2.state._fields, a2.state, r2[1:]):
            assert torch.equal(a, b), (B, name)
        exact_tc(False)
        f1 = m.decode_stream(x1, lengths=n1)
        f2 = m.decode_stream(x2, f1.state, lengths=n2)
        ra, rb = rel(a1.logits.cpu(), f1.logits.cpu()), rel(a2.logits.cpu(), f2.logits.cpu())
        print(f"B={B}: exact vs FFMA {ra:.2e} / {rb:.2e}")
        assert ra < 2 * FP32_TOL and rb < 2 * FP32_TOL, (B, ra, rb)


@pytest.mark.parametrize("shape", [dict(hidden_size=32, num_layers=3, num_classes=5),
                                   dict(hidden_size=70, num_layers=1, num_classes=3)])
def test_ffma_shapes(dev, exact_tc, ragged_calls, shape):
    """Shapes outside the tensor-core tier: ragged windows and a ragged stream within 1e-5 of float64."""
    exact_tc(True)
    m = make_model(dev, seed=3, **shape)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(37, 60, 8, generator=g) * 5
    _, want, _ = prefix_reference(m, x, 1)
    xd = x.to(dev)
    n = torch.randint(1, 61, (37,), generator=g)
    lg, _ = m.decode(padded(xd, n), lengths=n)
    r = rel(lg.cpu(), rows_at(want, n))
    worst = [r]

    def check(out, before, k, t):
        live = t > 0
        worst[0] = max(worst[0], rel(out.logits[torch.from_numpy(live).to(dev)].cpu(), rows_at(want[torch.from_numpy(live)], t[live])))
    run_ragged(m, xd, ragged_chunks(37, 60, seed=6, most=15), check)
    print(f"{shape}: windows {r:.2e}, stream {worst[0]:.2e}")
    assert worst[0] < FP32_TOL
    assert ragged_calls[0] == 0


def test_every_rcp_knob_value(dev, checkpoint, windows):
    """The launcher runs every instantiation of the x3_rcp_fma knob; each row is decode of its prefix bit for bit."""
    from neural_speech_decoding_b200 import _lib
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:70, :200].copy()).to(dev)
    n = torch.tensor([200, 1, 57, 133] * 17 + [9, 200])
    try:
        for nr in (0, 1, 2, 3):
            _lib.call("na_set_tuning", b"x3_rcp_fma", nr)
            lg, _ = m.decode(padded(x, n), lengths=n)
            for t in torch.unique(n).tolist():
                rows = (n == t).to(dev)
                assert torch.equal(lg[rows], m.decode(x[:, :t])[0][rows]), (nr, t)
    finally:
        _lib.call("na_set_tuning", b"x3_rcp_fma", 0)
