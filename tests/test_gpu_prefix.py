"""``EEG_LSTM.decode_prefixes`` on the GPU: the exact tensor-core kernel (``na_decoder_prefix_pool_x3``) and the FFMA
path (``na_attention_pool_prefix_f32``) against float64 -- the causal restatement of tests/test_prefix_host.py and
oracle.torch_ref.RefEEGLSTM on the truncated windows -- and against the existing eval paths.  Error of a prefix:
max|d| / max|ref| over the batch (DESIGN section 10f)."""
import numpy as np
import pytest
import torch

from tests.test_prefix_host import prefix_reference, rel_per_prefix, truncated_reference

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
# exact tensor-core path, a prefix in the middle of a window: measured 1.08e-5 at t = 175 of the shipped windows (median
# over the 25 prefixes 2.3e-6; 1.7e-6 for the whole window).  The pooled vector of a short prefix averages fewer steps of
# the per-step h, whose error from the fp16 hi + lo operand split is 6.2e-5 (DESIGN section 10d); decode(x[:, :t]) on the
# same tier computes the same h values.  The FFMA path holds FP32_TOL (2.2e-6 at the same prefix).
EXACT_PREFIX_TOL = 2e-5


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
    """Counts the calls of ops.decoder_prefix_pool_x3 (the exact tensor-core path)."""
    from neural_speech_decoding_b200 import ops
    n = [0]
    real = ops.decoder_prefix_pool_x3

    def counted(*a, **k):
        n[0] += 1
        return real(*a, **k)
    monkeypatch.setattr(ops, "decoder_prefix_pool_x3", counted)
    return n


def make_model(dev, sd=None, seed=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    if seed is not None:
        torch.manual_seed(seed)
    m = EEG_LSTM(**kw)
    if sd is not None:
        m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


@pytest.mark.parametrize("fused", [True, False])
def test_shipped_windows_against_float64(dev, checkpoint, windows, exact_tc, fused_calls, fused):
    """All 324 shipped windows at stride 25: every prefix within 1e-5 of the float64 restatement on the FFMA path (2e-5 on
    the exact tensor-core path, see EXACT_PREFIX_TOL), argmax identical."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"])
    out = m.decode_prefixes(x.to(dev), 25)
    assert fused_calls[0] == (1 if fused else 0)
    assert out.lengths.tolist() == list(range(25, 626, 25))
    assert [tuple(t.shape) for t in out[1:]] == [(324, 25, 3), (324, 25, 3)]
    lengths, want, _ = prefix_reference(m, x, 25)
    r = rel_per_prefix(out.logits, want)
    worst = int(lengths[int(r.argmax())])
    print(f"fused={fused}: worst prefix {float(r.max()):.2e} (t = {worst}), median {float(r.median()):.2e}")
    if fused:                                  # the existing exact-tier call on that prefix, for comparison
        lt, _ = m.decode(x[:, :worst].contiguous().to(dev))
        print(f"decode(x[:, :{worst}]) on the exact tier: {rel(lt.cpu(), truncated_reference(m, x, worst)):.2e}")
    assert float(r.max()) < (EXACT_PREFIX_TOL if fused else FP32_TOL)
    assert torch.equal(out.logits.cpu().argmax(dim=2), want.argmax(dim=2))
    # probs are the head kernel's softmax of its own logits
    assert float((out.probs.double() - torch.softmax(out.logits.double(), dim=2)).abs().max()) < 1e-6


@pytest.mark.parametrize("fused", [True, False])
def test_truncated_windows_against_reference(dev, checkpoint, windows, exact_tc, fused):
    """Stride 1 on the 324 shipped windows: the prefix of length t against RefEEGLSTM in float64 on x[:, :t]."""
    exact_tc(fused)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"])
    out = m.decode_prefixes(x.to(dev), 1)
    assert out.lengths.tolist() == list(range(1, 626))
    for t in (1, 2, 17, 125, 313, 624, 625):
        want = truncated_reference(m, x, t)
        got = out.logits[:, t - 1].cpu()
        r = rel(got, want)
        print(f"fused={fused} t={t}: {r:.2e}")
        assert r < (EXACT_PREFIX_TOL if fused else FP32_TOL), (t, r)
        assert torch.equal(got.argmax(dim=1), want.argmax(dim=1)), t


def test_agrees_with_decode(dev, checkpoint, windows, exact_tc):
    """The exact path against the existing exact-tier calls: the whole window against decode / decode_intermediates,
    and prefixes against decode on the truncated windows."""
    from neural_speech_decoding_b200 import ops
    exact_tc(True)
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"]).to(dev)
    out = m.decode_prefixes(x, 25)
    lg, _ = m.decode(x)
    r_last = rel(out.logits[:, -1].cpu(), lg.cpu())
    print(f"last prefix vs decode: {r_last:.2e}")
    assert r_last < 2e-6
    assert torch.equal(out.logits[:, -1].argmax(dim=1), lg.argmax(dim=1))
    head = [p.detach() for p in m._head_params()]
    pooled = ops.decoder_prefix_pool_x3(x, m._packed_x3(), head[0], head[1], 25)
    ex = m.decode_intermediates(x)
    r_pool = rel(pooled[:, -1].cpu(), ex.pooled.cpu())
    print(f"last pooled vector vs decode_intermediates: {r_pool:.2e}, bit-identical: {torch.equal(pooled[:, -1], ex.pooled)}")
    assert r_pool < 1e-6
    for t in (25, 100, 175, 250, 400, 600):
        lt, _ = m.decode(x[:, :t].contiguous())
        r = rel(out.logits[:, t // 25 - 1].cpu(), lt.cpu())
        print(f"t={t} vs decode(x[:, :t]): {r:.2e}")
        assert r < 2 * FP32_TOL, (t, r)


def _raw(m, x, stride, pad):
    """na_decoder_prefix_pool_x3 on a NaN-filled buffer `pad` elements longer than needed: every element of the result is
    written, nothing past it."""
    from neural_speech_decoding_b200 import _lib, ops
    B, T = x.shape[0], x.shape[1]
    P = -(-T // stride)
    n = B * P * 48
    buf = torch.full((n + pad,), float("nan"), dtype=torch.float32, device=x.device)
    head = [ops._f32c(t.detach()) for t in m._head_params()]
    _lib.call("na_decoder_prefix_pool_x3", x.data_ptr(), m._packed_x3().data_ptr(), head[0].data_ptr(), head[1].data_ptr(),
              buf.data_ptr(), T, B, stride, ops._stream())
    assert bool(torch.isnan(buf[n:]).all()), "write past B"
    assert bool(torch.isfinite(buf[:n]).all()), "element not written"
    return buf[:n].view(B, P, 48)


def test_tile_layouts_against_ffma(dev, checkpoint, exact_tc):
    """Row-replicated short tiles (R = 4, 2), full tiles, several tiles per CTA, and a partial last quarter: the raw call
    writes exactly [B][P][48], is bit-identical from run to run and to the API, and agrees with the FFMA path."""
    from neural_speech_decoding_b200 import ops
    m = make_model(dev, checkpoint)
    head = [ops._f32c(t.detach()) for t in m._head_params()]
    cases = [(1, 30, 7), (31, 30, 30), (33, 30, 31), (64, 30, 4), (65, 30, 1), (97, 29, 5), (128, 30, 6),
             (129, 30, 45), (300, 30, 8), (148 * 128 + 77, 3, 2)]
    for B, T, stride in cases:
        gen = torch.Generator().manual_seed(B + T)
        x = (torch.randn(B, T, 8, generator=gen) * 20.0).to(dev)
        got = _raw(m, x, stride, pad=4096)
        assert torch.equal(got, _raw(m, x, stride, pad=4096)), (B, T, stride)
        exact_tc(True)
        api = m.decode_prefixes(x, stride)
        assert torch.equal(api.logits, ops._prefix_head(got, head)[0]), (B, T, stride)
        exact_tc(False)
        try:
            ffma = m.decode_prefixes(x, stride)
            L = m.lstm.num_layers
            h = ops.window_zscore(x, T, T, False, True, False)
            for l in range(L):
                h = ops.lstm_layer_fwd(h, *m._packed(l), None, 1.0, False)[0]
            ffma_pooled = ops.attention_pool_prefix(h, B, head[0], head[1], stride)
        finally:
            exact_tc(True)
        r_pool, r_lg = rel(got.cpu(), ffma_pooled.cpu()), rel(api.logits.cpu(), ffma.logits.cpu())
        print(f"B={B} T={T} stride={stride}: pooled {r_pool:.2e}, logits {r_lg:.2e}")
        assert r_pool < 2 * FP32_TOL and r_lg < 2 * FP32_TOL, (B, T, stride, r_pool, r_lg)


def test_every_rcp_knob_value(dev, checkpoint, windows):
    """The launcher runs every instantiation of the x3_rcp_fma knob; each is within EXACT_PREFIX_TOL of float64."""
    from neural_speech_decoding_b200 import _lib
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:70, :200].copy())
    _, want, _ = prefix_reference(m, x, 9)
    try:
        for nr in (0, 1, 2, 3):
            _lib.call("na_set_tuning", b"x3_rcp_fma", nr)
            r = float(rel_per_prefix(m.decode_prefixes(x.to(dev), 9).logits, want).max())
            print(f"x3_rcp_fma={nr}: {r:.2e}")
            assert r < EXACT_PREFIX_TOL, (nr, r)
    finally:
        _lib.call("na_set_tuning", b"x3_rcp_fma", 0)


@pytest.mark.parametrize("shape", [dict(hidden_size=32, num_layers=3, num_classes=5),
                                   dict(hidden_size=100, num_layers=1, num_classes=16),
                                   dict(hidden_size=200, num_layers=2, num_classes=1),
                                   dict(hidden_size=300, num_layers=1, num_classes=3),
                                   dict(hidden_size=600, num_layers=1, num_classes=4)])
def test_other_shapes_on_ffma(dev, exact_tc, fused_calls, shape):
    """Shapes outside the tensor-core tier, one per instantiation of the FFMA pool kernel (H <= 64, 128, 256, 512,
    1024), within 1e-5 of float64."""
    exact_tc(True)
    m = make_model(dev, seed=3, **shape)
    g = torch.Generator().manual_seed(4)
    T = 40 if shape["hidden_size"] <= 64 else 17
    x = torch.randn(37, T, 8, generator=g) * 5
    for stride in (1, 6, 100):
        out = m.decode_prefixes(x.to(dev), stride)
        _, want, _ = prefix_reference(m, x, stride)
        r = float(rel_per_prefix(out.logits, want).max())
        print(f"{shape} stride={stride}: {r:.2e}")
        assert r < FP32_TOL, (shape, stride, r)
    assert fused_calls[0] == 0


def test_misaligned_view(dev, checkpoint, windows, exact_tc):
    """A contiguous view at an odd float offset gives the result of an aligned copy on both paths."""
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"][:45, :60].copy()).to(dev)
    buf = torch.empty(x.numel() + 1, dtype=torch.float32, device=dev)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    assert v.data_ptr() % 16 != 0
    for fused in (True, False):
        exact_tc(fused)
        a, b = m.decode_prefixes(x, 7), m.decode_prefixes(v, 7)
        assert torch.equal(a.logits, b.logits) and torch.equal(a.probs, b.probs), fused
