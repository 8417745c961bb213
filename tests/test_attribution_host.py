"""Host-side checks of EEG_LSTM.input_gradients / integrated_gradients: shapes, argument errors, which path runs, the
per-window gradient scaling and the quadrature.  No GPU: the FFMA path runs on tests/fake_lib.FakeLib (cpu_backend) and
the exact tensor-core path on tests/fake_attribution.FakeInputGradX3 (float64 autograd of the reference)."""
import math

import pytest
import torch

from oracle.torch_ref import RefEEGLSTM


@pytest.fixture
def fast(cpu_backend, monkeypatch):
    from neural_speech_decoding_b200 import ops
    from tests.fake_attribution import FakeInputGradX3
    fake = FakeInputGradX3()
    monkeypatch.setattr(ops, "decoder_input_grad_x3", fake)
    monkeypatch.setattr(ops, "EXACT_TC_TRAIN", True)
    return fake


def _model(checkpoint=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(0)
    m = EEG_LSTM(**kw)
    if checkpoint is not None:
        m.load_state_dict(checkpoint, strict=True)
    return m.eval()


def _ref_saliency(m, x, target):
    ref = RefEEGLSTM(input_size=m.lstm.input_size, hidden_size=m.lstm.hidden_size, num_layers=m.lstm.num_layers,
                     num_classes=m.fc[3].out_features).double().eval()
    ref.load_state_dict({k: v.double() for k, v in m.state_dict().items()})
    xg = x.double().requires_grad_(True)
    lg = ref(xg)
    (g,) = torch.autograd.grad(lg.gather(1, target[:, None]).sum(), xg)
    return lg, g


def test_shapes_and_empty_batch(fast, checkpoint, windows):
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:4, :30].copy())
    out = m.input_gradients(x)
    assert tuple(out.logits.shape) == (4, 3) and tuple(out.attributions.shape) == (4, 30, 8)
    assert out.target.dtype == torch.long and out.delta is None and out.attributions.dtype == torch.float32
    assert torch.equal(out.target, out.logits.argmax(dim=1))
    n = len(fast.calls)
    e = m.input_gradients(x[:0])
    assert tuple(e.logits.shape) == (0, 3) and tuple(e.attributions.shape) == (0, 30, 8) and tuple(e.target.shape) == (0,)
    ig = m.integrated_gradients(x[:0], steps=4)
    assert tuple(ig.attributions.shape) == (0, 30, 8) and tuple(ig.delta.shape) == (0,)
    assert len(fast.calls) == n                                    # no launch for B == 0


def test_errors(fast, checkpoint, windows):
    from neural_speech_decoding_b200 import ops
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:2, :20].copy())
    with pytest.raises(ValueError, match="out of range"):
        m.input_gradients(x, target=3)
    with pytest.raises(ValueError, match="out of range"):
        m.input_gradients(x, target=torch.tensor([0, -1]))
    with pytest.raises(ValueError, match="target must be"):
        m.input_gradients(x, target=torch.tensor([0, 1, 2]))
    with pytest.raises(ValueError, match="baseline"):
        m.integrated_gradients(x, baseline=torch.zeros(2, 20, 7))
    with pytest.raises(ValueError, match="steps"):
        m.integrated_gradients(x, steps=0)


def test_cpu_tensor_raises(checkpoint):
    m = _model(checkpoint)
    with pytest.raises(RuntimeError):
        m.input_gradients(torch.zeros(2, 10, 8))


@pytest.mark.parametrize("shape", [{}, {"hidden_size": 32, "num_layers": 3}])
@pytest.mark.parametrize("zscore", [False, True])
@pytest.mark.parametrize("exact_train", [False, True])
def test_routing(fast, monkeypatch, checkpoint, windows, shape, zscore, exact_train):
    from neural_speech_decoding_b200 import ops
    monkeypatch.setattr(ops, "EXACT_TC_TRAIN", exact_train)
    m = _model(checkpoint if not shape else None, **shape)
    m.zscore_input = zscore
    x = torch.from_numpy(windows["X"][:3, :16].copy())
    want_fast = exact_train and not shape and not zscore
    if zscore:                                 # the FFMA path has no gradient through the z-score stage
        with pytest.raises(RuntimeError, match="z-score"):
            m.input_gradients(x)
        assert not fast.calls
        return
    out = m.input_gradients(x, target=1)
    assert bool(fast.calls) == want_fast
    _, g = _ref_saliency(m, x, torch.full((3,), 1))
    d = (out.attributions.double() - g).abs().amax(dim=(1, 2)) / g.abs().amax(dim=(1, 2))
    assert float(d.max()) < 1e-5


def test_side_effects(fast, checkpoint, windows):
    m = _model(checkpoint).train()
    for p in m.parameters():
        p.grad = torch.ones_like(p)
    cache = dict(m._pack_cache)
    x = torch.from_numpy(windows["X"][:2, :12].copy())
    m.integrated_gradients(x, steps=2)
    assert m.training and dict(m._pack_cache) == cache
    assert all(torch.equal(p.grad, torch.ones_like(p)) for p in m.parameters())


def test_per_window_dz_scale():
    from neural_speech_decoding_b200 import ops
    dz = torch.tensor([[3.0, -0.5], [1e-6, 2e-6], [float("nan"), 1.0], [0.0, 0.0]])
    sdz, inv = ops._scale_dz_rows(dz)
    for b in (0, 1):
        s = 1.0 / float(inv[b])
        assert math.log2(s) == round(math.log2(s))                           # a power of two
        assert 32.0 < float(sdz[b].abs().max()) <= 64.0                       # max|dz_b| -> (2^5, 2^6]
        assert torch.equal(sdz[b] * inv[b], dz[b])                            # exact round trip
    assert torch.isnan(inv[2]) and torch.isnan(sdz[2]).all()                  # a NaN window keeps its NaN to itself
    assert torch.isfinite(inv[[0, 1, 3]]).all() and torch.equal(sdz[3], dz[3])


def test_quadrature(fast, monkeypatch, checkpoint, windows):
    """Midpoint weights: the batch holds the baseline, then steps x B windows at alpha_k = (k + 1/2) / steps."""
    m = _model(checkpoint)
    x = torch.from_numpy(windows["X"][:2, :10].copy())
    base = torch.full_like(x, 0.25)
    ig = m.integrated_gradients(x, target=torch.tensor([0, 2]), baseline=base, steps=4)
    shapes = [c[0] for c in fast.calls]
    assert shapes == [(2, 10, 8), (2 + 4 * 2, 10, 8)]
    assert torch.equal(fast.calls[1][1], torch.tensor([0, 2] * 5))
    # float64 midpoint quadrature of the reference
    want = torch.zeros(2, 10, 8, dtype=torch.float64)
    for k in range(4):
        a = (k + 0.5) / 4
        _, g = _ref_saliency(m, base + a * (x - base), torch.tensor([0, 2]))
        want += g / 4
    want *= (x - base).double()
    assert torch.allclose(ig.attributions.double(), want, rtol=1e-5, atol=1e-6 * float(want.abs().max()))
    lx, _ = _ref_saliency(m, x, torch.tensor([0, 2]))
    lb, _ = _ref_saliency(m, base, torch.tensor([0, 2]))
    dF = lx.gather(1, torch.tensor([[0], [2]]))[:, 0] - lb.gather(1, torch.tensor([[0], [2]]))[:, 0]
    assert torch.allclose(ig.delta.double(), want.sum(dim=(1, 2)) - dF, atol=1e-5)
