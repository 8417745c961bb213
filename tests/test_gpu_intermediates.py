"""EEG_LSTM.decode_intermediates on the GPU: attention weights over time, pooled vector and LayerNorm output from the
fused inference kernels, against the reference module read with forward hooks (the idiom the method replaces).
Tolerance: rel = max|d| / max|ref| per tensor."""
import numpy as np
import pytest
import torch

from oracle import numpy_oracle as no
from oracle.torch_ref import RefEEGLSTM

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
TC_TOL = 2e-2


def rel(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from neural_speech_decoding_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def make_model(dev, sd=None, seed=None, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    if seed is not None:
        torch.manual_seed(seed)
    m = EEG_LSTM(**kw)
    if sd is not None:
        m.load_state_dict(sd, strict=True)
    return m.to(dev).eval()


def hooked_reference(model, x_cpu):
    """fp32 CPU reference with forward hooks on attn and ln: (logits, attention [B,T], pooled [B,H], embedding [B,H])."""
    lstm = model.lstm
    ref = RefEEGLSTM(lstm.input_size, lstm.hidden_size, lstm.num_layers, model.fc[3].out_features)
    ref.load_state_dict({k: v.detach().float().cpu() for k, v in model.state_dict().items()}, strict=True)
    ref.eval()
    seen = {}
    h1 = ref.attn.register_forward_hook(lambda mod, i, o: seen.__setitem__("scores", o.squeeze(-1)))
    h2 = ref.ln.register_forward_hook(lambda mod, i, o: seen.update(pooled=i[0], emb=o))
    with torch.no_grad():
        logits = ref(x_cpu.float())
    h1.remove(); h2.remove()
    return logits.numpy(), torch.softmax(seen["scores"], dim=1).numpy(), seen["pooled"].numpy(), seen["emb"].numpy()


def check_against_reference(out, ref, tol):
    lg, att, zp, emb = ref
    assert rel(out.logits.cpu(), lg) < tol
    assert rel(out.attention.cpu(), att) < tol, rel(out.attention.cpu(), att)
    assert rel(out.pooled.cpu(), zp) < tol, rel(out.pooled.cpu(), zp)
    assert rel(out.embedding.cpu(), emb) < tol, rel(out.embedding.cpu(), emb)


def test_exact_tier_shipped_checkpoint_all_windows(dev, checkpoint, windows):
    from neural_speech_decoding_b200 import ops
    assert ops.EXACT_TC
    m = make_model(dev, checkpoint)
    x = torch.from_numpy(windows["X"])
    out = m.decode_intermediates(x.to(dev))
    assert [tuple(t.shape) for t in out] == [(324, 3), (324, 3), (324, 625), (324, 48), (324, 48)]
    assert all(t.dtype == torch.float32 and t.device == x.to(dev).device for t in out)
    check_against_reference(out, hooked_reference(m, x), FP32_TOL)
    assert np.abs(out.attention.double().sum(1).cpu().numpy() - 1.0).max() < 1e-6
    lg, pr = m.decode(x.to(dev))
    assert torch.equal(out.logits, lg) and torch.equal(out.probs, pr)


def _x3_raw(m, x, B, T, pad):
    """The exact-tier entry point on sentinel-filled buffers `pad` elements longer than needed."""
    from neural_speech_decoding_b200 import _lib, ops
    head = [ops._f32c(t) for t in m._head_params()]
    NC = head[6].shape[0]
    sent = -12345.0
    buf = lambda n: torch.full((n + pad,), sent, dtype=torch.float32, device=x.device)
    lg, pr, sc, zp, emb = buf(B * NC), buf(B * NC), buf(T * B), buf(B * 48), buf(B * 48)
    _lib.call("na_decoder_infer_x3_ex", x.data_ptr(), m._packed_x3().data_ptr(), *[t.data_ptr() for t in head],
              lg.data_ptr(), pr.data_ptr(), sc.data_ptr(), zp.data_ptr(), emb.data_ptr(), T, B, NC, ops._stream())
    for t in (lg, pr, sc, zp, emb):
        assert bool((t[-pad:] == sent).all()), "write past B"
    return (lg[:-pad].view(B, NC), pr[:-pad].view(B, NC), ops.attention_softmax(sc[:-pad].view(T, B)),
            zp[:-pad].view(B, 48), emb[:-pad].view(B, 48))


@pytest.mark.parametrize("T", [1, 2, 3, 30, 625])
def test_exact_tier_tile_layouts(dev, checkpoint, T):
    from neural_speech_decoding_b200 import ops
    m = make_model(dev, checkpoint)
    gen = torch.Generator().manual_seed(T)
    for B in [1, 31, 33, 64, 65, 129, 148 * 32 + 5, 148 * 128 + 77]:
        x = (torch.randn(B, T, 8, generator=gen) * 20.0).to(dev)
        got = _x3_raw(m, x, B, T, pad=4096)
        api = m.decode_intermediates(x)
        for a, b in zip(got, api):
            assert torch.equal(a, b), (B, T)
        ops.EXACT_TC = False
        try:
            ffma = m.decode_intermediates(x)
        finally:
            ops.EXACT_TC = True
        for name, a, b in zip(("logits", "probs", "attention", "pooled", "embedding"), got, ffma):
            if name != "probs":              # probs follow from the logits: a 1e-5 logit difference moves them by more
                assert rel(a.cpu(), b.cpu()) < FP32_TOL, (name, B, T, rel(a.cpu(), b.cpu()))
        assert rel(got[1].cpu(), torch.softmax(got[0].double(), dim=1).cpu()) < 1e-6
        if T == 1:
            assert bool((got[2] == 1.0).all())


@pytest.mark.parametrize("H", [48, 96, 144, 192])
def test_16bit_tier(dev, H):
    m = make_model(dev, seed=11 + H, hidden_size=H)
    gen = torch.Generator().manual_seed(H)
    x = (torch.randn(77, 40, 8, generator=gen) * 20.0).to(dev)
    exact = m.decode_intermediates(x)
    m.compute_dtype = torch.bfloat16
    half = m.decode_intermediates(x)
    lg, pr = m.decode(x)
    assert torch.equal(half.logits, lg) and torch.equal(half.probs, pr)
    for name, a, b in zip(half._fields, half, exact):
        assert rel(a.cpu(), b.cpu()) < TC_TOL, (name, H, rel(a.cpu(), b.cpu()))
    check_against_reference(exact, hooked_reference(m, x.cpu()), FP32_TOL)


@pytest.mark.parametrize("num_layers", [1, 3])
def test_generic_shapes_ffma(dev, num_layers):
    m = make_model(dev, seed=5 + num_layers, num_classes=5, hidden_size=32, num_layers=num_layers)
    gen = torch.Generator().manual_seed(num_layers)
    x = torch.randn(45, 100, 8, generator=gen) * 5.0
    out = m.decode_intermediates(x.to(dev))
    assert [tuple(t.shape) for t in out] == [(45, 5), (45, 5), (45, 100), (45, 32), (45, 32)]
    check_against_reference(out, hooked_reference(m, x), FP32_TOL)


def test_zscore_front_stage(dev, checkpoint, windows):
    m = make_model(dev, checkpoint)
    m.zscore_input = True
    X = windows["X"][:40]
    out = m.decode_intermediates(torch.from_numpy(X).to(dev))
    check_against_reference(out, hooked_reference(m, torch.from_numpy(no.zscore_window(X).astype(np.float32))), FP32_TOL)


def test_nan_window_and_bf16_input(dev, checkpoint, windows):
    m = make_model(dev, checkpoint)
    X = windows["X"][:9].copy()
    X[3, 100, 2] = np.nan
    out = m.decode_intermediates(torch.from_numpy(X).to(dev))
    att = out.attention.cpu().numpy()
    assert np.isnan(att[3]).all()
    assert np.isfinite(np.delete(att, 3, axis=0)).all()
    clean = m.decode_intermediates(torch.from_numpy(np.delete(X, 3, axis=0)).to(dev))
    assert torch.equal(torch.from_numpy(np.delete(att, 3, axis=0)), clean.attention.cpu())
    # bf16 input selects the 16-bit tier
    xb = torch.from_numpy(windows["X"][:20]).to(dev).bfloat16()
    half = m.decode_intermediates(xb)
    lg, _ = m.decode(xb)
    assert torch.equal(half.logits, lg)
    exact = m.decode_intermediates(xb.float())
    assert rel(half.attention.cpu(), exact.attention.cpu()) < TC_TOL


def test_predictor_explain(dev, checkpoint, windows, tmp_path):
    from neural_speech_decoding_b200.lstm_eeg_model import SimplePredictor

    class Identity:
        def transform(self, chunk):
            return chunk

    pth = tmp_path / "ck.pth"
    torch.save(dict(checkpoint), pth)
    p = SimplePredictor(str(pth), sr=125, preprocessor=Identity())
    probs, label, attention = p.explain(windows["X"][5])
    out = p.model.decode_intermediates(torch.from_numpy(windows["X"][5:6]).to(dev))
    assert attention.shape == (625,) and attention.dtype == np.float32
    assert np.array_equal(attention, out.attention[0].cpu().numpy())
    assert np.array_equal(probs, out.probs[0].cpu().numpy())
    assert label == p.class_names[int(np.argmax(probs))]
    probs_p, label_p = p.predict(windows["X"][5])
    assert np.array_equal(probs, probs_p) and label == label_p
