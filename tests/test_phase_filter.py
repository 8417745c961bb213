"""SURVEY 8(f) rank 1: the preprocessing filter in front of the decoder, on the GPU (opt-in).  Pins: the reference's own
filtered windows and the logits of its filtered path (tests/golden/ref_outputs_3class.npz)."""
import numpy as np
import pytest
import torch


def test_gpu_filter_is_opt_in():
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    with pytest.raises(PermissionError):
        PhaseCouplingFilterGPU()


@pytest.mark.gpu
def test_gpu_filter_matches_reference_windows_and_logits(windows, checkpoint, golden_dir):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    f = np.load(golden_dir / "ref_outputs_3class.npz")
    dev = torch.device("cuda:0")
    pre = PhaseCouplingFilterGPU(sr=125, tailoring_lambda=1.25e-29, device=dev, accept_noncommercial_terms=True)
    X = torch.from_numpy(windows["X"]).to(dev)
    Y = pre.transform_batch(X)
    pre.check()
    got = Y.cpu().numpy()
    want = f["filtered_subset"]
    sub = got[f["filtered_subset_idx"]]
    err = np.abs(sub - want).max(axis=(1, 2)) / np.abs(want).max(axis=(1, 2))
    assert err.max() < 1e-5, err.max()
    # single-window entry point (the reference's PreProcessor contract) == the batched one, bit for bit
    one = pre.transform(windows["X"][7])
    assert one.dtype == np.float32 and one.shape == (625, 8) and np.array_equal(one, got[7])
    with pytest.raises(ValueError):
        pre.transform(windows["X"][:2])
    # the whole live path on the GPU: filter -> decoder, against the reference's filtered-path logits of all 324 windows
    m = EEG_LSTM()
    m.load_state_dict(checkpoint, strict=True)
    m = m.to(dev).eval()
    with torch.inference_mode():
        logits = m(Y).cpu().numpy()
    ref = f["logits_filtered_b1"]
    assert np.abs(logits - ref).max() / np.abs(ref).max() < 5e-5
    margin = np.sort(ref, axis=1)
    safe = (margin[:, -1] - margin[:, -2]) > 1e-3
    assert safe.sum() >= 320 and np.array_equal(logits.argmax(1)[safe], ref.argmax(1)[safe])


@pytest.mark.gpu
def test_gpu_filter_random_windows_vs_oracle_and_predictor(checkpoint, tmp_path):
    from oracle.phase_filter import phase_coupling_filter
    from neural_speech_decoding_b200.lstm_eeg_model import SimplePredictor
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    rng = np.random.default_rng(3)
    t = np.arange(625)[:, None] / 125.0
    x = (rng.standard_normal((20, 625, 8)) * 2.0 + 3.0 * np.sin(2 * np.pi * (8 + np.arange(8))[None, None, :] * t[None])).astype(np.float32)
    x[3] = 0.0                                     # an all-zero window: phases are 0, P = 0, the filter is the identity
    # edge windows: a dead channel (r = 0 at every t, paired in the kernel's complex FFT with a live one), a constant
    # channel, a single nonzero sample, whole windows at 1e5 and 1e-30, one channel 30 decades below its FFT partner
    x[4, :, 2] = 0.0
    x[5, :, 5] = 0.0
    x[6, :, 1] = 4.0
    x[7, :, 6] = 0.0
    x[7, 300, 6] = -5.0
    x[8] *= np.float32(1e5)
    x[9] *= np.float32(1e-30)
    x[10, :, 3] *= np.float32(1e-30)
    dev = torch.device("cuda:0")
    for lam in (1.25e-29, 1e-25, 0.0):
        pre = PhaseCouplingFilterGPU(tailoring_lambda=lam, device=dev, accept_noncommercial_terms=True)
        got = pre.transform_batch(torch.from_numpy(x).to(dev)).cpu().numpy()
        pre.check()
        for i in range(x.shape[0]):
            want = phase_coupling_filter(x[i], lam)
            assert np.abs(got[i] - want).max() <= 1e-6 * np.abs(want).max(), (lam, i)
    assert np.array_equal(got[3], x[3])
    # SimplePredictor with the GPU front stage: predict_batch filters on the device (no per-window CPU loop)
    torch.save(checkpoint, tmp_path / "m.pth")
    pre = PhaseCouplingFilterGPU(device=dev, accept_noncommercial_terms=True)
    sp = SimplePredictor(str(tmp_path / "m.pth"), sr=125, preprocessor=pre)
    pb = sp.predict_batch(x)
    p0, label = sp.predict(x[0])
    assert pb.shape == (20, 3) and np.abs(pb[0] - p0).max() < 1e-6 and label in sp.class_names


@pytest.mark.gpu
def test_gpu_filter_nan_and_inf_windows():
    """A window with a NaN or Inf sample comes out non-finite where the reference's does (np.linalg.inv does not raise
    on NaN); it is not a singular system, so neither check() nor transform() raises, and the clean window next to it
    is bit-identical to its run alone."""
    from oracle.phase_filter import phase_coupling_filter
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    rng = np.random.default_rng(4)
    x = (rng.standard_normal((3, 625, 8)) * 2.0).astype(np.float32)
    x[1, 100, 3] = np.nan
    x[2, 400, 6] = np.inf
    dev = torch.device("cuda:0")
    pre = PhaseCouplingFilterGPU(device=dev, accept_noncommercial_terms=True)
    got = pre.transform_batch(torch.from_numpy(x).to(dev)).cpu().numpy()
    pre.check()
    with np.errstate(invalid="ignore"):
        for i in (1, 2):
            assert np.array_equal(np.isfinite(got[i]), np.isfinite(phase_coupling_filter(x[i]))), i
            assert np.array_equal(np.isfinite(pre.transform(x[i])), np.isfinite(got[i])), i
    assert np.isfinite(got[0]).all()
    assert np.array_equal(pre.transform(x[0]), got[0])


@pytest.mark.gpu
def test_gpu_filter_batch_layouts():
    """B = 1 and B = 148 * 8 + 3 (more CTAs than 8 per SM, a ragged last wave): every window bit-identical to its run
    alone."""
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    rng = np.random.default_rng(5)
    B = 148 * 8 + 3
    t = np.arange(625)[:, None] / 125.0
    x = (rng.standard_normal((B, 625, 8)) + 3.0 * np.sin(2 * np.pi * (8 + np.arange(8))[None, :] * t)[None]).astype(np.float32)
    dev = torch.device("cuda:0")
    pre = PhaseCouplingFilterGPU(device=dev, accept_noncommercial_terms=True)
    xd = torch.from_numpy(x).to(dev)
    full = pre.transform_batch(xd).cpu().numpy()
    pre.check()
    for i in range(B):
        assert np.array_equal(pre.transform_batch(xd[i:i + 1]).cpu().numpy()[0], full[i]), i


@pytest.mark.gpu
def test_gpu_filter_misaligned_view():
    """A contiguous view at a 4-byte offset is filtered like the aligned tensor (the kernel loads 16 bytes at a time)."""
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    x = torch.from_numpy((np.random.default_rng(6).standard_normal((3, 625, 8)) * 2.0).astype(np.float32)).cuda()
    buf = torch.empty(x.numel() + 1, device="cuda")
    view = buf[1:1 + x.numel()].view(x.shape)
    view.copy_(x)
    assert view.data_ptr() % 16 != 0
    pre = PhaseCouplingFilterGPU(device=torch.device("cuda:0"), accept_noncommercial_terms=True)
    assert torch.equal(pre.transform_batch(view), pre.transform_batch(x))
    pre.check()
