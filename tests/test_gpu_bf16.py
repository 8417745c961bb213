"""Tensor-core tier (tcgen05, bf16 operands / fp32 accumulate) against the fp32 reference.

Contract (BASELINE.json north_star): logits within 2e-2 of the reference (max|d| / max|ref|),
argmax class labels identical on the repo's EEG_data_collection windows.
"""
import numpy as np
import pytest
import torch

from oracle import numpy_oracle as no
from oracle.torch_ref import RefEEGLSTM

pytestmark = pytest.mark.gpu

BF16_TOL = 2e-2


def rel(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from neural_speech_decoding_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def bf16_model(dev, sd, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    m = EEG_LSTM(**kw)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval()
    m.compute_dtype = torch.bfloat16
    return m


def test_bf16_logits_and_argmax_on_all_windows(dev, checkpoint, windows, golden_dir):
    ref = np.load(golden_dir / "ref_outputs_3class.npz")["logits_raw_b1"]
    m = bf16_model(dev, checkpoint)
    with torch.inference_mode():
        got = m(torch.from_numpy(windows["X"]).to(dev)).cpu().numpy()
    assert got.shape == (324, 3) and np.isfinite(got).all()
    assert rel(got, ref) < BF16_TOL, rel(got, ref)
    assert np.array_equal(got.argmax(1), ref.argmax(1))
    # probabilities + ragged sizes (1 window; 130 windows = 2 tiles, second one almost empty)
    with torch.inference_mode():
        lg1, p1 = m.decode(torch.from_numpy(windows["X"][5:6]).to(dev))
        lg130, p130 = m.decode(torch.from_numpy(windows["X"][:130]).to(dev))
    assert rel(lg1.cpu().numpy(), ref[5:6]) < BF16_TOL
    assert np.array_equal(lg130.cpu().numpy(), got[:130])          # independent of batch / tile position
    np.testing.assert_allclose(p130.cpu().numpy(), no.softmax(lg130.cpu().numpy()), atol=2e-6)
    assert np.array_equal(lg1.cpu().numpy(), got[5:6])


def test_bf16_synthetic_512_and_many_tiles(dev, checkpoint):
    gen = torch.Generator(device="cpu").manual_seed(0)
    x = torch.randn(512, 625, 8, generator=gen) * 2.73
    refm = RefEEGLSTM().eval()
    refm.load_state_dict(checkpoint, strict=True)
    with torch.inference_mode():
        want = refm(x).numpy()
    m = bf16_model(dev, checkpoint)
    with torch.inference_mode():
        got = m(x.to(dev)).cpu().numpy()
    assert rel(got, want) < BF16_TOL, rel(got, want)
    margin = np.sort(want, axis=1)
    safe = (margin[:, -1] - margin[:, -2]) > 0.1                   # argmax is only defined up to the tolerance
    assert np.array_equal(got.argmax(1)[safe], want.argmax(1)[safe])
    # more tiles than SMs (persistent loop, tile-boundary state reset): 160 tiles x 128 short windows
    xs = torch.randn(160 * 128, 12, 8, generator=gen) * 2.73
    with torch.inference_mode():
        a = m(xs.to(dev)).cpu().numpy()
        m.compute_dtype = torch.float32
        b = m(xs.to(dev)).cpu().numpy()                             # exact tier
    # 20,480 random 12-step windows: bf16 operand rounding has a tail (a handful of windows whose
    # LayerNorm input is nearly constant amplify it), so this stress case is judged statistically
    err = np.abs(a - b).max(axis=1) / np.abs(b).max()
    assert np.isfinite(a).all()
    assert err.mean() < 2e-3 and err.max() < BF16_TOL, (err.mean(), err.max())      # the contract, on the worst window
    assert (a.argmax(1) != b.argmax(1)).mean() < 2e-3


def test_bf16_tile_modes_agree(dev, checkpoint):
    """Every tile layout of the v2 kernel (full 128-window tiles, a 3-quarter remainder, R = 2 and R = 4 row-replicated
    remainders, several tiles per CTA) gives bit-identical logits to the unreplicated layout, the v1 kernel agrees
    within the tier's rounding, and all of them match the exact fp32 tier."""
    from neural_speech_decoding_b200 import _lib, ops
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    gen = torch.Generator(device="cpu").manual_seed(3)
    m = bf16_model(dev, checkpoint)
    T = 40
    try:
        for quarters_per_cta in (1, 2, 3, 5, 6, 7):            # R=4 | R=2 | 3-quarter tile | 4+R4 | 4+R2 | 4+3
            B = sms * 32 * quarters_per_cta - 7                    # ragged last quarter
            x = (torch.randn(B, T, 8, generator=gen) * 2.73).to(dev)
            with torch.inference_mode():
                xt = ops.window_zscore(x, T, T, False, True, 2, 128)
                packed, head = m._packed_tc(), m._head_params()
                outs = {}
                for name, hs, rep in (("v2", 3, 1), ("v2_norep", 3, 0), ("v1", 2, 0)):
                    _lib.call("na_set_tuning", b"tc_infer_hs", hs)
                    _lib.call("na_set_tuning", b"tc_infer_rep", rep)
                    lg, pr = ops.decoder_infer_bf16(xt, packed, head, B, True)
                    outs[name] = lg.cpu().numpy()
                    np.testing.assert_allclose(pr.cpu().numpy(), no.softmax(outs[name]), atol=2e-6)
                m.compute_dtype = torch.float32
                exact = m(x).cpu().numpy()
                m.compute_dtype = torch.bfloat16
            assert np.array_equal(outs["v2"], outs["v2_norep"]), quarters_per_cta
            err = np.abs(outs["v2"] - exact).max(axis=1) / np.abs(exact).max()
            assert err.mean() < 2e-3 and np.quantile(err, 0.999) < BF16_TOL, (quarters_per_cta, err.mean(), err.max())
            err1 = np.abs(outs["v2"] - outs["v1"]).max(axis=1) / np.abs(exact).max()
            assert err1.mean() < 2e-3 and np.quantile(err1, 0.999) < BF16_TOL, (quarters_per_cta, err1.mean(), err1.max())
    finally:
        _lib.call("na_set_tuning", b"tc_infer_hs", 3)
        _lib.call("na_set_tuning", b"tc_infer_rep", 1)


def test_bf16_input_tensor_selects_tier_and_keeps_dtype(dev, checkpoint, windows):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    m = EEG_LSTM()
    m.load_state_dict(checkpoint, strict=True)
    m = m.to(dev).eval()
    x = torch.from_numpy(windows["X"][:8]).to(dev)
    with torch.inference_mode():
        y32 = m(x)
        y16 = m(x.bfloat16())
    assert y32.dtype == torch.float32 and y16.dtype == torch.bfloat16
    assert rel(y16.float().cpu().numpy(), y32.cpu().numpy()) < 3e-2


def test_bf16_five_class_and_trial_mean(dev, windows, golden_dir):
    from neural_speech_decoding_b200.tester import run_trials_batched
    f = np.load(golden_dir / "ref_5class.npz")
    sd = {k[3:]: torch.from_numpy(f[k]) for k in f.files if k.startswith("sd.")}
    m = bf16_model(dev, sd, num_classes=5)
    x = torch.from_numpy(windows["X"][f["sel"]]).to(dev)
    with torch.inference_mode():
        got = m(x).cpu().numpy()
    assert got.shape == (32, 5) and rel(got, f["logits"]) < BF16_TOL
    R, B = 10, 3
    w = windows["X"][:R * B].reshape(R, B, 625, 8)
    want = no.trial_mean(no.softmax(no.decoder_forward(w.reshape(R * B, 625, 8), {k: v.numpy() for k, v in sd.items()})).reshape(R, B, 5))
    avg = run_trials_batched(w, m)
    assert np.abs(avg - want).max() < 2e-2


# ---------------------------------------------------------------------------------------------
# training on the tensor-core tier (tcgen05 forward-with-save + fused BPTT/weight gradients)
# ---------------------------------------------------------------------------------------------
def grad_rel(model, ref_grads):
    out = {}
    aw = np.abs(ref_grads["attn.weight"]).max()
    gmax = max(float(np.abs(ref_grads[k]).max()) for k, _ in model.named_parameters())
    for k, p in model.named_parameters():
        r = ref_grads[k]
        scale = float(aw if k == "attn.bias" else np.abs(r).max())        # every tensor on its own scale, no floor
        out[k] = float(np.abs(p.grad.float().cpu().numpy() - r).max() / scale)
    return out


def test_bf16_training_gradients_eval_mode(dev, checkpoint, windows, golden_dir):
    g = np.load(golden_dir / "fp64_grads_3class_eval_b16.npz")
    sel = np.load(golden_dir / "ref_grads_3class_eval_b16.npz")
    m = bf16_model(dev, checkpoint)                       # eval mode: deterministic, autograd still works
    x = torch.from_numpy(windows["X"][sel["sel"]]).to(dev)
    y = torch.from_numpy(sel["y"]).to(dev)
    logits = m(x)
    assert rel(logits.detach().cpu().numpy(), sel["logits"]) < BF16_TOL
    loss = torch.nn.functional.cross_entropy(logits, y)
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < 2e-2
    worst = grad_rel(m, g)
    assert max(worst.values()) < BF16_TOL, worst
    # bit-reproducible (fixed-order reduction of the per-CTA TMEM partials)
    g1 = [p.grad.clone() for p in m.parameters()]
    m.zero_grad()
    torch.nn.functional.cross_entropy(m(x), y).backward()
    for a, p in zip(g1, m.parameters()):
        assert torch.equal(a, p.grad)


def test_bf16_training_with_injected_noise_and_many_tiles(dev, checkpoint):
    from oracle.torch_ref import explicit_forward
    torch.manual_seed(21)
    B, T, H = 300, 30, 48                                  # 3 tiles (384 padded), ragged
    x = torch.randn(B, T, 8) * 2.73
    y = torch.randint(0, 3, (B,))
    d1 = (torch.rand(1, B, T, H) >= 0.6).float()
    rr = torch.empty(B, 32).uniform_(1 / 8, 1 / 3)
    d2 = (torch.rand(B, 32) >= 0.6).float()
    sd = {k: v.double().requires_grad_(True) for k, v in checkpoint.items()}
    lr = torch.nn.functional.cross_entropy(explicit_forward(x.double(), sd, 2, 0.6, d1[0].double(), rr.double(), d2.double()), y)
    lr.backward()
    m = bf16_model(dev, checkpoint).train()
    m.inject_noise(drop1=d1, rrelu_slope=rr, drop2=d2)
    loss = torch.nn.functional.cross_entropy(m(x.to(dev)), y.to(dev))
    loss.backward()
    assert abs(loss.item() - lr.item()) < 2e-2
    worst = grad_rel(m, {k: v.grad.numpy() for k, v in sd.items()})
    assert max(worst.values()) < BF16_TOL, worst


def test_in_kernel_dropout_equals_mask_tensor_mode(dev, checkpoint):
    """The counter-based in-kernel dropout (no mask tensor) == the mask-tensor mode fed with the
    materialised mask, bit for bit (forward and all gradients); keep-rate and seeding behave.  Both runs pass
    p' = 1 - thresh16 / 65536, which makes the mask mode's scale 1 / (1 - p') exactly the generator's 65536 / thresh16."""
    from neural_speech_decoding_b200 import ops
    torch.manual_seed(3)
    B, T = 200, 40
    x = (torch.randn(B, T, 8) * 2.73).to(dev)
    y = torch.randint(0, 3, (B,)).to(dev)
    rr = torch.empty(B, 32).uniform_(1 / 8, 1 / 3).to(dev)
    d2 = (torch.rand(B, 32) >= 0.6).float().to(dev)
    seed, thresh = 123456789012345, int(round(0.4 * 65536))
    p = 1.0 - thresh / 65536
    m = bf16_model(dev, checkpoint).train()
    lstm = [m.lstm.layer(0), m.lstm.layer(1)]
    head = m._head_params()
    la = ops.decoder_train_forward_tc(x, lstm, head, p, False, (seed, thresh), rr, d2)
    torch.nn.functional.cross_entropy(la, y).backward()
    ga = [q.grad.clone() for q in m.parameters()]
    m.zero_grad()
    mask = ops.dropout_mask_u8(x, seed, thresh, T, 256)
    assert abs(mask.float().mean().item() - 0.4) < 0.01
    lb = ops.decoder_train_forward_tc(x, lstm, head, p, False, mask, rr, d2)
    torch.nn.functional.cross_entropy(lb, y).backward()
    assert torch.equal(la, lb), (la - lb).abs().max().item()
    for (k, _), g, q in zip(m.named_parameters(), ga, m.parameters()):
        assert torch.isfinite(g).all() and torch.equal(g, q.grad), k
    other = ops.dropout_mask_u8(x, seed + 1, thresh, T, 256)
    assert (other != mask).float().mean().item() > 0.3                            # a different seed decorrelates
    # module path: train-mode forward is stochastic, reproducible under torch.manual_seed
    torch.manual_seed(11); a = m(x)
    torch.manual_seed(11); b = m(x)
    torch.manual_seed(12); c = m(x)
    assert torch.equal(a, b) and not torch.equal(a, c)


def test_edge_shapes_and_bfloat16_module(dev, checkpoint, windows):
    """T = 1 and T = 2 windows (wavefront start-up), the z-score front stage on the tensor-core tier, and a
    module converted with .bfloat16() (bf16 parameters and inputs in, bf16 logits / gradients out)."""
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    gen = torch.Generator().manual_seed(9)
    refm = RefEEGLSTM().eval()
    refm.load_state_dict(checkpoint, strict=True)
    m = bf16_model(dev, checkpoint)
    for T in (1, 2, 3):
        x = torch.randn(200, T, 8, generator=gen) * 2.73
        with torch.inference_mode():
            got = m(x.to(dev)).cpu().numpy()
            want = refm(x).numpy()
        assert rel(got, want) < BF16_TOL, T
        y = torch.randint(0, 3, (200,), generator=gen)
        m.zero_grad()
        torch.nn.functional.cross_entropy(m(x.to(dev)), y.to(dev)).backward()      # T = 1: no recurrence at all
        assert all(torch.isfinite(p.grad).all() for p in m.parameters())
    # z-score front stage (K1 normalises, then the same decoder)
    m.zscore_input = True
    X = torch.from_numpy(windows["X"][:40])
    with torch.inference_mode():
        got = m(X.to(dev)).cpu().numpy()
        want = refm(torch.from_numpy(no.zscore_window(X.numpy()))).numpy()
    assert rel(got, want) < BF16_TOL
    m.zscore_input = False
    # .bfloat16() module
    mb = EEG_LSTM()
    mb.load_state_dict(checkpoint, strict=True)
    mb = mb.to(dev).bfloat16()
    xb = X[:16].to(dev).bfloat16()
    with torch.inference_mode():
        out = mb.eval()(xb)
    assert out.dtype == torch.bfloat16 and rel(out.float().cpu().numpy(), refm(X[:16]).detach().numpy()) < 5e-2
    mb.train()
    torch.nn.functional.cross_entropy(mb(xb).float(), torch.randint(0, 3, (16,)).to(dev)).backward()
    assert all(p.grad is not None and p.grad.dtype == torch.bfloat16 for p in mb.parameters())


# ---- wide hidden sizes (streamed-weight kernel, na_decoder_wide.cu) ------------------------------------------

def test_wide_h192_matches_reference_golden(dev, golden_dir):
    """BASELINE configs[4] architecture: the reference's own logits for EEG_LSTM(hidden_size=192) (seeded init,
    tests/golden/ref_stress_h192.npz, generated by importing the real reference)."""
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    f = np.load(golden_dir / "ref_stress_h192.npz")
    sd = {k[3:]: torch.from_numpy(f[k].copy()) for k in f.files if k.startswith("sd.")}
    m = EEG_LSTM(hidden_size=192)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval()
    m.compute_dtype = torch.bfloat16
    assert m.tc_wide_supported() and not m.tc_supported()
    with torch.inference_mode():
        lg, pr = m.decode(torch.from_numpy(f["x"]).to(dev))
    got = lg.cpu().numpy()
    assert rel(got, f["logits"]) < BF16_TOL, rel(got, f["logits"])
    assert np.array_equal(got.argmax(1), f["logits"].argmax(1))
    np.testing.assert_allclose(pr.cpu().numpy(), no.softmax(got), atol=2e-6)


@pytest.mark.parametrize("H,T,B", [(192, 37, 300), (144, 20, 130), (96, 50, 5), (192, 3, 148 * 128 + 77), (192, 1, 64)])
def test_wide_matches_exact_tier(dev, H, T, B):
    """Seeded random decoders of every wide size against the exact fp32 tier (itself pinned to the oracle):
    ragged batches, several tiles per CTA, T = 1 (flush-only pooling)."""
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(100 + H + T)
    m = EEG_LSTM(hidden_size=H, num_classes=5).to(dev).eval()
    with torch.no_grad():                                  # make the attention scores and the head non-trivial
        m.attn.weight.mul_(4.0); m.attn.bias.fill_(0.3)
        m.ln.weight.uniform_(0.5, 1.5); m.ln.bias.uniform_(-0.2, 0.2)
    gen = torch.Generator(device="cpu").manual_seed(H * 7 + B)
    x = (torch.randn(B, T, 8, generator=gen) * 2.73).to(dev)
    with torch.inference_mode():
        exact = m(x).cpu().numpy()
        m.compute_dtype = torch.bfloat16
        got = m(x).cpu().numpy()
        again = m(x).cpu().numpy()
    assert np.isfinite(got).all()
    assert np.array_equal(got, again)                      # deterministic, workspace re-use is clean
    err = np.abs(got - exact).max(axis=1) / np.abs(exact).max()
    assert err.mean() < 2e-3 and err.max() < BF16_TOL, (err.mean(), err.max())


def test_fused_input_entries_are_bit_identical(dev, checkpoint):
    """na_decoder_infer_bf16_x32 (fp32 [B,T,8] read directly, pack fused into the kernel) against the time-major fp16 entry
    point: same bits, incl. ragged batches and row-replicated short tiles."""
    from neural_speech_decoding_b200 import ops
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    gen = torch.Generator(device="cpu").manual_seed(11)
    m = bf16_model(dev, checkpoint)
    for B, T in ((1, 625), (77, 50), (148 * 32 * 5 - 3, 21)):
        x = (torch.randn(B, T, 8, generator=gen) * 2.73).to(dev)
        with torch.inference_mode():
            xt = ops.window_zscore(x, T, T, False, True, ops.NA_F16, ops.TC_TILE)
            a = ops.decoder_infer_bf16(xt, m._packed_tc(), m._head_params(), B, True)
            b = ops.decoder_infer_bf16_x32(x, m._packed_tc(), m._head_params(), True)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), (B, T)


def test_fp16_tier_input_range_and_nan(dev, checkpoint):
    """The 16-bit tier stores the input as fp16(x / 16) (the packed layer-0 W_ih carries the 16): raw ADC samples with a DC
    offset beyond fp16's 65,504 stay finite instead of turning the logits into NaN; inside the normal range nothing changes
    (same 2e-2 contract); a NaN sample poisons its own window only."""
    gen = torch.Generator(device="cpu").manual_seed(9)
    m = bf16_model(dev, checkpoint)
    x = torch.randn(40, 625, 8, generator=gen) * 2.73
    with torch.inference_mode():
        big = m((x + 1.0e5).to(dev)).cpu().numpy()                # 1e5 / 16 = 6,250: representable
        assert np.isfinite(big).all()
        m.compute_dtype = torch.float32
        want = m((x * 300.0).to(dev)).cpu().numpy()               # amplitudes of ~800 (max ~4,000): still the normal range
        m.compute_dtype = torch.bfloat16
        got = m((x * 300.0).to(dev)).cpu().numpy()
        assert rel(got, want) < BF16_TOL, rel(got, want)
        xn = x.clone()
        xn[3, 100, 2] = float("nan")
        out = m(xn.to(dev)).cpu().numpy()
    assert np.isnan(out[3]).all() and np.isfinite(np.delete(out, 3, axis=0)).all()
    # training forward / backward on the same tier: finite gradients for the offset input
    m.train()
    m.zero_grad()
    torch.nn.functional.cross_entropy(m((x[:8] + 1.0e5).to(dev)), torch.zeros(8, dtype=torch.long, device=dev)).backward()
    assert all(torch.isfinite(p.grad).all() for p in m.parameters())


@pytest.mark.parametrize("B,T", [(300, 30), (64, 7), (1, 3), (65, 12)])
def test_bf16_training_half_tiles_match_full_tiles(dev, checkpoint, B, T):
    """Half tiles (64 windows per tile, the two row copies split the hidden units -- used when a batch would leave more than
    half of the SMs idle) against full tiles: bit-identical logits, gradients equal up to the order of the fp32 weight-gradient
    accumulation, in eval mode and in train mode with the counter-based in-kernel dropout (same mask in both layouts)."""
    from neural_speech_decoding_b200 import ops
    gen = torch.Generator(device="cpu").manual_seed(B + T)
    x = (torch.randn(B, T, 8, generator=gen) * 2.73).to(dev)
    y = torch.randint(0, 3, (B,), generator=gen).to(dev)
    m = bf16_model(dev, checkpoint)
    def run(half, train):
        ops.TC_HALF_TILES = half
        m.train(train)
        m.zero_grad()
        torch.manual_seed(77)                      # same dropout seed / RReLU slopes / head dropout in both runs
        out = m(x)
        torch.nn.functional.cross_entropy(out, y).backward()
        return out.detach().clone(), [p.grad.clone() for p in m.parameters()]
    try:
        for train in (False, True):
            a, ga = run(True, train)
            b, gb = run(False, train)
            assert torch.isfinite(a).all() and torch.equal(a, b), (train, (a - b).abs().max().item())
            gmax = max(float(q.abs().max()) for q in gb)
            for (k, _), p, q in zip(m.named_parameters(), ga, gb):
                assert (p - q).abs().max().item() <= 2e-5 * gmax, (train, k, (p - q).abs().max().item(), gmax)
    finally:
        ops.TC_HALF_TILES = True


@pytest.mark.parametrize("half", [True, False])
@pytest.mark.parametrize("B,T", [(700, 34), (390, 41)])
def test_bf16_training_several_tiles_per_cta(dev, checkpoint, B, T, half):
    """The persistent training kernels with SEVERAL tiles per CTA (grid capped to 2 CTAs by the `train_max_ctas` test knob: the
    running mbarrier phases, the 2- / 3-stage TMA ring and the dW accumulators carry over from tile to tile) against one tile
    per CTA: bit-identical logits, gradients equal up to the order of the fp32 weight-gradient accumulation; eval and train
    mode (in-kernel dropout), full and half tiles, T not a multiple of the stage count."""
    from neural_speech_decoding_b200 import _lib, ops
    gen = torch.Generator(device="cpu").manual_seed(B + T)
    x = (torch.randn(B, T, 8, generator=gen) * 2.73).to(dev)
    y = torch.randint(0, 3, (B,), generator=gen).to(dev)
    m = bf16_model(dev, checkpoint)
    def run(cap, train):
        _lib.call("na_set_tuning", b"train_max_ctas", cap)
        m.train(train)
        m.zero_grad()
        torch.manual_seed(77)
        out = m(x)
        torch.nn.functional.cross_entropy(out, y).backward()
        return out.detach().clone(), [p.grad.clone() for p in m.parameters()]
    saved = ops.TC_HALF_TILES
    try:
        ops.TC_HALF_TILES = half
        for train in (False, True):
            a, ga = run(2, train)
            b, gb = run(0, train)
            assert torch.isfinite(a).all() and torch.equal(a, b), (train, (a - b).abs().max().item())
            gmax = max(float(q.abs().max()) for q in gb)
            for (k, _), p, q in zip(m.named_parameters(), ga, gb):
                assert (p - q).abs().max().item() <= 2e-5 * gmax, (train, k, (p - q).abs().max().item(), gmax)
    finally:
        _lib.call("na_set_tuning", b"train_max_ctas", 0)
        ops.TC_HALF_TILES = saved


# ---------------------------------------------------------------------------------------------
# wide decoders: training on the tensor cores (streamed-weight recurrence kernels + cuBLAS, csrc/na_wide_train.cu)
# ---------------------------------------------------------------------------------------------
def test_wide_training_stress_shape_vs_reference(dev, golden_dir):
    """BASELINE configs[4] (hidden_size = 192): logits, loss and every gradient of the 16-bit tensor-core training tier against
    float64 autograd of the reference module on the reference's own H = 192 fixture (2e-2 contract)."""
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    f = np.load(golden_dir / "ref_stress_h192.npz")
    sd = {k[3:]: torch.from_numpy(f[k]) for k in f.files if k.startswith("sd.")}
    m = EEG_LSTM(hidden_size=192)
    m.load_state_dict(sd, strict=True)
    m = m.to(dev).eval()
    m.compute_dtype = torch.bfloat16
    x, y = torch.from_numpy(f["x"]), torch.from_numpy(f["y"])
    logits = m(x.to(dev))
    assert rel(logits.detach().cpu().numpy(), f["logits"]) < BF16_TOL
    loss = torch.nn.functional.cross_entropy(logits, y.to(dev))
    loss.backward()
    assert abs(loss.item() - float(f["loss"])) < 2e-2
    ref = RefEEGLSTM(hidden_size=192).double().eval()
    ref.load_state_dict({k: v.double() for k, v in sd.items()}, strict=True)
    torch.nn.functional.cross_entropy(ref(x.double()), y).backward()
    truth = {k: p.grad.numpy() for k, p in ref.named_parameters()}
    worst = grad_rel(m, truth)
    worst.pop("attn.bias")                                  # analytically zero (softmax shift invariance): rounding noise on both sides
    assert max(worst.values()) < BF16_TOL, worst
    assert all(torch.isfinite(p.grad).all() for p in m.parameters())


@pytest.mark.parametrize("H,B,T", [(96, 150, 23), (144, 300, 9), (192, 5, 1)])
def test_wide_training_matches_exact_tier_with_noise(dev, H, B, T):
    """Seeded wide decoders in TRAIN mode with injected noise (inter-layer dropout mask, RReLU slopes, head dropout): the
    tensor-core tier against the exact fp32 tier (pinned to the oracle in test_gpu_parity.py), several tiles, ragged batch, T = 1."""
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(7 * H + B)
    m = EEG_LSTM(hidden_size=H, num_classes=5).to(dev).train()
    x = (torch.randn(B, T, 8) * 2.73).to(dev)
    y = torch.randint(0, 5, (B,)).to(dev)
    d1 = (torch.rand(1, B, T, H) >= 0.6).float()
    rr = torch.empty(B, 32).uniform_(1 / 8, 1 / 3)
    d2 = (torch.rand(B, 32) >= 0.6).float()
    m.inject_noise(drop1=d1, rrelu_slope=rr, drop2=d2)
    def run(dtype):
        m.compute_dtype = dtype
        m.zero_grad()
        out = m(x)
        torch.nn.functional.cross_entropy(out, y).backward()
        return out.detach().cpu().numpy(), {k: p.grad.detach().cpu().numpy().copy() for k, p in m.named_parameters()}
    lb, gb = run(torch.float32)
    la, ga = run(torch.bfloat16)
    assert np.isfinite(la).all() and rel(la, lb) < BF16_TOL, rel(la, lb)
    gmax = max(float(np.abs(v).max()) for v in gb.values())
    for k in ga:
        scale = np.abs(gb[k]).max()
        if k == "attn.bias" or (T == 1 and ("weight_hh" in k or k == "attn.weight")):
            scale = gmax
        assert np.abs(ga[k] - gb[k]).max() / scale < BF16_TOL, (k, np.abs(ga[k] - gb[k]).max() / scale)
