"""SURVEY 8(f) rank 4: collector-side filter chain.  PARITY UNPINNED (BrainFlow absent): the oracle is
oracle/filter_chain.py, a scipy restatement of BrainFlow's published algorithm."""
import numpy as np
import pytest
import torch
from scipy import signal

from oracle import filter_chain as fc


def test_butterworth_design_matches_scipy():
    """CPU: the from-first-principles SOS design has the same transfer function as scipy.signal.butter."""
    from neural_speech_decoding_b200 import filters
    w = np.linspace(0.01, np.pi - 0.01, 2000)
    cases = list(filters.COLLECTOR_CHAIN) + [("bandpass", 8.0, 13.0, 3), ("bandstop", 20.0, 30.0, 5), ("bandpass", 1.0, 60.0, 1)]
    for kind, lo, hi, order in cases:
        mine = filters.butter_band_sos(order, lo, hi, kind, 125.0)
        ref = signal.butter(order, [lo, hi], btype=kind, fs=125.0, output="sos")
        assert mine.shape == ref.shape == (order, 6)
        _, h1 = signal.sosfreqz(mine, worN=w)
        _, h2 = signal.sosfreqz(ref, worN=w)
        assert np.abs(h1 - h2).max() < 1e-11, (kind, lo, hi, order)
        assert np.all(np.abs(np.roots(s[3:])) < 1.0 for s in mine)            # stable
    with pytest.raises(ValueError):
        filters.butter_band_sos(2, 30.0, 70.0, "bandpass", 125.0)              # above Nyquist
    with pytest.raises(ValueError):
        filters.butter_band_sos(2, 3.0, 48.0, "lowpass", 125.0)


def test_oracle_cascade_matches_scipy_sosfilt():
    """CPU: the explicit-loop DirectFormII cascade of the oracle == scipy.signal.sosfilt (same recurrence)."""
    rng = np.random.default_rng(0)
    x = rng.standard_normal(300)
    sos = fc.scipy_sos("bandstop", 49.5, 50.5, 4, 125.0)
    got = fc.cascade(x, sos, np.zeros((4, 2)))
    np.testing.assert_allclose(got, signal.sosfilt(sos, x), rtol=0, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("carry", [True, False])
def test_filter_chain_matches_oracle(windows, carry):
    from neural_speech_decoding_b200 import filters
    rng = np.random.default_rng(1)
    raw = np.concatenate([windows["X"][:5] * 7.0 + 3.0,                         # recorded windows, rescaled + offset
                          (rng.standard_normal((3, 625, 8)) * 40 + 100 * np.sin(np.arange(625) * 2 * np.pi * 50 / 125)[None, :, None]
                           ).astype(np.float32)])                               # noise + strong 50 Hz mains
    got = filters.filter_windows(torch.from_numpy(raw).cuda(), carry_state=carry).cpu().numpy()
    sos_list = filters.chain_sos()
    for i in range(raw.shape[0]):
        want = fc.collector_chain(raw[i], sos_list=sos_list, carry_state=carry)           # same coefficients
        np.testing.assert_allclose(got[i], want, rtol=0, atol=2e-6), i
        want_scipy = fc.collector_chain(raw[i], carry_state=carry)                        # scipy's own design
        np.testing.assert_allclose(got[i], want_scipy, rtol=0, atol=5e-6), i
    # the 50 Hz line is gone, the mean is gone
    spec = np.abs(np.fft.rfft(got[-1][:, 0]))
    assert spec[250] < 1e-2 * np.abs(np.fft.rfft(raw[-1][:, 0]))[250]
    assert abs(got[-1].mean()) < 0.5


@pytest.mark.gpu
def test_filter_chain_options_and_errors(windows):
    from neural_speech_decoding_b200 import filters
    x = torch.from_numpy(windows["X"][:2]).cuda()
    y0 = filters.filter_windows(x, chain=(), detrend=True, round_decimals=-1).cpu().numpy()
    np.testing.assert_allclose(y0, windows["X"][:2] - windows["X"][:2].mean(axis=1, keepdims=True), atol=1e-6)
    y1 = filters.filter_windows(x, chain=(("bandpass", 8.0, 13.0, 3),), detrend=False, round_decimals=-1, carry_state=False).cpu().numpy()
    sos = signal.butter(3, [8.0, 13.0], btype="bandpass", fs=125.0, output="sos")
    want = signal.sosfilt(sos, signal.sosfilt(sos, windows["X"][0].astype(np.float64), axis=0)[::-1], axis=0)[::-1]
    np.testing.assert_allclose(y1[0], want, atol=2e-5)
    with pytest.raises(ValueError):
        filters.filter_windows(x[0])
    with pytest.raises(RuntimeError):
        filters.filter_windows(x.cpu())


# ---------------------------------------------------------------------------------------------------------------------
# Every compiled path of na_iir.cu against a float64 reference.  na_iir_chain picks its kernel from T, the largest filter
# order and the iir_occ3 knob: iir_chain_warp_kernel<LT, MAXS, OCC> with LT = 20 / 40 / 80 for T <= 640 / 1280 / 2560
# and MAXS = 4 / 8 for sections <= 4 / up to 8, iir_chain_kernel (tiled scratch) above 2560; C == 8 stages a window per
# CTA through shared memory (coop), any other C reads global memory directly, with a partial last CTA when B*C % 8 != 0.
# ---------------------------------------------------------------------------------------------------------------------
CHAINS = {
    "collector": fc.CHAIN,                                                    # 4 sections at most: MAXS = 4
    "order8": (("bandstop", 49.5, 50.5, 8), ("bandpass", 1.0, 40.0, 6)),     # 8 sections: MAXS = 8
    "none": (),                                                               # detrend and the cast only
}
LT_BOUNDARIES = [1, 2, 31, 33, 625, 640, 641, 1280, 1281, 2560, 2561, 5000]


def _raw(rng, B, T, C):
    """Noise, strong 50 Hz mains and a large DC offset (1e3 .. 1e5, either sign): the inputs the detrend is for."""
    t = np.arange(T)[None, :, None]
    dc = rng.uniform(1e3, 1e5, (B, 1, C)) * rng.choice([-1.0, 1.0], (B, 1, C))
    mains = 100.0 * np.sin(2 * np.pi * 50.0 * t / 125.0 + rng.uniform(0, 2 * np.pi, (B, 1, C)))
    return (rng.standard_normal((B, T, C)) * 40.0 + mains + dc).astype(np.float32)


def _ulps(got, ref):
    """Per series (axis 1 = time): |got - fp32(ref)| in fp32 ulps of the series' max |ref|."""
    ref32 = ref.astype(np.float32)
    ulp = np.spacing(np.abs(ref32).max(axis=1, keepdims=True))
    return np.abs(got.astype(np.float64) - ref32.astype(np.float64)) / ulp.astype(np.float64)


def _filter(x, **kw):
    from neural_speech_decoding_b200 import filters
    return filters.filter_windows(torch.from_numpy(x).cuda(), **kw).cpu().numpy()


@pytest.mark.parametrize("carry", [True, False])
@pytest.mark.parametrize("chain", ["collector", "order8"])
def test_sosfilt_reference_matches_cascade(chain, carry):
    """CPU: the vectorised sosfilt reference used at the large shapes == the explicit DirectFormII loops (sosfilt runs
    the transposed form, so they differ by rounding; the narrow order-8 notch amplifies it to ~1e-11)."""
    from neural_speech_decoding_b200 import filters
    rtol = {"collector": 1e-13, "order8": 1e-10}[chain]
    x = _raw(np.random.default_rng(5), 1, 625, 8)[0]
    sos = filters.chain_sos(CHAINS[chain])
    for detrend in (True, False):
        want = fc.zero_phase_chain(x, sos, carry_state=carry, detrend=detrend)
        got = fc.zero_phase_chain_sosfilt(x, sos, carry_state=carry, detrend=detrend)
        assert np.abs(got - want).max() <= rtol * np.abs(want).max(), (detrend, np.abs(got - want).max())


@pytest.mark.gpu
@pytest.mark.parametrize("chain", list(CHAINS))
@pytest.mark.parametrize("T", LT_BOUNDARIES)
def test_filter_chain_within_one_ulp(T, chain):
    """round_decimals=-1: every series within 1 fp32 ulp (of its max |ref|) of the float64 reference, at every LT
    boundary, coop (C = 8) and direct (C = 1, 5, 16; partial last CTAs), detrend and carry on and off."""
    from neural_speech_decoding_b200 import filters
    sos = filters.chain_sos(CHAINS[chain])
    for C in (8, 1, 5, 16):
        x = _raw(np.random.default_rng(T * 100 + C), 3, T, C)
        for detrend in (True, False):
            for carry in (True, False):
                got = _filter(x, chain=CHAINS[chain], detrend=detrend, carry_state=carry, round_decimals=-1)
                ref = fc.zero_phase_chain_sosfilt(x, sos, carry_state=carry, detrend=detrend)
                err = _ulps(got, ref).max()
                assert err <= 1.0, (C, detrend, carry, err)


@pytest.mark.gpu
@pytest.mark.parametrize("decimals", [7, 0])
def test_filter_chain_rounding(decimals):
    """np.round(., d) then the cast, negative zero cleared.  Rounding and the cast are monotone, so the output must lie
    between the rounded values of ref -/+ e (e: a float64 error bound); a value near a rounding tie may go either way."""
    from neural_speech_decoding_b200 import filters
    rng = np.random.default_rng(11)
    for T in (625, 1280, 2560, 5000):
        for C in (8, 5):
            amp = 10.0 ** rng.uniform(-4, 1.5, (3, 1, C))                   # 1e-4 .. 30: the 7th decimal is visible in fp32
            x = (_raw(rng, 3, T, C) * amp).astype(np.float32)
            for chain in ("collector", "order8"):
                got = _filter(x, chain=CHAINS[chain], round_decimals=decimals)
                ref = fc.zero_phase_chain_sosfilt(x, filters.chain_sos(CHAINS[chain]))
                e = 1e-9 * np.abs(ref).max(axis=1, keepdims=True)
                lo, hi = fc.collector_round(ref - e, decimals), fc.collector_round(ref + e, decimals)
                assert np.all((lo <= got) & (got <= hi)), (T, C, chain, np.abs(got - fc.collector_round(ref, decimals)).max())
                assert not np.any(np.signbit(got) & (got == 0)), (T, C, chain)
                if decimals == 0:
                    assert (got == 0).any() and (got < 0).any()             # small negative values were rounded to zero


@pytest.fixture
def set_iir_occ3():
    from neural_speech_decoding_b200 import _lib
    try:
        yield lambda v: _lib.call("na_set_tuning", b"iir_occ3", v)
    finally:
        _lib.call("na_set_tuning", b"iir_occ3", 2)


@pytest.mark.gpu
def test_filter_chain_iir_occ3_is_bit_identical(set_iir_occ3):
    """<20,4,1>, <20,4,2> and <20,4,3> differ only in their register budget."""
    rng = np.random.default_rng(12)
    for C in (8, 5):
        x = _raw(rng, 9, 625, C)
        out = {}
        for v in (1, 2, 3):
            set_iir_occ3(v)
            out[v] = _filter(x, round_decimals=-1)
        assert np.array_equal(out[1], out[2]) and np.array_equal(out[3], out[2]), C


@pytest.mark.gpu
@pytest.mark.parametrize("T", [625, 1280, 2560])
def test_filter_chain_coop_equals_direct(T):
    """[B,T,8] through shared memory == the same series as [B*8,T,1] read directly, bit for bit."""
    x = _raw(np.random.default_rng(T), 5, T, 8)
    xd = np.ascontiguousarray(x.transpose(0, 2, 1).reshape(40, T, 1))
    for chain in ("collector", "order8"):
        coop = _filter(x, chain=CHAINS[chain], round_decimals=-1)
        direct = _filter(xd, chain=CHAINS[chain], round_decimals=-1).reshape(5, 8, T).transpose(0, 2, 1)
        assert np.array_equal(coop, direct), chain


@pytest.mark.gpu
@pytest.mark.parametrize("T", [625, 1281, 2561])
def test_filter_chain_batch_invariance(T):
    """A window filtered alone == the same window inside a batch of 37."""
    for C in (8, 5):
        x = _raw(np.random.default_rng(T + C), 37, T, C)
        for chain in ("collector", "order8"):
            full = _filter(x, chain=CHAINS[chain], round_decimals=-1)
            for i in (0, 18, 36):
                assert np.array_equal(_filter(x[i:i + 1], chain=CHAINS[chain], round_decimals=-1)[0], full[i]), (C, chain, i)


@pytest.mark.gpu
@pytest.mark.parametrize("T,C", [(625, 8), (625, 5), (2561, 8)])
def test_filter_chain_nonfinite_series_are_isolated(T, C):
    """A NaN or Inf sample spoils its own series, as in the reference, and leaves every other series bit-identical."""
    from neural_speech_decoding_b200 import filters
    x = _raw(np.random.default_rng(T * C), 4, T, C)
    bad = x.copy()
    bad[1, T // 3, 2] = np.nan
    bad[2, T // 2, C - 1] = np.inf
    hit = np.zeros(x.shape, bool)
    hit[1, :, 2] = hit[2, :, C - 1] = True
    for chain in ("collector", "order8"):
        for detrend in (True, False):
            clean = _filter(x, chain=CHAINS[chain], detrend=detrend, round_decimals=-1)
            got = _filter(bad, chain=CHAINS[chain], detrend=detrend, round_decimals=-1)
            assert np.array_equal(got[~hit], clean[~hit]), (chain, detrend)
            with np.errstate(invalid="ignore"):
                ref = fc.zero_phase_chain_sosfilt(bad, filters.chain_sos(CHAINS[chain]), detrend=detrend)
            assert np.array_equal(np.isfinite(got), np.isfinite(ref)), (chain, detrend)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [625, 2561])
def test_filter_chain_misaligned_view(T):
    """A contiguous view at a 4-byte offset is filtered like the aligned tensor (the kernels load 16 bytes at a time)."""
    from neural_speech_decoding_b200 import filters
    x = torch.from_numpy(_raw(np.random.default_rng(T), 3, T, 8)).cuda()
    buf = torch.empty(x.numel() + 1, device="cuda")
    view = buf[1:1 + x.numel()].view(x.shape)
    view.copy_(x)
    assert view.data_ptr() % 16 != 0
    assert torch.equal(filters.filter_windows(view), filters.filter_windows(x))
