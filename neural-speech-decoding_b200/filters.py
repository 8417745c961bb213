"""Collector-side filter chain on the GPU (SURVEY 8(f) rank 4).

The reference records every training window through BrainFlow's ``DataFilter``
(``Neural_decoding_data_collector.py:109-127``): per channel, on the 625 most recent samples,

    detrend(CONSTANT) -> bandstop 39.5-40.5 Hz (order 4) -> bandpass 3-48 Hz (order 2)
                      -> bandstop 49.5-50.5 Hz (order 4) -> bandstop 59-61 Hz (order 4),

every filter ``BUTTERWORTH_ZERO_PHASE`` (forward pass, reverse, forward pass again, reverse), then
``np.round(x, 7)``.  The live path (``streaming_process.py``) does NOT apply it -- the train / serve skew of
SURVEY F8 -- so a host that wants recorded-like windows from a raw stream runs this chain first.

Design: Butterworth band filters as cascades of second-order sections, computed here from first principles
(analog prototype poles, Constantinides band transformation with exactly pre-warped band edges, bilinear map) in
float64; the arithmetic -- 28 serial biquad passes per series -- runs in ``na_iir_chain`` (one WARP per
(window, channel) series, float64, the series stays in registers: block-parallel recurrence + warp scan, no scratch;
``csrc/na_iir.cu``).

PARITY UNPINNED: BrainFlow (``brainflow==5.19.0``, C++ ``DSPFilters``) is not installed here, so the oracle
(``oracle/filter_chain.py``) restates its published algorithm with scipy; two details cannot be confirmed
without it and are parameters: section ordering (no effect beyond rounding) and whether the filter state is
reset between the forward and the backward pass (``carry_state``; BrainFlow re-uses the same filter object, so
the default carries it over).
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops

# (kind, f_lo, f_hi, order) in application order: Neural_decoding_data_collector.py:112-127
COLLECTOR_CHAIN: Tuple[Tuple[str, float, float, int], ...] = (
    ("bandstop", 39.5, 40.5, 4),
    ("bandpass", 3.0, 48.0, 2),
    ("bandstop", 49.5, 50.5, 4),
    ("bandstop", 59.0, 61.0, 4),
)


def butter_band_sos(order: int, f_lo: float, f_hi: float, kind: str, fs: float) -> np.ndarray:
    """Digital Butterworth band-pass / band-stop of prototype order ``order`` (2*order poles) as second-order
    sections ``[order, 6]`` = (b0, b1, b2, 1, a1, a2), unit gain in the pass band.

    Analog low-pass prototype poles p_k = exp(i pi (2k + order + 1) / (2 order)); band edges pre-warped
    w = 2 fs tan(pi f / fs); low-pass -> band-pass s -> (s^2 + w0^2) / (bw s) (band-stop: the reciprocal);
    bilinear z = (2 fs + s) / (2 fs - s).  Conjugate pole pairs are paired into sections."""
    if kind not in ("bandpass", "bandstop"):
        raise ValueError("kind must be 'bandpass' or 'bandstop'")
    if not (0.0 < f_lo < f_hi < fs / 2.0) or order < 1:
        raise ValueError("need 0 < f_lo < f_hi < fs/2 and order >= 1")
    k = np.arange(order)
    proto = np.exp(1j * np.pi * (2 * k + order + 1) / (2 * order))            # left half plane, |p| = 1
    w1, w2 = 2 * fs * np.tan(np.pi * f_lo / fs), 2 * fs * np.tan(np.pi * f_hi / fs)
    bw, w0 = w2 - w1, np.sqrt(w1 * w2)
    half = proto * bw / 2.0 if kind == "bandpass" else bw / (2.0 * proto)
    fs2 = 2.0 * fs
    bil = lambda sp: (fs2 + sp) / (fs2 - sp)                                  # bilinear map s -> z
    if kind == "bandpass":
        zpair = (1.0 + 0j, -1.0 + 0j)                                         # s = 0 -> z = 1, s = inf -> z = -1
    else:
        z0 = bil(1j * w0)
        zpair = (z0, np.conj(z0))                                             # the notch, on the unit circle
    pole_pairs = []
    for hp in half[np.imag(half) >= -1e-12 * np.abs(half)]:                   # one of each conjugate prototype pair (+ a real one)
        disc = np.sqrt(hp * hp - w0 * w0 + 0j)
        pa, pb = bil(hp + disc), bil(hp - disc)
        if abs(np.imag(hp)) <= 1e-12 * abs(hp):                               # real prototype pole: its two band poles share a section
            pole_pairs.append((pa, pb))
        else:                                                                 # complex: each band pole pairs with its conjugate
            pole_pairs.append((pa, np.conj(pa)))
            pole_pairs.append((pb, np.conj(pb)))
    if len(pole_pairs) != order:
        raise ValueError("internal error: section count")
    pole_pairs.sort(key=lambda pq: max(abs(pq[0]), abs(pq[1])))              # nearest-to-unit-circle last
    sos = np.zeros((order, 6))
    for i, (pa, pb) in enumerate(pole_pairs):
        bcoef = np.real(np.poly(zpair))
        acoef = np.real(np.poly([pa, pb]))
        sos[i] = [bcoef[0], bcoef[1], bcoef[2], 1.0, acoef[1], acoef[2]]
    # overall gain: 1 at the centre of the pass band (band-pass) / at DC (band-stop), put on the first section
    wc = bil(1j * w0) if kind == "bandpass" else 1.0 + 0j
    h = 1.0 + 0j
    for s in sos:
        h *= np.polyval(s[:3], wc) / np.polyval(s[3:], wc)
    sos[0, :3] /= np.abs(h)
    return sos


def chain_sos(chain: Sequence[Tuple[str, float, float, int]] = COLLECTOR_CHAIN, fs: float = 125.0) -> List[np.ndarray]:
    return [butter_band_sos(order, lo, hi, kind, fs) for kind, lo, hi, order in chain]


def filter_windows(x: torch.Tensor, fs: float = 125.0, chain: Sequence[Tuple[str, float, float, int]] = COLLECTOR_CHAIN,
                   detrend: bool = True, round_decimals: int = 7, carry_state: bool = True) -> torch.Tensor:
    """x fp32 ``[B,T,C]`` (CUDA) raw windows -> the collector's filtered windows, fp32 ``[B,T,C]``.
    ``round_decimals < 0`` disables the final ``np.round``."""
    ops._require_cuda(x)
    if x.dim() != 3:
        raise ValueError(f"filter_windows expects [B,T,C], got {tuple(x.shape)}")
    x = ops._aligned16(ops._f32c(x))
    B, T, C = x.shape
    sos = chain_sos(chain, fs)
    nsec = np.array([s.shape[0] for s in sos], dtype=np.int32)
    if len(sos) > 8 or (len(sos) and nsec.max() > 8):
        raise RuntimeError("filter_windows: at most 8 filters of at most 8 sections")
    coef = np.concatenate([s[:, [0, 1, 2, 4, 5]].reshape(-1) for s in sos] + [np.zeros(5)]).astype(np.float64)   # b0 b1 b2 a1 a2
    coef_d = torch.from_numpy(coef).to(x.device)
    nsec_d = torch.from_numpy(nsec).to(x.device)
    y = torch.empty_like(x)
    # only series longer than 2,560 samples go through the scratch-tiled one-thread-per-series kernel
    scratch = torch.empty((T * ((B * C + 127) // 128 * 128),), dtype=torch.float64, device=x.device) if T > 2560 else None
    if B * C:
        with torch.cuda.device(x.device):
            _lib.call("na_iir_chain", x.data_ptr(), y.data_ptr(), ops._ptr(scratch), coef_d.data_ptr(), nsec_d.data_ptr(),
                      len(sos), B, T, C, int(detrend), int(round_decimals), int(carry_state),
                      int(nsec.max()) if len(sos) else 0, ops._stream())
    return y


def chain_fma_per_sample(chain: Sequence[Tuple[str, float, float, int]] = COLLECTOR_CHAIN) -> int:
    """fp64 FMAs per sample of the warp-per-series kernel: every section is passed twice (zero phase), a pass costs
    2 (zero-state run) + 5 (real run) FMAs per sample."""
    return sum(2 * order * 7 for _, _, _, order in chain)
