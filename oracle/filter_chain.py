"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  CPU restatement of the collector's BrainFlow filter chain
(Neural_decoding_data_collector.py:109-127).  PARITY UNPINNED: brainflow==5.19.0 (C++ DSPFilters) is a third-party
dependency that is not installed in this image and not vendored in /root/reference, so this restates its
published algorithm: Butterworth designs from scipy.signal.butter (the same transfer functions DSPFilters'
Butterworth::Design::BandStop / BandPass produce), DirectFormII cascades, "zero phase" = process, reverse,
process again with the SAME filter object (state carried over), reverse."""
import numpy as np
from scipy import signal

CHAIN = (("bandstop", 39.5, 40.5, 4), ("bandpass", 3.0, 48.0, 2), ("bandstop", 49.5, 50.5, 4), ("bandstop", 59.0, 61.0, 4))


def scipy_sos(kind, lo, hi, order, fs):
    return signal.butter(order, [lo, hi], btype=kind, fs=fs, output="sos")


def cascade(x, sos, state):
    """DirectFormII biquad cascade over a 1-D float64 series, explicit loops; `state` [nsec, 2] is updated in place."""
    y = np.empty_like(x)
    for t in range(x.shape[0]):
        v = x[t]
        for s in range(sos.shape[0]):
            b0, b1, b2, _, a1, a2 = sos[s]
            w = v - a1 * state[s, 0] - a2 * state[s, 1]
            v = b0 * w + b1 * state[s, 0] + b2 * state[s, 1]
            state[s, 1] = state[s, 0]
            state[s, 0] = w
        y[t] = v
    return y


def collector_round(x, decimals):
    """The collector's output rule: np.round(x, decimals) (skipped for decimals < 0), negative zero cleared, float32."""
    x = np.asarray(x, dtype=np.float64)
    if decimals >= 0:
        x = np.round(x, decimals)
        x[x == 0] = 0.0
    return x.astype(np.float32)


def zero_phase_chain(window_TxC, sos_list, carry_state=True, detrend=True):
    """[T, C] -> [T, C] float64 before rounding: the explicit-loop restatement, one channel at a time."""
    x = np.asarray(window_TxC, dtype=np.float64)
    out = np.empty_like(x)
    for c in range(x.shape[1]):
        v = x[:, c].copy()
        if detrend:
            v = v - v.mean()
        for sos in sos_list:
            st = np.zeros((sos.shape[0], 2))
            v = cascade(v, sos, st)
            if not carry_state:
                st[:] = 0.0
            v = cascade(v[::-1].copy(), sos, st)[::-1].copy()
        out[:, c] = v
    return out


def zero_phase_chain_sosfilt(x, sos_list, carry_state=True, detrend=True, axis=-2):
    """zero_phase_chain for any number of series at once (default layout [..., T, C]), float64, with
    scipy.signal.sosfilt.  Carrying sosfilt's final state into the reversed pass continues the same filter, which is
    what carrying the DirectFormII state does; the two differ only by rounding."""
    x = np.asarray(x, dtype=np.float64)
    if detrend:
        x = x - x.mean(axis=axis, keepdims=True)
    for sos in sos_list:
        zshape = list(x.shape)
        zshape[axis] = 2
        zeros = np.zeros((sos.shape[0], *zshape))
        y, zf = signal.sosfilt(sos, x, axis=axis, zi=zeros)
        y, _ = signal.sosfilt(sos, np.flip(y, axis), axis=axis, zi=zf if carry_state else zeros)
        x = np.flip(y, axis)
    return np.ascontiguousarray(x)


def collector_chain(window_TxC, fs=125.0, sos_list=None, carry_state=True, detrend=True, decimals=7):
    """[T, C] float -> [T, C] float32, the values the collector would write (and the loader read back)."""
    sos_list = sos_list if sos_list is not None else [scipy_sos(k, lo, hi, o, fs) for k, lo, hi, o in CHAIN]
    return collector_round(zero_phase_chain(window_TxC, sos_list, carry_state, detrend), decimals)
