"""Host-memory stand-in for the sequence-LSTM entry points of libneuroalpha_b200.so (TEST INFRASTRUCTURE).

Extends tests/fake_lib.FakeLib with ``na_lstm_layer_fwd_f32_hx``, ``na_lstm_layer_bwd_f32_hx``,
``na_lstm_layer_wgrad_f32_hx`` and ``na_decoder_lstm_x3`` (plus the x3 weight packing it needs) in numpy, on raw HOST
pointers, so that ``EEG_LSTM.lstm(x, hx)`` and its autograd can be exercised where there is no GPU
(tests/test_lstm_sequence_host.py).  ``calls`` records which of the new entry points ran, in order.  The x3 "weight
image" here is the eight fp32 tensors back to back, not the kernel's fp16 layout.  The product never imports this module.
"""
from __future__ import annotations

import numpy as np

from tests.fake_lib import FakeLib, _arr, _sig

X3_BYTES = 40 * 3072
X3_SHAPES = [(192, 8), (192, 48), (192,), (192,), (192, 48), (192, 48), (192,), (192,)]


def _lstm_layer(x, w_ih, w_hh, bias, h, c):
    """x [T,N,K] float64 -> (h [T,N,H], c [T,N,H], gates [T,N,4H] activated i,f,g,o)."""
    H = w_hh.shape[1]
    hs, cs, gs = [], [], []
    for t in range(x.shape[0]):
        g = x[t] @ w_ih.T + h @ w_hh.T + bias
        i, f, gg, o = _sig(g[:, :H]), _sig(g[:, H:2 * H]), np.tanh(g[:, 2 * H:3 * H]), _sig(g[:, 3 * H:])
        c = f * c + i * gg
        h = o * np.tanh(c)
        hs.append(h); cs.append(c); gs.append(np.concatenate([i, f, gg, o], axis=1))
    return np.stack(hs), np.stack(cs), np.stack(gs)


class FakeLibSequence(FakeLib):
    def __init__(self):
        super().__init__()
        self.calls = []

    def na_lstm_layer_fwd_f32_hx(self, inp, wt, bias, hout, cout, gates, drop_mask, drop_scale, hout_drop,
                                 T, Bp, K, H, h_init, c_init, stream):
        self.calls.append("na_lstm_layer_fwd_f32_hx")
        if Bp % 32 or Bp <= 0:
            return self._fail("na_lstm_layer_fwd_f32: bad shape")
        if (h_init is None) != (c_init is None):
            return self._fail("na_lstm_layer_fwd_f32_hx: h_init and c_init must be given together")
        G = 4 * H
        W = _arr(wt, (K + H, G)).astype(np.float64)
        h0 = _arr(h_init, (Bp, H)).astype(np.float64) if h_init is not None else np.zeros((Bp, H))
        c0 = _arr(c_init, (Bp, H)).astype(np.float64) if c_init is not None else np.zeros((Bp, H))
        h, c, g = _lstm_layer(_arr(inp, (T, Bp, K)).astype(np.float64), W[:K].T, W[K:].T,
                              _arr(bias, (G,)).astype(np.float64), h0, c0)
        _arr(hout, (T, Bp, H))[...] = h
        if cout is not None:
            _arr(cout, (T, Bp, H))[...] = c
        if gates is not None:
            _arr(gates, (T, Bp, G))[...] = g
        if drop_mask is not None:
            _arr(hout_drop, (T, Bp, H))[...] = h * _arr(drop_mask, (T, Bp, H)) * drop_scale
        self.launches += 1
        return 0

    def na_lstm_layer_bwd_f32_hx(self, dh_out, gates, cstate, w_ih, w_hh, dgates, din, in_drop_mask, drop_scale,
                                 T, Bp, K, H, c_init, dh_last, dc_last, dh_init, dc_init, stream):
        self.calls.append("na_lstm_layer_bwd_f32_hx")
        G = 4 * H
        dho = _arr(dh_out, (T, Bp, H)).astype(np.float64)
        ga = _arr(gates, (T, Bp, G)).astype(np.float64)
        cs = _arr(cstate, (T, Bp, H)).astype(np.float64)
        wi, wh = _arr(w_ih, (G, K)).astype(np.float64), _arr(w_hh, (G, H)).astype(np.float64)
        mask = _arr(in_drop_mask, (T, Bp, K))
        zero = np.zeros((Bp, H))
        c_prev0 = _arr(c_init, (Bp, H)).astype(np.float64) if c_init is not None else zero
        dhrec = _arr(dh_last, (Bp, H)).astype(np.float64) if dh_last is not None else zero
        dc = _arr(dc_last, (Bp, H)).astype(np.float64) if dc_last is not None else zero
        for t in range(T - 1, -1, -1):
            i, f, g, o = ga[t, :, :H], ga[t, :, H:2 * H], ga[t, :, 2 * H:3 * H], ga[t, :, 3 * H:]
            cp = cs[t - 1] if t > 0 else c_prev0
            tc = np.tanh(cs[t])
            dh = dho[t] + dhrec
            dct = dc + dh * o * (1 - tc * tc)
            dc = dct * f
            pre = np.concatenate([dct * g * i * (1 - i), dct * cp * f * (1 - f), dct * i * (1 - g * g),
                                  dh * tc * o * (1 - o)], axis=1)
            _arr(dgates, (T, Bp, G))[t] = pre
            dhrec = pre @ wh
            if din is not None:
                v = pre @ wi
                _arr(din, (T, Bp, K))[t] = v * mask[t] * drop_scale if mask is not None else v
        if dh_init is not None:
            _arr(dh_init, (Bp, H))[...] = dhrec
        if dc_init is not None:
            _arr(dc_init, (Bp, H))[...] = dc
        self.launches += 1
        return 0

    def na_lstm_layer_wgrad_f32_hx(self, dgates, inp, h, dw_ih, dw_hh, db, partials, T, Bp, K, H, h_init, stream):
        self.calls.append("na_lstm_layer_wgrad_f32_hx")
        rc = self.na_lstm_layer_wgrad_f32(dgates, inp, h, dw_ih, dw_hh, db, partials, T, Bp, K, H, stream)
        if rc == 0 and h_init is not None:
            dg0 = _arr(dgates, (T, Bp, 4 * H))[0].astype(np.float64)
            out = _arr(dw_hh, (4 * H, H))
            out[...] = out + dg0.T @ _arr(h_init, (Bp, H)).astype(np.float64)
        return rc

    # -- exact tier, sequence output ----------------------------------------------------------
    def na_decoder_packed_x3_bytes(self):
        return X3_BYTES

    def na_decoder_pack_x3(self, w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1, packed, stream):
        flat = np.concatenate([_arr(p, s).ravel() for p, s in zip((w_ih0, w_hh0, b_ih0, b_hh0, w_ih1, w_hh1, b_ih1, b_hh1),
                                                                  X3_SHAPES)])
        _arr(packed, (X3_BYTES // 4,))[:flat.size] = flat
        self.launches += 1
        return 0

    def na_decoder_lstm_x3(self, x, packed, h_init, c_init, out, h_n, c_n, T, B, stream):
        self.calls.append("na_decoder_lstm_x3")
        if T < 1 or B < 1:
            return self._fail("na_decoder_lstm_x3: bad shape")
        if (h_init is None) != (c_init is None):
            return self._fail("na_decoder_lstm_x3: h_init and c_init must be given together")
        img = _arr(packed, (X3_BYTES // 4,)).astype(np.float64)
        ws, pos = [], 0
        for s in X3_SHAPES:
            n = int(np.prod(s))
            ws.append(img[pos:pos + n].reshape(s))
            pos += n
        hi = _arr(h_init, (2, B, 48)).astype(np.float64) if h_init is not None else np.zeros((2, B, 48))
        ci = _arr(c_init, (2, B, 48)).astype(np.float64) if c_init is not None else np.zeros((2, B, 48))
        cur = _arr(x, (B, T, 8)).astype(np.float64).transpose(1, 0, 2)
        hn, cn = _arr(h_n, (2, B, 48)), _arr(c_n, (2, B, 48))
        for l in range(2):
            w_ih, w_hh, b_ih, b_hh = ws[4 * l:4 * l + 4]
            h, c, _ = _lstm_layer(cur, w_ih, w_hh, b_ih + b_hh, hi[l], ci[l])
            hn[l], cn[l] = h[-1], c[-1]
            cur = h
        _arr(out, (B, T, 48))[...] = cur.transpose(1, 0, 2)
        self.launches += 1
        return 0
