"""Host-memory stand-in for the stream entry points of libneuroalpha_b200.so (TEST INFRASTRUCTURE).

Extends the sequence fake (``na_lstm_layer_fwd_f32_hx``, the x3 weight packing) and the prefix fake (the eval head tail)
with numpy versions of ``na_decoder_stream_x3`` and ``na_attention_pool_stream_f32`` on raw HOST pointers, in float64,
so that ``EEG_LSTM.decode_stream`` can be exercised where there is no GPU (tests/test_stream_host.py).  Like the real
library, both reject pointers that are not 16-byte aligned.  The product never imports this module.
"""
from __future__ import annotations

import numpy as np

from tests.fake_lib import RRELU_EVAL, _arr
from tests.fake_lib_sequence import X3_SHAPES, FakeLibSequence, _lstm_layer
from tests.test_prefix_host import FakeLibPrefix


def pool_steps(h, s, m, l, z):
    """The attention pool's online softmax over the steps of h [B,T,H] with scores s [B,T], from the state m / l [B],
    z [B,H] (float64; m = -inf, l = 0, z = 0 for a fresh pool) -> the state after the last step."""
    m, l, z = m.copy(), l.copy(), z.copy()
    with np.errstate(invalid="ignore"):
        for t in range(h.shape[1]):
            mn = np.maximum(m, s[:, t])
            sc = np.where(np.isneginf(m), 0.0, np.exp(m - mn))
            e = np.exp(s[:, t] - mn)
            l = l * sc + e
            z = z * sc[:, None] + e[:, None] * h[:, t]
            m = mn
    return m, l, z


def _aligned(*ptrs):
    return all(p is None or int(p) % 16 == 0 for p in ptrs)


class FakeLibStream(FakeLibSequence, FakeLibPrefix):
    def na_decoder_stream_x3(self, x, packed, aw, ab, lw, lb, w0, b0, w3, b3, h_in, c_in, m_in, l_in, z_in, logits, probs,
                             h_out, c_out, m_out, l_out, z_out, T, B, NC, stream):
        self.calls.append("na_decoder_stream_x3")
        if T < 1 or B < 1:
            return self._fail("na_decoder_stream_x3: bad shape")
        given = [p is not None for p in (h_in, c_in, m_in, l_in, z_in)]
        if any(given) and not all(given):
            return self._fail("na_decoder_stream_x3: h_in, c_in, m_in, l_in and z_in must be given together")
        if not _aligned(x, packed, h_in, c_in, m_in, l_in, z_in, logits, probs, h_out, c_out, m_out, l_out, z_out):
            return self._fail("na_decoder_stream_x3: not 16-byte aligned", -2)
        img = _arr(packed, (sum(int(np.prod(s)) for s in X3_SHAPES),)).astype(np.float64)
        ws, pos = [], 0
        for s in X3_SHAPES:
            n = int(np.prod(s))
            ws.append(img[pos:pos + n].reshape(s))
            pos += n
        f64 = lambda p, shape: _arr(p, shape).astype(np.float64)
        fresh = h_in is None
        hi = np.zeros((2, B, 48)) if fresh else f64(h_in, (2, B, 48))
        ci = np.zeros((2, B, 48)) if fresh else f64(c_in, (2, B, 48))
        cur = f64(x, (B, T, 8)).transpose(1, 0, 2)
        hn, cn = _arr(h_out, (2, B, 48)), _arr(c_out, (2, B, 48))
        for layer in range(2):
            w_ih, w_hh, b_ih, b_hh = ws[4 * layer:4 * layer + 4]
            h, c, _ = _lstm_layer(cur, w_ih, w_hh, b_ih + b_hh, hi[layer], ci[layer])
            hn[layer], cn[layer] = h[-1], c[-1]
            cur = h
        hb = cur.transpose(1, 0, 2)
        s = hb @ f64(aw, (48,)) + float(_arr(ab, (1,))[0])
        m0 = np.full(B, -np.inf) if fresh else f64(m_in, (B,))
        l0 = np.zeros(B) if fresh else f64(l_in, (B,))
        z0 = np.zeros((B, 48)) if fresh else f64(z_in, (B, 48))
        m, l, z = pool_steps(hb, s, m0, l0, z0)
        _arr(m_out, (B,))[...] = m
        _arr(l_out, (B,))[...] = l
        _arr(z_out, (B, 48))[...] = z
        P = self._head_params((aw, ab, lw, lb, w0, b0, w3, b3), 48, NC)
        lg = self._tail(z / l[:, None], P, float(RRELU_EVAL), 1.0)[4] @ P["w3"].T + P["b3"]
        _arr(logits, (B, NC))[...] = lg
        if probs is not None:
            e = np.exp(lg - lg.max(axis=1, keepdims=True))
            _arr(probs, (B, NC))[...] = e / e.sum(axis=1, keepdims=True)
        self.launches += 1
        return 0

    def na_attention_pool_stream_f32(self, h, aw, ab, m_in, l_in, z_in, pooled, m_out, l_out, z_out, T, B, Bp, H, stream):
        self.calls.append("na_attention_pool_stream_f32")
        if T < 1 or B < 1 or Bp < B:
            return self._fail("na_attention_pool_stream_f32: bad shape")
        given = [p is not None for p in (m_in, l_in, z_in)]
        if any(given) and not all(given):
            return self._fail("na_attention_pool_stream_f32: m_in, l_in and z_in must be given together")
        if not _aligned(h, m_in, l_in, z_in, pooled, m_out, l_out, z_out):
            return self._fail("na_attention_pool_stream_f32: not 16-byte aligned", -2)
        hb = _arr(h, (T, Bp, H)).astype(np.float64)[:, :B].transpose(1, 0, 2)
        s = hb @ _arr(aw, (H,)).astype(np.float64) + float(_arr(ab, (1,))[0])
        fresh = m_in is None
        m, l, z = pool_steps(hb, s, np.full(B, -np.inf) if fresh else _arr(m_in, (B,)).astype(np.float64),
                             np.zeros(B) if fresh else _arr(l_in, (B,)).astype(np.float64),
                             np.zeros((B, H)) if fresh else _arr(z_in, (B, H)).astype(np.float64))
        _arr(pooled, (B, H))[...] = z / l[:, None]
        _arr(m_out, (B,))[...] = m
        _arr(l_out, (B,))[...] = l
        _arr(z_out, (B, H))[...] = z
        self.launches += 1
        return 0
