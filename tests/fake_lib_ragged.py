"""Host-memory stand-in for the ragged stream entry points of libneuroalpha_b200.so (TEST INFRASTRUCTURE).

Extends the stream fake with numpy versions of ``na_decoder_stream_ragged_x3`` and ``na_attention_pool_stream_ragged_f32``
on raw HOST pointers, in float64, so that ``decode`` / ``decode_stream`` with ``lengths`` can be exercised where there is
no GPU (tests/test_ragged_host.py).  Row b takes steps t < lengths[b] only, as the kernels do; like the real library both
reject a NULL ``lengths`` and pointers that are not 16-byte aligned.  The product never imports this module.
"""
from __future__ import annotations

import ctypes

import numpy as np

from tests.fake_lib import RRELU_EVAL, _arr
from tests.fake_lib_sequence import X3_SHAPES, _lstm_layer
from tests.fake_lib_stream import FakeLibStream, _aligned, pool_steps


def _lengths(ptr, B, T):
    """int32 [B] at a host address, clamped to [0, T] as the kernels clamp it."""
    buf = (ctypes.c_int32 * B).from_address(int(ptr))
    return np.clip(np.ctypeslib.as_array(buf).astype(np.int64), 0, T)


def pool_rows(h, s, lens, m, l, z):
    """pool_steps where row b takes in its first lens[b] steps only -> the state after them."""
    m, l, z = m.copy(), l.copy(), z.copy()
    for b, n in enumerate(lens):
        m[b:b + 1], l[b:b + 1], z[b:b + 1] = pool_steps(h[b:b + 1, :n], s[b:b + 1, :n], m[b:b + 1], l[b:b + 1], z[b:b + 1])
    return m, l, z


class FakeLibRagged(FakeLibStream):
    def na_decoder_stream_ragged_x3(self, x, packed, aw, ab, lw, lb, w0, b0, w3, b3, h_in, c_in, m_in, l_in, z_in, lengths,
                                    logits, probs, h_out, c_out, m_out, l_out, z_out, T, B, NC, stream):
        self.calls.append("na_decoder_stream_ragged_x3")
        if T < 1 or B < 1:
            return self._fail("na_decoder_stream_ragged_x3: bad shape")
        if lengths is None:
            return self._fail("na_decoder_stream_ragged_x3: null pointer lengths")
        given = [p is not None for p in (h_in, c_in, m_in, l_in, z_in)]
        if any(given) and not all(given):
            return self._fail("na_decoder_stream_ragged_x3: h_in, c_in, m_in, l_in and z_in must be given together")
        if not _aligned(x, packed, h_in, c_in, m_in, l_in, z_in, lengths, logits, probs, h_out, c_out, m_out, l_out, z_out):
            return self._fail("na_decoder_stream_ragged_x3: not 16-byte aligned", -2)
        lens = _lengths(lengths, B, T)
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
        rows, last, empty = np.arange(B), np.maximum(lens - 1, 0), (lens == 0)[:, None]
        with np.errstate(invalid="ignore", over="ignore"):
            for layer in range(2):
                w_ih, w_hh, b_ih, b_hh = ws[4 * layer:4 * layer + 4]
                h, c, _ = _lstm_layer(cur, w_ih, w_hh, b_ih + b_hh, hi[layer], ci[layer])
                hn[layer] = np.where(empty, hi[layer], h[last, rows])
                cn[layer] = np.where(empty, ci[layer], c[last, rows])
                cur = h
            hb = cur.transpose(1, 0, 2)
            s = hb @ f64(aw, (48,)) + float(_arr(ab, (1,))[0])
            m0 = np.full(B, -np.inf) if fresh else f64(m_in, (B,))
            l0 = np.zeros(B) if fresh else f64(l_in, (B,))
            z0 = np.zeros((B, 48)) if fresh else f64(z_in, (B, 48))
            m, l, z = pool_rows(hb, s, lens, m0, l0, z0)
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

    def na_attention_pool_stream_ragged_f32(self, h, aw, ab, m_in, l_in, z_in, lengths, pooled, m_out, l_out, z_out, T, B,
                                            Bp, H, stream):
        self.calls.append("na_attention_pool_stream_ragged_f32")
        if T < 1 or B < 1 or Bp < B:
            return self._fail("na_attention_pool_stream_ragged_f32: bad shape")
        if lengths is None:
            return self._fail("na_attention_pool_stream_ragged_f32: null pointer lengths")
        given = [p is not None for p in (m_in, l_in, z_in)]
        if any(given) and not all(given):
            return self._fail("na_attention_pool_stream_ragged_f32: m_in, l_in and z_in must be given together")
        if not _aligned(h, m_in, l_in, z_in, lengths, pooled, m_out, l_out, z_out):
            return self._fail("na_attention_pool_stream_ragged_f32: not 16-byte aligned", -2)
        lens = _lengths(lengths, B, T)
        hb = _arr(h, (T, Bp, H)).astype(np.float64)[:, :B].transpose(1, 0, 2)
        fresh = m_in is None
        with np.errstate(invalid="ignore", over="ignore"):
            s = hb @ _arr(aw, (H,)).astype(np.float64) + float(_arr(ab, (1,))[0])
            m, l, z = pool_rows(hb, s, lens, np.full(B, -np.inf) if fresh else _arr(m_in, (B,)).astype(np.float64),
                                np.zeros(B) if fresh else _arr(l_in, (B,)).astype(np.float64),
                                np.zeros((B, H)) if fresh else _arr(z_in, (B, H)).astype(np.float64))
            _arr(pooled, (B, H))[...] = z / l[:, None]
        _arr(m_out, (B,))[...] = m
        _arr(l_out, (B,))[...] = l
        _arr(z_out, (B, H))[...] = z
        self.launches += 1
        return 0
