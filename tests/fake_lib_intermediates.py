"""Host-memory stand-in for the intermediates entry points of libneuroalpha_b200.so (TEST INFRASTRUCTURE).

Extends tests/fake_lib.FakeLib with ``na_head_fwd_f32_ex`` and ``na_attention_softmax_f32`` in numpy, on raw HOST
pointers, so that ``EEG_LSTM.decode_intermediates`` can be exercised on the generic path where there is no GPU
(tests/test_intermediates_host.py).  The product never imports this module.
"""
from __future__ import annotations

import numpy as np

from tests.fake_lib import FakeLib, _arr


class FakeLibIntermediates(FakeLib):
    def na_head_fwd_f32_ex(self, h, aw, ab, lw, lb, w0, b0, w3, b3, rrelu_slope, drop_mask, drop_scale,
                           logits, probs, scores_tm, pooled, embedding, stats, zpool, T, B, Bp, H, NC, stream):
        rc = self.na_head_fwd_f32(h, aw, ab, lw, lb, w0, b0, w3, b3, rrelu_slope, drop_mask, drop_scale,
                                  logits, probs, stats, zpool, T, B, Bp, H, NC, stream)
        if rc:
            return rc
        P = self._head_params((aw, ab, lw, lb, w0, b0, w3, b3), H, NC)
        hh = _arr(h, (T, Bp, H)).astype(np.float64)[:, :B]
        s = hh @ P["aw"] + P["ab"]                       # [T,B]
        e = np.exp(s - s.max(axis=0))
        zp = np.einsum("tb,tbh->bh", e, hh) / e.sum(axis=0)[:, None]
        if scores_tm is not None:
            _arr(scores_tm, (T, B))[...] = s
        if pooled is not None:
            _arr(pooled, (B, H))[...] = zp
        if embedding is not None:
            mean = zp.mean(axis=1, keepdims=True)
            var = ((zp - mean) ** 2).mean(axis=1, keepdims=True)
            _arr(embedding, (B, H))[...] = (zp - mean) / np.sqrt(var + 1e-5) * P["lw"] + P["lb"]
        return 0

    def na_attention_softmax_f32(self, scores_tm, attn, T, B, stream):
        if T < 1 or B < 1:
            return self._fail("na_attention_softmax_f32: bad shape")
        s = _arr(scores_tm, (T, B)).astype(np.float64).T
        e = np.exp(s - s.max(axis=1, keepdims=True))
        _arr(attn, (B, T))[...] = e / e.sum(axis=1, keepdims=True)
        self.launches += 1
        return 0
