"""Drop-in replacement of ``Neuro-Alpha-App/Utilities/lstm_eeg_model.py`` on B200.

Same public names (``CLASS_NAMES``, ``EEG_LSTM``, ``SimplePredictor``), same constructor
signatures and defaults, same 16-key ``state_dict`` layout, same ``forward(x) -> logits``
contract (reference lstm_eeg_model.py:11-101) -- but every arithmetic step runs in
hand-written sm_100a kernels (libneuroalpha_b200.so).  There is no CPU compute path:
``EEG_LSTM.forward`` on a CPU tensor raises.
"""
from __future__ import annotations

import math
import operator
from typing import Dict, List, NamedTuple, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import ops

CLASS_NAMES = ["Food", "Water", "BG-Noise"]      # reference lstm_eeg_model.py:11, verbatim


class DecoderOutputs(NamedTuple):
    """``EEG_LSTM.decode_intermediates``: everything the eval forward computes per window, fp32 on the device of ``x``.
    ``attention`` = softmax over time of ``attn(out)`` (reference lstm_eeg_model.py:36), ``pooled`` = the attention-weighted
    sum of the last LSTM layer's h (:37), ``embedding`` = ``ln(pooled)``, the input of ``fc`` (:38)."""
    logits: torch.Tensor        # [B, K]
    probs: torch.Tensor         # [B, K]
    attention: torch.Tensor     # [B, T]
    pooled: torch.Tensor        # [B, H]
    embedding: torch.Tensor     # [B, H]


class PrefixOutputs(NamedTuple):
    """``EEG_LSTM.decode_prefixes``: the eval forward of every prefix ``x[:, :t]`` of the windows, fp32 on the device of
    ``x``.  ``logits[:, j]`` is ``decode(x[:, :lengths[j]])[0]``."""
    lengths: torch.Tensor       # [P] long, t_j = min((j + 1) * stride, T); the last is T
    logits: torch.Tensor        # [B, P, K]
    probs: torch.Tensor         # [B, P, K]


class DecoderState(NamedTuple):
    """The state of B streams after the chunks ``EEG_LSTM.decode_stream`` has taken in, fp32 on the device of the chunks.
    ``h`` / ``c`` have nn.LSTM's ``h_n`` / ``c_n`` layout (the same as ``model.lstm``'s), batch dimension 1; the three
    attention-pool fields are the pool's online softmax over the steps seen so far, batch dimension 0: the running max
    ``m`` of the scores s_t = attn(h_t), ``sum_t exp(s_t - m)`` and ``sum_t exp(s_t - m) h_t`` (the pooled vector is
    ``pool_z / pool_sum[:, None]``).  Rows are independent: index, concatenate or reset them with plain torch (a fresh
    row is ``EEG_LSTM.initial_stream_state``'s: zeros, ``pool_max = -inf``)."""
    h: torch.Tensor             # [L, B, H]
    c: torch.Tensor             # [L, B, H]
    pool_max: torch.Tensor      # [B]
    pool_sum: torch.Tensor      # [B]
    pool_z: torch.Tensor        # [B, H]


class StreamOutputs(NamedTuple):
    """``EEG_LSTM.decode_stream``: the eval forward of everything each stream has received, and the state after the
    chunk (fp32 on the device of ``x``)."""
    logits: torch.Tensor        # [B, K]
    probs: torch.Tensor         # [B, K]
    state: DecoderState


class Attributions(NamedTuple):
    """``EEG_LSTM.input_gradients`` / ``integrated_gradients``: fp32 on the device of ``x``."""
    logits: torch.Tensor        # [B, K], at x
    target: torch.Tensor        # [B] long, the explained class of each window
    attributions: torch.Tensor  # [B, T, C]
    delta: Optional[torch.Tensor] = None    # [B] integrated gradients: sum(attributions) - (F(x) - F(baseline))


class LSTMParameters(nn.Module):
    """Parameter container with ``nn.LSTM``'s names, shapes, registration order and default init
    (U(-1/sqrt(H), 1/sqrt(H)) for every tensor, drawn in registration order), so that
    ``torch.manual_seed(s); EEG_LSTM()`` reproduces the reference's weights and the 16-key
    ``state_dict`` loads with ``strict=True`` (reference lstm_eeg_model.py:16-22, 81).

    Calling it is ``nn.LSTM(batch_first=True)``'s forward (see ``forward``).  ``EEG_LSTM.forward``,
    ``decode`` and ``decode_intermediates`` run their own fused kernels and never call it, so a forward
    hook on ``model.lstm`` fires only when the user calls ``model.lstm(...)``.
    """

    def __init__(self, input_size: int, hidden_size: int, num_layers: int, dropout: float):
        super().__init__()
        self.input_size, self.hidden_size, self.num_layers = input_size, hidden_size, num_layers
        self.dropout = float(dropout)
        self.batch_first = True
        self.bidirectional = False
        self._pack_cache: Dict[object, tuple] = {}         # shared with the owning EEG_LSTM (same dict object)
        for l in range(num_layers):
            k = input_size if l == 0 else hidden_size
            self.register_parameter(f"weight_ih_l{l}", nn.Parameter(torch.empty(4 * hidden_size, k)))
            self.register_parameter(f"weight_hh_l{l}", nn.Parameter(torch.empty(4 * hidden_size, hidden_size)))
            self.register_parameter(f"bias_ih_l{l}", nn.Parameter(torch.empty(4 * hidden_size)))
            self.register_parameter(f"bias_hh_l{l}", nn.Parameter(torch.empty(4 * hidden_size)))
        self.reset_parameters()

    def reset_parameters(self) -> None:
        stdv = 1.0 / math.sqrt(self.hidden_size) if self.hidden_size > 0 else 0.0
        for w in self.parameters():
            nn.init.uniform_(w, -stdv, stdv)

    def layer(self, l: int) -> List[torch.Tensor]:
        return [getattr(self, f"{n}_l{l}") for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]

    def extra_repr(self) -> str:
        return f"{self.input_size}, {self.hidden_size}, num_layers={self.num_layers}, batch_first=True, dropout={self.dropout}"

    def _cached_pack(self, slot, ps, make):
        key = tuple((p.data_ptr(), p._version, p.dtype) for p in ps)
        hit = self._pack_cache.get(slot)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                hit = (key, make())
            self._pack_cache[slot] = hit
        return hit[1]

    def _packed_x3(self):
        ps = self.layer(0) + self.layer(1)
        return self._cached_pack("x3", ps, lambda: ops.decoder_pack_x3(ps))

    def forward(self, input: torch.Tensor, hx: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
        """``nn.LSTM(batch_first=True)``: ``input`` [B,T,C] (or unbatched [T,C]) on a CUDA device, ``hx = (h_0, c_0)``
        [L,B,H] each ([L,H] unbatched; None = zeros) -> ``(output [B,T,H], (h_n, c_n))``, ``output`` = the last layer's
        h at every step, ``h_n`` / ``c_n`` [L,B,H] after the last step (``h_n`` before dropout).  Same argument checks
        and exceptions as nn.LSTM.  The result has the dtype of ``input``; the arithmetic is fp32.  Accuracy against
        float64 nn.LSTM (max|d| / max|ref| per tensor): 1e-5 on the FFMA path and for ``h_n`` / ``c_n``; on the fused
        path the per-step ``output`` of long windows is looser -- 6.2e-5 over the 625 steps of the shipped windows,
        tested at 1e-4 -- because the fp16 hi + lo operand split carries about 22 bits; ``ops.EXACT_TC = False`` selects
        the FFMA path for every call.

        In ``.train()`` mode with ``dropout > 0`` the output of every layer but the last is multiplied by a keep-mask
        ``torch.rand((B, T, H), device=input.device) >= dropout`` (drawn in layer order) and scaled by 1/(1-dropout).
        The owning model's ``compute_dtype`` and ``zscore_input`` do not apply: this sees the raw ``input``, as
        ``self.lstm(x)`` does in the reference.  The flagship shape (8 -> 48, 2 layers) in fp32 without autograd runs
        on the exact tensor-core kernel (``ops.EXACT_TC``); everything else, and every call that needs gradients, on the
        FFMA / generic kernels under ``ops.LSTMSequenceFunction`` (gradients w.r.t. input, weights and ``hx``)."""
        if input.dim() not in (2, 3):
            raise ValueError(f"LSTM: Expected input to be 2D or 3D, got {input.dim()}D instead")
        batched = input.dim() == 3
        x = input if batched else input.unsqueeze(0)
        h0 = c0 = None
        if hx is not None:
            h0, c0 = hx
            if batched and (h0.dim() != 3 or c0.dim() != 3):
                raise RuntimeError("For batched 3-D input, hx and cx should "
                                   f"also be 3-D but got ({h0.dim()}-D, {c0.dim()}-D) tensors")
            if not batched:
                if h0.dim() != 2 or c0.dim() != 2:
                    raise RuntimeError("For unbatched 2-D input, hx and cx should "
                                       f"also be 2-D but got ({h0.dim()}-D, {c0.dim()}-D) tensors")
                h0, c0 = h0.unsqueeze(1), c0.unsqueeze(1)
        w = self.weight_ih_l0
        if x.dtype != w.dtype:
            raise ValueError(f"RNN input dtype ({x.dtype}) does not match weight dtype ({w.dtype}). "
                             f"Convert input: input.to({w.dtype}), or convert model: model.to({x.dtype})")
        if x.size(-1) != self.input_size:
            raise RuntimeError(f"input.size(-1) must be equal to input_size. Expected {self.input_size}, "
                               f"got {x.size(-1)}")
        L, H = self.num_layers, self.hidden_size
        expected = (L, x.size(0), H)
        if h0 is not None:
            if h0.size() != expected:
                raise RuntimeError(f"Expected hidden[0] size {expected}, got {list(h0.size())}")
            if c0.size() != expected:
                raise RuntimeError(f"Expected hidden[1] size {expected}, got {list(c0.size())}")
        ops._require_cuda(x, h0, c0)          # raises on CPU tensors: there is no CPU fallback
        B, T = x.shape[0], x.shape[1]
        if B == 0:
            out, h_n, c_n = x.new_empty((0, T, H)), x.new_empty((L, 0, H)), x.new_empty((L, 0, H))
        else:
            needs_grad = torch.is_grad_enabled() and (
                x.requires_grad or any(p.requires_grad for p in self.parameters())
                or (h0 is not None and (h0.requires_grad or c0.requires_grad)))
            if (ops.EXACT_TC and (self.input_size, H, L) == (8, 48, 2) and x.dtype == torch.float32 and not needs_grad
                    and (not self.training or self.dropout == 0.0)):
                with torch.no_grad():
                    out, h_n, c_n = ops.decoder_lstm_x3(x.contiguous(), self._packed_x3(), h0, c0)
            else:
                masks = None
                if self.training and self.dropout > 0.0 and L > 1:
                    masks = [(torch.rand((B, T, H), device=x.device) >= self.dropout).float() for _ in range(L - 1)]
                flat = [t for l in range(L) for t in self.layer(l)]
                out, h_n, c_n = ops.LSTMSequenceFunction.apply(x, h0, c0, self.dropout, masks, *flat)
        out, h_n, c_n = (t if t.dtype == x.dtype else t.to(x.dtype) for t in (out, h_n, c_n))
        if not batched:
            return out.squeeze(0), (h_n.squeeze(1), c_n.squeeze(1))
        return out, (h_n, c_n)


class EEG_LSTM(nn.Module):
    """LSTM stack -> attention pool over time -> LayerNorm -> Linear(H,32) -> RReLU -> Dropout ->
    Linear(32,num_classes); reference lstm_eeg_model.py:13-39.

    ``forward(x)``: ``x`` float ``[B,T,C]`` on a CUDA device -> logits ``[B,num_classes]`` (dtype
    of ``x``).  ``.eval()`` disables the three stochastic ops (inter-layer LSTM dropout, RReLU
    noise, Dropout); ``.train()`` enables them.  ``zscore_input`` (extra, default off so that the
    contract stays the reference's) turns on the K1 per-window per-channel z-score front stage.
    """

    def __init__(self, input_size=8, hidden_size=48, num_layers=2, num_classes=3, dropout=0.60):
        super().__init__()
        self.lstm = LSTMParameters(input_size, hidden_size, num_layers, dropout if num_layers > 1 else 0.0)
        self.ln = nn.LayerNorm(hidden_size)
        self.attn = nn.Linear(hidden_size, 1)
        # containers only (names fc.0.* / fc.3.* as in the reference); never called, so forward hooks registered on
        # attn / ln / fc never fire -- decode_intermediates() returns what they would see
        self.fc = nn.Sequential(
            nn.Linear(hidden_size, 32),
            nn.RReLU(),
            nn.Dropout(dropout),
            nn.Linear(32, num_classes),
        )
        self.dropout_p = float(dropout)
        self.zscore_input = False
        # torch.float32: exact tier (1e-5 contract; at the flagship shape fp32-accurate tcgen05 kernels with
        # every operand split into fp16 hi + lo, FFMA kernels for the other shapes).  torch.bfloat16: 16-bit
        # tensor-core tier (tcgen05, IEEE fp16 operands / fp32 accumulate, 2e-2 contract -- north_star's
        # "bf16 path"); also selected by bf16 inputs or a .bfloat16() module.  Both tiers train.
        self.compute_dtype = torch.float32
        self._injected_noise: Optional[Dict[str, torch.Tensor]] = None
        self._pack_cache = self.lstm._pack_cache           # one cache: model.lstm(x) reuses the exact tier's weight image

    # -- helpers ---------------------------------------------------------------------------
    def _head_params(self) -> List[torch.Tensor]:
        return [self.attn.weight, self.attn.bias, self.ln.weight, self.ln.bias,
                self.fc[0].weight, self.fc[0].bias, self.fc[3].weight, self.fc[3].bias]

    def invalidate_packed_weights(self) -> None:
        """Drop the packed-weight caches.  They are keyed on (data_ptr, _version, dtype) of the parameters, which
        in-place updates through ``p.data`` (``p.data.copy_()``, EMA, weight clipping) do NOT bump: call this after
        such an update.  ``train()`` / ``eval()``, ``.to()`` / ``.cuda()`` / ``.half()`` and ``load_state_dict`` do it
        themselves."""
        self._pack_cache.clear()

    def train(self, mode: bool = True):
        self._pack_cache.clear()
        return super().train(mode)

    def _apply(self, fn, *args, **kwargs):
        self._pack_cache.clear()
        return super()._apply(fn, *args, **kwargs)

    def load_state_dict(self, *args, **kwargs):
        self._pack_cache.clear()
        out = super().load_state_dict(*args, **kwargs)
        self._pack_cache.clear()
        return out

    def _cached_pack(self, slot, ps, make):
        return self.lstm._cached_pack(slot, ps, make)

    def _packed(self, l: int):
        ps = self.lstm.layer(l)
        return self._cached_pack(l, ps, lambda: ops.pack_lstm_layer(*ps))

    def tc_supported(self) -> bool:
        """Shape implemented by the tensor-core tier (the flagship decoder)."""
        return (self.lstm.input_size == 8 and self.lstm.hidden_size == 48 and self.lstm.num_layers == 2
                and self.fc[3].out_features <= 16)

    def tc_wide_supported(self) -> bool:
        """Wide shapes of the tensor-core tier (streamed weights): BASELINE configs[4] and its neighbours."""
        return (self.lstm.input_size == 8 and self.lstm.hidden_size in ops.WIDE_HIDDEN and self.lstm.num_layers == 2
                and self.fc[3].out_features <= 16)

    def _packed_tc_wide(self):
        ps = self.lstm.layer(0) + self.lstm.layer(1) + [self.attn.weight, self.attn.bias]
        return self._cached_pack("tc_wide", ps, lambda: ops.decoder_pack_wide_bf16(ps[:8], ps[8], ps[9]))

    def _packed_x3(self):
        return self.lstm._packed_x3()

    def _packed_tc(self):
        ps = self.lstm.layer(0) + self.lstm.layer(1)
        return self._cached_pack("tc", ps, lambda: ops.decoder_pack_bf16(ps))

    def _tier(self, x: torch.Tensor, train: bool) -> str:
        """The kernel tier that runs ``x``: "tc" (16-bit tensor cores, flagship shape), "wide" (16-bit tensor cores,
        streamed weights), "x3" (fp32-accurate tensor cores, flagship shape) or "ffma" (FFMA / generic kernels, any
        shape).  The 16-bit tier is chosen by ``compute_dtype``, a bf16 ``x`` or a .bfloat16() module.  ``train``:
        ``forward``'s autograd path, where the tensor-core tiers give no d/dx and x3 has its own switch
        (``ops.EXACT_TC_TRAIN``) and also takes fp16 / bf16 ``x``; otherwise the eval path of ``decode``."""
        half = (self.compute_dtype == torch.bfloat16 or x.dtype == torch.bfloat16
                or self.attn.weight.dtype == torch.bfloat16)
        # a dropout rate within 1.5 / 65536 of 1 scales h0 past fp16's range on the flagship tensor-core tiers
        injected = (self._injected_noise or {}).get("drop1") is not None
        tc_train_ok = (not (train and self.training and self.lstm.dropout > 0.0)
                       or ops.tc_train_dropout_ok(self.dropout_p, mask_tensor=injected))
        if half and not (train and x.requires_grad):
            if self.tc_supported() and tc_train_ok:
                return "tc"
            if self.tc_wide_supported():
                return "wide"
        if train:
            if (ops.EXACT_TC_TRAIN and not half and self.tc_supported() and tc_train_ok and not x.requires_grad
                    and x.dtype in (torch.float32, torch.float16, torch.bfloat16)):
                return "x3"
        elif ops.EXACT_TC and not half and self.tc_supported() and x.dtype == torch.float32 and x.shape[0] > 0:
            return "x3"
        return "ffma"

    def _decode(self, x: torch.Tensor, ex: bool, want_probs: bool = True):
        """``decode`` (``ex`` False: (logits, probs)) and ``decode_intermediates`` (``ex`` True: the five fields of
        ``DecoderOutputs``, the op families' ``*_intermediates``) on the tier ``_tier`` picks.  The two families take
        the same arguments except ``want_probs``, which only the plain ones have."""
        probs = () if ex else (want_probs,)
        z = self.zscore_input
        tier = self._tier(x, train=False)
        with torch.no_grad():
            if tier == "tc":
                op = ops.decoder_infer_tc_intermediates if ex else ops.decoder_infer_tc
                return op(x, self._packed_tc(), self._head_params(), *probs, z)
            if tier == "wide":
                op = ops.decoder_infer_wide_intermediates if ex else ops.decoder_infer_wide
                return op(x, self._packed_tc_wide(), self._head_params(), self.lstm.hidden_size, *probs, z)
            if tier == "x3":
                # exact tier, flagship shape: fp32-accurate tensor-core kernel (fp16 hi/lo operand split); the optional
                # z-score stage is one K1 pass that leaves the windows batch-first in fp32
                if z:
                    x = ops.window_zscore(x, x.shape[1], x.shape[1], True, False, ops.NA_F32)
                op = ops.decoder_infer_x3_intermediates if ex else ops.decoder_infer_x3
                return op(x.contiguous(), self._packed_x3(), self._head_params(), *probs)
            L = self.lstm.num_layers
            op = ops.decoder_infer_intermediates if ex else ops.decoder_infer
            return op(x, [self.lstm.layer(l) for l in range(L)], [ops._f32c(t) for t in self._head_params()], *probs,
                      z, [self._packed(l) for l in range(L)])

    def decode(self, x: torch.Tensor, want_probs: bool = True, lengths=None):
        """Eval-mode forward without autograd: x [B,T,C] on CUDA -> (logits fp32 [B,K], probs fp32 [B,K] or
        empty).  Picks the tier from ``compute_dtype`` / the dtype of ``x`` / the parameters.

        ``lengths`` (a length-B sequence or 1-D integer tensor on any device, values in [1, T]) batches windows of
        different durations, as ``pack_padded_sequence`` does for nn.LSTM: row b is the forward of ``x[b, :lengths[b]]``
        alone, and ``x`` past a row's length is ignored whatever it holds, NaN included.  It runs ``decode_stream(x,
        lengths=lengths)`` from fresh streams and drops the state, so it has that call's contract: on the exact tier
        (``ops.EXACT_TC`` and the flagship shape) row b is ``decode(x[:, :lengths[b]])[b]`` bit for bit (whose error in
        mid-window is up to 2e-5 of float64, DESIGN 10f), elsewhere the FFMA kernels within 1e-5.  Eval arithmetic whatever
        ``self.training`` is; ``compute_dtype`` does not apply (a float16 / bfloat16 ``x`` is converted to fp32);
        ``zscore_input`` raises ``ValueError`` (its statistics would come from the whole padded window).  Reading the
        lengths for validation synchronises with the device once."""
        ops._require_cuda(x)
        if lengths is None:
            return self._decode(x, False, want_probs)
        out = self._stream(x, None, lengths, 1, "decode")
        return out.logits, out.probs if want_probs else torch.empty((0,), dtype=torch.float32, device=x.device)

    def decode_intermediates(self, x: torch.Tensor) -> DecoderOutputs:
        """Eval-mode forward without autograd that also returns the attention weights over time, the pooled vector and
        its LayerNorm output (``DecoderOutputs``, all fp32 on the device of ``x``).

        In the reference these are read with forward hooks on ``model.attn`` / ``model.ln``.  Here ``attn``, ``ln`` and
        ``fc`` are parameter containers that the fused kernels never call, so such hooks do not fire: this method
        replaces them.  The intermediates come from the same kernel launch as the logits, on the tier ``decode`` picks
        (same ``compute_dtype`` / input dtype / ``zscore_input`` handling), and carry that tier's accuracy contract;
        logits and probs are those of ``decode(x)``."""
        ops._require_cuda(x)
        B, T = x.shape[0], x.shape[1]
        if B == 0:
            H, K = self.lstm.hidden_size, self.fc[3].out_features
            e = lambda *shape: torch.empty(shape, dtype=torch.float32, device=x.device)
            return DecoderOutputs(e(0, K), e(0, K), e(0, T), e(0, H), e(0, H))
        return DecoderOutputs(*self._decode(x, True))

    def decode_prefixes(self, x: torch.Tensor, stride: int = 1) -> PrefixOutputs:
        """The decoder's output on every prefix of the windows, from one pass over them: ``x`` [B,T,C] on CUDA (T >= 1)
        -> ``PrefixOutputs(lengths, logits, probs)`` for the P = ceil(T / stride) prefixes ``x[:, :t_j]``, ``t_j =
        min((j + 1) * stride, T)`` (the last prefix is the whole window; a ``stride`` above T gives P = 1).  For an
        accuracy-versus-decision-time curve, or to stop as soon as the decoder is confident.

        ``logits[:, j]`` is ``decode(x[:, :t_j])[0]``, the reference's eval forward on the prefix, under the exact tier's
        1e-5 contract: the LSTM is causal and the attention pool is an online softmax, so the pool's state after step t
        is the pooled vector of ``x[:, :t+1]``; it is stored at every prefix end and the head runs on those vectors.  Eval
        arithmetic whatever ``self.training`` is; ``compute_dtype`` does not apply (a float16 / bfloat16 ``x`` is
        converted to fp32).  The flagship shape runs on the exact tensor-core kernel while ``ops.EXACT_TC`` is set, every
        other shape on the FFMA kernels.  ``zscore_input`` raises ``ValueError``: the z-score takes its statistics from
        the whole window, so a prefix of a normalised window is not a normalised prefix."""
        if x.dim() != 3:
            raise ValueError(f"expected x of shape [B,T,C], got {tuple(x.shape)}")
        ops._require_cuda(x)
        if x.shape[2] != self.lstm.input_size:
            raise RuntimeError(f"input.size(-1) must be equal to input_size. Expected {self.lstm.input_size}, got {x.shape[2]}")
        stride = operator.index(stride)
        if stride < 1:
            raise ValueError(f"stride must be >= 1, got {stride}")
        B, T = x.shape[0], x.shape[1]
        if T < 1:
            raise ValueError("decode_prefixes needs windows of at least one step")
        if self.zscore_input:
            raise ValueError("decode_prefixes: zscore_input normalises with the statistics of the whole window, so a "
                             "prefix of a normalised window is not a normalised prefix")
        lengths = ops.prefix_lengths(T, stride, x.device)
        if B == 0:
            K = self.fc[3].out_features
            e = torch.empty((0, lengths.numel(), K), dtype=torch.float32, device=x.device)
            return PrefixOutputs(lengths, e, e.clone())
        x32 = ops._aligned16(x.detach().float().contiguous())
        head = [p.detach() for p in self._head_params()]
        with torch.no_grad():
            if ops.EXACT_TC and self.tc_supported():
                logits, probs = ops.decoder_prefixes_x3(x32, self._packed_x3(), head, stride)
            else:
                L = self.lstm.num_layers
                logits, probs = ops.decoder_prefixes(x32, [self.lstm.layer(l) for l in range(L)], head, stride,
                                                     [self._packed(l) for l in range(L)])
        return PrefixOutputs(lengths, logits, probs)

    def initial_stream_state(self, B: int, device=None) -> DecoderState:
        """The ``DecoderState`` of B streams that have seen nothing: zeros, except ``pool_max = -inf``.  ``device``
        defaults to the parameters' device.  ``decode_stream(x, initial_stream_state(B))`` is ``decode_stream(x)`` bit
        for bit."""
        L, H = self.lstm.num_layers, self.lstm.hidden_size
        dev = self.attn.weight.device if device is None else torch.device(device)
        z = lambda *shape: torch.zeros(shape, dtype=torch.float32, device=dev)
        return DecoderState(z(L, B, H), z(L, B, H), torch.full((B,), -math.inf, dtype=torch.float32, device=dev),
                            z(B), z(B, H))

    def _check_stream_state(self, state, B: int, device) -> DecoderState:
        """``state`` as a ``DecoderState`` whose fields match chunks of B streams on ``device``; raises otherwise, naming
        the field: ``ValueError`` for the wrong number of fields or a dtype other than float32, ``RuntimeError`` for a
        shape or a device that does not match."""
        if not isinstance(state, tuple) or len(state) != 5:
            raise ValueError("state must be a DecoderState (h, c, pool_max, pool_sum, pool_z)")
        state = DecoderState(*state)
        L, H = self.lstm.num_layers, self.lstm.hidden_size
        want = {"h": (L, B, H), "c": (L, B, H), "pool_max": (B,), "pool_sum": (B,), "pool_z": (B, H)}
        for name, shape in want.items():
            t = getattr(state, name)
            if not isinstance(t, torch.Tensor):
                raise ValueError(f"state.{name} must be a tensor, got {type(t).__name__}")
            if tuple(t.shape) != shape:
                raise RuntimeError(f"state.{name} must have shape {list(shape)} for {B} streams, got {list(t.shape)}")
            if t.dtype != torch.float32:
                raise ValueError(f"state.{name} must be float32, got {t.dtype}")
            if t.device != device:
                raise RuntimeError(f"state.{name} is on {t.device}, the chunk on {device}")
        return state

    def decode_stream(self, x: torch.Tensor, state: Optional[DecoderState] = None, lengths=None) -> StreamOutputs:
        """The decoder on recordings that arrive a chunk at a time: ``x`` [B,T,C] on CUDA (T >= 1) is the next chunk of
        each of B streams, ``state`` the ``DecoderState`` the previous call returned (None: fresh streams) ->
        ``StreamOutputs(logits, probs, state)``.  ``logits`` is ``decode(torch.cat(chunks, dim=1))[0]``, the eval
        forward of everything each stream has received, at the cost of the new steps only: the LSTM carries its (h, c)
        and the attention pool its online softmax (max, sum, weighted sum) from chunk to chunk.  The returned state is
        new; the one passed in is never written.  For dynamic stopping on a live recording: after each chunk, compare
        ``probs.max(1)`` with a threshold (``scripts/accuracy_vs_time.py``).

        On the exact tier (``ops.EXACT_TC`` and the flagship shape) one fused kernel runs per call, and after each chunk
        the logits and probs are bit-identical to ``decode`` of everything streamed so far, and ``state.h`` /
        ``state.c`` to ``model.lstm``'s ``h_n`` / ``c_n``; every other shape runs on the FFMA kernels under the 1e-5
        contract.  Eval arithmetic whatever ``self.training`` is; ``compute_dtype`` does not apply (a float16 /
        bfloat16 ``x`` is converted to fp32).  ``zscore_input`` raises ``ValueError``: the z-score takes its statistics
        from the whole window, which a stream does not have.

        ``lengths`` serves streams that delivered different numbers of samples since the last call in one batch: a
        length-B sequence or 1-D integer tensor on any device, values in [0, T].  Row b then takes only ``x[b,
        :lengths[b]]``; ``x`` past a row's length is ignored whatever it holds, NaN included.  Row b's logits, probs and
        state are those of ``decode_stream(x[b:b+1, :lengths[b]], its state)``: on the exact tier bit for bit, with the
        logits of ``decode`` of everything the stream has received (error up to 2e-5 of float64 in mid-window, DESIGN
        10f / 10g), on the FFMA kernels within 1e-5.  A row given 0 steps returns its state unchanged, bit for bit, and
        the logits of that state: NaN for a stream that has seen nothing.  Reading the lengths for validation
        synchronises with the device once.  ``lengths=None`` is the call without them."""
        return self._stream(x, state, lengths, 0, "decode_stream")

    def _check_lengths(self, lengths, B: int, T: int, low: int, device) -> torch.Tensor:
        """``lengths`` as int32 [B] on ``device``; ``ValueError`` unless it is a length-B sequence or 1-D tensor of
        integers in [low, T].  Reads the values on the host (one synchronisation)."""
        t = lengths
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(lengths)
            if t.numel() == 0:                     # an empty sequence has no dtype to tell
                t = t.long()
        if t.dtype == torch.bool or t.dtype.is_floating_point or t.dtype.is_complex:
            raise ValueError(f"lengths must hold integers, got {t.dtype}")
        if tuple(t.shape) != (B,):
            raise ValueError(f"lengths must have shape [{B}] (one per row of x), got {list(t.shape)}")
        if B > 0:
            lo, hi = (int(v) for v in torch.stack(torch.aminmax(t)).tolist())
            if lo < low or hi > T:
                raise ValueError(f"lengths must lie in [{low}, {T}], got values in [{lo}, {hi}]")
        return t.to(device=device, dtype=torch.int32)

    def _stream(self, x: torch.Tensor, state, lengths, low: int, name: str) -> StreamOutputs:
        """``decode_stream``, and ``decode`` with ``lengths`` (``low`` = the smallest length allowed, ``name`` the
        caller's name in errors)."""
        if x.dim() != 3:
            raise ValueError(f"expected x of shape [B,T,C], got {tuple(x.shape)}")
        ops._require_cuda(x)
        if x.shape[2] != self.lstm.input_size:
            raise RuntimeError(f"input.size(-1) must be equal to input_size. Expected {self.lstm.input_size}, got {x.shape[2]}")
        B, T = x.shape[0], x.shape[1]
        stream = name == "decode_stream"
        if T < 1:
            raise ValueError(f"{name} needs {'chunks' if stream else 'windows'} of at least one step")
        if self.zscore_input:
            why = "which a stream does not have" if stream else "not those of each row's first lengths[b] steps"
            raise ValueError(f"{name}: zscore_input normalises with the statistics of the whole window, {why}")
        if state is not None:
            state = self._check_stream_state(state, B, x.device)
        if lengths is not None:
            lengths = self._check_lengths(lengths, B, T, low, x.device)
        if B == 0:
            K = self.fc[3].out_features
            e = torch.empty((0, K), dtype=torch.float32, device=x.device)
            return StreamOutputs(e, e.clone(), self.initial_stream_state(0, x.device))
        x32 = ops._aligned16(x.detach().float().contiguous())
        head = [p.detach() for p in self._head_params()]
        with torch.no_grad():
            L = self.lstm.num_layers
            if ops.EXACT_TC and self.tc_supported():
                if lengths is None:
                    out = ops.decoder_stream_chunk_x3(x32, self._packed_x3(), head, state)
                else:
                    out = ops.decoder_stream_chunk_ragged_x3(x32, self._packed_x3(), head, state, lengths)
            elif lengths is None:
                out = ops.decoder_stream_chunk(x32, [self.lstm.layer(l) for l in range(L)], head, state,
                                               [self._packed(l) for l in range(L)])
            else:
                out = ops.decoder_stream_chunk_ragged(x32, [self.lstm.layer(l) for l in range(L)], head, state, lengths,
                                                      [self._packed(l) for l in range(L)])
        return StreamOutputs(out[0], out[1], DecoderState(*out[2:]))

    def inject_noise(self, drop1: Optional[torch.Tensor] = None, rrelu_slope: Optional[torch.Tensor] = None,
                     drop2: Optional[torch.Tensor] = None) -> None:
        """Fix the train-mode noise of the NEXT forward calls (reproducible training / parity tests):
        ``drop1`` [L-1,B,T,H] 0/1 keep-mask of the inter-layer dropout, ``rrelu_slope`` [B,32],
        ``drop2`` [B,32] 0/1 keep-mask.  ``inject_noise()`` clears it."""
        if drop1 is None and rrelu_slope is None and drop2 is None:
            self._injected_noise = None
        else:
            self._injected_noise = {"drop1": drop1, "rrelu": rrelu_slope, "drop2": drop2}

    def _draw_noise(self, B: int, T: int, device, pad: int = ops.BATCH_ALIGN, mask_dtype=torch.float32,
                    skip_drop1: bool = False):
        """Train-mode noise as tensors (the kernels are deterministic functions of them): inter-layer
        dropout keep-masks (time-major padded, one per layer gap), RReLU slopes, head dropout mask."""
        p, L, H = self.dropout_p, self.lstm.num_layers, self.lstm.hidden_size
        Bp = ops.padded_batch(B, pad)
        inj = self._injected_noise or {}
        d1 = None
        if L > 1 and self.lstm.dropout > 0.0 and not skip_drop1:
            if inj.get("drop1") is not None:
                m = inj["drop1"].to(device=device, dtype=mask_dtype)             # [L-1,B,T,H]
                d1 = []
                for l in range(L - 1):
                    t = torch.zeros((T, Bp, H), dtype=mask_dtype, device=device)
                    t[:, :B] = m[l].permute(1, 0, 2)
                    d1.append(t)
            else:
                d1 = [(torch.rand((T, Bp, H), device=device) >= p).to(mask_dtype) for _ in range(L - 1)]
        if inj.get("rrelu") is not None:
            rr = inj["rrelu"].to(device=device, dtype=torch.float32).contiguous()
        else:
            rr = torch.empty((B, 32), device=device).uniform_(1.0 / 8.0, 1.0 / 3.0)
        d2 = None
        if p > 0.0:
            if inj.get("drop2") is not None:
                d2 = inj["drop2"].to(device=device, dtype=torch.float32).contiguous()
            else:
                d2 = (torch.rand((B, 32), device=device) >= p).float()
        return d1, rr, d2

    # -- input attributions -----------------------------------------------------------------
    def _targets(self, target, B: int, device) -> Optional[torch.Tensor]:
        if target is None:
            return None
        K = self.fc[3].out_features
        t = torch.as_tensor(target, dtype=torch.long, device=device)
        t = t.expand(B).contiguous() if t.dim() == 0 else t
        if t.shape != (B,):
            raise ValueError(f"target must be an int or a [B] = [{B}] tensor, got shape {tuple(t.shape)}")
        if B and (int(t.min()) < 0 or int(t.max()) >= K):
            raise ValueError(f"target out of range for {K} classes")
        return t

    def input_gradients(self, x: torch.Tensor, target=None) -> Attributions:
        """Saliency: ``d logits[b, target[b]] / d x[b]`` for every window, ``x`` [B,T,C] on CUDA -> ``Attributions(logits,
        target, attributions [B,T,C])``.  ``target``: an int or a [B] long tensor; default the argmax of each window's
        logits.  Eval-mode arithmetic whatever ``self.training`` is; parameter ``.grad``, the module's mode and its packed
        weights are left as they are.  ``compute_dtype`` does not apply: attributions always carry the fp32 contract.

        The flagship shape without ``zscore_input`` runs on the exact tensor-core kernels (``ops.decoder_input_grad_x3``)
        while ``ops.EXACT_TC_TRAIN`` is set.  Its accuracy is looser than the 1e-5 of the weight gradients, because a
        per-step dx does not average over time and windows.  On the 324 shipped windows (625 steps), max|d| / max|ref|
        against float64, on each window's own scale, is at most 4.3e-5 at the argmax class and 8.2e-5 at another class.
        That is the fp16 hi + lo operand split over the BPTT; it is tested at 2e-4.  With ``ops.EXACT_TC_TRAIN = False``
        every call takes the FFMA path: 9.6e-6 at the argmax class (4.8e-5 at another class, on one window).  Everything
        but the flagship shape, and ``zscore_input``, also runs on that path: torch autograd through the FFMA kernels
        (``ops.DecoderFunction``).  It has no gradient through the z-score stage, so ``zscore_input`` raises."""
        return self._input_gradients(x, target)

    def _input_gradients(self, x: torch.Tensor, target) -> Attributions:
        if x.dim() != 3:
            raise ValueError(f"expected x of shape [B,T,C], got {tuple(x.shape)}")
        ops._require_cuda(x)
        if x.shape[2] != self.lstm.input_size:
            raise RuntimeError(f"input.size(-1) must be equal to input_size. Expected {self.lstm.input_size}, got {x.shape[2]}")
        B = x.shape[0]
        tgt = self._targets(target, B, x.device)
        if B == 0:
            K = self.fc[3].out_features
            e = lambda *shape: torch.empty(shape, dtype=torch.float32, device=x.device)
            return Attributions(e(0, K), torch.empty((0,), dtype=torch.long, device=x.device), e(*x.shape))
        x32 = x.detach().float().contiguous()
        L = self.lstm.num_layers
        lstm_params = [[p.detach() for p in self.lstm.layer(l)] for l in range(L)]
        head = [p.detach() for p in self._head_params()]
        if ops.EXACT_TC_TRAIN and self.tc_supported() and not self.zscore_input:
            logits, dx = ops.decoder_input_grad_x3(x32, lstm_params, head, tgt)
        else:
            with torch.enable_grad():
                xg = x32.requires_grad_(True)
                logits = ops.decoder_train_forward(xg, lstm_params, head, self.dropout_p, self.zscore_input)
                pick = logits.argmax(dim=1) if tgt is None else tgt
                (dx,) = torch.autograd.grad(logits.gather(1, pick[:, None]).sum(), xg)
            logits = logits.detach().float()
        if tgt is None:
            tgt = logits.argmax(dim=1)
        return Attributions(logits, tgt, dx)

    def integrated_gradients(self, x: torch.Tensor, target=None, baseline: Optional[torch.Tensor] = None,
                             steps: int = 32) -> Attributions:
        """Integrated gradients (Sundararajan et al., 2017) of ``logits[b, target[b]]`` from ``baseline`` (default zeros: a
        flat signal) to ``x``, midpoint rule: ``alpha_k = (k + 1/2) / steps``, all ``B * steps`` interpolated windows as one
        batch through ``input_gradients``' path; ``attributions = (x - baseline) * mean_k grad``.  ``delta[b] =
        sum(attributions[b]) - (F(x) - F(baseline))`` is the completeness error.  It shrinks as ``steps`` grows once the
        steps resolve the path: on the shipped windows from a zero baseline, from 32 steps on (not from 8 to 16)."""
        if steps < 1:
            raise ValueError("steps must be >= 1")
        if x.dim() != 3:
            raise ValueError(f"expected x of shape [B,T,C], got {tuple(x.shape)}")
        x32 = x.detach().float()
        if baseline is None:
            base = torch.zeros_like(x32)
        else:
            if tuple(baseline.shape) != tuple(x.shape):
                raise ValueError(f"baseline must have the shape of x {tuple(x.shape)}, got {tuple(baseline.shape)}")
            base = baseline.detach().to(device=x32.device, dtype=torch.float32)
        at_x = self._input_gradients(x32, target)
        B = x.shape[0]
        if B == 0:
            return Attributions(at_x.logits, at_x.target, at_x.attributions, at_x.logits.new_empty((0,)))
        alpha = (torch.arange(steps, dtype=torch.float32, device=x32.device) + 0.5) / steps
        diff = x32 - base
        batch = torch.cat([base, (base[None] + alpha[:, None, None, None] * diff[None]).reshape(-1, *x.shape[1:])])
        run = self._input_gradients(batch, at_x.target.repeat(steps + 1))
        grads = run.attributions[B:].reshape(steps, *x.shape).mean(dim=0)
        attributions = diff * grads
        pick = lambda lg: lg.gather(1, at_x.target[:, None])[:, 0]
        delta = attributions.sum(dim=(1, 2)) - (pick(at_x.logits) - pick(run.logits[:B]))
        return Attributions(at_x.logits, at_x.target, attributions, delta)

    # -- forward ---------------------------------------------------------------------------
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 3:
            raise ValueError(f"EEG_LSTM.forward expects x of shape [B,T,C], got {tuple(x.shape)}")
        ops._require_cuda(x)          # raises on CPU tensors: there is no CPU fallback
        if x.shape[2] != self.lstm.input_size:
            raise RuntimeError(f"input.size(-1) must be equal to input_size. Expected {self.lstm.input_size}, "
                               f"got {x.shape[2]}")
        B, T, _ = x.shape
        if B == 0:
            return x.new_zeros((0, self.fc[3].out_features))
        L = self.lstm.num_layers
        lstm_params = [self.lstm.layer(l) for l in range(L)]
        head = self._head_params()
        needs_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))
        if not self.training and not needs_grad:
            logits, _ = self.decode(x, want_probs=False)
        else:
            d1 = rr = d2 = None
            tier = self._tier(x, train=True)
            if tier in ("tc", "x3"):
                # flagship shape on the tensor cores: tcgen05 forward + fused BPTT; tc with bf16 operands (2e-2 contract),
                # x3 fp32-accurate (operands split into fp16 hi + lo)
                drop1 = None
                if self.training:
                    injected = (self._injected_noise or {}).get("drop1") is not None
                    d1, rr, d2 = self._draw_noise(B, T, x.device, ops.TC_TILE, torch.uint8, skip_drop1=not injected)
                    if injected:
                        drop1 = d1[0]
                    elif self.lstm.dropout > 0.0:
                        # no mask tensor: the kernels generate (and the backward re-generates) the keep-bits from
                        # a counter-based hash; the seed comes from torch's CPU generator (torch.manual_seed)
                        drop1 = (int(torch.randint(0, 2 ** 62, (1,)).item()), ops.drop1_thresh16(self.dropout_p))
                train_forward = ops.decoder_train_forward_tc if tier == "tc" else ops.decoder_train_forward_x3
                logits = train_forward(x, lstm_params, head, self.dropout_p, self.zscore_input, drop1, rr, d2)
            elif tier == "wide":
                # wide shapes (BASELINE configs[4]) on the 16-bit tier: streamed-weight recurrence kernels + cuBLAS for the
                # time-parallel GEMMs; dropout / RReLU noise as tensors (time-major padded to 128)
                drop1 = None
                if self.training:
                    d1, rr, d2 = self._draw_noise(B, T, x.device, ops.TC_TILE)
                    drop1 = d1[0] if d1 is not None else None
                logits = ops.decoder_train_forward_wide_tc(x, lstm_params, head, self.dropout_p, self.zscore_input, drop1, rr, d2)
            else:
                if self.training:
                    d1, rr, d2 = self._draw_noise(B, T, x.device)
                logits = ops.decoder_train_forward(x, lstm_params, head, self.dropout_p, self.zscore_input,
                                                   d1, rr, d2)
        return logits if logits.dtype == x.dtype or not x.is_floating_point() else logits.to(x.dtype)


def _resolve_preprocessor():
    """The MindsAI filter stays what it is in the reference (a vendored, separately licensed CPU
    numpy package -- SURVEY 8(f) "next" #1).  Import it from wherever the reference app put it."""
    errors = []
    for mod in ("Utilities.preprocessor", "preprocessor"):
        try:
            return __import__(mod, fromlist=["PreProcessor"]).PreProcessor
        except ImportError as e:           # pragma: no cover - depends on the host app
            errors.append(f"{mod}: {e}")
    raise ImportError("PreProcessor (MindsAI filter wrapper, reference Utilities/preprocessor.py) is not "
                      "importable; pass `preprocessor=` explicitly. Tried: " + "; ".join(errors))


class SimplePredictor:
    """Reference lstm_eeg_model.py:42-101: preprocess [T,C] -> [1,T,C] -> logits -> softmax ->
    ``(probs float32[K], label)``.

    ``device`` keeps the reference's argument but means the I/O device only (``run_trials``
    hard-codes ``"cpu"``, tester.py:83): numpy in, numpy out; the model itself always lives on
    the current CUDA device and the H2D / D2H copies are explicit (SURVEY F11).
    ``preprocessor`` (extra, optional): an object with ``transform([T,C]) -> [T,C]``; default is
    the reference's ``PreProcessor(sr, tailoring_lambda)``.
    """

    def __init__(self, pth_path: str, sr: int, channel_order=None, input_size: int = 8, hidden_size: int = 48,
                 num_layers: int = 2, num_classes: int = 3, dropout: float = 0.60, device: str = "cpu",
                 tailoring_lambda: float = 1.25e-29, class_names=None, preprocessor=None):
        self.device = torch.device(device)
        self.compute_device = ops.compute_device(self.device)
        self.class_names = class_names or CLASS_NAMES
        self.pre = preprocessor if preprocessor is not None else _resolve_preprocessor()(sr=sr, tailoring_lambda=tailoring_lambda)
        self.model = EEG_LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers,
                              num_classes=num_classes, dropout=dropout)
        state = torch.load(pth_path, map_location="cpu")
        if isinstance(state, dict) and "state_dict" in state:     # raw state_dict or {"state_dict": ...}
            state = state["state_dict"]
        self.model.load_state_dict(state, strict=True)
        self.model.to(self.compute_device).eval()
        self._no_grad = torch.inference_mode

    def predict(self, chunk_TxC: np.ndarray):
        """chunk_TxC: np.ndarray [T,C] -> (probs np.ndarray [K] float32, label str)."""
        x = self.pre.transform(chunk_TxC)
        x_t = torch.from_numpy(np.ascontiguousarray(x[None, ...])).float().to(self.compute_device)
        with self._no_grad():
            _, probs = self.model.decode(x_t, want_probs=True)
            probs = probs[0].detach().cpu().numpy().astype(np.float32)
        y_idx = int(np.argmax(probs))
        return probs, self.class_names[y_idx]

    def explain(self, chunk_TxC: np.ndarray):
        """``predict`` plus the attention weights over time: chunk [T,C] -> (probs float32[K], label, attention
        float32[T]), with the same preprocessing.  The attention curve shows which part of the window drove the
        decision (forward hooks on ``model.attn`` do not fire in this implementation; see
        ``EEG_LSTM.decode_intermediates``)."""
        x = self.pre.transform(chunk_TxC)
        x_t = torch.from_numpy(np.ascontiguousarray(x[None, ...])).float().to(self.compute_device)
        with self._no_grad():
            out = self.model.decode_intermediates(x_t)
            probs = out.probs[0].detach().cpu().numpy().astype(np.float32)
            attention = out.attention[0].detach().cpu().numpy().astype(np.float32)
        y_idx = int(np.argmax(probs))
        return probs, self.class_names[y_idx], attention

    def attribute(self, chunk_TxC: np.ndarray, steps: int = 32):
        """``predict`` plus integrated gradients of the predicted class (``EEG_LSTM.integrated_gradients``, zero
        baseline): chunk [T,C] -> (probs float32[K], label, attributions float32[T,C]).  Same preprocessing as
        ``predict``; the attributions are with respect to the preprocessed window."""
        x = self.pre.transform(chunk_TxC)
        x_t = torch.from_numpy(np.ascontiguousarray(x[None, ...])).float().to(self.compute_device)
        with self._no_grad():
            _, probs = self.model.decode(x_t, want_probs=True)
            probs = probs[0].detach().cpu().numpy().astype(np.float32)
        y_idx = int(np.argmax(probs))
        out = self.model.integrated_gradients(x_t, target=y_idx, steps=steps)
        return probs, self.class_names[y_idx], out.attributions[0].detach().cpu().numpy().astype(np.float32)

    def predict_batch(self, chunks_BxTxC: np.ndarray, preprocess: bool = True) -> np.ndarray:
        """Batched sibling of ``predict``: [B,T,C] -> probs [B,K] (one H2D, one launch sequence, one D2H)."""
        if preprocess and hasattr(self.pre, "transform_batch"):
            # a batched GPU front stage (preprocess_gpu.PhaseCouplingFilterGPU, opt-in): one H2D, filter + decode on the device
            x_t = torch.from_numpy(np.ascontiguousarray(chunks_BxTxC, dtype=np.float32)).to(self.compute_device)
            x_t = self.pre.transform_batch(x_t)
        else:
            x = np.stack([self.pre.transform(c) for c in chunks_BxTxC]) if preprocess else np.asarray(chunks_BxTxC)
            x_t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(self.compute_device)
        with self._no_grad():
            _, probs = self.model.decode(x_t, want_probs=True)
        return probs.cpu().numpy().astype(np.float32)
