"""Drop-in replacement of ``Neuro-Alpha-App/Utilities/lstm_eeg_model.py`` on B200.

Same public names (``CLASS_NAMES``, ``EEG_LSTM``, ``SimplePredictor``), same constructor
signatures and defaults, same 16-key ``state_dict`` layout, same ``forward(x) -> logits``
contract (reference lstm_eeg_model.py:11-101) -- but every arithmetic step runs in
hand-written sm_100a kernels (libneuroalpha_b200.so).  There is no CPU compute path:
``EEG_LSTM.forward`` on a CPU tensor raises.
"""
from __future__ import annotations

import math
from typing import Dict, List, NamedTuple, Optional

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


class LSTMParameters(nn.Module):
    """Parameter container with ``nn.LSTM``'s names, shapes, registration order and default init
    (U(-1/sqrt(H), 1/sqrt(H)) for every tensor, drawn in registration order), so that
    ``torch.manual_seed(s); EEG_LSTM()`` reproduces the reference's weights and the 16-key
    ``state_dict`` loads with ``strict=True`` (reference lstm_eeg_model.py:16-22, 81).
    It holds no compute: the recurrence is ``torch.ops.neuroalpha.lstm_layer_fwd``.
    """

    def __init__(self, input_size: int, hidden_size: int, num_layers: int, dropout: float):
        super().__init__()
        self.input_size, self.hidden_size, self.num_layers = input_size, hidden_size, num_layers
        self.dropout = float(dropout)
        self.batch_first = True
        self.bidirectional = False
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
        self._pack_cache: Dict[object, tuple] = {}

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
        key = tuple((p.data_ptr(), p._version, p.dtype) for p in ps)
        hit = self._pack_cache.get(slot)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                hit = (key, make())
            self._pack_cache[slot] = hit
        return hit[1]

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
        ps = self.lstm.layer(0) + self.lstm.layer(1)
        return self._cached_pack("x3", ps, lambda: ops.decoder_pack_x3(ps))

    def _packed_tc(self):
        ps = self.lstm.layer(0) + self.lstm.layer(1)
        return self._cached_pack("tc", ps, lambda: ops.decoder_pack_bf16(ps))

    def decode(self, x: torch.Tensor, want_probs: bool = True):
        """Eval-mode forward without autograd: x [B,T,C] on CUDA -> (logits fp32 [B,K], probs fp32 [B,K] or
        empty).  Picks the tier from ``compute_dtype`` / the dtype of ``x`` / the parameters."""
        ops._require_cuda(x)
        bf16 = (self.compute_dtype == torch.bfloat16 or x.dtype == torch.bfloat16
                or self.attn.weight.dtype == torch.bfloat16)
        with torch.no_grad():
            if bf16 and self.tc_supported():
                return ops.decoder_infer_tc(x, self._packed_tc(), self._head_params(), want_probs, self.zscore_input)
            if bf16 and self.tc_wide_supported():
                return ops.decoder_infer_wide(x, self._packed_tc_wide(), self._head_params(), self.lstm.hidden_size,
                                              want_probs, self.zscore_input)
            if (ops.EXACT_TC and not bf16 and self.tc_supported() and x.dtype == torch.float32 and x.shape[0] > 0):
                # exact tier, flagship shape: fp32-accurate tensor-core kernel (fp16 hi/lo operand split); the optional
                # z-score stage is one K1 pass that leaves the windows batch-first in fp32
                if self.zscore_input:
                    x = ops.window_zscore(x, x.shape[1], x.shape[1], True, False, ops.NA_F32)
                return ops.decoder_infer_x3(x.contiguous(), self._packed_x3(), self._head_params(), want_probs)
            L = self.lstm.num_layers
            return ops.decoder_infer(x, [self.lstm.layer(l) for l in range(L)],
                                     [ops._f32c(t) for t in self._head_params()], want_probs, self.zscore_input,
                                     [self._packed(l) for l in range(L)])

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
        bf16 = (self.compute_dtype == torch.bfloat16 or x.dtype == torch.bfloat16
                or self.attn.weight.dtype == torch.bfloat16)
        with torch.no_grad():
            if bf16 and self.tc_supported():
                return DecoderOutputs(*ops.decoder_infer_tc_intermediates(x, self._packed_tc(), self._head_params(),
                                                                          self.zscore_input))
            if bf16 and self.tc_wide_supported():
                return DecoderOutputs(*ops.decoder_infer_wide_intermediates(x, self._packed_tc_wide(), self._head_params(),
                                                                            self.lstm.hidden_size, self.zscore_input))
            if ops.EXACT_TC and not bf16 and self.tc_supported() and x.dtype == torch.float32:
                if self.zscore_input:
                    x = ops.window_zscore(x, x.shape[1], x.shape[1], True, False, ops.NA_F32)
                return DecoderOutputs(*ops.decoder_infer_x3_intermediates(x.contiguous(), self._packed_x3(),
                                                                          self._head_params()))
            L = self.lstm.num_layers
            return DecoderOutputs(*ops.decoder_infer_intermediates(
                x, [self.lstm.layer(l) for l in range(L)], [ops._f32c(t) for t in self._head_params()],
                self.zscore_input, [self._packed(l) for l in range(L)]))

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
            bf16 = (self.compute_dtype == torch.bfloat16 or x.dtype == torch.bfloat16
                    or self.attn.weight.dtype == torch.bfloat16)
            if bf16 and self.tc_supported() and not x.requires_grad:
                # tensor-core tier: tcgen05 forward + fused BPTT (bf16 operands, 2e-2 contract)
                drop1 = None
                if self.training:
                    injected = (self._injected_noise or {}).get("drop1") is not None
                    d1, rr, d2 = self._draw_noise(B, T, x.device, ops.TC_TILE, torch.uint8, skip_drop1=not injected)
                    if injected:
                        drop1 = d1[0]
                    elif self.lstm.dropout > 0.0:
                        # no mask tensor: the kernels generate (and the backward re-generates) the keep-bits from
                        # a counter-based hash; the seed comes from torch's CPU generator (torch.manual_seed)
                        drop1 = (int(torch.randint(0, 2 ** 62, (1,)).item()), int(round((1.0 - self.dropout_p) * 65536)))
                logits = ops.decoder_train_forward_tc(x, lstm_params, head, self.dropout_p, self.zscore_input,
                                                      drop1, rr, d2)
            elif bf16 and self.tc_wide_supported() and not x.requires_grad:
                # wide shapes (BASELINE configs[4]) on the 16-bit tier: streamed-weight recurrence kernels + cuBLAS for the
                # time-parallel GEMMs; dropout / RReLU noise as tensors (time-major padded to 128)
                drop1 = None
                if self.training:
                    d1, rr, d2 = self._draw_noise(B, T, x.device, ops.TC_TILE)
                    drop1 = d1[0] if d1 is not None else None
                logits = ops.decoder_train_forward_wide_tc(x, lstm_params, head, self.dropout_p, self.zscore_input, drop1, rr, d2)
            elif (ops.EXACT_TC_TRAIN and not bf16 and self.tc_supported() and not x.requires_grad
                  and x.dtype in (torch.float32, torch.float16, torch.bfloat16)):
                # exact tier, flagship shape: fp32-accurate tensor-core training (operands split into fp16 hi + lo)
                drop1 = None
                if self.training:
                    injected = (self._injected_noise or {}).get("drop1") is not None
                    d1, rr, d2 = self._draw_noise(B, T, x.device, ops.TC_TILE, torch.uint8, skip_drop1=not injected)
                    if injected:
                        drop1 = d1[0]
                    elif self.lstm.dropout > 0.0:
                        drop1 = (int(torch.randint(0, 2 ** 62, (1,)).item()), int(round((1.0 - self.dropout_p) * 65536)))
                logits = ops.decoder_train_forward_x3(x, lstm_params, head, self.dropout_p, self.zscore_input,
                                                      drop1, rr, d2)
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
