"""Torch-facing operators over the C ABI: ``torch.ops.neuroalpha.*`` custom ops (CUDA only) and
the explicit autograd function of the whole decoder.

PyTorch is plumbing here -- device memory, streams, autograd bookkeeping.  Every arithmetic
step of the hot path runs in libneuroalpha_b200.so.  Calling an op with a CPU tensor raises:
there is deliberately no CPU implementation.

Internal activation layout is "time-major padded" (TMP): ``[T, Bp, F]`` with ``Bp`` the batch
rounded up to a multiple of 32 (see include/neuroalpha.h).
"""
from __future__ import annotations

import functools
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib

BATCH_ALIGN = 32
FC_HIDDEN = 32
NA_F32, NA_BF16 = 0, 1

HEAD_KEYS = ("attn.weight", "attn.bias", "ln.weight", "ln.bias",
             "fc.0.weight", "fc.0.bias", "fc.3.weight", "fc.3.bias")


def padded_batch(b: int, align: int = BATCH_ALIGN) -> int:
    return max(align, (b + align - 1) // align * align)


def _require_cuda(*tensors: Optional[Tensor]) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "neural_speech_decoding_b200: tensor on %s -- the decoder runs only on CUDA (sm_100a); "
                "there is no CPU fallback" % t.device)


def compute_device(io_device: torch.device) -> torch.device:
    """Device the kernels run on for a caller that names ``io_device`` (reference callers pass
    "cpu", tester.py:83): the named CUDA device, else the current one.  Raises without a GPU."""
    if io_device.type == "cuda":
        return io_device
    if not torch.cuda.is_available():
        raise RuntimeError("neural_speech_decoding_b200: no CUDA device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _f32c(t: Tensor) -> Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _aligned16(t: Tensor) -> Tensor:
    """t, or a copy of it when its data is not 16-byte aligned (a view at an odd offset): the kernels load 16 bytes at a
    time and the C ABI rejects such pointers."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _ptr(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _first_cuda_device(args, kwargs) -> Optional[torch.device]:
    for a in list(args) + list(kwargs.values()):
        if isinstance(a, Tensor):
            if a.is_cuda:
                return a.device
        elif isinstance(a, (list, tuple)):
            for t in a:
                if isinstance(t, Tensor) and t.is_cuda:
                    return t.device
    return None


def _device_guard(fn):
    """Run an op body on the device of its (first CUDA) tensor argument: the launch stream, the scratch
    allocations and the kernel's device all follow the data, not torch's current device
    (``SimplePredictor(device="cuda:1")`` / ``model.to("cuda:1")`` while cuda:0 is current)."""
    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = _first_cuda_device(args, kwargs)
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


def all_custom_ops():
    return [window_zscore, pack_lstm_layer, lstm_layer_fwd, lstm_layer_bwd, lstm_layer_wgrad, head_fwd,
            head_bwd, trial_mean, decoder_pack_bf16, decoder_infer_bf16, lstm2_fwd_train_bf16, lstm_bwd_bf16,
            dropout_mask_u8, head_tail_fwd, head_tail_bwd, decoder_infer_bf16_x32, decoder_pack_x3, decoder_infer_x3,
            decoder_pack_wide_bf16, decoder_infer_wide_bf16, x3_split_input, lstm_fwd_train_x3, lstm_bwd_x3, lstm_wgrad_x3,
            lstm_wide_fwd_train, lstm_wide_bwd, head_fwd_ex, attention_softmax, decoder_infer_bf16_ex,
            decoder_infer_bf16_x32_ex, decoder_infer_x3_ex, decoder_infer_wide_bf16_ex, lstm_layer_fwd_hx, lstm_layer_bwd_hx,
            lstm_layer_wgrad_hx, decoder_lstm_x3]


def launch_count() -> int:
    return _lib.query("na_launch_count")


# ------------------------------------------------------------------------------------------
# custom ops (kernel granularity)
# ------------------------------------------------------------------------------------------
@torch.library.custom_op("neuroalpha::window_zscore", mutates_args=(), device_types="cuda")
@_device_guard
def window_zscore(x: Tensor, T: int, hop: int, normalize: bool, time_major: bool, out16: int,
                  pad_to: int = BATCH_ALIGN) -> Tensor:
    """K1.  x: [B,T,C] batch or [n_samples,C] stream (then windows start every ``hop`` samples).

    Returns the windows ([B,T,C], or TMP [T,Bp,C] when ``time_major``), z-scored per window and
    channel when ``normalize`` (Frontend/app.py:166-170)."""
    _require_cuda(x)
    x = _f32c(x)
    if x.dim() == 3:
        B, T_, C = x.shape
        if T_ != T:
            raise RuntimeError(f"window_zscore: x has T={T_}, expected {T}")
        hop = T
    elif x.dim() == 2:
        n, C = x.shape
        B = 0 if n < T else (n - T) // hop + 1
    else:
        raise RuntimeError("window_zscore: x must be [B,T,C] or [n_samples,C]")
    Bp = padded_batch(B, pad_to) if time_major else B
    dt = {0: torch.float32, 1: torch.bfloat16, 2: torch.float16}[int(out16)]    # NA_F32 / NA_BF16 / NA_F16
    y = torch.empty((T, Bp, C) if time_major else (B, T, C), dtype=dt, device=x.device)
    if y.numel():
        _lib.call("na_window_zscore", x.data_ptr(), y.data_ptr(), B, T, C, hop, int(normalize),
                  int(time_major), Bp, int(out16), _stream())
    return y


@window_zscore.register_fake
def _(x, T, hop, normalize, time_major, out16, pad_to=BATCH_ALIGN):
    if x.dim() == 3:
        B, C = x.shape[0], x.shape[2]
    else:
        n, C = x.shape
        B = 0 if n < T else (n - T) // hop + 1
    dt = {0: torch.float32, 1: torch.bfloat16, 2: torch.float16}[int(out16)]
    return x.new_empty((T, padded_batch(B, pad_to), C) if time_major else (B, T, C), dtype=dt)


@torch.library.custom_op("neuroalpha::pack_lstm_layer", mutates_args=(), device_types="cuda")
@_device_guard
def pack_lstm_layer(w_ih: Tensor, w_hh: Tensor, b_ih: Tensor, b_hh: Tensor) -> Tuple[Tensor, Tensor]:
    _require_cuda(w_ih, w_hh, b_ih, b_hh)
    w_ih, w_hh, b_ih, b_hh = map(_f32c, (w_ih, w_hh, b_ih, b_hh))
    G, K = w_ih.shape
    H = G // 4
    wt = torch.empty((K + H, G), dtype=torch.float32, device=w_ih.device)
    bias = torch.empty((G,), dtype=torch.float32, device=w_ih.device)
    _lib.call("na_pack_lstm_layer", w_ih.data_ptr(), w_hh.data_ptr(), b_ih.data_ptr(), b_hh.data_ptr(),
              wt.data_ptr(), bias.data_ptr(), K, H, _stream())
    return wt, bias


@pack_lstm_layer.register_fake
def _(w_ih, w_hh, b_ih, b_hh):
    G, K = w_ih.shape
    return w_ih.new_empty((K + G // 4, G)), w_ih.new_empty((G,))


@torch.library.custom_op("neuroalpha::lstm_layer_fwd", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_layer_fwd(inp: Tensor, wt: Tensor, bias: Tensor, drop_mask: Optional[Tensor], drop_scale: float,
                   save: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """K3 forward of one layer.  inp TMP [T,Bp,K] -> (h, c, gates, h_drop); c/gates are empty
    unless ``save``; h_drop is empty unless ``drop_mask`` is given."""
    _require_cuda(inp, wt, bias, drop_mask)
    T, Bp, K = inp.shape
    H = bias.numel() // 4
    dev = inp.device
    h = torch.empty((T, Bp, H), dtype=torch.float32, device=dev)
    c = torch.empty((T, Bp, H) if save else (0,), dtype=torch.float32, device=dev)
    gates = torch.empty((T, Bp, 4 * H) if save else (0,), dtype=torch.float32, device=dev)
    h_drop = torch.empty((T, Bp, H) if drop_mask is not None else (0,), dtype=torch.float32, device=dev)
    _lib.call("na_lstm_layer_fwd_f32", inp.data_ptr(), wt.data_ptr(), bias.data_ptr(), h.data_ptr(),
              _ptr(c) if save else None, _ptr(gates) if save else None, _ptr(drop_mask), float(drop_scale),
              _ptr(h_drop) if drop_mask is not None else None, T, Bp, K, H, _stream())
    return h, c, gates, h_drop


@lstm_layer_fwd.register_fake
def _(inp, wt, bias, drop_mask, drop_scale, save):
    T, Bp, K = inp.shape
    H = bias.numel() // 4
    e = inp.new_empty((0,))
    return (inp.new_empty((T, Bp, H)), inp.new_empty((T, Bp, H)) if save else e,
            inp.new_empty((T, Bp, 4 * H)) if save else inp.new_empty((0,)),
            inp.new_empty((T, Bp, H)) if drop_mask is not None else inp.new_empty((0,)))


@torch.library.custom_op("neuroalpha::lstm_layer_bwd", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_layer_bwd(dh: Tensor, gates: Tensor, c: Tensor, w_ih: Tensor, w_hh: Tensor,
                   in_drop_mask: Optional[Tensor], drop_scale: float, need_din: bool) -> Tuple[Tensor, Tensor]:
    """Fused BPTT of one layer: (dgates TMP [T,Bp,4H], din TMP [T,Bp,K] or empty)."""
    _require_cuda(dh, gates, c, w_ih, w_hh, in_drop_mask)
    T, Bp, H = dh.shape
    K = w_ih.shape[1]
    dgates = torch.empty((T, Bp, 4 * H), dtype=torch.float32, device=dh.device)
    din = torch.empty((T, Bp, K) if need_din else (0,), dtype=torch.float32, device=dh.device)
    _lib.call("na_lstm_layer_bwd_f32", dh.data_ptr(), gates.data_ptr(), c.data_ptr(), w_ih.data_ptr(),
              w_hh.data_ptr(), dgates.data_ptr(), _ptr(din) if need_din else None, _ptr(in_drop_mask),
              float(drop_scale), T, Bp, K, H, _stream())
    return dgates, din


@lstm_layer_bwd.register_fake
def _(dh, gates, c, w_ih, w_hh, in_drop_mask, drop_scale, need_din):
    T, Bp, H = dh.shape
    return dh.new_empty((T, Bp, 4 * H)), dh.new_empty((T, Bp, w_ih.shape[1]) if need_din else (0,))


@torch.library.custom_op("neuroalpha::lstm_layer_wgrad", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_layer_wgrad(dgates: Tensor, inp: Tensor, h: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """(dW_ih [4H,K], dW_hh [4H,H], db [4H]) from dgates -- deterministic two-stage reduction."""
    _require_cuda(dgates, inp, h)
    T, Bp, G = dgates.shape
    K, H = inp.shape[2], h.shape[2]
    dev = dgates.device
    dw_ih = torch.empty((G, K), dtype=torch.float32, device=dev)
    dw_hh = torch.empty((G, H), dtype=torch.float32, device=dev)
    db = torch.empty((G,), dtype=torch.float32, device=dev)
    partials = torch.empty((_lib.query("na_wgrad_partial_floats", K, H),), dtype=torch.float32, device=dev)
    _lib.call("na_lstm_layer_wgrad_f32", dgates.data_ptr(), inp.data_ptr(), h.data_ptr(), dw_ih.data_ptr(),
              dw_hh.data_ptr(), db.data_ptr(), partials.data_ptr(), T, Bp, K, H, _stream())
    return dw_ih, dw_hh, db


@lstm_layer_wgrad.register_fake
def _(dgates, inp, h):
    G = dgates.shape[2]
    return dgates.new_empty((G, inp.shape[2])), dgates.new_empty((G, h.shape[2])), dgates.new_empty((G,))


@torch.library.custom_op("neuroalpha::lstm_layer_fwd_hx", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_layer_fwd_hx(inp: Tensor, wt: Tensor, bias: Tensor, drop_mask: Optional[Tensor], drop_scale: float,
                      h0: Optional[Tensor], c0: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """lstm_layer_fwd with save=True, starting from the initial state h0 / c0 [Bp,H] (both or neither; None = zeros):
    (h, c, gates, h_drop or empty)."""
    _require_cuda(inp, wt, bias, drop_mask, h0, c0)
    T, Bp, K = inp.shape
    H = bias.numel() // 4
    dev = inp.device
    h = torch.empty((T, Bp, H), dtype=torch.float32, device=dev)
    c = torch.empty((T, Bp, H), dtype=torch.float32, device=dev)
    gates = torch.empty((T, Bp, 4 * H), dtype=torch.float32, device=dev)
    h_drop = torch.empty((T, Bp, H) if drop_mask is not None else (0,), dtype=torch.float32, device=dev)
    _lib.call("na_lstm_layer_fwd_f32_hx", inp.data_ptr(), wt.data_ptr(), bias.data_ptr(), h.data_ptr(), c.data_ptr(),
              gates.data_ptr(), _ptr(drop_mask), float(drop_scale), _ptr(h_drop) if drop_mask is not None else None,
              T, Bp, K, H, _ptr(h0), _ptr(c0), _stream())
    return h, c, gates, h_drop


@lstm_layer_fwd_hx.register_fake
def _(inp, wt, bias, drop_mask, drop_scale, h0, c0):
    T, Bp, K = inp.shape
    H = bias.numel() // 4
    return (inp.new_empty((T, Bp, H)), inp.new_empty((T, Bp, H)), inp.new_empty((T, Bp, 4 * H)),
            inp.new_empty((T, Bp, H)) if drop_mask is not None else inp.new_empty((0,)))


@torch.library.custom_op("neuroalpha::lstm_layer_bwd_hx", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_layer_bwd_hx(dh: Tensor, gates: Tensor, c: Tensor, w_ih: Tensor, w_hh: Tensor, in_drop_mask: Optional[Tensor],
                      drop_scale: float, need_din: bool, c0: Optional[Tensor], dh_last: Tensor, dc_last: Tensor,
                      need_dhx: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """lstm_layer_bwd of a layer that started from c0 [Bp,H] (None = zeros), with the gradients w.r.t. its final h / c
    (dh_last / dc_last [Bp,H]) added at the last step: (dgates, din or empty, dh0 [Bp,H], dc0 [Bp,H]; both empty unless
    ``need_dhx``)."""
    _require_cuda(dh, gates, c, w_ih, w_hh, in_drop_mask, c0, dh_last, dc_last)
    T, Bp, H = dh.shape
    K = w_ih.shape[1]
    dev = dh.device
    dgates = torch.empty((T, Bp, 4 * H), dtype=torch.float32, device=dev)
    din = torch.empty((T, Bp, K) if need_din else (0,), dtype=torch.float32, device=dev)
    dh0 = torch.empty((Bp, H) if need_dhx else (0,), dtype=torch.float32, device=dev)
    dc0 = torch.empty((Bp, H) if need_dhx else (0,), dtype=torch.float32, device=dev)
    _lib.call("na_lstm_layer_bwd_f32_hx", dh.data_ptr(), gates.data_ptr(), c.data_ptr(), w_ih.data_ptr(), w_hh.data_ptr(),
              dgates.data_ptr(), _ptr(din) if need_din else None, _ptr(in_drop_mask), float(drop_scale), T, Bp, K, H,
              _ptr(c0), dh_last.data_ptr(), dc_last.data_ptr(), _ptr(dh0) if need_dhx else None,
              _ptr(dc0) if need_dhx else None, _stream())
    return dgates, din, dh0, dc0


@lstm_layer_bwd_hx.register_fake
def _(dh, gates, c, w_ih, w_hh, in_drop_mask, drop_scale, need_din, c0, dh_last, dc_last, need_dhx):
    T, Bp, H = dh.shape
    st = (Bp, H) if need_dhx else (0,)
    return (dh.new_empty((T, Bp, 4 * H)), dh.new_empty((T, Bp, w_ih.shape[1]) if need_din else (0,)), dh.new_empty(st),
            dh.new_empty(st))


@torch.library.custom_op("neuroalpha::lstm_layer_wgrad_hx", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_layer_wgrad_hx(dgates: Tensor, inp: Tensor, h: Tensor, h0: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor]:
    """lstm_layer_wgrad of a layer that started from h0 [Bp,H] (None = zeros): dW_hh includes dgates_0^T h0."""
    _require_cuda(dgates, inp, h, h0)
    T, Bp, G = dgates.shape
    K, H = inp.shape[2], h.shape[2]
    dev = dgates.device
    dw_ih = torch.empty((G, K), dtype=torch.float32, device=dev)
    dw_hh = torch.empty((G, H), dtype=torch.float32, device=dev)
    db = torch.empty((G,), dtype=torch.float32, device=dev)
    partials = torch.empty((_lib.query("na_wgrad_partial_floats", K, H),), dtype=torch.float32, device=dev)
    _lib.call("na_lstm_layer_wgrad_f32_hx", dgates.data_ptr(), inp.data_ptr(), h.data_ptr(), dw_ih.data_ptr(),
              dw_hh.data_ptr(), db.data_ptr(), partials.data_ptr(), T, Bp, K, H, _ptr(h0), _stream())
    return dw_ih, dw_hh, db


@lstm_layer_wgrad_hx.register_fake
def _(dgates, inp, h, h0):
    G = dgates.shape[2]
    return dgates.new_empty((G, inp.shape[2])), dgates.new_empty((G, h.shape[2])), dgates.new_empty((G,))


@torch.library.custom_op("neuroalpha::head_fwd", mutates_args=(), device_types="cuda")
@_device_guard
def head_fwd(h: Tensor, B: int, params: Sequence[Tensor], rrelu_slope: Optional[Tensor],
             drop_mask: Optional[Tensor], drop_scale: float, want_probs: bool,
             save: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """K4.  h TMP [T,Bp,H]; params in HEAD_KEYS order -> (logits [B,NC], probs, stats, zpool)."""
    _require_cuda(h, rrelu_slope, drop_mask, *params)
    T, Bp, H = h.shape
    NC = params[6].shape[0]
    dev = h.device
    logits = torch.empty((B, NC), dtype=torch.float32, device=dev)
    probs = torch.empty((B, NC) if want_probs else (0,), dtype=torch.float32, device=dev)
    stats = torch.empty((B, 2) if save else (0,), dtype=torch.float32, device=dev)
    zpool = torch.empty((B, H) if save else (0,), dtype=torch.float32, device=dev)
    _lib.call("na_head_fwd_f32", h.data_ptr(), *[p.data_ptr() for p in params], _ptr(rrelu_slope),
              _ptr(drop_mask), float(drop_scale), logits.data_ptr(), _ptr(probs) if want_probs else None,
              _ptr(stats) if save else None, _ptr(zpool) if save else None, T, B, Bp, H, NC, _stream())
    return logits, probs, stats, zpool


@head_fwd.register_fake
def _(h, B, params, rrelu_slope, drop_mask, drop_scale, want_probs, save):
    NC, H = params[6].shape[0], h.shape[2]
    return (h.new_empty((B, NC)), h.new_empty((B, NC) if want_probs else (0,)),
            h.new_empty((B, 2) if save else (0,)), h.new_empty((B, H) if save else (0,)))


def _ex_fake(like: Tensor, B: int, T: int, H: int, NC: int):
    f = torch.float32
    return (like.new_empty((B, NC), dtype=f), like.new_empty((B, NC), dtype=f), like.new_empty((T, B), dtype=f),
            like.new_empty((B, H), dtype=f), like.new_empty((B, H), dtype=f))


def _infer_fake(like: Tensor, B: int, NC: int, want_probs: bool):
    f = torch.float32
    return like.new_empty((B, NC), dtype=f), like.new_empty((B, NC) if want_probs else (0,), dtype=f)


def _infer_outputs(B: int, NC: int, dev, want_probs: bool = True, ex: Optional[Tuple[int, int]] = None) -> List[Tensor]:
    """Outputs of an eval kernel: logits [B,NC] and probs [B,NC] (empty unless ``want_probs``), then with ``ex`` = (T, H)
    the intermediates of its *_ex entry point: scores (time-major [T,B]), pooled [B,H], embedding [B,H]."""
    shapes = [(B, NC), (B, NC) if want_probs else (0,)] + ([(ex[0], B), (B, ex[1]), (B, ex[1])] if ex is not None else [])
    return [torch.empty(s, dtype=torch.float32, device=dev) for s in shapes]


def _out_ptrs(out: Sequence[Tensor], want_probs: bool) -> List[Optional[int]]:
    return [out[0].data_ptr(), _ptr(out[1]) if want_probs else None] + [t.data_ptr() for t in out[2:]]


def _infer_x32(op: str, x: Tensor, packed: Tensor, head: Sequence[Tensor], want_probs: bool, ex: bool):
    """Body of the eval ops that read the batch-first fp32 windows x [B,T,8] (entry point ``na_<op>``)."""
    _require_cuda(x, packed, *head)
    B, T, C = x.shape
    if x.dtype != torch.float32 or C != 8 or not x.is_contiguous():
        raise RuntimeError(f"{op}: x must be contiguous fp32 [B, T, 8]")
    head = [_f32c(t) for t in head]
    NC = head[6].shape[0]
    out = _infer_outputs(B, NC, x.device, want_probs, (T, 48) if ex else None)
    _lib.call("na_" + op, x.data_ptr(), packed.data_ptr(), *[t.data_ptr() for t in head], *_out_ptrs(out, want_probs),
              T, B, NC, _stream())
    return tuple(out)


def _infer_tmp(op: str, x_tmp: Tensor, packed: Tensor, head: Sequence[Tensor], B: int, H: Optional[int], want_probs: bool,
               ex: bool):
    """Body of the eval ops that read the time-major fp16 windows x_tmp [T,Bp,8] (entry point ``na_<op>``).  ``H``: the
    wide kernel's hidden size (it also takes its workspace), None for the flagship kernel."""
    _require_cuda(x_tmp, packed, *head)
    T, Bp, C = x_tmp.shape
    if x_tmp.dtype != TC_VALUE_DTYPE or C != 8 or Bp % TC_TILE:
        raise RuntimeError(f"{op}: x_tmp must be fp16 [T, Bp % 128 == 0, 8] (the tier's value format)")
    head = [_f32c(t) for t in head]
    NC = head[-2].shape[0]                                       # fc.3.weight (the wide kernel takes no attention vector)
    out = _infer_outputs(B, NC, x_tmp.device, want_probs, (T, H or 48) if ex else None)
    state = [] if H is None else [_wide_state(H, x_tmp.device).data_ptr()]
    _lib.call("na_" + op, x_tmp.data_ptr(), packed.data_ptr(), *[t.data_ptr() for t in head], *state,
              *_out_ptrs(out, want_probs), T, B, Bp, *([] if H is None else [H]), NC, _stream())
    return tuple(out)


def _with_attention(out) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """(logits, probs, scores [T,B], pooled, embedding) of a *_ex op -> the same with the attention weights [B,T]."""
    lg, pr, sc, zp, emb = out
    return lg, pr, attention_softmax(sc), zp, emb


@torch.library.custom_op("neuroalpha::head_fwd_ex", mutates_args=(), device_types="cuda")
@_device_guard
def head_fwd_ex(h: Tensor, B: int, params: Sequence[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """K4 in eval mode with its intermediates.  h TMP [T,Bp,H] -> (logits [B,NC], probs [B,NC], scores [T,B] time-major,
    pooled [B,H] (before LayerNorm), embedding [B,H] (LayerNorm output))."""
    _require_cuda(h, *params)
    T, Bp, H = h.shape
    NC = params[6].shape[0]
    logits, probs, scores, pooled, emb = _infer_outputs(B, NC, h.device, ex=(T, H))
    _lib.call("na_head_fwd_f32_ex", h.data_ptr(), *[p.data_ptr() for p in params], None, None, 1.0, logits.data_ptr(),
              probs.data_ptr(), scores.data_ptr(), pooled.data_ptr(), emb.data_ptr(), None, None, T, B, Bp, H, NC, _stream())
    return logits, probs, scores, pooled, emb


@head_fwd_ex.register_fake
def _(h, B, params):
    return _ex_fake(h, B, h.shape[0], h.shape[2], params[6].shape[0])


@torch.library.custom_op("neuroalpha::attention_softmax", mutates_args=(), device_types="cuda")
@_device_guard
def attention_softmax(scores_tm: Tensor) -> Tensor:
    """Time-major attention scores [T,B] -> attention weights [B,T] (softmax over time per window, fp32)."""
    _require_cuda(scores_tm)
    T, B = scores_tm.shape
    attn = torch.empty((B, T), dtype=torch.float32, device=scores_tm.device)
    if attn.numel():
        _lib.call("na_attention_softmax_f32", _f32c(scores_tm).data_ptr(), attn.data_ptr(), T, B, _stream())
    return attn


@attention_softmax.register_fake
def _(scores_tm):
    return scores_tm.new_empty((scores_tm.shape[1], scores_tm.shape[0]), dtype=torch.float32)


@torch.library.custom_op("neuroalpha::head_bwd", mutates_args=(), device_types="cuda")
@_device_guard
def head_bwd(dlogits: Tensor, h: Tensor, stats: Tensor, zpool: Tensor, params: Sequence[Tensor],
             rrelu_slope: Optional[Tensor], drop_mask: Optional[Tensor], drop_scale: float) -> Tuple[Tensor, Tensor]:
    """Backward of K4: (dh TMP [T,Bp,H], dparams packed in HEAD_KEYS order)."""
    _require_cuda(dlogits, h, stats, zpool, rrelu_slope, drop_mask, *params)
    T, Bp, H = h.shape
    B, NC = dlogits.shape
    dev = h.device
    dlogits = _f32c(dlogits)
    dh = torch.empty((T, Bp, H), dtype=torch.float32, device=dev)
    dparams = torch.empty((_lib.query("na_head_param_floats", H, NC),), dtype=torch.float32, device=dev)
    partials = torch.empty((_lib.query("na_head_partial_floats", B, H, NC),), dtype=torch.float32, device=dev)
    _lib.call("na_head_bwd_f32", dlogits.data_ptr(), h.data_ptr(), stats.data_ptr(), zpool.data_ptr(),
              *[p.data_ptr() for p in params], _ptr(rrelu_slope), _ptr(drop_mask), float(drop_scale),
              dh.data_ptr(), dparams.data_ptr(), partials.data_ptr(), T, B, Bp, H, NC, _stream())
    return dh, dparams


@head_bwd.register_fake
def _(dlogits, h, stats, zpool, params, rrelu_slope, drop_mask, drop_scale):
    H, NC = h.shape[2], dlogits.shape[1]
    n = H + 1 + 2 * H + FC_HIDDEN * H + FC_HIDDEN + FC_HIDDEN * NC + NC
    return h.new_empty(h.shape), h.new_empty((n,))


@torch.library.custom_op("neuroalpha::trial_mean", mutates_args=(), device_types="cuda")
@_device_guard
def trial_mean(x: Tensor) -> Tensor:
    """K5.  x [R, ...] fp32 -> mean over the leading (trial) axis with run_trials' exact rounding
    (tester.py:54,89,97)."""
    _require_cuda(x)
    x = _f32c(x)
    R = x.shape[0]
    out = torch.empty(x.shape[1:], dtype=torch.float32, device=x.device)
    _lib.call("na_trial_mean_f32", x.data_ptr(), out.data_ptr(), R, out.numel(), _stream())
    return out


@trial_mean.register_fake
def _(x):
    return x.new_empty(x.shape[1:])


TC_TILE = 128      # windows per CTA tile of the tensor-core tier (UMMA M)
# 16-bit VALUE format of the tier (EEG samples, h, weights): IEEE fp16 -- bounded range, 3 more mantissa
# bits than bf16 at the same tensor throughput.  Gradient operands (d gates) are bf16 inside the kernels.
TC_VALUE_DTYPE = torch.float16
NA_F16 = 2


@torch.library.custom_op("neuroalpha::decoder_pack_bf16", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_pack_bf16(lstm_flat: Sequence[Tensor]) -> Tensor:
    """The 8 nn.LSTM tensors (layer 0 then layer 1) -> UMMA B operands of the tensor-core tier."""
    _require_cuda(*lstm_flat)
    ts = [_f32c(t) for t in lstm_flat]
    if len(ts) != 8 or tuple(ts[0].shape) != (192, 8) or tuple(ts[4].shape) != (192, 48):
        raise RuntimeError("decoder_pack_bf16: the tensor-core tier implements input_size=8, hidden_size=48, num_layers=2")
    packed = torch.empty((_lib.query("na_decoder_packed_bf16_bytes"),), dtype=torch.uint8, device=ts[0].device)
    _lib.call("na_decoder_pack_bf16", *[t.data_ptr() for t in ts], packed.data_ptr(), _stream())
    return packed


@decoder_pack_bf16.register_fake
def _(lstm_flat):
    return lstm_flat[0].new_empty((2 * 22 * 3072,), dtype=torch.uint8)


@torch.library.custom_op("neuroalpha::decoder_infer_bf16", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_bf16(x_tmp: Tensor, packed: Tensor, head: Sequence[Tensor], B: int,
                       want_probs: bool) -> Tuple[Tensor, Tensor]:
    """Whole decoder forward on tcgen05 (bf16 operands, fp32 accumulate).  x_tmp: TMP bf16 [T,Bp,8]
    with Bp a multiple of 128 (window_zscore(..., time_major=True, bf16=True, pad_to=128))."""
    return _infer_tmp("decoder_infer_bf16", x_tmp, packed, head, B, None, want_probs, False)


@decoder_infer_bf16.register_fake
def _(x_tmp, packed, head, B, want_probs):
    return _infer_fake(x_tmp, B, head[6].shape[0], want_probs)


@torch.library.custom_op("neuroalpha::decoder_infer_bf16_x32", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_bf16_x32(x: Tensor, packed: Tensor, head: Sequence[Tensor], want_probs: bool) -> Tuple[Tensor, Tensor]:
    """Whole decoder forward on tcgen05 straight from the batch-first fp32 windows x [B,T,8] (the fp32 -> fp16
    time-major pack is fused into the kernel's producer warp)."""
    return _infer_x32("decoder_infer_bf16_x32", x, packed, head, want_probs, False)


@decoder_infer_bf16_x32.register_fake
def _(x, packed, head, want_probs):
    return _infer_fake(x, x.shape[0], head[6].shape[0], want_probs)


@torch.library.custom_op("neuroalpha::decoder_infer_bf16_ex", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_bf16_ex(x_tmp: Tensor, packed: Tensor, head: Sequence[Tensor],
                          B: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_bf16 with its intermediates: (logits, probs, scores [T,B] time-major, pooled [B,48], embedding [B,48])."""
    return _infer_tmp("decoder_infer_bf16_ex", x_tmp, packed, head, B, None, True, True)


@decoder_infer_bf16_ex.register_fake
def _(x_tmp, packed, head, B):
    return _ex_fake(x_tmp, B, x_tmp.shape[0], 48, head[6].shape[0])


@torch.library.custom_op("neuroalpha::decoder_infer_bf16_x32_ex", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_bf16_x32_ex(x: Tensor, packed: Tensor, head: Sequence[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_bf16_x32 with its intermediates: (logits, probs, scores [T,B] time-major, pooled, embedding)."""
    return _infer_x32("decoder_infer_bf16_x32_ex", x, packed, head, True, True)


@decoder_infer_bf16_x32_ex.register_fake
def _(x, packed, head):
    return _ex_fake(x, x.shape[0], x.shape[1], 48, head[6].shape[0])


FUSED_INPUT = True          # decoder_infer_tc: read fp32 [B,T,8] directly (False: K1 pack + time-major kernel; A/B timing)


def _infer_tc(x: Tensor, packed: Tensor, head_params: Sequence[Tensor], want_probs: bool, zscore: bool, ex: bool):
    """decoder_infer_tc (``ex`` False) and decoder_infer_tc_intermediates (``ex`` True, the *_ex kernels)."""
    _require_cuda(x)
    B, T, C = x.shape
    head = list(head_params)
    if FUSED_INPUT and not zscore and x.dtype == torch.float32 and C == 8 and B > 0:
        x = x.contiguous()
        if ex:
            return _with_attention(decoder_infer_bf16_x32_ex(x, packed, head))
        return decoder_infer_bf16_x32(x, packed, head, want_probs)
    xt = window_zscore(x, T, T, zscore, True, NA_F16, TC_TILE)
    if ex:
        return _with_attention(decoder_infer_bf16_ex(xt, packed, head, B))
    return decoder_infer_bf16(xt, packed, head, B, want_probs)


def decoder_infer_tc(x: Tensor, packed: Tensor, head_params: Sequence[Tensor], want_probs: bool = False,
                     zscore: bool = False) -> Tuple[Tensor, Tensor]:
    """Eval forward on the tensor-core tier.  x [B,T,8] fp32 (or bf16) -> (logits fp32, probs or empty).
    fp32 contiguous input without the z-score stage goes straight into the kernel; otherwise K1 packs the windows
    time-major in fp16 first (one read of x, one half-size write)."""
    return _infer_tc(x, packed, head_params, want_probs, zscore, False)


def decoder_infer_tc_intermediates(x: Tensor, packed: Tensor, head_params: Sequence[Tensor],
                                   zscore: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_tc with the intermediates: (logits, probs, attention [B,T], pooled [B,48], embedding [B,48]).
    Same input handling as decoder_infer_tc; the attention weights come from the kernel's scores by attention_softmax."""
    return _infer_tc(x, packed, head_params, True, zscore, True)


EXACT_TC = True             # exact tier, flagship shape, eval: fp16-split tcgen05 kernel (False: the FFMA kernels; A/B timing)


@torch.library.custom_op("neuroalpha::decoder_pack_x3", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_pack_x3(lstm_flat: Sequence[Tensor]) -> Tensor:
    """The 8 nn.LSTM tensors (layer 0 then layer 1) -> fp16 hi / lo UMMA operands of the exact tensor-core kernel."""
    _require_cuda(*lstm_flat)
    ts = [_f32c(t) for t in lstm_flat]
    if len(ts) != 8 or tuple(ts[0].shape) != (192, 8) or tuple(ts[4].shape) != (192, 48):
        raise RuntimeError("decoder_pack_x3: implements input_size=8, hidden_size=48, num_layers=2")
    packed = torch.empty((_lib.query("na_decoder_packed_x3_bytes"),), dtype=torch.uint8, device=ts[0].device)
    _lib.call("na_decoder_pack_x3", *[t.data_ptr() for t in ts], packed.data_ptr(), _stream())
    return packed


@decoder_pack_x3.register_fake
def _(lstm_flat):
    return lstm_flat[0].new_empty((40 * 3072,), dtype=torch.uint8)


@torch.library.custom_op("neuroalpha::decoder_infer_x3", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_x3(x: Tensor, packed: Tensor, head: Sequence[Tensor], want_probs: bool) -> Tuple[Tensor, Tensor]:
    """Whole decoder forward at fp32 accuracy on tcgen05 (operands split into fp16 hi + lo, three MMAs per product),
    straight from the batch-first fp32 windows x [B,T,8]."""
    return _infer_x32("decoder_infer_x3", x, packed, head, want_probs, False)


@decoder_infer_x3.register_fake
def _(x, packed, head, want_probs):
    return _infer_fake(x, x.shape[0], head[6].shape[0], want_probs)


@torch.library.custom_op("neuroalpha::decoder_infer_x3_ex", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_x3_ex(x: Tensor, packed: Tensor, head: Sequence[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_x3 with its intermediates: (logits, probs, scores [T,B] time-major, pooled [B,48], embedding [B,48])."""
    return _infer_x32("decoder_infer_x3_ex", x, packed, head, True, True)


@decoder_infer_x3_ex.register_fake
def _(x, packed, head):
    return _ex_fake(x, x.shape[0], x.shape[1], 48, head[6].shape[0])


@torch.library.custom_op("neuroalpha::decoder_lstm_x3", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_lstm_x3(x: Tensor, packed: Tensor, h0: Optional[Tensor], c0: Optional[Tensor]) -> Tuple[Tensor, Tensor, Tensor]:
    """The two LSTM layers of decoder_infer_x3 alone (same kernel and arithmetic; no pooling, no head): x [B,T,8] fp32,
    optional initial state h0 / c0 [2,B,48] (both or neither) -> (out [B,T,48] = the last layer's h at every step,
    h_n [2,B,48], c_n [2,B,48]).  Accuracy: see na_decoder_lstm_x3 in include/neuroalpha.h.  Inputs whose data is not
    16-byte aligned (a contiguous view at an odd offset) are copied: the kernel reads them with 16-byte loads."""
    _require_cuda(x, packed, h0, c0)
    B, T, C = x.shape
    if x.dtype != torch.float32 or C != 8:
        raise RuntimeError("decoder_lstm_x3: x must be fp32 [B, T, 8]")
    if (h0 is None) != (c0 is None):
        raise RuntimeError("decoder_lstm_x3: h0 and c0 must be given together")
    x = _aligned16(x.contiguous())
    if h0 is not None:
        if tuple(h0.shape) != (2, B, 48) or tuple(c0.shape) != (2, B, 48):
            raise RuntimeError(f"decoder_lstm_x3: h0 / c0 must be [2, {B}, 48]")
        h0, c0 = _aligned16(_f32c(h0)), _aligned16(_f32c(c0))
    dev = x.device
    out = torch.empty((B, T, 48), dtype=torch.float32, device=dev)
    h_n = torch.empty((2, B, 48), dtype=torch.float32, device=dev)
    c_n = torch.empty((2, B, 48), dtype=torch.float32, device=dev)
    _lib.call("na_decoder_lstm_x3", x.data_ptr(), packed.data_ptr(), _ptr(h0), _ptr(c0), out.data_ptr(), h_n.data_ptr(),
              c_n.data_ptr(), T, B, _stream())
    return out, h_n, c_n


@decoder_lstm_x3.register_fake
def _(x, packed, h0, c0):
    B, T = x.shape[0], x.shape[1]
    f = torch.float32
    return x.new_empty((B, T, 48), dtype=f), x.new_empty((2, B, 48), dtype=f), x.new_empty((2, B, 48), dtype=f)


def decoder_infer_x3_intermediates(x: Tensor, packed: Tensor,
                                   head_params: Sequence[Tensor]) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_x3 with the intermediates: (logits, probs, attention [B,T], pooled [B,48], embedding [B,48])."""
    return _with_attention(decoder_infer_x3_ex(x, packed, list(head_params)))


WIDE_HIDDEN = (96, 144, 192)          # hidden sizes of the streamed-weight tensor-core kernel (na_decoder_wide.cu)


@torch.library.custom_op("neuroalpha::decoder_pack_wide_bf16", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_pack_wide_bf16(lstm_flat: Sequence[Tensor], attn_w: Tensor, attn_b: Tensor) -> Tensor:
    """The 8 nn.LSTM tensors + the attention vector of a wide decoder (H in WIDE_HIDDEN, input_size 8, 2 layers)
    -> the weight image the wide kernel streams every step (MMA consumption order) + its score operand."""
    _require_cuda(*lstm_flat, attn_w, attn_b)
    ts = [_f32c(t) for t in lstm_flat]
    H = ts[1].shape[1]
    if len(ts) != 8 or H not in WIDE_HIDDEN or tuple(ts[0].shape) != (4 * H, 8) or tuple(ts[4].shape) != (4 * H, H):
        raise RuntimeError("decoder_pack_wide_bf16: implements input_size=8, hidden_size in (96, 144, 192), num_layers=2")
    packed = torch.empty((_lib.query("na_decoder_wide_packed_bytes", H),), dtype=torch.uint8, device=ts[0].device)
    _lib.call("na_decoder_pack_wide_bf16", *[t.data_ptr() for t in ts], _f32c(attn_w).data_ptr(), _f32c(attn_b).data_ptr(),
              packed.data_ptr(), H, _stream())
    return packed


@decoder_pack_wide_bf16.register_fake
def _(lstm_flat, attn_w, attn_b):
    H = lstm_flat[1].shape[1]
    nch = H // 48
    return lstm_flat[0].new_empty((nch * (2 + 3 * (H // 16)) * 6144 + (1 + H // 16) * 512,), dtype=torch.uint8)


_WIDE_STATE: dict = {}


def _wide_state(H: int, device) -> Tensor:
    """Per-device L2-resident workspace of the wide kernel (cell state + pooling accumulators of every CTA).
    One buffer per (device, H, stream): launches on one stream are ordered, so it is re-used."""
    key = (device.index, H, _stream())
    buf = _WIDE_STATE.get(key)
    if buf is None:
        buf = torch.empty((_lib.query("na_decoder_wide_state_bytes", H),), dtype=torch.uint8, device=device)
        _WIDE_STATE[key] = buf
    return buf


@torch.library.custom_op("neuroalpha::decoder_infer_wide_bf16", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_wide_bf16(x_tmp: Tensor, packed: Tensor, head: Sequence[Tensor], B: int, H: int,
                            want_probs: bool) -> Tuple[Tensor, Tensor]:
    """Whole wide-decoder forward on tcgen05 with streamed weights.  x_tmp as for decoder_infer_bf16;
    head = [ln.w, ln.b, fc0.w, fc0.b, fc3.w, fc3.b] (the attention vector is part of `packed`)."""
    return _infer_tmp("decoder_infer_wide_bf16", x_tmp, packed, head, B, H, want_probs, False)


@decoder_infer_wide_bf16.register_fake
def _(x_tmp, packed, head, B, H, want_probs):
    return _infer_fake(x_tmp, B, head[4].shape[0], want_probs)


@torch.library.custom_op("neuroalpha::decoder_infer_wide_bf16_ex", mutates_args=(), device_types="cuda")
@_device_guard
def decoder_infer_wide_bf16_ex(x_tmp: Tensor, packed: Tensor, head: Sequence[Tensor], B: int,
                               H: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_wide_bf16 with its intermediates: (logits, probs, scores [T,B] time-major, pooled [B,H], embedding [B,H])."""
    return _infer_tmp("decoder_infer_wide_bf16_ex", x_tmp, packed, head, B, H, True, True)


@decoder_infer_wide_bf16_ex.register_fake
def _(x_tmp, packed, head, B, H):
    return _ex_fake(x_tmp, B, x_tmp.shape[0], H, head[4].shape[0])


def _infer_wide(x: Tensor, packed: Tensor, head_params: Sequence[Tensor], H: int, want_probs: bool, zscore: bool,
                ex: bool):
    """decoder_infer_wide (``ex`` False) and decoder_infer_wide_intermediates (``ex`` True, the *_ex kernel)."""
    _require_cuda(x)
    B, T, C = x.shape
    # (Fusing the input pack into the wide kernel, as in decoder_infer_tc, was built and measured: bit-identical but slower --
    # 59.1 vs 56.0 ms at H = 192, T = 2500 -- because the producer warp's weight stream is that kernel's critical path; and the
    # extra code cost the default path 7 % through the instruction cache, so it was removed again.)
    xt = window_zscore(x, T, T, zscore, True, NA_F16, TC_TILE)
    if ex:
        return _with_attention(decoder_infer_wide_bf16_ex(xt, packed, list(head_params[2:]), B, H))
    return decoder_infer_wide_bf16(xt, packed, list(head_params[2:]), B, H, want_probs)


def decoder_infer_wide(x: Tensor, packed: Tensor, head_params: Sequence[Tensor], H: int, want_probs: bool = False,
                       zscore: bool = False) -> Tuple[Tensor, Tensor]:
    """Eval forward of a wide decoder on the tensor-core tier.  head_params in EEG_LSTM._head_params() order."""
    return _infer_wide(x, packed, head_params, H, want_probs, zscore, False)


def decoder_infer_wide_intermediates(x: Tensor, packed: Tensor, head_params: Sequence[Tensor], H: int,
                                     zscore: bool = False) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer_wide with the intermediates: (logits, probs, attention [B,T], pooled [B,H], embedding [B,H])."""
    return _infer_wide(x, packed, head_params, H, True, zscore, True)


# ------------------------------------------------------------------------------------------
# decoder-level forward / explicit autograd
# ------------------------------------------------------------------------------------------
def split_head_grads(dparams: Tensor, H: int, NC: int) -> List[Tensor]:
    """Unpack na_head_bwd_f32's dparams into tensors shaped like HEAD_KEYS."""
    sizes = [H, 1, H, H, FC_HIDDEN * H, FC_HIDDEN, FC_HIDDEN * NC, NC]
    shapes = [(1, H), (1,), (H,), (H,), (FC_HIDDEN, H), (FC_HIDDEN,), (NC, FC_HIDDEN), (NC,)]
    return [p.reshape(s) for p, s in zip(dparams.split(sizes), shapes)]


def _infer_ffma(x: Tensor, lstm_params: Sequence[Sequence[Tensor]], head_params: Sequence[Tensor], want_probs: bool,
                zscore: bool, packed: Optional[Sequence[Tuple[Tensor, Tensor]]], ex: bool):
    """decoder_infer (``ex`` False) and decoder_infer_intermediates (``ex`` True: the same LSTM launches, head_fwd_ex)."""
    _require_cuda(x)
    B, T, C = x.shape
    cur = window_zscore(x, T, T, zscore, True, False)
    for l, (w_ih, w_hh, b_ih, b_hh) in enumerate(lstm_params):
        wt, bias = packed[l] if packed is not None else pack_lstm_layer(w_ih, w_hh, b_ih, b_hh)
        cur = lstm_layer_fwd(cur, wt, bias, None, 1.0, False)[0]
    if ex:
        return _with_attention(head_fwd_ex(cur, B, list(head_params)))
    logits, probs, _, _ = head_fwd(cur, B, list(head_params), None, None, 1.0, want_probs, False)
    return logits, probs


def decoder_infer(x: Tensor, lstm_params: Sequence[Sequence[Tensor]], head_params: Sequence[Tensor],
                  want_probs: bool = False, zscore: bool = False,
                  packed: Optional[Sequence[Tuple[Tensor, Tensor]]] = None) -> Tuple[Tensor, Tensor]:
    """Eval-mode forward, nothing saved.  x [B,T,C] -> (logits [B,NC], probs or empty)."""
    return _infer_ffma(x, lstm_params, head_params, want_probs, zscore, packed, False)


def decoder_infer_intermediates(x: Tensor, lstm_params: Sequence[Sequence[Tensor]], head_params: Sequence[Tensor],
                                zscore: bool = False, packed: Optional[Sequence[Tuple[Tensor, Tensor]]] = None
                                ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """decoder_infer with the intermediates of the head: (logits, probs, attention [B,T], pooled [B,H], embedding [B,H]).
    The LSTM layers are the same launches; the head kernel writes the scores, the pooled vector and the LayerNorm output."""
    return _infer_ffma(x, lstm_params, head_params, True, zscore, packed, True)


def _save(ctx, tensors: Sequence[Tensor], optional: Sequence[Optional[Tensor]]) -> None:
    """ctx.save_for_backward of ``tensors`` and of the ``optional`` ones that are not None; ``_saved`` restores both."""
    ctx.optional_given = [t is not None for t in optional]
    ctx.save_for_backward(*tensors, *[t for t in optional if t is not None])


def _saved(ctx) -> Tuple[List[Tensor], List[Optional[Tensor]]]:
    """(tensors, optional) as given to ``_save``, with None in place of each optional tensor that was not given."""
    sv = list(ctx.saved_tensors)
    n = len(sv) - sum(ctx.optional_given)
    given = iter(sv[n:])
    return sv[:n], [next(given) if g else None for g in ctx.optional_given]


def _cast_grads(grads: Sequence[Tensor], dtypes: Sequence[torch.dtype]) -> List[Tensor]:
    """Each gradient in the dtype of its parameter (the kernels produce fp32; .bfloat16() modules want bf16)."""
    return [g.to(dt) if g.dtype != dt else g for g, dt in zip(grads, dtypes)]


class DecoderFunction(torch.autograd.Function):
    """x, 4*L LSTM tensors, 8 head tensors -> logits, with the backward written out by hand
    (fused BPTT + time-parallel weight-gradient reductions).  Noise tensors are inputs, so the
    function itself is deterministic."""

    @staticmethod
    def forward(ctx, x, num_layers, p, zscore, drop1_masks, rrelu_slope, drop2_mask, *params):
        _require_cuda(x, *params)
        ctx.param_dtypes = [t.dtype for t in params]
        B, T, C = x.shape
        lstm_flat, head = params[:4 * num_layers], [_f32c(t) for t in params[4 * num_layers:]]
        scale = 1.0 / (1.0 - p) if p < 1.0 else 0.0
        cur = window_zscore(x.detach(), T, T, zscore, True, False)
        saved, layer_in = [], cur
        for l in range(num_layers):
            w_ih, w_hh, b_ih, b_hh = (_f32c(t.detach()) for t in lstm_flat[4 * l:4 * l + 4])
            wt, bias = pack_lstm_layer(w_ih, w_hh, b_ih, b_hh)
            mask = drop1_masks[l] if (drop1_masks is not None and l < num_layers - 1) else None
            h, c, gates, h_drop = lstm_layer_fwd(layer_in, wt, bias, mask, scale, True)
            saved += [layer_in, h, c, gates, w_ih, w_hh]
            layer_in = h_drop if mask is not None else h
        logits, _, stats, zpool = head_fwd(layer_in, B, head, rrelu_slope, drop2_mask, scale, False, True)
        _save(ctx, [*saved, stats, zpool, *head], [*(drop1_masks or ()), rrelu_slope, drop2_mask])
        ctx.meta = (num_layers, scale, B, x.shape, zscore)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        num_layers, scale, B, xshape, zscore = ctx.meta
        sv, (*d1, rr, d2) = _saved(ctx)
        layers = [sv[6 * l:6 * l + 6] for l in range(num_layers)]
        stats, zpool = sv[6 * num_layers:6 * num_layers + 2]
        head = sv[6 * num_layers + 2:]

        top_in = layers[-1][1]          # the head consumed the raw h of the last layer (dropout is never applied after it)
        H = top_in.shape[2]
        NC = dlogits.shape[1]
        dh, dparams = head_bwd(dlogits.contiguous(), top_in, stats, zpool, head, rr, d2, scale)
        head_grads = split_head_grads(dparams, H, NC)

        need_dx = ctx.needs_input_grad[0]
        lstm_grads: List[Tensor] = [None] * (4 * num_layers)
        dx = None
        for l in range(num_layers - 1, -1, -1):
            layer_in, h, c, gates, w_ih, w_hh = layers[l]
            in_mask = d1[l - 1] if (d1 and l > 0) else None
            need_din = l > 0 or need_dx
            dgates, din = lstm_layer_bwd(dh, gates, c, w_ih, w_hh, in_mask, scale, need_din)
            dw_ih, dw_hh, db = lstm_layer_wgrad(dgates, layer_in, h)
            lstm_grads[4 * l:4 * l + 4] = [dw_ih, dw_hh, db, db.clone()]
            dh = din
        if need_dx:
            if zscore:
                raise RuntimeError("gradient w.r.t. x through the z-score front stage is not implemented")
            dx = dh[:, :B].permute(1, 0, 2).contiguous().reshape(xshape)
        return (dx, None, None, None, None, None, None, *_cast_grads([*lstm_grads, *head_grads], ctx.param_dtypes))


class LSTMSequenceFunction(torch.autograd.Function):
    """x [B,T,K], initial state h0 / c0 [L,B,H] (both or neither; None = zeros), 4*L LSTM tensors ->
    (out [B,T,H], h_n [L,B,H], c_n [L,B,H]): nn.LSTM(batch_first=True) on the FFMA / generic kernels, with the backward
    written out by hand (fused BPTT + time-parallel weight-gradient reductions) in the style of DecoderFunction.
    ``drop_masks``: None, or L-1 keep-masks [B,T,H] of 0/1; layer l+1 then reads h_l * mask_l / (1 - p).  All outputs
    fp32."""

    @staticmethod
    def forward(ctx, x, h0, c0, p, drop_masks, *params):
        _require_cuda(x, h0, c0, *params)
        ctx.param_dtypes = [t.dtype for t in params]
        ctx.hx_dtypes = None if h0 is None else (h0.dtype, c0.dtype)
        L = len(params) // 4
        B, T, _ = x.shape
        H = params[1].shape[1]
        Bp = padded_batch(B)
        scale = 1.0 / (1.0 - p) if p < 1.0 else 0.0

        def rows(t, lead):                  # [..., B, H] -> zero-padded [..., Bp, H] fp32 (TMP rows)
            z = torch.zeros((*lead, Bp, H), dtype=torch.float32, device=x.device)
            z[..., :B, :] = t.detach()
            return z

        h0p = rows(h0, (L,)) if h0 is not None else None
        c0p = rows(c0, (L,)) if c0 is not None else None
        masks = [rows(m.permute(1, 0, 2), (T,)) for m in drop_masks] if drop_masks is not None else None
        saved, h_n, c_n = [], [], []
        layer_in = window_zscore(_aligned16(_f32c(x.detach())), T, T, False, True, False)     # TMP copy of x, fp32
        for l in range(L):
            w_ih, w_hh, b_ih, b_hh = (_f32c(t.detach()) for t in params[4 * l:4 * l + 4])
            wt, bias = pack_lstm_layer(w_ih, w_hh, b_ih, b_hh)
            mask = masks[l] if (masks is not None and l < L - 1) else None
            h, c, gates, h_drop = lstm_layer_fwd_hx(layer_in, wt, bias, mask, scale,
                                                    None if h0p is None else h0p[l], None if c0p is None else c0p[l])
            saved += [layer_in, h, c, gates, w_ih, w_hh]
            h_n.append(h[T - 1, :B])
            c_n.append(c[T - 1, :B])
            layer_in = h_drop if mask is not None else h
        _save(ctx, saved, [h0p, c0p, *(masks or ())])
        ctx.meta = (L, scale, B, tuple(x.shape))
        return h[:, :B].permute(1, 0, 2).contiguous(), torch.stack(h_n), torch.stack(c_n)

    @staticmethod
    def backward(ctx, dout, dh_n, dc_n):
        L, scale, B, xshape = ctx.meta
        sv, (h0p, c0p, *masks) = _saved(ctx)
        layers = [sv[6 * l:6 * l + 6] for l in range(L)]
        T, Bp, H = layers[-1][1].shape

        def rows(t):
            z = torch.zeros((Bp, H), dtype=torch.float32, device=t.device)
            z[:B] = t
            return z

        dh = torch.zeros((T, Bp, H), dtype=torch.float32, device=dout.device)
        dh[:, :B] = dout.permute(1, 0, 2)                    # the top layer's h is the output
        need_dx = ctx.needs_input_grad[0]
        need_dhx = h0p is not None and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2])
        lstm_grads: List[Tensor] = [None] * (4 * L)
        dh0, dc0 = [None] * L, [None] * L
        for l in range(L - 1, -1, -1):
            layer_in, h, c, gates, w_ih, w_hh = layers[l]
            in_mask = masks[l - 1] if (masks and l > 0) else None
            need_din = l > 0 or need_dx
            dgates, din, dh0[l], dc0[l] = lstm_layer_bwd_hx(
                dh, gates, c, w_ih, w_hh, in_mask, scale, need_din, None if c0p is None else c0p[l],
                rows(dh_n[l].float()), rows(dc_n[l].float()), need_dhx)
            dw_ih, dw_hh, db = lstm_layer_wgrad_hx(dgates, layer_in, h, None if h0p is None else h0p[l])
            lstm_grads[4 * l:4 * l + 4] = [dw_ih, dw_hh, db, db.clone()]
            dh = din
        dx = dh[:, :B].permute(1, 0, 2).contiguous().reshape(xshape) if need_dx else None
        dh0_out = dc0_out = None
        if need_dhx:
            dh0_out = torch.stack([g[:B] for g in dh0]).to(ctx.hx_dtypes[0])
            dc0_out = torch.stack([g[:B] for g in dc0]).to(ctx.hx_dtypes[1])
        return (dx, dh0_out, dc0_out, None, None, *_cast_grads(lstm_grads, ctx.param_dtypes))


def decoder_train_forward(x: Tensor, lstm_params, head_params, p: float, zscore: bool = False,
                          drop1_masks=None, rrelu_slope=None, drop2_mask=None) -> Tensor:
    flat = [t for layer in lstm_params for t in layer]
    return DecoderFunction.apply(x, len(lstm_params), p, zscore, drop1_masks, rrelu_slope, drop2_mask,
                                 *flat, *head_params)


# ------------------------------------------------------------------------------------------
# tensor-core tier, training
# ------------------------------------------------------------------------------------------
@torch.library.custom_op("neuroalpha::lstm2_fwd_train_bf16", mutates_args=(), device_types="cuda")
@_device_guard
def lstm2_fwd_train_bf16(x_tmp: Tensor, packed: Tensor, mask: Optional[Tensor], seed: int, thresh16: int,
                         drop_scale: float, attn_w: Tensor, attn_b: Tensor,
                         B: int, half_stride: int = 0) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Training forward of the 2-layer LSTM on tcgen05 with the attention pool fused.  x_tmp fp16 TMP
    [T,Bp,8] (Bp % 128 == 0).  Inter-layer dropout: explicit ``mask`` u8 [T,Bp,48], or (mask None, thresh16 <
    65536) the in-kernel counter-based generator keyed by ``seed``, or none (thresh16 = 65536).
    -> (h0 TCL, h0d TCL or empty, c0 TCL32, h1 TCL, c1 TCL32, zpool [B,48], stats [B,2])."""
    _require_cuda(x_tmp, packed, mask, attn_w, attn_b)
    T, Bp, _ = x_tmp.shape
    dev = x_tmp.device
    has_drop = mask is not None or thresh16 < 65536
    tcl = lambda: torch.empty((T, Bp // TC_TILE, 6, TC_TILE, 8), dtype=TC_VALUE_DTYPE, device=dev)
    tcl32 = lambda: torch.empty((T, Bp // TC_TILE, 12, TC_TILE, 4), dtype=torch.float32, device=dev)
    h0, h1, c0, c1 = tcl(), tcl(), tcl32(), tcl32()
    h0d = tcl() if has_drop else torch.empty((0,), dtype=TC_VALUE_DTYPE, device=dev)
    zpool = torch.empty((B, 48), dtype=torch.float32, device=dev)
    stats = torch.empty((B, 2), dtype=torch.float32, device=dev)
    aw, ab = _f32c(attn_w), _f32c(attn_b)
    _lib.call("na_lstm2_fwd_train_bf16", x_tmp.data_ptr(), packed.data_ptr(), _ptr(mask), int(seed), int(thresh16),
              float(drop_scale), h0.data_ptr(), _ptr(h0d) if has_drop else None, c0.data_ptr(), h1.data_ptr(), None,
              c1.data_ptr(), aw.data_ptr(), ab.data_ptr(), zpool.data_ptr(), stats.data_ptr(), B, T, Bp, int(half_stride), _stream())
    return h0, h0d, c0, h1, c1, zpool, stats


@lstm2_fwd_train_bf16.register_fake
def _(x_tmp, packed, mask, seed, thresh16, drop_scale, attn_w, attn_b, B, half_stride=0):
    T, Bp, _ = x_tmp.shape
    tcl = lambda: x_tmp.new_empty((T, Bp // TC_TILE, 6, TC_TILE, 8))
    tcl32 = lambda: x_tmp.new_empty((T, Bp // TC_TILE, 12, TC_TILE, 4), dtype=torch.float32)
    has_drop = mask is not None or thresh16 < 65536
    return (tcl(), (tcl() if has_drop else x_tmp.new_empty((0,))), tcl32(), tcl(), tcl32(),
            x_tmp.new_empty((B, 48), dtype=torch.float32), x_tmp.new_empty((B, 2), dtype=torch.float32))


@torch.library.custom_op("neuroalpha::head_tail_fwd", mutates_args=(), device_types="cuda")
@_device_guard
def head_tail_fwd(zpool: Tensor, params: Sequence[Tensor], rrelu_slope: Optional[Tensor], drop_mask: Optional[Tensor],
                  drop_scale: float, want_probs: bool) -> Tuple[Tensor, Tensor]:
    """LayerNorm -> fc0 -> RReLU -> dropout -> fc3 (+softmax) on an already pooled z [B,H] (lstm_eeg_model.py:38-39)."""
    _require_cuda(zpool, rrelu_slope, drop_mask, *params)
    B, H = zpool.shape
    NC = params[6].shape[0]
    logits = torch.empty((B, NC), dtype=torch.float32, device=zpool.device)
    probs = torch.empty((B, NC) if want_probs else (0,), dtype=torch.float32, device=zpool.device)
    _lib.call("na_head_tail_fwd_f32", zpool.data_ptr(), *[p.data_ptr() for p in params], _ptr(rrelu_slope),
              _ptr(drop_mask), float(drop_scale), logits.data_ptr(), _ptr(probs) if want_probs else None, B, H, NC,
              _stream())
    return logits, probs


@head_tail_fwd.register_fake
def _(zpool, params, rrelu_slope, drop_mask, drop_scale, want_probs):
    B, NC = zpool.shape[0], params[6].shape[0]
    return zpool.new_empty((B, NC)), zpool.new_empty((B, NC) if want_probs else (0,))


@torch.library.custom_op("neuroalpha::head_tail_bwd", mutates_args=(), device_types="cuda")
@_device_guard
def head_tail_bwd(dlogits: Tensor, zpool: Tensor, params: Sequence[Tensor], rrelu_slope: Optional[Tensor],
                  drop_mask: Optional[Tensor], drop_scale: float) -> Tuple[Tensor, Tensor]:
    """Backward of head_tail_fwd: (dz [B,H], dparams packed like head_bwd with the attn slots zeroed)."""
    _require_cuda(dlogits, zpool, rrelu_slope, drop_mask, *params)
    B, H = zpool.shape
    NC = dlogits.shape[1]
    dev = zpool.device
    dlogits = _f32c(dlogits)
    dz = torch.empty((B, H), dtype=torch.float32, device=dev)
    dparams = torch.empty((_lib.query("na_head_param_floats", H, NC),), dtype=torch.float32, device=dev)
    partials = torch.empty((_lib.query("na_head_partial_floats", B, H, NC),), dtype=torch.float32, device=dev)
    _lib.call("na_head_tail_bwd_f32", dlogits.data_ptr(), zpool.data_ptr(), *[p.data_ptr() for p in params],
              _ptr(rrelu_slope), _ptr(drop_mask), float(drop_scale), dz.data_ptr(), dparams.data_ptr(),
              partials.data_ptr(), B, H, NC, _stream())
    return dz, dparams


@head_tail_bwd.register_fake
def _(dlogits, zpool, params, rrelu_slope, drop_mask, drop_scale):
    H, NC = zpool.shape[1], dlogits.shape[1]
    n = H + 1 + 2 * H + FC_HIDDEN * H + FC_HIDDEN + FC_HIDDEN * NC + NC
    return zpool.new_empty(zpool.shape), zpool.new_empty((n,))


@torch.library.custom_op("neuroalpha::dropout_mask_u8", mutates_args=(), device_types="cuda")
@_device_guard
def dropout_mask_u8(like: Tensor, seed: int, thresh16: int, T: int, Bp: int) -> Tensor:
    """The keep-mask the in-kernel generator produces for (seed, thresh16): u8 [T,Bp,48] on like.device."""
    _require_cuda(like)
    out = torch.empty((T, Bp, 48), dtype=torch.uint8, device=like.device)
    _lib.call("na_dropout_mask_u8", int(seed), int(thresh16), T, Bp, out.data_ptr(), _stream())
    return out


@dropout_mask_u8.register_fake
def _(like, seed, thresh16, T, Bp):
    return like.new_empty((T, Bp, 48), dtype=torch.uint8)


@torch.library.custom_op("neuroalpha::lstm_bwd_bf16", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_bwd_bf16(layer: int, act_in: Tensor, h: Tensor, c: Tensor, dh: Optional[Tensor], packed: Tensor, w_ih: Tensor,
                  w_hh: Tensor, in_mask: Optional[Tensor], seed: int, thresh16: int, drop_scale: float,
                  head: Sequence[Tensor], B: int, half_stride: int = 0) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Fused BPTT + weight gradients of one layer on tcgen05 -> (din TCL32 or empty, dW_ih, dW_hh, db, d_attn).
    ``head`` = [] (dh given) or [dz, stats, zpool, attn_w, attn_b] for layer 1 with the head backward fused:
    dh_t is rebuilt per step inside the kernel and d_attn [49] = (d attn_w | d attn_b) is returned."""
    _require_cuda(act_in, h, c, dh, packed, w_ih, w_hh, in_mask, *head)
    T, NT = c.shape[0], c.shape[1]
    Bp, H = NT * TC_TILE, 48
    dev = c.device
    w_ih, w_hh = _f32c(w_ih), _f32c(w_hh)
    din = torch.empty((T, NT, 12, TC_TILE, 4) if layer == 1 else (0,), dtype=torch.float32, device=dev)
    dw_ih, dw_hh = torch.empty_like(w_ih), torch.empty_like(w_hh)
    db = torch.empty((4 * H,), dtype=torch.float32, device=dev)
    fused = len(head) > 0
    d_attn = torch.empty((H + 1,) if fused else (0,), dtype=torch.float32, device=dev)
    hp = [_f32c(t) for t in head]
    zeros, scratch = _train_buffers(dev, "bf16", 12288, 36864 + 4 * _lib.query("na_train_bf16_partial_floats"))
    _lib.call("na_lstm_bwd_bf16", int(layer), act_in.data_ptr(), h.data_ptr(), c.data_ptr(),
              None if fused else _f32c(dh).data_ptr(), packed.data_ptr(), w_ih.data_ptr(), w_hh.data_ptr(),
              zeros.data_ptr(), _ptr(in_mask), int(seed), int(thresh16), float(drop_scale),
              _ptr(din) if layer == 1 else None, dw_ih.data_ptr(), dw_hh.data_ptr(), db.data_ptr(), scratch.data_ptr(),
              *([t.data_ptr() for t in hp] if fused else [None] * 5), int(B), _ptr(d_attn) if fused else None,
              T, Bp, int(half_stride), _stream())
    return din, dw_ih, dw_hh, db, d_attn


@lstm_bwd_bf16.register_fake
def _(layer, act_in, h, c, dh, packed, w_ih, w_hh, in_mask, seed, thresh16, drop_scale, head, B, half_stride=0):
    return (c.new_empty(c.shape if layer == 1 else (0,)), w_ih.new_empty(w_ih.shape, dtype=torch.float32),
            w_hh.new_empty(w_hh.shape, dtype=torch.float32), c.new_empty((192,)),
            c.new_empty((49,) if len(head) else (0,)))


def _scale_dz(dz: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """Gradient scaling of the tensor-core BPTT kernels: d(gates) cross the tensor pipe as fp16 (hi + lo pairs in the exact
    tier), so the gradient entering the recurrence -- dz, AFTER the LayerNorm backward, whose 1/sigma can amplify the
    logit gradient by orders of magnitude -- is scaled by an exact power of two that puts max|dz| at 2^6: a factor 2^10
    of headroom below fp16's 65,504 for the growth through din = dG.W and the recurrence, while values 2^-20 of the
    maximum still sit in fp16's normal range.  Everything downstream is linear in dz, so every LSTM / attention
    gradient is unscaled by the same power at the end.  All on the device, no host sync."""
    amax = dz.detach().abs().max().clamp_min(1e-30)
    s = torch.pow(2.0, 6.0 - torch.ceil(torch.log2(amax)))          # (torch.exp2 would JIT-compile via nvrtc)
    return dz * s, s, 1.0 / s


_TRAIN_BUFFERS: dict = {}


def _train_buffers(device, tag: str, zero_bytes: int, scratch_bytes: int):
    """Per (device, stream) zero block and scratch area of the training kernels (they used to be allocated -- and the zeros
    memset -- on every call).  Launches on one stream are ordered, so consecutive kernels may share the scratch."""
    key = (device.index, tag, _stream())
    hit = _TRAIN_BUFFERS.get(key)
    if hit is None or hit[1].numel() < scratch_bytes:
        hit = (torch.zeros((zero_bytes,), dtype=torch.uint8, device=device), torch.empty((scratch_bytes,), dtype=torch.uint8, device=device))
        _TRAIN_BUFFERS[key] = hit
    return hit


TC_HALF_TILES = True          # 16-bit training tier: half tiles for batches that leave more than half of the SMs idle (A/B knob)
_SM_COUNT: dict = {}


def _sm_count(device) -> int:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _SM_COUNT:
        _SM_COUNT[idx] = torch.cuda.get_device_properties(idx).multi_processor_count
    return _SM_COUNT[idx]


def _drop1_args(drop1, scale: float) -> Tuple[Optional[Tensor], int, int, float]:
    """``drop1`` of DecoderFunctionTC / X3 -> (mask, seed, thresh16, scale1) of the layer-0 training kernels: None (no
    inter-layer dropout), a u8 keep-mask (scaled like the head dropout), or ``(seed, thresh16)`` of the in-kernel
    counter-based generator."""
    if isinstance(drop1, tuple):
        seed, thresh16 = int(drop1[0]), int(drop1[1])
        return None, seed, thresh16, 65536.0 / thresh16 if thresh16 > 0 else 0.0   # exactly unbiased for the quantised keep-rate
    if drop1 is not None:
        return drop1, 0, 65536, scale
    return None, 0, 65536, 1.0


def _half_stride(B: int, device, half_tiles: bool) -> int:
    """``half_stride`` of the flagship training kernels: 0 for full tiles, else the padded batch for half tiles (64 windows
    per 128-row tile, the two row copies split the hidden units).  Half tiles are used (when ``half_tiles``, the tier's
    TC_HALF_TILES / X3_HALF_TILES) if the batch would leave more than half of the SMs without a tile: a tile then costs
    about half a step (strong scaling at small batches)."""
    half = half_tiles and 2 * ((B + TC_TILE - 1) // TC_TILE) <= _sm_count(device)
    return padded_batch(B, TC_TILE) if half else 0


def _half_tile_rows(mask: Tensor, B: int, Bp: int) -> Tensor:
    """A time-major keep-mask [T, >= B, 48] in the half-tile row layout [T, Bp, 48]: window b -> row (b // 64) * 128 + b % 64."""
    b_idx = torch.arange(B, device=mask.device)
    remapped = mask.new_zeros((mask.shape[0], Bp, mask.shape[2]))
    remapped[:, (b_idx // 64) * TC_TILE + b_idx % 64] = mask[:, :B]
    return remapped


def _tc_backward(ctx, dlogits: Tensor, zpool: Tensor, head: Sequence[Tensor], rr: Optional[Tensor], d2: Optional[Tensor],
                 scale: float, layers_bwd):
    """Backward of DecoderFunctionTC / X3 around the tier's two layer backwards.  The head tail backward (fp32, unscaled)
    gives dz, which _scale_dz scales; ``layers_bwd(dz)`` runs layer 1 (with the time loop of the head backward -- dh_t,
    d attn -- fused) and layer 0 and returns the scaled (dW_ih0, dW_hh0, db0, dW_ih1, dW_hh1, db1, d_attn)."""
    H, NC = 48, dlogits.shape[1]
    dz, dparams = head_tail_bwd(dlogits.contiguous(), zpool, head, rr, d2, scale)
    dz, _, inv_s = _scale_dz(dz)
    dw_ih0, dw_hh0, db0, dw_ih1, dw_hh1, db1, d_attn = layers_bwd(dz)
    torch._foreach_mul_([dw_ih0, dw_hh0, db0, dw_ih1, dw_hh1, db1, d_attn], inv_s)      # ONE launch unscales every scaled gradient
    head_grads = split_head_grads(torch.cat([d_attn, dparams[H + 1:]]), H, NC)
    grads = [dw_ih0, dw_hh0, db0, db0.clone(), dw_ih1, dw_hh1, db1, db1.clone(), *head_grads]
    return (None, None, None, None, None, None, *_cast_grads(grads, ctx.param_dtypes))


class DecoderFunctionTC(torch.autograd.Function):
    """Training step of the flagship decoder on the tensor-core tier: tcgen05 forward that saves h / c,
    fp32 head kernels, tcgen05 BPTT with the weight gradients accumulated in TMEM.  bf16 contract
    (logits and gradients within 2e-2 of the fp32 reference)."""

    @staticmethod
    def forward(ctx, x, p, zscore, drop1, rrelu_slope, drop2_mask, *params):
        """``drop1``: None (no inter-layer dropout), a u8 keep-mask [T,Bp,48], or ``(seed, thresh16)`` for the
        in-kernel counter-based generator (no mask tensor at all)."""
        _require_cuda(x, *params)
        ctx.param_dtypes = [t.dtype for t in params]
        if ctx.needs_input_grad[0]:
            raise RuntimeError("the tensor-core training tier does not produce d/dx; use compute_dtype=float32")
        B, T, C = x.shape
        lstm_flat, head = [t.detach() for t in params[:8]], [_f32c(t.detach()) for t in params[8:]]
        scale = 1.0 / (1.0 - p) if p < 1.0 else 0.0          # head dropout (and mask-tensor mode)
        mask, seed, thresh16, scale1 = _drop1_args(drop1, scale)
        half_stride = _half_stride(B, x.device, TC_HALF_TILES)
        xin = x.detach()
        if half_stride:
            nt = (B + 63) // 64
            if nt * 64 != B:
                xin = torch.cat([xin, xin.new_zeros((nt * 64 - B, T, C))])
            if mask is not None:
                mask = _half_tile_rows(mask, B, nt * TC_TILE)
            # pack first (fp16, time-major, 64 windows per tile), then mirror: rows 64..127 of every tile repeat rows 0..63 -- on
            # the 16-byte packed rows this copies a quarter of the bytes that mirroring the fp32 windows did
            xt = window_zscore(xin, T, T, zscore, True, NA_F16, 64)
            xt = xt.reshape(T, nt, 64, C)
            xt = torch.stack((xt, xt), dim=2).reshape(T, nt * TC_TILE, C)       # (the batched cat kernel: 1 KB contiguous runs)
        else:
            xt = window_zscore(xin, T, T, zscore, True, NA_F16, TC_TILE)
        packed = decoder_pack_bf16(lstm_flat)
        h0, h0d, c0, h1, c1, zpool, stats = lstm2_fwd_train_bf16(xt, packed, mask, seed, thresh16, scale1, head[0], head[1], B, half_stride)
        logits, _ = head_tail_fwd(zpool, head, rrelu_slope, drop2_mask, scale, False)
        w = [_f32c(t) for t in lstm_flat]
        _save(ctx, [xt, h0, h0d, c0, h1, c1, packed, stats, zpool, w[0], w[1], w[4], w[5], *head],
              [mask, rrelu_slope, drop2_mask])
        ctx.meta = (scale, B, seed, thresh16, scale1, half_stride)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        scale, B, seed, thresh16, scale1, half_stride = ctx.meta
        sv, (d1, rr, d2) = _saved(ctx)
        xt, h0, h0d, c0, h1, c1, packed, stats, zpool, w_ih0, w_hh0, w_ih1, w_hh1 = sv[:13]
        head = sv[13:]
        in1 = h0d if d1 is not None or thresh16 < 65536 else h0

        def layers_bwd(dz):
            din1, dw_ih1, dw_hh1, db1, d_attn = lstm_bwd_bf16(1, in1, h1, c1, None, packed, w_ih1, w_hh1, d1, seed, thresh16,
                                                              scale1, [dz, stats, zpool, head[0], head[1]], B, half_stride)
            _, dw_ih0, dw_hh0, db0, _ = lstm_bwd_bf16(0, xt, h0, c0, din1, packed, w_ih0, w_hh0, None, 0, 65536, 1.0, [], B,
                                                      half_stride)
            return dw_ih0, dw_hh0, db0, dw_ih1, dw_hh1, db1, d_attn
        return _tc_backward(ctx, dlogits, zpool, head, rr, d2, scale, layers_bwd)


def decoder_train_forward_tc(x: Tensor, lstm_params, head_params, p: float, zscore: bool = False,
                             drop1=None, rrelu_slope=None, drop2_mask=None) -> Tensor:
    flat = [t for layer in lstm_params for t in layer]
    return DecoderFunctionTC.apply(x, p, zscore, drop1, rrelu_slope, drop2_mask, *flat, *head_params)


# ------------------------------------------------------------------------------------------
# exact tier (fp32 contract), training on the tensor cores (csrc/na_train_x3.cu)
# ------------------------------------------------------------------------------------------
EXACT_TC_TRAIN = True        # flagship shape, no d/dx wanted: operand-split tcgen05 kernels (False: FFMA / generic kernels; A/B)
X3_HALF_TILES = True         # half tiles for the exact training tier when a batch fills less than half of the SMs (A/B knob)


def _tclx(T: int, Bp: int, dev) -> Tensor:
    return torch.empty((T, Bp // TC_TILE, 12, TC_TILE, 8), dtype=torch.float16, device=dev)


def _tcl32(T: int, Bp: int, dev) -> Tensor:
    return torch.empty((T, Bp // TC_TILE, 12, TC_TILE, 4), dtype=torch.float32, device=dev)


@torch.library.custom_op("neuroalpha::x3_split_input", mutates_args=(), device_types="cuda")
@_device_guard
def x3_split_input(x: Tensor, Bp: int, half_stride: int = 0) -> Tensor:
    """fp32 windows [B,T,8] -> XS fp16 [T, Bp/128, 2, 128, 8]: x / 16 split into hi and lo halves (padding rows zero).
    ``half_stride`` > 0: half tiles (window b in rows (b // 64) * 128 + b % 64 and + 64)."""
    _require_cuda(x)
    B, T, C = x.shape
    if x.dtype != torch.float32 or C != 8 or not x.is_contiguous() or Bp % TC_TILE or Bp < B:
        raise RuntimeError("x3_split_input: x must be contiguous fp32 [B, T, 8] and Bp a multiple of 128 >= B")
    xs = torch.empty((T, Bp // TC_TILE, 2, TC_TILE, 8), dtype=torch.float16, device=x.device)
    _lib.call("na_x3_split_input", x.data_ptr(), xs.data_ptr(), B, T, Bp, int(half_stride), _stream())
    return xs


@x3_split_input.register_fake
def _(x, Bp, half_stride=0):
    return x.new_empty((x.shape[1], Bp // TC_TILE, 2, TC_TILE, 8), dtype=torch.float16)


@torch.library.custom_op("neuroalpha::lstm_fwd_train_x3", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_fwd_train_x3(layer: int, inp: Tensor, packed: Tensor, attn_w: Tensor, attn_b: Tensor, mask: Optional[Tensor], seed: int,
                      thresh16: int, drop_scale: float, B: int, half_stride: int = 0) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Training forward of one layer at fp32 accuracy -> (h TCLX, hd TCLX or empty, c TCL32, zpool [B,48] or empty,
    stats [B,2] or empty).  Layer 0: ``inp`` = XS, ``hd`` = h after inter-layer dropout (when on); layer 1: ``inp`` = TCLX."""
    _require_cuda(inp, packed, attn_w, attn_b, mask)
    T, NT = inp.shape[0], inp.shape[1]
    Bp, dev = NT * TC_TILE, inp.device
    has_drop = layer == 0 and (mask is not None or thresh16 < 65536)
    h, c = _tclx(T, Bp, dev), _tcl32(T, Bp, dev)
    hd = _tclx(T, Bp, dev) if has_drop else torch.empty((0,), dtype=torch.float16, device=dev)
    zpool = torch.empty((B, 48) if layer == 1 else (0,), dtype=torch.float32, device=dev)
    stats = torch.empty((B, 2) if layer == 1 else (0,), dtype=torch.float32, device=dev)
    aw, ab = _f32c(attn_w), _f32c(attn_b)
    _lib.call("na_lstm_fwd_train_x3", int(layer), inp.data_ptr(), packed.data_ptr(), aw.data_ptr(), ab.data_ptr(),
              _ptr(mask) if layer == 0 else None, int(seed), int(thresh16) if layer == 0 else 65536, float(drop_scale),
              h.data_ptr(), _ptr(hd) if has_drop else None, c.data_ptr(), _ptr(zpool) if layer == 1 else None,
              _ptr(stats) if layer == 1 else None, int(B), T, Bp, int(half_stride), _stream())
    return h, hd, c, zpool, stats


@lstm_fwd_train_x3.register_fake
def _(layer, inp, packed, attn_w, attn_b, mask, seed, thresh16, drop_scale, B, half_stride=0):
    T, NT = inp.shape[0], inp.shape[1]
    has_drop = layer == 0 and (mask is not None or thresh16 < 65536)
    f32 = lambda *s: inp.new_empty(s, dtype=torch.float32)
    return (inp.new_empty((T, NT, 12, TC_TILE, 8)), inp.new_empty((T, NT, 12, TC_TILE, 8) if has_drop else (0,)),
            f32(T, NT, 12, TC_TILE, 4), f32(B, 48) if layer == 1 else f32(0), f32(B, 2) if layer == 1 else f32(0))


@torch.library.custom_op("neuroalpha::lstm_bwd_x3", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_bwd_x3(layer: int, act_in: Tensor, h: Tensor, c: Tensor, dh_in: Optional[Tensor], packed: Tensor,
                in_mask: Optional[Tensor], seed: int, thresh16: int, drop_scale: float, head: Sequence[Tensor],
                B: int, half_stride: int = 0) -> Tuple[Tensor, Tensor, Tensor]:
    """BPTT of one layer at fp32 accuracy -> (din TCL32 (layer 1) or empty, dg DGX, d_attn [49] or empty).
    ``head`` = [] (dh_in given) or [dz, stats, zpool, attn_w, attn_b]: layer 1 with the head backward's time loop fused."""
    _require_cuda(act_in, h, c, dh_in, packed, in_mask, *head)
    T, NT = c.shape[0], c.shape[1]
    Bp, dev = NT * TC_TILE, c.device
    din = _tcl32(T, Bp, dev) if layer == 1 else torch.empty((0,), dtype=torch.float32, device=dev)
    dg = torch.empty((T, NT, 48, TC_TILE, 8), dtype=torch.float16, device=dev)
    fused = len(head) > 0
    d_attn = torch.empty((52,) if fused else (0,), dtype=torch.float32, device=dev)
    hp = [_f32c(t) for t in head]
    zeros, scratch = _train_buffers(dev, "x3", 24576, 4 * _lib.query("na_train_x3_scratch_floats"))
    _lib.call("na_lstm_bwd_x3", int(layer), act_in.data_ptr(), h.data_ptr(), c.data_ptr(), None if fused else dh_in.data_ptr(),
              packed.data_ptr(), zeros.data_ptr(), _ptr(in_mask), int(seed), int(thresh16), float(drop_scale),
              _ptr(din) if layer == 1 else None, dg.data_ptr(), *([t.data_ptr() for t in hp] if fused else [None] * 5), int(B),
              _ptr(d_attn) if fused else None, scratch.data_ptr(), T, Bp, int(half_stride), _stream())
    return din, dg, d_attn[:49] if fused else d_attn


@lstm_bwd_x3.register_fake
def _(layer, act_in, h, c, dh_in, packed, in_mask, seed, thresh16, drop_scale, head, B, half_stride=0):
    T, NT = c.shape[0], c.shape[1]
    return (c.new_empty(c.shape if layer == 1 else (0,)), h.new_empty((T, NT, 48, TC_TILE, 8)),
            c.new_empty((49,) if len(head) else (0,)))


@torch.library.custom_op("neuroalpha::lstm_wgrad_x3", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_wgrad_x3(layer: int, dg: Tensor, act_in: Tensor, h: Tensor, half_stride: int = 0) -> Tuple[Tensor, Tensor, Tensor]:
    """Time-parallel weight gradients of one layer from d(gates) (DGX) and the saved activations:
    (dW_ih [192, 8 | 48], dW_hh [192, 48], db [192])."""
    _require_cuda(dg, act_in, h)
    T, NT = dg.shape[0], dg.shape[1]
    dev = dg.device
    dw_ih = torch.empty((192, 8 if layer == 0 else 48), dtype=torch.float32, device=dev)
    dw_hh = torch.empty((192, 48), dtype=torch.float32, device=dev)
    db = torch.empty((192,), dtype=torch.float32, device=dev)
    zeros, scratch = _train_buffers(dev, "x3", 24576, 4 * _lib.query("na_train_x3_scratch_floats"))
    _lib.call("na_lstm_wgrad_x3", int(layer), dg.data_ptr(), act_in.data_ptr(), h.data_ptr(), zeros.data_ptr(), dw_ih.data_ptr(),
              dw_hh.data_ptr(), db.data_ptr(), scratch.data_ptr(), T, NT * TC_TILE, int(half_stride), _stream())
    return dw_ih, dw_hh, db


@lstm_wgrad_x3.register_fake
def _(layer, dg, act_in, h, half_stride=0):
    f32 = lambda *s: dg.new_empty(s, dtype=torch.float32)
    return f32(192, 8 if layer == 0 else 48), f32(192, 48), f32(192)


def _x3_forward(x: Tensor, lstm_flat: Sequence[Tensor], head: Sequence[Tensor], p: float, zscore: bool, drop1,
                rrelu_slope: Optional[Tensor], drop2_mask: Optional[Tensor]):
    """Forward of the exact training tier with saves: x [B,T,8] -> (logits, saves (xs, h0, h0d, c0, h1, c1, packed, stats,
    zpool), the layer-0 keep-mask in its tile layout or None, meta (scale, B, seed, thresh16, scale1, half_stride)).
    ``lstm_flat`` / ``head``: detached tensors, the head ones fp32.  Used by DecoderFunctionX3 and, with no noise (eval
    arithmetic), by decoder_input_grad_x3."""
    B, T, C = x.shape
    scale = 1.0 / (1.0 - p) if p < 1.0 else 0.0          # head dropout (and mask-tensor mode)
    mask, seed, thresh16, scale1 = _drop1_args(drop1, scale)
    xin = x.detach()
    if xin.dtype != torch.float32:
        xin = xin.float()
    if zscore:
        xin = window_zscore(xin, T, T, True, False, NA_F32)
    half_stride = _half_stride(B, x.device, X3_HALF_TILES)
    Bp = ((B + 63) // 64) * TC_TILE if half_stride else padded_batch(B, TC_TILE)
    if half_stride and mask is not None:
        mask = _half_tile_rows(mask, B, Bp)
    xs = x3_split_input(xin.contiguous(), Bp, half_stride)
    packed = decoder_pack_x3(lstm_flat)
    h0, h0d, c0, _, _ = lstm_fwd_train_x3(0, xs, packed, head[0], head[1], mask, seed, thresh16, scale1, B, half_stride)
    has_drop = mask is not None or thresh16 < 65536
    h1, _, c1, zpool, stats = lstm_fwd_train_x3(1, h0d if has_drop else h0, packed, head[0], head[1], None, 0, 65536, 1.0, B, half_stride)
    logits, _ = head_tail_fwd(zpool, head, rrelu_slope, drop2_mask, scale, False)
    return logits, (xs, h0, h0d, c0, h1, c1, packed, stats, zpool), mask, (scale, B, seed, thresh16, scale1, half_stride)


class DecoderFunctionX3(torch.autograd.Function):
    """Training step of the flagship decoder at fp32 accuracy on the tensor cores (1e-5 contract on logits and
    gradients): operand-split tcgen05 forward with saves, fp32 head kernels, operand-split BPTT, time-parallel
    weight-gradient GEMMs.  No d/dx (the FFMA tier provides it; input attributions: decoder_input_grad_x3)."""

    @staticmethod
    def forward(ctx, x, p, zscore, drop1, rrelu_slope, drop2_mask, *params):
        _require_cuda(x, *params)
        ctx.param_dtypes = [t.dtype for t in params]
        if ctx.needs_input_grad[0]:
            raise RuntimeError("the tensor-core exact training tier does not produce d/dx")
        lstm_flat, head = [t.detach() for t in params[:8]], [_f32c(t.detach()) for t in params[8:]]
        logits, saves, mask, ctx.meta = _x3_forward(x, lstm_flat, head, p, zscore, drop1, rrelu_slope, drop2_mask)
        _save(ctx, [*saves, *head], [mask, rrelu_slope, drop2_mask])
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        scale, B, seed, thresh16, scale1, hs = ctx.meta
        sv, (d1, rr, d2) = _saved(ctx)
        xs, h0, h0d, c0, h1, c1, packed, stats, zpool = sv[:9]
        head = sv[9:]
        in1 = h0d if d1 is not None or thresh16 < 65536 else h0

        def layers_bwd(dz):
            din1, dg1, d_attn = lstm_bwd_x3(1, in1, h1, c1, None, packed, d1, seed, thresh16, scale1, [dz, stats, zpool, head[0], head[1]], B, hs)
            dw_ih1, dw_hh1, db1 = lstm_wgrad_x3(1, dg1, in1, h1, hs)
            del dg1
            _, dg0, _ = lstm_bwd_x3(0, xs, h0, c0, din1, packed, None, 0, 65536, 1.0, [], B, hs)
            dw_ih0, dw_hh0, db0 = lstm_wgrad_x3(0, dg0, xs, h0, hs)
            del dg0
            return dw_ih0, dw_hh0, db0, dw_ih1, dw_hh1, db1, d_attn.clone()     # (d_attn: a slice of the kernel's 52-float output)
        return _tc_backward(ctx, dlogits, zpool, head, rr, d2, scale, layers_bwd)


def decoder_train_forward_x3(x: Tensor, lstm_params, head_params, p: float, zscore: bool = False,
                             drop1=None, rrelu_slope=None, drop2_mask=None) -> Tensor:
    flat = [t for layer in lstm_params for t in layer]
    return DecoderFunctionX3.apply(x, p, zscore, drop1, rrelu_slope, drop2_mask, *flat, *head_params)


@torch.library.custom_op("neuroalpha::lstm_bwd_x3_dx", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_bwd_x3_dx(layer: int, act_in: Tensor, h: Tensor, c: Tensor, dh_in: Optional[Tensor], packed: Tensor,
                   head: Sequence[Tensor], dz_inv_scale: Optional[Tensor], B: int, half_stride: int = 0) -> Tensor:
    """BPTT of one layer for input attributions (no weight-gradient byproducts, no dropout) -> layer 1: din TCL32;
    layer 0: dx fp32 [B, T, 8], each window's row multiplied by ``dz_inv_scale[b]``.  ``head`` as in lstm_bwd_x3."""
    _require_cuda(act_in, h, c, dh_in, packed, dz_inv_scale, *head)
    T, NT = c.shape[0], c.shape[1]
    Bp, dev = NT * TC_TILE, c.device
    out = _tcl32(T, Bp, dev) if layer == 1 else torch.empty((B, T, 8), dtype=torch.float32, device=dev)
    fused = len(head) > 0
    hp = [_f32c(t) for t in head]
    zeros, _ = _train_buffers(dev, "x3", 24576, 4 * _lib.query("na_train_x3_scratch_floats"))
    _lib.call("na_lstm_bwd_x3_dx", int(layer), act_in.data_ptr(), h.data_ptr(), c.data_ptr(), None if fused else dh_in.data_ptr(),
              packed.data_ptr(), zeros.data_ptr(), None, 0, 65536, 1.0, out.data_ptr() if layer == 1 else None,
              *([t.data_ptr() for t in hp] if fused else [None] * 5), int(B), out.data_ptr() if layer == 0 else None,
              _f32c(dz_inv_scale).data_ptr() if layer == 0 else None, T, Bp, int(half_stride), _stream())
    return out


@lstm_bwd_x3_dx.register_fake
def _(layer, act_in, h, c, dh_in, packed, head, dz_inv_scale, B, half_stride=0):
    return c.new_empty(c.shape) if layer == 1 else c.new_empty((B, c.shape[0], 8))


def _scale_dz_rows(dz: Tensor) -> Tuple[Tensor, Tensor]:
    """_scale_dz per window, for per-window results: row b of dz is scaled by its own power of two 2^6 / 2^ceil(log2
    max|dz_b|), so a window whose dz is far below the batch maximum (LayerNorm's 1/sigma varies per window) keeps its low
    bits in the fp16 d(gates), and a NaN window leaves the others' scale alone.  Everything below dz is linear per
    window.  -> (scaled dz, the inverse factors [B])."""
    amax = dz.abs().amax(dim=1, keepdim=True).clamp_min(1e-30)
    s = torch.pow(2.0, 6.0 - torch.ceil(torch.log2(amax)))
    return dz * s, (1.0 / s).reshape(-1).contiguous()


def _input_grad_x3_round(x: Tensor, lstm_flat: Sequence[Tensor], head: Sequence[Tensor], target: Optional[Tensor]):
    logits, saves, _, meta = _x3_forward(x, lstm_flat, head, 0.0, False, None, None, None)
    xs, h0, _, c0, h1, c1, packed, stats, zpool = saves
    B, hs = meta[1], meta[5]
    tgt = logits.argmax(dim=1) if target is None else target
    dlogits = torch.zeros_like(logits).scatter_(1, tgt[:, None], 1.0)
    dz, _ = head_tail_bwd(dlogits, zpool, head, None, None, 1.0)
    dz, inv_s = _scale_dz_rows(dz)
    din1 = lstm_bwd_x3_dx(1, h0, h1, c1, None, packed, [dz, stats, zpool, head[0], head[1]], None, B, hs)
    del h1, c1
    dx = lstm_bwd_x3_dx(0, xs, h0, c0, din1, packed, [], inv_s, B, hs)
    return logits, tgt, dx


def decoder_input_grad_x3(x: Tensor, lstm_params, head_params, target: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """Saliency of the flagship decoder on the exact tensor-core tier, eval arithmetic (no dropout, RReLU at its eval
    slope): x fp32 [B,T,8] -> (logits [B,K], dx = d logits[b, target[b]] / d x[b] fp32 [B,T,8]).  ``target``: long [B], or
    None for the argmax of each window's logits.  Runs without autograd: the forward of DecoderFunctionX3, the head tail
    backward of a one-hot dlogits, then both layers' BPTT without weight gradients.  Batches above one round of full
    tiles (SMs x 128 windows) run round by round; each round saves about 1 MB per 625-step window."""
    _require_cuda(x, target)
    B, T, C = x.shape
    with torch.no_grad():
        lstm_flat = [t.detach() for layer in lstm_params for t in layer]
        head = [_f32c(t.detach()) for t in head_params]
        rnd = _sm_count(x.device) * TC_TILE
        if B <= rnd:
            logits, _, dx = _input_grad_x3_round(x, lstm_flat, head, target)
            return logits, dx
        parts = [_input_grad_x3_round(x[i:i + rnd], lstm_flat, head, None if target is None else target[i:i + rnd])
                 for i in range(0, B, rnd)]
        return torch.cat([q[0] for q in parts]), torch.cat([q[2] for q in parts])


# ------------------------------------------------------------------------------------------
# wide decoders (H = 96 / 144 / 192): training on the tensor cores, 16-bit tier (csrc/na_wide_train.cu)
# ------------------------------------------------------------------------------------------
def _to_wtl(x2d: Tensor, T: int, Bp: int, H: int) -> Tensor:
    """row-major [T*Bp, F] -> WTL [T, NT, H/48 * 3, P, 128, 16 bytes]: thread = (row, 16-unit group g of task k) owns P
    16-byte pieces, the lanes of a warp are contiguous within a piece.  F = 4H (gates, torch order gate * H + unit ->
    accumulator column order (u/4)*16 + gate*4 + u%4 within the group) or F = H (h, c, dh: unit order).  One transpose copy."""
    nt, nch = Bp // TC_TILE, H // 48
    if x2d.shape[1] == 4 * H:
        v = x2d.view(T, nt, TC_TILE, 2, 2, nch, 3, 4, 4)                  # t, tile, row, gate/2, gate%2, k, g, q, ur
        return v.permute(0, 1, 5, 6, 7, 3, 2, 4, 8).reshape(T, nt, nch * 3, 8, TC_TILE, 8).contiguous()
    epp = 16 // x2d.element_size()                                       # elements per 16-byte piece
    v = x2d.view(T, nt, TC_TILE, nch, 3, 16 // epp, epp)                  # t, tile, row, k, g, piece, e
    return v.permute(0, 1, 3, 4, 5, 2, 6).reshape(T, nt, nch * 3, 16 // epp, TC_TILE, epp).contiguous()   # (reshape alone may return a view)


def _from_wtl(w: Tensor, T: int, Bp: int, H: int) -> Tensor:
    """WTL -> row-major [T*Bp, F] (the inverse of _to_wtl)."""
    nt, nch = Bp // TC_TILE, H // 48
    if w.shape[3] == 8 and w.dtype == torch.float16 and w.shape[5] == 8:  # gates / d(gates)
        v = w.view(T, nt, nch, 3, 4, 2, TC_TILE, 2, 4)                    # t, tile, k, g, q, gate/2, row, gate%2, ur
        return v.permute(0, 1, 6, 5, 7, 2, 3, 4, 8).reshape(T * Bp, 4 * H).contiguous()
    v = w.view(T, nt, nch, 3, w.shape[3], TC_TILE, w.shape[5])           # t, tile, k, g, piece, row, e
    return v.permute(0, 1, 5, 2, 3, 4, 6).reshape(T * Bp, H).contiguous()


def _wide_images(w_hh: Tensor, H: int):
    """The two streamed weight images of a layer (see include/neuroalpha.h): forward [nch][H/16][2][192][8] and
    backward [nch][12][2][H][8], fp16."""
    nch = H // 48
    n = torch.arange(192, device=w_hh.device)
    j, gate = (n // 16) * 4 + n % 4, (n % 16) // 4
    rows = (gate[None, :] * H + 48 * torch.arange(nch, device=w_hh.device)[:, None] + j[None, :])        # [nch, 192] torch rows
    wt = w_hh.detach().float()[rows]                                                                    # [nch, 192 (n), H (k)]
    fwd = wt.reshape(nch, 192, H // 16, 2, 8).permute(0, 2, 3, 1, 4).contiguous().to(torch.float16)     # [nch][ks][c2][n][e]
    bwd = wt.permute(0, 2, 1).reshape(nch, H, 12, 2, 8).permute(0, 2, 3, 1, 4).contiguous().to(torch.float16)   # [nch][ks][c2][n_out][e]
    return fwd, bwd


@torch.library.custom_op("neuroalpha::lstm_wide_fwd_train", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_wide_fwd_train(gx: Tensor, w_image: Tensor, H: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Serial part of one wide layer's training forward.  gx: WTL fp16 [T, NT, H/48 * 3, 8, 128, 8] -> (gates WTL, h WTL fp16
    [.., 2, 128, 8], c WTL fp32 [.., 4, 128, 4])."""
    _require_cuda(gx, w_image)
    T, NT = gx.shape[0], gx.shape[1]
    gates = torch.empty_like(gx)                                        # [T, NT, nch * 3, 8, 128, 8]
    h = torch.empty(gx.shape[:3] + (2, TC_TILE, 8), dtype=torch.float16, device=gx.device)
    c = torch.empty(gx.shape[:3] + (4, TC_TILE, 4), dtype=torch.float32, device=gx.device)
    _lib.call("na_lstm_wide_fwd_train", gx.data_ptr(), w_image.data_ptr(), gates.data_ptr(), h.data_ptr(), c.data_ptr(), T, NT * TC_TILE,
              int(H), _stream())
    return gates, h, c


@lstm_wide_fwd_train.register_fake
def _(gx, w_image, H):
    return (gx.new_empty(gx.shape), gx.new_empty(gx.shape[:3] + (2, TC_TILE, 8)),
            gx.new_empty(gx.shape[:3] + (4, TC_TILE, 4), dtype=torch.float32))


@torch.library.custom_op("neuroalpha::lstm_wide_bwd", mutates_args=(), device_types="cuda")
@_device_guard
def lstm_wide_bwd(gates: Tensor, c: Tensor, dh_in: Tensor, w_image: Tensor, H: int) -> Tensor:
    """Serial part of one wide layer's BPTT: (gates, c, dh_in) WTL -> d(gates) WTL fp16."""
    _require_cuda(gates, c, dh_in, w_image)
    T, NT = gates.shape[0], gates.shape[1]
    dg = torch.empty_like(gates)
    ws = torch.empty((_lib.query("na_wide_train_ws_floats", int(H)),), dtype=torch.float32, device=gates.device)
    _lib.call("na_lstm_wide_bwd", gates.data_ptr(), c.data_ptr(), dh_in.data_ptr(), w_image.data_ptr(), dg.data_ptr(), ws.data_ptr(),
              T, NT * TC_TILE, int(H), _stream())
    return dg


@lstm_wide_bwd.register_fake
def _(gates, c, dh_in, w_image, H):
    return gates.new_empty(gates.shape)


def _mm_f32(a: Tensor, b: Tensor) -> Tensor:
    """fp16 x fp16 -> fp32 GEMM (cuBLAS, fp32 accumulate AND fp32 output: sums over millions of rows must not round to fp16)."""
    try:
        return torch.mm(a, b, out_dtype=torch.float32)
    except TypeError:                                  # older torch: chunk the reduction dimension and accumulate in fp32
        out = torch.zeros((a.shape[0], b.shape[1]), dtype=torch.float32, device=a.device)
        step = 1 << 18
        for i in range(0, a.shape[1], step):
            out += a[:, i:i + step].float() @ b[i:i + step].float()
        return out


class DecoderFunctionWideTC(torch.autograd.Function):
    """Training step of a wide decoder (hidden_size 96 / 144 / 192, 2 layers) on the 16-bit tensor-core tier: cuBLAS for
    everything that is parallel over time, the streamed-weight recurrence kernels for the serial part of every layer and
    direction, the fp32 head kernels.  2e-2 contract."""

    @staticmethod
    def forward(ctx, x, p, zscore, drop1, rrelu_slope, drop2_mask, *params):
        _require_cuda(x, *params)
        ctx.param_dtypes = [t.dtype for t in params]
        if ctx.needs_input_grad[0]:
            raise RuntimeError("the tensor-core training tier does not produce d/dx; use compute_dtype=float32")
        B, T, C = x.shape
        lstm, head = [t.detach() for t in params[:8]], [_f32c(t.detach()) for t in params[8:]]
        H = lstm[1].shape[1]
        scale = 1.0 / (1.0 - p) if p < 1.0 else 0.0
        Bp = padded_batch(B, TC_TILE)
        dev = x.device
        xin = x.detach().float()
        if zscore:
            xin = window_zscore(xin, T, T, True, False, NA_F32)
        xt = torch.zeros((T, Bp, C), dtype=torch.float32, device=dev)
        xt[:, :B] = xin.permute(1, 0, 2)
        layer_in = xt.reshape(T * Bp, C)
        saved, h_rows = [], []
        mask = None
        for l in range(2):
            w_ih, w_hh, b_ih, b_hh = lstm[4 * l:4 * l + 4]
            fimg, bimg = _wide_images(w_hh, H)
            if l == 0:          # K = 8: fp32 GEMM (raw EEG can exceed fp16's range), rounded to fp16 afterwards
                gx2d = torch.addmm((b_ih + b_hh).float(), layer_in, w_ih.float().t()).to(torch.float16)
            else:
                gx2d = torch.addmm((b_ih + b_hh).to(torch.float16), layer_in, w_ih.to(torch.float16).t())
            gates, h, c = lstm_wide_fwd_train(_to_wtl(gx2d, T, Bp, H), fimg, H)
            del gx2d
            h2d = _from_wtl(h, T, Bp, H)                                         # [T*Bp, H] fp16, unit order
            saved += [gates, c, bimg, layer_in if l == 0 else None]
            h_rows.append(h2d)
            if l == 0:
                if drop1 is not None:                                            # inter-layer dropout (lstm_eeg_model.py:21)
                    mask = drop1.reshape(T * Bp, H).to(torch.float16)
                    layer_in = h2d * mask * scale
                else:
                    layer_in = h2d
        h1 = h_rows[1].float().reshape(T, Bp, H)
        logits, _, stats, zpool = head_fwd(h1, B, head, rrelu_slope, drop2_mask, scale, False, True)
        _save(ctx, [*saved[:7], h_rows[0], h_rows[1], layer_in if mask is not None else h_rows[0], stats, zpool, *lstm, *head],
              [mask, rrelu_slope, drop2_mask])
        ctx.meta = (scale, B, T, Bp, H)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        scale, B, T, Bp, H = ctx.meta
        sv, (mask, rr, d2) = _saved(ctx)
        gates0, c0, bimg0, x2d, gates1, c1, bimg1, h0_2d, h1_2d, in1_2d, stats, zpool = sv[:12]
        lstm, head = sv[12:20], sv[20:28]
        dev = dlogits.device
        NC = dlogits.shape[1]
        h1 = h1_2d.float().reshape(T, Bp, H)
        dh1, dparams = head_bwd(dlogits.contiguous(), h1, stats, zpool, head, rr, d2, scale)
        del h1
        dh1, _, inv_s = _scale_dz(dh1)       # d(gates) are fp16: the gradient entering the recurrence, scaled (max|dh| -> 2^6)
        zeros_h = torch.zeros((Bp, H), dtype=torch.float16, device=dev)
        def layer_bwd(gates, c, bimg, dh2d, in2d, h2d, w_ih):
            dg = lstm_wide_bwd(gates, c, _to_wtl(dh2d, T, Bp, H), bimg, H)
            dg2d = _from_wtl(dg, T, Bp, H)                                       # [T*Bp, 4H] fp16, torch gate order
            del dg
            dgt = dg2d.t()
            in16 = in2d if in2d.dtype == torch.float16 else in2d.to(torch.float16)
            dw_ih = _mm_f32(dgt, in16)
            hprev = torch.cat([zeros_h, h2d[:-Bp]])                               # h_{t-1}
            dw_hh = _mm_f32(dgt, hprev)
            db = _mm_f32(dgt, torch.ones((dg2d.shape[0], 8), dtype=torch.float16, device=dev))[:, 0].contiguous()
            return dg2d, dw_ih, dw_hh, db
        dg1, dw_ih1, dw_hh1, db1 = layer_bwd(gates1, c1, bimg1, dh1.reshape(T * Bp, H), in1_2d, h1_2d, lstm[4])
        del dh1
        din1 = _mm_f32(dg1, lstm[4].to(torch.float16))                            # [T*Bp, H] fp32 (still scaled by s)
        del dg1
        if mask is not None:
            din1 = din1 * mask * scale
        # layer 0: its input is the raw fp32 window; x can exceed fp16's range, so the weight gradient uses x / 16 (exact) and is rescaled
        x16 = (x2d * 0.0625).to(torch.float16)
        dg0, dw_ih0, dw_hh0, db0 = layer_bwd(gates0, c0, bimg0, din1, x16, h0_2d, lstm[0])
        dw_ih0 = dw_ih0 * 16.0
        del dg0, din1
        head_grads = split_head_grads(dparams, H, NC)
        db0, db1 = db0 * inv_s, db1 * inv_s
        grads = [dw_ih0 * inv_s, dw_hh0 * inv_s, db0, db0.clone(), dw_ih1 * inv_s, dw_hh1 * inv_s, db1, db1.clone(), *head_grads]
        return (None, None, None, None, None, None, *_cast_grads(grads, ctx.param_dtypes))


def decoder_train_forward_wide_tc(x: Tensor, lstm_params, head_params, p: float, zscore: bool = False,
                                  drop1=None, rrelu_slope=None, drop2_mask=None) -> Tensor:
    flat = [t for layer in lstm_params for t in layer]
    return DecoderFunctionWideTC.apply(x, p, zscore, drop1, rrelu_slope, drop2_mask, *flat, *head_params)
