"""GPU version of the preprocessing step that precedes the decoder on every live window (SURVEY 8(f) rank 1).

The reference filters each ``[T, C]`` window on the CPU before it reaches the model
(``Utilities/preprocessor.py:21-36`` -> the vendored ``mindsai_filter_python`` package, ``core.py:14-48``;
0.76 ms per window and core -- three orders of magnitude slower than the GPU decoder it feeds).  This module runs
the same mathematics for whole batches in one kernel (``csrc/na_phase.cu``):

    analytic signal per channel (Hilbert transform)  ->  instantaneous phases
    P[i, j] = sum_t sin^2(phase_i - phase_j),  P <- D^-1 P D^-1  (D = sqrt(clip(diag P, 1e-12)))
    y = (I + lambda P^T P)^-1 x

**Opt-in only.**  The method belongs to MindsApplied Incorporated (patent pending; their reference implementation is
licensed under the Polyform Noncommercial License 1.0.0 -- ``Utilities/MindsAI/LICENSE``, ``PATENTS.md`` in the
reference tree).  Nothing here is copied from it -- the kernel is written from the published mathematics -- but *using*
the method is subject to their terms, so the class refuses to construct unless the caller states
``accept_noncommercial_terms=True``, and nothing in this package enables it by default:
``SimplePredictor`` keeps calling the host application's own ``PreProcessor`` unless it is handed this object.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, ops

T_WINDOW, N_CHANNELS = 625, 8


class PhaseCouplingFilterGPU:
    """Drop-in for the reference's ``PreProcessor`` (``transform([T, C]) -> [T, C]``, float32) plus the batched
    ``transform_batch([B, T, C])`` that the GPU path is for.  ``tailoring_lambda`` as in
    ``PreProcessor(sr, tailoring_lambda=1.25e-29)`` (``sr`` is accepted and unused there as well)."""

    def __init__(self, sr: int = 125, tailoring_lambda: float = 1.25e-29, device=None, accept_noncommercial_terms: bool = False):
        if not accept_noncommercial_terms:
            raise PermissionError(
                "PhaseCouplingFilterGPU implements MindsApplied's phase-coupling filter (patent pending; reference implementation "
                "under the Polyform Noncommercial License 1.0.0).  It is opt-in: pass accept_noncommercial_terms=True if your use "
                "is permitted by those terms; otherwise keep the host application's own PreProcessor.")
        self.sr = sr
        self.tailoring_lambda = float(tailoring_lambda)
        self.device = ops.compute_device(torch.device(device) if device is not None else torch.device("cpu"))
        k = np.arange(T_WINDOW, dtype=np.float64)
        ang = -2.0 * np.pi * k / T_WINDOW
        self._twiddle = torch.from_numpy(np.stack([np.cos(ang), np.sin(ang)], axis=1).reshape(-1).copy()).to(self.device)

    def transform_batch(self, x: torch.Tensor) -> torch.Tensor:
        """x fp32 ``[B, 625, 8]`` on the CUDA device -> filtered windows, same shape / dtype / device."""
        ops._require_cuda(x)
        if x.dim() != 3 or x.shape[1] != T_WINDOW or x.shape[2] != N_CHANNELS:
            raise ValueError(f"Expected windows of shape [B, {T_WINDOW}, {N_CHANNELS}], got {tuple(x.shape)}")
        x = ops._aligned16(ops._f32c(x))
        y = torch.empty_like(x)
        if x.shape[0] == 0:
            return y
        status = torch.zeros((4,), dtype=torch.int32, device=x.device)
        tw = self._twiddle if self._twiddle.device == x.device else self._twiddle.to(x.device)
        with torch.cuda.device(x.device):
            _lib.call("na_phase_coupling_filter", x.data_ptr(), y.data_ptr(), tw.data_ptr(), self.tailoring_lambda,
                      status.data_ptr(), x.shape[0], T_WINDOW, N_CHANNELS, ops._stream())
        self._last_status = status           # checked lazily: no host sync on the hot path
        return y

    def check(self) -> None:
        """Raise ``numpy.linalg.LinAlgError`` (what the reference's ``np.linalg.inv`` raises) if a window of the last
        batch had a singular system: an exactly zero pivot, as LAPACK reports it.  A window holding NaN or Inf is not
        singular; like the reference, its output is NaN."""
        st = getattr(self, "_last_status", None)
        if st is not None and int(st[0].item()) != 0:
            raise np.linalg.LinAlgError("Singular matrix")

    def transform(self, chunk_samples_by_channels: np.ndarray) -> np.ndarray:
        """``[samples, channels]`` float32 numpy -> filtered ``[samples, channels]`` float32 numpy (reference contract,
        preprocessor.py:21-36, same ``ValueError`` on a non-2D chunk)."""
        x = np.asarray(chunk_samples_by_channels)
        if x.ndim != 2:
            raise ValueError(f"Expected 2D array [samples, channels], got {x.shape}")
        xt = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)[None]).to(self.device)
        out = self.transform_batch(xt)[0].cpu().numpy()
        self.check()
        return out
