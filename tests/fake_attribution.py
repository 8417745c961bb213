"""Host stand-in for ops.decoder_input_grad_x3 (TEST INFRASTRUCTURE): the same (logits, dx) from float64 autograd of
oracle.torch_ref.RefEEGLSTM, so that EEG_LSTM.input_gradients / integrated_gradients can be exercised on the fast path
where there is no GPU (tests/test_attribution_host.py).  Records every call.  The product never imports this module."""
from __future__ import annotations

import torch

from oracle.torch_ref import RefEEGLSTM

_NAMES = ("attn.weight", "attn.bias", "ln.weight", "ln.bias", "fc.0.weight", "fc.0.bias", "fc.3.weight", "fc.3.bias")


class FakeInputGradX3:
    def __init__(self):
        self.calls = []

    def __call__(self, x, lstm_params, head_params, target=None):
        self.calls.append((tuple(x.shape), None if target is None else target.clone()))
        H, K = lstm_params[0][1].shape[1], head_params[6].shape[0]
        ref = RefEEGLSTM(input_size=x.shape[2], hidden_size=H, num_layers=len(lstm_params), num_classes=K).double().eval()
        sd = {f"lstm.{n}_l{l}": p for l, layer in enumerate(lstm_params)
              for n, p in zip(("weight_ih", "weight_hh", "bias_ih", "bias_hh"), layer)}
        sd.update(zip(_NAMES, head_params))
        ref.load_state_dict({k: v.detach().double() for k, v in sd.items()})
        with torch.enable_grad():
            xg = x.detach().double().requires_grad_(True)
            logits = ref(xg)
            pick = logits.argmax(dim=1) if target is None else target
            (dx,) = torch.autograd.grad(logits.gather(1, pick[:, None]).sum(), xg)
        return logits.detach().float(), dx.float()
