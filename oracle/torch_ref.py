"""Torch-CPU restatement of the reference decoder (TEST INFRASTRUCTURE).

Two forms:

* ``RefEEGLSTM`` -- the reference module restated from its torch building blocks
  (``nn.LSTM``/``nn.LayerNorm``/``nn.Linear``/``nn.RReLU``/``nn.Dropout``), i.e. the
  same CPU arithmetic the reference runs (oneDNN ``aten::mkldnn_rnn_layer``).  It is
  the CPU arm timed by ``bench.py`` (``cpu_baseline.kind = "port"``) because
  ``/root/reference`` does not exist on the GPU box.
  Restates Neuro-Alpha-App/Utilities/lstm_eeg_model.py:13-39.
* ``explicit_forward`` -- the same maths written out cell by cell in differentiable
  torch ops so that the train-mode noise (LSTM inter-layer dropout :21, RReLU slope
  :27, Dropout :28) can be injected and autograd gives the matching gradients.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

RRELU_EVAL_SLOPE = (1.0 / 8.0 + 1.0 / 3.0) / 2.0


class RefEEGLSTM(nn.Module):
    def __init__(self, input_size=8, hidden_size=48, num_layers=2, num_classes=3, dropout=0.60):
        super().__init__()
        self.lstm = nn.LSTM(input_size=input_size, hidden_size=hidden_size, num_layers=num_layers,
                            batch_first=True, dropout=dropout if num_layers > 1 else 0.0)
        self.ln = nn.LayerNorm(hidden_size)
        self.attn = nn.Linear(hidden_size, 1)
        self.fc = nn.Sequential(nn.Linear(hidden_size, 32), nn.RReLU(), nn.Dropout(dropout),
                                nn.Linear(32, num_classes))

    def forward(self, x):
        out, _ = self.lstm(x)
        w = torch.softmax(self.attn(out).squeeze(-1), dim=1)
        out = (out * w.unsqueeze(-1)).sum(dim=1)
        return self.fc(self.ln(out))


def explicit_forward(x, sd, num_layers=2, p=0.6, drop1_mask=None, rrelu_slope=None, drop2_mask=None, drop1_scale=None):
    """x [B,T,C]; sd: name -> tensor (may require grad).  Returns logits [B,K].

    Masks are 0/1 tensors; scaling by 1/(1-p) (0 for p = 1) is applied here, as torch's dropout does.  ``drop1_scale``
    replaces that factor for the inter-layer dropout (the in-kernel generator of the tensor-core tiers scales by
    65536 / thresh16).
    """
    scale = 1.0 / (1.0 - p) if p < 1.0 else 0.0
    scale1 = scale if drop1_scale is None else drop1_scale
    inp = x
    for l in range(num_layers):
        w_ih, w_hh = sd[f"lstm.weight_ih_l{l}"], sd[f"lstm.weight_hh_l{l}"]
        bias = sd[f"lstm.bias_ih_l{l}"] + sd[f"lstm.bias_hh_l{l}"]
        B, T, _ = inp.shape
        H = w_hh.shape[1]
        h = inp.new_zeros(B, H)
        c = inp.new_zeros(B, H)
        pre = inp @ w_ih.t() + bias
        hs = []
        for t in range(T):
            g = pre[:, t] + h @ w_hh.t()
            i, f, gg, o = g.split(H, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(gg)
            h = torch.sigmoid(o) * torch.tanh(c)
            hs.append(h)
        inp = torch.stack(hs, dim=1)
        if drop1_mask is not None and l < num_layers - 1:
            inp = inp * drop1_mask * scale1
    out = inp
    scores = out @ sd["attn.weight"][0] + sd["attn.bias"][0]
    w = torch.softmax(scores, dim=1)
    z = (out * w.unsqueeze(-1)).sum(dim=1)
    z = F.layer_norm(z, (z.shape[-1],), sd["ln.weight"], sd["ln.bias"], 1e-5)
    a = z @ sd["fc.0.weight"].t() + sd["fc.0.bias"]
    slope = RRELU_EVAL_SLOPE if rrelu_slope is None else rrelu_slope
    a = torch.where(a >= 0, a, a * slope)
    if drop2_mask is not None:
        a = a * drop2_mask * scale
    return a @ sd["fc.3.weight"].t() + sd["fc.3.bias"]
