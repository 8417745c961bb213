"""Predicted accuracy of the exact tier's input attributions (ops.decoder_input_grad_x3): a CPU simulation of the split
BPTT's dx = d logits[target] / dx over the 324 shipped windows (625 steps), against float64.  Prints the worst per-window
max|d| / max|ref| for the argmax target and for the next class.  CPU only, a few minutes.

    python scripts/x3_dx_split_error.py

What the simulation rounds as the kernels do: the forward as scripts/x3_split_error.py "split std" (operands split into fp16
hi + lo, products hi.hi + hi.lo + lo.hi, fp32 sums; layer 0 stores x / 16 against 16 W_ih), the gradient entering the
recurrence scaled per window to max|dz_b| in (2^5, 2^6], d(gates) in fp32 and split the same way for the three products
of every step (dh_rec = dG . W_hh, din = dG . W_ih1, dx = dG . 16 W_ih0 / 16).  The head and the attention pooling
backward stay in float64 (the kernels run them in fp32, whose error is far below the split's).
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle.torch_ref import RefEEGLSTM  # noqa: E402

ck = np.load(ROOT / "tests" / "golden" / "checkpoint_3class.npz")
sd = {str(k): torch.from_numpy(ck[str(k)].copy()).double() for k in ck["__order__"]}
X = torch.from_numpy(np.load(ROOT / "tests" / "golden" / "eeg_windows.npz")["X"].copy()).double()
H = 48
f32 = lambda a: a.float().double()


def split(v):
    hi = v.half().double()
    return hi, (v - hi).half().double()


def mm(a, w, exact):                      # a [B,K] . w [K,N]
    if exact:
        return a @ w
    ah, al = split(a)
    wh, wl = split(w)
    return f32(ah @ wh + ah @ wl + al @ wh)


def lstm(x, l, exact):
    wi, wh = sd[f"lstm.weight_ih_l{l}"], sd[f"lstm.weight_hh_l{l}"]
    b = sd[f"lstm.bias_ih_l{l}"] + sd[f"lstm.bias_hh_l{l}"]
    if not exact:
        b = sum(split(f32(b)))
    xs, wis = (x / 16, wi * 16) if (l == 0 and not exact) else (x, wi)
    B, T = x.shape[:2]
    h, c = torch.zeros(B, H, dtype=torch.float64), torch.zeros(B, H, dtype=torch.float64)
    hs, cs, gs = [], [], []
    for t in range(T):
        pre = mm(xs[:, t], wis.T, exact) + mm(h, wh.T, exact) + b
        i, f, g, o = pre.split(H, dim=1)
        i, f, g, o = torch.sigmoid(i), torch.sigmoid(f), torch.tanh(g), torch.sigmoid(o)
        if not exact:
            i, f, g, o = f32(i), f32(f), f32(g), f32(o)
        c = f * c + i * g
        h = o * torch.tanh(c)
        if not exact:
            c, h = f32(c), f32(h)
        hs.append(h), cs.append(c), gs.append((i, f, g, o))
    return torch.stack(hs, 1), cs, gs


def bptt(dh_in, cs, gs, l, exact, dxs=None):
    """dh_in [B,T,H] -> d(input) [B,T,K]."""
    wi, wh = sd[f"lstm.weight_ih_l{l}"], sd[f"lstm.weight_hh_l{l}"]
    wis = wi * 16 if (l == 0 and not exact) else wi
    B, T = dh_in.shape[:2]
    dh_rec, dc = torch.zeros(B, H, dtype=torch.float64), torch.zeros(B, H, dtype=torch.float64)
    din = torch.zeros(B, T, wi.shape[1], dtype=torch.float64)
    for t in range(T - 1, -1, -1):
        i, f, g, o = gs[t]
        c, cp = cs[t], (cs[t - 1] if t else torch.zeros_like(cs[t]))
        dh = dh_in[:, t] + dh_rec
        tc = torch.tanh(c)
        dct = dh * o * (1 - tc * tc) + dc
        dG = torch.cat([dct * g * i * (1 - i), dct * cp * f * (1 - f), dct * i * (1 - g * g), dh * tc * o * (1 - o)], 1)
        if not exact:
            dG = f32(dG)
        dc = dct * f
        dh_rec = mm(dG, wh, exact)
        d = mm(dG, wis, exact)
        din[:, t] = d if exact else d / 16 if l == 0 else d
    return din


def saliency(exact, target):
    h0, cs0, gs0 = lstm(X, 0, exact)
    h1, cs1, gs1 = lstm(h0, 1, exact)
    ref = RefEEGLSTM().double().eval()
    ref.load_state_dict(sd)
    hv = h1.clone().requires_grad_(True)
    s = ref.attn(hv).squeeze(-1)
    z = (torch.softmax(s, dim=1)[..., None] * hv).sum(1)
    lg = ref.fc(ref.ln(z))
    tgt = lg.argmax(1) if target is None else target
    (dh1,) = torch.autograd.grad(lg.gather(1, tgt[:, None]).sum(), hv)   # the head + pooling backward, float64
    inv = torch.ones(X.shape[0], 1, 1, dtype=torch.float64)
    if not exact:                                                       # per-window power of two, as _scale_dz_rows
        amax = dh1.abs().amax(dim=(1, 2), keepdim=True).clamp_min(1e-30)
        sc = 2.0 ** (6.0 - torch.ceil(torch.log2(amax)))
        dh1, inv = dh1 * sc, 1 / sc
    din1 = bptt(dh1, cs1, gs1, 1, exact)
    if not exact:
        din1 = f32(din1)
    return bptt(din1, cs0, gs0, 0, exact) * inv, tgt


if __name__ == "__main__":
    ref_a, tgt = saliency(True, None)
    for name, t in (("argmax", tgt), ("next class", (tgt + 1) % 3)):
        want = ref_a if name == "argmax" else saliency(True, t)[0]
        got = saliency(False, t)[0]
        err = (got - want).abs().amax(dim=(1, 2)) / want.abs().amax(dim=(1, 2))
        print(f"{name}: worst per-window max|d|/max|ref| {float(err.max()):.3g}, median {float(err.median()):.3g}", flush=True)
