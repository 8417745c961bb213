"""Where the fused exact-tier kernel's per-step LSTM error comes from: a numpy simulation of the two-layer recurrence
over the 324 shipped windows (625 steps), with each error source switched on alone, against float64.  Prints
max|d| / max|ref| of the last layer's h over all steps.  CPU only, a few minutes.

    python scripts/x3_split_error.py

  operands: fp64 | fp32 (FFMA kernels) | split (fp16 hi + lo, products hi.hi + hi.lo + lo.hi: the tensor-core kernel)
            | split4 (also lo.lo)
  activations: std (sigmoid / tanh rounded to fp32) | alg (the kernel's ex2 / rcp combination, cell_granule_exact;
            ex2 and rcp exactly rounded, so the MUFU approximations' own error is not included)
"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ck = dict(np.load(ROOT / "tests" / "golden" / "checkpoint_3class.npz"))
ck = {k: v.astype(np.float64) for k, v in ck.items() if k != "__order__"}
X = np.load(ROOT / "tests" / "golden" / "eeg_windows.npz")["X"].astype(np.float64)
f32 = lambda a: np.asarray(a, np.float32).astype(np.float64)
def split(v):
    hi = np.asarray(v, np.float16).astype(np.float64)
    lo = np.asarray(v - hi, np.float16).astype(np.float64)
    return hi, lo
def mm(a, w, mode):               # a [B,K], w [G,K]
    if mode == "fp64": return a @ w.T
    if mode == "fp32": return f32(a @ w.T)
    ah, al = split(a); wh, wl = split(w)
    if mode == "split4": return f32(ah @ wh.T + ah @ wl.T + al @ wh.T + al @ wl.T)
    return f32(ah @ wh.T + ah @ wl.T + al @ wh.T)
def act(pre, c, H, mode):
    i, f, g, o = pre[:, :H], pre[:, H:2*H], pre[:, 2*H:3*H], pre[:, 3*H:]
    if mode == "fp64":
        sg = lambda v: 1/(1+np.exp(-v)); cn = sg(f)*c + sg(i)*np.tanh(g); return cn, sg(o)*np.tanh(cn)
    if mode == "std":
        sg = lambda v: f32(1/(1+f32(np.exp(-v)))); cn = f32(sg(f)*c + f32(sg(i)*f32(np.tanh(g)))); return cn, f32(sg(o)*f32(np.tanh(cn)))
    L2 = float(np.float32(1.4426950408889634))
    ex2 = lambda a: f32(2.0 ** f32(np.minimum(a, 40.0)))
    ei, ef = ex2(f32(-L2*i)), ex2(f32(-L2*f)); eg, eo = ex2(f32(-2*L2*g)), ex2(f32(-L2*o))
    dig = f32(f32(1+ei)*f32(1+eg)); df = f32(1+ef)
    num = f32(c*dig + f32(f32(1-eg)*df))
    cn = f32(num * f32(1/f32(df*dig)))
    ec = ex2(f32(-2*L2*cn)); dh = f32(f32(1+eo)*f32(1+ec))
    return cn, f32(f32(1-ec)*f32(1/dh))
def run(mm_mode, act_mode):
    B, T, _ = X.shape; H = 48
    inp = X
    for l in range(2):
        wi, wh = ck[f"lstm.weight_ih_l{l}"], ck[f"lstm.weight_hh_l{l}"]
        if l == 0 and mm_mode.startswith("split"): wi_s, xs = wi*16, inp/16
        else: wi_s, xs = wi, inp
        b = ck[f"lstm.bias_ih_l{l}"] + ck[f"lstm.bias_hh_l{l}"]
        if mm_mode != "fp64": b = f32(b)
        if mm_mode.startswith("split"): bh, bl = split(b); b = bh + bl
        h = np.zeros((B, H)); c = np.zeros((B, H)); outs = []
        for t in range(T):
            pre = mm(xs[:, t], wi_s, mm_mode) + mm(h, wh, mm_mode) + b
            if mm_mode != "fp64": pre = f32(pre)
            c, h = act(pre, c, H, act_mode); outs.append(h)
        inp = np.stack(outs, 1)
    return inp
ref = run("fp64", "fp64")
np.seterr(over="ignore")
for mmm, am in [("split", "alg"), ("split", "std"), ("split4", "std"), ("fp32", "alg"), ("fp32", "std")]:
    o = run(mmm, am); print(mmm, am, np.abs(o - ref).max() / np.abs(ref).max(), flush=True)
