"""Cost of input attributions at the flagship shape: EEG_LSTM.input_gradients on the exact tensor-core path against the
FFMA fallback (ops.EXACT_TC_TRAIN = False), alternated in one run, with decode for scale; integrated gradients of the 324
shipped windows at steps = 32; and the layer-0 BPTT kernel with and without its dx MMAs (lstm_bwd_x3 vs lstm_bwd_x3_dx at
the same size).  16,384 seeded windows of 625 x 8, the shipped checkpoint, CUDA events.  Prints one JSON object; the
card's name, power limit and SM clocks are read in the same run.

    python scripts/time_attribution.py [--windows 16384] [--reps 5]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench                                                     # noqa: E402  (synth_windows, load_checkpoint)
from neural_speech_decoding_b200 import ops                      # noqa: E402
from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock, max_clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_clock": clock, "max_sm_clock": max_clock}
    except Exception as e:                                       # pragma: no cover - depends on the host
        return {"name": torch.cuda.get_device_name(), "power_limit": f"not read ({e})"}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def stats(samples):
    s = sorted(samples)
    return {"median_ms": s[len(s) // 2], "min_ms": s[0], "max_ms": s[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_attribution.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    m = EEG_LSTM().to(dev).eval()
    m.load_state_dict(bench.load_checkpoint(), strict=True)
    N = args.windows
    x = bench.synth_windows(N, seed=1000).to(dev)
    res = {"card": card(), "windows": N, "T": int(x.shape[1]), "reps": args.reps}

    def fast():
        m.input_gradients(x)

    def ffma():
        saved = ops.EXACT_TC_TRAIN
        ops.EXACT_TC_TRAIN = False
        try:
            m.input_gradients(x)
        finally:
            ops.EXACT_TC_TRAIN = saved

    def decode():
        m.decode(x, want_probs=False)

    for fn in (fast, ffma, decode):                              # warm-up of every shape
        fn()
    torch.cuda.synchronize()
    t = {"fast": [], "ffma": [], "decode": []}
    for _ in range(args.reps):                                   # alternated
        for name, fn in (("fast", fast), ("ffma", ffma), ("decode", decode)):
            t[name].append(timed(fn))
    for name in t:
        res[f"{name}_ms"] = stats(t[name])
        res[f"{name}_windows_per_s"] = N / (res[f"{name}_ms"]["median_ms"] * 1e-3)

    # integrated gradients: the shipped windows, steps = 32 (one batch of 324 x 33 windows)
    X = torch.from_numpy(np.load(ROOT / "tests" / "golden" / "eeg_windows.npz")["X"].copy()).to(dev)
    ig = lambda: m.integrated_gradients(X, steps=32)
    ig()
    res["ig_324x32_ms"] = stats([timed(ig) for _ in range(args.reps)])

    # the layer-0 BPTT with and without the dx MMAs, same inputs (the forward and layer 1 run once, outside the timing)
    lstm_flat = [p.detach() for l in range(2) for p in m.lstm.layer(l)]
    head = [ops._f32c(p.detach()) for p in m._head_params()]
    with torch.no_grad():
        logits, saves, _, meta = ops._x3_forward(x, lstm_flat, head, 0.0, False, None, None, None)
        xs, h0, _, c0, h1, c1, packed, st, zpool = saves
        B, hs = meta[1], meta[5]
        dl = torch.zeros_like(logits).scatter_(1, logits.argmax(dim=1)[:, None], 1.0)
        dz, _ = ops.head_tail_bwd(dl, zpool, head, None, None, 1.0)
        dz, inv = ops._scale_dz_rows(dz)
        din1 = ops.lstm_bwd_x3_dx(1, h0, h1, c1, None, packed, [dz, st, zpool, head[0], head[1]], None, B, hs)
        del h1, c1
        wg = lambda: ops.lstm_bwd_x3(0, xs, h0, c0, din1, packed, None, 0, 65536, 1.0, [], B, hs)
        dx = lambda: ops.lstm_bwd_x3_dx(0, xs, h0, c0, din1, packed, [], inv, B, hs)
        wg(), dx()
        torch.cuda.synchronize()
        k = {"bwd_l0_weight_grad_outputs": [], "bwd_l0_dx": []}
        for _ in range(args.reps):
            k["bwd_l0_weight_grad_outputs"].append(timed(wg))
            k["bwd_l0_dx"].append(timed(dx))
    for name in k:
        res[f"{name}_ms"] = stats(k[name])
    print(json.dumps(res))


if __name__ == "__main__":
    main()
