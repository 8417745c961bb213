"""Accuracy against decision time: the decoder's prediction on every prefix of the labelled windows, from one
EEG_LSTM.decode_prefixes pass.  For each prefix length it prints the accuracy against the filename labels and the share
of windows whose argmax already equals the one of the whole window.

    python scripts/accuracy_vs_time.py [--data tests/golden/eeg_windows.npz | CSV_DIR] [--checkpoint model.pth]
                                       [--classes food,water,backgroundnoise] [--stride 25] [--sr 125] [--json]

``--data``: what ``trainer.load_windows`` reads (a ``.npz`` with X and prefix, or a directory of ``*.csv`` windows named
``<class>_...``); windows whose prefix is not in ``--classes`` are skipped.  ``--checkpoint``: a ``state_dict`` saved by
``trainer.py`` (or ``{"state_dict": ...}``); default the shipped 3-class checkpoint.  Needs a GPU.
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM   # noqa: E402
from neural_speech_decoding_b200.trainer import DEFAULT_CLASSES, load_windows   # noqa: E402


def load_state(path):
    if path is None:
        ck = np.load(ROOT / "tests" / "golden" / "checkpoint_3class.npz")
        return {str(k): torch.from_numpy(ck[str(k)].copy()) for k in ck["__order__"]}
    state = torch.load(path, map_location="cpu")
    return state["state_dict"] if isinstance(state, dict) and "state_dict" in state else state


def model_for(state):
    """An EEG_LSTM with the shape the state_dict describes."""
    L = sum(1 for k in state if k.startswith("lstm.weight_ih_l"))
    H = state["lstm.weight_hh_l0"].shape[1]
    m = EEG_LSTM(input_size=state["lstm.weight_ih_l0"].shape[1], hidden_size=H, num_layers=L,
                 num_classes=state["fc.3.weight"].shape[0])
    m.load_state_dict(state, strict=True)
    return m


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--data", default=str(ROOT / "tests" / "golden" / "eeg_windows.npz"))
    ap.add_argument("--checkpoint", default=None)
    ap.add_argument("--classes", default=",".join(DEFAULT_CLASSES))
    ap.add_argument("--stride", type=int, default=25, help="prefix stride in samples (25 = 0.2 s at 125 Hz)")
    ap.add_argument("--sr", type=float, default=125.0, help="sampling rate in Hz (625 samples = 5 s)")
    ap.add_argument("--json", action="store_true", help="one JSON object instead of the table")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("accuracy_vs_time.py runs the decoder on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    classes = [c.strip() for c in args.classes.split(",") if c.strip()]
    X, y = load_windows(args.data, classes)
    m = model_for(load_state(args.checkpoint)).to(dev).eval()
    if m.fc[3].out_features != len(classes):
        raise SystemExit(f"the checkpoint has {m.fc[3].out_features} classes, --classes names {len(classes)}")
    out = m.decode_prefixes(torch.from_numpy(X).to(dev), args.stride)
    pred = out.logits.argmax(dim=2).cpu()                      # [N, P]
    labels = torch.from_numpy(y)
    acc = (pred == labels[:, None]).double().mean(dim=0)
    agree = (pred == pred[:, -1:]).double().mean(dim=0)
    rows = [{"samples": int(t), "seconds": t / args.sr, "accuracy": float(a), "agrees_with_full": float(g)}
            for t, a, g in zip(out.lengths.tolist(), acc, agree)]
    if args.json:
        print(json.dumps({"data": args.data, "checkpoint": args.checkpoint or "shipped", "windows": len(y),
                          "classes": classes, "stride": args.stride, "prefixes": rows}, indent=1))
        return
    print(f"{len(y)} windows of {X.shape[1]} samples, classes {classes}, checkpoint {args.checkpoint or 'shipped'}")
    print(f"{'samples':>8} {'seconds':>8} {'accuracy':>9} {'agrees with full window':>24}")
    for r in rows:
        print(f"{r['samples']:8d} {r['seconds']:8.2f} {r['accuracy']:9.4f} {r['agrees_with_full']:24.4f}")


if __name__ == "__main__":
    main()
