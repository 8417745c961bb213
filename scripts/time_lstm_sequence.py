"""Cost of ``model.lstm(x)`` (nn.LSTM's contract, sequence output) at the bench's workload: 40,960 seeded windows of
625 x 8 and the shipped checkpoint, eval mode without autograd.  Medians of CUDA-event timings for the fused exact-tier
kernel (``na_decoder_lstm_x3``), for ``decode(x)`` (the same kernel with pooling and head instead of the sequence
stores) and for the FFMA path of the same call (``ops.EXACT_TC = False``), the write rate of the [B,T,48] fp32 output,
and the largest difference between the two paths.  Prints one JSON object; the card name and power limit are read in
the same run.

    python scripts/time_lstm_sequence.py [--windows 40960] [--reps 20]
"""
import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))
import bench                                                     # noqa: E402  (synth_windows, load_checkpoint)
from neural_speech_decoding_b200 import ops                      # noqa: E402
from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM  # noqa: E402
from time_intermediates import card, time_ms                     # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=40960)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_lstm_sequence.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    m = EEG_LSTM().to(dev).eval()
    m.load_state_dict(bench.load_checkpoint(), strict=True)
    N = args.windows
    x = bench.synth_windows(N, seed=1000).to(dev)               # 819 MB in, 4.9 GB out: larger than the L2
    T = x.shape[1]
    out_bytes = N * T * 48 * 4
    res = {"card": card(), "windows": N, "T": T, "output_bytes": out_bytes}
    with torch.inference_mode():
        fused = time_ms(lambda: m.lstm(x), args.reps)
        fused["output_GB_per_s"] = out_bytes / (fused["median_ms"] * 1e-3) / 1e9
        res["lstm_fused"] = fused
        res["decode"] = time_ms(lambda: m.decode(x, want_probs=True), args.reps)
        a = m.lstm(x)
        ops.EXACT_TC = False
        try:
            res["lstm_ffma"] = time_ms(lambda: m.lstm(x), max(3, args.reps // 4), warmup=1)
            b = m.lstm(x)
        finally:
            ops.EXACT_TC = True
        res["fused_speedup_vs_ffma"] = res["lstm_ffma"]["median_ms"] / fused["median_ms"]
        res["fused_vs_decode"] = fused["median_ms"] / res["decode"]["median_ms"]
        res["max_rel_diff_fused_vs_ffma"] = {
            name: float((p - q).abs().max() / q.abs().max()) for name, p, q in
            (("output", a[0], b[0]), ("h_n", a[1][0], b[1][0]), ("c_n", a[1][1], b[1][1]))}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
