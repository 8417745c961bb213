"""Cost of EEG_LSTM.decode_intermediates against decode at the bench's workload (40,960 seeded windows of 625 x 8, the
shipped checkpoint), on both flagship tiers: whole call, each kernel alone (CUDA events), and the attention softmax pass
in GB/s (it reads the [T][B] scores three times and writes the [B][T] weights once).  Prints one JSON object; the card
name and power limit are read in the same run.

    python scripts/time_intermediates.py [--windows 40960] [--reps 20]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench                                                     # noqa: E402  (synth_windows, load_checkpoint)
from neural_speech_decoding_b200 import ops                      # noqa: E402
from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                       # pragma: no cover - depends on the host
        return {"name": torch.cuda.get_device_name(), "power_limit": f"not read ({e})"}


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    samples = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        samples.append(e0.elapsed_time(e1))
    samples.sort()
    return {"median_ms": samples[len(samples) // 2], "min_ms": samples[0], "max_ms": samples[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=40960)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_intermediates.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    m = EEG_LSTM().to(dev).eval()
    m.load_state_dict(bench.load_checkpoint(), strict=True)
    N = args.windows
    x = bench.synth_windows(N, seed=1000).to(dev)               # 819 MB at 40,960 windows: larger than the L2
    T = x.shape[1]
    head = [ops._f32c(t) for t in m._head_params()]
    res = {"card": card(), "windows": N, "T": T, "tiers": {}}
    with torch.inference_mode():
        for tier, dtype in (("exact", torch.float32), ("16-bit", torch.bfloat16)):
            m.compute_dtype = dtype
            r = {"decode": time_ms(lambda: m.decode(x, want_probs=True), args.reps),
                 "decode_intermediates": time_ms(lambda: m.decode_intermediates(x), args.reps)}
            if tier == "exact":
                pk = m._packed_x3()
                r["kernel_default"] = time_ms(lambda: ops.decoder_infer_x3(x, pk, head, True), args.reps)
                r["kernel_ex"] = time_ms(lambda: ops.decoder_infer_x3_ex(x, pk, head), args.reps)
                sc = ops.decoder_infer_x3_ex(x, pk, head)[2]
            else:
                pk = m._packed_tc()
                r["kernel_default"] = time_ms(lambda: ops.decoder_infer_bf16_x32(x, pk, head, True), args.reps)
                r["kernel_ex"] = time_ms(lambda: ops.decoder_infer_bf16_x32_ex(x, pk, head), args.reps)
                sc = ops.decoder_infer_bf16_x32_ex(x, pk, head)[2]
            sm = time_ms(lambda: ops.attention_softmax(sc), args.reps * 5)
            nbytes = 4 * T * N * 4                               # 3 reads of the scores + 1 write of the weights
            sm["bytes"] = nbytes
            sm["GB_per_s"] = nbytes / (sm["median_ms"] * 1e-3) / 1e9
            r["attention_softmax_kernel"] = sm
            r["overhead_vs_decode"] = r["decode_intermediates"]["median_ms"] / r["decode"]["median_ms"] - 1.0
            res["tiers"][tier] = r
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
