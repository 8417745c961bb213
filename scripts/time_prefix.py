"""Cost of EEG_LSTM.decode_prefixes against decode at the bench's workload (40,960 seeded windows of 625 x 8, the shipped
checkpoint, exact tier): decode(x), decode_prefixes(x, stride) at stride 1, 25 and 125, the naive loop of one decode call
per prefix at stride 125, and the two kernels of the exact path alone (the prefix pool and the head tail over the B * P
pooled rows).  CUDA-event medians, the paths alternated in one process (one sample of each per round).  Prints one JSON
object; the card name, power limit and max SM clock are read in the same run.

    python scripts/time_prefix.py [--windows 40960] [--reps 15]
    python scripts/time_prefix.py --profile DIR      # a separate run: torch.profiler of decode and decode_prefixes at
                                                     # stride 1 and 25, per-kernel device times -> DIR/prefix_kernels.json
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


def profile(m, x, out_dir):
    """Device time per kernel of decode(x) and decode_prefixes(x, stride) at stride 1 and 25, from torch.profiler."""
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as torch_profile
    out_dir.mkdir(parents=True, exist_ok=True)
    calls = {"decode": lambda: m.decode(x, want_probs=True), "prefixes_s1": lambda: m.decode_prefixes(x, 1),
             "prefixes_s25": lambda: m.decode_prefixes(x, 25)}
    res = {"card": card(), "windows": x.shape[0], "T": x.shape[1], "kernels_us": {}}
    with torch.inference_mode():
        for name, fn in calls.items():
            fn()
            torch.cuda.synchronize()
            with torch_profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                torch.cuda.synchronize()
            res["kernels_us"][name] = {e.key: round(e.device_time_total, 1) for e in prof.key_averages()
                                       if e.device_time_total > 0}
    (out_dir / "prefix_kernels.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res, indent=1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=40960)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--profile", type=Path, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_prefix.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    m = EEG_LSTM().to(dev).eval()
    m.load_state_dict(bench.load_checkpoint(), strict=True)
    N = args.windows
    x = bench.synth_windows(N, seed=1000).to(dev)               # 819 MB at 40,960 windows: larger than the L2
    T = x.shape[1]
    head = [ops._f32c(t) for t in m._head_params()]
    pk = m._packed_x3()
    if args.profile is not None:
        return profile(m, x, args.profile)
    pooled = {s: ops.decoder_prefix_pool_x3(x, pk, head[0], head[1], s) for s in (1, 25)}

    def naive(stride):
        for t in ops.prefix_lengths(T, stride).tolist():
            m.decode(x[:, :t], want_probs=True)

    paths = {
        "decode": lambda: m.decode(x, want_probs=True),
        "prefixes_s1": lambda: m.decode_prefixes(x, 1),
        "prefixes_s25": lambda: m.decode_prefixes(x, 25),
        "prefixes_s125": lambda: m.decode_prefixes(x, 125),
        "naive_loop_s125": lambda: naive(125),
        "kernel_decode": lambda: ops.decoder_infer_x3(x, pk, head, True),
        "kernel_prefix_pool_s1": lambda: ops.decoder_prefix_pool_x3(x, pk, head[0], head[1], 1),
        "kernel_prefix_pool_s25": lambda: ops.decoder_prefix_pool_x3(x, pk, head[0], head[1], 25),
        "head_tail_s1": lambda: ops._prefix_head(pooled[1], head),
        "head_tail_s25": lambda: ops._prefix_head(pooled[25], head),
    }
    samples = {k: [] for k in paths}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.inference_mode():
        for fn in paths.values():                                # warm-up: every shape of the timed rounds
            fn()
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for k, fn in paths.items():
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                samples[k].append(e0.elapsed_time(e1))
    res = {"card": card(), "windows": N, "T": T, "reps": args.reps, "ms": {}}
    for k, v in samples.items():
        v.sort()
        res["ms"][k] = {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}
    med = {k: v["median"] for k, v in res["ms"].items()}
    res["ratio_to_decode"] = {k: med[k] / med["decode"] for k in ("prefixes_s1", "prefixes_s25", "prefixes_s125",
                                                                  "naive_loop_s125")}
    res["naive_over_prefixes_s125"] = med["naive_loop_s125"] / med["prefixes_s125"]
    # the naive loop re-runs the recurrence from step 0 for every prefix: its cost grows with sum(t_j) / T prefixes'
    # worth of decode; at stride 25 and 1 it is estimated from the per-step cost it shows at stride 125
    steps125 = float(ops.prefix_lengths(T, 125).sum()) / T
    per_window_pass = med["naive_loop_s125"] / steps125
    for s in (25, 1):
        est = per_window_pass * float(ops.prefix_lengths(T, s).sum()) / T
        res[f"naive_loop_s{s}_estimated_ms"] = est
        res[f"naive_over_prefixes_s{s}_estimated"] = est / med[f"prefixes_s{s}"]
    res["pooled_bytes_s1"] = N * T * 48 * 4
    res["pooled_bytes_s25"] = N * ops.num_prefixes(T, 25) * 48 * 4
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
