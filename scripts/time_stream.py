"""Cost of EEG_LSTM.decode_stream at the bench's workload (40,960 seeded windows of 625 x 8, the shipped checkpoint, exact
tier): the whole window streamed in chunks of 625, 125, 25 and 5 steps (summed over the calls), against decode(x) and
against decode_prefixes(x, chunk), which computes the same logits offline; the naive growing-window loop (one decode of
x[:, :t] per chunk end) at chunk 125; and the latency of one 25-step call at B = 1 and at B = 18,944 (one round of full
tiles on 148 SMs).  The chunks are contiguous tensors sliced before the timing, as a live source would deliver them.
CUDA-event medians, the paths alternated in one process (one sample of each per round).  Prints one JSON object; the
card name, power limit and max SM clock are read in the same run.

    python scripts/time_stream.py [--windows 40960] [--reps 9]
    python scripts/time_stream.py --profile DIR      # a separate run: torch.profiler of decode and of the stream at
                                                     # chunk 25 and 5, per-kernel device times -> DIR/stream_kernels.json
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
from time_prefix import card                                     # noqa: E402
from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM  # noqa: E402

CHUNKS = (625, 125, 25, 5)


def chunked(x, n):
    return [x[:, t:t + n].contiguous() for t in range(0, x.shape[1], n)]


def run_stream(m, chunks):
    state = None
    for c in chunks:
        out = m.decode_stream(c, state)
        state = out.state
    return out


def profile(m, x, out_dir):
    """Device time per kernel of decode(x) and of streaming x in chunks of 25 and 5 steps, from torch.profiler."""
    from torch.profiler import ProfilerActivity
    from torch.profiler import profile as torch_profile
    out_dir.mkdir(parents=True, exist_ok=True)
    parts = {n: chunked(x, n) for n in (25, 5)}
    calls = {"decode": lambda: m.decode(x, want_probs=True), "stream_c25": lambda: run_stream(m, parts[25]),
             "stream_c5": lambda: run_stream(m, parts[5])}
    res = {"card": card(), "windows": x.shape[0], "T": x.shape[1], "kernels_us": {}, "wall_ms": {}}
    with torch.inference_mode():
        for name, fn in calls.items():
            fn()
            torch.cuda.synchronize()
            with torch_profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
                fn()
                torch.cuda.synchronize()
            res["kernels_us"][name] = {e.key: {"device_us": round(e.device_time_total, 1), "count": e.count}
                                       for e in prof.key_averages() if e.device_time_total > 0}
    (out_dir / "stream_kernels.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res, indent=1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=40960)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--profile", type=Path, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_stream.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    m = EEG_LSTM().to(dev).eval()
    m.load_state_dict(bench.load_checkpoint(), strict=True)
    N = args.windows
    x = bench.synth_windows(N, seed=1000).to(dev)               # 819 MB at 40,960 windows: larger than the L2
    T = x.shape[1]
    if args.profile is not None:
        return profile(m, x, args.profile)
    parts = {n: chunked(x, n) for n in CHUNKS}
    full = 148 * 128
    lat = {}
    for B in (1, full):                                         # the state after 100 steps, and the next 25-step chunk
        xb = x[:B] if B <= N else x.repeat((B + N - 1) // N, 1, 1)[:B]
        lat[B] = (m.decode_stream(xb[:, :100].contiguous()).state, xb[:, 100:125].contiguous())

    def naive(n):
        for t in range(n, T + 1, n):
            m.decode(x[:, :t], want_probs=True)

    paths = {"decode": lambda: m.decode(x, want_probs=True)}
    for n in CHUNKS:
        paths[f"stream_c{n}"] = (lambda n: lambda: run_stream(m, parts[n]))(n)
        paths[f"prefixes_s{n}"] = (lambda n: lambda: m.decode_prefixes(x, n))(n)
    paths["naive_loop_c125"] = lambda: naive(125)
    for B, (st, c) in lat.items():
        paths[f"call_c25_B{B}"] = (lambda st, c: lambda: m.decode_stream(c, st))(st, c)
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
    res["stream_over_decode"] = {n: med[f"stream_c{n}"] / med["decode"] for n in CHUNKS}
    res["stream_over_prefixes"] = {n: med[f"stream_c{n}"] / med[f"prefixes_s{n}"] for n in CHUNKS}
    res["stream_per_call_ms"] = {n: med[f"stream_c{n}"] / len(parts[n]) for n in CHUNKS}
    res["naive_loop_c125_over_stream_c125"] = med["naive_loop_c125"] / med["stream_c125"]
    res["targets"] = {"c125_within_1.1x_decode": res["stream_over_decode"][125] <= 1.1,
                      "c25_within_1.5x_decode": res["stream_over_decode"][25] <= 1.5}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
