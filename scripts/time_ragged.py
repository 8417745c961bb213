"""Cost of per-row lengths in EEG_LSTM.decode / decode_stream at the bench's workload (40,960 seeded windows of 625 x 8,
the shipped checkpoint, exact tier):

* decode(x) against decode(x, lengths=625 everywhere) and decode(x, lengths=random in [1, 625]);
* the kernel alone: ops.decoder_stream_ragged_x3 (kStream + kRagged) against ops.decoder_stream_x3 (kStream) on the
  same 625-step windows from a fresh state, without the API's validation;
* a live stream of 25 polls of 0.2 s at 125 Hz: per-row chunk lengths drawn from {24, 25, 26} in one ragged call per
  poll, against uniform 25-step chunks (one plain call per poll), and against grouping the rows by length (one plain
  call per distinct length, with the state gathered and scattered per group).

The chunks, lengths and group indices are built before the timing, as a live source would deliver them.  CUDA-event
medians, the paths alternated in one process (one sample of each per round).  Prints one JSON object; the card name,
power limit and max SM clock are read in the same run.

    python scripts/time_ragged.py [--windows 40960] [--reps 9]
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
from neural_speech_decoding_b200 import ops                      # noqa: E402
from neural_speech_decoding_b200.lstm_eeg_model import DecoderState, EEG_LSTM  # noqa: E402

POLLS, POLL_STEPS = 25, (24, 25, 26)


def polls(x, seed):
    """25 polls: per-row lengths from POLL_STEPS, each poll's [B, 26, 8] chunk (NaN past a row's length) and, per distinct
    length, the row indices and their contiguous [rows, n, 8] chunk."""
    g = torch.Generator().manual_seed(seed)
    B, dev = x.shape[0], x.device
    src = torch.cat([x, x[:, :POLLS * 2]], dim=1)               # room for 25 polls of up to 26 steps
    done = torch.zeros(B, dtype=torch.int64)
    out = []
    for _ in range(POLLS):
        n = torch.tensor(POLL_STEPS)[torch.randint(0, len(POLL_STEPS), (B,), generator=g)]
        idx = (done[:, None] + torch.arange(max(POLL_STEPS))).to(dev)
        chunk = torch.gather(src, 1, idx[:, :, None].expand(-1, -1, x.shape[2])).contiguous()
        chunk[torch.arange(max(POLL_STEPS), device=dev)[None, :] >= n.to(dev)[:, None]] = float("nan")
        groups = []
        for k in POLL_STEPS:
            rows = (n == k).nonzero().squeeze(1).to(dev)
            groups.append((rows, chunk[rows, :k].contiguous()))
        out.append((n, chunk, groups))
        done += n
    return out


def run_ragged(m, ps):
    state = None
    for n, chunk, _ in ps:
        state = m.decode_stream(chunk, state, lengths=n).state
    return state


def run_uniform(m, chunks):
    state = None
    for c in chunks:
        state = m.decode_stream(c, state).state
    return state


def run_grouped(m, ps, B, dev):
    """One plain decode_stream per distinct length of each poll, the state gathered and scattered per group."""
    state = m.initial_stream_state(B, dev)
    for _, _, groups in ps:
        new = [s.clone() for s in state]
        for rows, chunk in groups:
            sub = DecoderState(*[s[:, rows] if s.dim() == 3 else s[rows] for s in state])
            out = m.decode_stream(chunk, sub).state
            for s, o in zip(new, out):
                if s.dim() == 3:
                    s[:, rows] = o
                else:
                    s[rows] = o
        state = DecoderState(*new)
    return state


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=40960)
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_ragged.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    m = EEG_LSTM().to(dev).eval()
    m.load_state_dict(bench.load_checkpoint(), strict=True)
    N = args.windows
    x = bench.synth_windows(N, seed=1000).to(dev)               # 819 MB at 40,960 windows: larger than the L2
    T = x.shape[1]
    g = torch.Generator().manual_seed(7)
    full = torch.full((N,), T, dtype=torch.int64)
    rnd = torch.randint(1, T + 1, (N,), generator=g)
    x_rnd = x.clone()
    x_rnd[torch.arange(T, device=dev)[None, :] >= rnd.to(dev)[:, None]] = float("nan")
    packed, head = m._packed_x3(), [p.detach() for p in m._head_params()]
    full_dev = full.to(device=dev, dtype=torch.int32)
    ps = polls(x, seed=3)
    uniform = [x[:, t:t + 25].contiguous() for t in range(0, T, 25)]

    paths = {
        "decode": lambda: m.decode(x),
        "decode_lengths_full": lambda: m.decode(x, lengths=full),
        "decode_lengths_random": lambda: m.decode(x_rnd, lengths=rnd),
        "kernel_stream": lambda: ops.decoder_stream_x3(x, packed, head, None, None, None, None, None),
        "kernel_ragged": lambda: ops.decoder_stream_ragged_x3(x, packed, head, None, None, None, None, None, full_dev),
        "polls_ragged": lambda: run_ragged(m, ps),
        "polls_uniform_c25": lambda: run_uniform(m, uniform),
        "polls_grouped": lambda: run_grouped(m, ps, N, dev),
    }
    samples = {k: [] for k in paths}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.inference_mode():
        n0 = ops.launch_count()
        run_grouped(m, ps, N, dev)
        grouped_launches = ops.launch_count() - n0
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
        a, b = m.decode(x), m.decode(x, lengths=full)
        same_full = bool(torch.equal(a[0], b[0]))
    res = {"card": card(), "windows": N, "T": T, "reps": args.reps, "ms": {}}
    for k, v in samples.items():
        v.sort()
        res["ms"][k] = {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}
    med = {k: v["median"] for k, v in res["ms"].items()}
    res["decode_lengths_full_over_decode"] = med["decode_lengths_full"] / med["decode"]
    res["decode_lengths_random_over_decode"] = med["decode_lengths_random"] / med["decode"]
    res["kernel_ragged_over_stream"] = med["kernel_ragged"] / med["kernel_stream"]
    res["polls_ragged_over_uniform"] = med["polls_ragged"] / med["polls_uniform_c25"]
    res["polls_grouped_over_ragged"] = med["polls_grouped"] / med["polls_ragged"]
    res["grouped_launches_per_poll"] = grouped_launches / POLLS
    res["decode_lengths_full_bit_identical"] = same_full
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
