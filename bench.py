#!/usr/bin/env python
"""Headline benchmark of the NeuroAlpha decoder hot path (BASELINE.json: "EEG windows/sec").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic EEG: BASELINE.json configs[1],
i.e. R=10 trials x B=4096 sessions of [625,8] windows per GPU (40,960 windows), decoder forward +
class softmax + run_trials' 10-trial probability averaging, fp32, shipped 3-class weights.

  value : windows/s with the windows already resident in HBM (CUDA events, max over ranks), measured on the
          fp32-contract tier (decoder_infer_x3_kernel: fp32-accurate tcgen05, every operand split into fp16 hi + lo,
          1e-5 parity) -- the reference's arithmetic is fp32, so this is the like-for-like headline; the 16-bit tier
          (north_star's "bf16 path", IEEE fp16 operands, 2e-2 contract) is the named extra "fp16_tier"
  e2e   : the same through the public host API (run_trials_batched on PINNED HOST windows):
          H2D of every trial + D2H of the averaged probabilities inside the timed region
  roofline / cpu_baseline / clocks / gpu_launches / train : see DESIGN.md "Measurement"

Multi-GPU (torchrun, one rank per GPU): inference shards by batch with no data-path collective
(weak scaling: every rank decodes its own 40,960 windows); the "train" leg is data-parallel with
one flat NCCL gradient all-reduce.

--impl reference times the reference's CPU implementation of the same path on the host cores
(oracle/torch_ref.py RefEEGLSTM -- the reference module restated from the same torch building
blocks; the reference itself is Python and /root/reference does not exist on the GPU box).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

T, C, H, NC = 625, 8, 48, 3
R_TRIALS, B_SESSIONS = 10, 4096
FWD_FLOPS_PER_WINDOW = 36_603_264            # SURVEY 8(a), base K=3
FWDBWD_FLOPS_PER_WINDOW = 107_889_792
L1_KERNEL_FLOPS_PER_WINDOW = 2 * (48 + 48) * 192 * T      # layer-1 recurrence kernel: [x_t|h] . W, K=96
L0_KERNEL_FLOPS_PER_WINDOW = 2 * (8 + 48) * 192 * T
INPUT_SIGMA = 2.73                            # matches the CSV corpus (SURVEY 8d)
NCU_TRAFFIC_BYTES_40960 = 823.51e6 + 7.36e6   # dram__bytes_read.sum + dram__bytes_write.sum, profiles/r1_tc2_fused_ncu_full.csv
# the same two counters for decoder_infer_x3_kernel (one launch over 40,960 windows)
NCU_TRAFFIC_BYTES_40960_X3 = 823.19e6 + 5.96e6
NCU_TRAFFIC_SOURCE_X3 = "profiles/r2_x3_ncu_full.csv"


def load_checkpoint():
    ck = np.load(ROOT / "tests" / "golden" / "checkpoint_3class.npz")
    return {str(k): torch.from_numpy(ck[str(k)].copy()) for k in ck["__order__"]}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [s.strip() for s in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def synth_windows(n, seed, pin=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.empty((n, T, C), dtype=torch.float32, pin_memory=pin)
    chunk = 4096
    for i in range(0, n, chunk):
        x[i:i + chunk] = torch.randn((min(chunk, n - i), T, C), generator=g) * INPUT_SIGMA
    return x


# ---------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference)
# ---------------------------------------------------------------------------------------------
def cpu_decode_pass(model, x_rb, R, B):
    """One bounded sample of the workload on the host: R x B windows, chunks of 512, softmax,
    10-trial mean (tester.py:89,97 semantics)."""
    from oracle import trial_mean
    probs = []
    with torch.inference_mode():
        for i in range(0, x_rb.shape[0], 512):
            probs.append(torch.softmax(model(x_rb[i:i + 512]), dim=-1))
    p = torch.cat(probs).numpy().reshape(R, B, NC)
    return trial_mean(p)


def cpu_arm(steps, warmup, R=10, B=256):
    from oracle.torch_ref import RefEEGLSTM
    torch.set_num_threads(os.cpu_count() or 1)
    m = RefEEGLSTM().eval()
    m.load_state_dict(load_checkpoint(), strict=True)
    x = synth_windows(R * B, seed=0)
    for _ in range(warmup):
        cpu_decode_pass(m, x, R, B)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cpu_decode_pass(m, x, R, B)
        times.append(time.perf_counter() - t0)
    return {"windows_per_s": R * B / statistics.median(times), "ms_per_step": 1e3 * statistics.median(times),
            "cores": torch.get_num_threads(), "sample": f"{R} trials x {B} sessions = {R * B} windows [625,8] per step, "
            f"chunks of 512, fp32, median of {steps} after {warmup} warm-up", "times": times}


def cpu_train_arm(B=512, reps=3):
    """SURVEY 8(d): the reference module's train step on the host -- B = 512, train mode (dropout, RReLU noise),
    mean cross-entropy, Adam lr 1e-3; one warm-up, median of ``reps``."""
    from oracle.torch_ref import RefEEGLSTM
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    m = RefEEGLSTM().train()
    m.load_state_dict(load_checkpoint(), strict=True)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    x = synth_windows(B, seed=2000)
    y = torch.randint(0, NC, (B,), generator=torch.Generator(device="cpu").manual_seed(1))
    times = []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        opt.zero_grad()
        torch.nn.functional.cross_entropy(m(x), y).backward()
        opt.step()
        if i:
            times.append(time.perf_counter() - t0)
    return {"value": B / statistics.median(times), "unit": "windows/s", "ms_per_step": 1e3 * statistics.median(times),
            "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"one train step of B={B} windows [625,8] (fwd + bwd + Adam), train mode, fp32, median of {reps} after 1 warm-up"}


def config1_labels():
    d = np.load(ROOT / "tests" / "golden" / "eeg_windows.npz")
    idx = {"food": 0, "water": 1, "backgroundnoise": 2}           # CLASS_NAMES order (lstm_eeg_model.py:11); yes / no excluded
    keep = [i for i, s in enumerate(d["prefix"]) if str(s) in idx]
    return d["X"], np.array(keep), np.array([idx[str(d["prefix"][i])] for i in keep], dtype=np.int64)


def config1_epoch(model, X, keep, y, to_dev):
    """BASELINE configs[0]: fp32 forward over all 324 repo windows + one training epoch (the 179 three-class windows,
    batch 32, CE, Adam lr 1e-3 -- the recipe is ours, SURVEY F2).  Returns (forward seconds, epoch seconds, last loss)."""
    sync = torch.cuda.synchronize if to_dev is not None else (lambda: None)
    xa = torch.from_numpy(X)
    model.eval()
    sync(); t0 = time.perf_counter()
    with torch.inference_mode():
        xin = xa.to(to_dev) if to_dev is not None else xa
        out = model(xin)
        out = out.cpu() if to_dev is not None else out
    sync(); t_fwd = time.perf_counter() - t0
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    order = np.random.default_rng(0).permutation(len(keep))
    sync(); t0 = time.perf_counter()
    loss = None
    for s0 in range(0, len(order), 32):
        ix = order[s0:s0 + 32]
        xb, yb = torch.from_numpy(X[keep[ix]]), torch.from_numpy(y[ix])
        if to_dev is not None:
            xb, yb = xb.to(to_dev), yb.to(to_dev)
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(model(xb), yb)
        loss.backward()
        opt.step()
    last = float(loss.item())
    sync(); t_ep = time.perf_counter() - t0
    return t_fwd, t_ep, last


def config1_leg(dev):
    """configs[0] on both sides in the same run: the CPU port and this module (exact tier) on the repo's own windows."""
    from oracle.torch_ref import RefEEGLSTM
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    X, keep, y = config1_labels()
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    ref = RefEEGLSTM()
    ref.load_state_dict(load_checkpoint(), strict=True)
    cf, ce, cl = config1_epoch(ref, X, keep, y, None)
    torch.manual_seed(0)
    m = EEG_LSTM().to(dev)
    m.load_state_dict(load_checkpoint(), strict=True)
    config1_epoch(m, X, keep, y, dev)                      # warm-up (allocator, weight packs)
    m.load_state_dict(load_checkpoint(), strict=True)
    gf, ge, gl = config1_epoch(m, X, keep, y, dev)
    return {"workload": "configs[0]: fp32 forward over the 324 EEG_data_collection windows + one training epoch over the 179 "
                        "food / water / backgroundnoise windows (batch 32, CE, Adam lr 1e-3), shipped .pth weights",
            "cpu": {"forward_ms": 1e3 * cf, "forward_windows_per_s": 324 / cf, "epoch_ms": 1e3 * ce,
                    "epoch_windows_per_s": len(keep) / ce, "cores": torch.get_num_threads(), "kind": "port", "last_loss": cl},
            "gpu": {"forward_ms": 1e3 * gf, "forward_windows_per_s": 324 / gf, "epoch_ms": 1e3 * ge,
                    "epoch_windows_per_s": len(keep) / ge, "tier": "exact (fp32 contract)", "last_loss": gl,
                    "timing": "host wall clock incl. H2D / D2H and optimizer (6 steps of <= 32 windows: launch-latency bound)"}}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_arm(max(1, args.steps), max(1, args.warmup))
    line = {
        "impl": "reference", "metric": "EEG windows/sec (decoder fwd + softmax + 10-trial mean)",
        "value": r["windows_per_s"], "unit": "windows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: 3-class decoder inference + 10-trial averaging, bounded CPU sample",
                   "trials": 10, "sessions": 256, "T": T, "C": C},
        "cpu_baseline": {"value": r["windows_per_s"], "unit": "windows/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["windows_per_s"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
NUMA_BINDING = [None]


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        # each rank on the CPUs (and the NUMA node) next to its GPU: the e2e leg's pinned buffers are first-touched there
        from neural_speech_decoding_b200.dp import bind_to_gpu_numa
        NUMA_BINDING[0] = bind_to_gpu_numa(local)
        # NCCL prints its version banner on STDOUT when the communicator is created; stdout must carry
        # exactly one JSON line, so fd 1 points at stderr until the first collective has run.
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            t = torch.zeros(1, device=torch.device("cuda", local))
            dist.all_reduce(t)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    return world, rank, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(v, world, dev):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return v


def time_steps(fn, steps, warmup, world, dev):
    for _ in range(warmup):
        fn()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier(world)
    return max_over_ranks(e0.elapsed_time(e1), world, dev)      # ms, max over ranks


def h2d_ceiling(host, dev, world, reps=3):
    """Platform ceiling of the e2e leg: every rank copies its pinned 819 MB step input with plain cudaMemcpyAsync at the
    same time (barrier, CUDA events, max over ranks).  Aggregate GB/s = world x bytes / time."""
    buf = torch.empty_like(host, device=dev)
    def cp():
        buf.copy_(host, non_blocking=True)
    ms = time_steps(cp, reps, 1, world, dev) / reps
    del buf
    return {"per_gpu_gbs": host.numel() * 4 / (ms * 1e-3) / 1e9, "aggregate_gbs": world * host.numel() * 4 / (ms * 1e-3) / 1e9,
            "ms_per_copy": ms, "bytes_per_gpu": host.numel() * 4, "concurrent_ranks": world,
            "what": "all ranks copy their pinned step input at once (cudaMemcpyAsync, one call), max over ranks"}


def run_gpu_arm(args):
    from neural_speech_decoding_b200 import _lib, ops
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    from neural_speech_decoding_b200.tester import run_trials_batched
    _lib.load()                                     # fail loudly without the CUDA library
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    peaks = measured_peaks()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count

    model = EEG_LSTM().to(dev).eval()
    model.load_state_dict(load_checkpoint(), strict=True)
    R, B = R_TRIALS, B_SESSIONS
    n_win = R * B
    host = synth_windows(n_win, seed=1000 + rank, pin=True).reshape(R, B, T, C)
    x_dev = host.to(dev)                            # 819 MB per rank: larger than the 126 MB L2
    x_flat = x_dev.reshape(n_win, T, C)

    def step_device():
        with torch.inference_mode():
            logits, p = model.decode(x_flat, want_probs=True)
            return {"logits": logits, "probs": p, "avg_probs": ops.trial_mean(p.reshape(R, B, NC))}

    def step_e2e():
        return run_trials_batched(host, model)      # pinned host in, numpy out

    def measure(dtype):
        model.compute_dtype = dtype
        sampler = ClockSampler(local).start() if rank == 0 else None
        last = [None]                               # what the last step returned (--dump-outputs)

        def step():
            last[0] = step_device()
        for _ in range(args.warmup):
            step()
        l0 = ops.launch_count()
        ms = time_steps(step, args.steps, 0, world, dev)
        launches = ops.launch_count() - l0
        clocks = sampler.stop() if sampler else None
        e_steps = max(1, min(args.steps, 10))
        ms_e2e = time_steps(step_e2e, e_steps, 2, world, dev)
        return {"value": world * n_win * args.steps / (ms * 1e-3), "ms_per_step": ms / args.steps,
                "e2e_value": world * n_win * e_steps / (ms_e2e * 1e-3), "e2e_ms_per_step": ms_e2e / e_steps,
                "launches": launches, "clocks": clocks, "outputs": last[0]}

    fp = measure(torch.float32)                     # fp32-contract tier: the headline (the reference computes in fp32)
    h16 = measure(torch.bfloat16)                   # 16-bit tensor-core tier (fp16 operands, 2e-2 contract): named extra
    ceiling = h2d_ceiling(host, dev, world)

    # ---- dominant kernels alone, CUDA events on the launching stream -------------------------------
    reps = max(3, min(args.steps, 10))
    n_full, n_short = sms * 128, sms * 32           # one full round of 128-window tiles / one round of row-replicated quarter tiles
    with torch.inference_mode():
        head = model._head_params()
        packed_x3 = model._packed_x3()
        ms_x3 = time_steps(lambda: ops.decoder_infer_x3(x_flat, packed_x3, head, True), reps, 2, 1, dev) / reps
        ms_x3_full = time_steps(lambda: ops.decoder_infer_x3(x_flat[:n_full], packed_x3, head, True), reps, 2, 1, dev) / reps
        ms_x3_short = time_steps(lambda: ops.decoder_infer_x3(x_flat[:n_short], packed_x3, head, True), reps, 2, 1, dev) / reps
        model.compute_dtype = torch.bfloat16
        xt16 = ops.window_zscore(x_flat, T, T, False, True, ops.NA_F16, ops.TC_TILE)
        packed_tc = model._packed_tc()
        ms_tc_tm = time_steps(lambda: ops.decoder_infer_bf16(xt16, packed_tc, head, n_win, True), reps, 2, 1, dev) / reps
        ms_tc = time_steps(lambda: ops.decoder_infer_bf16_x32(x_flat, packed_tc, head, True), reps, 2, 1, dev) / reps
        ms_tc_full = time_steps(lambda: ops.decoder_infer_bf16_x32(x_flat[:n_full], packed_tc, head, True), reps, 2, 1, dev) / reps
        ms_tc_short = time_steps(lambda: ops.decoder_infer_bf16_x32(x_flat[:n_short], packed_tc, head, True), reps, 2, 1, dev) / reps
        ms_pack16 = time_steps(lambda: ops.window_zscore(x_flat, T, T, False, True, ops.NA_F16, ops.TC_TILE), reps, 2, 1, dev) / reps
        ms_z = time_steps(lambda: ops.window_zscore(x_flat, T, T, True, False, False), reps, 2, 1, dev) / reps
        del xt16
        packed = [model._packed(l) for l in range(2)]
        xt = ops.window_zscore(x_flat, T, T, False, True, False)
        h0 = ops.lstm_layer_fwd(xt, packed[0][0], packed[0][1], None, 1.0, False)[0]
        del xt
        ms_l1 = time_steps(lambda: ops.lstm_layer_fwd(h0, packed[1][0], packed[1][1], None, 1.0, False)[0], 3, 1, 1, dev) / 3
        # K4 / K5 alone (SURVEY 8(d)): the standalone pooling head over a [T, Bp, 48] fp32 tensor (fused into the inference
        # kernels; standalone in the FFMA tier), and the 10-trial mean
        ms_k4 = time_steps(lambda: ops.head_fwd(h0, n_win, head, None, None, 1.0, True, False), 3, 1, 1, dev) / 3
        k4_bytes = h0.numel() * 4
        del h0
        pr = torch.rand(R, B, NC, device=dev)
        ms_k5 = time_steps(lambda: ops.trial_mean(pr), reps, 2, 1, dev) / reps
    x3_tflops = FWD_FLOPS_PER_WINDOW * n_win / (ms_x3 * 1e-3) / 1e12
    tc_tflops = FWD_FLOPS_PER_WINDOW * n_win / (ms_tc * 1e-3) / 1e12
    l1_tflops = L1_KERNEL_FLOPS_PER_WINDOW * n_win / (ms_l1 * 1e-3) / 1e12

    # ---- single-window latency: what one `SimplePredictor.predict`-style call costs (numpy [625,8] in -> probs out) ----
    def one_window_latency(dtype):
        model.compute_dtype = dtype
        w = host[0, 0].numpy()
        lat = []
        with torch.inference_mode():
            for i in range(60):
                t0 = time.perf_counter()
                xg = torch.from_numpy(w[None]).to(dev)
                _, p = model.decode(xg, want_probs=True)
                p = p[0].cpu().numpy()
                lat.append((time.perf_counter() - t0) * 1e3)
        return statistics.median(lat[10:])
    lat_exact, lat_h16 = one_window_latency(torch.float32), one_window_latency(torch.bfloat16)

    # ---- CSV ingestion kernel (SURVEY 8f rank 2): 4,096 files of the collector's format, byte work ------------------
    import io
    from neural_speech_decoding_b200 import ingest
    files = []
    for i in range(64):
        bio = io.BytesIO()
        np.savetxt(bio, host[0, i].numpy(), delimiter=",", fmt="%.7f")
        files.append(bio.getvalue())
    files = files * 64
    off = np.zeros(len(files) + 1, dtype=np.int64)
    np.cumsum([len(f) for f in files], out=off[1:])
    text_dev = torch.frombuffer(bytearray(b"".join(files)), dtype=torch.uint8).to(dev)
    off_dev = torch.from_numpy(off).to(dev)
    ms_csv = time_steps(lambda: ingest.parse_csv_bytes(text_dev, off_dev), reps, 2, 1, dev) / reps
    csv_bytes = int(off[-1]) + len(files) * T * C * 4
    del text_dev

    # ---- collector-side filter chain (SURVEY 8f rank 4): all 40,960 windows of the step ----------------------------
    from neural_speech_decoding_b200 import filters
    ms_filt = time_steps(lambda: filters.filter_windows(x_flat), 3, 1, 1, dev) / 3
    filt_bytes = n_win * C * T * (4 + 4)            # algorithmic: one fp32 read + one fp32 write per sample
    filt_flops = n_win * C * T * filters.chain_fma_per_sample() * 2
    # ---- preprocessing front stage (SURVEY 8f rank 1, opt-in): the step in front of the decoder on every live window ----
    from neural_speech_decoding_b200.preprocess_gpu import PhaseCouplingFilterGPU
    pre = PhaseCouplingFilterGPU(device=dev, accept_noncommercial_terms=True)      # benchmark of the opt-in stage
    ms_pre = time_steps(lambda: pre.transform_batch(x_flat), 3, 1, 1, dev) / 3
    pre_cpu = None
    if rank == 0 and not args.no_cpu:
        from oracle.phase_filter import phase_coupling_filter
        wins = host[0, :24].numpy()
        t0 = time.perf_counter()
        for wv in wins:
            phase_coupling_filter(wv)
        pre_cpu = len(wins) / (time.perf_counter() - t0)
    torch.cuda.empty_cache()

    # ---- measured CUDA-core fp32 peak (FFMA probe) -------------------------------------------------
    out = torch.zeros(4, device=dev)
    blocks, iters = sms * 8, 1 << 16
    def probe():
        _lib.call("na_ffma_probe", out.data_ptr(), blocks, iters, torch.cuda.current_stream().cuda_stream)
    ms_probe = time_steps(probe, 3, 2, 1, dev) / 3
    ffma_peak = blocks * 256 * 2 * 16 * iters / (ms_probe * 1e-3) / 1e12

    train = None
    if not args.no_train:
        train = train_leg(args, world, rank, dev)
    stress = stress_leg(dev, peaks) if (rank == 0 and not args.no_stress) else None
    config1 = config1_leg(dev) if (rank == 0 and not args.no_cpu) else None

    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**fp["outputs"], **{f"fp16_tier_{k}": v for k, v in h16["outputs"].items()}})
    # the CPU arm runs on rank 0 after every timed GPU region (it would perturb the other ranks' host threads otherwise)
    cpu = cpu_arm(3, 1) if not args.no_cpu else None
    cpu_train = cpu_train_arm() if (not args.no_cpu and not args.no_train) else None
    peak = peaks["bf16_tflops"]     # the kernel is timed alone -> burst figure
    e2e_bytes = n_win * T * C * 4
    line = {
        "metric": "EEG windows/sec (decoder fwd + softmax + 10-trial mean)", "value": fp["value"], "unit": "windows/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": fp["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32-accurate (tcgen05: every operand split into fp16 hi + lo, 3 MMAs per product, fp32 accumulate; "
                 "fp32 cell state / pooling / head; ex2 + rcp activations) -- 1e-5 contract vs the fp32 reference",
        "data": "synthetic",
        "config": {"workload": "configs[1]: 3-class decoder (T=625,C=8,H=48,L=2) batched inference + run_trials "
                               "10-trial probability averaging, shipped .pth weights",
                   "trials": R, "sessions_per_gpu": B, "windows_per_step_per_gpu": n_win,
                   "l2_policy": "inputs larger than L2 (819 MB fp32 windows per step per GPU)",
                   "parallelism": f"batch-shard x{world}, no collective",
                   "parity": "tests/test_gpu_parity.py: logits within 1e-5 of the fp32 reference, argmax identical on the 324 repo windows"},
        "e2e": {"value": fp["e2e_value"], "unit": "windows/s", "ms_per_step": fp["e2e_ms_per_step"],
                "h2d_bytes_per_step": e2e_bytes, "d2h_bytes_per_step": B * NC * 4,
                "api": "neural_speech_decoding_b200.tester.run_trials_batched(pinned host fp32 [R,B,T,C]) -> numpy [B,K]",
                "h2d_gbs_per_gpu": e2e_bytes / (fp["e2e_ms_per_step"] * 1e-3) / 1e9,
                "h2d_ceiling": ceiling,
                "frac_of_h2d_ceiling": (e2e_bytes / (fp["e2e_ms_per_step"] * 1e-3) / 1e9) / ceiling["per_gpu_gbs"],
                "rank0_cpu_binding": (f"{len(NUMA_BINDING[0])} CPUs local to the GPU (NVML affinity)" if NUMA_BINDING[0] else "none")},
        "gpu_launches": fp["launches"],
        "clocks": fp["clocks"],
        "roofline": {
            "kernel": "decoder_infer_x3_kernel (tcgen05/TMEM, fp32-accurate: K1 read + K2 + K3 + K4 fused, fp32 [B,T,8] windows -> probabilities)",
            "bound": "tensor", "achieved": x3_tflops, "peak": peak, "unit": "TFLOP/s", "frac": x3_tflops / peak,
            "peak_source": peaks["source"] + " cuBLAS bf16 (burst: kernel timed alone)",
            "issued_tflops_3x": 3 * x3_tflops,
            "traffic": NCU_TRAFFIC_BYTES_40960_X3 * n_win / 40960, "traffic_source": NCU_TRAFFIC_SOURCE_X3,
            "algorithmic_bytes_per_launch": n_win * (T * C * 4 + NC * 8),
            "algorithmic_flops_per_launch": FWD_FLOPS_PER_WINDOW * n_win,
            "ms_per_launch": ms_x3,
            # north_star's mandatory recurrence metric, both regimes: a full round of 128-window tiles (throughput regime,
            # every SM sub-partition saturated) and a round of row-replicated 32-window tiles (the dependent-chain latency)
            "per_timestep_latency_us": {"full_tile_round": ms_x3_full * 1e3 / T, "short_tile_chain": ms_x3_short * 1e3 / T,
                                        "windows_full_round": n_full, "windows_short_round": n_short,
                                        "what": "kernel time of one round / 625 steps (layer 0 and layer 1 of a step are software-pipelined)"},
            # the pipe that actually bounds the kernel: 7 MUFU per cell update (5 ex2 + 2 rcp) on the 16-lane/clk/SM pipe
            "xu_pipe": mufu_pipe(n_win, ms_x3, fp["clocks"], X3_MUFU_PER_CELL),
            "note": "MUFU-bound, not tensor-bound: 1250 dependent cell updates per window; the accurate activations cost "
                    "ex2 + rcp (tanh.approx is 5e-4) -- see DESIGN.md section 6a; the 40,960-window step is 2.16 rounds of 148 tiles, "
                    "its remainder runs as row-replicated short tiles",
            "k1_zscore_f32": {"kernel": "window_zscore_vec_kernel (z-score, fp32 in/out)", "bound": "hbm",
                              "achieved": n_win * T * C * 8 / (ms_z * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                              "unit": "GB/s", "frac": n_win * T * C * 8 / (ms_z * 1e-3) / 1e9 / peaks["hbm_gbs"]},
            "k1_window_pack": {"kernel": "window_pack16_tmp_kernel (fp32 -> time-major fp16)", "bound": "hbm",
                               "achieved": n_win * T * C * 6 / (ms_pack16 * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                               "unit": "GB/s", "frac": n_win * T * C * 6 / (ms_pack16 * 1e-3) / 1e9 / peaks["hbm_gbs"]},
            "k4_head": {"kernel": "head_fwd_kernel (attention score, online softmax over time, pooling, LayerNorm, MLP, softmax; standalone)",
                        "bound": "hbm", "achieved": k4_bytes / (ms_k4 * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": k4_bytes / (ms_k4 * 1e-3) / 1e9 / peaks["hbm_gbs"], "ms_per_launch": ms_k4,
                        "note": "h [625, Bp, 48] fp32 read once (120,000 B per window); in the tensor-core inference kernels K4 is fused and "
                                "this traffic does not exist"},
            "k5_trial_mean": {"kernel": "trial_mean_kernel (ordered fp32 sum of 10 trials, one division: tester.py:54,89,97)", "bound": "hbm",
                              "achieved": (R + 1) * B * NC * 4 / (ms_k5 * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                              "frac": (R + 1) * B * NC * 4 / (ms_k5 * 1e-3) / 1e9 / peaks["hbm_gbs"], "us_per_launch": ms_k5 * 1e3,
                              "note": "540 KB per launch: launch-latency-bound, not HBM-bound"},
            "csv_parse": {"kernel": "csv_parse_kernel (4,096 files of 625x8 '%.7f' text -> fp32; includes the status D2H check)",
                          "bound": "hbm", "achieved": csv_bytes / (ms_csv * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                          "frac": csv_bytes / (ms_csv * 1e-3) / 1e9 / peaks["hbm_gbs"], "files_per_s": 4096 / (ms_csv * 1e-3)},
            "filter_chain": {"kernel": "iir_chain_warp_kernel (detrend + 4 zero-phase Butterworth band filters, float64, one warp per "
                                       "(window, channel) series, the series lives in registers: no scratch)",
                             "bound": "hbm", "achieved": filt_bytes / (ms_filt * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": filt_bytes / (ms_filt * 1e-3) / 1e9 / peaks["hbm_gbs"], "windows_per_s": n_win / (ms_filt * 1e-3),
                             "algorithmic_bytes": filt_bytes, "fp64_tflops": filt_flops / (ms_filt * 1e-3) / 1e12,
                             "note": "8 B of DRAM traffic per sample (algorithmic); the binding pipe is fp64 FMA, not HBM",
                             "parity": "unpinned (BrainFlow absent): tests/test_filters.py vs the scipy restatement"},
            "phase_filter": {"kernel": "phase_coupling_filter_kernel (opt-in front stage: radix-5 FFT Hilbert transform, 28 pairwise phase sums, "
                                       "8x8 fp64 solve, mix; one CTA per window, float64)",
                             "bound": "hbm", "achieved": n_win * T * C * 8 / (ms_pre * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": n_win * T * C * 8 / (ms_pre * 1e-3) / 1e9 / peaks["hbm_gbs"], "windows_per_s": n_win / (ms_pre * 1e-3),
                             "ms_per_40960_windows": ms_pre,
                             "cpu_windows_per_s_per_core": pre_cpu, "cpu_kind": "port (oracle/phase_filter.py, numpy float64, one core)",
                             "note": "nominally HBM-bound byte work (40 KB per window); actually bound by fp64 arithmetic and shared-memory "
                                     "latency of the 8 FFTs per window",
                             "parity": "tests/test_phase_filter.py: the reference's own filtered windows (1e-5) and filtered-path logits"},
            "ffma_kernels": {"kernel": "lstm_fwd_h48_kernel<KIN=48> (layer-1 recurrence, exact fp32 FFMA; other shapes / A-B reference)",
                             "bound": "cuda-core fp32 (FFMA issue)", "achieved": l1_tflops, "peak": ffma_peak,
                             "unit": "TFLOP/s", "frac": l1_tflops / ffma_peak, "peak_source": "na_ffma_probe measured in this run",
                             "ms_per_launch": ms_l1},
        },
        "fp16_tier": {
            "what": "north_star's \"bf16 path\": 16-bit tensor-core tier, 2e-2 contract (secondary; NOT like-for-like with the fp32 reference)",
            "dtype": "IEEE fp16 operands (x / 16, h, weights), fp32 accumulate / cell state / pooling / head; tanh.approx activations",
            "value": h16["value"], "unit": "windows/s", "ms_per_step": h16["ms_per_step"],
            "e2e": {"value": h16["e2e_value"], "unit": "windows/s", "ms_per_step": h16["e2e_ms_per_step"]},
            "gpu_launches": h16["launches"], "clocks": h16["clocks"],
            "vs_cpu": (h16["value"] / world / cpu["windows_per_s"]) if cpu else None,
            "parity": "tests/test_gpu_bf16.py: logits within 2e-2 of the fp32 reference, argmax identical on the 324 repo windows",
            "roofline": {"kernel": "decoder_infer_v2_kernel", "bound": "tensor", "achieved": tc_tflops, "peak": peak, "unit": "TFLOP/s",
                         "frac": tc_tflops / peak, "ms_per_launch": ms_tc, "ms_per_launch_time_major_fp16_input": ms_tc_tm,
                         "traffic": NCU_TRAFFIC_BYTES_40960 * n_win / 40960, "traffic_source": "profiles/r1_tc2_fused_ncu_full.csv",
                         "per_timestep_latency_us": {"full_tile_round": ms_tc_full * 1e3 / T, "short_tile_chain": ms_tc_short * 1e3 / T},
                         "xu_pipe": mufu_pipe(n_win, ms_tc, h16["clocks"], V2_MUFU_PER_CELL)},
        },
    }
    line["single_window_latency_ms"] = {"exact_fp32": lat_exact, "fp16_tier": lat_h16,
                                         "what": "host numpy [625,8] -> H2D -> decoder forward + softmax -> D2H probabilities, median of 50 "
                                                 "(reference on its CPU: ~13.5 ms per window, SURVEY 8a12)"}
    if cpu:
        line["cpu_baseline"] = {"value": cpu["windows_per_s"], "unit": "windows/s", "cores": cpu["cores"],
                                "kind": "port", "sample": cpu["sample"]}
    if train:
        if cpu_train:
            train["cpu_baseline"] = cpu_train
            train["fp32_exact"]["vs_cpu"] = train["fp32_exact"]["value"] / world / cpu_train["value"]
        line["train"] = train
    if stress:
        line["stress"] = stress
    if config1:
        line["config1"] = config1
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, arrays):
    """Rank 0's results of the last timed step, one float32 ``<name>.npy`` each: per tier the [40960, 3] logits and
    probabilities and the [4096, 3] 10-trial means (2.6 MB in all).  The inputs are seeded, so two builds run with the
    same arguments can be compared output for output."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(d / f"{name}.npy", t.float().cpu().numpy())


X3_MUFU_PER_CELL, V2_MUFU_PER_CELL = 7, 5


def mufu_pipe(n_win, ms, clocks, per_cell):
    """The pipe that actually bounds the decoder kernels: ``per_cell`` MUFU results per hidden unit, layer and step on the
    16-results/clk/SM transcendental pipe (measured: scripts/ubench/mufu_rate.cu, 31.4 results/ns/SM at 1.965 GHz)."""
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    ops_ = n_win * T * 2 * H * per_cell
    ach, peak = ops_ / (ms * 1e-3) / 1e9, 16 * 148 * mhz * 1e-3
    return {"bound": "MUFU (transcendental pipe): 16 results/clk/SM x 148 SMs x SM clock under load", "achieved": ach, "peak": peak,
            "unit": "G MUFU results/s", "frac": ach / peak, "sm_mhz": mhz, "mufu_per_cell": per_cell}


def stress_leg(dev, peaks):
    """BASELINE configs[4]: EEG_LSTM(hidden_size=192), T = 2500 (4x longer windows, 4x wider LSTM), synthetic EEG,
    one full round of 148 x 128 windows, eval forward on the streamed-weight tensor-core kernel
    (na_decoder_wide.cu).  Seeded default init (there is no shipped checkpoint of that shape)."""
    from neural_speech_decoding_b200 import ops
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    Hs, Ts, Bs = 192, 2500, 148 * 128
    flops = 2 * Ts * (4 * Hs * (C + Hs) + 4 * Hs * 2 * Hs) + 4 * Ts * Hs + 2 * 32 * Hs + 2 * 32 * NC
    torch.manual_seed(0)
    m = EEG_LSTM(hidden_size=Hs).to(dev).eval()
    m.compute_dtype = torch.bfloat16
    g = torch.Generator(device="cpu").manual_seed(77)
    x = torch.empty((Bs, Ts, C), dtype=torch.float32, device=dev)
    for i in range(0, Bs, 1024):                       # 1.5 GB of fp32 windows, generated in slabs
        x[i:i + 1024] = (torch.randn((min(1024, Bs - i), Ts, C), generator=g) * INPUT_SIGMA).to(dev)
    with torch.inference_mode():
        xt = ops.window_zscore(x, Ts, Ts, False, True, ops.NA_F16, ops.TC_TILE)
        packed, head = m._packed_tc_wide(), m._head_params()
        ms_k = time_steps(lambda: ops.decoder_infer_wide_bf16(xt, packed, head[2:], Bs, Hs, True), 3, 2, 1, dev) / 3
        del xt
        ms = time_steps(lambda: m.decode(x, want_probs=True), 3, 1, 1, dev) / 3
        # the exact-fp32 tier (generic kernels) on a bounded slice, for the ratio
        m.compute_dtype = torch.float32
        ms32 = time_steps(lambda: m.decode(x[:256], want_probs=True), 1, 1, 1, dev)
    # ---- configs[4] "... and BPTT backward": one train step (fwd + BPTT + Adam) at the stress shape -----------------
    fb = 3 * flops - 2 * Ts * 4 * Hs * C                   # fwd + bwd, no dX of layer 0
    def train_step_time(dtype, Bt):
        torch.manual_seed(0)
        mt = EEG_LSTM(hidden_size=Hs).to(dev).train()
        mt.compute_dtype = dtype
        opt = torch.optim.Adam(mt.parameters(), lr=1e-3)
        yt = torch.randint(0, NC, (Bt,), generator=torch.Generator(device="cpu").manual_seed(5)).to(dev)
        def tstep():
            opt.zero_grad()
            torch.nn.functional.cross_entropy(mt(x[:Bt]), yt).backward()
            opt.step()
        ms_t = time_steps(tstep, 1, 1, 1, dev)
        del mt, opt
        torch.cuda.empty_cache()
        return ms_t
    Bt16, Bt32 = 2048, 256
    ms_t16 = train_step_time(torch.bfloat16, Bt16)
    ms_t32 = train_step_time(torch.float32, Bt32)
    train = {"value": Bt16 / (ms_t16 * 1e-3), "unit": "windows/s", "ms_per_step": ms_t16, "batch": Bt16,
             "tier": "16-bit tensor-core tier: lstm_wide_fwd_kernel<4> / lstm_wide_bwd_kernel<4> (tcgen05, weights streamed by TMA, the "
                     "recurrent state resident) for the serial part of every layer and direction + cuBLAS for the time-parallel GEMMs",
             "achieved_tflops": fb * Bt16 / (ms_t16 * 1e-3) / 1e12,
             "parity": "tests/test_gpu_bf16.py::test_wide_training_* (the reference's H=192 fixture vs float64 autograd, 2e-2; train-mode noise vs the exact tier)",
             "fp32_exact": {"value": Bt32 / (ms_t32 * 1e-3), "unit": "windows/s", "ms_per_step": ms_t32, "batch": Bt32,
                            "tier": "generic FFMA forward-with-save + fused BPTT + time-parallel weight gradients",
                            "parity": "tests/test_gpu_parity.py::test_stress_shape_h192 (gradients within 1e-5 of the fp64 truth)"},
             "note": "2,048 windows = 16 tiles: the serial kernels occupy 16 of 148 SMs (the saves are 27 MB per window; memory, not "
                     "SMs, bounds the batch)"}
    del x
    torch.cuda.empty_cache()
    tf = flops * Bs / (ms_k * 1e-3) / 1e12
    return {"workload": "configs[4]: EEG_LSTM(hidden_size=192), T=2500, C=8, 18,944 synthetic windows, eval forward",
            "train": train,
            "value": Bs / (ms * 1e-3), "unit": "windows/s", "ms_per_pass": ms,
            "kernel": "decoder_infer_wide_kernel<4> (tcgen05; activations resident, weights streamed by TMA from L2)",
            "ms_per_launch": ms_k, "per_timestep_latency_us": ms_k * 1e3 / Ts,
            "flops_per_window": flops, "achieved_tflops": tf,
            "frac_of_bf16_sustained_peak": tf / peaks["bf16_tflops_sustained"], "frac_of_bf16_burst_peak": tf / peaks["bf16_tflops"],
            "fp32_exact_windows_per_s": 256 / (ms32 * 1e-3),
            "parity": "tests/test_gpu_bf16.py::test_wide_*: reference golden (H=192) and the exact tier, 2e-2 contract",
            "note": "stress.train: the 16-bit tier trains at this shape on the tensor cores since round 2"}


def train_leg(args, world, rank, dev):
    """BASELINE configs[2]: data-parallel training of the 3-class decoder on synthetic EEG, GLOBAL batch
    65,536 (fixed as N grows: per-GPU batch 65,536/N, micro-batched), train mode (inter-layer dropout,
    RReLU noise, dropout), mean CE over the global batch, one flat NCCL all-reduce, Adam (optim.FusedAdam: one launch).
    Headline: tensor-core tier; the exact-fp32 tier is timed beside it on a bounded global batch."""
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    from neural_speech_decoding_b200.dp import DataParallelTrainer
    from neural_speech_decoding_b200.optim import FusedAdam

    def run(dtype, global_batch, micro, steps):
        torch.manual_seed(0)
        model = EEG_LSTM().to(dev)
        model.load_state_dict(load_checkpoint(), strict=True)
        model.train()
        model.compute_dtype = dtype
        per_gpu = global_batch // world
        # micro-batches of `micro` windows (default 148 x 128 = one tile per SM) + one ragged remainder: the per-GPU batch is
        # exactly global_batch / world, whatever the SM count
        micro = min(per_gpu, micro)
        micros = [micro] * (per_gpu // micro) + ([per_gpu % micro] if per_gpu % micro else [])
        x = synth_windows(micro, seed=2000 + rank).to(dev)
        g = torch.Generator(device="cpu").manual_seed(1 + rank)
        y = torch.randint(0, NC, (micro,), generator=g).to(dev)
        trainer = DataParallelTrainer(model, FusedAdam(model.parameters(), lr=1e-3), world_size=world)
        batches = [(x[:m], y[:m]) for m in micros]

        def step():
            trainer.step(batches, global_batch=per_gpu * world)

        ms = time_steps(step, steps, 3, world, dev)      # 3 warm-up steps (1 left NCCL / allocator warm-up inside the timed region at N = 8)
        wps = world * per_gpu * steps / (ms * 1e-3)
        return {"value": wps, "unit": "windows/s", "ms_per_step": ms / steps, "global_batch": per_gpu * world,
                "per_gpu_batch": per_gpu, "micro_batch": micro, "micro_batches": micros, "steps": steps,
                "achieved_tflops_per_gpu": FWDBWD_FLOPS_PER_WINDOW * wps / world / 1e12}

    def dp_equivalence(dtype):
        """N-rank DP gradient (each rank its shard, one NCCL all-reduce) == the same global batch on ONE rank.
        Eval-mode autograd (no noise) so both sides are deterministic; executed inside the multi-GPU bench run because
        the driver's pytest box has one GPU."""
        import torch.distributed as dist
        nb = 64 * world
        xg = synth_windows(nb, seed=4242).to(dev)                       # same global batch on every rank
        yg = torch.randint(0, NC, (nb,), generator=torch.Generator(device="cpu").manual_seed(7)).to(dev)
        def grads(xs, ys, ws):
            torch.manual_seed(0)
            m2 = EEG_LSTM().to(dev)
            m2.load_state_dict(load_checkpoint(), strict=True)
            m2.eval()
            m2.compute_dtype = dtype
            tr = DataParallelTrainer(m2, torch.optim.SGD(m2.parameters(), lr=0.0), world_size=ws)
            tr.backward_only([(xs, ys)], global_batch=nb)
            return tr.bucket.flat.clone()
        sl = slice(rank * 64, rank * 64 + 64)
        g_dp = grads(xg[sl], yg[sl], world)
        g_one = grads(xg, yg, 1)
        err = ((g_dp - g_one).abs().max() / g_one.abs().max()).reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        return float(err.item())

    steps = max(1, min(args.steps, 5))
    tc = run(torch.bfloat16, args.train_batch, args.train_micro, steps)
    tc.update({"dtype": "fp16 tensor-core operands (tcgen05), fp32 accumulate / cell state / weight gradients",
               "optimizer": "Adam lr=1e-3 (optim.FusedAdam: torch.optim.Adam's update, one launch for all 16 tensors)",
               "scaling": "strong (global batch fixed)",
               "allreduce": "one flat fp32 bucket (127 KB), NCCL" if world > 1 else "none (1 GPU)",
               "parity": "tests/test_gpu_bf16.py: gradients within 2e-2 of the fp64 oracle",
               "frac_of_bf16_sustained_peak": tc["achieved_tflops_per_gpu"] / measured_peaks()["bf16_tflops_sustained"]})
    fp = run(torch.float32, args.train_batch, args.train_micro, min(steps, 3))      # the same configs[2] step on the fp32-contract tier
    tc["fp32_exact"] = {k: fp[k] for k in ("value", "unit", "ms_per_step", "global_batch", "micro_batch", "achieved_tflops_per_gpu")}
    tc["fp32_exact"]["parity"] = "tests/test_gpu_parity.py: logits and gradients within 1e-5 of the fp64 truth / the reference's autograd"
    tc["fp32_exact"]["kernels"] = ("lstm_fwd_x3_kernel<0/1>, lstm_bwd_x3_kernel<1/0>, lstm_wgrad_x3_kernel<1/0> (tcgen05, operands split into "
                                   "fp16 hi + lo: 3 MMAs per product, fp32 accumulate; ex2 / rcp activations)")
    tc["fp32_exact"]["frac_of_bf16_sustained_peak_issued_3x"] = 3 * fp["achieved_tflops_per_gpu"] / measured_peaks()["bf16_tflops_sustained"]
    if world > 1:
        e16, e32 = dp_equivalence(torch.bfloat16), dp_equivalence(torch.float32)
        tc["dp_equivalence"] = {"what": f"max|g_DP({world} ranks, NCCL all-reduce) - g_single| / max|g| over the flat gradient bucket, "
                                        f"global batch {64 * world}, eval-mode autograd",
                                "fp16_tier": e16, "fp32_exact": e32, "tolerance": {"fp16_tier": 1e-4, "fp32_exact": 1e-5},
                                "ok": bool(e16 < 1e-4 and e32 < 1e-5)}
        if not tc["dp_equivalence"]["ok"] and rank == 0:
            print(f"WARNING: DP equivalence outside tolerance: {tc['dp_equivalence']}", file=sys.stderr)
    return tc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-stress", action="store_true")
    ap.add_argument("--train-batch", type=int, default=65536, help="GLOBAL batch of the train leg (configs[2])")
    ap.add_argument("--train-micro", type=int, default=148 * 128, help="windows per micro-batch (default: one 128-window tile per SM)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (both tiers) to DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    run_gpu_arm(args)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
