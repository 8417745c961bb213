"""Save what every kernel tier of EEG_LSTM computes, from seeded inputs, so that two builds can be compared bit for bit.

Tiers: x3 (fp32, flagship shape), tc (compute_dtype bf16, flagship), wide (bf16, hidden_size 96, short windows) and FFMA
(hidden_size 32 with 3 layers; the flagship with ops.EXACT_TC / EXACT_TC_TRAIN off).  The flagship tensor-core tiers run
one batch small enough for half tiles and one above 148 x 64 windows, which takes full tiles.  For each: ``decode``
(with and without the z-score stage), ``decode_intermediates``, ``forward`` logits and every parameter gradient in eval
mode and in train mode (injected noise, and noise drawn under torch.manual_seed), and ``model.lstm(x, hx)`` on the fused
path (eval, no autograd) and on the autograd path (train mode, with gradients).  Uses only the public API.

    python scripts/dump_tier_outputs.py --out DIR            # one .npz per case
    python scripts/dump_tier_outputs.py --compare DIR_A DIR_B  # every array equal bit for bit (NaNs included)?
"""
import argparse
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from neural_speech_decoding_b200 import ops                      # noqa: E402
from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM  # noqa: E402

# name: (model kwargs, compute_dtype, exact tensor-core tiers on, batch sizes, T)
CASES = {
    "x3": ({}, torch.float32, True, (200, 9600), 625),
    "tc": ({}, torch.bfloat16, True, (200, 9600), 625),
    "wide": ({"hidden_size": 96}, torch.bfloat16, True, (300,), 96),
    "ffma_h32x3": ({"hidden_size": 32, "num_layers": 3}, torch.float32, True, (100,), 120),
    "ffma_flagship": ({}, torch.float32, False, (150,), 200),
}


def arr(t):
    t = t.detach()
    return (t.float() if t.dtype == torch.bfloat16 else t).cpu().numpy()


def run_case(name, kw, cdt, exact, B, T, dev):
    ops.EXACT_TC = ops.EXACT_TC_TRAIN = exact
    out = {}
    torch.manual_seed(11)
    m = EEG_LSTM(**kw).to(dev)
    m.compute_dtype = cdt
    L, H, K = m.lstm.num_layers, m.lstm.hidden_size, m.fc[3].out_features
    g = torch.Generator().manual_seed(B)
    x = (torch.randn((B, T, 8), generator=g) * 2.5).to(dev)
    y = torch.randint(0, K, (B,), generator=g).to(dev)

    m.eval()
    for z in (False, True):
        m.zscore_input = z
        lg, pr = m.decode(x)
        out[f"decode_z{int(z)}_logits"], out[f"decode_z{int(z)}_probs"] = arr(lg), arr(pr)
        for f, t in zip(("logits", "probs", "attention", "pooled", "embedding"), m.decode_intermediates(x)):
            out[f"ex_z{int(z)}_{f}"] = arr(t)
    m.zscore_input = False

    def fwd_bwd(tag):
        m.zero_grad(set_to_none=True)
        logits = m(x)
        torch.nn.functional.cross_entropy(logits.float(), y).backward()
        out[f"{tag}_logits"] = arr(logits)
        for k, p in m.named_parameters():
            out[f"{tag}_grad_{k}"] = arr(p.grad)

    fwd_bwd("eval")
    m.train()
    drop1 = (torch.rand((L - 1, B, T, H), generator=g) >= m.dropout_p).float().to(dev)
    rr = torch.empty((B, 32)).uniform_(1 / 8, 1 / 3, generator=g).to(dev)
    drop2 = (torch.rand((B, 32), generator=g) >= m.dropout_p).float().to(dev)
    m.inject_noise(drop1, rr, drop2)
    fwd_bwd("train_injected")
    m.inject_noise()
    torch.manual_seed(5)
    fwd_bwd("train_seeded")

    h0 = (torch.randn((L, B, H), generator=g) * 0.5).to(dev)
    c0 = torch.randn((L, B, H), generator=g).to(dev)
    m.eval()
    with torch.no_grad():
        o, (hn, cn) = m.lstm(x, (h0, c0))
    out["lstm_eval_out"], out["lstm_eval_hn"], out["lstm_eval_cn"] = arr(o), arr(hn), arr(cn)
    m.train()
    m.zero_grad(set_to_none=True)
    xg, h0g, c0g = x.clone().requires_grad_(True), h0.clone().requires_grad_(True), c0.clone().requires_grad_(True)
    torch.manual_seed(6)
    o, (hn, cn) = m.lstm(xg, (h0g, c0g))
    (o.square().mean() + hn.sum() + cn.mean()).backward()
    out["lstm_train_out"], out["lstm_train_hn"], out["lstm_train_cn"] = arr(o), arr(hn), arr(cn)
    out["lstm_grad_x"], out["lstm_grad_h0"], out["lstm_grad_c0"] = arr(xg.grad), arr(h0g.grad), arr(c0g.grad)
    for k, p in m.lstm.named_parameters():
        out[f"lstm_grad_{k}"] = arr(p.grad)
    return out


def compare(a: Path, b: Path) -> int:
    bad, n = [], 0
    names = sorted(p.name for p in a.glob("*.npz"))
    if names != sorted(p.name for p in b.glob("*.npz")) or not names:
        print(f"different case files: {names} vs {sorted(p.name for p in b.glob('*.npz'))}")
        return 1
    for f in names:
        da, db = np.load(a / f), np.load(b / f)
        if sorted(da.files) != sorted(db.files):
            bad.append(f"{f}: different arrays")
            continue
        for k in da.files:
            u, v = da[k], db[k]
            n += 1
            same = u.dtype == v.dtype and u.shape == v.shape and np.array_equal(
                u.view(f"u{u.dtype.itemsize}"), v.view(f"u{v.dtype.itemsize}"))
            if not same:
                bad.append(f"{f}:{k}")
    print(f"{n} arrays compared, {len(bad)} differ" + ("".join("\n  " + s for s in bad)))
    return 1 if bad else 0


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", type=Path)
    ap.add_argument("--compare", type=Path, nargs=2)
    args = ap.parse_args()
    if args.compare:
        sys.exit(compare(*args.compare))
    args.out.mkdir(parents=True, exist_ok=True)
    dev = torch.device("cuda")
    for name, (kw, cdt, exact, batches, T) in CASES.items():
        for B in batches:
            out = run_case(name, kw, cdt, exact, B, T, dev)
            np.savez(args.out / f"{name}_B{B}.npz", **out)
            print(f"{name} B={B}: {len(out)} arrays", flush=True)


if __name__ == "__main__":
    main()
