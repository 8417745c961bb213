"""The fp32 FFMA tier (generic LSTM kernels, head kernels, weight-gradient reductions) at every size its C ABI accepts,
against float64 references on the CPU.

The tier runs every model shape the tensor-core kernels do not, every backward that wants d/dx, and it is the anchor the
tensor-core tiers are tested against.  Its ABI accepts 1 <= K <= 4096, 1 <= H <= 1024 and 1 <= NC <= 16, so the cases
sit on both sides of every edge the kernels have:
- the generic kernels change how a thread maps to hidden units at H = 512 (512 threads a CTA at most) and loop the BPTT
  contraction over K + H columns beyond 512;
- the head is compiled for H <= 64 / 128 / 256 / 512 / 1024 with 8 / 4 / 2 / 1 / 1 time steps per chunk;
- B = 1, 9 and 41 leave windows of padding in the 8-window CTAs of the LSTM kernels and in the head's 8-warp CTAs;
- T = 1 .. 17 end the head's time chunks at every remainder.

Judgement: max|d| / max|ref| per tensor within 1e-5.  A gradient that vanishes analytically is judged on the largest
gradient of the call instead: attn.bias always (softmax over time is shift-invariant), dW_hh and d attn.weight at T = 1,
and at H = 1 everything upstream of the LayerNorm and d ln.weight (a LayerNorm over one unit outputs ln.bias whatever its
input).  The module cases also judge d attn.weight at T = 2 that way: with two steps it is alpha_0 alpha_1 (g_0 - g_1)
(h_0 - h_1) summed over windows, a product of two step differences of an LSTM's output.  At (K, H, L, T) = (1, 1024, 3,
2) it is 2.5e-5 of the largest gradient, and a relative 1e-7 change of the top layer's h moves it by 5e-6 of itself, so
the fp32 rounding of h alone puts it near 1e-5 (measured on an NVIDIA B200: 1.4e-5; every other tensor within 3.3e-6).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.torch_ref import RRELU_EVAL_SLOPE, RefEEGLSTM

pytestmark = pytest.mark.gpu

TOL = 1e-5
P = 0.6                                   # EEG_LSTM's default dropout
SCALE = 1.0 / (1.0 - P)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from neural_speech_decoding_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


@pytest.fixture
def ffma_tier():
    """The flagship-shape switches off, so that every call below runs on the FFMA kernels."""
    from neural_speech_decoding_b200 import ops
    saved = ops.EXACT_TC, ops.EXACT_TC_TRAIN
    ops.EXACT_TC = ops.EXACT_TC_TRAIN = False
    yield
    ops.EXACT_TC, ops.EXACT_TC_TRAIN = saved


def err(got, want, scale=None):
    got = np.asarray(got.detach().cpu() if torch.is_tensor(got) else got, np.float64)
    want = np.asarray(want.detach().cpu() if torch.is_tensor(want) else want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    s = np.abs(want).max() if scale is None else scale
    return float(np.abs(got - want).max() / max(float(s), 1e-300))


def judge(errors):
    bad = {k: v for k, v in errors.items() if not v < TOL}
    assert not bad, f"bad={bad} all={errors}"


def gmax_of(grads):
    return max(float(np.abs(g.detach().cpu().numpy()).max()) for g in grads.values())


def judge_grads(got, want, T, H, near_vanishing=()):
    """got / want: name -> gradient, each judged on its own scale unless it vanishes (module docstring)."""
    vanishing = {"attn.bias", *near_vanishing}
    if T == 1:
        vanishing |= {k for k in want if "weight_hh" in k or k == "attn.weight"}
    if H == 1:
        vanishing |= {k for k in want if k.startswith(("lstm.", "attn.", "ln.weight"))}
    gmax = gmax_of(want)
    return {f"d{k}": err(got[k], want[k], gmax if k in vanishing else None) for k in want}


def tail_f64(z, prm, rr, d2):
    """LayerNorm -> fc0 -> RReLU(slopes) -> dropout -> fc3 in the dtype of z.  rr None: eval slope; d2 None: no dropout."""
    _, _, ln_w, ln_b, w0, b0, w3, b3 = prm
    zn = F.layer_norm(z, (z.shape[-1],), ln_w, ln_b, 1e-5)
    a = zn @ w0.t() + b0
    a = torch.where(a >= 0, a, a * (RRELU_EVAL_SLOPE if rr is None else rr))
    if d2 is not None:
        a = a * d2 * SCALE
    return a @ w3.t() + b3, zn


def head_f64(h, prm, rr, d2):
    """Attention pool over time + tail.  h [B,T,H] -> (logits, scores [B,T], pooled, embedding)."""
    s = h @ prm[0][0] + prm[1][0]
    z = (h * torch.softmax(s, dim=1).unsqueeze(-1)).sum(dim=1)
    logits, zn = tail_f64(z, prm, rr, d2)
    return logits, s, z, zn


def train_forward_f64(x, sd, L, masks, rr, d2):
    """The decoder in train mode with given noise, cell by cell; masks[l] [B,T,H] is the keep-mask after layer l."""
    inp = x
    for l in range(L):
        w_ih, w_hh = sd[f"lstm.weight_ih_l{l}"], sd[f"lstm.weight_hh_l{l}"]
        b = sd[f"lstm.bias_ih_l{l}"] + sd[f"lstm.bias_hh_l{l}"]
        B, T, _ = inp.shape
        H = w_hh.shape[1]
        h = c = inp.new_zeros(B, H)
        pre = inp @ w_ih.t() + b
        hs = []
        for t in range(T):
            i, f, g, o = (pre[:, t] + h @ w_hh.t()).split(H, dim=1)
            c = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
            h = torch.sigmoid(o) * torch.tanh(c)
            hs.append(h)
        inp = torch.stack(hs, dim=1)
        if l < L - 1:
            inp = inp * masks[l] * SCALE
    return head_f64(inp, [sd[k] for k in ("attn.weight", "attn.bias", "ln.weight", "ln.bias", "fc.0.weight",
                                           "fc.0.bias", "fc.3.weight", "fc.3.bias")], rr, d2)[0]


# ---------------------------------------------------------------------------------------------
# (a) EEG_LSTM on the FFMA tier
# ---------------------------------------------------------------------------------------------
# (input_size, hidden_size, num_layers, num_classes, B, T): every H edge of the generic and head kernels
# (H = 300: layer 1 has K + H = 600; H >= 505 with K = 8: layer 0 has K + H > 512; H > 512: two units a thread),
# input_size 1 / 8 / 37 / 1000 / 4096, 1-3 layers, NC 1 / 3 / 16, B 1 / 9 / 41, T 1 / 2 / 7 / 9 / 17
MODULE_SHAPES = [
    (8, 1, 2, 3, 9, 7),
    (1, 31, 1, 1, 41, 9),
    (37, 32, 3, 16, 1, 17),
    (8, 33, 2, 3, 9, 2),
    (8, 64, 1, 16, 41, 1),
    (37, 65, 2, 1, 9, 17),
    (1, 128, 2, 3, 1, 9),
    (8, 129, 3, 3, 9, 7),
    (1000, 256, 1, 3, 9, 2),
    (8, 257, 2, 16, 41, 7),
    (8, 300, 2, 3, 9, 9),
    (37, 504, 1, 1, 9, 2),
    (8, 505, 2, 3, 1, 7),
    (1, 512, 1, 16, 9, 17),
    (8, 513, 2, 3, 9, 1),
    (8, 672, 1, 3, 41, 2),
    (37, 673, 2, 16, 9, 7),
    (1000, 1023, 1, 3, 9, 9),
    (8, 1024, 2, 3, 9, 17),
    (1, 1024, 3, 16, 41, 2),
    (4096, 16, 1, 3, 9, 7),
    (4096, 1, 2, 1, 41, 2),
]


@pytest.mark.parametrize("train", [False, True], ids=["eval", "train"])
@pytest.mark.parametrize("K,H,L,NC,B,T", MODULE_SHAPES)
def test_module_vs_float64(dev, ffma_tier, K, H, L, NC, B, T, train):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(1000 * H + K + 7 * L + T)
    ref = RefEEGLSTM(K, H, L, NC).eval()
    sd = {k: v.double() for k, v in ref.state_dict().items()}            # fp32 values, evaluated in float64
    ref.double().load_state_dict(sd, strict=True)
    x = torch.randn(B, T, K).double()
    y = torch.randint(0, NC, (B,))
    m = EEG_LSTM(K, H, L, NC).to(dev)
    m.load_state_dict({k: v.float() for k, v in sd.items()}, strict=True)
    errors = {}
    if train:
        masks = [(torch.rand(B, T, H) >= P).double() for _ in range(L - 1)]
        rr = torch.empty(B, 32, dtype=torch.float64).uniform_(1 / 8, 1 / 3).float().double()
        d2 = (torch.rand(B, 32) >= P).double()
        sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        xr = x.clone().requires_grad_(True)
        want = train_forward_f64(xr, sdg, L, masks, rr, d2)
        m.train()
        m.inject_noise(drop1=torch.stack(masks).float() if L > 1 else None, rrelu_slope=rr.float(), drop2=d2.float())
        ref_grads = lambda: {k: v.grad for k, v in sdg.items()}
    else:
        xr = x.clone().requires_grad_(True)
        want = ref(xr)
        m.eval()
        with torch.no_grad():                              # the inference launches (nothing saved)
            errors["logits_infer"] = err(m(x.float().to(dev)), want)
        ref_grads = lambda: {k: p.grad for k, p in ref.named_parameters()}
    lr = F.cross_entropy(want, y)
    lr.backward()
    xg = x.float().to(dev).requires_grad_(True)
    logits = m(xg)
    loss = F.cross_entropy(logits, y.to(dev))
    loss.backward()
    assert m._tier(xg, train=True) == "ffma"
    errors["logits"] = err(logits, want)
    errors["loss"] = abs(loss.item() - lr.item()) / max(1.0, abs(lr.item()))
    errors["dx"] = err(xg.grad, xr.grad, gmax_of(ref_grads()) if H == 1 else None)
    errors.update(judge_grads({k: p.grad for k, p in m.named_parameters()}, ref_grads(), T, H,
                              ["attn.weight"] if T == 2 else []))
    judge(errors)


# ---------------------------------------------------------------------------------------------
# (b) one layer through the C ABI with an initial state, dropout on both sides and gradients from outside the sequence
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,H", [(8, 504), (8, 505), (512, 512), (1, 1024), (1000, 25), (37, 1024)])
def test_layer_abi_with_initial_state(dev, K, H):
    from neural_speech_decoding_b200 import ops
    torch.manual_seed(K + H)
    B, T = 9, 5
    Bp = ops.padded_batch(B)
    lstm = torch.nn.LSTM(K, H, 1, batch_first=True).double()          # fp32-initialised values in float64
    x = torch.randn(B, T, K).double()
    in_mask = (torch.rand(B, T, K) >= P).double()
    out_mask = (torch.rand(B, T, H) >= P).double()
    h0, c0 = torch.randn(B, H).double() * 0.5, torch.randn(B, H).double()
    dh_out = torch.randn(B, T, H).double()
    dh_last, dc_last = torch.randn(B, H).double(), torch.randn(B, H).double()

    # float64: u = x * in_mask * scale is the layer's input (what the layer below hands up), stepped one call per t so
    # that every c_t is seen
    xr, h0r, c0r = (t.clone().requires_grad_(True) for t in (x, h0, c0))
    u = xr * in_mask * SCALE
    state, hs, cs = (h0r[None], c0r[None]), [], []
    for t in range(T):
        out, state = lstm(u[:, t:t + 1], state)
        hs.append(out[:, 0])
        cs.append(state[1][0])
    h_ref, c_ref = torch.stack(hs, 1), torch.stack(cs, 1)
    ((h_ref * dh_out).sum() + (state[0][0] * dh_last).sum() + (state[1][0] * dc_last).sum()).backward()

    def tmp(t):                                           # [B,T,n] -> zero-padded TMP [T,Bp,n] fp32 on the device
        z = torch.zeros(t.shape[1], Bp, t.shape[2])
        z[:, :B] = t.detach().permute(1, 0, 2).float()
        return z.to(dev)

    def rows(t):                                          # [B,H] -> zero-padded [Bp,H]
        z = torch.zeros(Bp, t.shape[1])
        z[:B] = t.detach().float()
        return z.to(dev)

    w_ih, w_hh, b_ih, b_hh = (p.detach().float().to(dev).contiguous() for p in
                              (lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0))
    u_tmp = tmp(u)
    wt, bias = ops.pack_lstm_layer(w_ih, w_hh, b_ih, b_hh)
    h, c, gates, h_drop = ops.lstm_layer_fwd_hx(u_tmp, wt, bias, tmp(out_mask), SCALE, rows(h0), rows(c0))
    dgates, din, dh0, dc0 = ops.lstm_layer_bwd_hx(tmp(dh_out), gates, c, w_ih, w_hh, tmp(in_mask), SCALE, True, rows(c0),
                                                  rows(dh_last), rows(dc_last), True)
    dw_ih, dw_hh, db = ops.lstm_layer_wgrad_hx(dgates, u_tmp, h, rows(h0))
    bm = lambda t: t[:, :B].permute(1, 0, 2)             # TMP -> [B,T,n], live rows
    judge({"h": err(bm(h), h_ref), "c": err(bm(c), c_ref), "h_drop": err(bm(h_drop), h_ref * out_mask * SCALE),
           "din": err(bm(din), xr.grad), "dh0": err(dh0[:B], h0r.grad), "dc0": err(dc0[:B], c0r.grad),
           "dW_ih": err(dw_ih, lstm.weight_ih_l0.grad), "dW_hh": err(dw_hh, lstm.weight_hh_l0.grad),
           "db": err(db, lstm.bias_ih_l0.grad)})
    # padding windows: zero inputs and zero incoming gradients give finite states and exactly zero gradients (the
    # reductions sum over every row, padding included)
    for name, t in {"h": h, "c": c, "gates": gates, "h_drop": h_drop}.items():
        assert torch.isfinite(t).all(), name
    for name, t in {"dgates": dgates[:, B:], "din": din[:, B:], "dh0": dh0[B:], "dc0": dc0[B:]}.items():
        assert torch.count_nonzero(t) == 0, name


# ---------------------------------------------------------------------------------------------
# (c) the head at every <JPL, CH> instantiation
# ---------------------------------------------------------------------------------------------
def chunk(H):
    return 8 if H <= 64 else 4 if H <= 128 else 2 if H <= 256 else 1


def head_params(H, NC, gen, attn_scale=1.0):
    lin = lambda o, i: (torch.rand(o, i, generator=gen, dtype=torch.float64) * 2 - 1) / np.sqrt(i)
    return [lin(1, H) * attn_scale, torch.randn(1, generator=gen, dtype=torch.float64),
            1 + 0.2 * torch.randn(H, generator=gen, dtype=torch.float64), 0.1 * torch.randn(H, generator=gen, dtype=torch.float64),
            lin(32, H), 0.1 * torch.randn(32, generator=gen, dtype=torch.float64),
            lin(NC, 32), 0.1 * torch.randn(NC, generator=gen, dtype=torch.float64)]


def run_head(dev, H, T, NC, B, attn_scale=1.0, seed=0):
    """Every head entry point at one shape against float64; returns (errors, float64 scores)."""
    from neural_speech_decoding_b200 import ops
    gen = torch.Generator().manual_seed(seed)
    Bp = ops.padded_batch(B)
    prm = [p.float().double() for p in head_params(H, NC, gen, attn_scale)]      # fp32-representable
    h = torch.tanh(torch.randn(B, T, H, generator=gen, dtype=torch.float64)).float().double()
    rr = torch.empty(B, 32, dtype=torch.float64).uniform_(1 / 8, 1 / 3, generator=gen).float().double()
    d2 = (torch.rand(B, 32, generator=gen) >= P).double()
    dlogits = torch.randn(B, NC, generator=gen, dtype=torch.float64).float().double()

    h_tmp = torch.full((T, Bp, H), float("nan"))          # padding windows are never read
    h_tmp[:, :B] = h.permute(1, 0, 2).float()
    h_tmp = h_tmp.to(dev)
    pg = [p.float().to(dev).contiguous() for p in prm]
    rr_g, d2_g = rr.float().to(dev), d2.float().to(dev)
    names = ["attn.weight", "attn.bias", "ln.weight", "ln.bias", "fc.0.weight", "fc.0.bias", "fc.3.weight", "fc.3.bias"]
    e = {}

    # train mode: forward with RReLU slopes and dropout, backward
    hr = h.clone().requires_grad_(True)
    pr = [p.clone().requires_grad_(True) for p in prm]
    lg_ref, s_ref, z_ref, _ = head_f64(hr, pr, rr, d2)
    (lg_ref * dlogits).sum().backward()
    logits, probs, stats, zpool = ops.head_fwd(h_tmp, B, pg, rr_g, d2_g, SCALE, True, True)
    e["logits"] = err(logits, lg_ref)
    e["probs"] = err(probs, torch.softmax(lg_ref, dim=1))
    e["zpool"] = err(zpool, z_ref)
    dh, dparams = ops.head_bwd(dlogits.float().to(dev), h_tmp, stats, zpool, pg, rr_g, d2_g, SCALE)
    want = dict(zip(names, [p.grad for p in pr]))
    e["dh"] = err(dh[:, :B].permute(1, 0, 2), hr.grad, gmax_of(want) if H == 1 else None)
    assert torch.count_nonzero(dh[:, B:]) == 0                                    # padding rows of dh are zeroed
    e.update(judge_grads(dict(zip(names, ops.split_head_grads(dparams, H, NC))), want, T, H))

    # the saved zpool through the tail-only forward: the same arithmetic as the full forward's, bit for bit
    tail_logits, tail_probs = ops.head_tail_fwd(zpool, pg, rr_g, d2_g, SCALE, True)
    assert torch.equal(tail_logits, logits) and torch.equal(tail_probs, probs)

    # tail forward / backward from the float64 pooled vector
    z32 = z_ref.detach().float().double().requires_grad_(True)
    pt = [p.clone().requires_grad_(True) for p in prm]
    tl_ref, _ = tail_f64(z32, pt, rr, d2)
    (tl_ref * dlogits).sum().backward()
    tl, _ = ops.head_tail_fwd(z32.detach().float().to(dev), pg, rr_g, d2_g, SCALE, False)
    e["tail_logits"] = err(tl, tl_ref)
    dz, dtail = ops.head_tail_bwd(dlogits.float().to(dev), z32.detach().float().to(dev), pg, rr_g, d2_g, SCALE)
    want = {k: p.grad for k, p in zip(names[2:], pt[2:])}
    e["tail_dz"] = err(dz, z32.grad, gmax_of(want) if H == 1 else None)
    tg = dict(zip(names, ops.split_head_grads(dtail, H, NC)))
    assert torch.count_nonzero(tg["attn.weight"]) == 0 and torch.count_nonzero(tg["attn.bias"]) == 0
    e.update({f"tail_{k}": v for k, v in judge_grads({k: tg[k] for k in names[2:]}, want, T, H).items()})

    # eval mode with the intermediates
    lg_e, s_e, z_e, zn_e = head_f64(h, prm, None, None)
    logits, probs, scores, pooled, emb = ops.head_fwd_ex(h_tmp, B, pg)
    e.update({"ex_logits": err(logits, lg_e), "ex_probs": err(probs, torch.softmax(lg_e, dim=1)),
              "ex_scores": err(scores.t(), s_e), "ex_pooled": err(pooled, z_e), "ex_embedding": err(emb, zn_e)})
    return e, s_e


@pytest.mark.parametrize("H", [1, 64, 65, 128, 129, 256, 257, 512, 513, 1024])
def test_head_every_instantiation(dev, H):
    CH = chunk(H)
    for T in sorted({CH - 1, CH, CH + 1, 625} - {0}):
        for NC in (1, 16):
            B = 9 if T == 625 else 41
            errors, _ = run_head(dev, H, T, NC, B, seed=H * 7919 + T * 31 + NC)
            judge({f"T={T} NC={NC} {k}": v for k, v in errors.items()})


@pytest.mark.parametrize("H", [1, 64, 129, 257, 1024])
def test_head_online_softmax_rescales_across_chunks(dev, H):
    """attn.weight scaled so that the scores of a window span more than 80: every new running maximum rescales what the
    earlier chunks accumulated, by factors down to exp(-80)."""
    errors, scores = run_head(dev, H, 625, 3, 9, attn_scale=120.0 if H == 1 else 60.0, seed=H)
    span = (scores.max(dim=1).values - scores.min(dim=1).values).min().item()
    assert span > 80, span
    judge(errors)
