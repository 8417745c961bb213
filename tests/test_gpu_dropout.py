"""The in-kernel inter-layer dropout of the two flagship tensor-core training tiers (exact: csrc/na_train_x3.cu, 16-bit:
csrc/na_train_tc.cu + na_train_fwd2.cuh) against references.

In train mode ``EEG_LSTM`` passes ``(seed, thresh16)`` to the layer-0 forward and the layer-1 backward, which regenerate
the keep-bits from a counter-based hash (``dropout_keep8``); no mask tensor exists.  These tests pin that path:

* the generator (``ops.dropout_mask_u8``) equals the numpy restatement ``oracle.dropout_hash`` bit for bit;
* generator mode equals mask-tensor mode fed with the materialised mask, bit for bit (logits and all 16 gradients), on
  full tiles, half tiles and a capped grid -- the kernels share every instruction after the keep-bits;
* generator mode against float64 autograd of ``explicit_forward`` with the same mask and the generator's scale 65536 /
  thresh16: the exact tier within 1e-5 on every tensor's own scale, the 16-bit tier within its 2e-2 contract;
* the ends of thresh16: 0 (drop everything) and 1, whose scale 65536 does not fit the fp16 operands.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import dropout_hash as dh
from oracle.torch_ref import explicit_forward

pytestmark = pytest.mark.gpu

EXACT_TOL = 1e-5
BF16_TOL = 2e-2
TH06 = 26214                         # round(0.4 * 65536): the module's thresh16 at its default p = 0.6


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from neural_speech_decoding_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def make_model(dev, sd, **kw):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    m = EEG_LSTM(**kw)
    m.load_state_dict(sd, strict=True)
    return m.to(dev)


class Layout:
    """Tile layout of both training tiers for the duration of a ``with``: "full", "half" or "capped" (full tiles, the grid
    capped to 2 CTAs so that every CTA loops over several tiles); "default" leaves the library's choice."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        from neural_speech_decoding_b200 import _lib, ops
        self.saved = (ops.X3_HALF_TILES, ops.TC_HALF_TILES)
        if self.name != "default":
            ops.X3_HALF_TILES = ops.TC_HALF_TILES = self.name == "half"
        if self.name == "capped":
            _lib.call("na_set_tuning", b"train_max_ctas", 2)
        return self

    def __exit__(self, *exc):
        from neural_speech_decoding_b200 import _lib, ops
        ops.X3_HALF_TILES, ops.TC_HALF_TILES = self.saved
        _lib.call("na_set_tuning", b"train_max_ctas", 0)


def train_fn(tier):
    from neural_speech_decoding_b200 import ops
    return ops.decoder_train_forward_x3 if tier == "x3" else ops.decoder_train_forward_tc


def run_ops(m, tier, x, y, p, drop1, rr, d2):
    """One training step through ``ops`` -> (logits, the 16 parameter gradients in named_parameters order)."""
    m.zero_grad()
    lstm, head = [m.lstm.layer(l) for l in range(2)], m._head_params()
    out = train_fn(tier)(x, lstm, head, p, False, drop1, rr, d2)
    F.cross_entropy(out, y).backward()
    return out.detach().clone(), [q.grad.detach().clone() for q in m.parameters()]


def inputs(B, T, seed, windows=None):
    gen = torch.Generator().manual_seed(seed)
    if windows is None:
        x = torch.randn(B, T, 8, generator=gen) * 2.73
    else:
        x = torch.from_numpy(windows["X"][:B, :T].copy())
    y = torch.randint(0, 3, (B,), generator=gen)
    rr = torch.empty(B, 32).uniform_(1 / 8, 1 / 3, generator=gen)
    d2 = (torch.rand(B, 32, generator=gen) >= 0.6).float()
    return x, y, rr, d2


def gen_mask(x_dev, seed, th, B, T):
    """The generator's keep-mask of windows 0..B-1 as [B, T, 48] float64 (the full-tile key: row t * padded_batch + b)."""
    from neural_speech_decoding_b200 import ops
    mask = ops.dropout_mask_u8(x_dev, seed, th, T, ops.padded_batch(B, ops.TC_TILE))
    return mask, mask[:, :B].permute(1, 0, 2).double().cpu()


def fp64_reference(sd, x, y, p, m1, scale1, rr, d2):
    """float64 autograd of the cell-by-cell restatement -> (logits, loss, gradients by parameter name)."""
    sd64 = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    logits = explicit_forward(x.double(), sd64, 2, p, m1, rr.double(), d2.double(), drop1_scale=scale1)
    loss = F.cross_entropy(logits, y)
    loss.backward()
    return logits.detach().numpy(), loss.item(), {k: v.grad.numpy() for k, v in sd64.items()}


def grad_errors(m, grads, ref, tier, T):
    """max|d| / scale per tensor.  The scale is the tensor's own max|ref|, except for gradients that vanish analytically:
    attn.bias (softmax over time is shift-invariant) and, at T = 1, weight_hh* and attn.weight are judged on the largest
    gradient of the model (the exact tier, check_grads' rule); the 16-bit tier judges attn.bias on attn.weight's scale
    (grad_rel's rule) where that is not zero."""
    names = [k for k, _ in m.named_parameters()]
    gmax = max(float(np.abs(ref[k]).max()) for k in names)
    aw = float(np.abs(ref["attn.weight"]).max())
    out = {}
    for k, g in zip(names, grads):
        scale = float(np.abs(ref[k]).max())
        if T == 1 and ("weight_hh" in k or k in ("attn.weight", "attn.bias")):
            scale = gmax
        elif k == "attn.bias":
            scale = gmax if tier == "x3" else aw
        out[k] = float(np.abs(g.float().cpu().numpy() - ref[k]).max() / scale)
    return out


def check_against_fp64(tag, m, tier, T, logits, y, grads, ref, limits=None):
    """Logits on max|ref logits|, the loss absolutely, every gradient by grad_errors' rule; the exact tier within 1e-5,
    the 16-bit tier within 2e-2.  ``limits``: tensor name -> the measured bound of a case where the tier's arithmetic does
    not reach its contract (see the cases that pass one); every other tensor keeps the contract."""
    ref_logits, ref_loss, ref_grads = ref
    tol = EXACT_TOL if tier == "x3" else BF16_TOL
    lg = logits.float().cpu().numpy()
    assert np.isfinite(lg).all(), tag
    lerr = float(np.abs(lg - ref_logits).max() / np.abs(ref_logits).max())
    loss_err = abs(F.cross_entropy(logits.float(), y).item() - ref_loss)
    errs = grad_errors(m, grads, ref_grads, tier, T)
    worst = max(errs, key=errs.get)
    print(f"DROPOUT-FP64 {tag} tier={tier} logits={lerr:.2e} loss={loss_err:.2e} worst_grad={worst}:{errs[worst]:.2e}")
    assert lerr < tol and loss_err < tol, (tag, lerr, loss_err)
    bad = {k: v for k, v in errs.items() if not v < (limits or {}).get(k, tol)}
    assert not bad, (tag, bad, errs)


# ---------------------------------------------------------------------------------------------
# (a) the generator == its numpy restatement
# ---------------------------------------------------------------------------------------------
SEEDS = [0, 1, 2 ** 32 - 1, 2 ** 32, 0x2F6B_91C3_5A07_D4E9, 2 ** 64 - 1]
THRESH = [0, 1, 26214, 32768, 65535, 65536]


@pytest.mark.parametrize("T,Bp", [(1, 1), (3, 37), (625, 128), (7, 4096)])
@pytest.mark.parametrize("seed", SEEDS)
def test_generator_equals_restatement(dev, seed, T, Bp):
    from neural_speech_decoding_b200 import ops
    like = torch.empty(1, device=dev)
    for th in THRESH:
        got = ops.dropout_mask_u8(like, seed, th, T, Bp).cpu().numpy()
        want = dh.dropout_mask_u8(seed, th, T, Bp)
        assert got.shape == (T, Bp, 48) and got.dtype == np.uint8
        assert np.array_equal(got, want), (seed, th, T, Bp, int((got != want).sum()))


# ---------------------------------------------------------------------------------------------
# (b) generator mode == mask-tensor mode, bit for bit
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["full", "half", "capped"])
@pytest.mark.parametrize("B,T", [(300, 37), (65, 12), (129, 2)])
@pytest.mark.parametrize("tier", ["x3", "tc"])
def test_generator_mode_equals_mask_mode(dev, checkpoint, tier, B, T, layout):
    """``p' = 1 - thresh16 / 65536`` makes the mask mode's scale 1 / (1 - p') exactly the generator's 65536 / thresh16 (in
    double and in fp32); ``p`` also sets the head dropout's scale, so both runs pass p'.  Then the only difference between
    the runs is where the keep-bits come from: the half-tile layout re-lays the mask tensor (ops._half_tile_rows) while the
    generator keys on the full-tile row, and the backward regenerates the forward's bits at row t + 1."""
    from neural_speech_decoding_b200 import ops
    x, y, rr, d2 = inputs(B, T, 1000 + B + T)
    x, y, rr, d2 = x.to(dev), y.to(dev), rr.to(dev), d2.to(dev)
    m = make_model(dev, checkpoint).train()
    if tier == "tc":
        m.compute_dtype = torch.bfloat16
    seed = 0x5DEECE66D_1234 + B
    for th in (TH06, 40000):
        p = 1.0 - th / 65536
        assert 1.0 / (1.0 - p) == 65536.0 / th
        mask = ops.dropout_mask_u8(x, seed, th, T, ops.padded_batch(B, ops.TC_TILE))
        with Layout(layout):
            a, ga = run_ops(m, tier, x, y, p, (seed, th), rr, d2)
            b, gb = run_ops(m, tier, x, y, p, mask, rr, d2)
        assert torch.isfinite(a).all()
        assert torch.equal(a, b), (th, (a - b).abs().max().item())
        for (k, _), u, v in zip(m.named_parameters(), ga, gb):
            assert torch.isfinite(u).all() and torch.equal(u, v), (th, k, (u - v).abs().max().item())


# ---------------------------------------------------------------------------------------------
# (c) generator mode against float64
# ---------------------------------------------------------------------------------------------
OPS_CASES = [(300, 37), (65, 12), (1, 1), (129, 2)]
# The 16-bit tier at B = 65, T = 12 (these inputs): the layer-0 gradients are up to 9.5e-2 from float64 on their own scale,
# the same on full and half tiles (layer 1: weight_ih 7.5e-2, bias 4.5e-2, weight_hh 2.4e-2; attn.weight, which the
# layer-1 BPTT also computes, 3.0e-2), while the exact tier is within 2.3e-6 of the same reference and mask, and generator mode
# equals mask mode bit for bit (test_generator_mode_equals_mask_mode).  Measured on an NVIDIA B200, this is the tier's fp16
# operand rounding on a small batch, not the dropout path or the ragged tile: other inputs at B = 65, T = 12 are within
# 3e-3, and with no dropout at all the tier is 6.9e-2 off on weight_ih_l0 in eval mode at B = 66, T = 12 and 3.4e-2 on
# weight_hh_l0 at B = 300, T = 12 (DESIGN §5, "Accuracy of the gradients").  The LayerNorm and fc tensors keep the 2e-2 contract.
TC_65_12_LIMITS = {**{f"lstm.{w}_l{l}": 0.12 for w in ("weight_ih", "weight_hh", "bias_ih", "bias_hh") for l in (0, 1)},
                   "attn.weight": 0.05}


@pytest.mark.parametrize("tier,B,T", [("tc", B, T) for B, T in OPS_CASES] + [("x3", B, T) for B, T in OPS_CASES])
def test_generator_mode_vs_fp64_through_ops(dev, checkpoint, tier, B, T):
    """Full and half tiles at the module's default p = 0.6 (thresh16 26214): the inter-layer dropout scaled by 65536 /
    thresh16, the head dropout by 1 / (1 - p)."""
    x, y, rr, d2 = inputs(B, T, 2000 + B + T)
    xd = x.to(dev)
    seed = 0x0123_4567_89AB_CDEF ^ B
    _, m1 = gen_mask(xd, seed, TH06, B, T)
    ref = fp64_reference(checkpoint, x, y, 0.6, m1, 65536.0 / TH06, rr, d2)
    m = make_model(dev, checkpoint).train()
    for layout in ("full", "half"):
        with Layout(layout):
            logits, grads = run_ops(m, tier, xd, y.to(dev), 0.6, (seed, TH06), rr.to(dev), d2.to(dev))
        limits = TC_65_12_LIMITS if (tier, B, T) == ("tc", 65, 12) else None
        check_against_fp64(f"B={B} T={T} {layout}", m, tier, T, logits, y.to(dev), grads, ref, limits)


def module_step(m, x, y, rr, d2, s):
    """The trainer's path: train mode, RReLU slopes and head dropout injected, the inter-layer dropout's seed the first
    CPU draw after torch.manual_seed(s)."""
    m.train()
    m.inject_noise(rrelu_slope=rr, drop2=d2)
    m.zero_grad()
    torch.manual_seed(s)
    out = m(x)
    F.cross_entropy(out, y).backward()
    return out.detach().clone(), [q.grad.detach().clone() for q in m.parameters()]


# The exact tier on 64 shipped windows x 625 steps in train mode: attn.weight 2.37e-5 and lstm.weight_ih_l0 1.43e-5 from
# float64 on their own scales (logits 1.2e-6, every other tensor within 6.4e-6), the same in mask-tensor mode (2.30e-5), so
# not the generator.  Measured on an NVIDIA B200, the error grows with T and with the noise: 1.9e-6 at T = 100, 6.4e-6 at
# T = 300, 7.1e-6 in eval mode at T = 625, 1.15e-5 at T = 625 with the head noise alone; the FFMA tier is 1.4e-6 and CPU
# fp32 autograd 3.3e-6 on the same case (DESIGN §6c, "Accuracy at production length").  Every other tensor keeps 1e-5.
X3_625_LIMITS = {"attn.weight": 3e-5, "lstm.weight_ih_l0": 3e-5}
MODULE_CASES = [(0.6, 64, 625, True), (0.25, 300, 37, False), (0.9, 300, 37, False)]


@pytest.mark.parametrize("tier,p,B,T,shipped", [(tier, *c) for tier in ("tc", "x3") for c in MODULE_CASES])
def test_generator_mode_vs_fp64_through_module(dev, checkpoint, windows, tier, p, B, T, shipped):
    """``EEG_LSTM(dropout=p)`` with the shipped weights in train mode, the layout the library picks (half tiles at these
    batches): the seed is rebuilt the way forward draws it and thresh16 = round((1 - p) * 65536)."""
    x, y, rr, d2 = inputs(B, T, 3000 + B + T, windows if shipped else None)
    d2 = (torch.rand(B, 32, generator=torch.Generator().manual_seed(B)) >= p).float()
    xd = x.to(dev)
    s = 4242 + B
    torch.manual_seed(s)
    seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    th = int(round((1.0 - p) * 65536))
    _, m1 = gen_mask(xd, seed, th, B, T)
    ref = fp64_reference(checkpoint, x, y, p, m1, 65536.0 / th, rr, d2)
    m = make_model(dev, checkpoint, dropout=p)
    if tier == "tc":
        m.compute_dtype = torch.bfloat16
    assert m._tier(xd, train=True) == tier
    logits, grads = module_step(m, xd, y.to(dev), rr.to(dev), d2.to(dev), s)
    again, _ = module_step(m, xd, y.to(dev), rr.to(dev), d2.to(dev), s)
    assert torch.equal(logits, again)                        # reproducible under torch.manual_seed
    other, _ = module_step(m, xd, y.to(dev), rr.to(dev), d2.to(dev), s + 1)
    assert not torch.equal(logits, other)                    # and a different seed draws a different mask
    limits = X3_625_LIMITS if (tier, T) == ("x3", 625) else None
    check_against_fp64(f"module p={p} B={B} T={T}", m, tier, T, logits, y.to(dev), grads, ref, limits)


# ---------------------------------------------------------------------------------------------
# (d) the ends of thresh16
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tier", ["x3", "tc"])
def test_thresh16_zero_drops_everything(dev, checkpoint, tier):
    """thresh16 = 0 (scale 0): layer 1 sees zeros, so layer 0 and layer 1's input weights get exactly zero gradients; every
    other tensor matches float64 on its own scale (grad_errors' rule)."""
    B, T = 130, 9
    x, y, rr, d2 = inputs(B, T, 77)
    ref = fp64_reference(checkpoint, x, y, 0.6, torch.zeros(B, T, 48, dtype=torch.float64), 0.0, rr, d2)
    m = make_model(dev, checkpoint).train()
    logits, grads = run_ops(m, tier, x.to(dev), y.to(dev), 0.6, (99, 0), rr.to(dev), d2.to(dev))
    names = [k for k, _ in m.named_parameters()]
    ref_logits, ref_loss, ref_grads = ref
    zero = {k for k in names if k.endswith("_l0") or k == "lstm.weight_ih_l1"}
    for k, g in zip(names, grads):
        if k in zero:
            assert not ref_grads[k].any() and not g.any(), k
    tol = EXACT_TOL if tier == "x3" else BF16_TOL
    assert np.abs(logits.cpu().numpy() - ref_logits).max() / np.abs(ref_logits).max() < tol
    with np.errstate(invalid="ignore"):                      # 0 / 0 on the tensors checked for exact zeros above
        errs = grad_errors(m, grads, ref_grads, tier, T)
    bad = {k: v for k, v in errs.items() if k not in zero and not v < tol}
    assert not bad, (bad, errs)


@pytest.mark.parametrize("half", [False, True])
def test_module_dropout_one(dev, checkpoint, half):
    """p = 1: thresh16 = 0 and the head dropout is total too, so every logit is fc.3.bias and only fc.3.bias gets a
    gradient, as in float64."""
    B, T = 70, 11
    x, y, rr, d2 = inputs(B, T, 5)
    d2 = torch.zeros(B, 32)
    ref_logits, _, ref_grads = fp64_reference(checkpoint, x, y, 1.0, torch.zeros(B, T, 48, dtype=torch.float64), 0.0, rr, d2)
    m = make_model(dev, checkpoint, dropout=1.0)
    if half:
        m.compute_dtype = torch.bfloat16
    assert m._tier(x.to(dev), train=True) == ("tc" if half else "x3")
    logits, grads = module_step(m, x.to(dev), y.to(dev), rr.to(dev), d2.to(dev), 1)
    assert torch.equal(logits, m.fc[3].bias.detach()[None].expand(B, -1))
    assert np.abs(logits.cpu().numpy() - ref_logits).max() == 0.0
    for (k, _), g in zip(m.named_parameters(), grads):
        if k == "fc.3.bias":
            assert np.abs(g.cpu().numpy() - ref_grads[k]).max() / np.abs(ref_grads[k]).max() < EXACT_TOL
        else:
            assert not g.any(), k


def saturating_input(B, T, seed):
    """Windows that drive layer 0's gates to saturation (|h0| within fp32 rounding of 1 on many units)."""
    gen = torch.Generator().manual_seed(seed)
    return torch.sign(torch.randn(B, T, 8, generator=gen)) * 400.0


def test_thresh16_one_exceeds_fp16_operands(dev, checkpoint):
    """thresh16 = 1 scales a kept h0 by 65536, and from |h0| >= 0.99976 that is past fp16's 65504, where both tiers hold
    the dropped h0 (the exact tier as its fp16 hi half).  Measured on an NVIDIA B200 before the ops refused it: the 16-bit
    tier gave non-finite logits on 2 of these 128 windows and non-finite gradients.  So the tensor-core training ops refuse
    a drop scale past 65504, in generator and in mask-tensor mode; thresh16 = 2 (scale 32768) still fits."""
    B, T = 128, 12
    x = saturating_input(B, T, 3).to(dev)
    m = make_model(dev, checkpoint).train()
    lstm, head = [m.lstm.layer(l) for l in range(2)], [h.detach() for h in m._head_params()]
    rr, d2 = torch.full((B, 32), 0.2, device=dev), torch.ones(B, 32, device=dev)
    for tier in ("x3", "tc"):
        with pytest.raises(ValueError, match="fp16"):
            train_fn(tier)(x, lstm, head, 0.6, False, (7, 1), rr, d2)
        with pytest.raises(ValueError, match="fp16"):
            train_fn(tier)(x, lstm, head, 1 - 1 / 65536, False, torch.ones(T, 128, 48, dtype=torch.uint8, device=dev), rr, d2)
    for tier in ("x3", "tc"):
        out = train_fn(tier)(x, lstm, head, 0.6, False, (7, 2), rr, d2)
        assert torch.isfinite(out).all(), tier


@pytest.mark.parametrize("half", [False, True])
def test_module_dropout_past_fp16_trains_on_ffma(dev, checkpoint, half):
    """p = 1 - 1 / 65536 (thresh16 = 1, scale 65536) on h-saturating windows: the module trains on the FFMA tier, which is
    finite and near float64 with the same (injected) masks.  The saturated layer-1 gates leave gradients that vanish
    on their own scale, and the scale amplifies fp32 rounding, so the gradients are checked for finiteness."""
    p = 1 - 1 / 65536
    B, T = 40, 12
    x = saturating_input(B, T, 4)
    gen = torch.Generator().manual_seed(6)
    y = torch.randint(0, 3, (B,), generator=gen)
    d1 = (torch.rand(1, B, T, 48, generator=gen) >= 0.6).float()
    rr = torch.empty(B, 32).uniform_(1 / 8, 1 / 3, generator=gen)
    d2 = (torch.rand(B, 32, generator=gen) >= 0.6).float()
    ref_logits, ref_loss, ref_grads = fp64_reference(checkpoint, x, y, p, d1[0].double(), None, rr, d2)
    assert np.isfinite(ref_logits).all()
    m = make_model(dev, checkpoint, dropout=p).train()
    if half:
        m.compute_dtype = torch.bfloat16
    xd = x.to(dev)
    assert m._tier(xd, train=True) == "ffma"
    m.inject_noise(drop1=d1, rrelu_slope=rr, drop2=d2)
    logits = m(xd)
    loss = F.cross_entropy(logits, y.to(dev))
    loss.backward()
    lg = logits.detach().cpu().numpy()
    assert np.isfinite(lg).all()
    # a scale of 65536 turns fp32's rounding of h0 (2^-24) into 2^-8 absolute in layer 1's input: measured 1.5e-2 from
    # float64 on the logits, a property of the problem at this scale, not of the tier
    assert np.abs(lg - ref_logits).max() / np.abs(ref_logits).max() < 5e-2
    for k, q in m.named_parameters():
        assert torch.isfinite(q.grad).all(), k
