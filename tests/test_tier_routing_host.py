"""Which kernel tier ``EEG_LSTM.decode``, ``decode_intermediates`` and ``forward`` pick, checked on the CPU.

Every tier entry point in ``ops`` (and the pack ops and ``window_zscore``) is replaced by a recorder that returns zeros of
the right shape, so these tests see the routing alone: the rules over ``compute_dtype``, the input and module dtypes, the
shape, the batch size, eval / eval with parameter gradients / train, ``x.requires_grad``, ``ops.EXACT_TC`` /
``ops.EXACT_TC_TRAIN`` and ``zscore_input``.  In train mode they also check the noise each training tier receives under
``torch.manual_seed``: seeded runs depend on the order of those draws.
"""
import itertools

import pytest
import torch

F32, F16, BF16 = torch.float32, torch.float16, torch.bfloat16
T = 12
SEED = 1234
SHAPES = {"flagship": {}, "h96": {"hidden_size": 96}, "h32x3": {"hidden_size": 32, "num_layers": 3},
          "k17": {"num_classes": 17}}


def expected_tier(m, x, grad_path: bool) -> str:
    """The routing rules, stated independently of the model code."""
    from neural_speech_decoding_b200 import ops
    lstm, K = m.lstm, m.fc[3].out_features
    half = BF16 in (m.compute_dtype, x.dtype, m.attn.weight.dtype)
    tc = (lstm.input_size, lstm.hidden_size, lstm.num_layers) == (8, 48, 2) and K <= 16
    wide = lstm.input_size == 8 and lstm.hidden_size in (96, 144, 192) and lstm.num_layers == 2 and K <= 16
    if not grad_path:
        if half and tc:
            return "tc"
        if half and wide:
            return "wide"
        if ops.EXACT_TC and not half and tc and x.dtype == F32 and x.shape[0] > 0:
            return "x3"
        return "ffma"
    no_dx = not x.requires_grad
    if half and tc and no_dx:
        return "tc"
    if half and wide and no_dx:
        return "wide"
    if ops.EXACT_TC_TRAIN and not half and tc and no_dx and x.dtype in (F32, F16, BF16):
        return "x3"
    return "ffma"


class Recorder:
    def __init__(self, monkeypatch):
        from neural_speech_decoding_b200 import ops
        self.calls = []
        rec = self.calls.append

        def two(x, head, want_probs):
            B, K = x.shape[0], head[6].shape[0]
            return torch.zeros(B, K), torch.zeros((B, K) if want_probs else (0,))

        def five(x, head):
            B, K, H = x.shape[0], head[6].shape[0], head[2].shape[0]
            return torch.zeros(B, K), torch.zeros(B, K), torch.zeros(B, x.shape[1]), torch.zeros(B, H), torch.zeros(B, H)

        def train(tier):
            def f(x, lstm_params, head_params, p, zscore=False, drop1=None, rrelu_slope=None, drop2_mask=None):
                rec(dict(tier=tier, fam="train", x=x, zscore=zscore, p=p, drop1=drop1, rr=rrelu_slope, d2=drop2_mask))
                return torch.zeros(x.shape[0], head_params[6].shape[0])
            return f

        def infer_tc(x, packed, head_params, want_probs=False, zscore=False):
            rec(dict(tier="tc", fam="decode", x=x, zscore=zscore, want_probs=want_probs))
            return two(x, head_params, want_probs)

        def infer_tc_ex(x, packed, head_params, zscore=False):
            rec(dict(tier="tc", fam="ex", x=x, zscore=zscore))
            return five(x, head_params)

        def infer_wide(x, packed, head_params, H, want_probs=False, zscore=False):
            rec(dict(tier="wide", fam="decode", x=x, zscore=zscore, want_probs=want_probs, H=H))
            return two(x, head_params, want_probs)

        def infer_wide_ex(x, packed, head_params, H, zscore=False):
            rec(dict(tier="wide", fam="ex", x=x, zscore=zscore, H=H))
            return five(x, head_params)

        def infer_x3(x, packed, head, want_probs):
            rec(dict(tier="x3", fam="decode", x=x, want_probs=want_probs))
            return two(x, head, want_probs)

        def infer_x3_ex(x, packed, head_params):
            rec(dict(tier="x3", fam="ex", x=x))
            return five(x, head_params)

        def infer(x, lstm_params, head_params, want_probs=False, zscore=False, packed=None):
            rec(dict(tier="ffma", fam="decode", x=x, zscore=zscore, want_probs=want_probs, layers=len(lstm_params)))
            return two(x, head_params, want_probs)

        def infer_ex(x, lstm_params, head_params, zscore=False, packed=None):
            rec(dict(tier="ffma", fam="ex", x=x, zscore=zscore, layers=len(lstm_params)))
            return five(x, head_params)

        def window_zscore(x, T, hop, normalize, time_major, out16, pad_to=32):
            out = x.float() + 0.0
            rec(dict(tier=None, fam="zscore", x=x, out=out, normalize=normalize, time_major=time_major, out16=out16))
            return out

        u8 = lambda *a, **k: torch.zeros(1, dtype=torch.uint8)
        for name, fn in dict(decoder_infer_tc=infer_tc, decoder_infer_tc_intermediates=infer_tc_ex,
                             decoder_infer_wide=infer_wide, decoder_infer_wide_intermediates=infer_wide_ex,
                             decoder_infer_x3=infer_x3, decoder_infer_x3_intermediates=infer_x3_ex,
                             decoder_infer=infer, decoder_infer_intermediates=infer_ex,
                             decoder_train_forward=train("ffma"), decoder_train_forward_tc=train("tc"),
                             decoder_train_forward_wide_tc=train("wide"), decoder_train_forward_x3=train("x3"),
                             window_zscore=window_zscore, decoder_pack_bf16=u8, decoder_pack_x3=u8,
                             decoder_pack_wide_bf16=u8,
                             pack_lstm_layer=lambda *a: (torch.zeros(1), torch.zeros(1))).items():
            monkeypatch.setattr(ops, name, fn)

    def take(self):
        out, self.calls[:] = list(self.calls), []
        return out


def _model(shape, mdt):
    from neural_speech_decoding_b200.lstm_eeg_model import EEG_LSTM
    torch.manual_seed(0)
    m = EEG_LSTM(**SHAPES[shape])
    return m.to(mdt) if mdt != F32 else m


def _check_tier_call(calls, want, fam, m, x):
    """One call into tier ``want`` of family ``fam`` (the x3 tier is preceded by the K1 z-score pass when zscore_input is
    on), with the model's zscore flag and the model's x."""
    if want == "x3" and fam != "train" and m.zscore_input:
        zs, call = calls
        assert zs["fam"] == "zscore" and zs["x"] is x and zs["normalize"] and not zs["time_major"] and zs["out16"] == 0
        assert call["x"] is zs["out"]
    else:
        (call,) = calls
        assert call["x"] is x
    assert (call["tier"], call["fam"]) == (want, fam)
    if call["tier"] != "x3" or fam == "train":
        assert call["zscore"] == m.zscore_input
    if call["tier"] == "wide" and fam != "train":
        assert call["H"] == m.lstm.hidden_size
    if call["tier"] == "ffma" and fam != "train":
        assert call["layers"] == m.lstm.num_layers
    return call


@pytest.mark.parametrize("mdt", [F32, BF16], ids=["module_f32", "module_bf16"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_decode_routing(cpu_backend, monkeypatch, shape, mdt):
    from neural_speech_decoding_b200 import ops
    from neural_speech_decoding_b200.lstm_eeg_model import DecoderOutputs
    rec = Recorder(monkeypatch)
    m = _model(shape, mdt).eval()
    K, H = m.fc[3].out_features, m.lstm.hidden_size
    for cdt, xdt, B, exact, z, xrg in itertools.product((F32, BF16), (F32, F16, BF16), (0, 5), (True, False),
                                                         (False, True), (False, True)):
        monkeypatch.setattr(ops, "EXACT_TC", exact)
        m.compute_dtype, m.zscore_input = cdt, z
        x = torch.randn(B, T, 8).to(xdt).requires_grad_(xrg)
        want = expected_tier(m, x, grad_path=False)
        ctx = (cdt, xdt, B, exact, z, xrg)
        for want_probs in (True, False):
            lg, pr = m.decode(x, want_probs=want_probs)
            call = _check_tier_call(rec.take(), want, "decode", m, x)
            assert call["want_probs"] == want_probs, ctx
            assert lg.shape == (B, K) and pr.shape == ((B, K) if want_probs else (0,)), ctx
        out = m.decode_intermediates(x)
        assert isinstance(out, DecoderOutputs)
        assert [tuple(t.shape) for t in out] == [(B, K), (B, K), (B, T), (B, H), (B, H)], ctx
        calls = rec.take()
        if B == 0:
            assert calls == [], ctx          # empty DecoderOutputs without a launch
        else:
            _check_tier_call(calls, want, "ex", m, x)


@pytest.mark.parametrize("mode", ["eval", "eval_param_grad", "train"])
@pytest.mark.parametrize("mdt", [F32, BF16], ids=["module_f32", "module_bf16"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_forward_routing(cpu_backend, monkeypatch, shape, mdt, mode):
    from neural_speech_decoding_b200 import ops
    rec = Recorder(monkeypatch)
    m = _model(shape, mdt).train(mode == "train")
    if mode == "eval":
        m.requires_grad_(False)
    K = m.fc[3].out_features
    for cdt, xdt, B, exact, exact_train, z, xrg in itertools.product(
            (F32, BF16), (F32, F16, BF16), (0, 5), (True, False), (True, False), (False, True), (False, True)):
        monkeypatch.setattr(ops, "EXACT_TC", exact)
        monkeypatch.setattr(ops, "EXACT_TC_TRAIN", exact_train)
        m.compute_dtype, m.zscore_input = cdt, z
        x = torch.randn(B, T, 8).to(xdt).requires_grad_(xrg)
        grad_path = mode != "eval" or xrg
        ctx = (cdt, xdt, B, exact, exact_train, z, xrg)
        torch.manual_seed(SEED)
        logits = m(x)
        assert logits.shape == (B, K) and logits.dtype == xdt, ctx
        calls = rec.take()
        if B == 0:
            assert calls == [], ctx
            continue
        want = expected_tier(m, x, grad_path)
        if not grad_path:
            call = _check_tier_call(calls, want, "decode", m, x)
            assert not call["want_probs"], ctx
            continue
        call = _check_tier_call(calls, want, "train", m, x)
        assert call["p"] == m.dropout_p, ctx
        _check_noise(call, want, m, B, injected={} if mode == "train" else None)


def _expected_noise(tier, m, B, injected):
    """The noise a train-mode forward draws after torch.manual_seed(SEED), in draw order, as the tier receives it:
    (drop1, rrelu_slope, drop2)."""
    p, L, H = m.dropout_p, m.lstm.num_layers, m.lstm.hidden_size
    pad = 32 if tier == "ffma" else 128
    Bp = max(pad, -(-B // pad) * pad)
    mask_dtype = torch.uint8 if tier in ("tc", "x3") else F32
    torch.manual_seed(SEED)
    d1 = None
    if L > 1 and m.lstm.dropout > 0.0:
        if injected.get("drop1") is not None:
            d1 = []
            for l in range(L - 1):
                t = torch.zeros((T, Bp, H), dtype=mask_dtype)
                t[:, :B] = injected["drop1"][l].permute(1, 0, 2).to(mask_dtype)
                d1.append(t)
        elif tier not in ("tc", "x3"):           # the flagship tensor-core tiers generate the keep-bits in the kernel
            d1 = [(torch.rand((T, Bp, H)) >= p).to(mask_dtype) for _ in range(L - 1)]
    rr = injected["rrelu"] if injected.get("rrelu") is not None else torch.empty((B, 32)).uniform_(1.0 / 8.0, 1.0 / 3.0)
    d2 = None
    if p > 0.0:
        d2 = injected["drop2"] if injected.get("drop2") is not None else (torch.rand((B, 32)) >= p).float()
    if tier == "ffma":
        return d1, rr, d2
    drop1 = d1[0] if d1 is not None else None
    if tier in ("tc", "x3") and d1 is None and m.lstm.dropout > 0.0:
        drop1 = (int(torch.randint(0, 2 ** 62, (1,)).item()), int(round((1.0 - p) * 65536)))
    return drop1, rr, d2


def _same(a, b):
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and a.dtype == b.dtype and torch.equal(a, b)
    if isinstance(a, list):
        return isinstance(b, list) and len(a) == len(b) and all(_same(u, v) for u, v in zip(a, b))
    return a == b


def _check_noise(call, tier, m, B, injected):
    """``injected`` None: no noise at all (eval mode with autograd)."""
    got = (call["drop1"], call["rr"], call["d2"])
    if injected is None:
        assert got == (None, None, None)
        return
    want = _expected_noise(tier, m, B, injected)
    for name, g, w in zip(("drop1", "rrelu_slope", "drop2"), got, want):
        assert _same(g, w), (tier, name, g, w)


@pytest.mark.parametrize("inject", ["none", "drop1", "all"])
@pytest.mark.parametrize("tier", ["tc", "x3", "wide", "ffma", "ffma_3_layers"])
def test_train_noise_seeded_and_injected(cpu_backend, monkeypatch, tier, inject):
    """The (drop1, rrelu_slope, drop2) each training tier receives, drawn under torch.manual_seed or injected."""
    from neural_speech_decoding_b200 import ops
    rec = Recorder(monkeypatch)
    monkeypatch.setattr(ops, "EXACT_TC_TRAIN", True)
    shape, cdt = {"tc": ("flagship", BF16), "x3": ("flagship", F32), "wide": ("h96", BF16), "ffma": ("k17", F32),
                  "ffma_3_layers": ("h32x3", F32)}[tier]
    m = _model(shape, F32).train()
    m.compute_dtype = cdt
    L, H, B = m.lstm.num_layers, m.lstm.hidden_size, 5
    injected = {}
    if inject != "none":
        g = torch.Generator().manual_seed(7)
        injected["drop1"] = (torch.rand((L - 1, B, T, H), generator=g) >= 0.6).float()
        if inject == "all":
            injected["rrelu"] = torch.empty((B, 32)).uniform_(0.15, 0.3, generator=g)
            injected["drop2"] = (torch.rand((B, 32), generator=g) >= 0.6).float()
        m.inject_noise(injected["drop1"], injected.get("rrelu"), injected.get("drop2"))
    x = torch.randn(B, T, 8)
    tier = tier.split("_")[0]
    for _ in range(2):                       # the same seed gives the same noise again
        torch.manual_seed(SEED)
        m(x)
        (call,) = rec.take()
        assert call["tier"] == tier
        _check_noise(call, tier, m, B, injected)
