"""The conv stack launch by launch on the B200: every tensor-core launch is recomputed in float64 from the operand
planes the GPU itself stored for its input (tests/precision_emulation.py) and its stored output must agree within

    |gpu - emu| <= beta * S + allowance(emu)

where S = pool(conv(|W|, |a|)) + |b| (carried through an in-launch intermediate layer), beta is the launch's bar
below and allowance(emu) the representation error of the output row format (pe.allowance: half an fp16 ulp,
2^-22 for hi | lo, ...).  A lost correction term is a
systematic error of ~2^-12 S; the bars sit at least 4x below such defects, except where
test_precision_emulation.SEPARATION records otherwise and why.

Variants are those of test_gpu_model.py::test_every_layer_against_oracle, plus weight-scale cases that push F8's
operands to the edges of the e4m3 range."""
import json
import logging
import math
import os

import numpy as np
import pytest
import torch

from oracle import preprocess_oracle as pp
from riser_b200.config import AttrDict
from riser_b200 import Model, synth, PREC_F16, PREC_F16_W2, PREC_F16_X3, PREC_F16_F8
from riser_b200.model import F8_A_SHIFT
from tests import precision_emulation as pe

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")
CFG = AttrDict({"cnn": {"n_layers": 12, "depth": 1, "channels": synth.CHANNELS, "kernels": [3] * 12,
                        "n_classes": 2, "classifier": "gap_fc"}})
LENGTHS = [4096, 5001, 7108, 12048, 12047, 8615, 4097]
MAX_LEN = 12048
POISON = 7.5

# name -> (RISER_FUSE_L0, precision, extra environment); the variants of test_every_layer_against_oracle
VARIANTS = {
    "f0-f16": (0, PREC_F16, {}), "f0-w2": (0, PREC_F16_W2, {}), "f0-x3": (0, PREC_F16_X3, {}),
    "f2-f16": (2, PREC_F16, {}), "f2-w2": (2, PREC_F16_W2, {}), "f2-x3": (2, PREC_F16_X3, {}),
    "f0-f8": (0, PREC_F16_F8, {}), "f2-f8": (2, PREC_F16_F8, {}),
    "f0-f8-from1": (0, PREC_F16_F8, {"RISER_F8_FROM": "1"}), "f2-f8-from1": (2, PREC_F16_F8, {"RISER_F8_FROM": "1"}),
    "f2-f8-from3": (2, PREC_F16_F8, {"RISER_F8_FROM": "3"}), "f2-f8-from6": (2, PREC_F16_F8, {"RISER_F8_FROM": "6"}),
    "f2-x3-flat": (2, PREC_F16_X3, {"RISER_EO": "0"}), "f0-f16-flat": (0, PREC_F16, {"RISER_EO": "0"}),
    "f2-f8-nopair": (2, PREC_F16_F8, {"RISER_PAIR": "0"}),
    "f2-f8-nofuse23": (2, PREC_F16_F8, {"RISER_FUSE23": "0"}), "f2-x3-nofuse23": (2, PREC_F16_X3, {"RISER_FUSE23": "0"}),
    "f2-x3-nokc": (2, PREC_F16_X3, {"RISER_KC": "0"}), "f2-f8-nokc": (2, PREC_F16_F8, {"RISER_KC": "0"}),
}
# default configuration, weights (and biases) of one layer scaled: layer-5 inputs up to ~850 / ~3,400 (beyond
# e4m3's 448), a layer whose weights sit 2^-10 lower (per-layer exponent, e4m3 weight subnormals), and a factor that
# is not a power of two
SCALES = {"l4x64": (4, 64.0, True), "l4x256": (4, 256.0, True), "l7w2m10": (7, 2.0 ** -10, False),
          "l6x37.5": (6, 37.5, True)}

# beta per term set, indexed by the first conv layer of the launch (1..11): 4x the largest max|gpu - emu| / S
# measured over every variant and scale case below (MEASURED: one B200, 1,000 W power limit), rounded up to a power
# of two and at least 2^-20.  Layer 1 includes layer 0 when the plan fuses it; in the F16 / W2 modes layer 0's
# single-fp16 output then flips at rounding ties, hence their bar there.  RMS_BAR bounds the RMS of that excess over
# every output the same way: a lost term is systematic and moves the RMS, accumulation noise mostly does not.
MEASURED = {
    pe.F16: [4.23e-05, 4.02e-08, 1.04e-07, 1.8e-07, 1.27e-07, 1.01e-07, 1.56e-07, 1.32e-07, 1.62e-07, 2.22e-07, 5.85e-07],
    pe.W2: [4.97e-05, 1.85e-07, 1.48e-07, 1.82e-07, 1.88e-07, 3.75e-07, 2.93e-07, 3.02e-07, 4.79e-07, 5.23e-07, 1.06e-06],
    pe.X3: [4.79e-07, 5.44e-07, 5.87e-07, 8.61e-07, 8.63e-07, 6.93e-07, 8.87e-07, 8.69e-07, 1.36e-06, 1.41e-06, 1.53e-06],
    pe.F8: [2.3e-06, 1.66e-08, 2.61e-08, 3.21e-08, 6.29e-08, 9.37e-08, 9.79e-08, 2.56e-07, 2.2e-07, 3.79e-07, 1.75e-06],
}
BETA = {t: [2.0 ** max(-20, math.ceil(math.log2(4 * m))) if m > 0 else 2.0 ** -20 for m in ms]
        for t, ms in MEASURED.items()}
RMS_BAR = {pe.F16: 2.0 ** -19, pe.W2: 2.0 ** -19, pe.X3: 2.0 ** -19, pe.F8: 2.0 ** -19}   # measured 2.3 / 2.3 / 2.9 / 2.8e-7
TERMS_NAME = {pe.F16: "F16", pe.W2: "W2", pe.X3: "X3", pe.F8: "F8"}


def _state(scale=None):
    sd = {k: v.clone() for k, v in synth.state_dict(0).items()}
    if scale:
        i, f, with_bias = scale
        sd[f"layers.{i}.0.weight"] *= f
        if with_bias:
            sd[f"layers.{i}.0.bias"] *= f
    return sd


def _inputs():
    rng = np.random.default_rng(0)
    normed = [pp.mad_normalise(synth.body(rng, n)) for n in LENGTHS]
    x = torch.full((len(LENGTHS), MAX_LEN), POISON)            # poison beyond each read's length
    for b, v in enumerate(normed):
        x[b, :len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float64)).float()
    return x.cuda(), torch.tensor(LENGTHS, dtype=torch.int32).cuda()


def _launches(plan, n):
    """(first, last) conv layer of every tensor-core launch, from the plan."""
    out, i = [], 1
    while i < n:
        j = i + 1 if i + 1 < n and plan.layer_format(i + 1) < 0 else i
        out.append((i, j))
        i = j + 1
    return out


def _planes64(planes, b, rows):
    return tuple(p[b, :rows].double() for p in planes)


def _check_format(planes, fmt, val, ctx):
    """The stored split is the one the format specifies: |lo| <= ulp(hi) / 2, a8 = e4m3(a 2^-F8_A_SHIFT) to a step."""
    hi = planes[0]
    if fmt == 2:
        lo = planes[1]
    elif fmt == 3:
        lo = planes[2] * 2.0 ** -(9 - pe.F8_LO_SHIFT)
        a8 = planes[1] * 2.0 ** F8_A_SHIFT
        bad = (a8 - val).abs() > 2.0 ** -3 * val.abs() + 2.0 ** (F8_A_SHIFT - 9)
        assert not bool(bad.any()), f"{ctx}: a8 is not e4m3(a * 2^-{F8_A_SHIFT})"
    else:
        return
    bad = lo.abs() > 2.0 ** -11 * hi.abs() * (1 + 2.0 ** -9) + 2.0 ** -24
    assert not bool(bad.any()), f"{ctx}: |lo| exceeds half an fp16 ulp of hi (split not round-to-nearest)"


def run_variant(fuse, precision, env, monkeypatch, scale=None):
    """Runs one forward and checks every launch; returns {launch key: (max ratio, rms ratio)}."""
    monkeypatch.setenv("RISER_FUSE_L0", str(fuse))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    state = _state(scale)
    model = Model(state, CFG, LOG, "mRNA", precision=precision)
    x, lens = _inputs()
    n = model.n_layers
    feat = torch.zeros(len(LENGTHS), synth.CHANNELS[-1], device="cuda")
    probs = model.classify_batch(x, lens, max_len=MAX_LEN, feat=feat)
    torch.cuda.synchronize()
    plan = model.plan(len(LENGTHS), MAX_LEN)
    assert plan.fused_layer0 == bool(fuse)
    W = [state[f"layers.{i}.0.weight"].cuda() for i in range(n)]
    Bs = [state[f"layers.{i}.0.bias"].cuda() for i in range(n)]
    packs = {}
    stats, failures = {}, []
    for (i, j) in _launches(plan, n):
        fmt_in = plan.layer_format(i)
        fmt_out = plan.layer_format(j + 1) if j + 1 < n else 0
        terms = pe.terms_of(abs(fmt_in), precision)
        key = f"L{i}{'+' + str(j) if j > i else ''}{'+0' if i == 1 and plan.fused_layer0 else ''}:" \
              f"{TERMS_NAME[terms]}:{plan.layer_kernel(i)}"
        src = None if (i == 1 and plan.fused_layer0) else plan.planes(i, n)
        out = plan.planes(j + 1, n, fmt_out or None)
        worst, sq, cnt = 0.0, 0.0, 0
        for b, L0 in enumerate(LENGTHS):
            rows_in, rows_out = L0 >> i, L0 >> (j + 1)
            if src is None:                                   # layer 0 inside layer 1's launch
                xs = x[b, :L0]
                a0 = pe.layer0_tc(xs, state["layers.0.0.weight"].cuda(), state["layers.0.0.bias"].cuda())
                s_in = pe.layer0_bound(xs, W[0], Bs[0])
                planes = pe.split_act(a0, fmt_in)
            else:
                planes = _planes64(src, b, rows_in)
                s_in = pe.act_value(planes, fmt_in).abs()
            for li in range(i, j + 1):
                if li not in packs:
                    packs[li] = pe.pack_weights(W[li])
                terms_l = pe.terms_of(fmt_in if li == i else 2, precision)
                y = pe.layer(planes, fmt_in if li == i else 2, W[li], Bs[li], terms_l, wp=packs[li])
                s_in = pe.bound(s_in, W[li], Bs[li])
                if li < j:                                    # conv_eo2_kernel's intermediate: hi + lo planes
                    planes = pe.split_act(y, 2)
            S = s_in
            got_planes = _planes64(out, b, out[0].shape[1])
            got = pe.act_value(got_planes, fmt_out)
            tail = torch.cat([p[rows_out:].reshape(-1) for p in got_planes])
            if bool((tail != 0).any()):
                failures.append((key, b, "rows beyond the valid length are not zero"))
            got = got[:rows_out]
            _check_format(tuple(p[:rows_out] for p in got_planes), fmt_out, got, f"{key} read {b}")
            d = (got - y).abs()
            if not bool(torch.isfinite(got).all()):
                failures.append((key, b, "non-finite output"))
                continue
            excess = (d - pe.allowance(y, fmt_out)).clamp_min(0) / S.clamp_min(1e-30)   # beyond the output's rounding
            worst = max(worst, float(excess.max()))
            sq += float((excess ** 2).sum())
            cnt += d.numel()
        rms = math.sqrt(sq / max(cnt, 1))
        stats[key] = (worst, rms)
        beta = BETA[terms][i - 1]
        if worst > beta or rms > RMS_BAR[terms]:
            failures.append((key, f"max {worst:.3g} (beta {beta:.3g})", f"rms {rms:.3g} (bar {RMS_BAR[terms]:.3g})"))
    record = os.environ.get("RISER_PRECISION_RECORD")
    if record:
        with open(record, "a") as f:
            f.write(json.dumps({"variant": [fuse, precision, env, scale], "stats": stats}) + "\n")
    # head: feat = float64 mean of the GPU's own act_n rows; probs = softmax of the head on that feat
    act = plan.planes(n, n)[0].double()
    want_feat = torch.stack([act[b, :L0 >> n].mean(0) for b, L0 in enumerate(LENGTHS)])
    fd = (feat.double() - want_feat).abs().max().item()
    assert fd <= 2.0 ** -22 * want_feat.abs().max().item() + 1e-30, ("feat", fd)
    logits = feat.double() @ state["classifier.2.weight"].double().cuda().T + state["classifier.2.bias"].double().cuda()
    pd = (probs.double() - torch.softmax(logits, 1)).abs().max().item()
    assert pd <= 1e-6, ("probs", pd)
    assert not failures, failures


@pytest.mark.parametrize("name", list(VARIANTS))
def test_every_launch_against_emulation(name, monkeypatch):
    fuse, precision, env = VARIANTS[name]
    run_variant(fuse, precision, env, monkeypatch)


@pytest.mark.parametrize("name", list(SCALES))
def test_f8_weight_scales_against_emulation(name, monkeypatch):
    run_variant(2, PREC_F16_F8, {}, monkeypatch, scale=SCALES[name])
