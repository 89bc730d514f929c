"""The dedicated ConvNet kernels of csrc/convnet.cu at shapes other than the shipped network's.

Model sends every k = 3, depth-1, 'gap_fc', two-class ConvNet with 2..16 layers and a layer 0 of at most 64 channels
to these kernels, and riser_plan_create picks each layer's kernel, N tile, row format and layout from the shape.  The
shapes below are picked so that the shape alone (default environment) makes the plan choose what the shipped network
never does; PLANS pins those choices, so that a change of a plan heuristic updates this table on purpose.  Each shape
is then checked in every precision three ways: every tensor-core launch against the float64 emulation of its operand
formats (tests/precision_emulation.py), layer0_kernel against float64 where layer 0 is not fused, and the
probabilities end to end against the float64 reference module.  `first80` is the one shape the kernels cannot take
(layer 0 wider than 64 channels): Model runs it on GenericConvNet."""
import logging
import math

import numpy as np
import pytest
import torch

from oracle import control_oracle as ctl
from oracle import preprocess_oracle as pp
from oracle.convnet_module import ConvNet as RefConvNet
from riser_b200 import Model, decide, synth, _lib, PREC_F16, PREC_F16_W2, PREC_F16_X3, PREC_F16_F8
from riser_b200.config import AttrDict, CNN_SHIPPED
from tests import precision_emulation as pe
from tests.test_gpu_model import PROB_TOL
from tests.test_gpu_precision import BETA, RMS_BAR, POISON, check_every_launch

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")

SHAPES = {
    "two_fused_last": [18, 30],
    "narrow16": [16, 40, 96, 200],
    "kc18": [18, 26, 56, 72, 130],
    "fused24": [24, 32, 33, 47, 80, 129, 257],
    "first64": [64, 64, 100, 300, 600],
    "deep13": [8, 16, 16, 24, 32, 48, 64, 96, 128, 192, 256, 384, 512],
    "first80": [80, 96, 128],
}
GENERIC = {"first80"}
PRECISIONS = {"f16": PREC_F16, "w2": PREC_F16_W2, "x3": PREC_F16_X3, "f8": PREC_F16_F8}
MAX_LEN = 16000

F01, TC, EO, EO2, PAIR = "fused01_kernel", "conv_tc_kernel", "conv_eo_kernel", "conv_eo2_kernel", "conv_pair_kernel"
# shape -> precision -> (fused_layer0, one row per conv layer 1..n-1: (layer_kernel, layer_format, layer_eo, N tile))
PLANS = {
    "two_fused_last": {
        "f16": (False, [(TC, 1, 0, 32)]),
        "w2": (False, [(TC, 1, 0, 32)]),
        "x3": (False, [(TC, 2, 0, 32)]),
        "f8": (False, [(TC, 2, 0, 32)]),
    },
    "narrow16": {
        "f16": (False, [(TC, 1, 0, 48), (EO, 1, 1, 96), (TC, 1, 0, 208)]),
        "w2": (False, [(TC, 1, 0, 48), (EO, 1, 1, 96), (TC, 1, 0, 208)]),
        "x3": (False, [(TC, 2, 0, 48), (EO, 2, 1, 96), (TC, 2, 0, 208)]),
        "f8": (False, [(TC, 2, 0, 48), (EO, 2, 1, 96), (TC, 2, 0, 208)]),
    },
    "kc18": {
        "f16": (True, [(F01, 1, 0, 32), (EO, 1, 1, 64), (EO, 1, 1, 80), (TC, 1, 0, 144)]),
        "w2": (True, [(F01, 1, 0, 32), (EO, 1, 1, 64), (EO, 1, 1, 80), (TC, 1, 0, 144)]),
        "x3": (True, [(F01, 2, 0, 32), (EO, 2, 1, 64), (EO, 2, 1, 80), (TC, 2, 0, 144)]),
        "f8": (True, [(F01, 2, 0, 32), (EO, 2, 1, 64), (EO, 2, 1, 80), (TC, 2, 0, 144)]),
    },
    "fused24": {
        "f16": (True, [(F01, 1, 0, 32), (EO, 1, 1, 48), (EO, 1, 1, 48), (EO, 1, 1, 80), (TC, 1, 0, 144), (TC, 1, 0, 144)]),
        "w2": (True, [(F01, 1, 0, 32), (EO, 1, 1, 48), (EO, 1, 1, 48), (EO, 1, 1, 80), (TC, 1, 0, 144), (TC, 1, 0, 144)]),
        "x3": (True, [(F01, 2, 0, 32), (EO2, 2, 1, 48), (EO2, -1, 1, 48), (EO, 2, 1, 80), (TC, 2, 0, 144), (TC, 2, 0, 144)]),
        "f8": (True, [(F01, 2, 0, 32), (EO2, 2, 1, 48), (EO2, -1, 1, 48), (EO, 2, 1, 80), (TC, 3, 0, 144), (PAIR, 3, 0, 144)]),
    },
    "first64": {
        "f16": (False, [(TC, 1, 0, 64), (EO, 1, 1, 112), (TC, 1, 0, 160), (TC, 1, 0, 208)]),
        "w2": (False, [(TC, 1, 0, 64), (EO, 1, 1, 112), (TC, 1, 0, 160), (TC, 1, 0, 208)]),
        "x3": (False, [(TC, 2, 0, 64), (EO, 2, 1, 112), (TC, 2, 0, 160), (TC, 2, 0, 208)]),
        "f8": (False, [(TC, 2, 0, 64), (EO, 2, 1, 112), (TC, 2, 0, 160), (TC, 2, 0, 208)]),
    },
    "deep13": {
        "f16": (False, [(TC, 1, 0, 16), (EO, 1, 1, 16), (EO, 1, 1, 32), (EO, 1, 1, 32), (TC, 1, 0, 48), (TC, 1, 0, 64), (TC, 1, 0, 96), (TC, 1, 0, 128), (TC, 1, 0, 192), (TC, 1, 0, 256), (TC, 1, 0, 192), (TC, 1, 0, 256)]),
        "w2": (False, [(TC, 1, 0, 16), (EO, 1, 1, 16), (EO, 1, 1, 32), (EO, 1, 1, 32), (TC, 1, 0, 48), (TC, 1, 0, 64), (TC, 1, 0, 96), (TC, 1, 0, 128), (TC, 1, 0, 192), (TC, 1, 0, 256), (TC, 1, 0, 192), (TC, 1, 0, 256)]),
        "x3": (False, [(TC, 2, 0, 16), (EO2, 2, 1, 16), (EO2, -1, 1, 32), (EO, 2, 1, 32), (TC, 2, 0, 48), (TC, 2, 0, 64), (TC, 2, 0, 96), (TC, 2, 0, 128), (TC, 2, 0, 192), (TC, 2, 0, 256), (TC, 2, 0, 192), (TC, 2, 0, 256)]),
        "f8": (False, [(TC, 2, 0, 16), (EO2, 2, 1, 16), (EO2, -1, 1, 32), (EO, 2, 1, 32), (TC, 3, 0, 48), (TC, 3, 0, 64), (TC, 3, 0, 96), (PAIR, 3, 0, 128), (PAIR, 3, 0, 192), (PAIR, 3, 0, 256), (PAIR, 3, 0, 192), (PAIR, 3, 0, 256)]),
    },
}


def _cfg(name):
    ch = SHAPES[name]
    return AttrDict({"model": "cnn", "cnn": {"n_layers": len(ch), "depth": 1, "channels": ch, "kernels": [3] * len(ch),
                                             "n_classes": 2, "classifier": "gap_fc"}})


def _state(name):
    return synth.generic_cnn_state_dict(_cfg(name).cnn, 3)


def _plan_rows(plan, n):
    eo = _lib.lib().riser_plan_layer_eo
    return plan.fused_layer0, [(plan.layer_kernel(i), plan.layer_format(i), int(eo(plan._handle, i)),
                                plan.layer_info(i + 1)[4]) for i in range(1, n)]


def _cases(shapes):
    return [pytest.param(s, p, id=f"{s}-{p}") for s in shapes for p in PRECISIONS]


DEDICATED = [s for s in SHAPES if s not in GENERIC]
UNFUSED = [s for s in DEDICATED if not PLANS[s]["f16"][0]]


def _uses_kc(name, p):
    """fused01_kernel runs its K-concatenated form (fused01_kernel<4>) when riser_model_create builds the operand for
    it: F16_X3 and an even layer 0 of at most 20 channels (layer 1 then has one 32-wide N tile)."""
    c0 = SHAPES[name][0]
    return PRECISIONS[p] == PREC_F16_X3 and c0 <= 20 and c0 % 2 == 0


def _pair_n_last(name, i, n_tile):
    """conv_pair_kernel's N tiles of layer i: 256 wide but the last, which takes the rest of cout_p."""
    cout_p = -(-SHAPES[name][i] // n_tile) * n_tile
    return cout_p - (-(-cout_p // 256) - 1) * 256, min(256, cout_p)


@pytest.mark.parametrize("name,prec", _cases(SHAPES))
def test_plan_choices_are_pinned(name, prec):
    model = Model(_state(name), _cfg(name), LOG, "mRNA", precision=PRECISIONS[prec])
    if name in GENERIC:
        assert model._generic is not None
        return
    assert model._generic is None
    fused, rows = _plan_rows(model.plan(3, MAX_LEN), model.n_layers)
    assert (fused, rows) == PLANS[name][prec], (fused, rows)


def test_plan_table_reaches_what_the_shipped_plan_does_not():
    shipped = {}
    for prec, p in PRECISIONS.items():
        model = Model(synth.state_dict(0), AttrDict({"cnn": dict(CNN_SHIPPED)}), LOG, "mRNA", precision=p)
        for kernel, _, _, nt in _plan_rows(model.plan(3, MAX_LEN), 12)[1]:
            shipped.setdefault(kernel, set()).add(nt)
    reached = set()
    for name, by_prec in PLANS.items():
        ch = SHAPES[name]
        n = len(ch)
        for prec, (fused, rows) in by_prec.items():
            if fused and rows[0][0] == F01 and ch[0] != 20:
                reached.add("fused01_kernel, layer 0 width != 20, K-concatenated" if _uses_kc(name, prec)
                            else "fused01_kernel, layer 0 width != 20, three passes")
            if not fused and ch[0] <= 16:
                reached.add("layer0_kernel <= 16 channels")
            if not fused and ch[0] == 64:
                reached.add("layer0_kernel 64 channels")
            for i, (kernel, _, _, nt) in enumerate(rows, 1):
                if kernel in (EO, EO2) and nt not in shipped[kernel]:
                    reached.add(f"{kernel} at an N tile the shipped plan does not use")
                if kernel == PAIR:
                    n_last, n_tile = _pair_n_last(name, i, nt)
                    if n_last < n_tile:
                        reached.add("conv_pair_kernel with a narrower last N tile")
            if n != 12:
                reached.add("a layer other than 11 writes the fp32 last activation")
            if n == 2:
                reached.add("n_layers == 2")
            if n >= 13:
                reached.add("n_layers >= 13")
    assert reached == {
        "fused01_kernel, layer 0 width != 20, K-concatenated", "fused01_kernel, layer 0 width != 20, three passes",
        "layer0_kernel <= 16 channels", "layer0_kernel 64 channels",
        f"{EO} at an N tile the shipped plan does not use", f"{EO2} at an N tile the shipped plan does not use",
        "conv_pair_kernel with a narrower last N tile", "a layer other than 11 writes the fp32 last activation",
        "n_layers == 2", "n_layers >= 13"}, reached


# Bars per term set, from the shipped network's table (test_gpu_precision.BETA, RMS_BAR), not loosened: a launch that
# contains layer 0 takes the shipped layer-1 bar, every other launch the largest shipped bar of layers 2..11.  The widths
# here stay within the shipped ones, so no K is longer than what those bars were measured at.
# Measured max |gpu - emu| / S on one B200 (1,000 W power limit), per shape, F16 / W2 / X3 / F8, launches without layer 0
# (with it):
#   two_fused_last 2.1e-07  5.4e-07  8.6e-07  8.6e-07
#   narrow16       2.6e-07  5.3e-07  7.5e-07  7.5e-07
#   kc18           3.2e-07 (4.5e-05)  6.7e-07 (3.5e-05)  8.7e-07 (2.6e-07)  8.7e-07 (2.6e-07)
#   fused24        2.5e-07 (3.8e-05)  4.7e-07 (4.1e-05)  7.0e-07 (2.0e-07)  6.7e-07 (2.0e-07)
#   first64        4.0e-07  7.2e-07  1.1e-06  1.1e-06
#   deep13         2.4e-07  4.6e-07  8.1e-07  6.4e-07
# against bars of 3.8e-06 / 7.6e-06 / 7.6e-06 / 7.6e-06 (2.4e-04 / 2.4e-04 / 3.8e-06 / 1.5e-05 with layer 0); the RMS
# of every launch stayed <= 1.8e-07 (bar 1.9e-06).
def _beta(i, terms, with_l0):
    return BETA[terms][0] if with_l0 else max(BETA[terms][1:])


@pytest.mark.parametrize("name,prec", _cases(DEDICATED))
def test_every_launch_against_emulation(name, prec):
    n = len(SHAPES[name])
    lengths = [L for L in (4096, 4097, 9999, MAX_LEN, 8193) if L >= 2 ** n]
    _, stats = check_every_launch(_state(name), _cfg(name), PRECISIONS[prec], lengths, MAX_LEN, _beta,
                                  record=[name, prec])
    print(name, prec, {k: f"{m:.3g} / {r:.3g}" for k, (m, r) in stats.items()})


def _batch(normed, lengths, rows=None):
    """fp32 [rows, MAX_LEN] on the device, POISON past each read's length; rows > len(lengths) repeats the reads."""
    K = len(lengths)
    x = torch.full((K, MAX_LEN), POISON)
    for b, v in enumerate(normed):
        x[b, :len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float64)).float()
    idx = torch.arange(rows or K) % K
    return x[idx].cuda(), torch.tensor(lengths, dtype=torch.int32)[idx].cuda()


def _reads(n, seed):
    """Lengths of the ragged batch: 4096, 4097, odd, max_len, 0, 2^n - 1 and, for deep networks, lengths between
    4096 and 2^n; normalised bodies (empty for length 0)."""
    lengths = [4096, 4097, 9999, MAX_LEN, 0, 2 ** n - 1, 8192, 8193, 5001, 12347]
    rng = np.random.default_rng(seed)
    return lengths, [pp.mad_normalise(synth.body(rng, L)) if L else np.zeros(0) for L in lengths]


@pytest.mark.parametrize("name,prec", _cases(UNFUSED))
def test_unfused_layer0_against_float64(name, prec):
    """layer0_kernel's act_1: fp32 conv + bias + ReLU + max-pool rounded to layer 1's row format, against float64.
    Beyond the format's allowance, the fp32 arithmetic (three fmas) adds at most 3 * 2^-24 S, and the lo plane of a
    hi | lo row, an fp16 itself, has the subnormal step 2^-24 below 2^-14 (measured max excess / S on one B200:
    8e-08 for single fp16 rows; 1.8e-06 for hi | lo rows without the 2^-25 term)."""
    state = _state(name)
    model = Model(state, _cfg(name), LOG, "mRNA", precision=PRECISIONS[prec])
    lengths, normed = _reads(model.n_layers, 11)
    x, lens = _batch(normed, lengths)
    model.classify_batch(x, lens, max_len=MAX_LEN)
    torch.cuda.synchronize()
    plan = model.plan(len(lengths), MAX_LEN)
    assert not plan.fused_layer0
    fmt = plan.layer_format(1)
    planes = plan.planes(1, model.n_layers)
    w0, b0 = state["layers.0.0.weight"].cuda(), state["layers.0.0.bias"].cuda()
    worst = 0.0
    for b, L in enumerate(lengths):
        got_planes = tuple(p[b].double() for p in planes)
        rows = L >> 1
        assert all(bool((p[rows:] == 0).all()) for p in got_planes), (b, "rows beyond the valid length are not zero")
        if not rows:
            continue
        xs = x[b, :L].double()
        want = pe.exact_layer(xs[:, None], w0, b0)
        S = pe.layer0_bound(xs, w0, b0)
        d = (pe.act_value(got_planes, fmt)[:rows] - want).abs()
        excess = (d - pe.allowance(want, fmt) - (2.0 ** -25 if fmt == 2 else 0)).clamp_min(0) / S.clamp_min(1e-30)
        worst = max(worst, float(excess.max()))
    print(name, prec, f"layer 0: max excess / S {worst:.3g}")
    assert worst <= 2.0 ** -22, worst


def _reference(name, normed, lengths):
    net = RefConvNet(_cfg(name).cnn).double()
    net.load_state_dict({k: v.double() for k, v in _state(name).items()})
    n = len(SHAPES[name])
    want = np.full((len(lengths), 2), np.nan)
    with torch.no_grad():
        for b, (v, L) in enumerate(zip(normed, lengths)):
            if L >= 2 ** n:
                want[b] = torch.softmax(net(torch.from_numpy(np.asarray(v, dtype=np.float64))[None]), 1)[0].numpy()
    return want


@pytest.mark.parametrize("name,prec", _cases(SHAPES))
def test_probs_against_reference(name, prec):
    """A ragged batch repeated to 300 rows: the first copy against the float64 reference one read at a time, NaN rows
    for reads shorter than 2^n_layers and for length 0, every replica bit-identical to the first, and decide() on these
    probabilities against the control rule."""
    p = PRECISIONS[prec]
    model = Model(_state(name), _cfg(name), LOG, "mRNA", precision=p)
    n = model.n_layers
    lengths, normed = _reads(n, 12)
    K, R = len(lengths), 300
    x, lens = _batch(normed, lengths, R)
    probs = model.classify_batch(x, lens, max_len=MAX_LEN)
    got = probs.cpu().numpy()
    want = _reference(name, normed, lengths)
    live = [b for b, L in enumerate(lengths) if L >= 2 ** n]
    dead = [b for b in range(K) if b not in live]
    err = np.abs(got[:K][live] - want[live]).max()
    print(name, prec, f"max |dp| {err:.3g}")
    assert err < PROB_TOL[p], err
    assert np.isnan(got[:K][dead]).all()
    src = np.arange(R) % K
    rep = np.isin(src, live)
    assert np.array_equal(got[rep], got[src[rep]])
    assert np.isnan(got[~rep]).all()
    lens_h = lens.cpu().numpy()
    for mode in ("enrich", "deplete"):
        for thr in (0.9, 0.3, 0.5):
            dec = decide(probs[None], lens, thr, mode, MAX_LEN).cpu().numpy()
            for b in range(R):
                if lens_h[b] == 0:
                    assert dec[b] == ctl.SKIPPED
                    continue
                want_d = ctl.decide([torch.tensor(got[b, 1])], [torch.tensor(got[b, 0])], int(lens_h[b]), MAX_LEN,
                                    thr, mode)
                assert dec[b] == want_d, (mode, thr, b)


def test_classify_refuses_reads_too_short_for_the_last_pool():
    """Model.classify takes the reference's contract: a signal that leaves no row for the last pool raises."""
    model = Model(_state("deep13"), _cfg("deep13"), LOG, "mRNA")
    assert model._generic is None
    rng = np.random.default_rng(13)
    y = pp.mad_normalise(synth.body(rng, 8192))
    with pytest.raises(RuntimeError):
        model.classify(y[:8191])
    with pytest.raises(RuntimeError):
        model.classify(y[:4096])
    got = model.classify(y).cpu().numpy()
    want = _reference("deep13", [y], [8192])[0]
    assert np.abs(got - want).max() < PROB_TOL[PREC_F16_F8]
