"""CPU checks of the float64 launch emulation (tests/precision_emulation.py) the GPU per-launch test relies on:
its terms agree with an independent restatement, its intrinsic error per layer is the recorded one, every defect it
can inject is at least 4x above the GPU bar of test_gpu_precision.py, and the F16_F8 operands keep their accuracy
for activations beyond e4m3's 448."""
import math

import numpy as np
import pytest
import torch

from oracle import preprocess_oracle as pp
from riser_b200 import synth
from tests import precision_emulation as pe
from tests.test_gpu_precision import BETA

LENGTHS = (12048, 8615, 5001)
N_LAYERS = 12

# intrinsic max|emu - exact| / S per layer 1..11 (each layer fed the exact float64 input, synthetic model 0, the
# reads above), measured with this emulation; asserted with a 2x margin
INTRINSIC = {
    pe.X3: [6.2e-08, 4.8e-08, 4.1e-08, 3.3e-08, 2.8e-08, 2.2e-08, 1.7e-08, 1.3e-08, 1.2e-08, 9.0e-09, 6.0e-09],
    pe.F8: [1.62e-05, 1.22e-05, 1.00e-05, 6.89e-06, 5.18e-06, 4.02e-06, 2.95e-06, 2.45e-06, 2.44e-06, 1.95e-06,
            1.37e-06],
}


def _state():
    return {k: v.double() for k, v in synth.state_dict(0).items()}


@pytest.fixture(scope="module")
def chain():
    """Exact float64 inputs of layers 1..11 for the three reads: [read][layer] -> [L_i, C]."""
    sd = _state()
    rng = np.random.default_rng(0)
    out = []
    for n in LENGTHS:
        a = torch.from_numpy(np.asarray(pp.mad_normalise(synth.body(rng, n)), dtype=np.float64))[:, None]
        acts = [a]
        for i in range(N_LAYERS - 1):
            a = pe.exact_layer(a, sd[f"layers.{i}.0.weight"], sd[f"layers.{i}.0.bias"])
            acts.append(a)
        out.append(acts)
    return out


def _wb(i, sd=None):
    sd = sd or synth.state_dict(0)
    return sd[f"layers.{i}.0.weight"], sd[f"layers.{i}.0.bias"]


def _rel(y, ref, S):
    return float(((y - ref).abs() / S).max())


def _e4m3_ref(x):
    """Round to nearest-even e4m3 (3 mantissa bits, min normal 2^-6, subnormal step 2^-9), saturated at 448."""
    x = np.clip(np.asarray(x, dtype=np.float64), -448.0, 448.0)
    e = np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -6)))
    step = 2.0 ** (e - 3)
    return np.round(x / step) * step                     # np.round: half to even


def test_terms_match_independent_restatement():
    g = np.random.default_rng(3)
    L, cin, cout = 37, 24, 40
    w32 = (g.normal(0, 0.2, (cout, cin, 3))).astype(np.float32)
    b32 = g.normal(0, 0.05, cout).astype(np.float32)
    a = np.abs(g.normal(0, 3, (L, cin))) * (g.random((L, cin)) < 0.8)
    a[0, 0], a[1, 1] = 3000.0, 1e-3                     # past the old a8 range; an e4m3 subnormal
    e = 12 - math.frexp(float(np.abs(w32).max()))[1]
    v = w32.astype(np.float64) * 2.0 ** e
    whi = v.astype(np.float16).astype(np.float64)
    wlo = (v - whi).astype(np.float16).astype(np.float64)
    ahi = a.astype(np.float16).astype(np.float64)
    alo = (a - ahi).astype(np.float16).astype(np.float64)
    sa, sl = pe.F8_A_SHIFT, pe.F8_LO_SHIFT
    a8, lo8 = _e4m3_ref(a * 2.0 ** -sa), _e4m3_ref((a - ahi) * 2.0 ** (9 - sl))
    w8a, w8l = _e4m3_ref((v - whi) * 2.0 ** sa), _e4m3_ref(v * 2.0 ** -(9 - sl))

    def ref(terms):
        out = np.zeros((L // 2, cout))
        for t in range(L // 2):
            acc = np.zeros((2, cout))
            for p in range(2):
                for k in range(3):
                    r = 2 * t + p + k - 1
                    if 0 <= r < L:
                        acc[p] += sum(x[r] @ wt[:, :, k].T for x, wt in terms)
            out[t] = np.maximum(acc.max(0) * 2.0 ** -e + b32, 0)
        return out

    want = {pe.X3: ref([(ahi, whi), (alo, whi), (ahi, wlo)]), pe.F8: ref([(ahi, whi), (a8, w8a), (lo8, w8l)])}
    at, wt, bt = torch.from_numpy(a), torch.from_numpy(w32), torch.from_numpy(b32)
    for terms, fmt in ((pe.X3, 2), (pe.F8, 3)):
        got = pe.layer(pe.split_act(at, fmt), fmt, wt, bt, terms).numpy()
        np.testing.assert_allclose(got, want[terms], rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(pe.e4m3(torch.linspace(-500, 500, 20001, dtype=torch.float64)).numpy(),
                                  _e4m3_ref(np.linspace(-500, 500, 20001)))


def _intrinsic(chain, i, terms, mutant=None, sd=None):
    w, b = _wb(i, sd)
    fmt = 2 if terms == pe.X3 else 3
    wp = pe.pack_weights(w)
    worst = 0.0
    for acts in chain:
        a = acts[i]
        y = pe.layer(pe.split_act(a, fmt, mutant), fmt, w, b, terms, mutant, wp)
        worst = max(worst, _rel(y, pe.exact_layer(a, w.double(), b.double()), pe.bound(a.abs(), w, b)))
    return worst


@pytest.mark.parametrize("terms", [pe.X3, pe.F8])
def test_intrinsic_error_per_layer(chain, terms):
    got = [_intrinsic(chain, i, terms) for i in range(1, N_LAYERS)]
    bad = [(i + 1, g, r) for i, (g, r) in enumerate(zip(got, INTRINSIC[terms])) if not (r / 2 <= g <= 2 * r)]
    assert not bad, f"(layer, measured, recorded): {bad}; all: {['%.3g' % g for g in got]}"


IN_FMT = {pe.W2: 1, pe.X3: 2, pe.F8: 3}


def separation(chain, terms):
    """{(layer, mutant): deviation / beta} where deviation = max over outputs of (|stored(bad) - good| - allowance(good))
    / S: the quantity test_gpu_precision asserts, for a GPU that computed `bad` exactly and stored it."""
    fmt = IN_FMT[terms]
    out = {}
    for i in range(1, N_LAYERS):
        w, b = _wb(i)
        wp = pe.pack_weights(w)
        fmt_out = 0 if i == N_LAYERS - 1 else fmt
        for m in pe.MUTANTS[terms]:
            dev = 0.0
            for acts in chain:
                a = acts[i]
                S = pe.bound(a.abs(), w, b)
                good = pe.layer(pe.split_act(a, fmt), fmt, w, b, terms, None, wp)
                bad = pe.stored(pe.layer(pe.split_act(a, fmt, m), fmt, w, b, terms, m, wp), fmt_out)
                dev = max(dev, float(((bad - good).abs() - pe.allowance(good, fmt_out)).clamp_min(0).div(S).max()))
            out[(i, m)] = dev / BETA[terms][i - 1]
    return out


@pytest.mark.parametrize("terms", [pe.W2, pe.X3, pe.F8])
def test_mutants_stand_4x_above_the_gpu_bar(chain, terms):
    """Each injected defect moves some output of every layer by >= 4 beta S beyond the output format's rounding."""
    ratios = separation(chain, terms)
    weak = {k: round(r, 2) for k, r in ratios.items()
            if r < SEPARATION.get((terms, k[0]), 4.0) and k[1] not in NOT_SEPARABLE.get(terms, ())}
    assert not weak, f"(layer, mutant): deviation / beta below the required separation: {weak}"


# mutants that change the computed value by about as little as the fp32 accumulation does: with hi = fp16(a) either
# way, a8 = e4m3(hi 2^-3) and e4m3(a 2^-3) differ only at e4m3 rounding ties; a truncated hi leaves hi + lo exact
# (X3) and a truncated e4m3 operand moves a term of ~2^-12 S by one e4m3 step (F8: 0.5-2.6 beta in layers 1, 8, 10,
# 11).  The GPU test checks the stored split instead (|lo| <= ulp(hi) / 2, a8 to one e4m3 step).
NOT_SEPARABLE = {pe.X3: ("trunc",), pe.F8: ("a8_from_hi", "trunc")}
# Layer 11's bars (2^-17, from a measured 1.1-1.8e-6) stand only 3.5x below a lost correction term (W2, X3, F8) and,
# F8, 1.7x below a halved one (lo_scale_2p8): its K = 3 x 1135 accumulates the most fp32 truncation on the GPU.  W2's
# layer-1 launch includes layer 0, whose single-fp16 output flips at rounding ties against the float64 emulation; its
# bar (2^-12) is 0.6x of a lost W_lo there, so that launch does not see the defect (layers 2-10 do, 8.7x or more).
SEPARATION = {(pe.W2, 11): 1.5, (pe.X3, 11): 1.5, (pe.F8, 11): 1.5, (pe.W2, 1): 0.5}


# weight-scale cases: layer whose weights (and bias) are scaled, factor, scale the bias too, the F8 layers checked
# (every layer downstream of the scaled one).  l4x64 / l4x256 put layer-5 inputs at up to ~820 / ~3,280, beyond
# e4m3's 448; l6x37.5 is a factor that is not a power of two.
F8_RANGE = {"l4x64": (4, 64.0, True, (5, 6, 7, 8, 9, 10, 11)), "l4x256": (4, 256.0, True, (5, 6, 7, 8, 9, 10, 11)),
            "l6x37.5": (6, 37.5, True, (7, 8, 9, 10, 11)), "l7w2m10": (7, 2.0 ** -10, False, (7, 8, 9, 10, 11))}
# Activations far BELOW the synthetic heads' O(1-15) lie outside F8's range for any fixed pair of shifts: with layer
# 7's weights x 2^-10 (its bias not), layer 8's inputs are ~0.05 and the e4m3 operands reach their subnormals.  Layer 8
# is then 3.3x its in-range error (the unshifted operands: 2.6x); test_no_static_shift_keeps_small_activations_in_range
# shows that no shift pair does better than 2x.  LOW_RANGE_BAR is this case's own bar, in units of the in-range error.
LOW_RANGE = "l7w2m10"
LOW_RANGE_BAR = 4.0


_CHAINS = {}


def _scaled_chain(case):
    if case in _CHAINS:
        return _CHAINS[case]
    j, f, with_bias, _ = F8_RANGE[case]
    sd = _state()
    sd[f"layers.{j}.0.weight"] = sd[f"layers.{j}.0.weight"] * f
    if with_bias:
        sd[f"layers.{j}.0.bias"] = sd[f"layers.{j}.0.bias"] * f
    rng = np.random.default_rng(0)
    out = []
    for n in LENGTHS[:2]:
        a = torch.from_numpy(np.asarray(pp.mad_normalise(synth.body(rng, n)), dtype=np.float64))[:, None]
        acts = [a]
        for i in range(N_LAYERS - 1):
            a = pe.exact_layer(a, sd[f"layers.{i}.0.weight"], sd[f"layers.{i}.0.bias"])
            acts.append(a)
        out.append(acts)
    _CHAINS[case] = out, {k: v.float() for k, v in sd.items()}
    return _CHAINS[case]


def _f8_range_errors(case, shifts, layers=None):
    """{layer: F8 intrinsic max|emu - exact| / S / the layer's in-range value} with the given (a, lo) shifts."""
    chain, sd = _scaled_chain(case)
    sa, sl = shifts
    out = {}
    for i in layers or F8_RANGE[case][3]:
        w, b = _wb(i, sd)
        wp = pe.pack_weights(w, sa, sl)
        worst = 0.0
        for acts in chain:
            a = acts[i]
            y = pe.epilogue(pe.conv_acc(pe.split_act(a, 3, None, sa, sl), 3, wp, pe.F8), wp["e"], b.double())
            worst = max(worst, _rel(y, pe.exact_layer(a, w.double(), b.double()), pe.bound(a.abs(), w, b)))
        out[i] = worst / INTRINSIC[pe.F8][i - 1]
    return out


@pytest.mark.parametrize("case", [c for c in F8_RANGE if c != LOW_RANGE])
def test_f8_accuracy_beyond_448(case):
    """F8's intrinsic error in every layer downstream of the scaled one stays within 2x of its in-range value."""
    got = _f8_range_errors(case, (pe.F8_A_SHIFT, pe.F8_LO_SHIFT))
    bad = {i: round(g, 2) for i, g in got.items() if g > 2.0}
    assert not bad, f"layer: measured / in-range {bad}"


def test_f8_small_activations_recorded_limit():
    got = _f8_range_errors(LOW_RANGE, (pe.F8_A_SHIFT, pe.F8_LO_SHIFT))
    bad = {i: round(g, 2) for i, g in got.items() if g > LOW_RANGE_BAR}
    assert not bad, f"layer: measured / in-range {bad}"


def test_no_static_shift_keeps_small_activations_in_range():
    """Layer 8 of the small-activation case exceeds 2x its in-range error for every (a, lo) shift pair that keeps the
    high-range case l4x256 within 2x, and for the unshifted operands: the limit is the format's, not the choice."""
    for sa in range(0, 6):
        for sl in range(0, 3):
            low = _f8_range_errors(LOW_RANGE, (sa, sl), (8,))[8]
            if low <= 2.0:
                high = max(_f8_range_errors("l4x256", (sa, sl), (5, 8)).values())
                assert high > 2.0, ((sa, sl), low, high)


def test_unshifted_f8_operands_saturate_beyond_448():
    """Without the exponent shifts (a8 = e4m3(a), lo8 = e4m3((a - hi) 2^9)) layer 5 degrades 3.7x at inputs of ~820
    and 13x at ~3,280: the defect the a8 shift removes."""
    for case, factor in (("l4x64", 3.0), ("l4x256", 10.0)):
        got = _f8_range_errors(case, (0, 0), (5,))
        assert got[5] > factor, (case, got)
