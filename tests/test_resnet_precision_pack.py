"""CPU: the ResNet's operand formats per precision mode.  pack_tc_weights against a byte-for-byte restatement (torch's
float16 / float8_e4m3fn casts, the SWIZZLE_64B order written out row by row); the e4m3 activation and weight rows of
F16_F8 against a scalar round-to-nearest-even e4m3 encoder, near saturation and in the subnormal range; the F8
weight operands at the scale _scale_exponent picks; and every lost correction term of the GPU's per-launch check
(tests/test_gpu_resnet_precision.py) standing at least 4x above its bar."""
import math

import numpy as np
import pytest
import torch

from oracle import preprocess_oracle as pp
from riser_b200 import synth
from riser_b200.model import F8_A_SHIFT, F8_LO_SHIFT, PREC_F16, PREC_F16_F8, PREC_F16_W2, PREC_F16_X3
from riser_b200.resnet import _fold, _scale_exponent, pack_tc_weights
from tests import resnet_emulation as emu
from tests.test_gpu_resnet_precision import BETA

MODES = {"f16": PREC_F16, "w2": PREC_F16_W2, "x3": PREC_F16_X3, "f8": PREC_F16_F8}


def e4m3_ref(x):
    """One float -> its e4m3 byte: round to nearest even, saturated to +-448 (__NV_SATFINITE), subnormal step 2^-9."""
    s = 0x80 if math.copysign(1.0, x) < 0 else 0
    a = abs(x)
    if a >= 448.0:
        return s | 0x7E
    if a < 2.0 ** -6:
        return s | int(round(a * 2.0 ** 9))             # 8 = the smallest normal, 2^-6, code 0x08
    m, ex = math.frexp(a)
    E = ex - 1
    q = int(round(a * 2.0 ** (3 - E)))                 # exact scaling: Python's round is half-to-even here
    if q == 16:
        E, q = E + 1, 8
    code = ((E + 7) << 3) | (q - 8)
    return s | min(code, 0x7E)


def e4m3_val(b):
    s = -1.0 if b & 0x80 else 1.0
    E, q = (b >> 3) & 15, b & 7
    return s * (q * 2.0 ** -9 if E == 0 else (8 + q) * 2.0 ** (E - 10))


def f16(x):
    return float(np.float16(np.float32(x)))


def restate_image(w, n_pad, cin_p, e, mode):
    """The image pack_tc_weights documents, built one 64-byte row at a time."""
    cout, cin, K = w.shape
    kb = (cin_p + 31) // 32
    ws = (w.double() * 2.0 ** e).float()
    n_planes = 1 if mode == PREC_F16 else 2
    img = bytearray()
    for t in range(K):
        for b in range(kb):
            for plane in range(n_planes):
                for r in range(n_pad):
                    row = bytearray(64)
                    for j in range(32):
                        c = 32 * b + j
                        v = float(ws[r, c, t]) if (r < cout and c < cin) else 0.0
                        hi = f16(v)
                        lo = np.float32(v) - np.float32(hi)
                        if plane == 0:
                            row[2 * j:2 * j + 2] = np.float16(hi).tobytes()
                        elif mode != PREC_F16_F8:
                            row[2 * j:2 * j + 2] = np.float16(lo).tobytes()
                        else:
                            row[j] = e4m3_ref(float(lo) * 2.0 ** F8_A_SHIFT)
                            row[32 + j] = e4m3_ref(v * 2.0 ** -(9 - F8_LO_SHIFT))
                    out = bytearray(64)
                    for ch in range(4):                      # 16-byte chunk ch lands at ch ^ ((r >> 1) & 3)
                        dst = ch ^ ((r >> 1) & 3)
                        out[16 * dst:16 * dst + 16] = row[16 * ch:16 * ch + 16]
                    img += out
    return bytes(img)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("shape,e", [((20, 20, 3), 9), ((40, 45, 1), 12), ((16, 8, 3), -3)])
def test_weight_image_matches_restatement(mode, shape, e):
    g = torch.Generator().manual_seed(sum(shape) + e)
    w = torch.randn(*shape, generator=g) * 2.0 ** -2
    w[0, 0, 0] = 60000.0 * 2.0 ** -e                   # near fp16's top: W_lo 2^3 reaches 128
    w.view(-1)[5:40] *= 2.0 ** -14                      # tiny weights: their e4m3 operands are subnormal or zero
    cout, cin, _ = shape
    n_pad, cin_p = (cout + 15) & ~15, (cin + 7) & ~7
    got = pack_tc_weights(w, n_pad, cin_p, e, MODES[mode])
    assert got.dtype == torch.uint8
    assert bytes(got.numpy()) == restate_image(w, n_pad, cin_p, e, MODES[mode])
    if mode == "x3":                                    # the default mode's image: the same call without a mode
        assert torch.equal(got, pack_tc_weights(w, n_pad, cin_p, e))


def test_e4m3_rows_restated():
    """F8 activation row [e4m3(a 2^-3) | e4m3((a - hi) 2^9)] and weight row [e4m3(W_lo 2^3) | e4m3(W 2^-9)] as the
    emulation (and pack_tc_weights) computes them, against the scalar encoder: saturation at |a| = 3584, the
    subnormal range, ties."""
    vals = [0.0, -0.0, 1e-9, 2.0 ** -12, 2.0 ** -9 * 3.5, 2.0 ** -6 * 0.99, 2.0 ** -6, 0.3, -1.7, 17.123, 255.9,
            3583.0, 3584.0, 3700.0, 3839.9, -3900.0, 5e4, 65504.0]
    rng = np.random.default_rng(3)
    vals += list(rng.normal(0, 1, 200) * 2.0 ** rng.integers(-14, 12, 200))
    a = torch.tensor(vals, dtype=torch.float32).to(torch.float64)
    hi, a8, lo8 = emu.split(a, emu.F8)
    for i, v in enumerate(a.tolist()):
        h = f16(v)
        assert float(hi[i]) == h
        assert e4m3_ref(float(a8[i])) == e4m3_ref(v * 2.0 ** -F8_A_SHIFT), v
        assert float(a8[i]) == e4m3_val(e4m3_ref(v * 2.0 ** -F8_A_SHIFT)), v
        assert float(lo8[i]) == e4m3_val(e4m3_ref((v - h) * 2.0 ** (9 - F8_LO_SHIFT))), v
    # e4m3's largest finite value, not NaN: a8 rounds to 448 from |a| = 3456 up and is clamped there above 3584
    assert [float(a8[vals.index(v)]) for v in (3583.0, 3584.0, 3700.0, -3900.0, 65504.0)] == [448.0, 448.0, 448.0, -448.0, 448.0]
    assert float(a8[vals.index(255.9)]) == 32.0
    # weight rows: the emulation's operands equal the bytes of the packed image
    w = torch.tensor(vals[:-2], dtype=torch.float32).view(1, -1, 1) * 2.0 ** -4
    wp = emu.weights(w, 4)
    for i in range(w.shape[1]):
        v = float(w[0, i, 0]) * 16.0
        lo = float(np.float32(v) - np.float32(f16(v)))
        assert float(wp["w8a"][0, i, 0]) == e4m3_val(e4m3_ref(lo * 2.0 ** F8_A_SHIFT)), v
        assert float(wp["w8l"][0, i, 0]) == e4m3_val(e4m3_ref(v * 2.0 ** -(9 - F8_LO_SHIFT))), v


@pytest.mark.parametrize("name", ["basic", "bottleneck"])
def test_f8_weight_operands_at_layer_scale(name):
    """At the scale _scale_exponent picks (max |W 2^e| in [2^11, 2^12)) the e4m3 weight operands are far from
    saturation (|W 2^-9| <= 8, |W_lo 2^3| <= 8: 448 is e4m3's largest), W 2^-9 is normal for every weight above 2^-8 of the layer's largest,
    and what the subnormal ones lose is below 2^-20 of the largest term either row carries."""
    cfg = synth.RESNET_CONFIGS[name]
    sd = {k: torch.as_tensor(v).float() for k, v in synth.resnet_state_dict(cfg, 0).items()}
    prefixes = sorted({k[:-len(".0.weight")] for k in sd if k.startswith("layers.") and k.endswith(".0.weight")})
    for p in prefixes:
        w, _ = _fold(sd[p + ".0.weight"], None, tuple(sd[p + ".1" + s] for s in
                                                       (".weight", ".bias", ".running_mean", ".running_var")))
        e = _scale_exponent(w)
        wp = emu.weights(w, e)
        v = w.double() * 2.0 ** e
        vmax = float(v.abs().max())
        assert 2.0 ** 11 <= vmax < 2.0 ** 12
        assert float(wp["w8l"].abs().max()) <= 8 and float(wp["w8a"].abs().max()) <= 8
        big = v.abs() >= vmax * 2.0 ** -8
        assert bool((wp["w8l"][big].abs() >= 2.0 ** -6).all())
        # subnormal steps 2^-9: the loss in weight units, against the largest weight
        loss_l = float(((wp["w8l"] - v * 2.0 ** -9).abs() * 2.0 ** 9)[~big].max()) if (~big).any() else 0.0
        loss_a = float((wp["w8a"] * 2.0 ** -3 - (v - wp["hi"])).abs().max())
        print(f"{name} {p}: e {e}, {int((~big).sum())} of {v.numel()} weights below 2^-8 max, "
              f"W row loss {loss_l / vmax:.1e}, W_lo row loss {loss_a / vmax:.1e} of max")
        assert loss_l * 2.0 ** -11 / vmax < 2.0 ** -20     # the lo8 operand it meets is <= 2^-11 of |a|
        assert loss_a / vmax < 2.0 ** -15


@pytest.fixture(scope="module")
def signals():
    bodies = synth.ragged_bodies(7, 3, 6000, 12048)
    return [pp.mad_normalise(b) for b in bodies]


@pytest.mark.parametrize("name", ["basic", "bottleneck"])
def test_lost_terms_stand_above_beta(signals, name):
    """Each lost correction term (W_lo in W2 and X3, a_lo in X3, either e4m3 term in F8) moves every launch by at least
    4x the bar of its mode and launch kind, on the excess quantity the GPU test asserts (with the fused launches'
    intermediate allowance)."""
    worst = {}
    for ln in emu.cpu_launches(name, signals[:2]):
        for mode_name, mode in MODES.items():
            y, S, allow = emu.run_launch(ln, mode)
            for m in emu.MUTANTS.get(mode, ()):
                ym, _, _ = emu.run_launch(ln, mode, m)
                ratio = emu.excess(ym, y, S, allow) / BETA[(mode_name, ln["kind"])]
                k = (mode_name, ln["kind"], m)
                worst[k] = min(worst.get(k, math.inf), ratio)
    for k, r in sorted(worst.items()):
        print(f"{name} {k}: smallest mutant / beta {r:.1f}")
        assert r >= 4, (k, r)
