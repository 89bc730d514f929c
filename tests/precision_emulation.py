"""Float64 emulation of what one tensor-core launch of the conv stack (csrc/convnet.cu) is specified to compute,
given the operand planes it reads (test infrastructure; runs on whatever device the tensors live on).

Activations are [rows, channels] float64 tensors of ONE read, rows = its valid length; rows beyond it are zero in
the kernels, which is the convolution's 'same' padding.  Weights are the checkpoint's float32 [cout, cin, 3].

Row formats (riser_plan_layer_format): 1 = fp16, 2 = fp16 hi | fp16 lo, 3 = fp16 hi | e4m3 a8 | e4m3 lo8 with
a8 = e4m3(a * 2^-F8_A_SHIFT) and lo8 = e4m3((a - hi) * 2^(9 - F8_LO_SHIFT)).  Planes are held in stored units
(a8 and lo8 as the e4m3 values, not rescaled).

Term sets of one conv layer (the weights carry a per-layer power-of-two scale 2^e, undone in the epilogue):
  F16: a_hi W_hi          W2: + a_hi W_lo          X3: a_hi W_hi + a_lo W_hi + a_hi W_lo
  F8 : a_hi W_hi + a8 e4m3(W_lo 2^F8_A_SHIFT) + lo8 e4m3(W 2^-(9 - F8_LO_SHIFT))

Mutants: the same computation with one defect, named by a string:
  drop_alo / drop_wlo   X3 without a_lo W_hi / a_hi W_lo (W2: without a_hi W_lo)
  drop_a8 / drop_lo8    F8 without the a8 (W_lo) / the lo8 (a_lo) product
  lo_scale_2p8          lo8 written as (a - hi) * 2^(8 - F8_LO_SHIFT): the a_lo term halved
  a8_from_hi            a8 = e4m3(hi * 2^-F8_A_SHIFT) instead of e4m3(a * 2^-F8_A_SHIFT)
  trunc                 every rounding of the activation split truncates instead of rounding to nearest
Encoding mutants (a8_from_hi, lo_scale_2p8, trunc) act where activations are split (split_act); the others where
terms are summed (conv_acc).
"""
import math

import torch

from riser_b200.model import F8_A_SHIFT, F8_LO_SHIFT

F16, W2, X3, F8 = 0, 1, 2, 3
E4M3_MAX = 448.0
F16_MAX = 65504.0
MUTANTS = {W2: ("drop_wlo",), X3: ("drop_alo", "drop_wlo", "trunc"),
           F8: ("drop_a8", "drop_lo8", "lo_scale_2p8", "a8_from_hi", "trunc")}


def _toward_zero(x, r, dt, int_dt):
    """r = x rounded to nearest in dt (as float64); step the ones whose magnitude grew one code toward zero."""
    q = x.to(dt)
    up = r.abs() > x.abs()
    bits = q.view(int_dt)
    bits = torch.where(up & (bits & 0x7FFF if int_dt == torch.int16 else bits & 0x7F).ne(0), bits - 1, bits)
    return bits.view(dt).to(torch.float64)


def fp16(x, trunc=False):
    """fp16 round-to-nearest (or toward zero), saturated to +-65504 as the epilogues' sat_half2 does."""
    x = x.clamp(-F16_MAX, F16_MAX)
    r = x.to(torch.float16).to(torch.float64)
    return _toward_zero(x, r, torch.float16, torch.int16) if trunc else r


def e4m3(x, trunc=False):
    """__nv_cvt_float_to_fp8(x, __NV_SATFINITE, __NV_E4M3): torch's cast returns NaN above 448, so clamp first."""
    x = x.clamp(-E4M3_MAX, E4M3_MAX)
    r = x.to(torch.float8_e4m3fn).to(torch.float64)
    return _toward_zero(x, r, torch.float8_e4m3fn, torch.uint8) if trunc else r


def split_act(a, fmt, mutant=None, a_shift=None, lo_shift=None):
    """The planes an epilogue stores for the value a (float64): (hi,), (hi, lo) or (hi, a8, lo8)."""
    sa = F8_A_SHIFT if a_shift is None else a_shift
    sl = F8_LO_SHIFT if lo_shift is None else lo_shift
    tr = mutant == "trunc"
    hi = fp16(a, tr)
    if fmt == 1:
        return (hi,)
    if fmt == 2:
        return hi, fp16(a - hi, tr)
    a8 = e4m3((hi if mutant == "a8_from_hi" else a) * 2.0 ** -sa, tr)
    lo8 = e4m3((a - hi) * 2.0 ** ((8 if mutant == "lo_scale_2p8" else 9) - sl), tr)
    return hi, a8, lo8


def act_value(planes, fmt, lo_shift=None):
    """The value a stored row stands for (Plan.activation's decoding)."""
    sl = F8_LO_SHIFT if lo_shift is None else lo_shift
    if fmt == 2:
        return planes[0] + planes[1]
    if fmt == 3:
        return planes[0] + planes[2] * 2.0 ** -(9 - sl)
    return planes[0]


def half_ulp16(y):
    """Half the fp16 spacing at |y| (2^-25 in the subnormal range): fp16 round-to-nearest moves y by at most this."""
    e = torch.floor(torch.log2(y.abs().clamp_min(2.0 ** -14)))
    return 2.0 ** (e - 11)


def stored(y, fmt):
    """The value an epilogue's output row carries for y: rounded to the format and decoded (0 = fp32, the head)."""
    if fmt == 0:
        return y.to(torch.float32).to(torch.float64)
    return act_value(split_act(y, fmt), fmt)


def allowance(y, fmt, lo_shift=None):
    """Largest |stored(y) - y| the output format allows: its representation error, per element.  fp16: half an ulp;
    hi | lo: 2^-22; F8 rows: lo8's 3 mantissa bits on |a - hi| <= half an fp16 ulp, plus half of e4m3's subnormal
    step 2^-9 in value units, plus what lo8 loses to saturation above |a| = 2048 (2^-3 at most below 4096); fp32: 2^-24."""
    sl = F8_LO_SHIFT if lo_shift is None else lo_shift
    if fmt == 1:
        return half_ulp16(y) * (1 + 2.0 ** -20)
    if fmt == 2:
        return 2.0 ** -22 * y.abs() + 2.0 ** -48
    if fmt == 3:                                   # + lo8's saturation at 448 once half an ulp of hi exceeds it
        h = half_ulp16(y)
        return 2.0 ** -4 * h + 2.0 ** -(19 - sl) + (h - E4M3_MAX * 2.0 ** -(9 - sl)).clamp_min(0)
    return 2.0 ** -24 * y.abs() + 2.0 ** -149


def weight_exponent(w):
    """riser_model_create: the weights are stored times 2^e, e = 12 - frexp exponent of max|w|, clamped to +-24."""
    wmax = float(w.abs().max())
    if not (wmax > 0 and math.isfinite(wmax)):
        return 0
    return max(-24, min(24, 12 - math.frexp(wmax)[1]))


def pack_weights(w, a_shift=None, lo_shift=None):
    """Weight operands of one layer in scaled units, [cout, cin, 3] float64: hi, lo, w8a, w8l and the exponent e."""
    sa = F8_A_SHIFT if a_shift is None else a_shift
    sl = F8_LO_SHIFT if lo_shift is None else lo_shift
    e = weight_exponent(w)
    v = w.to(torch.float32).to(torch.float64) * 2.0 ** e        # exact: a power-of-two scale of a float32
    hi = v.to(torch.float16).to(torch.float64)
    d = v - hi                                                  # exact in float32, as the host computes it
    return {"e": e, "hi": hi, "lo": d.to(torch.float16).to(torch.float64),
            "w8a": e4m3(d * 2.0 ** sa), "w8l": e4m3(v * 2.0 ** -(9 - sl))}


def conv(a, w):
    """'same' Conv1d, k = 3, of a [L, cin] with w [cout, cin, 3] (no bias): [L, cout]."""
    z = a.new_zeros(1, a.shape[1])
    p = torch.cat([z, a, z])
    L = a.shape[0]
    return sum(p[k:k + L] @ w[:, :, k].T for k in range(3))


def pool(y):
    """MaxPool1d(2, 2) over rows: the valid rows of the next layer are L // 2."""
    n = y.shape[0] // 2
    return torch.maximum(y[0:2 * n:2], y[1:2 * n:2])


def conv_acc(planes, fmt, wp, terms, mutant=None):
    """The fp32 accumulator of the layer, in scaled weight units, computed exactly."""
    hi = planes[0]
    if terms == F16:
        return conv(hi, wp["hi"])
    if terms == W2:
        return conv(hi, wp["hi"] if mutant == "drop_wlo" else wp["hi"] + wp["lo"])
    if terms == X3:
        acc = conv(hi, wp["hi"])
        if mutant != "drop_alo":
            acc = acc + conv(planes[1], wp["hi"])
        if mutant != "drop_wlo":
            acc = acc + conv(hi, wp["lo"])
        return acc
    assert fmt == 3
    acc = conv(hi, wp["hi"])
    if mutant != "drop_a8":
        acc = acc + conv(planes[1], wp["w8a"])
    if mutant != "drop_lo8":
        acc = acc + conv(planes[2], wp["w8l"])
    return acc


def epilogue(acc, e, bias):
    """max-pool, acc * 2^-e + bias, ReLU (the epilogues' fmaxf(fmaf(max(ev, ov), inv_scale, b), 0))."""
    return torch.relu(pool(acc) * 2.0 ** -e + bias)


def layer(planes, fmt, w, bias, terms, mutant=None, wp=None):
    """One conv layer from its stored input planes: the float64 value its epilogue rounds to the output format."""
    wp = pack_weights(w) if wp is None else wp
    return epilogue(conv_acc(planes, fmt, wp, terms, mutant), wp["e"], bias.to(torch.float64))


def exact_layer(a, w, bias):
    """Conv1d + ReLU + MaxPool in float64 (the operation itself)."""
    return torch.relu(pool(conv(a, w.to(torch.float64))) + bias.to(torch.float64))


def bound(a_abs, w, bias):
    """S: the same conv with |W| and |a| plus |b|, max-pooled.  |error| <= beta * S survives ReLU and the pool."""
    return pool(conv(a_abs, w.to(torch.float64).abs())) + bias.to(torch.float64).abs()


def layer0_tc(x, w0, b0):
    """Layer 0 as fused01_kernel computes it on the tensor pipe (DESIGN section 4): x (clamped to the fp16 range) and
    the taps split hi + lo in fp16, the bias as hi + lo through a column of ones, x_lo * w_lo dropped; then the
    mid-epilogue's max-pool and ReLU.  x: float [L] signal of one read -> [L // 2, cout0] float64."""
    x = x.to(torch.float64).clamp(-F16_MAX, F16_MAX)[:, None]
    xh = fp16(x)
    xl = fp16(x - xh)
    w = w0.to(torch.float32).to(torch.float64)
    wh = w.to(torch.float16).to(torch.float64)
    wl = (w - wh).to(torch.float16).to(torch.float64)
    b = b0.to(torch.float32).to(torch.float64)
    bh = b.to(torch.float16).to(torch.float64)
    bl = (b - bh).to(torch.float16).to(torch.float64)
    y = conv(xh, wh) + conv(xl, wh) + conv(xh, wl) + bh + bl
    return torch.relu(pool(y))


def layer0_bound(x, w0, b0):
    return pool(conv(x.to(torch.float64).abs()[:, None], w0.to(torch.float64).abs())) + b0.to(torch.float64).abs()


def terms_of(fmt, precision):
    """Term set a layer runs from its input format and the model's precision mode."""
    return {2: X3, 3: F8}.get(fmt, W2 if precision == W2 else F16)
