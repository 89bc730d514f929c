"""Float64 emulation of what one launch of the ResNet's tensor-core kernel (riser_res_tc_ex, csrc/resnet_tc.cu) is
specified to compute in each precision mode, from the fp32 input it reads (test infrastructure, beside
precision_emulation.py whose fp16 / e4m3 roundings it shares; runs on whatever device the tensors live on).

Activations are [rows, channels] float64 tensors of ONE read, rows = its valid length (rows beyond it read as zero).
Weights are the folded float32 [cout, cin, k]; the kernel multiplies them by 2^e (e = resnet._scale_exponent) and
undoes it in the epilogue.

Operands per mode (the kernel converts fp32 activations itself, so a launch's operands follow from its input):
  F16: a_hi W_hi      W2: a_hi (W_hi + W_lo)      X3: a_hi W_hi + a_lo W_hi + a_hi W_lo
  F8 : a_hi W_hi + a8 e4m3(W_lo 2^F8_A_SHIFT) + lo8 e4m3(W 2^-(9 - F8_LO_SHIFT)),
       a8 = e4m3(a 2^-F8_A_SHIFT), lo8 = e4m3((a - a_hi) 2^(9 - F8_LO_SHIFT))
A fused BasicBlock: mid = ReLU(conv1(x) + b1) on rows [0, n_out), converted to the mode's operands in the kernel,
then out = ReLU(conv2(mid) + shortcut conv(x) + b2 + residual).  The GPU's mid is its fp32 accumulation, which can
round to the neighbouring fp16 (or e4m3) code where the float64 value lies near a rounding midpoint; `mid_allowance`
bounds what such a flip moves the output by.

Mutants (a lost correction term): drop_wlo (W2, X3), drop_alo (X3), drop_a8 / drop_lo8 (F8).
"""
import torch

from riser_b200.model import F8_A_SHIFT, F8_LO_SHIFT, PREC_F16 as F16, PREC_F16_F8 as F8, PREC_F16_W2 as W2, \
    PREC_F16_X3 as X3
from tests.precision_emulation import e4m3, fp16

MUTANTS = {W2: ("drop_wlo",), X3: ("drop_alo", "drop_wlo"), F8: ("drop_a8", "drop_lo8")}
E4M3_SAT_A = 448.0 * 2.0 ** F8_A_SHIFT        # |a| at which a8 = e4m3(a 2^-F8_A_SHIFT) saturates: 3584


def split(a, mode):
    """The A operand planes the kernel builds from the value a: (hi,), (hi, lo) or (hi, a8, lo8)."""
    hi = fp16(a)
    if mode == X3:
        return hi, fp16(a - hi)
    if mode == F8:
        return hi, e4m3(a * 2.0 ** -F8_A_SHIFT), e4m3((a - hi) * 2.0 ** (9 - F8_LO_SHIFT))
    return (hi,)


def weights(w, e):
    """Weight operands in scaled units (w 2^e), [cout, cin, k] float64: hi, lo, w8a, w8l."""
    v = w.to(torch.float32).to(torch.float64) * 2.0 ** e       # exact: a power-of-two scale of a float32
    hi = v.to(torch.float16).to(torch.float64)
    d = v - hi                                                  # exact in float32, as the host computes it
    return {"e": e, "hi": hi, "lo": d.to(torch.float16).to(torch.float64),
            "w8a": e4m3(d * 2.0 ** F8_A_SHIFT), "w8l": e4m3(v * 2.0 ** -(9 - F8_LO_SHIFT))}


def conv(a, w, stride, pad, n_out):
    """Conv1d of a [n_in, cin] (zero outside) with w [cout, cin, k]: rows [0, n_out) of the output."""
    k = w.shape[2]
    n = stride * max(n_out - 1, 0) + k
    p = a.new_zeros(max(n, pad + a.shape[0]), a.shape[1])
    p[pad:pad + a.shape[0]] = a
    return sum(p[t:t + stride * (n_out - 1) + 1:stride] @ w[:, :, t].T for t in range(k))


def acc(planes, wp, mode, stride, pad, n_out, mutant=None):
    """The launch's fp32 accumulator in scaled weight units, computed exactly."""
    hi = planes[0]
    if mode == F16:
        return conv(hi, wp["hi"], stride, pad, n_out)
    if mode == W2:
        return conv(hi, wp["hi"] if mutant == "drop_wlo" else wp["hi"] + wp["lo"], stride, pad, n_out)
    y = conv(hi, wp["hi"], stride, pad, n_out)
    if mode == X3:
        if mutant != "drop_alo":
            y = y + conv(planes[1], wp["hi"], stride, pad, n_out)
        if mutant != "drop_wlo":
            y = y + conv(hi, wp["lo"], stride, pad, n_out)
        return y
    if mutant != "drop_a8":
        y = y + conv(planes[1], wp["w8a"], stride, pad, n_out)
    if mutant != "drop_lo8":
        y = y + conv(planes[2], wp["w8l"], stride, pad, n_out)
    return y


def single(x, n_out, w, b, e, stride, pad, mode, residual=None, relu=True, mutant=None):
    """One conv launch: (emulated output, bound S = conv(|a|, |W|) + |b| (+ |residual|)), [n_out, cout]."""
    w64 = w.to(torch.float64)
    y = acc(split(x, mode), weights(w, e), mode, stride, pad, n_out, mutant) * 2.0 ** -e + b.to(torch.float64)
    S = conv(x.abs(), w64.abs(), stride, pad, n_out) + b.to(torch.float64).abs()
    if residual is not None:
        y = y + residual
        S = S + residual.abs()
    return (torch.relu(y) if relu else y), S


def fused(x, n_out, c1, c2, sc, stride, mode, residual=None, mutant=None):
    """A fused BasicBlock launch.  c1 = (w1, b1, e1), c2 = (w2, b2, e2), sc = shortcut weight [cout, cin, 1] or None
    (its bias folded into b2, its scale e2).  -> (output, S, mid, S1) with S = conv2(|mid|, |W2|) + conv(|x|, |Wsc|)
    + |b2| (+ |residual|) and S1 the bound of the intermediate."""
    (w1, b1, e1), (w2, b2, e2) = c1, c2
    mid, S1 = single(x, n_out, w1, b1, e1, stride, 1, mode, mutant=mutant)
    wp2 = weights(w2, e2)
    a2 = acc(split(mid, mode), wp2, mode, 1, 1, n_out, mutant)
    S = conv(mid, w2.to(torch.float64).abs(), 1, 1, n_out) + b2.to(torch.float64).abs()
    if sc is not None:
        a2 = a2 + acc(split(x, mode), weights(sc, e2), mode, stride, 0, n_out, mutant)
        S = S + conv(x.abs(), sc.to(torch.float64).abs(), stride, 0, n_out)
    y = a2 * 2.0 ** -e2 + b2.to(torch.float64)
    if residual is not None:
        y = y + residual
        S = S + residual.abs()
    return torch.relu(y), S, mid, S1


def mid_allowance(mid, S1, w2, e2, mode, delta=2.0 ** -20):
    """What the GPU's intermediate, within delta * S1 of the float64 one, can move conv2 by through a different
    operand code: per plane, |plane(mid + d) - plane(mid - d)| against |that plane's weights| (F16 hi.W_hi, W2
    hi.(W_hi + W_lo), X3 hi.(W_hi + W_lo) + lo.W_hi, F8 hi.W_hi + a8.w8a + lo8.w8l), in output units."""
    d = delta * S1
    n_out = mid.shape[0]
    wp = weights(w2, e2)
    hi_w = wp["hi"] + wp["lo"] if mode in (W2, X3) else wp["hi"]
    plane_w = {F16: [hi_w], W2: [hi_w], X3: [hi_w, wp["hi"]], F8: [hi_w, wp["w8a"], wp["w8l"]]}[mode]
    out = mid.new_zeros(n_out, w2.shape[0])
    for p_hi, p_lo, w in zip(split(mid + d, mode), split(mid - d, mode), plane_w):
        out = out + conv((p_hi - p_lo).abs(), w.abs(), 1, 1, n_out)
    return out * 2.0 ** -e2


def excess(gpu, emu, S, allow=None):
    """max over elements of (|gpu - emu| - allowance) / S: the quantity the per-launch bars hold (0 where S = 0)."""
    d = (gpu - emu).abs()
    if allow is not None:
        d = (d - allow).clamp_min(0)
    return float(torch.where(S > 0, d / S.clamp_min(1e-300), d * 1e300).max()) if d.numel() else 0.0


def cpu_launches(name, signals, seed=0):
    """The tensor-core launches of ResNetModel's forward for the synthetic configuration `name`, restated on the CPU
    for a few normalised signals: dicts with kind ("fused" / "single"), the folded weights, scales and the launch's
    float32 input per read (as float64 [rows, channels]), each block's input computed exactly from the previous one.
    Basic blocks are fused launches, bottleneck convolutions single ones (as on the GPU)."""
    import torch.nn.functional as F
    from riser_b200 import synth
    from riser_b200.resnet import _fold, _scale_exponent
    from oracle import resnet_oracle as ro
    cfg = synth.RESNET_CONFIGS[name]
    sd = {k: torch.as_tensor(v).float() for k, v in synth.resnet_state_dict(cfg, seed).items()
          if not k.endswith("num_batches_tracked")}

    def bn(p):
        return tuple(sd[p + s] for s in (".weight", ".bias", ".running_mean", ".running_var"))

    def folded(p):
        return _fold(sd[p + ".0.weight"], None, bn(p + ".1"))

    out = []
    for sig in signals:
        with torch.no_grad():
            h = torch.as_tensor(sig, dtype=torch.float32)[None, None]
            h = F.conv1d(h, sd["conv_block.0.weight"], sd["conv_block.0.bias"], stride=cfg["stride"],
                         padding=cfg["padding"])
            h = F.max_pool1d(torch.relu(ro._bn(h, sd, "conv_block.1")), 2, stride=2, padding=1)
        h = h[0].T.to(torch.float64)                               # [rows, channels]
        cin = cfg["channels"][0]
        for i in range(cfg["n_layers"]):
            cout = cfg["channels"][i]
            for j in range(cfg["blocks"][i]):
                stride = 2 if (i > 0 and j == 0) else 1
                p = f"layers.{i}.{j}"
                sc = folded(p + ".shortcut") if (cin != cout or stride != 1) else None
                x = h.float().to(torch.float64)                       # the launch reads float32
                if cfg["block"] != "bottleneck":
                    (w1, b1), (w2, b2) = folded(p + ".blocks.0"), folded(p + ".blocks.1")
                    n_out = (x.shape[0] + 2 - 3) // stride + 1
                    e1, e2 = _scale_exponent(w1), _scale_exponent(w2, *([sc[0]] if sc is not None else []))
                    b2s = b2 + (sc[1] if sc is not None else 0)
                    out.append(dict(kind="fused", x=x, n_out=n_out, c1=(w1, b1, e1), c2=(w2, b2s, e2),
                                    sc=None if sc is None else sc[0], stride=stride, residual=None if sc else x,
                                    name=p))
                    h, _, _, _ = fused(x, n_out, (w1, b1, e1), (w2, b2s, e2), None if sc is None else sc[0], stride,
                                       X3, residual=None if sc else x)
                else:
                    res = x
                    n_out = (x.shape[0] - 1) // stride + 1
                    if sc is not None:
                        e = _scale_exponent(sc[0])
                        out.append(dict(kind="single", x=x, n_out=n_out, w=sc[0], b=sc[1], e=e, stride=stride, pad=0,
                                        residual=None, relu=False, name=p + ".shortcut"))
                        res, _ = single(x, n_out, sc[0], sc[1], e, stride, 0, X3, relu=False)
                        res = res.float().to(torch.float64)
                    y = x
                    for k, (s, pad) in enumerate(((1, 0), (stride, 1), (1, 0))):
                        w, b = folded(p + f".blocks.{k}")
                        e = _scale_exponent(w)
                        n_k = (y.shape[0] + 2 * pad - w.shape[2]) // s + 1
                        r = res if k == 2 else None
                        out.append(dict(kind="single", x=y, n_out=n_k, w=w, b=b, e=e, stride=s, pad=pad, residual=r,
                                        relu=True, name=p + f".blocks.{k}"))
                        y, _ = single(y, n_k, w, b, e, s, pad, X3, residual=r)
                        y = y.float().to(torch.float64)
                    h = y
                cin = cout
    return out


def run_launch(ln, mode, mutant=None):
    """A cpu_launches entry in `mode` (optionally with a mutant): (output, S, allowance or None)."""
    if ln["kind"] == "single":
        y, S = single(ln["x"], ln["n_out"], ln["w"], ln["b"], ln["e"], ln["stride"], ln["pad"], mode,
                      residual=ln["residual"], relu=ln["relu"], mutant=mutant)
        return y, S, None
    y, S, mid, S1 = fused(ln["x"], ln["n_out"], ln["c1"], ln["c2"], ln["sc"], ln["stride"], mode,
                          residual=ln["residual"], mutant=mutant)
    return y, S, mid_allowance(mid, S1, ln["c2"][0], ln["c2"][2], mode)
