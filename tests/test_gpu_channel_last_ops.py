"""The channel-last building blocks of the ResNet variant and the generic ConvNet, op by op, against plain float64
references at the shapes the model-level tests do not reach: riser_res_tc_ex (csrc/resnet_tc.cu) with a read that fits
one tile, more work items than resident CTAs, both staging depths and 8,191 tiles per read; riser_conv1d_cl (tiled and
per-element kernels), riser_stem_pool_cl (templated and generic kernels), riser_maxpool1d_pad_cl, riser_len_chain and
riser_gap_linear_softmax (csrc/resnet.cu).  Then the models built on them at lengths whose last stage fits one tile.

Conventions of every op test:
  * the output is filled with a NaN bit pattern before the launch; rows at or beyond a read's output length must still
    hold it afterwards (ResNetModel and GenericConvNet reuse their activation buffers on that contract), and input rows
    at or beyond a read's length are NaN, so a kernel that reads one shows it;
  * batches are ragged, with empty reads between live ones and a read of length 1;
  * each read's rows equal the same launch on that read alone (B = 1, same padded lengths) bit for bit: every output
    row's arithmetic is independent of the batch, so this needs no tolerance and catches item-decode, skip and
    staging-slot errors that a tolerance would hide."""
import functools
import logging
import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import preprocess_oracle as pp
from oracle import resnet_oracle as ro
from riser_b200 import Model, _lib, synth
from riser_b200.config import AttrDict
from riser_b200.resnet import _scale_exponent, pack_tc_weights
from tests import resnet_emulation as emu
from tests.test_gpu_resnet_precision import BETA, MODES, PROB_BAR, _model

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")
POISON = 0x7FBADBAD                     # a NaN bit pattern no kernel computes
U = 2.0 ** -24                          # unit roundoff of float32
F64 = torch.float64


def gamma(n):
    return n * U / (1.0 - n * U)


def _p(t):
    return _lib.ptr(t)


def _i32(v):
    return torch.tensor(v, dtype=torch.int32, device="cuda")


def _poisoned(*shape):
    return torch.full(shape, POISON, dtype=torch.int32, device="cuda").view(torch.float32)


def _randn(seed, *shape, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


def _seed(name):
    return zlib.crc32(name.encode())


def _nan_beyond(x, lens):
    """Rows at or beyond each read's length (dim 1) become NaN."""
    rows = torch.arange(x.shape[1], device=x.device)
    x[rows[None, :] >= torch.as_tensor(lens, device=x.device).long()[:, None]] = float("nan")
    return x


def _assert_unwritten(out, len_out):
    rows = torch.arange(out.shape[1], device=out.device)
    dead = rows[None, :] >= torch.as_tensor(len_out, device=out.device).long()[:, None]
    assert bool((out.view(torch.int32)[dead] == POISON).all()), "a row at or beyond len_out was written"


def _assert_finite(rows, what):
    """Every value of a read's valid rows is finite: a row left unwritten (the NaN poison) or computed from an input row
    beyond the read's length (NaN) fails here, before any comparison whose fold could drop a NaN."""
    assert bool(torch.isfinite(rows).all()), what


def _assert_same_bits(a, b, what):
    assert torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32)), what


def _conv_len(n, k, s, p):
    """Output length of Conv1d(k, s, p) on n samples (0 for an empty read)."""
    return 0 if n <= 0 or n + 2 * p < k else (n + 2 * p - k) // s + 1


# ---------------------------------------------------------------------------------------------- riser_res_tc_ex
LOUT = (1, 37, 126, 127, 128, 129, 252, 253, 257, 1000)     # 1, 2 and 3 tiles per read at both tile heights (128 / 126)
ALL = ("f16", "w2", "x3", "f8")
SINGLE = {   # name: (cin, cout, taps, stride, residual, relu, modes); n1 = cout padded to 16, cin_p = cin padded to 8
    "k1s1-c8-n16": (5, 12, 1, 1, False, 1, ALL),
    "k3s1-c24-n80": (20, 67, 3, 1, True, 1, ALL),            # cout_p 72 < n1 80
    "k3s2-c40-n128": (40, 128, 3, 2, False, 0, ALL),         # 2 n1 = 256: stacked [W_hi; W_lo] (W2, X3)
    "k3s2-c24-n256": (24, 256, 3, 2, True, 1, ALL),          # 2 n1 > 256: separate W_lo MMAs
    "k1s1-c72-n80": (67, 80, 1, 1, True, 0, ALL),
    "k1s2-c40-n144": (40, 140, 1, 2, False, 1, ALL),
    "k1s1-c256-n16": (256, 16, 1, 1, False, 1, ("f16", "w2")),   # cin_p 256 fits shared memory without a lo A tile
    "k3s1-c256-n16": (256, 16, 3, 1, True, 1, ("f16",)),
}
FUSED = {    # name: (cin, cmid, cout, stride, modes); identity shortcut at stride 1 with cin = cout, else a 1x1 conv
    "id-c24-m40": (24, 40, 24, 1, ALL),
    "id-c40-m24": (40, 24, 40, 1, ALL),
    "id-c67-m45": (67, 45, 67, 1, ("f16", "w2")),
    "sc-s2-c20-m30-o45": (20, 30, 45, 2, ALL),
    "sc-s2-c45-m67": (45, 67, 67, 2, ("f16",)),
}


def _pad8(c):
    return (c + 7) & ~7


def _pad16(c):
    return (c + 15) & ~15


def _folded(seed, cout, cin, k):
    w = _randn(seed, cout, cin, k, scale=math.sqrt(2.0 / (cin * k))).cpu()
    return w, _randn(seed + 1, cout, scale=0.1).cpu()


def _padded(v, n):
    out = torch.zeros(n)
    out[:v.shape[0]] = v
    return out.cuda()


def _single_launch(name, mode, cin, cout, taps, stride, residual, relu):
    w, b = _folded(_seed(name), cout, cin, taps)
    e, n1 = _scale_exponent(w), _pad16(cout)
    cin_p = _pad8(cin)
    return dict(kind="single", cin=cin, cin_p=cin_p, cout=cout, cout_p=_pad8(cout), taps=taps, stride=stride,
                pad=(taps - 1) // 2, residual=residual, identity=False, relu=relu, mode=mode, n1=n1, n2=0, cmid_p=0,
                w1=pack_tc_weights(w, n1, cin_p, e, MODES[mode]).cuda(), w2=None, wsc=None, b1=_padded(b, n1),
                b2=None, e1=e, e2=0, w=w.cuda(), b=b.cuda())


def _fused_launch(name, mode, cin, cmid, cout, stride):
    s = _seed(name)
    (w1, b1), (w2, b2) = _folded(s, cmid, cin, 3), _folded(s + 2, cout, cmid, 3)
    identity = stride == 1 and cin == cout
    wsc, bsc = (None, None) if identity else _folded(s + 4, cout, cin, 1)
    e1 = _scale_exponent(w1)
    e2 = _scale_exponent(w2, *([] if identity else [wsc]))
    n1, n2, cin_p, cmid_p = _pad16(cmid), _pad16(cout), _pad8(cin), _pad8(cmid)
    b2s = b2 if identity else b2 + bsc
    p = MODES[mode]
    return dict(kind="fused", cin=cin, cin_p=cin_p, cout=cout, cout_p=_pad8(cout), taps=3, stride=stride, pad=1,
                residual=identity, identity=identity, relu=1, mode=mode, n1=n1, n2=n2, cmid_p=cmid_p,
                w1=pack_tc_weights(w1, n1, cin_p, e1, p).cuda(), w2=pack_tc_weights(w2, n2, cmid_p, e2, p).cuda(),
                wsc=None if identity else pack_tc_weights(wsc, n2, cin_p, e2, p).cuda(), b1=_padded(b1, n1),
                b2=_padded(b2s, n2), e1=e1, e2=e2, c1=(w1.cuda(), b1.cuda(), e1), c2=(w2.cuda(), b2s.cuda(), e2),
                sc=None if identity else wsc.cuda())


def _res_tc(ln, x, len_in, len_out, Lout_pad, residual):
    out = _poisoned(x.shape[0], Lout_pad, ln["cout_p"])
    _lib.check(_lib.lib().riser_res_tc_ex(
        _p(x), _p(len_in), _p(len_out), _p(out), _p(residual), _p(ln["w1"]), _p(ln["w2"]), _p(ln["wsc"]), _p(ln["b1"]),
        _p(ln["b2"]), 2.0 ** -ln["e1"], 2.0 ** -ln["e2"], x.shape[0], x.shape[1], Lout_pad, ln["cin_p"], ln["cmid_p"],
        ln["cout_p"], ln["n1"], ln["n2"], ln["taps"], ln["stride"], ln["relu"], _lib.stream_ptr(), MODES[ln["mode"]]),
        "riser_res_tc_ex")
    return out


def _smem(ln):
    return _lib.lib().riser_res_tc_smem_ex(ln["cin_p"], ln["cmid_p"], ln["n1"], ln["n2"], ln["taps"], ln["stride"],
                                           1 if ln["kind"] == "fused" else 0, 1 if ln["wsc"] is not None else 0,
                                           MODES[ln["mode"]])


def _raw_stages(ln, max_smem):
    """The staging depth riser_res_tc_ex picks (its host code, restated): a second raw input buffer when one more does
    not lower the CTAs per SM, which are limited by shared memory, by the 512 TMEM columns an SM has and to 8."""
    def acc_cols(n):
        cat = ln["mode"] in ("x3", "w2") and 2 * n <= 256          # [W_hi; W_lo] stacked: 2n accumulator columns
        return ((2 * n if cat else n) + 31) // 32 * 32
    cols = acc_cols(ln["n1"]) + (acc_cols(ln["n2"]) if ln["kind"] == "fused" else 0)
    tmem = 1 << max(5, (cols - 1).bit_length())
    smem = _smem(ln)
    ctas = min(max(1, min(512 // tmem, 227 * 1024 // (smem + 1024))), 8)
    raw_rows = 258 if ln["stride"] == 2 else 128 + ln["taps"] - 1
    raw = (raw_rows * ln["cin_p"] * 4 + 127) & ~127
    return 2 if smem + raw <= max_smem and 227 * 1024 // (smem + raw + 1024) >= ctas else 1


def _lens_in(Lin_pad, B):
    pattern = [Lin_pad, 0, 1, Lin_pad // 2 + 1] if B == 4 else \
        [Lin_pad, 0, 1, (Lin_pad // 2) | 1, 0, Lin_pad - 1, (2 * Lin_pad) // 3]
    return [min(max(v, 0), Lin_pad) for v in pattern[:B]]


def _inputs(ln, lens_in, Lin_pad, Lout_pad):
    """x [B, Lin_pad, cin_p] (padding channels 0, rows beyond a read NaN), len_out, residual or None."""
    B = len(lens_in)
    seed = _seed(f"{ln['kind']}{ln['cin']}{ln['cout']}{Lin_pad}{B}")
    x = torch.zeros(B, Lin_pad, ln["cin_p"], device="cuda")
    x[:, :, :ln["cin"]] = _randn(seed, B, Lin_pad, ln["cin"], scale=2.0)
    len_out = [_conv_len(n, ln["taps"], ln["stride"], ln["pad"]) for n in lens_in]
    _nan_beyond(x, lens_in)
    res = None
    if ln["identity"]:
        res = x
    elif ln["residual"]:
        res = torch.zeros(B, Lout_pad, ln["cout_p"], device="cuda")
        res[:, :, :ln["cout"]] = _randn(seed + 7, B, Lout_pad, ln["cout"])
        _nan_beyond(res, len_out)
    return x, len_out, res


def _emulate(ln, x, res, b, n_in, n_out):
    """(emulated output, S, allowance or None) of read b in float64 (tests/resnet_emulation.py)."""
    mode = MODES[ln["mode"]]
    xb = x[b, :n_in, :ln["cin"]].to(F64)
    rb = None if res is None else res[b, :n_out, :ln["cout"]].to(F64)
    if ln["kind"] == "single":
        y, S = emu.single(xb, n_out, ln["w"], ln["b"], ln["e1"], ln["stride"], ln["pad"], mode, residual=rb,
                          relu=bool(ln["relu"]))
        return y, S, None
    y, S, mid, S1 = emu.fused(xb, n_out, ln["c1"], ln["c2"], ln["sc"], ln["stride"], mode, residual=rb)
    assert float(mid.abs().max()) < emu.E4M3_SAT_A
    return y, S, emu.mid_allowance(mid, S1, ln["c2"][0], ln["e2"], mode)


def _check_res_tc(ln, lens_in, Lin_pad, Lout_pad, reads=None, solo=True):
    """One batched launch: poison beyond len_out, |gpu - emu| <= beta S (+ the intermediate's allowance) for `reads`
    (default: every live read), each of them equal to its solo launch bit for bit, padding channels 0."""
    x, len_out, res = _inputs(ln, lens_in, Lin_pad, Lout_pad)
    assert float(torch.nan_to_num(x, nan=0.0).abs().max()) < emu.E4M3_SAT_A
    li, lo = _i32(lens_in), _i32(len_out)
    out = _res_tc(ln, x, li, lo, Lout_pad, res)
    torch.cuda.synchronize()
    _assert_unwritten(out, len_out)
    worst = 0.0
    for b in (range(len(lens_in)) if reads is None else reads):
        n = len_out[b]
        if n == 0:
            continue
        _assert_finite(out[b, :n], f"read {b}: a valid row is NaN or unwritten")
        y, S, allow = _emulate(ln, x, res, b, lens_in[b], n)
        worst = max(worst, emu.excess(out[b, :n, :ln["cout"]].to(F64), y, S, allow))
        assert bool((out[b, :n, ln["cout"]:] == 0).all()), "padding channels must stay 0"
        if solo:
            one = _res_tc(ln, x[b:b + 1], li[b:b + 1], lo[b:b + 1], Lout_pad, None if res is None else res[b:b + 1])
            _assert_same_bits(out[b, :n], one[0, :n], f"read {b}: batched launch != the same launch on the read alone")
    beta = BETA[(ln["mode"], ln["kind"])]
    print(f"{ln['kind']} {ln['mode']} Lout_pad {Lout_pad} B {len(lens_in)}: max excess/S {worst:.3e} (beta {beta:.3e})")
    assert worst <= beta, worst


def _sweep(shapes):
    cases = []
    for j, (name, spec) in enumerate(shapes.items()):
        modes = spec[-1]
        for i, L in enumerate(LOUT):
            mode, B = modes[(i + j) % len(modes)], (4, 7)[(i + j) % 2]
            cases.append(pytest.param(name, mode, L, B, id=f"{name}-{mode}-L{L}-B{B}"))
    return cases


def _launch(kind, name, mode):
    return _single_launch(name, mode, *SINGLE[name][:-1]) if kind == "single" else \
        _fused_launch(name, mode, *FUSED[name][:-1])


@pytest.mark.parametrize("name,mode,Lout_pad,B", _sweep(SINGLE))
def test_res_tc_single_conv(name, mode, Lout_pad, B):
    ln = _launch("single", name, mode)
    Lin_pad = ln["stride"] * Lout_pad
    _check_res_tc(ln, _lens_in(Lin_pad, B), Lin_pad, Lout_pad)


@pytest.mark.parametrize("name,mode,Lout_pad,B", _sweep(FUSED))
def test_res_tc_fused_block(name, mode, Lout_pad, B):
    ln = _launch("fused", name, mode)
    Lin_pad = ln["stride"] * Lout_pad
    _check_res_tc(ln, _lens_in(Lin_pad, B), Lin_pad, Lout_pad)


def test_res_tc_sweep_covers_both_staging_depths():
    """Every shape of the sweep is one the kernel takes, and the sweep runs both staging depths in both modes, with a
    fused identity block at depth 1 (its shortcut is read back from the one staging buffer before the next prefetch)."""
    max_smem = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    seen = set()
    for kind, shapes in (("single", SINGLE), ("fused", FUSED)):
        for case in _sweep(shapes):
            name, mode = case.values[:2]
            ln = _launch(kind, name, mode)
            assert 0 < _smem(ln) <= max_smem, (name, mode)
            seen.add((kind, _raw_stages(ln, max_smem), ln["identity"]))
    assert {("single", 1, False), ("single", 2, False), ("fused", 1, True), ("fused", 2, True)} <= seen, seen
    assert any(k == "fused" and not ident for k, _, ident in seen)


@pytest.mark.parametrize("kind,name,mode", [("single", "k1s1-c8-n16", "x3"), ("single", "k3s1-c24-n80", "f8"),
                                            ("fused", "id-c24-m40", "x3"), ("fused", "id-c24-m40", "f16")])
def test_res_tc_many_items_per_cta(kind, name, mode):
    """300 ragged reads x 1,000 rows: more items than 148 SMs x 8 CTAs, so every CTA walks several items and the next
    item's prefetch, the second staging slot and the mbarrier parities all run (the model-level batches give each CTA
    one item at most)."""
    ln = _launch(kind, name, mode)
    B, Lout_pad = 300, 1000
    Lin_pad = ln["stride"] * Lout_pad
    tile = 128 if kind == "single" else 126
    n_items = B * -(-Lout_pad // tile)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert n_items > sms * 8, n_items
    g = np.random.Generator(np.random.PCG64(_seed(name + mode)))
    lens = g.integers(0, Lin_pad + 1, size=B)
    lens[g.random(B) < 0.25] = Lin_pad
    lens[::17] = 0
    lens[5] = 1
    lens = [int(v) for v in lens]
    reads = sorted(set(range(0, B, 10)) | {1, 5, B - 2, B - 1})
    _check_res_tc(ln, lens, Lin_pad, Lout_pad, reads=reads)


def test_res_tc_8191_tiles_per_read():
    """2^13 - 1 tiles per read, B = 66, only reads 64 and 65 live: the last items of the launch (read 64's last tile
    and read 65's) decode to the right read.  len_in / len_out carry one extra entry 0, so that an item decoded one
    read too far finds an empty read rather than memory past the arrays (about 2.2 GB each for input and output)."""
    ln = _single_launch("t8191", "x3", 8, 8, 1, 1, False, 1)
    assert (ln["cin_p"], ln["cout_p"], ln["n1"]) == (8, 8, 16)
    B, Lout_pad = 66, 8191 * 128
    x = torch.full((B, Lout_pad, 8), float("nan"), device="cuda")
    x[64:66] = _randn(8191, 2, Lout_pad, 8)
    lens = [0] * 64 + [Lout_pad, Lout_pad] + [0]
    li = _i32(lens)
    out = _res_tc(ln, x, li, li, Lout_pad, None)
    torch.cuda.synchronize()
    for b in range(B):
        n = lens[b]
        assert bool((out[b, n:].view(torch.int32) == POISON).all()), b
        if n:
            y, S, _ = _emulate(ln, x, None, b, n, n)
            ex = emu.excess(out[b, :n].to(F64), y, S)
            print(f"read {b}: max excess/S {ex:.3e}")
            assert ex <= BETA[("x3", "single")], (b, ex)
    del x, out
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- riser_conv1d_cl
def _conv1d_cl(x, len_in, w, b, res, len_out, Lout_pad, Cin, Cout, K, stride, pad, relu):
    out = _poisoned(x.shape[0], Lout_pad, Cout)
    _lib.check(_lib.lib().riser_conv1d_cl(_p(x), _p(len_in), _p(w), _p(b), _p(res), _p(out), _p(len_out), x.shape[0],
                                          x.shape[1], Lout_pad, Cin, Cout, K, stride, pad, relu, _lib.stream_ptr()),
               "riser_conv1d_cl")
    return out


def _tile_rows(Cout):
    """Position-tile height the tiled kernel can reach (riser_conv1d_cl's host code): 256 / (CT / 4) rows of threads
    x 8 positions, CT = all output channels up to 128, else 64."""
    c4 = (Cout + 3) & ~3
    ct = c4 if c4 <= 128 else 64
    return (256 // (ct // 4)) * 8


def _conv1d_cases():
    cases, i = [], 0
    pairs = [(ci, co) for ci in (1, 8, 67, 128) for co in (3, 67, 130, 256)]
    for K in (1, 3, 5, 19):
        for pad in sorted({0, (K - 1) // 2, 5}):
            for stride in (1, 2, 3):
                Cin, Cout = pairs[i % len(pairs)]
                T = _tile_rows(Cout)
                Lout_pad = (T - 1, T, T + 1, 2 * T + 3)[i % 4]
                cases.append(pytest.param(K, stride, pad, Cin, Cout, Lout_pad, i % 3 == 0, i % 2, i % 5 == 0,
                                          id=f"k{K}s{stride}p{pad}-{Cin}to{Cout}-L{Lout_pad}" + ("-naive" if i % 5 == 0 else "")))
                i += 1
    # weights of one channel tile over 200 KB: only the per-element kernel takes the shape
    assert 3 * 512 * 128 * 4 > 200 * 1024
    cases.append(pytest.param(3, 1, 1, 512, 128, 130, True, 1, False, id="k3s1p1-512to128-L130-untiled"))
    return cases


@pytest.mark.parametrize("K,stride,pad,Cin,Cout,Lout_pad,residual,relu,naive", _conv1d_cases())
def test_conv1d_cl(monkeypatch, K, stride, pad, Cin, Cout, Lout_pad, residual, relu, naive):
    """Against float64 F.conv1d per read: |gpu - ref| <= gamma_n S, n = K Cin + 2 (the fp32 FMA chain, the bias and the
    residual), S = conv(|x|, |w|) + |b| (+ |residual|) -- a rigorous bound for any order of the sum."""
    if naive:
        monkeypatch.setenv("RISER_RESNET_NAIVE", "1")
    name = f"conv{K}{stride}{pad}{Cin}{Cout}{Lout_pad}"
    Lin_pad = max(1, (Lout_pad - 1) * stride + K - 2 * pad)
    lens = [Lin_pad, 0, 1, Lin_pad // 2 + 1, Lin_pad - 1, 0, (2 * Lin_pad) // 3]
    lens = [min(max(v, 0), Lin_pad) for v in lens]
    len_out = [_conv_len(n, K, stride, pad) for n in lens]
    assert max(len_out) == Lout_pad
    B = len(lens)
    s = _seed(name)
    x = _nan_beyond(_randn(s, B, Lin_pad, Cin), lens)
    wt = _randn(s + 1, Cout, Cin, K, scale=1.0 / math.sqrt(Cin * K))        # [Cout, Cin, K] as torch has it
    w = wt.permute(2, 1, 0).contiguous()                                       # [K][Cin][Cout] as the kernel reads it
    bias = _randn(s + 2, Cout, scale=0.1)
    res = _nan_beyond(_randn(s + 3, B, Lout_pad, Cout), len_out) if residual else None
    li, lo = _i32(lens), _i32(len_out)
    out = _conv1d_cl(x, li, w, bias, res, lo, Lout_pad, Cin, Cout, K, stride, pad, relu)
    torch.cuda.synchronize()
    _assert_unwritten(out, len_out)
    bar = gamma(K * Cin + 2)
    worst = 0.0
    for b in range(B):
        n, m = lens[b], len_out[b]
        if m == 0:
            continue
        xb = x[b, :n].to(F64).T[None]
        ref = F.conv1d(xb, wt.to(F64), bias.to(F64), stride=stride, padding=pad)[0].T
        S = F.conv1d(xb.abs(), wt.to(F64).abs(), bias.to(F64).abs(), stride=stride, padding=pad)[0].T
        assert ref.shape[0] == m
        if res is not None:
            ref, S = ref + res[b, :m].to(F64), S + res[b, :m].to(F64).abs()
        if relu:
            ref = torch.relu(ref)
        _assert_finite(out[b, :m], f"read {b}: a valid row is NaN or unwritten")
        worst = max(worst, float(((out[b, :m].to(F64) - ref).abs() / S.clamp_min(1e-300)).max()))
        one = _conv1d_cl(x[b:b + 1], li[b:b + 1], w, bias, None if res is None else res[b:b + 1], lo[b:b + 1],
                         Lout_pad, Cin, Cout, K, stride, pad, relu)
        _assert_same_bits(out[b, :m], one[0, :m], f"read {b}: batched != alone")
    print(f"max |gpu - ref| / S = {worst:.3e}, gamma_{K * Cin + 2} = {bar:.3e}")
    assert worst <= bar, worst


# ---------------------------------------------------------------------------------------------- riser_stem_pool_cl
def _stem(x, len_in, w, b, len_conv, len_out, Lout_pad, Cp, K, stride, pad):
    out = _poisoned(x.shape[0], Lout_pad, Cp)
    _lib.check(_lib.lib().riser_stem_pool_cl(_p(x), x.stride(0), _p(len_in), _p(w), _p(b), _p(out), _p(len_conv),
                                             _p(len_out), x.shape[0], Lout_pad, Cp, K, stride, pad, _lib.stream_ptr()),
               "riser_stem_pool_cl")
    return out


@pytest.mark.parametrize("Cp", [4, 24, 32])
@pytest.mark.parametrize("K,stride,pad", [(19, 3, 5), (7, 2, 3), (32, 1, 0), (1, 1, 0)],
                         ids=["k19s3-template", "k7s2", "k32s1", "k1s1"])
def test_stem_pool_cl(K, stride, pad, Cp):
    """Conv1d(1 -> Cp) + ReLU + MaxPool1d(2, 2, padding=1) against float64 on each read alone, pooled lengths around
    the 128- and 256-position tiles, a read shorter than the kernel, one with a single conv position, an empty one.
    Bar gamma_{K+1} S (the bias and K FMAs; ReLU and max add no error), S = the larger conv(|x|, |w|) + |b| of the
    two pooled positions."""
    # pooled length P = n_conv // 2 + 1: n_conv = 2 P - 2 or 2 P - 1
    n_convs = [2 * P - 2 + (P & 1) for P in (127, 128, 129, 255, 256, 257, 511, 512, 513)]
    lens = [(nc - 1) * stride + K - 2 * pad + (i % stride) for i, nc in enumerate(n_convs)]
    lens[1:1] = [0]                                                           # an empty read between live ones
    lens += [K - 2 * pad, K - 1]                                              # one conv position; shorter than K
    n_conv = [_conv_len(n, K, stride, pad) for n in lens]
    assert 1 in n_conv and (K == 1 or any(0 < n < K for n in lens))
    len_out = [nc // 2 + 1 if nc > 0 else 0 for nc in n_conv]
    Lout_pad, ld = max(len_out) + 2, max(lens) + 5
    B = len(lens)
    s = _seed(f"stem{K}{stride}{pad}{Cp}")
    x = _nan_beyond(_randn(s, B, ld), lens)
    wt = _randn(s + 1, Cp, 1, K, scale=1.0 / math.sqrt(K))
    bias = _randn(s + 2, Cp, scale=0.1)
    w = wt[:, 0, :].T.contiguous()                                            # [K][Cp]
    li, lc, lo = _i32(lens), _i32(n_conv), _i32(len_out)
    out = _stem(x, li, w, bias, lc, lo, Lout_pad, Cp, K, stride, pad)
    torch.cuda.synchronize()
    _assert_unwritten(out, len_out)
    bar, worst = gamma(K + 1), 0.0
    for b in range(B):
        m = len_out[b]
        if m == 0:
            continue
        xb = x[b, :lens[b]].to(F64)[None, None]
        conv = F.conv1d(xb, wt.to(F64), bias.to(F64), stride=stride, padding=pad)
        S = F.conv1d(xb.abs(), wt.to(F64).abs(), bias.to(F64).abs(), stride=stride, padding=pad)
        assert conv.shape[-1] == n_conv[b]
        ref = F.max_pool1d(torch.relu(conv), 2, stride=2, padding=1)[0].T
        S = F.max_pool1d(S, 2, stride=2, padding=1)[0].T
        assert ref.shape[0] == m
        _assert_finite(out[b, :m], f"read {b}: a valid row is NaN or unwritten")
        worst = max(worst, float(((out[b, :m].to(F64) - ref).abs() / S.clamp_min(1e-300)).max()))
        one = _stem(x[b:b + 1], li[b:b + 1], w, bias, lc[b:b + 1], lo[b:b + 1], Lout_pad, Cp, K, stride, pad)
        _assert_same_bits(out[b, :m], one[0, :m], f"read {b}: batched != alone")
    print(f"max |gpu - ref| / S = {worst:.3e}, gamma_{K + 1} = {bar:.3e}")
    assert worst <= bar, worst


# ---------------------------------------------------------------------------------------------- riser_maxpool1d_pad_cl
@pytest.mark.parametrize("pad", [0, 1])
def test_maxpool1d_pad_cl(pad):
    """Exactly F.max_pool1d(2, 2, padding=pad) of each read, at odd, even, 1 and 0 lengths."""
    C, Lin_pad = 67, 301
    lens = [301, 0, 1, 2, 3, 0, 8, 9, 250, 251, 300]
    len_out = [(n + 2 * pad) // 2 if n > 0 else 0 for n in lens]
    Lout_pad = Lin_pad // 2 + 1
    x = _nan_beyond(_randn(_seed(f"pool{pad}"), len(lens), Lin_pad, C), lens)
    li, lo = _i32(lens), _i32(len_out)

    def run(x, li, lo):
        out = _poisoned(x.shape[0], Lout_pad, C)
        _lib.check(_lib.lib().riser_maxpool1d_pad_cl(_p(x), _p(li), _p(out), _p(lo), x.shape[0], Lin_pad, Lout_pad, C,
                                                     pad, _lib.stream_ptr()), "riser_maxpool1d_pad_cl")
        return out
    out = run(x, li, lo)
    torch.cuda.synchronize()
    _assert_unwritten(out, len_out)
    for b, n in enumerate(lens):
        if len_out[b] == 0:
            continue
        ref = F.max_pool1d(x[b, :n].T[None].to(F64), 2, stride=2, padding=pad)[0].T.float()
        assert ref.shape[0] == len_out[b]
        _assert_same_bits(out[b, :len_out[b]], ref, f"read {b} (length {n})")
        _assert_same_bits(out[b, :len_out[b]], run(x[b:b + 1], li[b:b + 1], lo[b:b + 1])[0, :len_out[b]], b)


# ---------------------------------------------------------------------------------------------- riser_len_chain
@functools.lru_cache(maxsize=None)
def _torch_len(n, k, s, p):
    """The length torch itself produces for op (k, s, p) on n samples (k < 0: MaxPool1d(2, 2, padding p)); 0 where
    torch refuses the input."""
    try:
        z = torch.zeros(1, 1, n)
        if k < 0:
            return int(F.max_pool1d(z, 2, stride=2, padding=p).shape[-1])
        return int(F.conv1d(z, torch.zeros(1, 1, k), stride=s, padding=p).shape[-1])
    except RuntimeError:
        return 0


def _chains():
    out = []
    for name, cfg in synth.RESNET_CONFIGS.items():
        out.append((name, _model(name, None).chain))
    for name, cfg in synth.GENERIC_CNN_CONFIGS.items():
        m = Model(synth.generic_cnn_state_dict(cfg, 0), AttrDict({"model": "cnn", "cnn": cfg}), LOG, "mRNA")
        out.append((name, m._generic.chain))
    return out


def test_len_chain_matches_torch():
    """Every op of both ResNet configurations and every generic ConvNet configuration, n = 0 ... 600 and a few large n:
    exactly the output lengths torch's own conv1d / max_pool1d produce, op after op."""
    ns = list(range(601)) + [4095, 4096, 6000, 7108, 10120, 12048, 100003, 1 << 20]
    for name, chain in _chains():
        ops = [tuple(int(v) for v in r) for r in chain.cpu().tolist()]
        got = torch.empty(len(ops), len(ns), dtype=torch.int32, device="cuda")
        _lib.check(_lib.lib().riser_len_chain(_p(_i32(ns)), len(ns), _p(chain), len(ops), _p(got), _lib.stream_ptr()),
                   "riser_len_chain")
        got = got.cpu().numpy()
        for i, n in enumerate(ns):
            for j, op in enumerate(ops):
                n = _torch_len(n, *op) if n > 0 else 0
                assert got[j, i] == n, (name, ns[i], j, op, int(got[j, i]), n)


# ---------------------------------------------------------------------------------------------- riser_gap_linear_softmax
@pytest.mark.parametrize("n_classes", [1, 2, 3, 32])
@pytest.mark.parametrize("C", [8, 72, 256, 1024])
def test_gap_linear_softmax(C, n_classes):
    """Against float64, lengths 0, 1, 251 and 5,000 (a length-0 row is NaN).  The bar, per probability:
      feat_c = (sum of L float32 terms) / L: L - 1 additions and a division, |df_c| <= gamma_L sum_t |x_tc| / L;
      logit_j = sum_c feat_c w_jc + b_j in any order (lane FMA chains, shuffle tree, bias): C + 1 terms,
        |dl_j| <= gamma_{C+1} (sum_c |feat_c w_jc| + |b_j|) + sum_c |w_jc| |df_c|;
      softmax: l_j - max rounds once, a further logit perturbation of u |l_j - max|; softmax's Jacobian has row sums
        sum_j |dp_i / dl_j| = 2 p_i (1 - p_i) <= 1/2, so |dp_i| <= max_j |dl_j| / 2; expf (2 ulp = 4u relative), the
        sum of n_classes terms and the division add at most (n_classes + 10) u p_i."""
    lens = [5000, 0, 1, 251]
    B, L_pad = len(lens), 5000
    s = _seed(f"head{C}{n_classes}")
    x = _nan_beyond(_randn(s, B, L_pad, C), lens)
    w = _randn(s + 1, n_classes, C, scale=3.0 / math.sqrt(C))
    bias = _randn(s + 2, n_classes, scale=0.5)
    li = _i32(lens)

    def run(x, li):
        probs = _poisoned(x.shape[0], n_classes)
        _lib.check(_lib.lib().riser_gap_linear_softmax(_p(x), _p(li), _p(w), _p(bias), _p(probs), x.shape[0], L_pad, C,
                                                       n_classes, _lib.stream_ptr()), "riser_gap_linear_softmax")
        return probs
    probs = run(x, li)
    torch.cuda.synchronize()
    w64, b64 = w.to(F64), bias.to(F64)
    for b, L in enumerate(lens):
        _assert_same_bits(probs[b], run(x[b:b + 1], li[b:b + 1])[0], f"read {b}: batched != alone")
        if L == 0:
            assert bool(torch.isnan(probs[b]).all())
            continue
        xb = x[b, :L].to(F64)
        f = xb.sum(0) / L
        df = gamma(L) * xb.abs().sum(0) / L
        logit = w64 @ f + b64
        dl = gamma(C + 1) * ((w64 * (f.abs() + df)).abs().sum(1) + b64.abs()) + w64.abs() @ df
        p = torch.softmax(logit, 0)
        dl = dl + U * ((logit.max() - logit).abs() + 2 * dl.max())
        bar = 0.5 * dl.max() + (n_classes + 10) * U * p
        err = (probs[b].to(F64) - p).abs()
        assert bool((err <= bar).all()), (b, float(err.max()), float(bar.min()))


# ---------------------------------------------------------------------------------------------- the models
def _ragged(seed, B, L, lo):
    normed = [np.asarray(pp.mad_normalise(v), dtype=np.float64) for v in synth.ragged_bodies(seed, B, lo, L)]
    x = torch.full((B, L), 9.0)                          # poison the padding: never read as signal
    for b, v in enumerate(normed):
        x[b, :len(v)] = torch.from_numpy(v).float()
    return normed, x.cuda(), _i32([len(v) for v in normed])


def _batch_equals_solo(model, x, n, L, probs):
    for b in range(x.shape[0]):
        one = model.classify_batch(x[b:b + 1], n[b:b + 1], max_len=L)
        _assert_same_bits(probs[b], one[0], f"read {b}: batched != alone")


@functools.lru_cache(maxsize=None)
def _oracle(name, L):
    normed, _, _ = _ragged(L, 16, L, L // 2)
    sd = synth.resnet_state_dict(synth.RESNET_CONFIGS[name], 0)
    return np.stack([ro.classify(sd, synth.RESNET_CONFIGS[name], v).numpy() for v in normed])


@pytest.mark.parametrize("L", [4096, 6000])
@pytest.mark.parametrize("mode", ["x3", "f8"])
@pytest.mark.parametrize("name", ["basic", "bottleneck"])
def test_resnet_model_where_the_last_stage_fits_one_tile(name, mode, L):
    """At max_len 4,096 and 6,000 the last stage has 86 / 125 rows: one tile per read.  Every read's probabilities
    against the reference restatement, and each row equal to the same call on that read alone."""
    _, x, n = _ragged(L, 16, L, L // 2)
    model = _model(name, MODES[mode])
    probs = model.classify_batch(x, n, max_len=L).clone()
    want = _oracle(name, L)
    err = float(np.abs(probs.cpu().numpy() - want).max())
    print(f"{name} {mode} at {L}: max |dp| {err:.2e}")
    assert err < PROB_BAR[(name, mode)], err
    _batch_equals_solo(model, x, n, L, probs)


def test_evaluate_ladder_with_the_resnet():
    """riser_b200.evaluate with a basic X3 ResNetModel: every rung (4,096 / 7,108 / 10,120) of every read against the
    reference restatement on that prefix."""
    from riser_b200 import Kit, SignalProcessor
    from riser_b200 import evaluate as ev
    cfg = synth.RESNET_CONFIGS["basic"]
    sd = synth.resnet_state_dict(cfg, 0)
    bodies = synth.ragged_bodies(41, 16, 4096, 12048)
    reads = [(f"r{i}", b) for i, b in enumerate(bodies)]
    lines = ev.evaluate(reads, _model("basic", None), SignalProcessor(Kit.create_from_version("RNA002")), "RNA002",
                        already_trimmed=True)
    assert len(lines) == len(reads)
    worst = {}
    for (rid, body), ln in zip(reads, lines):
        preds = ln.rstrip("\n").split("\t")[6].split(";")
        rungs = [L for L in ev.ladder("RNA002") if L <= len(body)]
        assert len(preds) == len(rungs), (rid, preds)
        for L, pr in zip(rungs, preds):
            k, vals = pr.split(":")
            assert int(k) == L
            got = np.array([float(v) for v in vals.split(",")])
            want = ro.classify(sd, cfg, pp.mad_normalise(body[:L])).numpy()
            assert np.isfinite(got).all(), (rid, L, got)
            worst[L] = max(worst.get(L, 0.0), float(np.abs(got - want).max()))
    print(f"max |dp| per rung: {worst}")
    assert all(v < 2e-4 for v in worst.values()), worst


def test_generic_convnet_batch_equals_solo_at_2048():
    """k5_fc at max_len 2,048: layer 4 (k = 3, tensor cores) runs at 128 rows, one tile per read."""
    cfg = synth.GENERIC_CNN_CONFIGS["k5_fc"]
    model = Model(synth.generic_cnn_state_dict(cfg, 0), AttrDict({"model": "cnn", "cnn": cfg}), LOG, "mRNA")
    assert model._generic.layers[4][0].tc is not None
    _, x, n = _ragged(77, 8, 2048, 700)
    probs = model.classify_batch(x, n, max_len=2048).clone()
    assert bool(torch.isfinite(probs).all())
    _batch_equals_solo(model, x, n, 2048, probs)


def test_resnet_empty_batch():
    model = _model("basic", None)
    x = torch.zeros(0, 4096, device="cuda")
    assert tuple(model.classify_batch(x, _i32([]), max_len=4096).shape) == (0, 2)
