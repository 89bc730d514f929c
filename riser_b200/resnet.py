"""ResNet variant of the classifier (riser/nets/resnet.py) behind the same Model call surface.

The reference can only select it in train.py:177-178 (``config.model == 'resnet'``,
``ResNet(config.resnet)``) and ships no config or weights for it, so the hyper-parameters are
whatever the caller's config says: ``channels, kernel, padding, stride, block, n_layers,
blocks, n_classes`` (resnet.py:73-102).  BatchNorm (eval mode) is folded into the convolution
weights here on the host.  The residual blocks run on the tensor pipe (csrc/resnet_tc.cu: tcgen05 implicit GEMM,
fp16 operand planes, fp32 accumulation in TMEM) -- a BasicBlock as ONE launch whose intermediate
activation never leaves the SM, the convolutions of a BottleneckBlock (and blocks whose weights do not fit
shared memory fused) one launch each with the residual added in the epilogue; the stem (Cin = 1, K = 19: 3 % of the
FLOPs), its max-pool and the head stay on the fp32 CUDA-core kernels of csrc/resnet.cu, which also remain the
fallback for shapes the tensor-core kernel does not take (``RISER_RESNET_TC=0`` forces them everywhere).
Activations are fp32 channel-last [B][L][C_p] with the channels padded to a multiple of 8 (zero weights / biases in
the padding, so the padding channels stay zero through every layer).

Precision (``ResNetModel(..., precision=)``, the PREC_* modes of model.py) applies to the tensor-core launches only:
F16_X3 (the default, ``precision=None``: a_hi W_hi + a_lo W_hi + a_hi W_lo), F16_W2 (a_hi (W_hi + W_lo)), F16 (a_hi
W_hi) and F16_F8 (a_hi W_hi + one e4m3 pass carrying both correction terms, as the ConvNet's default).  The stem, its
max-pool, the head and every convolution that falls back to the CUDA cores stay fp32 whatever the mode.
"""
import os

import numpy as np
import torch

from . import _lib
from .model import F8_A_SHIFT, F8_LO_SHIFT, PREC_F16, PREC_F16_F8, PREC_F16_W2, PREC_F16_X3

EPS = 1e-5


def _pad8(c):
    return (int(c) + 7) & ~7


def _pad16(c):
    return (int(c) + 15) & ~15


def _scale_exponent(*ws):
    """Power of two that brings the largest weight magnitude into [2^11, 2^12): keeps the fp16 lo plane out of the
    subnormal range (as csrc/convnet.cu does for the ConvNet)."""
    wmax = max(float(w.abs().max()) for w in ws)
    if not np.isfinite(wmax) or wmax <= 0.0:
        return 0
    return int(max(-24, min(24, 12 - np.frexp(wmax)[1])))


E4M3_MAX = 448.0


def e4m3_bytes(x):
    """float32 -> e4m3 bytes, rounded to nearest and saturated to +-448 (__nv_cvt_float_to_fp8 with __NV_SATFINITE;
    torch's cast alone gives NaN above the range)."""
    return x.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).view(torch.uint8)


def pack_tc_weights(w, n_pad, cin_p, e, precision=PREC_F16_X3):
    """Folded conv weight [Cout, Cin, K] fp32 -> the operand image riser_res_tc_ex reads in mode `precision`:
    [tap][K block of 32 channels][plane][n_pad rows][64 bytes], every 64-byte row with its 16-byte chunks at
    ``chunk ^ ((row >> 1) & 3)`` (K-major SWIZZLE_64B), weights w = W 2^e.  Planes: F16 [hi]; F16_W2 and F16_X3 [hi, lo]
    (hi = fp16(w), lo = fp16(w - hi): for a tap and K block the hi rows are followed by the lo rows, so the stacked
    operand [W_hi; W_lo] is one tile); F16_F8 [hi, e4m3 row] with the row [e4m3((w - hi) 2^F8_A_SHIFT) x32 |
    e4m3(w 2^-(9 - F8_LO_SHIFT)) x32] of the K block's 32 channels."""
    cout, cin, K = w.shape
    kb = (cin_p + 31) // 32
    ws = (w.double() * (2.0 ** e)).float()
    hi = ws.half()
    d = ws - hi.float()                                          # exact in float32

    def plane(src):                       # [cout, cin, K] -> bytes [K][kb][n_pad][32 x element]
        full = torch.zeros(K, n_pad, kb * 32, dtype=src.dtype)
        full[:, :cout, :cin] = src.permute(2, 0, 1)
        return full.view(K, n_pad, kb, 32).permute(0, 2, 1, 3).contiguous().view(torch.uint8)

    if precision == PREC_F16:
        planes = [plane(hi)]
    elif precision in (PREC_F16_W2, PREC_F16_X3):
        planes = [plane(hi), plane(d.half())]
    elif precision == PREC_F16_F8:
        w8 = torch.cat([plane(e4m3_bytes(d * 2.0 ** F8_A_SHIFT)), plane(e4m3_bytes(ws * 2.0 ** -(9 - F8_LO_SHIFT)))],
                       dim=3)
        planes = [plane(hi), w8]
    else:
        raise ValueError(f"unknown precision mode {precision}")
    P = len(planes)
    chunks = torch.stack(planes, dim=2).view(K, kb, P, n_pad, 4, 16)
    rows = torch.arange(n_pad)
    out = torch.empty_like(chunks)
    for c in range(4):
        dst = c ^ ((rows >> 1) & 3)
        out[:, :, :, rows, dst] = chunks[:, :, :, rows, c]
    return out.contiguous().view(-1)


def _fold(w, b, bn):
    """Conv weight [Cout, Cin, K] (+ optional bias) followed by eval-mode BatchNorm1d -> one
    conv with w' = w * g / sqrt(var + eps), b' = beta + (b - mean) * g / sqrt(var + eps)."""
    g, beta, mean, var = bn
    scale = g / torch.sqrt(var + EPS)
    wf = w * scale[:, None, None]
    bf = beta + ((b if b is not None else 0.0) - mean) * scale
    return wf, bf


class _Conv:
    """One folded convolution: CUDA-core weights [K][Cin_p][Cout_p] (zero padded), and -- when the tensor-core kernel
    takes the shape -- its operand image."""
    def __init__(self, w, b, stride, pad, device, pad_cin=True):
        self.cout, self.cin, self.k = w.shape
        self.stride, self.pad = stride, pad
        self.cin_p = _pad8(self.cin) if pad_cin else self.cin
        self.cout_p = _pad8(self.cout)
        wp = torch.zeros(self.k, self.cin_p, self.cout_p)
        wp[:, :self.cin, :self.cout] = w.permute(2, 1, 0)
        bp = torch.zeros(self.cout_p)
        bp[:self.cout] = b
        self.w = wp.contiguous().to(device)                        # [K][Cin_p][Cout_p]
        self.b = bp.contiguous().to(device)
        self.w_host, self.b_host = w, b
        self.tc = None

    def out_len(self, n):
        return torch.clamp((n + 2 * self.pad - self.k) // self.stride + 1, min=0).to(torch.int32)

    def tc_ok(self):
        return self.k in (1, 3) and self.stride in (1, 2) and self.pad == (self.k - 1) // 2 and self.cin_p % 8 == 0 \
            and _pad16(self.cout) <= 256

    def build_tc(self, device, max_smem, precision=PREC_F16_X3):
        """Operand image for the single-conv mode of riser_res_tc_ex (None if the shape is not supported)."""
        if not self.tc_ok():
            return None
        n1 = _pad16(self.cout)
        need = _lib.lib().riser_res_tc_smem_ex(self.cin_p, 0, n1, 0, self.k, self.stride, 0, 0, precision)
        if need == 0 or need > max_smem:
            return None
        e = _scale_exponent(self.w_host)
        bias = torch.zeros(n1)
        bias[:self.cout] = self.b_host
        self.tc = dict(w=pack_tc_weights(self.w_host, n1, self.cin_p, e, precision).to(device), bias=bias.to(device),
                       inv=float(2.0 ** -e), e=e, n1=n1)
        return self.tc


class _FusedBasic:
    """Operand images of a whole BasicBlock for the fused mode of riser_res_tc."""
    def __init__(self, conv1, conv2, shortcut, device, precision=PREC_F16_X3):
        n1, n2 = _pad16(conv1.cout), _pad16(conv2.cout)
        e1 = _scale_exponent(conv1.w_host)
        e2 = _scale_exponent(conv2.w_host, *([shortcut.w_host] if shortcut is not None else []))
        self.w1 = pack_tc_weights(conv1.w_host, n1, conv1.cin_p, e1, precision).to(device)
        self.w2 = pack_tc_weights(conv2.w_host, n2, conv2.cin_p, e2, precision).to(device)
        self.wsc = None if shortcut is None else \
            pack_tc_weights(shortcut.w_host, n2, shortcut.cin_p, e2, precision).to(device)
        self.e1, self.e2 = e1, e2
        b1 = torch.zeros(n1)
        b1[:conv1.cout] = conv1.b_host
        b2 = torch.zeros(n2)
        b2[:conv2.cout] = conv2.b_host
        if shortcut is not None:
            b2[:shortcut.cout] += shortcut.b_host
        self.b1, self.b2 = b1.to(device), b2.to(device)
        self.inv1, self.inv2 = float(2.0 ** -e1), float(2.0 ** -e2)
        self.n1, self.n2 = n1, n2


class ResNetModel():
    def __init__(self, state, config, logger, target, precision=None):
        """precision: PREC_F16, PREC_F16_W2, PREC_F16_X3 or PREC_F16_F8 for the tensor-core launches; None = F16_X3."""
        self.target = target
        self.precision = PREC_F16_X3 if precision is None else int(precision)
        if self.precision not in (PREC_F16, PREC_F16_W2, PREC_F16_X3, PREC_F16_F8):
            raise ValueError(f"unknown precision mode {precision}")
        self.logger = logger
        self.device = _lib.require_device()
        self.logger.info('Using %s device', self.device)
        c = config.resnet if hasattr(config, "resnet") else config
        sd = state if isinstance(state, dict) else torch.load(state, map_location=torch.device('cpu'))
        sd = {k: torch.as_tensor(v).detach().to("cpu", torch.float32) for k, v in sd.items()
              if not k.endswith("num_batches_tracked")}
        self.c = c
        self.n_classes = int(c.n_classes)
        dev = self.device

        def bn(prefix):
            return tuple(sd[prefix + s] for s in (".weight", ".bias", ".running_mean", ".running_var"))

        def conv_bn(prefix, stride, pad, bias=None, pad_cin=True):
            w, b = _fold(sd[prefix + ".0.weight"], bias, bn(prefix + ".1"))
            return _Conv(w, b, stride, pad, dev, pad_cin=pad_cin)

        self.use_tc = os.environ.get("RISER_RESNET_TC", "1") != "0"
        self.fused_stem = os.environ.get("RISER_RESNET_FUSED_STEM", "1") != "0"
        max_smem = torch.cuda.get_device_properties(dev).shared_memory_per_block_optin
        L_ = _lib.lib()
        self.stem = conv_bn("conv_block", int(c.stride), int(c.padding), bias=sd["conv_block.0.bias"], pad_cin=False)
        self.blocks = []
        self.n_tc_fused = self.n_tc_convs = self.n_cuda_core_convs = 0
        cin = int(c.channels[0])
        for i in range(int(c.n_layers)):
            cout = int(c.channels[i])
            for j in range(int(c.blocks[i])):
                stride = 2 if (i > 0 and j == 0) else 1
                p = f"layers.{i}.{j}"
                shortcut = None
                if cin != cout or stride != 1:                              # resnet.py:45-47
                    shortcut = conv_bn(p + ".shortcut", stride, 0)
                if c.block == "bottleneck":
                    convs = [conv_bn(p + ".blocks.0", 1, 0), conv_bn(p + ".blocks.1", stride, 1),
                             conv_bn(p + ".blocks.2", 1, 0)]
                else:
                    convs = [conv_bn(p + ".blocks.0", stride, 1), conv_bn(p + ".blocks.1", 1, 1)]
                fused = None
                if self.use_tc:
                    if c.block != "bottleneck" and all(cv.tc_ok() for cv in convs):
                        need = L_.riser_res_tc_smem_ex(convs[0].cin_p, convs[1].cin_p, _pad16(convs[0].cout),
                                                       _pad16(convs[1].cout), 3, stride, 1,
                                                       1 if shortcut is not None else 0, self.precision)
                        if 0 < need <= max_smem:
                            fused = _FusedBasic(convs[0], convs[1], shortcut, dev, self.precision)
                    if fused is None:
                        for cv in convs + ([shortcut] if shortcut is not None else []):
                            cv.build_tc(dev, max_smem, self.precision)
                if fused is not None:
                    self.n_tc_fused += 1
                else:
                    for cv in convs + ([shortcut] if shortcut is not None else []):
                        if cv.tc is not None:
                            self.n_tc_convs += 1
                        else:
                            self.n_cuda_core_convs += 1
                self.blocks.append((convs, shortcut, fused))
                cin = cout
        self.c_last = cin
        self.c_last_p = _pad8(cin)
        fc = torch.zeros(self.n_classes, self.c_last_p)
        fc[:, :cin] = sd["decoder.2.weight"]
        self.fc_w = fc.contiguous().to(dev)
        self.fc_b = sd["decoder.2.bias"].contiguous().to(dev)
        self._acts = {}
        # (kernel, stride, padding) of every op of the main chain, kernel < 0 = the stem's max-pool (riser_len_chain)
        chain = [(self.stem.k, self.stem.stride, self.stem.pad), (-1, 2, 1)]
        for convs, _, _ in self.blocks:
            chain += [(cv.k, cv.stride, cv.pad) for cv in convs]
        self.n_chain = len(chain)
        self.chain = torch.tensor(chain, dtype=torch.int32).contiguous().to(dev)
        self.logger.debug('ResNet blocks: %d fused on tcgen05, %d convs on tcgen05, %d on CUDA cores',
                          self.n_tc_fused, self.n_tc_convs, self.n_cuda_core_convs)

    # ------------------------------------------------------------------ launches
    def _buf(self, key, *shape):
        # rows at or beyond a read's length are never read by any kernel (each takes the per-read lengths), so the
        # activation buffers need no clearing and are reused from call to call
        t = self._acts.get((key,) + shape)
        if t is None:
            t = self._acts[(key,) + shape] = torch.empty(*shape, dtype=torch.float32, device=self.device)
        return t

    def _conv_args(self, cv, x, n_in, L_in, n_out, out, residual, relu):
        """Arguments of riser_res_tc(_ex) for a single-conv launch, up to the stream."""
        t = cv.tc
        return (_lib.ptr(x), _lib.ptr(n_in), _lib.ptr(n_out), _lib.ptr(out), _lib.ptr(residual), _lib.ptr(t["w"]), None,
                None, _lib.ptr(t["bias"]), None, t["inv"], 1.0, x.shape[0], L_in, out.shape[1], cv.cin_p, 0, cv.cout_p,
                t["n1"], 0, cv.k, cv.stride, 1 if relu else 0)

    def _fused_args(self, fb, convs, x, n_in, L_in, n_out, out, residual):
        """Arguments of riser_res_tc(_ex) for a fused BasicBlock launch, up to the stream."""
        c1, c2 = convs
        return (_lib.ptr(x), _lib.ptr(n_in), _lib.ptr(n_out), _lib.ptr(out), _lib.ptr(residual), _lib.ptr(fb.w1),
                _lib.ptr(fb.w2), _lib.ptr(fb.wsc), _lib.ptr(fb.b1), _lib.ptr(fb.b2), fb.inv1, fb.inv2, x.shape[0], L_in,
                out.shape[1], c1.cin_p, c2.cin_p, c2.cout_p, fb.n1, fb.n2, 3, c1.stride, 1)

    def _conv(self, cv, x, n_in, L_in, n_out, residual=None, relu=True):
        B = x.shape[0]
        L_out = max(1, (L_in + 2 * cv.pad - cv.k) // cv.stride + 1)
        out = self._buf(id(cv), B, L_out, cv.cout_p)
        if cv.tc is not None:
            _lib.check(_lib.lib().riser_res_tc_ex(*self._conv_args(cv, x, n_in, L_in, n_out, out, residual, relu),
                                                  _lib.stream_ptr(), self.precision), "riser_res_tc")
            return out, L_out
        _lib.check(_lib.lib().riser_conv1d_cl(_lib.ptr(x), _lib.ptr(n_in), _lib.ptr(cv.w), _lib.ptr(cv.b),
                                              _lib.ptr(residual), _lib.ptr(out), _lib.ptr(n_out), B, L_in, L_out,
                                              cv.cin_p, cv.cout_p, cv.k, cv.stride, cv.pad, 1 if relu else 0,
                                              _lib.stream_ptr()), "riser_conv1d_cl")
        return out, L_out

    def _fused_block(self, fb, convs, shortcut, x, n_in, L_in, n_out):
        """A whole BasicBlock in one launch (csrc/resnet_tc.cu, fused mode)."""
        B = x.shape[0]
        c1, c2 = convs
        L_out = max(1, (L_in + 2 - 3) // c1.stride + 1)
        out = self._buf(id(fb), B, L_out, c2.cout_p)
        residual = x if shortcut is None else None              # identity shortcut: same layout as the output
        _lib.check(_lib.lib().riser_res_tc_ex(*self._fused_args(fb, convs, x, n_in, L_in, n_out, out, residual),
                                              _lib.stream_ptr(), self.precision), "riser_res_tc")
        return out, L_out

    def classify_batch(self, x, lens, max_len=None, probs=None, **_unused):
        """x: fp32 [B, ld] normalised signals on the device, lens int32 [B].  -> probs [B, n_classes]."""
        B = x.shape[0]
        if probs is None:
            probs = torch.empty(B, self.n_classes, dtype=torch.float32, device=self.device)
        if B == 0:
            return probs
        L0 = int(max_len if max_len is not None else x.shape[1])
        lens = lens.to(torch.int32)
        # valid lengths after every op of the main chain, one launch (stem conv, stem pool, every block conv)
        n_all = self._acts.get(("len", B))
        if n_all is None:
            n_all = self._acts[("len", B)] = torch.empty(self.n_chain, B, dtype=torch.int32, device=self.device)
        _lib.check(_lib.lib().riser_len_chain(_lib.ptr(lens), B, _lib.ptr(self.chain), self.n_chain, _lib.ptr(n_all),
                                              _lib.stream_ptr()), "riser_len_chain")
        st = self.stem
        if st.cin == 1 and st.k <= 32 and self.fused_stem:
            # conv + BN + ReLU + max-pool in one launch: the conv output (the largest activation) is never stored
            L = max(1, (L0 + 2 * st.pad - st.k) // st.stride + 1)
            L_p = L // 2 + 1
            pooled = self._buf("pool", B, L_p, st.cout_p)
            xc = x if (x.stride(1) == 1 and x.dtype == torch.float32) else x.contiguous()
            _lib.check(_lib.lib().riser_stem_pool_cl(_lib.ptr(xc), xc.stride(0), _lib.ptr(lens), _lib.ptr(st.w),
                                                     _lib.ptr(st.b), _lib.ptr(pooled), _lib.ptr(n_all[0]),
                                                     _lib.ptr(n_all[1]), B, L_p, st.cout_p, st.k, st.stride, st.pad,
                                                     _lib.stream_ptr()), "riser_stem_pool_cl")
        else:
            xin = x[:, :L0].contiguous().view(B, L0, 1)
            h, L = self._conv(st, xin, lens, L0, n_all[0])
            L_p = L // 2 + 1                                               # MaxPool1d(2, 2, padding=1)
            pooled = self._buf("pool", B, L_p, st.cout_p)
            _lib.check(_lib.lib().riser_maxpool1d_cl(_lib.ptr(h), _lib.ptr(n_all[0]), _lib.ptr(pooled),
                                                     _lib.ptr(n_all[1]), B, L, L_p, st.cout_p, _lib.stream_ptr()),
                       "riser_maxpool1d_cl")
        h, n, L, j = pooled, n_all[1], L_p, 2
        for convs, shortcut, fused in self.blocks:
            n_block = n_all[j + len(convs) - 1]             # the shortcut's output is as long as the block's
            if fused is not None:
                h, L = self._fused_block(fused, convs, shortcut, h, n, L, n_block)
                n = n_block
                j += len(convs)
                continue
            res = h
            if shortcut is not None:
                res, _ = self._conv(shortcut, h, n, L, n_block, relu=False)
            y, ny, Ly = h, n, L
            for k, cv in enumerate(convs):
                last = k == len(convs) - 1
                y, Ly = self._conv(cv, y, ny, Ly, n_all[j], residual=res if last else None, relu=True)
                ny = n_all[j]
                j += 1
            h, n, L = y, ny, Ly
        _lib.check(_lib.lib().riser_gap_linear_softmax(_lib.ptr(h), _lib.ptr(n), _lib.ptr(self.fc_w),
                                                       _lib.ptr(self.fc_b), _lib.ptr(probs), B, L, self.c_last_p,
                                                       self.n_classes, _lib.stream_ptr()),
                   "riser_gap_linear_softmax")
        return probs

    def classify(self, signal):
        """riser/model.py:22-28 for the ResNet: 1-D numpy -> Tensor[n_classes] on the device."""
        signal = np.asarray(signal)
        n = signal.shape[0]
        x = torch.from_numpy(signal).to(self.device, dtype=torch.float).view(1, n)
        lens = torch.tensor([n], dtype=torch.int32, device=self.device)
        return self.classify_batch(x, lens, max_len=n)[0]
