"""Host-side mirror of riser/model.py (Model) backed by the sm_100a network kernels
in csrc/convnet.cu.

``Model(state, config, logger, target)`` and ``Model.classify(signal)`` keep the
reference's signature and behaviour (riser/model.py:7-28) so ``riser.py:41`` and
``control.py:69`` work unchanged; ``classify_batch`` is the additive batched entry
the rewritten loop uses.  A config with ``model: resnet`` (train.py:177-178) builds the
ResNet variant instead (``resnet.ResNetModel``, same call surface).  There is no CPU
fallback: constructing a Model without an sm_100 device raises.
"""
import ctypes

import numpy as np
import torch

from . import _lib

PREC_F16 = 0       # one tcgen05 pass, fp16 weights
PREC_F16_W2 = 1    # two passes, weights split hi + lo (exact to ~22 bits)
PREC_F16_X3 = 2    # three passes, weights and activations split hi + lo: fp32-class
PREC_F16_F8 = 3    # fp16 pass + one e4m3 pass carrying both hi/lo correction terms (2 pass-equivalents)
DEFAULT_PRECISION = PREC_F16_F8
MIN_LENGTH = 4096  # riser/preprocess.py:8 -- 12 stride-2 pools
# F16_F8 rows carry a8 = e4m3(a * 2^-F8_A_SHIFT) and lo8 = e4m3((a - hi) * 2^(9 - F8_LO_SHIFT)); the weight operands
# of the e4m3 pass carry the opposite powers of two (csrc/convnet.cu kF8AScale / kF8LoScale, which these must match)
F8_A_SHIFT = 3
F8_LO_SHIFT = 0
DEFAULT_CHUNK = 0    # 0 = whole batch in one plan (every launch covers the whole batch)


class Plan:
    """A launch plan (TMA tensor maps + geometry) for one (batch, max length) shape,
    with the activation workspace it owns."""
    def __init__(self, model, B, max_len):
        L = _lib.lib()
        self.B, self.max_len = B, max_len
        nbytes = L.riser_workspace_bytes(model._handle, B, max_len)
        self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=model.device)
        self._handle = ctypes.c_void_p()
        _lib.check(L.riser_plan_create(ctypes.byref(self._handle), model._handle, B, max_len,
                                       _lib.ptr(self.workspace), nbytes, _lib.stream_ptr()),
                   "riser_plan_create")
        self.launches = L.riser_forward_launches(self._handle)
        self.fused_layer0 = bool(L.riser_plan_fused_layer0(self._handle))

    def layer_info(self, i):
        off, rows, cp, c, nt = ctypes.c_int64(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        _lib.check(_lib.lib().riser_plan_layer_info(self._handle, i, ctypes.byref(off), ctypes.byref(rows),
                                                    ctypes.byref(cp), ctypes.byref(c), ctypes.byref(nt)),
                   "riser_plan_layer_info")
        return off.value, rows.value, cp.value, c.value, nt.value

    def layer_format(self, i):
        """Row format of layer i's input buffer: 1 = fp16, 2 = fp16 hi | lo, 3 = fp16 hi | e4m3 a | e4m3 lo (0: head)."""
        return int(_lib.lib().riser_plan_layer_format(self._handle, i))

    def layer_kernel(self, i):
        """Name of the kernel that runs conv layer i in this plan (riser_plan_layer_kernel)."""
        k = int(_lib.lib().riser_plan_layer_kernel(self._handle, i))
        return {0: "conv_tc_kernel", 1: "conv_eo_kernel", 2: "conv_pair_kernel", 3: "fused01_kernel",
                5: "conv_eo2_kernel"}.get(k, "?")

    def planes(self, i, n_layers, fmt=None):
        """Layer i's input buffer as the planes it stores, each [B, rows_per_read, channels] in its stored dtype:
        (hi, lo) fp16 for format 2, (hi fp16, a8 e4m3, lo8 e4m3) for format 3, (x,) otherwise (fp16; fp32 for the
        head's input).  `fmt` = row format, by default the one the plan reports (layer_format)."""
        if fmt is None:
            fmt = self.layer_format(i) or 1
            if fmt < 0:
                raise ValueError(f"layer {i}'s input is never materialised in this plan (fused into the previous launch)")
        off, rows, cp, c, _ = self.layer_info(i)
        dt = torch.float32 if i == n_layers else torch.float16
        nbytes = self.B * rows * cp * (4 if i == n_layers else 2)
        full = self.workspace[off:off + nbytes].view(dt)
        if i != n_layers and _lib.lib().riser_plan_layer_eo(self._handle, i):
            # even / odd plane layout: [parity][b][t // 2] -> [b][t]
            full = full.view(2, self.B, rows // 2, cp).permute(1, 2, 0, 3).reshape(self.B, rows, cp)
        else:
            full = full.view(self.B, rows, cp)
        half = cp // 2
        if fmt == 2 and i != n_layers:      # hi + lo planes side by side
            return full[:, :, :c], full[:, :, half:half + c]
        if fmt == 3 and i != n_layers:      # [hi fp16 | a8 e4m3 | lo8 e4m3] (bytes)
            raw = full.contiguous().view(torch.uint8).view(self.B, rows, cp * 2)
            a8 = raw[:, :, 2 * half:2 * half + c].contiguous().view(torch.float8_e4m3fn)
            lo8 = raw[:, :, 3 * half:3 * half + c].contiguous().view(torch.float8_e4m3fn)
            return full[:, :, :c], a8, lo8
        return (full[:, :, :c],)

    def activation(self, i, n_layers, planes=None):
        """Layer i's input buffer as a [B, rows_per_read, channels] tensor (tests); `planes` = row format,
        by default the one the plan reports (layer_format)."""
        p = self.planes(i, n_layers, planes)
        if len(p) == 2:
            return p[0].float() + p[1].float()
        if len(p) == 3:                    # hi + (a - hi), the e4m3 a8 is only an MMA operand
            return p[0].float() + p[2].float() * 2.0 ** -(9 - F8_LO_SHIFT)
        return p[0]

    def __del__(self):
        try:
            if self._handle:
                _lib.lib().riser_plan_destroy(self._handle)
        except Exception:
            pass


class Model():
    def __new__(cls, state=None, config=None, logger=None, target=None, precision=None):
        # a checkpoint trained with `model: resnet` (the reference's train.py) comes with a `resnet:` section and no
        # `cnn:` one: Model then is the ResNet variant (riser_b200/resnet.py), with the same call surface
        if cls is Model and getattr(config, "model", "cnn") == "resnet":
            from .resnet import ResNetModel
            return ResNetModel(state, config, logger, target, precision=precision)
        return super().__new__(cls)

    def __init__(self, state, config, logger, target, precision=None):
        self.target = target

        # Logger
        self.logger = logger

        # Device to run model on (riser/model.py:13-15; no CPU fallback here)
        self.device = self._get_device()
        self.logger.info('Using %s device', self.device)

        # Weights: a path to a .pth state-dict as riser.py:40 passes, or a state-dict
        c = config.cnn
        if isinstance(state, dict):
            sd = state
        else:
            sd = torch.load(state, map_location=torch.device('cpu'))
        self.precision = DEFAULT_PRECISION if precision is None else precision
        self._handle = ctypes.c_void_p()
        self._plans = {}
        self._build(sd, c)

    # ------------------------------------------------------------------ construction
    def _build(self, sd, c):
        """Shape checks mirror what ConvNet(config.cnn).load_state_dict would enforce
        (riser/nets/cnn.py:8-41, riser/model.py:18-19)."""
        self._generic = None
        if (c.classifier != 'gap_fc' or int(c.depth) != 1 or int(c.n_classes) != 2
                or any(int(k) != 3 for k in c.kernels[:c.n_layers]) or int(c.n_layers) < 2):
            # not the shipped shape (riser/model/*.yaml:6-12) the kernels of csrc/convnet.cu are written for: depth > 1,
            # other odd kernel sizes, 'gap' head, n_classes != 2 run on the generic channel-last ops
            # (riser/nets/cnn.py:8-65 in full; convnet_generic.py says what is still refused and why)
            from .convnet_generic import GenericConvNet
            self._generic = GenericConvNet(sd, c, self.device, self.logger)
            self.channels = [int(x) for x in c.channels[:int(c.n_layers)]]
            self.n_layers = int(c.n_layers)
            return
        n = int(c.n_layers)
        channels = [int(x) for x in c.channels[:n]]
        expected = {}
        cin = 1
        for i, cout in enumerate(channels):
            expected[f"layers.{i}.0.weight"] = (cout, cin, 3)
            expected[f"layers.{i}.0.bias"] = (cout,)
            cin = cout
        expected["classifier.2.weight"] = (2, channels[-1])
        expected["classifier.2.bias"] = (2,)
        missing = [k for k in expected if k not in sd]
        unexpected = [k for k in sd if k not in expected]
        if missing or unexpected:
            raise RuntimeError(f"Error(s) in loading state_dict for ConvNet: missing keys {missing}, "
                               f"unexpected keys {unexpected}")
        host = {}
        for k, shape in expected.items():
            t = torch.as_tensor(sd[k]).detach().to("cpu", torch.float32).contiguous()
            if tuple(t.shape) != shape:
                raise RuntimeError(f"size mismatch for {k}: checkpoint {tuple(t.shape)} vs model {shape}")
            host[k] = t
        self._host = host          # keep alive during the call
        self.channels = channels
        self.n_layers = n
        ch = (ctypes.c_int * n)(*channels)
        wp = (ctypes.c_void_p * n)(*[host[f"layers.{i}.0.weight"].data_ptr() for i in range(n)])
        bp = (ctypes.c_void_p * n)(*[host[f"layers.{i}.0.bias"].data_ptr() for i in range(n)])
        _lib.check(_lib.lib().riser_model_create(ctypes.byref(self._handle), n, ch, wp, bp,
                                                 ctypes.c_void_p(host["classifier.2.weight"].data_ptr()),
                                                 ctypes.c_void_p(host["classifier.2.bias"].data_ptr()),
                                                 self.precision, self.device.index or 0),
                   "riser_model_create")
        del self._host

    def _get_device(self):
        return _lib.require_device()

    def __del__(self):
        try:
            self._plans.clear()
            if self._handle:
                _lib.lib().riser_model_destroy(self._handle)
        except Exception:
            pass

    # ------------------------------------------------------------------ inference
    def plan(self, B, max_len):
        key = (int(B), int(max_len))
        p = self._plans.get(key)
        if p is None:
            p = self._plans[key] = Plan(self, key[0], key[1])
        return p

    def classify(self, signal):
        """riser/model.py:22-28: 1-D numpy (float64, or int64 zeros) -> Tensor[2] =
        (p_off_target, p_on_target) on the device."""
        signal = np.asarray(signal)
        if self._generic is not None:
            if signal.ndim != 1 or signal.shape[0] < self._generic.min_length:
                raise RuntimeError(f"signal of length {signal.shape} is shorter than {self._generic.min_length} samples")
            return self._generic.classify(signal)
        if signal.ndim != 1 or signal.shape[0] < MIN_LENGTH:
            # the reference dies in the 12th MaxPool1d for shorter input
            raise RuntimeError(f"signal of length {signal.shape} is shorter than {MIN_LENGTH} samples")
        n = signal.shape[0]
        ld = (n + 1023) & ~1023
        x = torch.zeros(1, ld, dtype=torch.float32, device=self.device)
        x[0, :n] = torch.from_numpy(signal).to(self.device, dtype=torch.float)
        lens = torch.tensor([n], dtype=torch.int32, device=self.device)
        return self.classify_batch(x, lens, max_len=ld)[0]

    def classify_batch(self, x, lens, max_len=None, probs=None, feat=None, chunk=None, events=None):
        """x: fp32 [B, ld] normalised signals on the device (8-byte aligned rows, even
        ld), lens: int32 [B] valid lengths (>= 4096; shorter -> NaN row).
        Returns probs fp32 [B, 2] on the device.  No synchronisation.

        chunk: optionally run the network over sub-batches of this many reads, one plan
        and one forward each (bounds the workspace; each launch covers its whole sub-batch).
        events: optional list; (start, end) torch.cuda.Event pairs bracketing layer 0 +
        the tcgen05 conv layers of every sub-batch are appended (bench.py's roofline;
        ``time_layer0`` gives the layer-0 share to subtract)."""
        if self._generic is not None:
            return self._generic.classify_batch(x, lens, max_len=max_len, probs=probs)
        B = x.shape[0]
        max_len = int(max_len if max_len is not None else x.shape[1])
        if probs is None:
            probs = torch.empty(B, 2, dtype=torch.float32, device=self.device)
        if B == 0:
            return probs
        chunk = int(chunk or DEFAULT_CHUNK or B)
        L = _lib.lib()
        stream = _lib.stream_ptr()
        for lo in range(0, B, chunk):
            n = min(chunk, B - lo)
            p = self.plan(n, max_len)
            xs, ls, ps = x[lo:lo + n], lens[lo:lo + n], probs[lo:lo + n]
            fs = None if feat is None else feat[lo:lo + n]
            if events is None:
                _lib.check(L.riser_forward(p._handle, _lib.ptr(xs), x.stride(0), _lib.ptr(ls), _lib.ptr(ps),
                                           _lib.ptr(fs), stream), "riser_forward")
                continue
            # stages 0 (tile activity flags + layer 0 unless fused) and 1 (the conv layers) bracketed
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for stage in range(3):
                _lib.check(L.riser_forward_stage(p._handle, stage, _lib.ptr(xs), x.stride(0), _lib.ptr(ls),
                                                 _lib.ptr(ps), _lib.ptr(fs), stream), "riser_forward_stage")
                if stage == 1:
                    e1.record()
            events.append((e0, e1))
        return probs

    def time_layer0(self, x, lens, max_len, iters=3):
        """Device time (ms) of the layer-0 launches alone (same chunk loop as a forward)."""
        p = self.plan(x.shape[0], max_len)
        L, stream = _lib.lib(), _lib.stream_ptr()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for k in range(iters + 1):
            if k == 1:
                e0.record()
            _lib.check(L.riser_forward_stage(p._handle, 3, _lib.ptr(x), x.stride(0), _lib.ptr(lens), None, None,
                                             stream), "riser_forward_stage")
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / iters

    def launches(self, B, max_len, chunk=None):
        """Kernels one classify_batch call launches."""
        if B <= 0:
            return 0
        if self._generic is not None:
            return self._generic.launches(B)
        chunk = int(chunk or DEFAULT_CHUNK or B)
        return sum(self.plan(min(chunk, B - lo), max_len).launches for lo in range(0, B, chunk))


def decide(probs, lens, threshold, mode, max_len):
    """riser/control.py:75-82 on the device: probs fp32 [M, B, 2], lens int32 [B]
    (0 = skipped) -> uint8 [B] decision codes (include/riser_b200.h)."""
    M, B = probs.shape[0], probs.shape[1]
    out = torch.empty(B, dtype=torch.uint8, device=probs.device)
    mode_code = {"enrich": 0, "deplete": 1}[mode]
    _lib.check(_lib.lib().riser_decide(_lib.ptr(probs), _lib.ptr(lens), B, M, float(threshold), mode_code,
                                       int(max_len), _lib.ptr(out), _lib.stream_ptr()), "riser_decide")
    return out
