"""Train a ConvNet (riser/nets/cnn.py:8-65) or the ResNet variant (riser/nets/resnet.py, ``ResNetTrainer``;
``make_trainer`` picks by ``config.model``) on the GPU from the normalised windows ``retrain.preprocess_reads``
produces, and write checkpoints that ``riser_b200.Model`` and the reference's networks load.

The reference trains with ``train.py`` on pytorch_lightning; this module is the same optimisation problem on the
package's own kernels, not a restatement of Lightning:
  * ``ConvNetTrainer`` holds fp32 master weights on the device and runs one step as
    forward  -- the GenericConvNet op sequence: ``riser_conv1d_cl`` (bias + ReLU fused) for every convolution,
                ``riser_maxpool1d_pad_cl`` (pad 0), ``riser_len_chain`` for the per-layer lengths of a ragged batch,
                every post-ReLU output kept;
    head     -- ``riser_gap_linear_ce_bwd``: average pool + linear + nn.CrossEntropyLoss (mean), with its gradients;
    backward -- per convolution ``riser_relu_pool_bwd_cl`` (ReLU + pool, or ReLU alone inside a layer of depth > 1),
                ``riser_conv1d_wgrad_cl`` (weight and bias gradients, tcgen05) and, for the input gradient,
                ``riser_conv1d_cl`` with the tap-flipped, transposed weight;
    update   -- ``torch.optim.Adam(lr=config.learning_rate)`` (elementwise, torch is the plumbing).
  * ``fit`` loops over epochs: every epoch draws shuffled batches from every window-length set (train.py's 2 s, 3 s
    and 4 s tensors) in one seeded interleaved order -- NOT a line-by-line restatement of Lightning's
    ``CombinedLoader`` --, validates, and writes ``<prefix>_latest.pth`` and, on a new lowest validation loss,
    ``<prefix>_best.pth``.
No CPU path: every op is a kernel of libriser_b200.so."""
import functools

import numpy as np
import torch
from torch import nn

from . import _lib
from .config import AttrDict
from .convnet_generic import check_supported


def _on_own_device(method):
    """Runs a trainer method with the trainer's device current, whatever device the calling thread has current: every
    launch goes to _lib.stream_ptr(), the current device's stream, and must go to the device that holds the buffers."""
    @functools.wraps(method)
    def guarded(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return method(self, *args, **kwargs)
    return guarded


def _cnn_config(config):
    c = config["cnn"] if "cnn" in config else config
    return c if isinstance(c, AttrDict) else AttrDict(c)


def default_init_state(cnn, seed):
    """The weights torch's default init gives ConvNet(config.cnn) (riser/nets/cnn.py:8-65) under
    torch.manual_seed(seed), under the reference's state-dict keys: the parametrised modules are created in the
    reference's order (the layers, ``depth`` Conv1d each, then the classifier's Linear or 1 x 1 Conv1d), so the RNG
    draws the same values.  The CPU RNG state of the caller is left as it was."""
    cnn = AttrDict(cnn)
    check_supported(cnn)
    sd, cin = {}, 1
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        for i in range(int(cnn.n_layers)):
            cout, k = int(cnn.channels[i]), int(cnn.kernels[i])
            for d in range(int(cnn.depth)):
                conv = nn.Conv1d(cin if d == 0 else cout, cout, k, stride=1, padding='same')
                sd[f"layers.{i}.{2 * d}.weight"], sd[f"layers.{i}.{2 * d}.bias"] = conv.weight.detach(), conv.bias.detach()
            cin = cout
        nc = int(cnn.n_classes)
        head, key = (nn.Linear(cin, nc), "classifier.2") if cnn.classifier == 'gap_fc' else (nn.Conv1d(cin, nc, 1), "classifier.0")
        sd[key + ".weight"], sd[key + ".bias"] = head.weight.detach(), head.bias.detach()
    return sd


class ConvNetTrainer:
    def __init__(self, config, state=None, seed=0, logger=None):
        c = _cnn_config(config)
        check_supported(c)
        self.device = _lib.require_device()
        self.logger = logger
        self.n_layers, self.depth = int(c.n_layers), int(c.depth)
        self.channels = [int(x) for x in c.channels[:self.n_layers]]
        self.kernels = [int(k) for k in c.kernels[:self.n_layers]]
        self.n_classes = int(c.n_classes)
        self.classifier = c.classifier
        self.min_length = 1 << self.n_layers          # the last pool needs two rows
        if state is None:
            state = default_init_state(c, seed)
        # (key, shape) of every parameter in the reference's state-dict order; convs[i][d] = (weight key, bias key)
        self.shapes, self.convs = {}, []
        cin = 1
        for i, (cout, k) in enumerate(zip(self.channels, self.kernels)):
            row = []
            for d in range(self.depth):
                wk, bk = f"layers.{i}.{2 * d}.weight", f"layers.{i}.{2 * d}.bias"
                self.shapes[wk], self.shapes[bk] = (cout, cin if d == 0 else cout, k), (cout,)
                row.append((wk, bk))
            self.convs.append(row)
            cin = cout
        pre = "classifier.2" if self.classifier == 'gap_fc' else "classifier.0"
        self.head_w, self.head_b = pre + ".weight", pre + ".bias"
        self.shapes[self.head_w] = (self.n_classes, cin) if self.classifier == 'gap_fc' else (self.n_classes, cin, 1)
        self.shapes[self.head_b] = (self.n_classes,)
        missing = [k for k in self.shapes if k not in state]
        unexpected = [k for k in state if k not in self.shapes]
        if missing or unexpected:
            raise RuntimeError(f"Error(s) in loading state_dict for ConvNet: missing keys {missing}, "
                               f"unexpected keys {unexpected}")
        self.params = {}
        for k, shape in self.shapes.items():
            t = torch.as_tensor(state[k]).detach().to(self.device, torch.float32).contiguous()
            if tuple(t.shape) != shape:
                raise RuntimeError(f"size mismatch for {k}: checkpoint {tuple(t.shape)} vs model {shape}")
            p = nn.Parameter(t.clone())
            p.grad = torch.zeros_like(p)
            self.params[k] = p
        lr = c.get("learning_rate", config.get("learning_rate", 1e-3))
        self.optimizer = torch.optim.Adam(list(self.params.values()), lr=float(lr))
        # per convolution: the forward weight [K][Cin][Cout] and the dgrad weight [K][Cout][Cin] (taps flipped)
        self._wf, self._wd = {}, {}
        for row in self.convs:
            for wk, _ in row:
                co, ci, k = self.shapes[wk]
                self._wf[wk] = torch.empty(k, ci, co, device=self.device)
                self._wd[wk] = torch.empty(k, co, ci, device=self.device)
        self._zero_bias = torch.zeros(max(self.channels + [1]), device=self.device)
        chain = []
        for k in self.kernels:
            chain += [(k, 1, (k - 1) // 2)] * self.depth + [(-1, 2, 0)]
        self.n_chain = len(chain)
        self.chain = torch.tensor(chain, dtype=torch.int32).to(self.device)
        self._bufs = {}
        self.reducer = None           # a data-parallel replica's side of the reductions (riser_b200.parallel)

    # ------------------------------------------------------------------ buffers of one (B, L) shape
    def _shape_bufs(self, B, L):
        key = (B, L)
        s = self._bufs.get(key)
        if s is not None:
            return s
        dev, f32 = self.device, torch.float32
        s = {"lens": torch.empty(self.n_chain, B, dtype=torch.int32, device=dev), "Y": [], "P": [], "gY": [], "gP": []}
        Li, ws, cin = L, 0, 1
        for i, cout in enumerate(self.channels):
            s["Y"].append([torch.empty(B, Li, cout, dtype=f32, device=dev) for _ in range(self.depth)])
            s["gY"].append([torch.empty(B, Li, cout, dtype=f32, device=dev) for _ in range(self.depth)])
            Lp = max(1, Li // 2)
            s["P"].append(torch.empty(B, Lp, cout, dtype=f32, device=dev))
            s["gP"].append(torch.empty(B, Lp, cout, dtype=f32, device=dev))
            for d in range(self.depth):
                ws = max(ws, _lib.lib().riser_conv1d_wgrad_workspace_bytes(B, Li, cin if d == 0 else cout, cout,
                                                                            self.kernels[i]))
            cin, Li = cout, Lp
        s["ws"] = torch.empty(max(ws, 16) // 4 + 4, dtype=f32, device=dev)
        s["ws_bytes"] = s["ws"].numel() * 4
        C = self.channels[-1]
        s["loss"] = torch.empty(B, dtype=f32, device=dev)
        s["loss_mean"] = torch.empty(1, dtype=f32, device=dev)
        s["logits"] = torch.empty(B, self.n_classes, dtype=f32, device=dev)
        s["dlogits"] = torch.empty(B, self.n_classes, dtype=f32, device=dev)
        s["feat"] = torch.empty(B, C, dtype=f32, device=dev)
        s["dfc_w"] = torch.empty(self.n_classes, C, dtype=f32, device=dev)
        s["dfc_b"] = torch.empty(self.n_classes, dtype=f32, device=dev)
        self._bufs[key] = s
        return s

    # ------------------------------------------------------------------ inputs
    @_on_own_device
    def _inputs(self, x, lens, labels):
        if x.dim() != 2:
            raise ValueError(f"x must be [B, L], got {tuple(x.shape)}")
        B, L = x.shape
        if lens.device.type == "cpu":
            lens_h = lens.to(torch.int64)
            if lens_h.shape != (B,):
                raise ValueError(f"lens must be [{B}], got {tuple(lens.shape)}")
            if B and (int(lens_h.min()) < self.min_length or int(lens_h.max()) > L):
                raise ValueError(f"read lengths must lie in [{self.min_length}, {L}] (2**n_layers samples leave one "
                                 "row for the last pool), got "
                                 f"[{int(lens_h.min())}, {int(lens_h.max())}]")
        if labels.device.type == "cpu":
            lab = labels.to(torch.int64)
            if B and (int(lab.min()) < 0 or int(lab.max()) >= self.n_classes):
                raise ValueError(f"labels must lie in [0, {self.n_classes}), got [{int(lab.min())}, {int(lab.max())}]")
        x = x.to(self.device, torch.float32).contiguous()
        lens = lens.to(self.device, torch.int32).contiguous()
        labels = labels.to(self.device, torch.int64).contiguous()
        return x, lens, labels

    # ------------------------------------------------------------------ forward + head + backward
    def _run(self, x, lens, labels, backward=True):
        lib, stream, ptr = _lib.lib(), _lib.stream_ptr(), _lib.ptr
        B, L = x.shape
        s = self._shape_bufs(B, L)
        n_all = s["lens"]
        _lib.check(lib.riser_len_chain(ptr(lens), B, ptr(self.chain), self.n_chain, ptr(n_all), stream),
                   "riser_len_chain")
        for row in self.convs:
            for wk, _ in row:
                self._wf[wk].copy_(self.params[wk].detach().permute(2, 1, 0))
        # forward
        h, n_in, Li, cin, j = x.view(B, L, 1), lens, L, 1, 0
        conv_len = []                  # per layer: the valid lengths of its convolutions' outputs, then of its pool
        for i, (cout, k) in enumerate(zip(self.channels, self.kernels)):
            for d in range(self.depth):
                wk, bk = self.convs[i][d]
                y = s["Y"][i][d]
                _lib.check(lib.riser_conv1d_cl(ptr(h), ptr(n_in), ptr(self._wf[wk]), ptr(self.params[bk]), None, ptr(y),
                                               ptr(n_all[j]), B, Li, Li, cin if d == 0 else cout, cout, k, 1,
                                               (k - 1) // 2, 1, stream), "riser_conv1d_cl")
                h, n_in = y, n_all[j]
                j += 1
            p = s["P"][i]
            Lp = p.shape[1]
            _lib.check(lib.riser_maxpool1d_pad_cl(ptr(h), ptr(n_in), ptr(p), ptr(n_all[j]), B, Li, Lp, cout, 0, stream),
                       "riser_maxpool1d_pad_cl")
            conv_len.append((n_in, n_all[j]))
            h, n_in, Li, cin = p, n_all[j], Lp, cout
            j += 1
        # head: loss and its gradients
        C = self.channels[-1]
        gh = s["gP"][-1]
        fc_w, fc_b = self.params[self.head_w], self.params[self.head_b]
        # without the backward pass (evaluate) the head's gradients go to scratch: the parameters' .grad stay as they were
        dw, db = (fc_w.grad, fc_b.grad) if backward else (s["dfc_w"], s["dfc_b"])
        _head(self.reducer if backward else None, h, n_in, fc_w, fc_b, labels, Li, C, self.n_classes, s, dw, db, gh)
        if backward:
            self._backward(s, x, lens, conv_len, B, L)
        return s

    def _backward(self, s, x, lens, conv_len, B, L):
        lib, stream, ptr = _lib.lib(), _lib.stream_ptr(), _lib.ptr
        for row in self.convs:
            for wk, _ in row:
                w, k = self.params[wk].detach(), self.shapes[wk][2]
                for t in range(k):
                    self._wd[wk][t].copy_(w[:, :, k - 1 - t])
        for i in reversed(range(self.n_layers)):
            cout, k = self.channels[i], self.kernels[i]
            cin = 1 if i == 0 else self.channels[i - 1]
            Li = s["Y"][i][0].shape[1]
            n_conv, _ = conv_len[i]
            dp = s["gP"][i]
            gz = s["gY"][i][self.depth - 1]
            _lib.check(lib.riser_relu_pool_bwd_cl(ptr(s["Y"][i][self.depth - 1]), ptr(dp), ptr(n_conv), ptr(gz), B, Li,
                                                  dp.shape[1], cout, 1, stream), "riser_relu_pool_bwd_cl")
            for d in reversed(range(self.depth)):
                wk, bk = self.convs[i][d]
                ci = cin if d == 0 else cout
                if d > 0:
                    xin = s["Y"][i][d - 1]
                elif i > 0:
                    xin = s["P"][i - 1]
                else:
                    xin = x.view(B, L, 1)
                _lib.check(lib.riser_conv1d_wgrad_cl(ptr(gz), ptr(xin), ptr(n_conv), B, Li, ci, cout, k,
                                                     ptr(self.params[wk].grad), ptr(self.params[bk].grad), ptr(s["ws"]),
                                                     s["ws_bytes"], stream), "riser_conv1d_wgrad_cl")
                if i == 0 and d == 0:
                    break
                # input gradient: the same convolution with the flipped, transposed weight
                gx = s["gY"][i][d - 1] if d > 0 else s["gP"][i - 1]
                _lib.check(lib.riser_conv1d_cl(ptr(gz), ptr(n_conv), ptr(self._wd[wk]), ptr(self._zero_bias), None,
                                               ptr(gx), ptr(n_conv), B, Li, Li, cout, ci, k, 1, (k - 1) // 2, 0, stream),
                           "riser_conv1d_cl (dgrad)")
                if d > 0:
                    gz = s["gY"][i][d - 1]
                    _lib.check(lib.riser_relu_pool_bwd_cl(ptr(s["Y"][i][d - 1]), ptr(gx), ptr(n_conv), ptr(gz), B, Li,
                                                          Li, cout, 0, stream), "riser_relu_pool_bwd_cl")

    # ------------------------------------------------------------------ public surface
    @_on_own_device
    def step(self, x, lens, labels):
        """One Adam step on the batch: x fp32 [B, ld] normalised windows, read b valid for lens[b] samples
        (2**n_layers <= lens[b] <= ld), labels int64 class indices.  Returns the mean loss as a 0-dim device tensor
        (a view of a buffer the next step at the same shape overwrites).  With x, lens and labels already on the
        device a step after the first at its shape neither allocates nor synchronises; it then does not check lens
        or labels either (a read that is too short or a label out of range makes the loss NaN and contributes no
        gradient).  lens / labels given as CPU tensors are checked and raise ValueError."""
        x, lens, labels = self._inputs(x, lens, labels)
        s = self._run(x, lens, labels)
        self.optimizer.step()
        return s["loss_mean"][0]

    @_on_own_device
    def gradients(self, x, lens, labels):
        """The loss gradients of the batch at the current weights, keyed like the state-dict (device tensors)."""
        x, lens, labels = self._inputs(x, lens, labels)
        self._run(x, lens, labels)
        return {k: p.grad.clone() for k, p in self.params.items()}

    @_on_own_device
    def evaluate(self, x, lens, labels):
        """(mean loss, number of reads whose argmax class is the label) at the current weights."""
        x, lens, labels = self._inputs(x, lens, labels)
        if x.shape[0] == 0:
            return float("nan"), 0
        s = self._run(x, lens, labels, backward=False)
        correct = int((s["logits"].argmax(dim=1) == labels).sum())
        return float(s["loss_mean"][0]), correct

    def state_dict(self):
        """CPU fp32 tensors under the reference's key names (loadable by riser_b200.Model and ConvNet)."""
        return {k: p.detach().to("cpu").clone() for k, p in self.params.items()}


# ---------------------------------------------------------------- ResNet (riser/nets/resnet.py)
BN_MOMENTUM, BN_EPS = 0.1, 1e-5           # nn.BatchNorm1d's defaults (resnet.py:23,29,80)
HEAD_MAX_CLASSES = 32                     # riser_gap_linear_ce_bwd's limit


def _resnet_config(config):
    c = config["resnet"] if "resnet" in config else config
    return c if isinstance(c, AttrDict) else AttrDict(c)


def _resnet_layout(c):
    """The convolutions of ResNet(c) in the key order of riser_b200.synth.resnet_state_dict: the stem, then per block
    (its key prefix, its convolutions, its shortcut, whether the shortcut is applied).  A convolution is
    (conv key, BN key, cin, cout, kernel, stride, padding)."""
    ch = [int(v) for v in c.channels]
    stem = ("conv_block.0", "conv_block.1", 1, ch[0], int(c.kernel), int(c.stride), int(c.padding))
    blocks, cin = [], ch[0]
    for i in range(int(c.n_layers)):
        cout = ch[i]
        for j in range(int(c.blocks[i])):
            s, p = 2 if (i > 0 and j == 0) else 1, f"layers.{i}.{j}"
            if c.block == "bottleneck":
                mid = cout // 4
                dims = [(cin, mid, 1, 1, 0), (mid, mid, 3, s, 1), (mid, cout, 1, 1, 0)]
            else:
                dims = [(cin, cout, 3, s, 1), (cout, cout, 3, 1, 1)]
            convs = [(f"{p}.blocks.{k}.0", f"{p}.blocks.{k}.1") + d for k, d in enumerate(dims)]
            blocks.append((p, convs, (f"{p}.shortcut.0", f"{p}.shortcut.1", cin, cout, 1, s, 0), cin != cout or s != 1))
            cin = cout
    return stem, blocks, cin


def check_resnet_supported(c):
    """Raise NotImplementedError for a ResNet configuration the training kernels do not take."""
    if c.block not in ("basic", "bottleneck"):
        raise NotImplementedError(f"ResNet block {c.block!r}: 'basic' or 'bottleneck'")
    if not 1 <= int(c.n_classes) <= HEAD_MAX_CLASSES:
        raise NotImplementedError(f"n_classes {c.n_classes}: the loss kernel takes 1 to {HEAD_MAX_CLASSES} classes")
    if not 1 <= int(c.kernel) <= 32 or int(c.stride) < 1 or int(c.padding) < 0:
        raise NotImplementedError(f"stem Conv1d(kernel {c.kernel}, stride {c.stride}, padding {c.padding}): the weight "
                                  "gradient takes kernels of 1 to 32 taps")


def resnet_default_init_state(c, seed):
    """The weights torch's default init gives a ResNet(c) (riser/nets/resnet.py) under torch.manual_seed(seed), under
    the reference's state-dict keys: Conv1d / Linear kaiming-uniform with their bias, BatchNorm1d weight 1, bias 0,
    running statistics 0 / 1, num_batches_tracked 0.  The modules are created in this order, which decides what the RNG
    draws: the stem's Conv1d (with bias), then for every block its main-branch Conv1d's and then its shortcut's 1 x 1
    Conv1d (created in every block, as resnet.py:21-24 does), then the decoder's Linear -- the key order of
    riser_b200.synth.resnet_state_dict and of oracle/resnet_module.py; the reference's own construction order is not
    restated.  The CPU RNG state of the caller is left as it was."""
    c = AttrDict(c)
    check_resnet_supported(c)
    stem, blocks, cin = _resnet_layout(c)
    sd = {}

    def conv_bn(ck, bk, ci, co, k, s, p, bias=False):
        conv = nn.Conv1d(ci, co, k, stride=s, padding=p, bias=bias)
        sd[ck + ".weight"] = conv.weight.detach()
        if bias:
            sd[ck + ".bias"] = conv.bias.detach()
        for name, v in nn.BatchNorm1d(co).state_dict().items():
            sd[f"{bk}.{name}"] = v

    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        conv_bn(*stem, bias=True)
        for _, convs, sc, _ in blocks:
            for cv in convs + [sc]:
                conv_bn(*cv)
        head = nn.Linear(cin, int(c.n_classes))
        sd["decoder.2.weight"], sd["decoder.2.bias"] = head.weight.detach(), head.bias.detach()
    return sd


class ResNetTrainer:
    """Trains ResNet(config.resnet) (riser/nets/resnet.py) on the GPU with the surface of ConvNetTrainer, so ``fit``
    trains it unchanged.  One step:
      forward  -- every convolution on ``riser_conv1d_cl`` (fp32, a zero bias where the Conv1d has none), its raw output
                  kept; ``riser_bn_stats_cl`` (batch statistics over the valid rows, float64; the running statistics
                  and num_batches_tracked updated in ``step`` only); ``riser_bn_apply_cl`` for BN [+ shortcut] [+ ReLU]
                  (a block's BN2(conv2) + BN_sc(conv_sc) + ReLU in one pass); ``riser_maxpool1d_pad_cl`` (padding 1);
                  ``riser_len_chain``;
      head     -- ``riser_gap_linear_ce_bwd``;
      backward -- ``riser_bn_bwd_cl`` (the block output's ReLU mask applied once, its result also the shortcut's
                  gradient), ``riser_conv1d_wgrad_ex`` (tcgen05) for every weight gradient, ``riser_conv1d_cl`` with the
                  tap-flipped weight for stride-1 input gradients and ``riser_conv1d_dgrad_cl`` for strided ones (the
                  shortcut's gradient added through their residual), ``riser_relu_pool_bwd_cl`` (pool 2) for the stem;
      update   -- ``torch.optim.Adam(lr=learning_rate)`` over the parameters that get a gradient.
    A ragged batch's BatchNorm statistics are over the valid rows of every read (torch's at equal lengths), so its
    gradient is not the mean of per-read gradients.  The shortcut parameters of identity blocks (built by the reference,
    never used) are carried unchanged into ``state_dict``."""

    def __init__(self, config, state=None, seed=0, logger=None):
        c = _resnet_config(config)
        check_resnet_supported(c)
        self.device = _lib.require_device()
        self.logger = logger
        self.n_classes = int(c.n_classes)
        self.stem, self.blocks, self.c_last = _resnet_layout(c)
        lib = _lib.lib()
        if lib.riser_conv1d_wgrad_ex_workspace_bytes(1, 1, 1, self.stem[3], self.stem[4]) == 0:
            raise NotImplementedError(f"stem kernel {self.stem[4]}: outside the weight gradient's limit")
        ref = resnet_default_init_state(c, seed)          # the keys, their order and shapes
        if state is None:
            state = ref
        missing = [k for k in ref if k not in state]
        unexpected = [k for k in state if k not in ref]
        if missing or unexpected:
            raise RuntimeError(f"Error(s) in loading state_dict for ResNet: missing keys {missing}, "
                               f"unexpected keys {unexpected}")
        self.keys = list(ref)
        unused = set()
        for _, _, sc, applied in self.blocks:
            if not applied:
                unused |= {k for k in ref if k.startswith(sc[0] + ".") or k.startswith(sc[1] + ".")}
        self.params, self.buffers, self.frozen = {}, {}, {}
        for k in self.keys:
            v = torch.as_tensor(state[k]).detach()
            if tuple(v.shape) != tuple(ref[k].shape):
                raise RuntimeError(f"size mismatch for {k}: checkpoint {tuple(v.shape)} vs model {tuple(ref[k].shape)}")
            if k in unused:
                self.frozen[k] = v.to("cpu").clone()
            elif k.endswith("num_batches_tracked"):
                self.buffers[k] = v.to(self.device, torch.int64).clone()
            elif k.endswith(("running_mean", "running_var")):
                self.buffers[k] = v.to(self.device, torch.float32).contiguous().clone()
            else:
                p = nn.Parameter(v.to(self.device, torch.float32).contiguous().clone())
                p.grad = torch.zeros_like(p)
                self.params[k] = p
        lr = c.get("learning_rate", config.get("learning_rate", 1e-3))
        self.optimizer = torch.optim.Adam(list(self.params.values()), lr=float(lr))
        # per convolution: forward weight [K][Cin][Cout] and input-gradient weight [K][Cout][Cin] (taps flipped for the
        # stride-1 ones, which run on riser_conv1d_cl; as they are for riser_conv1d_dgrad_cl)
        self.convs = [self.stem]
        for _, convs, sc, applied in self.blocks:
            self.convs += convs + ([sc] if applied else [])
        self._wf, self._wd = {}, {}
        for ck, _, ci, co, k, _, _ in self.convs:
            self._wf[ck] = torch.empty(k, ci, co, device=self.device)
            self._wd[ck] = torch.empty(k, co, ci, device=self.device)
        self._zero = torch.zeros(max(max(cv[2], cv[3]) for cv in self.convs), device=self.device)
        chain = [self.stem[4:7], (-1, 2, 1)]
        for _, convs, _, _ in self.blocks:
            chain += [cv[4:7] for cv in convs]
        self.chain_host = chain
        self.n_chain = len(chain)
        self.chain = torch.tensor(chain, dtype=torch.int32).to(self.device)
        self.stats = {cv[1]: (torch.empty(cv[3], device=self.device), torch.empty(cv[3], device=self.device))
                      for cv in self.convs}
        self.bn_ws = torch.empty(lib.riser_bn_workspace_bytes(max(cv[3] for cv in self.convs)) // 4 + 4,
                                 device=self.device)
        self._bufs = {}
        self.reducer = None           # a data-parallel replica's side of the reductions (riser_b200.parallel)

    # ------------------------------------------------------------------ buffers of one (B, L) shape
    def _shape_bufs(self, B, L):
        s = self._bufs.get((B, L))
        if s is not None:
            return s
        dev, lib = self.device, _lib.lib()

        def buf(Lx, C):
            return torch.empty(B, Lx, C, device=dev)

        def out_len(cv, Lx):
            return max(1, (Lx + 2 * cv[6] - cv[4]) // cv[5] + 1)

        # Y: convolution outputs, A: their BN + ReLU, H: block outputs, g*: their gradients; gM: a block's output
        # gradient through its ReLU mask; gin: a shortcut convolution's input gradient
        s = {"lens": torch.empty(self.n_chain, B, dtype=torch.int32, device=dev), "Y": {}, "A": {}, "gY": {}, "gA": {},
             "H": {}, "gH": {}, "gM": {}, "gin": {}}
        ws = 0
        L0 = out_len(self.stem, L)
        Lp = L0 // 2 + 1
        for key in ("Y", "A", "gY", "gA"):
            s[key][self.stem[0]] = buf(L0, self.stem[3])
        s["P"], s["gP"] = buf(Lp, self.stem[3]), buf(Lp, self.stem[3])
        ws = max(ws, lib.riser_conv1d_wgrad_ex_workspace_bytes(B, L0, 1, self.stem[3], self.stem[4]))
        Li = Lp
        for p, convs, sc, applied in self.blocks:
            L_in, Lx = Li, Li
            for k, cv in enumerate(convs):
                Lo = out_len(cv, Lx)
                s["Y"][cv[0]], s["gY"][cv[0]] = buf(Lo, cv[3]), buf(Lo, cv[3])
                if k < len(convs) - 1:
                    s["A"][cv[0]], s["gA"][cv[0]] = buf(Lo, cv[3]), buf(Lo, cv[3])
                ws = max(ws, lib.riser_conv1d_wgrad_ex_workspace_bytes(B, Lo, cv[2], cv[3], cv[4]))
                Lx = Lo
            s["H"][p], s["gH"][p], s["gM"][p] = buf(Lx, convs[-1][3]), buf(Lx, convs[-1][3]), buf(Lx, convs[-1][3])
            if applied:
                s["Y"][sc[0]], s["gY"][sc[0]] = buf(Lx, sc[3]), buf(Lx, sc[3])
                s["gin"][p] = buf(L_in, sc[2])
                ws = max(ws, lib.riser_conv1d_wgrad_ex_workspace_bytes(B, Lx, sc[2], sc[3], 1))
            Li = Lx
        s["ws"] = torch.empty(max(ws, 16) // 4 + 4, device=dev)
        C = self.c_last
        for k, shape in dict(loss=(B,), loss_mean=(1,), logits=(B, self.n_classes), dlogits=(B, self.n_classes),
                             feat=(B, C), dfc_w=(self.n_classes, C), dfc_b=(self.n_classes,)).items():
            s[k] = torch.empty(*shape, device=dev)
        self._bufs[(B, L)] = s
        return s

    # ------------------------------------------------------------------ inputs
    def _check_lengths(self, lens_h, L):
        """Host-side lengths: every op of the chain keeps at least one row per read, and every BatchNorm sees more
        than one value per channel (torch raises on that in training)."""
        if lens_h.numel() and (int(lens_h.min()) < 1 or int(lens_h.max()) > L):
            raise ValueError(f"read lengths must lie in [1, {L}], got [{int(lens_h.min())}, {int(lens_h.max())}]")
        n = lens_h.clone()
        for j, (k, st, pd) in enumerate(self.chain_host):
            if k < 0:
                n = torch.div(n + 2 * pd, 2, rounding_mode="floor")
            else:
                n = torch.clamp(torch.div(n + 2 * pd - k, st, rounding_mode="floor") + 1, min=0)
            if n.numel() and int(n.min()) < 1:
                raise ValueError(f"a read of {int(lens_h[int(n.argmin())])} samples leaves no row after op {j} "
                                 f"(kernel, stride, padding) = {self.chain_host[j]}")
            if k >= 0 and int(n.sum()) < 2:
                raise ValueError(f"op {j} leaves {int(n.sum())} value per channel for BatchNorm's batch statistics "
                                 "(more than 1 needed)")

    @_on_own_device
    def _inputs(self, x, lens, labels):
        if x.dim() != 2:
            raise ValueError(f"x must be [B, L], got {tuple(x.shape)}")
        B, L = x.shape
        if lens.device.type == "cpu":
            lens_h = lens.to(torch.int64)
            if lens_h.shape != (B,):
                raise ValueError(f"lens must be [{B}], got {tuple(lens.shape)}")
            self._check_lengths(lens_h, L)
        if labels.device.type == "cpu":
            lab = labels.to(torch.int64)
            if B and (int(lab.min()) < 0 or int(lab.max()) >= self.n_classes):
                raise ValueError(f"labels must lie in [0, {self.n_classes}), got [{int(lab.min())}, {int(lab.max())}]")
        x = x.to(self.device, torch.float32).contiguous()
        lens = lens.to(self.device, torch.int32).contiguous()
        labels = labels.to(self.device, torch.int64).contiguous()
        return x, lens, labels

    # ------------------------------------------------------------------ forward + head + backward
    def _conv(self, cv, h, n_in, L_in, y, n_out, bias=None):
        _lib.check(_lib.lib().riser_conv1d_cl(_lib.ptr(h), _lib.ptr(n_in), _lib.ptr(self._wf[cv[0]]),
                                              _lib.ptr(self._zero if bias is None else bias), None, _lib.ptr(y),
                                              _lib.ptr(n_out), h.shape[0], L_in, y.shape[1], cv[2], cv[3], cv[4],
                                              cv[5], cv[6], 0, _lib.stream_ptr()), "riser_conv1d_cl")

    def _bn_stats(self, cv, y, n, mode):
        """mode 'train': batch statistics, 'step': also update the running ones, 'eval': the running statistics."""
        if mode == "eval":
            return self.buffers[cv[1] + ".running_mean"], self.buffers[cv[1] + ".running_var"]
        mean, var = self.stats[cv[1]]
        run = [None] * 3
        if mode == "step":
            run = [self.buffers[cv[1] + k] for k in (".running_mean", ".running_var", ".num_batches_tracked")]
        if self.reducer is not None:
            self.reducer.bn_stats(cv, y, n, mean, var, run)
            return mean, var
        _lib.check(_lib.lib().riser_bn_stats_cl(_lib.ptr(y), _lib.ptr(n), y.shape[0], y.shape[1], cv[3], _lib.ptr(mean),
                                                _lib.ptr(var), *[_lib.ptr(t) for t in run], BN_MOMENTUM,
                                                _lib.ptr(self.bn_ws), self.bn_ws.numel() * 4, _lib.stream_ptr()),
                   "riser_bn_stats_cl")
        return mean, var

    def _bn_apply(self, cv, y, n, stats, out, relu, residual=None, res=None):
        P = _lib.ptr
        g, b = self.params[cv[1] + ".weight"], self.params[cv[1] + ".bias"]
        rs = [None] * 4 if res is None else [res[1][0], res[1][1], self.params[res[0][1] + ".weight"],
                                            self.params[res[0][1] + ".bias"]]
        _lib.check(_lib.lib().riser_bn_apply_cl(P(y), P(n), y.shape[0], y.shape[1], cv[3], P(stats[0]), P(stats[1]),
                                                P(g), P(b), P(residual), *[P(t) for t in rs], BN_EPS, 1 if relu else 0,
                                                P(out), _lib.stream_ptr()), "riser_bn_apply_cl")

    def _run(self, x, lens, labels, mode):
        """mode: 'step' (gradients, running statistics updated), 'train' (gradients only) or 'eval' (loss only)."""
        lib, ptr = _lib.lib(), _lib.ptr
        B, L = x.shape
        s = self._shape_bufs(B, L)
        n_all = s["lens"]
        _lib.check(lib.riser_len_chain(ptr(lens), B, ptr(self.chain), self.n_chain, ptr(n_all), _lib.stream_ptr()),
                   "riser_len_chain")
        for cv in self.convs:
            self._wf[cv[0]].copy_(self.params[cv[0] + ".weight"].detach().permute(2, 1, 0))
        st = self.stem
        Y0, A0 = s["Y"][st[0]], s["A"][st[0]]
        self._conv(st, x.view(B, L, 1), lens, L, Y0, n_all[0], bias=self.params[st[0] + ".bias"])
        stats = {st[1]: self._bn_stats(st, Y0, n_all[0], mode)}
        self._bn_apply(st, Y0, n_all[0], stats[st[1]], A0, True)
        _lib.check(lib.riser_maxpool1d_pad_cl(ptr(A0), ptr(n_all[0]), ptr(s["P"]), ptr(n_all[1]), B, A0.shape[1],
                                              s["P"].shape[1], st[3], 1, _lib.stream_ptr()), "riser_maxpool1d_pad_cl")
        h, n, Lh, j = s["P"], n_all[1], s["P"].shape[1], 2
        trace = []                                # per block: (input, its lengths, per conv (input, n_in, n_out))
        for p, convs, sc, applied in self.blocks:
            h_in, n_in, L_in = h, n, Lh
            ins = []
            for k, cv in enumerate(convs):
                y = s["Y"][cv[0]]
                self._conv(cv, h, n, Lh, y, n_all[j])
                ins.append((h, n, n_all[j]))
                stats[cv[1]] = self._bn_stats(cv, y, n_all[j], mode)
                if k < len(convs) - 1:
                    self._bn_apply(cv, y, n_all[j], stats[cv[1]], s["A"][cv[0]], True)
                    h = s["A"][cv[0]]
                n, Lh = n_all[j], y.shape[1]
                j += 1
            res = None
            if applied:
                ysc = s["Y"][sc[0]]
                self._conv(sc, h_in, n_in, L_in, ysc, n)
                stats[sc[1]] = self._bn_stats(sc, ysc, n, mode)
                res = (sc, stats[sc[1]])
            last = convs[-1]
            self._bn_apply(last, s["Y"][last[0]], n, stats[last[1]], s["H"][p], True,
                           residual=s["Y"][sc[0]] if applied else h_in, res=res)
            h = s["H"][p]
            trace.append((h_in, n_in, ins))
        C = self.c_last
        gh = s["gH"][self.blocks[-1][0]]
        fc_w, fc_b = self.params["decoder.2.weight"], self.params["decoder.2.bias"]
        dw, db = (fc_w.grad, fc_b.grad) if mode != "eval" else (s["dfc_w"], s["dfc_b"])
        _head(self.reducer if mode != "eval" else None, h, n, fc_w, fc_b, labels, Lh, C, self.n_classes, s, dw, db,
              gh)
        if mode != "eval":
            self._backward(s, x, lens, n_all, stats, trace)
        return s

    def _bn_bwd(self, cv, dout, mask, y, n, stats, dx, dy_out=None):
        if self.reducer is not None:
            self.reducer.bn_bwd(cv, dout, mask, y, n, stats, dx, dy_out)
            return
        P = _lib.ptr
        g = self.params[cv[1] + ".weight"]
        _lib.check(_lib.lib().riser_bn_bwd_cl(P(dout), P(mask), P(y), P(n), y.shape[0], y.shape[1], cv[3],
                                              P(stats[0]), P(stats[1]), P(g), BN_EPS, P(g.grad),
                                              P(self.params[cv[1] + ".bias"].grad), P(dx), P(dy_out),
                                              P(self.bn_ws), self.bn_ws.numel() * 4, _lib.stream_ptr()),
                   "riser_bn_bwd_cl")

    def _wgrad(self, s, cv, dz, n_out, x, n_in, db=None):
        _lib.check(_lib.lib().riser_conv1d_wgrad_ex(_lib.ptr(dz), _lib.ptr(x), _lib.ptr(n_out), _lib.ptr(n_in),
                                                    dz.shape[0], dz.shape[1], x.shape[1], cv[2], cv[3], cv[4], cv[5],
                                                    cv[6], _lib.ptr(self.params[cv[0] + ".weight"].grad),
                                                    _lib.ptr(db), _lib.ptr(s["ws"]), s["ws"].numel() * 4,
                                                    _lib.stream_ptr()), "riser_conv1d_wgrad_ex")

    def _dgrad(self, cv, dz, n_out, dx, n_in, residual=None):
        lib, P = _lib.lib(), _lib.ptr
        if cv[5] == 1:
            _lib.check(lib.riser_conv1d_cl(P(dz), P(n_out), P(self._wd[cv[0]]), P(self._zero), P(residual), P(dx),
                                           P(n_in), dz.shape[0], dz.shape[1], dx.shape[1], cv[3], cv[2], cv[4], 1,
                                           cv[4] - 1 - cv[6], 0, _lib.stream_ptr()), "riser_conv1d_cl (dgrad)")
        else:
            _lib.check(lib.riser_conv1d_dgrad_cl(P(dz), P(n_out), P(self._wd[cv[0]]), P(residual), P(dx), P(n_in),
                                                 dz.shape[0], dz.shape[1], dx.shape[1], cv[2], cv[3], cv[4], cv[5],
                                                 cv[6], _lib.stream_ptr()), "riser_conv1d_dgrad_cl")

    def _bn_backward_order(self):
        """The convolutions whose BatchNorm _backward differentiates, in its order (self.convs is the forward's)."""
        order = []
        for _, convs, sc, applied in reversed(self.blocks):
            order += [convs[-1]] + ([sc] if applied else []) + convs[-2::-1]
        return order + [self.stem]

    def _backward(self, s, x, lens, n_all, stats, trace):
        for cv in self.convs:
            w = self.params[cv[0] + ".weight"].detach()
            self._wd[cv[0]].copy_((w.flip(2) if cv[5] == 1 else w).permute(2, 0, 1))
        for bi in reversed(range(len(self.blocks))):
            p, convs, sc, applied = self.blocks[bi]
            h_in, n_in, ins = trace[bi]
            g_in = s["gH"][self.blocks[bi - 1][0]] if bi > 0 else s["gP"]
            last = convs[-1]
            n_out = ins[-1][2]
            gm = s["gM"][p]
            # the block output's ReLU mask, applied once: gm feeds the main branch's BN and the shortcut
            self._bn_bwd(last, s["gH"][p], s["H"][p], s["Y"][last[0]], n_out, stats[last[1]], s["gY"][last[0]],
                         dy_out=gm)
            res = gm
            if applied:
                gsc = s["gY"][sc[0]]
                self._bn_bwd(sc, gm, None, s["Y"][sc[0]], n_out, stats[sc[1]], gsc)
                self._wgrad(s, sc, gsc, n_out, h_in, n_in)
                res = s["gin"][p]
                self._dgrad(sc, gsc, n_out, res, n_in)
            for k in reversed(range(len(convs))):
                cv = convs[k]
                xin, nk_in, nk_out = ins[k]
                dz = s["gY"][cv[0]]
                self._wgrad(s, cv, dz, nk_out, xin, nk_in)
                if k > 0:
                    prev = convs[k - 1]
                    self._dgrad(cv, dz, nk_out, s["gA"][prev[0]], nk_in)
                    self._bn_bwd(prev, s["gA"][prev[0]], s["A"][prev[0]], s["Y"][prev[0]], nk_in, stats[prev[1]],
                                 s["gY"][prev[0]])
                else:
                    self._dgrad(cv, dz, nk_out, g_in, nk_in, residual=res)
        st = self.stem
        B, L = x.shape
        A0 = s["A"][st[0]]
        _lib.check(_lib.lib().riser_relu_pool_bwd_cl(_lib.ptr(A0), _lib.ptr(s["gP"]), _lib.ptr(n_all[0]),
                                                     _lib.ptr(s["gA"][st[0]]), B, A0.shape[1], s["gP"].shape[1], st[3],
                                                     2, _lib.stream_ptr()), "riser_relu_pool_bwd_cl")
        self._bn_bwd(st, s["gA"][st[0]], None, s["Y"][st[0]], n_all[0], stats[st[1]], s["gY"][st[0]])
        self._wgrad(s, st, s["gY"][st[0]], n_all[0], x.view(B, L, 1), lens, db=self.params[st[0] + ".bias"].grad)

    # ------------------------------------------------------------------ public surface
    @_on_own_device
    def step(self, x, lens, labels):
        """One Adam step on the batch (x fp32 [B, ld] normalised windows, read b valid for lens[b] samples, labels
        int64), with BatchNorm's batch statistics; the running statistics and num_batches_tracked are updated once.
        Returns the mean loss as a 0-dim device tensor (a view of a buffer the next step at the same shape overwrites).
        With x, lens and labels on the device a step after the first at its shape neither allocates nor synchronises,
        and does not check lens or labels; lens / labels given as CPU tensors are checked and raise ValueError."""
        x, lens, labels = self._inputs(x, lens, labels)
        s = self._run(x, lens, labels, "step")
        self.optimizer.step()
        return s["loss_mean"][0]

    @_on_own_device
    def gradients(self, x, lens, labels):
        """The loss gradients of the batch at the current weights (batch statistics; the running statistics stay as
        they are), keyed like the state-dict (device tensors)."""
        x, lens, labels = self._inputs(x, lens, labels)
        self._run(x, lens, labels, "train")
        return {k: p.grad.clone() for k, p in self.params.items()}

    @_on_own_device
    def evaluate(self, x, lens, labels):
        """(mean loss, number of reads whose argmax class is the label) in eval mode (the running statistics)."""
        x, lens, labels = self._inputs(x, lens, labels)
        if x.shape[0] == 0:
            return float("nan"), 0
        s = self._run(x, lens, labels, "eval")
        correct = int((s["logits"].argmax(dim=1) == labels).sum())
        return float(s["loss_mean"][0]), correct

    def state_dict(self):
        """CPU tensors under the reference's keys, in synth.resnet_state_dict's order (loadable by riser_b200.Model with
        ``model: resnet`` and by the reference's ResNet): fp32 parameters and running statistics, num_batches_tracked
        int64, the unused shortcut tensors as they were given."""
        out = {}
        for k in self.keys:
            src = self.params.get(k, self.buffers.get(k))
            out[k] = self.frozen[k].clone() if src is None else src.detach().to("cpu").clone()
        return out


def _head(reducer, h, n, fc_w, fc_b, labels, L_pad, C, n_classes, s, dw, db, dh):
    """The loss head (riser_gap_linear_ce_bwd).  A data-parallel replica in training (reducer set) divides by the
    global batch and writes its share of the mean loss where the replicas' gradient exchange adds them up."""
    lib, ptr, B = _lib.lib(), _lib.ptr, h.shape[0]
    if reducer is None:
        _lib.check(lib.riser_gap_linear_ce_bwd(ptr(h), ptr(n), ptr(fc_w), ptr(fc_b), ptr(labels), B, L_pad, C,
                                               n_classes, ptr(s["loss"]), ptr(s["loss_mean"]), ptr(s["logits"]),
                                               ptr(s["dlogits"]), ptr(s["feat"]), ptr(dw), ptr(db), ptr(dh),
                                               _lib.stream_ptr()), "riser_gap_linear_ce_bwd")
    else:
        _lib.check(lib.riser_gap_linear_ce_bwd_ex(ptr(h), ptr(n), ptr(fc_w), ptr(fc_b), ptr(labels), B, reducer.batch,
                                                  L_pad, C, n_classes, ptr(s["loss"]), ptr(reducer.loss),
                                                  ptr(s["logits"]), ptr(s["dlogits"]), ptr(s["feat"]), ptr(dw), ptr(db),
                                                  ptr(dh), _lib.stream_ptr()), "riser_gap_linear_ce_bwd_ex")


def model_of(config):
    """``config.model`` ('cnn' when absent)."""
    model = (config.get("model") if isinstance(config, dict) else getattr(config, "model", None)) or "cnn"
    if model not in ("cnn", "resnet"):
        raise NotImplementedError(f"model {model!r}: 'cnn' or 'resnet'")
    return model


def make_trainer(config, state=None, seed=0, logger=None, devices=None):
    """ConvNetTrainer or ResNetTrainer by ``config.model`` ('cnn' when absent), as the reference's train.py:175-184
    and riser_b200.Model choose the network.  ``devices`` naming more than one GPU: a
    riser_b200.parallel.DataParallelTrainer over them; one device: the single-device trainer built on it."""
    model = model_of(config)
    if devices is not None:
        from .parallel import DataParallelTrainer, check_devices
        devices = check_devices(devices)
        if len(devices) > 1:
            return DataParallelTrainer(config, devices, state=state, seed=seed, logger=logger)
        with torch.cuda.device(devices[0]):
            return make_trainer(config, state=state, seed=seed, logger=logger)
    cls = ResNetTrainer if model == "resnet" else ConvNetTrainer
    return cls(config, state=state, seed=seed, logger=logger)


# ---------------------------------------------------------------- data (riser/data.py)
def load_tensors(negative_pt, positive_pt):
    """Negative then positive windows (torch.load'ed [N, L] tensors or paths to them), labels 0 then 1."""
    neg = negative_pt if torch.is_tensor(negative_pt) else torch.load(negative_pt)
    pos = positive_pt if torch.is_tensor(positive_pt) else torch.load(positive_pt)
    x = torch.cat([neg, pos]).to(torch.float32)
    y = torch.cat([torch.zeros(len(neg), dtype=torch.int64), torch.ones(len(pos), dtype=torch.int64)])
    return x, y


def fit(trainer, train_sets, val_sets, epochs, batch_size, out_prefix, seed=0, logger=None):
    """Train for ``epochs`` epochs.  train_sets / val_sets: lists of (x [N, L], labels [N]), one per window length.
    Each epoch shuffles every set, cuts it into batches of ``batch_size`` and runs them in one seeded interleaved
    order; then it validates (loss averaged over reads, accuracy), writes ``<out_prefix>_latest.pth`` and, when the
    validation loss is the lowest so far, ``<out_prefix>_best.pth``.  Returns the per-epoch history."""
    rng = np.random.Generator(np.random.PCG64(seed))
    dev = trainer.device

    def upload(sets):
        out = []
        for x, y in sets:
            x = torch.as_tensor(x, dtype=torch.float32)
            y = torch.as_tensor(y, dtype=torch.int64)
            trainer._inputs(x[:1], torch.tensor([x.shape[1]], dtype=torch.int32), y)      # checks length and labels
            out.append((x.to(dev).contiguous(), y.to(dev)))
        return out

    train, val = upload(train_sets), upload(val_sets)
    best, history = float("inf"), []
    for epoch in range(epochs):
        batches = []
        for si, (x, _) in enumerate(train):
            perm = rng.permutation(x.shape[0])
            batches += [(si, perm[k:k + batch_size]) for k in range(0, len(perm), batch_size)]
        order = rng.permutation(len(batches))
        train_loss = torch.zeros((), device=dev)
        for bi in order:
            si, idx = batches[bi]
            x, y = train[si]
            idx = torch.from_numpy(idx).to(dev)
            xb = x.index_select(0, idx)
            lens = torch.full((xb.shape[0],), xb.shape[1], dtype=torch.int32, device=dev)
            train_loss += trainer.step(xb, lens, y.index_select(0, idx))
        total, correct, n = 0.0, 0, 0
        for x, y in val:
            for k in range(0, x.shape[0], batch_size):
                xb, yb = x[k:k + batch_size], y[k:k + batch_size]
                lens = torch.full((xb.shape[0],), xb.shape[1], dtype=torch.int32, device=dev)
                loss, c = trainer.evaluate(xb, lens, yb)
                total += loss * xb.shape[0]
                correct += c
                n += xb.shape[0]
        val_loss = total / max(n, 1)
        val_acc = correct / max(n, 1)
        rec = {"epoch": epoch, "train_loss": float(train_loss) / max(len(batches), 1), "val_loss": val_loss,
               "val_acc": val_acc}
        history.append(rec)
        if logger is not None:
            logger.info("epoch %d: train loss %.5f, val loss %.5f, val acc %.4f", epoch, rec["train_loss"], val_loss,
                        val_acc)
        sd = trainer.state_dict()
        torch.save(sd, f"{out_prefix}_latest.pth")
        if val_loss < best:
            best = val_loss
            torch.save(sd, f"{out_prefix}_best.pth")
    return history
