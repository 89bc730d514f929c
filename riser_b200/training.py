"""Train a ConvNet (riser/nets/cnn.py:8-65) on the GPU from the normalised windows ``retrain.preprocess_reads``
produces, and write checkpoints that ``riser_b200.Model`` and the reference's ``ConvNet`` both load.

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
import numpy as np
import torch
from torch import nn

from . import _lib
from .config import AttrDict
from .convnet_generic import check_supported


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
        _lib.check(lib.riser_gap_linear_ce_bwd(ptr(h), ptr(n_in), ptr(fc_w), ptr(fc_b), ptr(labels), B, Li, C,
                                               self.n_classes, ptr(s["loss"]), ptr(s["loss_mean"]), ptr(s["logits"]),
                                               ptr(s["dlogits"]), ptr(s["feat"]), ptr(dw), ptr(db), ptr(gh), stream),
                   "riser_gap_linear_ce_bwd")
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

    def gradients(self, x, lens, labels):
        """The loss gradients of the batch at the current weights, keyed like the state-dict (device tensors)."""
        x, lens, labels = self._inputs(x, lens, labels)
        self._run(x, lens, labels)
        return {k: p.grad.clone() for k, p in self.params.items()}

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
