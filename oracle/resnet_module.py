"""torch nn.Module restatement of riser/nets/resnet.py (ResNet, BasicBlock, BottleneckBlock) for training, with the
reference's state-dict keys.  Test infrastructure, see oracle/__init__.

``forward(x)`` is the plain module in train or eval mode.  ``forward(x, lens)`` runs a ragged batch ``x`` [B, L] whose
read b is valid for ``lens[b]`` samples the way riser_b200's ResNetTrainer does: every op sees zeros (max-pool: -inf)
outside each read's valid rows, BatchNorm's training statistics are over the valid rows of every read (the running
statistics are updated from them), and the average pool is over each read's valid rows.  At equal lengths that is the
plain module.  ``force`` (with ``lens``) replaces ReLU masks and max-pool choices by given ones, so that a float64
reference can take an fp32 forward's decisions: ``force[name]`` is a bool [B, C, L] mask for the ReLU after ``name``
("conv_block" and every "layers.i.j.blocks.k" but the last of a block, and "layers.i.j" for the block output), and
``force["pool"]`` a bool [B, C, L_pool] that is True where the stem's max-pool takes the second row of its window.

Modules are registered -- and torch's default init draws -- in this order: the stem (Conv1d with bias, BatchNorm1d),
then for every block its main-branch convolutions and BatchNorms, then its shortcut Conv1d and BatchNorm1d, then the
decoder's Linear.  That is the key order of riser_b200.synth.resnet_state_dict; the reference's own construction order
is not part of this checkout.  The shortcut's parameters exist in every block (resnet.py:21-24), used or not."""
import torch
import torch.nn.functional as F
from torch import nn


def _get(c, k):
    return c[k] if isinstance(c, dict) else getattr(c, k)


def _conv_bn(cin, cout, k, stride=1, padding=0, relu=True):
    """resnet.py:26-37: Conv1d (no bias) -> BatchNorm1d [-> ReLU]."""
    mods = [nn.Conv1d(cin, cout, k, stride=stride, padding=padding, bias=False), nn.BatchNorm1d(cout)]
    return nn.Sequential(*(mods + ([nn.ReLU()] if relu else [])))


class ResidualBlock(nn.Module):
    """resnet.py:39-70: BasicBlock (k3 / stride s, k3) or BottleneckBlock (1x1, k3 / stride s, 1x1 with cout / 4
    channels inside); output ReLU(main + shortcut), the shortcut BN(Conv1d 1x1, stride s) when cin != cout or s != 1."""

    def __init__(self, cin, cout, stride, kind):
        super().__init__()
        if kind == "bottleneck":
            mid = cout // 4
            self.blocks = nn.Sequential(_conv_bn(cin, mid, 1), _conv_bn(mid, mid, 3, stride, 1),
                                        _conv_bn(mid, cout, 1, relu=False))
        elif kind == "basic":
            self.blocks = nn.Sequential(_conv_bn(cin, cout, 3, stride, 1), _conv_bn(cout, cout, 3, 1, 1, relu=False))
        else:
            raise NotImplementedError(f"block {kind!r}")
        self.shortcut = nn.Sequential(nn.Conv1d(cin, cout, 1, stride=stride, bias=False), nn.BatchNorm1d(cout))
        self.apply_shortcut = cin != cout or stride != 1

    def forward(self, x):
        res = self.shortcut(x) if self.apply_shortcut else x
        return F.relu(self.blocks(x) + res)


class ResNet(nn.Module):
    def __init__(self, c):
        super().__init__()
        ch = [int(v) for v in _get(c, "channels")]
        self.conv_block = nn.Sequential(
            nn.Conv1d(1, ch[0], int(_get(c, "kernel")), stride=int(_get(c, "stride")), padding=int(_get(c, "padding"))),
            nn.BatchNorm1d(ch[0]), nn.ReLU(), nn.MaxPool1d(2, 2, padding=1))
        layers, cin = [], ch[0]
        for i in range(int(_get(c, "n_layers"))):
            blocks = []
            for j in range(int(_get(c, "blocks")[i])):
                blocks.append(ResidualBlock(cin, ch[i], 2 if (i > 0 and j == 0) else 1, _get(c, "block")))
                cin = ch[i]
            layers.append(nn.Sequential(*blocks))
        self.layers = nn.Sequential(*layers)
        self.decoder = nn.Sequential(nn.AdaptiveAvgPool1d(1), nn.Flatten(1), nn.Linear(cin, int(_get(c, "n_classes"))))

    def forward(self, x, lens=None, force=None):
        if lens is None:
            return self.decoder(self.layers(self.conv_block(x.unsqueeze(1))))
        return self._masked(x, [int(n) for n in lens], force or {})

    # ---------------------------------------------------------------- ragged batch
    def _bn(self, bn, y, m):
        n = float(m.sum())
        if bn.training:
            mean = torch.where(m, y, 0).sum((0, 2)) / n
            d = torch.where(m, y - mean[None, :, None], 0)
            var = (d * d).sum((0, 2)) / n
            with torch.no_grad():
                bn.running_mean.mul_(1 - bn.momentum).add_(bn.momentum * mean)
                bn.running_var.mul_(1 - bn.momentum).add_(bn.momentum * var * n / (n - 1))
                bn.num_batches_tracked += 1
        else:
            mean, var = bn.running_mean, bn.running_var
        return (y - mean[None, :, None]) / torch.sqrt(var[None, :, None] + bn.eps) * bn.weight[None, :, None] + \
            bn.bias[None, :, None]

    @staticmethod
    def _mask(lens, L, dev):
        return (torch.arange(L, device=dev)[None, :] < torch.tensor(lens, device=dev)[:, None])[:, None, :]

    def _relu(self, y, m, name, force):
        keep = force[name][..., :y.shape[2]] if name in force else y > 0
        return torch.where(m & keep, y, 0)

    def _conv(self, conv, h, lens):
        out = [max(0, (n + 2 * conv.padding[0] - conv.kernel_size[0]) // conv.stride[0] + 1) for n in lens]
        y = conv(h)
        return y, out, self._mask(out, y.shape[2], y.device)

    def _masked(self, x, lens, force):
        dev = x.device
        m = self._mask(lens, x.shape[1], dev)
        h = torch.where(m, x.unsqueeze(1), 0)
        conv, bn = self.conv_block[0], self.conv_block[1]
        y, lens, m = self._conv(conv, h, lens)
        h = self._relu(self._bn(bn, y, m), m, "conv_block", force)
        # MaxPool1d(2, 2, padding 1): window p = (h[2p - 1], h[2p]), -inf outside the read
        hp = torch.where(m, h, float("-inf"))
        if hp.shape[2] % 2:
            hp = torch.cat([hp, torch.full_like(hp[:, :, :1], float("-inf"))], 2)
        hp = torch.cat([torch.full_like(hp[:, :, :1], float("-inf")), hp, torch.full_like(hp[:, :, :1], float("-inf"))], 2)
        Lp = y.shape[2] // 2 + 1                                  # MaxPool1d's output length
        first, second = hp[:, :, 0::2][..., :Lp], hp[:, :, 1::2][..., :Lp]
        take2 = force["pool"][..., :first.shape[2]] if "pool" in force else (second > first) | torch.isnan(second)
        lens = [n // 2 + 1 if n > 0 else 0 for n in lens]
        m = self._mask(lens, first.shape[2], dev)
        h = torch.where(m, torch.where(take2, second, first), 0)
        for i, layer in enumerate(self.layers):
            for j, blk in enumerate(layer):
                name = f"layers.{i}.{j}"
                y_in, lens_in = h, lens
                for k, cb in enumerate(blk.blocks):
                    y, lens, m = self._conv(cb[0], h, lens)
                    h = self._bn(cb[1], y, m)
                    if k < len(blk.blocks) - 1:
                        h = self._relu(h, m, f"{name}.blocks.{k}", force)
                if blk.apply_shortcut:
                    ys, _, _ = self._conv(blk.shortcut[0], y_in, lens_in)
                    res = self._bn(blk.shortcut[1], ys, m)
                else:
                    res = y_in
                h = self._relu(h + res, m, name, force)
        n = torch.tensor(lens, device=dev, dtype=h.dtype)[:, None]
        return self.decoder[2](h.sum(2) / n)


def initial_state(c, seed):
    """The state-dict of ResNet(c) as torch's default init draws it under torch.manual_seed(seed)."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        return {k: v.detach().clone() for k, v in ResNet(c).state_dict().items()}
