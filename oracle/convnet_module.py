"""torch nn.Module restatement of riser/nets/cnn.py:8-65 (ConvNet, every configuration riser_b200 implements: depth >= 1,
odd kernels, 'gap_fc' and 'gap' heads, any n_classes).  Test infrastructure, see oracle/__init__.

Modules are created in the order the reference's ``__init__`` creates them -- the layers (``_make_layer``, cnn.py:52-65:
``depth`` x [Conv1d(k, stride 1, padding='same') + ReLU], then MaxPool1d(2, 2)), then the classifier (cnn.py:24-39)
-- so that under the same ``torch.manual_seed`` torch's default init draws the same weights as the reference's
``ConvNet(config.cnn)``.  State-dict keys are the reference's.  The tests use it as the float64 / fp32 autograd reference
of training and pin it against the reference's own outputs (tests/golden/convnet_generic.npz, and oracle/convnet_oracle
for the shipped shape)."""
import torch
from torch import nn


def _get(c, k):
    return c[k] if isinstance(c, dict) else getattr(c, k)


class ConvNet(nn.Module):
    def __init__(self, c):
        super().__init__()
        n, depth = int(_get(c, "n_layers")), int(_get(c, "depth"))
        channels, kernels = list(_get(c, "channels"))[:n], list(_get(c, "kernels"))[:n]
        layers, cin = [], 1
        for i in range(n):
            layers.append(self._make_layer(cin, int(channels[i]), int(kernels[i]), depth))
            cin = int(channels[i])
        self.layers = nn.Sequential(*layers)
        nc, head = int(_get(c, "n_classes")), _get(c, "classifier")
        if head == "gap_fc":                                    # cnn.py:28-33
            self.classifier = nn.Sequential(nn.AdaptiveAvgPool1d(1), nn.Flatten(1), nn.Linear(cin, nc))
        elif head == "gap":                                     # cnn.py:35-39
            self.classifier = nn.Sequential(nn.Conv1d(cin, nc, 1), nn.AdaptiveAvgPool1d(1), nn.Flatten(1))
        else:
            raise NotImplementedError(f"classifier {head!r}")

    @staticmethod
    def _make_layer(cin, cout, k, depth):
        mods = []
        for d in range(depth):
            mods += [nn.Conv1d(cin if d == 0 else cout, cout, k, stride=1, padding="same"), nn.ReLU(inplace=True)]
        mods.append(nn.MaxPool1d(2, 2))
        return nn.Sequential(*mods)

    def forward(self, x):                                       # cnn.py:43-50: [B, L] -> [B, n_classes]
        return self.classifier(self.layers(x.unsqueeze(1)))


def initial_state(c, seed):
    """The state-dict of ConvNet(c) as torch's default init draws it under torch.manual_seed(seed)."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        return {k: v.detach().clone() for k, v in ConvNet(c).state_dict().items()}
