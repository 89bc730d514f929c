"""CPU: the ResNet the training tests compare against (oracle/resnet_module.py) is pinned against the eval-mode oracle and
the reference's own outputs, its ragged-batch (masked) training mode equals torch's BatchNorm at equal lengths, and the
trainer's initial weights (riser_b200.training.resnet_default_init_state) are the ones that module draws."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import preprocess_oracle as pp, resnet_oracle
from oracle.resnet_module import ResNet, initial_state
from riser_b200 import synth
from riser_b200.training import resnet_default_init_state

CONFIGS = synth.RESNET_CONFIGS


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_module_matches_eval_oracle(name):
    cfg = CONFIGS[name]
    sd = synth.resnet_state_dict(cfg, 0)
    net = ResNet(cfg).eval()
    net.load_state_dict(sd)                                     # strict: the reference's keys, shortcuts included
    assert list(net.state_dict()) == list(sd)
    x = torch.randn(3, 5000, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        want = resnet_oracle.logits(sd, cfg, x)
        assert torch.equal(net(x), want)
        assert torch.allclose(net(x, [5000] * 3), want, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_module_matches_reference_golden_probabilities(golden_dir, name):
    g = np.load(os.path.join(golden_dir, "resnet_probs.npz"))
    bodies = synth.ragged_bodies(int(g["seed"]), 24, 4096, 12048)
    cfg = CONFIGS[name]
    net = ResNet(cfg).eval()
    net.load_state_dict(synth.resnet_state_dict(cfg, 0))
    with torch.no_grad():
        for i in (0, 5, 11, 23):
            x = torch.from_numpy(np.asarray(pp.mad_normalise(bodies[i]), dtype=np.float32))[None]
            assert np.abs(F.softmax(net(x), 1)[0].numpy() - g[f"probs_{name}"][i]).max() < 1e-6, i


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_masked_training_mode_equals_batch_norm_at_equal_lengths(name):
    """At equal lengths the ragged-batch path is torch's training-mode BatchNorm: logits, gradients and the running
    statistics (and num_batches_tracked) after the step."""
    cfg = CONFIGS[name]
    sd = synth.resnet_state_dict(cfg, 1)
    plain, masked = ResNet(cfg).double().train(), ResNet(cfg).double().train()
    plain.load_state_dict(sd)
    masked.load_state_dict(sd)
    x = torch.randn(3, 3000, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    a, b = plain(x), masked(x, [3000] * 3)
    assert torch.allclose(a, b, rtol=1e-12, atol=1e-11)
    a.square().sum().backward()
    b.square().sum().backward()
    for (k, p), q in zip(plain.named_parameters(), masked.parameters()):
        if p.grad is None:
            assert q.grad is None, k                            # the unused shortcut parameters
        else:
            assert torch.allclose(p.grad, q.grad, rtol=1e-9, atol=1e-11), k
    for (k, u), v in zip(plain.named_buffers(), masked.buffers()):
        assert torch.allclose(u.double(), v.double(), rtol=1e-12, atol=1e-14), k


def test_masked_statistics_ignore_padding():
    """A read's padding changes nothing: a batch of one short read padded with garbage equals the read alone."""
    cfg = CONFIGS["basic"]
    sd = synth.resnet_state_dict(cfg, 2)
    n1, n2 = ResNet(cfg).double().train(), ResNet(cfg).double().train()
    n1.load_state_dict(sd)
    n2.load_state_dict(sd)
    x = torch.randn(1, 4000, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    padded = torch.cat([x, torch.full((1, 900), 1e6, dtype=torch.float64)], 1)
    assert torch.allclose(n1(x), n2(padded, [4000]), rtol=1e-12, atol=1e-11)
    for (k, u), v in zip(n1.named_buffers(), n2.buffers()):
        assert torch.allclose(u.double(), v.double(), rtol=1e-12, atol=1e-14), k


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_initial_weights_are_the_modules(name):
    cfg = CONFIGS[name]
    want = initial_state(cfg, 5)
    got = resnet_default_init_state(cfg, 5)
    assert list(got) == list(want) == list(synth.resnet_state_dict(cfg, 0))
    for k in want:
        assert got[k].dtype == want[k].dtype and torch.equal(got[k], want[k]), k
    assert not torch.equal(got["conv_block.0.weight"], resnet_default_init_state(cfg, 6)["conv_block.0.weight"])
    state = torch.random.get_rng_state()
    resnet_default_init_state(cfg, 6)
    assert torch.equal(torch.random.get_rng_state(), state)          # the caller's RNG is left alone
