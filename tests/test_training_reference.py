"""CPU: the reference ConvNet the training tests compare against (oracle/convnet_module.py) is pinned against the
reference's own outputs, and the trainer's initial weights (riser_b200.training.default_init_state) are the ones that
module -- built in riser/nets/cnn.py's construction order -- draws under the same seed."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import convnet_oracle, preprocess_oracle as pp
from oracle.convnet_module import ConvNet, initial_state
from riser_b200 import synth
from riser_b200.config import CNN_SHIPPED
from riser_b200.training import default_init_state

CONFIGS = dict(synth.GENERIC_CNN_CONFIGS, shipped=CNN_SHIPPED)


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_initial_weights_follow_the_reference_construction_order(name):
    want = initial_state(CONFIGS[name], 5)
    got = default_init_state(CONFIGS[name], 5)
    assert list(got) == list(want)
    for k in want:
        assert torch.equal(got[k], want[k]), k
    state = torch.random.get_rng_state()
    default_init_state(CONFIGS[name], 6)
    assert torch.equal(torch.random.get_rng_state(), state)          # the caller's RNG is left alone


@pytest.mark.parametrize("name", sorted(synth.GENERIC_CNN_CONFIGS))
def test_module_matches_reference_golden_probabilities(golden_dir, name):
    g = np.load(os.path.join(golden_dir, "convnet_generic.npz"))
    cfg = synth.GENERIC_CNN_CONFIGS[name]
    net = ConvNet(cfg)
    net.load_state_dict(synth.generic_cnn_state_dict(cfg, 0))
    bodies = synth.ragged_bodies(int(g["seed_reads"]), len(g["lengths"]), 700, 5000)
    with torch.no_grad():
        probs = np.stack([F.softmax(net(torch.from_numpy(np.asarray(pp.mad_normalise(b), dtype=np.float32))[None]), 1)[0]
                          .numpy() for b in bodies])
    assert np.abs(probs - g[f"probs_{name}"]).max() < 1e-5


def test_module_matches_shipped_oracle():
    net = ConvNet(CNN_SHIPPED)
    sd = synth.state_dict(0)
    net.load_state_dict(sd)
    x = torch.randn(2, 5000, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        assert torch.allclose(net(x), convnet_oracle.logits(sd, x), rtol=1e-5, atol=1e-5)
