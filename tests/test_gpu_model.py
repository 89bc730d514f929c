"""GPU parity of the network forward (csrc/convnet.cu through the C ABI) against the
oracle (torch CPU fp32 restatement of riser/nets/cnn.py + riser/model.py) and the
golden probabilities produced by the reference's own Model.classify.

Tolerances (north star): softmax probabilities within 1e-3 absolute; decisions identical
except where the reference probability lies within 1e-3 of the threshold."""
import logging
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import preprocess_oracle as pp
from oracle import convnet_oracle as net
from oracle import control_oracle as ctl
from riser_b200.config import AttrDict
from riser_b200 import Model, decide, synth, PREC_F16, PREC_F16_W2, PREC_F16_X3, PREC_F16_F8
from tests.golden import make_golden_params as P

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")
CFG = AttrDict({"cnn": {"n_layers": 12, "depth": 1, "channels": synth.CHANNELS, "kernels": [3] * 12,
                        "n_classes": 2, "classifier": "gap_fc"}})
# north-star bar: 1e-3 absolute.  X3 (the default) meets it with margin (observed max 1.5e-4,
# limited by the tensor cores' truncating fp32 accumulation); W2 / F16 are opt-in fast modes.
PROB_TOL = {PREC_F16_X3: 1e-3, PREC_F16_F8: 1e-3, PREC_F16_W2: 3e-3, PREC_F16: 5e-3}   # F16 = opt-in fast mode, outside the 1e-3 bar


def to_device_batch(normed, ld=None):
    n = np.array([len(x) for x in normed], dtype=np.int32)
    ld = ld or int((n.max() + 3) & ~3)
    x = torch.zeros(len(normed), ld, dtype=torch.float32)
    for b, v in enumerate(normed):
        x[b, :len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float64)).float()
    return x.cuda(), torch.from_numpy(n).cuda()


def oracle_layers(state, x):
    """Per-layer pooled activations [C, L_i] of one read (fp32)."""
    h = x.view(1, 1, -1)
    outs = []
    for i in range(12):
        h = F.max_pool1d(F.relu(F.conv1d(h, state[f"layers.{i}.0.weight"], state[f"layers.{i}.0.bias"],
                                         padding="same")), 2, 2)
        outs.append(h[0])
    return outs


# pytest numbers the tuple-valued cases by position ("precision11"); their ids are pinned so that a case keeps its
# id when the list in front of it changes
@pytest.mark.parametrize("fuse,precision", [(0, PREC_F16), (0, PREC_F16_W2), (0, PREC_F16_X3),
                                            (2, PREC_F16), (2, PREC_F16_W2), (2, PREC_F16_X3), (0, PREC_F16_F8), (2, PREC_F16_F8)] +
                         [pytest.param(f, p, id=f"{f}-precision{k}") for k, (f, p) in enumerate([
                                            (0, (PREC_F16_F8, 1)), (2, (PREC_F16_F8, 1)), (2, (PREC_F16_F8, 3)),
                                            (2, (PREC_F16_X3, "flat")), (0, (PREC_F16, "flat")),
                                            (2, (PREC_F16_F8, "nopair"))], 11)] +
                         [pytest.param(f, p, id=f"{f}-precision{k}") for k, (f, p) in enumerate([
                                            (2, (PREC_F16_F8, 6)),
                                            (2, (PREC_F16_F8, "nofuse23")), (2, (PREC_F16_X3, "nofuse23")),
                                            (2, (PREC_F16_X3, "nokc")), (2, (PREC_F16_F8, "nokc"))], 20)])
def test_every_layer_against_oracle(fuse, precision, monkeypatch):
    monkeypatch.setenv("RISER_FUSE_L0", str(fuse))
    if isinstance(precision, tuple) and precision[1] == "flat":     # without the even / odd plane layout
        precision = precision[0]
        monkeypatch.setenv("RISER_EO", "0")
    elif isinstance(precision, tuple) and precision[1] == "nopair":   # e4m3 layers on single CTAs (conv_tc_kernel<F8>)
        precision = precision[0]                                       # instead of CTA pairs (cta_group::2, the default)
        monkeypatch.setenv("RISER_PAIR", "0")
    elif isinstance(precision, tuple) and precision[1] == "nokc":      # layer 1's hi / lo terms as three plane passes
        precision = precision[0]                                        # (fused01_kernel<2>) instead of one K = 64 pass
        monkeypatch.setenv("RISER_KC", "0")
    elif isinstance(precision, tuple) and precision[1] == "nofuse23":  # layers 2 and 3 as two conv_eo_kernel launches
        precision = precision[0]
        monkeypatch.setenv("RISER_FUSE23", "0")
    elif isinstance(precision, tuple):                                # first layer that runs the e4m3 correction pass
        precision, f8_from = precision
        monkeypatch.setenv("RISER_F8_FROM", str(f8_from))
    rng = np.random.default_rng(0)
    lengths = [4096, 5001, 7108, 12048, 12047, 8615, 4097]
    normed = [pp.mad_normalise(synth.body(rng, n)) for n in lengths]
    state = synth.state_dict(0)
    model = Model(state, CFG, LOG, "mRNA", precision=precision)
    x, lens = to_device_batch(normed)
    feat = torch.zeros(len(lengths), 1702, device="cuda")
    probs = model.classify_batch(x, lens, max_len=12048, feat=feat)
    torch.cuda.synchronize()
    plan = model.plan(len(lengths), 12048)
    assert plan.fused_layer0 == bool(fuse)
    report = []
    for b, v in enumerate(normed):
        want = oracle_layers(state, torch.from_numpy(np.asarray(v, dtype=np.float64)).float())
        for i in range(2 if plan.fused_layer0 else 1, 13):
            if plan.layer_format(i) < 0:                           # computed inside the previous layer's launch
                continue                                           # (conv_eo2_kernel): checked through the layers after it
            act = plan.activation(i, 12)[b].float().cpu()          # decoded by the row format the plan reports
            w = want[i - 1].T                                  # [L_i, C]
            L = w.shape[0]
            err = (act[:L] - w).abs().max().item()
            scale = w.abs().max().item()
            tail = act[L:].abs().max().item() if act.shape[0] > L else 0.0
            report.append((b, i, L, err / scale, tail))
    tol = 5e-4 if precision in (PREC_F16_X3, PREC_F16_F8) else 1e-2
    bad = [r for r in report if r[3] > tol or r[4] != 0.0]
    assert not bad, "layer mismatches (read, layer, L, rel err, tail max): %s" % bad[:12]
    want_feat = net.features(state, torch.zeros(0)) if False else None
    ofeat = torch.stack([net.features(state, torch.from_numpy(np.asarray(v, dtype=np.float64)).float()[None])[0]
                         for v in normed])
    rel = ((feat.cpu() - ofeat).norm() / ofeat.norm()).item()
    assert rel < (1e-4 if precision == PREC_F16_X3 else 3e-4 if precision == PREC_F16_F8 else 2e-3), rel
    want_p = net.classify_ragged(state, normed)
    assert np.abs(probs.cpu().numpy() - want_p).max() < PROB_TOL[precision]


@pytest.mark.parametrize("precision", [PREC_F16, PREC_F16_W2, PREC_F16_X3, PREC_F16_F8])
def test_probs_against_reference_golden(golden_dir, precision):
    g = np.load(os.path.join(golden_dir, "convnet_probs.npz"))
    bodies = P.norm_inputs()
    normed = [pp.mad_normalise(x) for x in bodies]
    x, lens = to_device_batch(normed)
    worst = {}
    for target in g["targets"]:
        model = Model(synth.state_dict(synth.TARGET_SEEDS[str(target)]), CFG, LOG, str(target),
                      precision=precision)
        probs = model.classify_batch(x, lens, max_len=12048).cpu().numpy()
        want = g[f"probs_{target}"]
        d = np.abs(probs - want).max(axis=1)
        worst[str(target)] = (float(d.max()), float(d.mean()))
        assert d.max() < PROB_TOL[precision], (target, worst)
        # decisions identical except where the reference p is within 1e-3 of the threshold
        for thr in (0.9, 0.5, 0.99):
            on_ref, on_got = want[:, 1] > np.float32(thr), probs[:, 1] > np.float32(thr)
            near = np.abs(want[:, 1] - thr) <= 1e-3
            assert np.all((on_ref == on_got) | near)
    print("worst |dp| (max, mean):", worst)


def test_classify_drop_in_and_short_input():
    state = synth.state_dict(0)
    model = Model(state, CFG, LOG, "mRNA")
    assert model.target == "mRNA"
    rng = np.random.default_rng(4)
    y = pp.mad_normalise(synth.body(rng, 6000))
    p = model.classify(y)                       # float64 ndarray in, Tensor[2] out (model.py:22-28)
    p_off, p_on = p
    want = net.classify(state, y)
    assert abs(p_on.item() - want[1].item()) < 1e-3 and abs(p_off.item() + p_on.item() - 1) < 1e-6
    assert bool(p_on > 0.9) == bool(want[1] > 0.9) or abs(want[1].item() - 0.9) < 1e-3
    z = model.classify(np.zeros(5000, dtype=np.int64))      # MAD == 0 read: int64 zeros (preprocess.py:123)
    assert abs(z[1].item() - net.classify(state, np.zeros(5000, dtype=np.int64))[1].item()) < 1e-3
    with pytest.raises(RuntimeError):
        model.classify(y[:4095])
    with pytest.raises(RuntimeError):
        Model({k: v for k, v in state.items() if k != "classifier.2.bias"}, CFG, LOG, "x")


def test_fixed_batch_rna004_shapes():
    """BASELINE config 2 shapes: fixed length 8,615 (reference-faithful) and 16,000 (as named)."""
    state = synth.state_dict(0)
    model = Model(state, CFG, LOG, "mRNA")
    for L in (8615, 16000):
        X = synth.body_batch(7, 6, L)
        normed = [pp.mad_normalise(x) for x in X]
        x, lens = to_device_batch(normed)
        probs = model.classify_batch(x, lens, max_len=L).cpu().numpy()
        want = net.classify_ragged(state, normed)
        assert np.abs(probs - want).max() < 1e-3, (L, np.abs(probs - want).max())


def test_decide_kernel_matches_control_rule():
    rng = np.random.default_rng(8)
    B, M = 600, 3
    p_on = rng.random((M, B)).astype(np.float32)
    p_on[:, :50] = np.float32(0.9)                   # exactly at threshold: strict '>' fails
    p_on[:, 50:80] = np.nextafter(np.float32(0.9), np.float32(1))
    probs = np.stack([1 - p_on, p_on], axis=2).astype(np.float32)
    probs[0, 90:95] = np.nan
    lens = rng.integers(4096, 12049, size=B).astype(np.int32)
    lens[::7] = 12048
    lens[5::11] = 0
    for mode in ("enrich", "deplete"):
        for thr in (0.9, 0.3, 0.5):
            got = decide(torch.from_numpy(probs).cuda(), torch.from_numpy(lens).cuda(), thr, mode, 12048).cpu().numpy()
            for b in range(B):
                if lens[b] == 0:
                    assert got[b] == ctl.SKIPPED
                    continue
                on = [torch.tensor(probs[m, b, 1]) for m in range(M)]
                off = [torch.tensor(probs[m, b, 0]) for m in range(M)]
                assert got[b] == ctl.decide(on, off, int(lens[b]), 12048, thr, mode), (mode, thr, b)


@pytest.mark.parametrize("precision", [PREC_F16, PREC_F16_X3, PREC_F16_F8])
def test_plan_reuse_with_stale_activations_and_skipped_reads(precision):
    """Tiles that lie wholly beyond a read's valid length are skipped, so the activation
    buffers keep stale rows from earlier batches; results must not depend on them.  Batch 1
    fills every buffer with full-length reads, batch 2 reuses the plan with short reads and
    skipped (length 0) reads in other positions."""
    rng = np.random.default_rng(21)
    state = synth.state_dict(1)
    model = Model(state, CFG, LOG, "mtRNA", precision=precision)
    B = 10
    first = [pp.mad_normalise(synth.body(rng, 12048)) for _ in range(B)]
    x, lens = to_device_batch(first, ld=12048)
    p1 = model.classify_batch(x, lens, max_len=12048).cpu().numpy()
    assert np.abs(p1 - net.classify_ragged(state, first)).max() < PROB_TOL[precision]
    lengths = [4096, 0, 5000, 12048, 0, 4097, 9000, 0, 6001, 4500]
    second = [pp.mad_normalise(synth.body(rng, n)) if n else np.zeros(0) for n in lengths]
    x2 = torch.zeros(B, 12048)
    for b, v in enumerate(second):
        x2[b, :len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float64)).float()
    # poison the padding beyond each read's length: it must never be read as signal
    for b, n in enumerate(lengths):
        x2[b, n:] = 7.5
    lens2 = torch.tensor(lengths, dtype=torch.int32).cuda()
    p2 = model.classify_batch(x2.cuda(), lens2, max_len=12048).cpu().numpy()
    live = [b for b, n in enumerate(lengths) if n]
    want = net.classify_ragged(state, [second[b] for b in live])
    assert np.abs(p2[live] - want).max() < PROB_TOL[precision]
    assert np.isnan(p2[[b for b, n in enumerate(lengths) if not n]]).all()
    # and again with the long reads: buffers now hold the short batch's leftovers
    p3 = model.classify_batch(x, lens, max_len=12048).cpu().numpy()
    assert np.array_equal(p3, p1)


@pytest.mark.parametrize("max_len", [16000, 12048, 8615, 4099, 4096, 9999])
def test_random_ragged_batches_all_boundaries(max_len):
    """Random ragged lengths (and a few zeros) for several max_len values, default precision: work items of the
    fused layers 0+1 (255 pooled outputs) and of the even/odd layers straddle read boundaries at arbitrary offsets,
    Lp parities differ, and the shortest reads end long before the tiles do."""
    rng = np.random.default_rng(1000 + max_len)
    state = synth.state_dict(2)
    model = Model(state, CFG, LOG, "globin")
    B = 23
    lengths = [int(x) for x in rng.integers(4096, max_len + 1, size=B)]
    lengths[0], lengths[1], lengths[-1] = max_len, 4096, max_len
    lengths[5] = 0
    if max_len > 4097:
        lengths[7] = 4097
    normed = [pp.mad_normalise(synth.body(rng, n)) if n else np.zeros(0) for n in lengths]
    ld = (max_len + 3) & ~3
    x = torch.full((B, ld), 3.25)                      # poison beyond each read's length
    for b, v in enumerate(normed):
        x[b, :len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float64)).float()
    lens = torch.tensor(lengths, dtype=torch.int32).cuda()
    probs = model.classify_batch(x.cuda(), lens, max_len=max_len).cpu().numpy()
    live = [b for b, n in enumerate(lengths) if n]
    want = net.classify_ragged(state, [normed[b] for b in live])
    assert np.abs(probs[live] - want).max() < 1e-3, np.abs(probs[live] - want).max()
    assert np.isnan(probs[5]).all()


def test_full_size_batch_replication_invariance():
    """BASELINE config 2 at full size (4096 x 16,000): the batch is 37 distinct reads (ragged, one skipped)
    repeated to 4096 rows.  Every replica must give bit-identical probabilities whatever its row (tiles of
    different CTAs, different positions inside work items), and the first copies must match the oracle."""
    rng = np.random.default_rng(77)
    state = synth.state_dict(0)
    model = Model(state, CFG, LOG, "mRNA")
    B, L, K = 4096, 16000, 37
    lengths = [int(v) for v in rng.integers(4096, L + 1, size=K)]
    lengths[0], lengths[3], lengths[9] = L, 4096, 0
    normed = [pp.mad_normalise(synth.body(rng, n)) if n else np.zeros(0) for n in lengths]
    xk = torch.zeros(K, L)
    for b, v in enumerate(normed):
        xk[b, :len(v)] = torch.from_numpy(np.asarray(v, dtype=np.float64)).float()
    idx = torch.arange(B) % K
    x = xk[idx].cuda()
    lens = torch.tensor(lengths, dtype=torch.int32)[idx].cuda()
    probs = model.classify_batch(x, lens, max_len=L).cpu().numpy()
    first = probs[:K]
    live = [b for b in range(K) if lengths[b]]
    want = net.classify_ragged(state, [normed[b] for b in live])
    assert np.abs(first[live] - want).max() < 1e-3
    rep = probs.reshape(-1)[: (B // K) * K * 2].reshape(B // K, K, 2)
    assert np.array_equal(rep[:, live], np.broadcast_to(first[live], rep[:, live].shape))
    assert np.isnan(rep[:, 9]).all()
