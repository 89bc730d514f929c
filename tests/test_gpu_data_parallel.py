"""GPU: data-parallel training (riser_b200/parallel.py) against the one-device trainers.

Every check runs in two layouts: "shared" puts two replicas on cuda:0 (the same split, reductions, events and host
threads, on one GPU) and "two" puts them on cuda:0 and cuda:1 (peer-to-peer loads over NVLink); "two" is skipped
when fewer than two GPUs are visible.  Run the whole file on a box with at least two B200s."""
import ctypes
import logging

import numpy as np
import pytest
import torch

from riser_b200 import _lib, synth
from riser_b200.config import AttrDict, CNN_SHIPPED
from riser_b200.parallel import DataParallelTrainer, split
from riser_b200.training import ConvNetTrainer, ResNetTrainer, fit, make_trainer

pytestmark = pytest.mark.gpu
P = _lib.ptr
LOG = logging.getLogger("test")
TWO = pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one box")
LAYOUTS = ["shared", pytest.param("two", marks=TWO)]
NOISE_ONLY = ("conv_block.0.bias",)      # exact gradient 0 (a training-mode BatchNorm follows): rounding only


@pytest.fixture(scope="module")
def dev():
    return _lib.require_device()


def _devices(layout):
    return [0, 0] if layout == "shared" else [0, 1]


def _dp(cfg, layout, state=None, seed=0):
    if layout == "two":
        return DataParallelTrainer(cfg, [0, 1], state=state, seed=seed)
    tr = DataParallelTrainer.__new__(DataParallelTrainer)
    tr._build(cfg, [0, 0], state, seed, None)
    return tr


def _batch(lens, ld, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.full((len(lens), ld), float("nan"))                 # padding never read
    for b, n in enumerate(lens):
        x[b, :n] = torch.randn(n, generator=g)
    return x


def _rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm()).item()


# ---------------------------------------------------------------- the reduction kernel
@pytest.mark.parametrize("layout", LAYOUTS)
def test_peer_reduce_is_the_device_order_sum(dev, layout):
    devices = _devices(layout)
    if layout == "two":
        _lib.check(_lib.lib().riser_peer_enable((ctypes.c_int * 2)(0, 1), 2), "riser_peer_enable")
    rng = np.random.default_rng(5)
    for n, lo, hi in [(1, 0, 1), (3, 0, 3), (5, 1, 5), (1027, 0, 1027), (1027, 3, 1026), (4096, 0, 4096),
                      (100003, 7, 99999), (8, 4, 4), (0, 0, 0)]:
        # magnitudes across 2^30 so that the order of the sums changes the result
        host = [(rng.standard_normal(max(n, 1)) * 2.0 ** rng.integers(-15, 15, max(n, 1))).astype(np.float32)
                for _ in devices]
        src = [torch.from_numpy(h).to(f"cuda:{d}") for h, d in zip(host, devices)]
        want = host[0].copy()
        for h in host[1:]:
            want = (want + h).astype(np.float32)
        ptrs = (ctypes.c_void_p * len(src))(*[t.data_ptr() for t in src])
        outs = []
        for d in sorted(set(devices)):
            with torch.cuda.device(d):
                dst = torch.full((max(n, 1),), 7.0, device=f"cuda:{d}")
                _lib.check(_lib.lib().riser_peer_reduce_f32(ptrs, len(src), P(dst), lo, hi, _lib.stream_ptr()),
                           "riser_peer_reduce_f32")
                outs.append(dst.cpu().numpy())
        for out in outs:
            assert np.array_equal(out[lo:hi].view(np.uint32), want[lo:hi].view(np.uint32)), (n, lo, hi)
            assert (out[:lo] == 7.0).all() and (out[hi:n] == 7.0).all()
        # unaligned sources take the scalar path, with the same bits
        if n > 8:
            ptrs1 = (ctypes.c_void_p * len(src))(*[t.data_ptr() + 4 for t in src])
            with torch.cuda.device(devices[0]):
                dst = torch.zeros(n, device=f"cuda:{devices[0]}")
                _lib.check(_lib.lib().riser_peer_reduce_f32(ptrs1, len(src), P(dst), 0, n - 1, _lib.stream_ptr()),
                           "riser_peer_reduce_f32")
                assert np.array_equal(dst.cpu().numpy()[:n - 1].view(np.uint32), want[1:].view(np.uint32))
    with pytest.raises(_lib.RiserError):
        _lib.check(_lib.lib().riser_peer_reduce_f32((ctypes.c_void_p * 9)(*[src[0].data_ptr()] * 9), 9,
                                                    P(src[0]), 0, 1, _lib.stream_ptr()), "nine sources")


@pytest.mark.parametrize("G", range(2, 9))
def test_peer_reduce_adds_the_sources_in_device_order(dev, G):
    """G sources on one GPU, with values for which the order of the fp32 sums shows: source 0 is 2^24 + 2k (the
    spacing of fp32 there is 2), the others are 1.  In device order every + 1 is a tie that rounds to even, so most
    of them are lost; summing the ones first keeps them.  Then random magnitudes across 2^40."""
    rng = np.random.default_rng(G)
    n = 4099
    big = (2.0 ** 24 + 2 * rng.integers(0, 1000, n)).astype(np.float32)
    host = [big] + [np.ones(n, np.float32) for _ in range(G - 1)]
    want = host[0].copy()
    for h in host[1:]:
        want = (want + h).astype(np.float32)
    rev = host[-1].copy()                            # the reverse order: the small ones first
    for h in host[-2::-1]:
        rev = (rev + h).astype(np.float32)
    assert np.array_equal(want, rev) == (G == 2)     # the order matters from G = 3 on
    # random magnitudes too
    host_r = [(rng.standard_normal(n) * 2.0 ** rng.integers(-20, 20, n)).astype(np.float32) for _ in range(G)]
    want_r = host_r[0].copy()
    for h in host_r[1:]:
        want_r = (want_r + h).astype(np.float32)
    for hs, w in ((host, want), (host_r, want_r)):
        src = [torch.from_numpy(h).to(dev) for h in hs]
        ptrs = (ctypes.c_void_p * G)(*[t.data_ptr() for t in src])
        for lo, hi in ((0, n), (3, n - 2)):
            dst = torch.zeros(n, device=dev)
            _lib.check(_lib.lib().riser_peer_reduce_f32(ptrs, G, P(dst), lo, hi, _lib.stream_ptr()),
                       "riser_peer_reduce_f32")
            assert np.array_equal(dst.cpu().numpy()[lo:hi].view(np.uint32), w[lo:hi].view(np.uint32)), (G, lo, hi)


def test_split_batch_norm_matches_the_one_call_path(dev):
    """G = 1 of the split BatchNorm is riser_bn_stats_cl / riser_bn_bwd_cl bit for bit; three slices of the batch give
    the whole batch's statistics and sums within float64 rounding."""
    lib = _lib.lib()
    g = torch.Generator().manual_seed(4)
    lens = [700, 1, 555, 699, 3, 700]
    B, L, C = len(lens), 700, 45
    y = (torch.randn(B, L, C, generator=g) * 3 + 1).to(dev)
    dout = torch.randn(B, L, C, generator=g).to(dev)
    gamma = (torch.rand(C, generator=g) + 0.5).to(dev)
    n = torch.tensor(lens, dtype=torch.int32, device=dev)
    ws = torch.empty(lib.riser_bn_workspace_bytes(C) // 4 + 4, device=dev)
    wsb = ws.numel() * 4
    s = _lib.stream_ptr()

    def one_call():
        mean, var = torch.empty(C, device=dev), torch.empty(C, device=dev)
        run = [torch.zeros(C, device=dev), torch.ones(C, device=dev), torch.zeros((), dtype=torch.int64, device=dev)]
        _lib.check(lib.riser_bn_stats_cl(P(y), P(n), B, L, C, P(mean), P(var), *[P(t) for t in run], 0.1, P(ws), wsb,
                                         s), "stats")
        out = [torch.empty(C, device=dev), torch.empty(C, device=dev), torch.empty_like(y)]
        _lib.check(lib.riser_bn_bwd_cl(P(dout), None, P(y), P(n), B, L, C, P(mean), P(var), P(gamma), 1e-5,
                                       *[P(t) for t in out], None, P(ws), wsb, s), "bwd")
        return [mean, var] + run + out

    def split_calls(G):
        parts = [(torch.empty(lib.riser_bn_partial_bytes(C) // 8, dtype=torch.float64, device=dev),
                  torch.empty(lib.riser_bn_partial_bytes(C) // 8, dtype=torch.float64, device=dev)) for _ in range(G)]
        mean, var = torch.empty(C, device=dev), torch.empty(C, device=dev)
        run = [torch.zeros(C, device=dev), torch.ones(C, device=dev), torch.zeros((), dtype=torch.int64, device=dev)]
        cuts = split(B, G)
        for (lo, hi), (ps, _) in zip(cuts, parts):
            _lib.check(lib.riser_bn_stats_partial_cl(P(y[lo:hi]), P(n[lo:hi]), hi - lo, L, C, P(ps), P(ws), wsb, s),
                       "stats partial")
        sp = (ctypes.c_void_p * G)(*[p[0].data_ptr() for p in parts])
        _lib.check(lib.riser_bn_stats_finalize_cl(sp, G, C, P(mean), P(var), *[P(t) for t in run], 0.1, s), "fin")
        for (lo, hi), (_, pb) in zip(cuts, parts):
            _lib.check(lib.riser_bn_bwd_partial_cl(P(dout[lo:hi]), None, P(y[lo:hi]), P(n[lo:hi]), hi - lo, L, C,
                                                   P(mean), P(var), 1e-5, P(pb), P(ws), wsb, s), "bwd partial")
        bp = (ctypes.c_void_p * G)(*[p[1].data_ptr() for p in parts])
        dg, db, dx = torch.empty(C, device=dev), torch.empty(C, device=dev), torch.empty_like(y)
        for r, (lo, hi) in enumerate(cuts):
            g2, b2 = torch.empty(C, device=dev), torch.empty(C, device=dev)
            _lib.check(lib.riser_bn_bwd_finalize_cl(bp, G, int(r == 0), P(dout[lo:hi]), None, P(y[lo:hi]),
                                                    P(n[lo:hi]), hi - lo, L, C, P(mean), P(var), P(gamma), 1e-5,
                                                    P(g2), P(b2), P(dx[lo:hi]), None, P(ws), wsb, s), "bwd fin")
            if r == 0:
                dg, db = g2, b2
            else:
                assert (g2 == 0).all() and (b2 == 0).all()
        return [mean, var] + run + [dg, db, dx]

    want = one_call()
    for a, b in zip(split_calls(1), want):
        assert torch.equal(a, b)
    m = (torch.arange(L, device=dev)[None, :] < n[:, None].long())[..., None].expand(B, L, C)
    got = split_calls(3)
    for i, (a, b) in enumerate(zip(got, want)):
        if i == 4:
            assert int(a) == int(b) == 1
        elif i == 7:
            assert _rel(a[m], b[m]) < 1e-7
        else:
            assert _rel(a, b) < 1e-7, i


# ---------------------------------------------------------------- whole networks against the one-device trainer
CNN_CASES = {
    "shipped": (CNN_SHIPPED, [12048] * 4, [4096, 6001, 8615, 12048], 12048),
    "k5_fc": (synth.GENERIC_CNN_CONFIGS["k5_fc"], [1024] * 4, [64, 333, 1024, 1000], 1024),
}


def _compare_convnet(cfg, lens, ld, layout, seed=1):
    one = ConvNetTrainer(cfg, seed=3)
    dp = _dp(cfg, layout, state=one.state_dict())
    try:
        x = _batch(lens, ld, seed)
        labels = torch.tensor([b % int(cfg["n_classes"]) for b in range(len(lens))])
        lens_t = torch.tensor(lens, dtype=torch.int32)
        want = one.gradients(x, lens_t, labels)
        got = dp.gradients(x, lens_t, labels)
        torch.cuda.synchronize()
        s1 = one._bufs[(len(lens), ld)]
        for rep, (lo, hi) in zip(dp.replicas, split(len(lens), len(dp.replicas))):
            if hi > lo:
                s = rep.trainer._bufs[(hi - lo, ld)]
                assert torch.equal(s["loss"].cpu(), s1["loss"][lo:hi].cpu())
                assert torch.equal(s["logits"].cpu(), s1["logits"][lo:hi].cpu())
                assert torch.equal(s["dlogits"].cpu(), s1["dlogits"][lo:hi].cpu())
        errs = {k: _rel(got[k], want[k]) for k in want}
        worst = max(errs, key=errs.get)
        print(f"B {len(lens)}: worst relative gradient difference to the one-device step {errs[worst]:.1e} ({worst})")
        assert errs[worst] <= 1e-5, (worst, errs[worst])
        assert abs(float(dp.replicas[0].loss[0]) - float(s1["loss_mean"][0])) <= 1e-6 * abs(float(s1["loss_mean"][0]))
    finally:
        dp.close()


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("name", sorted(CNN_CASES))
@pytest.mark.parametrize("ragged", [False, True])
def test_convnet_gradients_match_one_device(dev, layout, name, ragged):
    cfg, equal, uneven, ld = CNN_CASES[name]
    _compare_convnet(cfg, uneven if ragged else equal, ld, layout)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("B", [3, 1])
def test_convnet_uneven_and_empty_slices(dev, layout, B):
    cfg, _, uneven, ld = CNN_CASES["k5_fc"]
    _compare_convnet(cfg, uneven[:B], ld, layout)


def _compare_resnet(cfg, lens, ld, layout, steps=True):
    cfg = {"model": "resnet", "resnet": dict(cfg)}
    one = ResNetTrainer(cfg, state=synth.resnet_state_dict(cfg["resnet"], 0))
    dp = _dp(cfg, layout, state=one.state_dict())
    try:
        x = _batch(lens, ld, 2)
        labels = torch.tensor([b % 2 for b in range(len(lens))])
        lens_t = torch.tensor(lens, dtype=torch.int32)
        want = one.gradients(x, lens_t, labels)
        got = dp.gradients(x, lens_t, labels)
        torch.cuda.synchronize()
        st = {k: _rel(dp.replicas[0].trainer.stats[k][i], one.stats[k][i]) for k in one.stats for i in (0, 1)
              if one.stats[k][i].norm() > 0}
        assert max(st.values()) <= 1e-7, max(st.values())
        for rep in dp.replicas[1:]:                   # every replica finalised the same statistics
            assert all(torch.equal(rep.trainer.stats[k][i].cpu(), dp.replicas[0].trainer.stats[k][i].cpu())
                       for k in one.stats for i in (0, 1))
        errs = {k: _rel(got[k], want[k]) for k in want if k not in NOISE_ONLY}
        worst = max(errs, key=errs.get)
        stem = want["conv_block.0.weight"].norm()
        noise = max(((got[k] - want[k]).norm() / stem).item() for k in NOISE_ONLY)
        print(f"B {len(lens)}: BN statistics {max(st.values()):.1e}, worst gradient {errs[worst]:.1e} ({worst}), "
              f"stem bias {noise:.1e} of the stem weight gradient")
        assert errs[worst] <= 1e-5, (worst, errs[worst])
        assert noise < 1e-4
        if steps:
            one.step(x, lens_t, labels)
            dp.step(x, lens_t, labels)
            a, b = dp.state_dict(), one.state_dict()
            for k in b:
                if k.endswith("num_batches_tracked"):
                    assert int(a[k]) == int(b[k]), k
                elif "running" in k:
                    assert _rel(a[k], b[k]) <= 1e-6, (k, _rel(a[k], b[k]))
    finally:
        dp.close()


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("name", sorted(synth.RESNET_CONFIGS))
@pytest.mark.parametrize("lens", [[12048] * 4, [12048, 5000, 8615, 4096, 12047], [12048, 4096, 7000], [9000]],
                         ids=["equal", "ragged", "B3", "B1"])
def test_resnet_matches_one_device(dev, layout, name, lens):
    _compare_resnet(synth.RESNET_CONFIGS[name], lens, 12048, layout)


def _one_row_length(tr):
    """The shortest read whose last BatchNorm sees exactly one row."""
    for L in range(1, 4096):
        n = torch.tensor([L])
        ok = True
        for k, st, pd in tr.chain_host:
            n = (n + 2 * pd) // 2 if k < 0 else torch.clamp((n + 2 * pd - k) // st + 1, min=0)
            ok &= int(n.min()) >= 1
        if ok and int(n) == 1:
            return L
    raise AssertionError("no such length")


@pytest.mark.parametrize("layout", LAYOUTS)
def test_single_value_rule_on_the_global_batch(dev, layout):
    cfg = synth.RESNET_CONFIGS["basic"]
    one = ResNetTrainer(cfg, seed=0)
    L = _one_row_length(one)
    x, lens, labels = _batch([L, L], L, 3), torch.tensor([L, L], dtype=torch.int32), torch.tensor([0, 1])
    with pytest.raises(ValueError):
        one.gradients(x[:1], lens[:1], labels[:1])              # one read alone: refused
    _compare_resnet(cfg, [L, L], L, layout, steps=False)      # one read per replica: accepted, the global batch


# ---------------------------------------------------------------- replicas, determinism, fit, refusals
def _five_steps(cfg, layout, state):
    dp = _dp(cfg, layout, state=state)
    try:
        for k in range(5):
            lens = [1024, 700, 1024, 512, 900] if k % 2 else [1024] * 4
            x = _batch(lens, 1024, 50 + k)
            dp.step(x, torch.tensor(lens, dtype=torch.int32), torch.tensor([b % 2 for b in range(len(lens))]))
        torch.cuda.synchronize()
        out = []
        for rep in dp.replicas:
            tr = rep.trainer
            opt = {f"{k}.{s}": v.cpu() for k, p in tr.params.items() for s, v in tr.optimizer.state[p].items()}
            bufs = {k: v.cpu() for k, v in getattr(tr, "buffers", {}).items()}
            out.append(dict(tr.state_dict(), **opt, **bufs))
        return out
    finally:
        dp.close()


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("model", ["cnn", "resnet"])
def test_replicas_stay_identical_and_runs_repeat(dev, layout, model):
    if model == "cnn":
        cfg = dict(synth.GENERIC_CNN_CONFIGS["k5_fc"], learning_rate=1e-3)
        state = ConvNetTrainer(cfg, seed=0).state_dict()
    else:
        cfg = {"model": "resnet", "resnet": dict(synth.RESNET_CONFIGS["basic"], learning_rate=1e-3)}
        state = None
    a, b = _five_steps(cfg, layout, state), _five_steps(cfg, layout, state)
    for run in (a, b):
        for other in run[1:]:
            assert list(other) == list(run[0])
            for k in run[0]:
                assert torch.equal(other[k], run[0][k]), k
    for k in a[0]:
        assert torch.equal(a[0][k], b[0][k]), k


@pytest.mark.parametrize("layout", LAYOUTS)
def test_fit_matches_one_device(dev, layout, tmp_path):
    """fit on the data-parallel trainer from a trained-like state at lr 1e-4: the epoch-0 losses of the one-device
    fit of the same global batches; checkpoints load in Model and in the reference module."""
    from riser_b200 import Model
    from oracle.resnet_module import ResNet as RefResNet
    cfg = {"model": "resnet", "resnet": dict(synth.RESNET_CONFIGS["basic"], learning_rate=1e-4)}
    state = synth.resnet_state_dict(cfg["resnet"], 0)
    g = torch.Generator().manual_seed(9)
    train = [(torch.randn(10, 4096, generator=g), torch.randint(0, 2, (10,), generator=g))]
    val = [(torch.randn(6, 4096, generator=g), torch.randint(0, 2, (6,), generator=g))]
    one = make_trainer(cfg, state=state)
    h1 = fit(one, train, val, 1, 4, str(tmp_path / "one"), seed=1)
    if layout == "two":
        dp = make_trainer(cfg, state=state, devices=[0, 1])
        assert isinstance(dp, DataParallelTrainer)
    else:
        dp = _dp(cfg, layout, state=state)
    try:
        h2 = fit(dp, train, val, 1, 4, str(tmp_path / "dp"), seed=1)
    finally:
        dp.close()
    for k in ("train_loss", "val_loss"):
        assert abs(h2[0][k] - h1[0][k]) <= 1e-4 * abs(h1[0][k]), (k, h1, h2)
    for suffix in ("_latest.pth", "_best.pth"):
        sd = torch.load(str(tmp_path / ("dp" + suffix)))
        Model(sd, AttrDict(cfg), LOG, "dp")
        RefResNet(cfg["resnet"]).load_state_dict(sd)


@TWO
def test_fit_on_devices_listed_out_of_order(dev, tmp_path):
    """devices=[1, 0] from a caller whose current device is 0: training and validation run on the replicas' own
    devices, and the epoch's losses match the one-device fit."""
    cfg = {"model": "cnn", "cnn": dict(synth.GENERIC_CNN_CONFIGS["k5_fc"]), "learning_rate": 1e-4}
    state = ConvNetTrainer(cfg, seed=0).state_dict()
    g = torch.Generator().manual_seed(11)
    train = [(torch.randn(10, 1024, generator=g), torch.randint(0, 2, (10,), generator=g))]
    val = [(torch.randn(6, 1024, generator=g), torch.randint(0, 2, (6,), generator=g))]
    torch.cuda.set_device(0)
    h1 = fit(make_trainer(cfg, state=state), train, val, 1, 4, str(tmp_path / "one"), seed=1)
    dp = make_trainer(cfg, state=state, devices=[1, 0])
    try:
        assert dp.device == torch.device("cuda", 1)
        h2 = fit(dp, train, val, 1, 4, str(tmp_path / "dp"), seed=1)
    finally:
        dp.close()
    assert torch.cuda.current_device() == 0
    for k in ("train_loss", "val_loss"):
        assert abs(h2[0][k] - h1[0][k]) <= 1e-4 * abs(h1[0][k]), (k, h1, h2)
    single = make_trainer(cfg, state=state, devices=[1])          # a one-device trainer on device 1, used from 0
    assert type(single) is ConvNetTrainer and single.device == torch.device("cuda", 1)
    x, y = val[0]
    lens = torch.full((6,), 1024, dtype=torch.int32)
    assert single.evaluate(x, lens, y) == ConvNetTrainer(cfg, state=state).evaluate(x, lens, y)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_empty_global_batch_is_refused(dev, layout):
    cfg = synth.GENERIC_CNN_CONFIGS["k5_fc"]
    dp = _dp(cfg, layout)
    try:
        with pytest.raises(ValueError):
            dp.step(torch.zeros(0, 1024), torch.zeros(0, dtype=torch.int32), torch.zeros(0, dtype=torch.int64))
    finally:
        dp.close()


def test_refusals_and_single_device(dev):
    cfg = synth.GENERIC_CNN_CONFIGS["k5_fc"]
    with pytest.raises(ValueError):
        DataParallelTrainer(cfg, [0, 0])
    with pytest.raises(ValueError):
        make_trainer(cfg, devices=[0, "cuda:0"])
    with pytest.raises(ValueError):
        DataParallelTrainer(cfg, list(range(9)))
    assert type(make_trainer(cfg, devices=[0])) is ConvNetTrainer
    assert type(make_trainer({"model": "resnet", "resnet": synth.RESNET_CONFIGS["basic"]}, devices=[0])) is ResNetTrainer
