"""Training the ResNet variant on the GPU (riser_b200.training.ResNetTrainer, csrc/train_resnet.cu, riser_conv1d_wgrad_ex
and the padded pool's backward in csrc/train.cu): the new ops one by one against float64, whole-network gradients and
Adam steps against float64 autograd of oracle/resnet_module, learning, fit() through make_trainer, the checkpoint round
trip into riser_b200.Model and the reference module, determinism and the refusals."""
import logging
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.resnet_module import ResNet as RefResNet
from riser_b200 import Model, _lib, synth
from riser_b200.config import AttrDict
from riser_b200.training import ResNetTrainer, fit, make_trainer

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")

# riser_conv1d_wgrad_ex: |gpu - f64| <= BETA * S, S = sum |dZ| |X| (riser_conv1d_wgrad_cl's bar)
BETA = 5e-5
TINY = 1e-30
# per tensor |gpu - f64| / |f64| (Frobenius norms): whole-network gradients, parameters after 10 Adam steps
GRAD_BAR = 1e-4
ADAM_BAR = 1e-3
CONFIGS = sorted(synth.RESNET_CONFIGS)
P = _lib.ptr


@pytest.fixture(scope="module")
def dev():
    return _lib.require_device()


def _call(name, *args):
    _lib.check(getattr(_lib.lib(), name)(*args), name)


def _poison(t, lens):
    """t [B, L, C] with NaN in every row at or beyond its read's length."""
    t = t.clone()
    for b, n in enumerate(lens):
        t[b, n:] = float("nan")
    return t


def _rows(lens, L, dev=None):
    return (torch.arange(L, device=dev)[None, :] < torch.as_tensor(lens, device=dev)[:, None])[:, :, None]


def _out_lens(lens, K, s, p):
    return [max(0, (n + 2 * p - K) // s + 1) for n in lens]


# ---------------------------------------------------------------- strided, padded wgrad and dgrad
CONV_CASES = [
    # (Cin, Cout, K, stride, pad, input lengths, Lin_pad)
    (1, 20, 19, 3, 5, [12048, 0, 1, 9, 4097, 12047], 12048),
    (20, 30, 3, 2, 1, [2008, 0, 1, 2, 1003, 1500], 2008),
    (20, 30, 1, 2, 0, [2008, 0, 1, 2, 1003, 1500], 2008),
    (30, 30, 3, 1, 1, [1004, 0, 1, 2, 777], 1004),
    (64, 16, 1, 1, 0, [502, 0, 1, 300], 502),
    (8, 16, 4, 2, 1, [301, 0, 1, 2, 3, 150], 301),
    (128, 256, 1, 2, 0, [251, 1, 125, 250], 251),
]


def _conv_case(case, dev):
    cin, cout, K, s, p, lens_in, Lin = CONV_CASES[case]
    Lout = (Lin + 2 * p - K) // s + 1
    lens_out = _out_lens(lens_in, K, s, p)
    g = torch.Generator().manual_seed(100 + case)
    B = len(lens_in)
    x = torch.relu(torch.randn(B, Lin, cin, generator=g))
    dz = torch.randn(B, Lout, cout, generator=g) * torch.exp(torch.randn(B, Lout, 1, generator=g))
    w = torch.randn(cout, cin, K, generator=g) / (cin * K) ** 0.5
    return (cin, cout, K, s, p, lens_in, lens_out, Lin, Lout,
            _poison(x, lens_in).to(dev), _poison(dz, lens_out).to(dev), w.to(dev))


def _conv_ref(x, dz, w, lens_in, lens_out, s, p):
    """float64 dW, db, dX of the masked convolution, and S = sum |dZ| |X| per weight."""
    xm = torch.nan_to_num(x.double()) * _rows(lens_in, x.shape[1], x.device)
    dzm = torch.nan_to_num(dz.double()) * _rows(lens_out, dz.shape[1], dz.device)
    W = w.double().requires_grad_(True)
    X = xm.permute(0, 2, 1).contiguous().requires_grad_(True)
    (F.conv1d(X, W, stride=s, padding=p) * dzm.permute(0, 2, 1)).sum().backward()
    Wa = torch.ones_like(W).requires_grad_(True)
    (F.conv1d(X.detach().abs(), Wa, stride=s, padding=p) * dzm.abs().permute(0, 2, 1)).sum().backward()
    dx = X.grad.permute(0, 2, 1) * _rows(lens_in, x.shape[1], x.device)
    return W.grad, dzm.sum((0, 1)), dx, Wa.grad, dzm.abs().sum((0, 1))


def _wgrad_ex(dz, x, lo, li, cin, cout, K, s, p, bias=True):
    B, Lout = dz.shape[:2]
    nb = _lib.lib().riser_conv1d_wgrad_ex_workspace_bytes(B, Lout, cin, cout, K)
    assert nb > 0
    ws = torch.empty(nb // 4 + 1, device=dz.device)
    dw = torch.empty(cout, cin, K, device=dz.device)
    db = torch.empty(cout, device=dz.device) if bias else None
    _call("riser_conv1d_wgrad_ex", P(dz), P(x), P(lo), P(li), B, Lout, x.shape[1], cin, cout, K, s, p, P(dw), P(db),
          P(ws), ws.numel() * 4, _lib.stream_ptr())
    return dw, db


@pytest.mark.parametrize("case", range(len(CONV_CASES)))
def test_wgrad_ex_against_float64(dev, case):
    cin, cout, K, s, p, lens_in, lens_out, Lin, Lout, x, dz, w = _conv_case(case, dev)
    li = torch.tensor(lens_in, dtype=torch.int32, device=dev)
    lo = torch.tensor(lens_out, dtype=torch.int32, device=dev)
    dw, db = _wgrad_ex(dz, x, lo, li, cin, cout, K, s, p)
    dw2, db2 = _wgrad_ex(dz, x, lo, li, cin, cout, K, s, p)
    assert torch.equal(dw, dw2) and torch.equal(db, db2), "two launches differ"
    dw3, _ = _wgrad_ex(dz, x, lo, li, cin, cout, K, s, p, bias=False)
    assert torch.equal(dw, dw3)
    rw, rb, _, sw, sb = _conv_ref(x, dz, w, lens_in, lens_out, s, p)
    ew = ((dw.double() - rw).abs() / (sw + TINY)).max().item()
    eb = ((db.double() - rb).abs() / (sb + TINY)).max().item()
    print(f"wgrad_ex Cin {cin} Cout {cout} K {K} stride {s} pad {p}: max |err| / S  dW {ew:.2e}  db {eb:.2e}")
    assert torch.isfinite(dw).all() and torch.isfinite(db).all()
    assert ((dw.double() - rw).abs() <= BETA * sw + TINY).all(), ew
    assert ((db.double() - rb).abs() <= BETA * sb + TINY).all(), eb
    if s == 1 and K % 2 == 1 and p == (K - 1) // 2:           # riser_conv1d_wgrad_cl's case: the same bits
        B = len(lens_in)
        nb = _lib.lib().riser_conv1d_wgrad_workspace_bytes(B, Lin, cin, cout, K)
        ws = torch.empty(nb // 4 + 1, device=dev)
        dwc, dbc = torch.empty_like(dw), torch.empty_like(db)
        _call("riser_conv1d_wgrad_cl", P(dz), P(x), P(li), B, Lin, cin, cout, K, P(dwc), P(dbc), P(ws), ws.numel() * 4,
              _lib.stream_ptr())
        assert torch.equal(dwc, dw) and torch.equal(dbc, db)


@pytest.mark.parametrize("case", range(len(CONV_CASES)))
@pytest.mark.parametrize("with_residual", [False, True])
def test_dgrad_against_float64(dev, case, with_residual):
    cin, cout, K, s, p, lens_in, lens_out, Lin, Lout, x, dz, w = _conv_case(case, dev)
    B = len(lens_in)
    li = torch.tensor(lens_in, dtype=torch.int32, device=dev)
    lo = torch.tensor(lens_out, dtype=torch.int32, device=dev)
    res = _poison(torch.randn(B, Lin, cin, generator=torch.Generator().manual_seed(case)), lens_in).to(dev) \
        if with_residual else None
    wd = w.permute(2, 0, 1).contiguous()                        # [K][Cout][Cin]
    outs = []
    for _ in range(2):
        dx = torch.full((B, Lin, cin), 7.0, device=dev)
        _call("riser_conv1d_dgrad_cl", P(dz), P(lo), P(wd), P(res), P(dx), P(li), B, Lout, Lin, cin, cout, K, s, p,
              _lib.stream_ptr())
        outs.append(dx)
    assert torch.equal(outs[0], outs[1]), "two launches differ"
    _, _, want, _, _ = _conv_ref(x, dz, w, lens_in, lens_out, s, p)
    if res is not None:
        want = want + torch.nan_to_num(res.double()) * _rows(lens_in, Lin, dev)
    got = outs[0].double()
    assert torch.isfinite(got).all()
    assert (got[~_rows(lens_in, Lin, dev).expand_as(got)] == 0).all()
    err = ((got - want).norm() / want.norm()).item()
    print(f"dgrad Cin {cin} Cout {cout} K {K} stride {s} pad {p} residual {with_residual}: relative error {err:.2e}")
    assert err < 1e-6


# ---------------------------------------------------------------- BatchNorm
def _bn_gpu(y, lens, gamma, beta, dout, res=None, res_p=None, relu=True, update=False, run=None):
    """stats (+ update), apply (+ residual, normalised when res_p), backward with the output's ReLU mask."""
    dev = y.device
    B, L, C = y.shape
    ln = torch.tensor(lens, dtype=torch.int32, device=dev)
    ws = torch.empty(_lib.lib().riser_bn_workspace_bytes(C) // 4 + 4, device=dev)
    mean, var = torch.empty(C, device=dev), torch.empty(C, device=dev)
    r = run if update else [None] * 3
    _call("riser_bn_stats_cl", P(y), P(ln), B, L, C, P(mean), P(var), *[P(t) for t in r], 0.1, P(ws), ws.numel() * 4,
          _lib.stream_ptr())
    rmv = [None] * 4
    if res_p is not None:
        rm, rv = torch.empty(C, device=dev), torch.empty(C, device=dev)
        _call("riser_bn_stats_cl", P(res), P(ln), B, L, C, P(rm), P(rv), None, None, None, 0.1, P(ws), ws.numel() * 4,
              _lib.stream_ptr())
        rmv = [rm, rv, res_p[0], res_p[1]]
    out = torch.full_like(y, 3.0)
    _call("riser_bn_apply_cl", P(y), P(ln), B, L, C, P(mean), P(var), P(gamma), P(beta), P(res), *[P(t) for t in rmv],
          1e-5, 1 if relu else 0, P(out), _lib.stream_ptr())
    dg, dbt, dx, dyo = torch.empty(C, device=dev), torch.empty(C, device=dev), torch.empty_like(y), torch.empty_like(y)
    _call("riser_bn_bwd_cl", P(dout), P(out if relu else None), P(y), P(ln), B, L, C, P(mean), P(var), P(gamma), 1e-5,
          P(dg), P(dbt), P(dx), P(dyo), P(ws), ws.numel() * 4, _lib.stream_ptr())
    return dict(mean=mean, var=var, out=out, dgamma=dg, dbeta=dbt, dx=dx, dy=dyo)


def _bn_ref(y, lens, gamma, beta, dout, relu=True):
    """float64 masked training-mode BN + ReLU and its autograd (torch's F.batch_norm at equal lengths)."""
    dev = y.device
    m = _rows(lens, y.shape[1], dev)
    n = float(sum(lens))
    Y = torch.nan_to_num(y.double()).requires_grad_(True)
    G, Bt = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    mean = torch.where(m, Y, 0).sum((0, 1)) / n
    var = (torch.where(m, Y - mean, 0) ** 2).sum((0, 1)) / n
    out = (Y - mean) / torch.sqrt(var + 1e-5) * G + Bt
    if relu:
        out = F.relu(out)
    (torch.where(m, out, 0) * torch.nan_to_num(dout.double())).sum().backward()
    return dict(mean=mean.detach(), var=var.detach(), out=out.detach(), dgamma=G.grad, dbeta=Bt.grad, dx=Y.grad), n


def _rel(a, b):
    return ((a.double() - b).norm() / b.norm()).item()


@pytest.mark.parametrize("ragged", [False, True])
def test_batch_norm_against_float64(dev, ragged):
    g = torch.Generator().manual_seed(21 + ragged)
    lens = [700, 0, 1, 2, 555, 699] if ragged else [700] * 4
    B, L, C = len(lens), 700, 45
    y = torch.randn(B, L, C, generator=g) * 3 + torch.randn(C, generator=g) * 2
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    dout = torch.randn(B, L, C, generator=g)
    yd, dd = _poison(y, lens).to(dev), _poison(dout, lens).to(dev)
    run = [torch.randn(C, generator=g).to(dev), (torch.rand(C, generator=g) + 0.5).to(dev),
           torch.tensor(7, dtype=torch.int64, device=dev)]
    run0 = [t.clone() for t in run]
    got = _bn_gpu(yd, lens, gamma.to(dev), beta.to(dev), dd, update=True, run=run)
    again = _bn_gpu(yd, lens, gamma.to(dev), beta.to(dev), dd)
    for k in got:
        assert torch.equal(got[k], again[k]), k                  # two launches, the same bits
    want, n = _bn_ref(yd, lens, gamma.to(dev), beta.to(dev), dd)
    m = _rows(lens, L, dev).expand(B, L, C)
    if not ragged:                                           # torch's own training-mode BatchNorm
        rm, rv = run0[0].double().clone(), run0[1].double().clone()
        tb = F.batch_norm(torch.nan_to_num(yd.double()).permute(0, 2, 1), rm, rv, gamma.double().to(dev),
                          beta.double().to(dev), training=True, momentum=0.1, eps=1e-5)
        assert torch.allclose(F.relu(tb).permute(0, 2, 1), want["out"], rtol=1e-12, atol=1e-12)
    else:
        rm = 0.9 * run0[0].double() + 0.1 * want["mean"]
        rv = 0.9 * run0[1].double() + 0.1 * want["var"] * n / (n - 1)
    errs = dict(mean=_rel(got["mean"], want["mean"]), var=_rel(got["var"], want["var"]),
                out=_rel(torch.where(m, got["out"], 0), torch.where(m, want["out"], 0)),
                dgamma=_rel(got["dgamma"], want["dgamma"]), dbeta=_rel(got["dbeta"], want["dbeta"]),
                dx=_rel(got["dx"], want["dx"]), running_mean=_rel(run[0], rm), running_var=_rel(run[1], rv))
    print(f"batch norm (ragged {ragged}) relative errors: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert max(errs.values()) < 1e-6, errs
    assert int(run[2]) == 8
    assert (got["dx"][~m] == 0).all() and (got["dy"][~m] == 0).all()
    assert torch.equal(got["dy"][m], torch.where(got["out"] > 0, dd, 0)[m])


def test_batch_norm_with_normalised_residual(dev):
    """BN2(y) + BN_sc(r) + ReLU in one apply pass, against float64."""
    g = torch.Generator().manual_seed(31)
    lens = [300, 1, 257]
    B, L, C = len(lens), 300, 30
    y, r = torch.randn(B, L, C, generator=g), torch.randn(B, L, C, generator=g) * 2 + 1
    gam, bet = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    gr, br = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    yd, rd = _poison(y, lens).to(dev), _poison(r, lens).to(dev)
    got = _bn_gpu(yd, lens, gam.to(dev), bet.to(dev), torch.zeros_like(yd), res=rd, res_p=(gr.to(dev), br.to(dev)))
    m = _rows(lens, L, dev)
    n = float(sum(lens))

    def bn(t, ga, be):
        t = torch.nan_to_num(t.double())
        mu = torch.where(m, t, 0).sum((0, 1)) / n
        v = (torch.where(m, t - mu, 0) ** 2).sum((0, 1)) / n
        return (t - mu) / torch.sqrt(v + 1e-5) * ga.double().to(dev) + be.double().to(dev)
    want = torch.where(m, F.relu(bn(yd, gam, bet) + bn(rd, gr, br)), 0)
    err = _rel(torch.where(m, got["out"], 0), want)
    print(f"BN + normalised residual + ReLU: relative error {err:.1e}")
    assert err < 1e-6


# ---------------------------------------------------------------- stem pool backward
@pytest.mark.parametrize("L", [18, 17])
def test_padded_pool_bwd_equals_torch(dev, L):
    g = torch.Generator().manual_seed(L)
    lens = [L, 0, 1, 2, 3, L - 1, 8]
    B, C = len(lens), 7
    z = torch.randint(-1, 3, (B, L, C), generator=g).float()      # many ties, zeros and negatives
    y = torch.relu(z)
    Lp = L // 2 + 1
    dp = torch.randn(B, Lp, C, generator=g)
    want = torch.zeros(B, L, C)
    for b, n in enumerate(lens):
        if n == 0:
            continue
        zb = z[b, :n].T.unsqueeze(0).clone().requires_grad_(True)
        out = F.max_pool1d(F.relu(zb), 2, 2, padding=1)
        out.backward(dp[b, :out.shape[2]].T.unsqueeze(0))
        want[b, :n] = zb.grad[0].T
    yd, dp_d = _poison(y, lens).to(dev), _poison(dp, [n // 2 + 1 if n else 0 for n in lens]).to(dev)
    lens_d = torch.tensor(lens, dtype=torch.int32, device=dev)
    outs = []
    for _ in range(2):
        got = torch.full((B, L, C), 7.0, device=dev)
        _call("riser_relu_pool_bwd_cl", P(yd), P(dp_d), P(lens_d), P(got), B, L, Lp, C, 2, _lib.stream_ptr())
        outs.append(got.cpu())
    assert torch.equal(outs[0], outs[1])
    assert torch.equal(outs[0], want)


# ---------------------------------------------------------------- whole network
def _batch(lens, ld, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.full((len(lens), ld), float("nan"))                 # padding never read
    for b, n in enumerate(lens):
        x[b, :n] = torch.randn(n, generator=g)
    return x


def _decisions(tr, s, B, dev):
    """The trainer's fp32 ReLU masks and stem max-pool choices, as oracle/resnet_module's ``force``."""
    n_all = s["lens"]
    force = {}
    st = tr.stem
    A0 = s["A"][st[0]]
    force["conv_block"] = (A0 > 0).permute(0, 2, 1)
    valid = _rows(n_all[0].long(), A0.shape[1], dev)
    hp = torch.where(valid, A0, float("-inf")).permute(0, 2, 1)
    pad = torch.full_like(hp[:, :, :1], float("-inf"))
    hp = torch.cat([pad, hp] + [pad] * (1 + hp.shape[2] % 2), 2)
    Lp = s["P"].shape[1]
    first, second = hp[:, :, 0::2][..., :Lp], hp[:, :, 1::2][..., :Lp]
    force["pool"] = (second > first) | torch.isnan(second)
    for p, convs, _, _ in tr.blocks:
        for k, cv in enumerate(convs[:-1]):
            force[f"{p}.blocks.{k}"] = (s["A"][cv[0]] > 0).permute(0, 2, 1)
        force[p] = (s["H"][p] > 0).permute(0, 2, 1)
    return force


def _ref_grads(cfg, state, x, lens, labels, dev, force=None):
    net = RefResNet(cfg).double().to(dev).train()
    net.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in state.items()})
    net.zero_grad()
    xd = torch.nan_to_num(x.double()).to(dev)
    F.cross_entropy(net(xd, lens, force), labels.to(dev)).backward()
    return {k: p.grad.detach().cpu() for k, p in net.named_parameters() if p.grad is not None}


# the stem convolution's bias feeds a training-mode BatchNorm, which removes it: its exact gradient is 0 and what any
# fp32 computation returns is rounding; it is checked against the stem weight gradient's norm instead
NOISE_ONLY = ("conv_block.0.bias",)


@pytest.mark.parametrize("name", CONFIGS)
@pytest.mark.parametrize("ragged", [False, True])
def test_network_gradients_against_float64(dev, name, ragged):
    cfg = synth.RESNET_CONFIGS[name]
    lens = [12048, 5000, 8615, 4096, 12047] if ragged else [12048] * 6
    ld = 12048
    tr = ResNetTrainer(cfg, seed=3)
    state = tr.state_dict()
    x = _batch(lens, ld, 1)
    labels = torch.tensor([b % 2 for b in range(len(lens))])
    lens_t = torch.tensor(lens, dtype=torch.int32)
    got = {k: v.cpu() for k, v in tr.gradients(x, lens_t, labels).items()}
    torch.cuda.synchronize()
    s = tr._bufs[(len(lens), ld)]
    force = _decisions(tr, s, len(lens), dev)
    want = _ref_grads(cfg, state, x, lens, labels, dev, force)
    plain = _ref_grads(cfg, state, x, lens, labels, dev)
    assert set(got) == set(want)
    errs = {k: ((got[k].double() - want[k]).norm() / want[k].norm()).item() for k in want if k not in NOISE_ONLY}
    free = {k: ((got[k].double() - plain[k]).norm() / plain[k].norm()).item() for k in errs}
    worst = max(errs, key=errs.get)
    print(f"{name} (ragged {ragged}): worst relative gradient error {errs[worst]:.2e} ({worst}); with float64's own "
          f"ReLU / pool decisions {max(free.values()):.2e}")
    print("  " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    for k in NOISE_ONLY:
        ratio = (got[k].norm() / want["conv_block.0.weight"].norm()).item()
        print(f"  {k}: |gpu| {got[k].norm().item():.2e} (float64 {want[k].norm().item():.2e}), "
              f"{ratio:.1e} of the stem weight gradient")
        assert ratio < 1e-4
    assert errs[worst] <= GRAD_BAR, (worst, errs[worst])
    # gradients() used the batch statistics and left the running ones alone
    assert all(torch.equal(tr.state_dict()[k], state[k]) for k in state)


@pytest.mark.parametrize("name", CONFIGS)
def test_adam_steps_against_float64(dev, name):
    """Ten Adam steps from a trained-like state (synth.resnet_state_dict: BatchNorm away from its zero-bias init) at
    lr 1e-4.  From torch's default init, or at lr 1e-3, the trajectory itself amplifies rounding: torch's own fp32
    autograd then ends 4.9e-3 to 2.5e-1 away from float64 (measured on a B200; DESIGN.md, "Training the ResNet").
    Measured here (B200): worst parameter 3.4e-6 (basic), 7.1e-5 (bottleneck); torch fp32 4.0e-6, 1.8e-4."""
    cfg = dict(synth.RESNET_CONFIGS[name], learning_rate=1e-4)
    tr = ResNetTrainer(cfg, state=synth.resnet_state_dict(cfg, 0))
    start = tr.state_dict()
    net = RefResNet(cfg).double().to(dev).train()
    net.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in start.items()})
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)             # skips the parameters that get no gradient
    B, ld = 4, 4096
    stem_bias = []                  # (gpu, float64) stem conv bias at every step's forward
    for step in range(10):
        stem_bias.append((tr.params["conv_block.0.bias"].detach().double().cpu(),
                          net.conv_block[0].bias.detach().cpu().clone()))
        x = _batch([ld] * B, ld, 100 + step)
        labels = torch.tensor([(b + step) % 2 for b in range(B)])
        tr.step(x.to(dev), torch.full((B,), ld, dtype=torch.int32, device=dev), labels.to(dev))
        opt.zero_grad()
        F.cross_entropy(net(x.double().to(dev)), labels.to(dev)).backward()
        opt.step()
    got = tr.state_dict()
    ref = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    assert list(got) == list(ref)
    # The stem bias's exact gradient is 0 (a training-mode BatchNorm follows), so Adam moves it by rounding noise; the
    # stem BN's batch mean follows that bias exactly and its running mean records it.  Remove the bias's share from the
    # running mean: sum over steps k of momentum (1 - momentum)^(9 - k) (bias_gpu_k - bias_f64_k).
    share = sum(0.1 * 0.9 ** (9 - k) * (g - r) for k, (g, r) in enumerate(stem_bias))
    got = dict(got, **{"conv_block.1.running_mean": got["conv_block.1.running_mean"].double() - share})
    errs = {k: ((got[k].double() - ref[k]).norm() / ref[k].norm()).item() for k in ref
            if got[k].is_floating_point() and k not in tr.frozen and k not in NOISE_ONLY}
    worst = max(errs, key=errs.get)
    params = [k for k in errs if k in tr.params]
    print(f"{name}, 10 Adam steps: worst relative error {errs[worst]:.2e} ({worst}); parameters "
          f"{max(errs[k] for k in params):.2e}, running statistics {max(errs[k] for k in errs if k not in params):.2e}")
    assert errs[worst] <= ADAM_BAR
    for k in got:
        if k.endswith("num_batches_tracked"):
            assert got[k].dtype == torch.int64 and int(got[k]) == int(start[k]) + (0 if k in tr.frozen else 10), k
        if k in tr.frozen:
            assert torch.equal(got[k], start[k]), k                 # unused shortcut tensors: bitwise unchanged


def _two_class(seed, n, length):
    from oracle import preprocess_oracle as pp
    bodies = synth.body_batch(seed, n, length)
    x = torch.tensor(np.stack([np.asarray(pp.mad_normalise(b), dtype=np.float32) for b in bodies]))
    return x, torch.tensor([r & 1 for r in range(n)])


@pytest.mark.parametrize("name", CONFIGS)
def test_loss_falls_on_two_class_data(dev, name):
    tr = ResNetTrainer(dict(synth.RESNET_CONFIGS[name], learning_rate=2e-3), seed=1)
    x, y = _two_class(4, 64, 2048)
    x, y = x.to(dev), y.to(dev)
    lens = torch.full((16,), 2048, dtype=torch.int32, device=dev)
    losses = []
    for step in range(40):
        k = (step * 16) % 64
        losses.append(float(tr.step(x[k:k + 16], lens, y[k:k + 16])))
    print(f"{name}: loss over 40 steps: first 5 {np.mean(losses[:5]):.4f}, last 5 {np.mean(losses[-5:]):.4f}")
    assert np.mean(losses[-5:]) < 0.8 * np.mean(losses[:5])


def test_fit_end_to_end_through_make_trainer(dev, tmp_path):
    cfg = AttrDict({"model": "resnet", "resnet": dict(synth.RESNET_CONFIGS["basic"]), "learning_rate": 2e-3})
    (x2, y2), (x3, y3), (xv, yv) = _two_class(1, 16, 2048), _two_class(2, 8, 3072), _two_class(3, 8, 2048)
    tr = make_trainer(cfg, seed=0)
    assert isinstance(tr, ResNetTrainer)
    prefix = str(tmp_path / "run")
    hist = fit(tr, [(x2, y2), (x3, y3)], [(xv, yv)], epochs=2, batch_size=8, out_prefix=prefix, seed=7, logger=LOG)
    assert len(hist) == 2 and all(np.isfinite(h["val_loss"]) for h in hist)
    for suffix in ("_latest.pth", "_best.pth"):
        sd = torch.load(prefix + suffix)
        assert list(sd) == list(synth.resnet_state_dict(cfg.resnet, 0))
        RefResNet(cfg.resnet).load_state_dict(sd)
    best = ResNetTrainer(cfg, state=torch.load(prefix + "_best.pth"))
    loss, _ = best.evaluate(xv, torch.full((8,), 2048, dtype=torch.int32), yv)
    assert abs(loss - min(h["val_loss"] for h in hist)) < 1e-5


@pytest.mark.parametrize("name", CONFIGS)
def test_checkpoint_round_trip(dev, name):
    cfg = AttrDict({"model": "resnet", "resnet": dict(synth.RESNET_CONFIGS[name]), "learning_rate": 1e-3})
    tr = ResNetTrainer(cfg, seed=2)
    for step in range(3):
        x = _batch([4096] * 8, 4096, 50 + step)
        tr.step(x, torch.full((8,), 4096, dtype=torch.int32), torch.tensor([b % 2 for b in range(8)]))
    sd = tr.state_dict()
    ref = synth.resnet_state_dict(cfg.resnet, 0)
    assert list(sd) == list(ref) and all(sd[k].dtype == ref[k].dtype for k in sd)
    net = RefResNet(cfg.resnet).eval()
    net.load_state_dict(sd)                                       # strict
    model = Model(sd, cfg, LOG, "mRNA")
    assert type(model).__name__ == "ResNetModel"
    lens = [12048, 4096, 9001, 5000]
    x = _batch(lens, 12048, 9)
    probs = model.classify_batch(x.to(dev), torch.tensor(lens, dtype=torch.int32, device=dev), max_len=12048).cpu()
    with torch.no_grad():
        logits = torch.cat([net(x[b:b + 1, :n]) for b, n in enumerate(lens)])
    err = (probs - F.softmax(logits, 1)).abs().max().item()
    print(f"{name} round trip: max |dp| {err:.2e}")
    assert err < 2e-4
    labels = torch.tensor([0, 1, 1, 0])
    want = F.cross_entropy(logits, labels).item()
    # evaluate() on equal-length reads (fit's use) against the eval-mode oracle
    xe = x[:, :4096].contiguous()
    loss, _ = tr.evaluate(xe, torch.full((4,), 4096, dtype=torch.int32), labels)
    with torch.no_grad():
        want_e = F.cross_entropy(net(xe), labels).item()
    print(f"{name} evaluate: loss {loss:.6f}, oracle {want_e:.6f} (ragged oracle {want:.6f})")
    assert abs(loss - want_e) <= 1e-4 * max(1.0, abs(want_e))


def test_steps_are_deterministic(dev):
    cfg = synth.RESNET_CONFIGS["bottleneck"]
    state = ResNetTrainer(cfg, seed=4).state_dict()
    runs = []
    for _ in range(2):
        tr = ResNetTrainer(cfg, state=state)
        for step in range(3):
            lens = [4096, 3001, 4000, 2222]
            tr.step(_batch(lens, 4096, 60 + step), torch.tensor(lens, dtype=torch.int32), torch.tensor([0, 1, 0, 1]))
        runs.append(tr.state_dict())
    assert all(torch.equal(runs[0][k], runs[1][k]) for k in runs[0])


def test_refusals(dev):
    base = synth.RESNET_CONFIGS["basic"]
    with pytest.raises(NotImplementedError):
        ResNetTrainer(dict(base, n_classes=33))
    with pytest.raises(NotImplementedError):
        ResNetTrainer(dict(base, block="preact"))
    with pytest.raises(NotImplementedError):
        ResNetTrainer(dict(base, kernel=33))
    with pytest.raises(NotImplementedError):
        make_trainer({"model": "tcn"})
    assert isinstance(make_trainer({"model": "resnet", "resnet": dict(base)}), ResNetTrainer)
    tr = ResNetTrainer(base)
    x = torch.zeros(2, 64)
    with pytest.raises(ValueError):
        tr.step(x, torch.tensor([64, 0], dtype=torch.int32), torch.tensor([0, 1]))    # a zero-length read
    with pytest.raises(ValueError):
        tr.step(x[:1], torch.tensor([9], dtype=torch.int32), torch.tensor([0]))       # one value per BN channel
    with pytest.raises(ValueError):
        tr.step(x, torch.tensor([64, 64], dtype=torch.int32), torch.tensor([0, 2]))
