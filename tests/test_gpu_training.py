"""Training on the GPU (riser_b200/training.py, csrc/train.cu): the backward kernels op by op against float64, whole-network
gradients against float64 torch autograd of the reference architecture, Adam steps, the checkpoint round trip into
riser_b200.Model and the reference module, fit() end to end, and the refusals."""
import logging
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from riser_b200 import Model, _lib, synth
from riser_b200.config import AttrDict, CNN_SHIPPED
from oracle.convnet_module import ConvNet as RefConvNet
from riser_b200.training import ConvNetTrainer, fit, load_tensors

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")

# riser_conv1d_wgrad_cl: |gpu - f64| <= BETA * S + TINY, S = sum |dZ| |X|.  Measured on a B200, max |err| / S: 2.2e-5
# (Cin 1135 x Cout 1702, 160 rows), 1.4e-5 (Cin 67 x Cout 337, K 5), 7.3e-6 (Cin 1, K 3), 3.6e-6 (Cin 20 x Cout 30 over
# 30,120 rows); the float64 emulation of the format (tests/test_training_precision.py) reaches 3.5e-6 and one bf16 pass
# without the lo planes 1.6e-3
BETA = 5e-5
TINY = 1e-30
# whole-network gradients against float64 autograd that takes the GPU forward's own ReLU / max-pool decisions, and
# parameters after 10 Adam steps: per tensor, |gpu - f64| / |f64| (Frobenius norms)
GRAD_BAR = 1e-4
ADAM_BAR = 1e-3


@pytest.fixture(scope="module")
def dev():
    return _lib.require_device()


def _call(name, *args):
    _lib.check(getattr(_lib.lib(), name)(*args), name)


P = _lib.ptr


# ---------------------------------------------------------------- wgrad
def _wgrad_ref(dz, x, lens, K):
    """float64 dW [Cout][Cin][K], db, and S for the masked, shifted GEMM."""
    B, L, cout = dz.shape
    cin = x.shape[2]
    mask = (torch.arange(L, device=dz.device)[None, :] < lens[:, None].long()).double()[:, :, None]
    dzm = torch.nan_to_num(dz.double()) * mask
    xm = torch.nan_to_num(x.double()) * mask
    pad = (K - 1) // 2
    dw = torch.empty(cout, cin, K, dtype=torch.float64, device=dz.device)
    s = torch.empty_like(dw)
    a, aa = dzm.reshape(-1, cout), dzm.abs().reshape(-1, cout)
    for j in range(K):
        sh = j - pad
        xs = torch.zeros_like(xm)
        if sh >= 0:
            xs[:, :L - sh] = xm[:, sh:]
        else:
            xs[:, -sh:] = xm[:, :L + sh]
        xs = xs.reshape(-1, cin)
        dw[:, :, j] = a.T @ xs
        s[:, :, j] = aa.T @ xs.abs()
    return dw, dzm.sum(dim=(0, 1)), s, aa.sum(0)


def _wgrad_gpu(dz, x, lens, K):
    B, L, cout = dz.shape
    cin = x.shape[2]
    nb = _lib.lib().riser_conv1d_wgrad_workspace_bytes(B, L, cin, cout, K)
    assert nb > 0
    ws = torch.empty(nb // 4 + 1, device=dz.device)
    dw = torch.empty(cout, cin, K, device=dz.device)
    db = torch.empty(cout, device=dz.device)
    _call("riser_conv1d_wgrad_cl", P(dz), P(x), P(lens), B, L, cin, cout, K, P(dw), P(db), P(ws), ws.numel() * 4,
          _lib.stream_ptr())
    return dw, db


WGRAD_CASES = [
    # (Cin, Cout, K, lens, L_pad)
    (1, 20, 3, [0, 1, 7, 300, 299], 304),
    (20, 30, 3, [6024, 0, 6023, 1, 4097], 6024),
    (20, 30, 1, [33, 0, 17], 40),
    (20, 30, 5, [501, 64, 3], 512),
    (67, 337, 5, [187, 0, 95, 1], 188),
    (67, 20, 3, [1000, 999], 1000),
    (1135, 1702, 3, [5, 4, 5, 1, 0, 5, 3, 5] * 4, 5),
    (1135, 30, 1, [11, 6, 9], 12),
    (20, 1702, 3, [9, 2, 9], 9),
    (20, 30, 3, None, 6024),          # about 2**22 rows: 697 full reads of 6,024
]


@pytest.mark.parametrize("case", range(len(WGRAD_CASES)))
def test_wgrad_against_float64(dev, case):
    cin, cout, K, lens, L = WGRAD_CASES[case]
    if lens is None:
        lens = [L] * 697
    g = torch.Generator(device="cpu").manual_seed(case)
    B = len(lens)
    lens_t = torch.tensor(lens, dtype=torch.int32)
    dz = torch.randn(B, L, cout, generator=g) * torch.exp(torch.randn(B, L, 1, generator=g) * 2)
    x = torch.relu(torch.randn(B, L, cin, generator=g))
    pad_rows = torch.arange(L)[None, :] >= lens_t[:, None].long()
    dz[pad_rows] = float("nan")                     # rows at or beyond len must never be read
    x[pad_rows] = float("nan")
    dz, x, lens_d = dz.to(dev), x.to(dev), lens_t.to(dev)
    dw, db = _wgrad_gpu(dz, x, lens_d, K)
    dw2, db2 = _wgrad_gpu(dz, x, lens_d, K)
    assert torch.equal(dw, dw2) and torch.equal(db, db2), "two launches differ"
    rw, rb, s, sb = _wgrad_ref(dz, x, lens_d, K)
    ew = ((dw.double() - rw).abs() / (s + TINY)).max().item()
    eb = ((db.double() - rb).abs() / (sb + TINY)).max().item()
    print(f"wgrad Cin {cin} Cout {cout} K {K} rows {B * L}: max |err| / S  dW {ew:.2e}  db {eb:.2e}")
    assert torch.isfinite(dw).all() and torch.isfinite(db).all()
    assert ((dw.double() - rw).abs() <= BETA * s + TINY).all(), ew
    assert ((db.double() - rb).abs() <= BETA * sb + TINY).all(), eb


# ---------------------------------------------------------------- ReLU + pool backward
@pytest.mark.parametrize("pool", [1, 0])
def test_relu_pool_bwd_equals_torch(dev, pool):
    g = torch.Generator().manual_seed(5 + pool)
    lens = [9, 0, 1, 8, 17, 16]
    B, L, C = len(lens), 18, 7
    z = torch.randint(-1, 3, (B, L, C), generator=g).float()      # many equal pairs, zeros and negatives
    y = torch.relu(z)
    Lp = L // 2 if pool else L
    dp = torch.randn(B, Lp, C, generator=g)
    want = torch.zeros(B, L, C)
    for b, n in enumerate(lens):
        if n == 0 or (pool and n < 2):
            continue
        zb = z[b, :n].T.unsqueeze(0).clone().requires_grad_(True)       # [1, C, n] as the reference runs it
        out = F.relu(zb)
        if pool:
            out = F.max_pool1d(out, 2, 2)
        out.backward(dp[b, :out.shape[2]].T.unsqueeze(0))
        want[b, :n] = zb.grad[0].T
    yd = y.clone()
    for b, n in enumerate(lens):
        yd[b, n:] = float("nan")
    got = torch.full((B, L, C), 7.0, device=dev)
    yd, dp_d, lens_d = yd.to(dev), dp.to(dev), torch.tensor(lens, dtype=torch.int32).to(dev)
    _call("riser_relu_pool_bwd_cl", P(yd), P(dp_d), P(lens_d), P(got), B, L, Lp, C, pool, _lib.stream_ptr())
    assert torch.equal(got.cpu(), want)


# ---------------------------------------------------------------- head
def test_head_against_float64(dev):
    g = torch.Generator().manual_seed(11)
    lens = [5, 1, 3, 5, 2]
    B, L, C, nc = len(lens), 5, 1702, 3
    h = torch.relu(torch.randn(B, L, C, generator=g))
    w = torch.randn(nc, C, generator=g) * 0.05
    bias = torch.randn(nc, generator=g)
    labels = torch.tensor([0, 2, 1, 1, 0])
    hd = h.clone()
    for b, n in enumerate(lens):
        hd[b, n:] = float("nan")
    out = {k: torch.empty(*s, device=dev) for k, s in
           dict(loss=(B,), mean=(1,), logits=(B, nc), dlog=(B, nc), feat=(B, C), dw=(nc, C), db=(nc,), dh=(B, L, C)).items()}
    ins = [hd.to(dev), torch.tensor(lens, dtype=torch.int32).to(dev), w.to(dev), bias.to(dev), labels.to(dev)]
    _call("riser_gap_linear_ce_bwd", *[P(t) for t in ins], B, L, C, nc, P(out["loss"]), P(out["mean"]), P(out["logits"]),
          P(out["dlog"]), P(out["feat"]), P(out["dw"]), P(out["db"]), P(out["dh"]), _lib.stream_ptr())
    h64 = h.double().requires_grad_(True)
    w64, b64 = w.double().requires_grad_(True), bias.double().requires_grad_(True)
    feat = torch.stack([h64[b, :n].mean(0) for b, n in enumerate(lens)])
    logits = feat @ w64.T + b64
    per = F.cross_entropy(logits, labels, reduction="none")
    loss = per.mean()
    loss.backward()

    def rel(a, b):
        return ((a.cpu().double() - b.detach()).norm() / b.detach().norm()).item()

    errs = dict(loss=rel(out["mean"][0], loss), per=rel(out["loss"], per), dw=rel(out["dw"], w64.grad),
                db=rel(out["db"], b64.grad), dh=rel(out["dh"], h64.grad), logits=rel(out["logits"], logits))
    print("head relative errors:", {k: f"{v:.1e}" for k, v in errs.items()})
    assert max(errs.values()) <= 1e-6, errs


# ---------------------------------------------------------------- whole network
def _batch(lens, ld, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.full((len(lens), ld), float("nan"))                 # padding never read
    for b, n in enumerate(lens):
        x[b, :n] = torch.randn(n, generator=g)
    return x


def _ref_grads(cfg, state, x, lens, labels, dev, dtype=torch.float64):
    """torch autograd of the reference architecture (float64, or fp32 without TF32), one read at a time at its own
    length, mean loss."""
    net = RefConvNet(cfg).to(dtype).to(dev)
    net.load_state_dict({k: v.to(dtype) for k, v in state.items()})
    net.zero_grad()
    total = 0.0
    for b, n in enumerate(lens):
        xb = x[b:b + 1, :n].to(dtype).to(dev)
        loss = F.cross_entropy(net(xb).reshape(1, -1), labels[b:b + 1].to(dev)) / len(lens)
        loss.backward()
        total += loss.item()
    return {k: p.grad.detach().cpu() for k, p in net.named_parameters()}, total


def _masked_ref(cfg, state, x, lens, labels, bufs, dev):
    """float64 autograd of the reference architecture, one read at a time at its own length, mean loss -- with every
    ReLU mask and max-pool choice taken from the trainer's saved fp32 forward (``bufs``, the trainer's buffers of the
    batch's shape), so that a near-tie decided the other way in fp32 does not count as an error.  Returns the parameter
    gradients, the per-layer relative error of the GPU's dZ against the float64 one, and how many ReLU / pool decisions
    the float64 values alone would have taken the other way."""
    net = RefConvNet(cfg).double().to(dev)
    net.load_state_dict({k: v.double() for k, v in state.items()})
    net.zero_grad()
    depth = int(cfg["depth"])
    flips = {"relu": 0, "pool": 0}
    zs = []
    for b, n in enumerate(lens):
        h, ni = x[b:b + 1, :n].double().to(dev).unsqueeze(1), n
        for i, layer in enumerate(net.layers):
            for d in range(depth):
                z = layer[2 * d](h)
                z.retain_grad()
                zs.append((i, d, b, ni, z))
                m = bufs["Y"][i][d][b, :ni].T > 0
                flips["relu"] += int(((z[0] > 0) != m).sum())
                h = z * m
            k = ni // 2
            yg = bufs["Y"][i][depth - 1][b, :2 * k]
            second = ((yg[1::2] > yg[0::2]) | torch.isnan(yg[1::2])).T          # torch's rule on the GPU's values
            flips["pool"] += int(((h[0, :, 1:2 * k:2] > h[0, :, 0:2 * k:2]) != second).sum())
            idx = 2 * torch.arange(k, device=dev)[None, :] + second.long()
            h, ni = torch.gather(h[0], 1, idx)[None], k
        loss = F.cross_entropy(net.classifier(h).reshape(1, -1), labels[b:b + 1].to(dev)) / len(lens)
        loss.backward()
    num, den = {}, {}
    for i, d, b, ni, z in zs:
        ref = z.grad[0].T
        got = bufs["gY"][i][d][b, :ni].double()
        num[(i, d)] = num.get((i, d), 0.0) + float(((got - ref) ** 2).sum())
        den[(i, d)] = den.get((i, d), 0.0) + float((ref ** 2).sum())
    dz_err = {key: (num[key] / den[key]) ** 0.5 if den[key] > 0 else 0.0 for key in num}
    return {k: p.grad.detach().cpu() for k, p in net.named_parameters()}, dz_err, flips


NET_CASES = {
    "shipped": (CNN_SHIPPED, [4096, 6001, 8615, 12048], 12048),
    "deep_gap": (synth.GENERIC_CNN_CONFIGS["deep_gap"], [300, 517, 1024, 777], 1024),
    "k5_fc": (synth.GENERIC_CNN_CONFIGS["k5_fc"], [64, 333, 1024, 1000], 1024),
}


@pytest.mark.parametrize("name", sorted(NET_CASES))
def test_network_gradients_against_float64(dev, name):
    cfg, lens, ld = NET_CASES[name]
    tr = ConvNetTrainer(cfg, seed=3)
    state = tr.state_dict()
    x = _batch(lens, ld, 1)
    labels = torch.tensor([b % int(cfg["n_classes"]) for b in range(len(lens))])
    lens_t = torch.tensor(lens, dtype=torch.int32)
    got = {k: v.cpu() for k, v in tr.gradients(x, lens_t, labels).items()}
    torch.cuda.synchronize()
    want, dz_err, flips = _masked_ref(cfg, state, x, lens, labels, tr._bufs[(len(lens), ld)], dev)
    plain, _ = _ref_grads(cfg, state, x, lens, labels, dev)
    assert set(got) == set(want)

    def rel(a, b, k):
        return ((a[k].double() - b[k]).norm() / b[k].norm()).item()

    errs = {k: rel(got, want, k) for k in want}
    print(f"{name}: {flips['relu']} ReLU and {flips['pool']} max-pool decisions of the fp32 forward differ from float64's; "
          "relative gradient errors against float64 with the GPU's decisions / without: " +
          ", ".join(f"{k} {errs[k]:.1e} / {rel(got, plain, k):.1e}" for k in want))
    print(f"{name}: relative dZ error per conv: " + ", ".join(f"{i}.{d} {e:.1e}" for (i, d), e in sorted(dz_err.items())))
    worst = max(errs, key=errs.get)
    assert errs[worst] <= GRAD_BAR, (worst, errs[worst])
    # a ragged batch's gradient is the mean of the per-read gradients (the same ops; only the split of wgrad's row sums
    # differs)
    acc = {k: torch.zeros_like(v) for k, v in got.items()}
    for b, n in enumerate(lens):
        one = tr.gradients(x[b:b + 1, :n].contiguous(), lens_t[b:b + 1], labels[b:b + 1])
        for k in acc:
            acc[k] += one[k].cpu() / len(lens)
    ragged = {k: ((acc[k] - got[k]).norm() / got[k].norm()).item() for k in acc}
    print(f"{name}: ragged batch vs mean of per-read gradients, worst {max(ragged.values()):.1e}")
    for k in acc:
        assert ragged[k] <= 1e-5, (k, ragged[k])


def test_adam_steps_against_float64(dev):
    cfg = dict(synth.GENERIC_CNN_CONFIGS["k5_fc"], learning_rate=1e-3)
    tr = ConvNetTrainer(cfg, seed=0)
    net = RefConvNet(cfg).double().to(dev)
    net.load_state_dict({k: v.double() for k, v in tr.state_dict().items()})
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    B, ld = 8, 512
    for step in range(10):
        x = _batch([ld] * B, ld, 100 + step)
        labels = torch.tensor([(b + step) % 2 for b in range(B)])
        tr.step(x.to(dev), torch.full((B,), ld, dtype=torch.int32, device=dev), labels.to(dev))
        opt.zero_grad()
        F.cross_entropy(net(x.double().to(dev)), labels.to(dev)).backward()
        opt.step()
    got = tr.state_dict()
    errs = {k: ((got[k].double() - p.detach().cpu()).norm() / p.detach().cpu().norm()).item()
            for k, p in net.named_parameters()}
    worst = max(errs, key=errs.get)
    print(f"10 Adam steps: worst relative parameter error {errs[worst]:.2e} ({worst})")
    assert errs[worst] <= ADAM_BAR


def _two_class(seed, n, length):
    from oracle import preprocess_oracle as pp
    bodies = synth.body_batch(seed, n, length)
    x = torch.tensor(np.stack([np.asarray(pp.mad_normalise(b), dtype=np.float32) for b in bodies]))
    return x, torch.tensor([r & 1 for r in range(n)])


def test_loss_falls_on_two_class_data(dev):
    cfg = dict(synth.GENERIC_CNN_CONFIGS["k5_fc"], learning_rate=2e-3)
    tr = ConvNetTrainer(cfg, seed=1)
    x, y = _two_class(4, 64, 1024)
    x, y = x.to(dev), y.to(dev)
    lens = torch.full((16,), 1024, dtype=torch.int32, device=dev)
    losses = []
    for step in range(50):
        k = (step * 16) % 64
        losses.append(float(tr.step(x[k:k + 16], lens, y[k:k + 16])))
    print(f"loss over 50 steps: first 5 {np.mean(losses[:5]):.4f}, last 5 {np.mean(losses[-5:]):.4f}")
    assert np.mean(losses[-5:]) < 0.8 * np.mean(losses[:5])


def test_checkpoint_round_trip(dev):
    cfg = AttrDict({"model": "cnn", "cnn": dict(CNN_SHIPPED), "learning_rate": 1e-4})
    tr = ConvNetTrainer(cfg, seed=2)
    lens = [4096, 12048, 7000]
    x = _batch(lens, 12048, 9)
    tr.step(x, torch.tensor(lens, dtype=torch.int32), torch.tensor([0, 1, 1]))
    sd = tr.state_dict()
    model = Model(sd, cfg, LOG, "mRNA")
    assert model._generic is None                              # the dedicated kernels of csrc/convnet.cu
    xz = torch.nan_to_num(x, nan=0.0)
    probs = model.classify_batch(xz.to(dev), torch.tensor(lens, dtype=torch.int32, device=dev), max_len=12048).cpu()
    net = RefConvNet(cfg.cnn)
    net.load_state_dict(sd)
    with torch.no_grad():
        want = torch.cat([F.softmax(net(xz[b:b + 1, :n]), dim=1) for b, n in enumerate(lens)])
    err = (probs - want).abs().max().item()
    print(f"round trip: max |dp| {err:.2e}")
    assert err < 1e-3


def test_fit_end_to_end(dev, tmp_path):
    cfg = dict(synth.GENERIC_CNN_CONFIGS["k5_fc"], learning_rate=2e-3)
    (x2, y2), (x3, y3), (xv, yv) = _two_class(1, 24, 256), _two_class(2, 16, 384), _two_class(3, 16, 256)
    neg, pos = x2[y2 == 0], x2[y2 == 1]
    xa, ya = load_tensors(neg, pos)
    assert torch.equal(ya, torch.tensor([0] * len(neg) + [1] * len(pos)))
    runs = []
    for r in range(2):
        prefix = str(tmp_path / f"run{r}")
        hist = fit(ConvNetTrainer(cfg, seed=0), [(xa, ya), (x3, y3)], [(xv, yv)], epochs=3, batch_size=8,
                   out_prefix=prefix, seed=7, logger=LOG)
        assert os.path.exists(prefix + "_latest.pth") and os.path.exists(prefix + "_best.pth")
        runs.append((prefix, hist))
    (p0, h0), (p1, h1) = runs
    assert h0 == h1
    for suffix in ("_latest.pth", "_best.pth"):
        a, b = torch.load(p0 + suffix), torch.load(p1 + suffix)
        assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    lens = torch.full((16,), 256, dtype=torch.int32)
    best = ConvNetTrainer(cfg, state=torch.load(p0 + "_best.pth")).evaluate(xv, lens, yv)[0]
    latest = ConvNetTrainer(cfg, state=torch.load(p0 + "_latest.pth")).evaluate(xv, lens, yv)[0]
    assert best <= latest
    assert abs(best - min(h["val_loss"] for h in h0)) < 1e-6


def test_refusals(dev):
    cfg = synth.GENERIC_CNN_CONFIGS["k5_fc"]
    with pytest.raises(NotImplementedError):
        ConvNetTrainer(dict(cfg, kernels=[3, 4, 3, 5, 3]))
    with pytest.raises(NotImplementedError):
        ConvNetTrainer(dict(cfg, classifier="fc"))
    tr = ConvNetTrainer(cfg)
    x = torch.zeros(2, 64)
    with pytest.raises(ValueError):
        tr.step(x, torch.tensor([64, 16], dtype=torch.int32), torch.tensor([0, 1]))     # 5 pools need 32 samples
    with pytest.raises(ValueError):
        tr.step(x, torch.tensor([64, 64], dtype=torch.int32), torch.tensor([0, 2]))
    with pytest.raises(ValueError):
        tr.gradients(x, torch.tensor([64, 64], dtype=torch.int32), torch.tensor([-1, 0]))


def test_evaluate_leaves_gradients_and_plain_dict_config(dev):
    cfg = {"model": "cnn", "cnn": dict(synth.GENERIC_CNN_CONFIGS["k5_fc"]), "learning_rate": 1e-3}
    tr = ConvNetTrainer(cfg, seed=0)                                  # a plain dict with a 'cnn' section
    x = _batch([512, 300], 512, 3)
    lens, labels = torch.tensor([512, 300], dtype=torch.int32), torch.tensor([0, 1])
    g = tr.gradients(x, lens, labels)
    loss, correct = tr.evaluate(x[:, :300].contiguous(), torch.tensor([300, 300], dtype=torch.int32), torch.tensor([1, 1]))
    assert np.isfinite(loss) and 0 <= correct <= 2
    for k, p in tr.params.items():
        assert torch.equal(p.grad, g[k]), k
