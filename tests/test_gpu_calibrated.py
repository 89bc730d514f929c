"""GPU: the calibrated (float32 pA) input mode end to end -- riser_polya_end_f32 bit for bit against numpy's float32
evaluation of riser/preprocess.py:42-79 (oracle.polya_end, tests/calibrated_reference.py), SignalProcessor.trim_polyA /
get_polyA_end on float32, BatchedClassifier(signal_dtype=np.float32) against the oracle's serial loop with the
float32 normaliser, and SequencerControl driving a calibrated client."""
import logging

import numpy as np
import pytest
import torch

from oracle import control_oracle as ctl
from oracle import convnet_oracle as net
from oracle import preprocess_oracle as pp
from oracle import refshim
from tests import calibrated_reference as cref
from riser_b200 import (Kit, SignalProcessor, Model, BatchedClassifier, RaggedBatch, SequencerControl, synth, sim,
                        _lib)
from riser_b200.config import shipped_config

pytestmark = pytest.mark.gpu
LOG = logging.getLogger("test")
f32 = np.float32
RES, MAX_W = 500, 512


@pytest.fixture(scope="module")
def proc():
    return SignalProcessor(Kit.create_from_version("RNA002"))


def calibrate(sig, scale, offset):
    return ((sig.astype(f32) + f32(offset)) * f32(scale)).astype(f32)


def expected(x):
    """(start, end, stats [W, 4]) as numpy computes them for float32 x; the scan covers the first 512 windows."""
    x = x[:MAX_W * RES]
    st = cref.polya_window_stats(x).astype(f32)
    start = end = None
    for w, (med, mad, mean, rolling) in enumerate(st):
        change = (mean - rolling) / rolling * 100
        if not start and change > 20 and mad <= 20:
            start = w * RES
        if start and not end and mad > 20:
            end = w * RES
    assert end == pp.polya_end(x)
    return start, end, st


def check_against_numpy(ends, starts, stats, sigs):
    found = 0
    for b, x in enumerate(sigs):
        start, end, st = expected(x)
        assert ends[b] == (-1 if end is None else end), b
        assert starts[b] == (-1 if start is None else start), b
        got = stats[b, :len(st)]
        assert np.array_equal(got.view(np.uint32), st.view(np.uint32)), (b, np.argwhere(got != st)[:4])
        found += end is not None
    return found


def run_f32(proc, sigs):
    batch = RaggedBatch(sigs, torch.device("cuda"), dtype=np.float32)
    starts = torch.empty(batch.B, dtype=torch.int32, device="cuda")
    ends, stats = proc.polya_end_device(batch, return_stats=True, starts=starts)
    assert stats.dtype == torch.float32 and stats.shape[2] == 4
    return ends.cpu().numpy(), starts.cpu().numpy(), stats.cpu().numpy()


def prefixes(seed, n, rng):
    reads = synth.raw_reads(seed, n, min_body=2000, max_body=16000, frac_no_polya=0.1, frac_const=0.02)
    out = []
    for i, (_, s) in enumerate(reads):
        k = int(rng.integers(1, len(s) // RES + 1))
        cut = [k * RES, k * RES - 1, int(rng.integers(0, len(s) + 1)), len(s)][i % 4]
        out.append(s[:max(cut, 0)])
    return out


@pytest.mark.parametrize("cal", ["0.1759/3.2", "0.684/10", "1.3/-20", "random"])
def test_polya_f32_matches_numpy(proc, cal):
    """400 ragged prefixes per calibration (1,600 in all): ends, starts and every per-window statistic."""
    rng = np.random.default_rng(len(cal))
    raw = prefixes(21 + len(cal), 400, rng)
    if cal == "random":
        sigs = [calibrate(s, rng.uniform(0.5, 2.0), rng.uniform(-30, 30)) for s in raw]
    else:
        scale, offset = map(float, cal.split("/"))
        sigs = [calibrate(s, scale, offset) for s in raw]
    ends, starts, stats = run_f32(proc, sigs)
    found = check_against_numpy(ends, starts, stats, sigs)
    if cal == "0.1759/3.2":
        assert found < 10              # the MAD thresholds are ADC-sized: a pA window rarely exceeds 20
    else:
        assert found > 50
    print(f"[{cal}] {found} / {len(sigs)} poly(A) ends found")


def test_polya_f32_corner_cases(proc):
    rng = np.random.default_rng(5)
    sigs = []
    # tied middle ranks, constant windows, negative values
    sigs.append(np.round(rng.normal(-40, 3, 9000)).astype(f32))
    sigs.append(np.full(6000, -7.25, f32))
    sigs.append(np.concatenate([np.full(3000, 80.0, f32), np.full(3000, -0.0, f32), np.full(2000, 0.0, f32)]))
    t = np.round(rng.normal(60, 20, 8000)).astype(f32)
    t[::2] = 60.0
    sigs.append(t)
    # rolling mean near 0: signal centred on zero
    for s in synth.raw_reads(8, 6, min_body=6000, max_body=9000):
        a = s[1].astype(f32)
        sigs.append(calibrate(s[1], 0.684, -float(np.mean(a))))
    # lengths 500k, 500k - 1, fewer than 500 samples, more than 512 windows
    base = calibrate(synth.raw_reads(9, 1, min_body=15000, max_body=15000)[0][1], 0.684, 10)
    for n in (0, 1, 499, 500, 999, 1000, 1499, 1500, 4999, 5000):
        sigs.append(base[:n])
    long = calibrate(np.tile(synth.raw_reads(10, 1, min_body=16000, max_body=16000)[0][1], 20)[:260_123], 1.3, -20)
    sigs.append(long)
    # the mean change one float32 ulp either side of 20 (and exactly 20), built by hand: windows 0-2 at r, window
    # 3 at m (MAD 0), window 4 noisy (MAD > 20)
    for target in (np.nextafter(f32(20), f32(21)), f32(20), np.nextafter(f32(20), f32(19))):
        r, m = _mean_change_pair(target)
        x = np.concatenate([np.full(1500, r, f32), np.full(500, m, f32), rng.normal(m, 200, 1000).astype(f32)])
        _, end, st = expected(x)
        change = (st[3, 2] - st[3, 3]) / st[3, 3] * 100
        assert change == target and (end == 2000) == (target > 20)
        sigs.append(x)
    ends, starts, stats = run_f32(proc, sigs)
    check_against_numpy(ends, starts, stats, sigs)
    assert ends[-3] == 2000 and ends[-2] == -1 and ends[-1] == -1


def _mean_change_pair(target):
    """Constant levels r (rolling) and m (window) whose float32 mean change is exactly ``target``."""
    rs = np.nextafter(f32(100), f32(200)) + np.arange(-300, 300, dtype=f32) * np.spacing(f32(100))
    ms = np.nextafter(f32(120), f32(200)) + np.arange(-300, 300, dtype=f32) * np.spacing(f32(120))
    mean_r = np.array([np.mean(np.full(1000, v, f32)) for v in rs], dtype=f32)
    mean_m = np.array([np.mean(np.full(500, v, f32)) for v in ms], dtype=f32)
    ch = ((mean_m[None, :] - mean_r[:, None]) / mean_r[:, None] * f32(100)).astype(f32)
    i, j = np.argwhere(ch == target)[0]
    return rs[i], ms[j]


def test_polya_f32_odd_phases(proc):
    """Reads starting at every 4-byte phase of a 16-byte line (scalar loads) give what aligned reads give."""
    rng = np.random.default_rng(6)
    sigs = [calibrate(s, 0.684, 10) for s in prefixes(31, 64, rng)]
    offs, pos = [], 0
    for b, s in enumerate(sigs):
        pos += 1 + (b % 4)
        offs.append(pos)
        pos += len(s)
    flat = np.zeros(pos + 8, f32)
    for o, s in zip(offs, sigs):
        flat[o:o + len(s)] = s
    assert any(o % 4 for o in offs)
    dev = torch.device("cuda")
    sig = torch.from_numpy(flat).to(dev)
    off = torch.tensor(offs + [pos], dtype=torch.int64, device=dev)
    n = torch.tensor([len(s) for s in sigs], dtype=torch.int32, device=dev)
    B, max_w = len(sigs), max(1, max(len(s) for s in sigs) // RES)
    ends = torch.empty(B, dtype=torch.int32, device=dev)
    starts = torch.empty(B, dtype=torch.int32, device=dev)
    stats = torch.zeros(B, max_w, 4, dtype=torch.float32, device=dev)
    _lib.check(_lib.lib().riser_polya_end_f32(_lib.ptr(sig), _lib.ptr(off), _lib.ptr(n), B, _lib.ptr(ends),
                                              _lib.ptr(starts), _lib.ptr(stats), max_w, _lib.stream_ptr()),
               "riser_polya_end_f32")
    e, s, st = ends.cpu().numpy(), starts.cpu().numpy(), stats.cpu().numpy()
    check_against_numpy(e, s, st, sigs)
    e2, s2, st2 = run_f32(proc, sigs)
    assert np.array_equal(e, e2) and np.array_equal(s, s2)


def test_trim_and_get_polya_end_float32(proc):
    """riser/preprocess.py:87-102 on float32: only found ends are cached, a cached end short-circuits detection, the
    cut is at end + 1; integer input keeps the int16 route; a mixed batch is refused."""
    reads = synth.raw_reads(12, 40, min_body=3000, max_body=14000, frac_no_polya=0.2)
    items = [(rid, calibrate(s, 0.684, 10)) for rid, s in reads]
    cache_g, cache_o = {}, {}
    for rid, x in items:
        assert proc.get_polyA_end(x) == pp.polya_end(x)
        got, tg = proc.trim_polyA(x, rid, cache_g)
        want, to = pp.trim_polya(x, rid, cache_o)
        assert tg == to and got.dtype == f32 and np.array_equal(got, want)
    assert cache_g == cache_o and len(cache_g) > 15
    for rid, x in items:                     # cache hits: the shorter prefix is cut where the cached end says
        got, tg = proc.trim_polyA(x[:4000], rid, cache_g)
        want, to = pp.trim_polya(x[:4000], rid, cache_o)
        assert tg == to and np.array_equal(got, want)
    batch = [x for _, x in items[:8]]
    assert np.array_equal(proc.get_polyA_end_batch(batch),
                          [-1 if e is None else e for e in (pp.polya_end(x) for x in batch)])
    with pytest.raises(TypeError):
        proc.get_polyA_end_batch([batch[0], reads[1][1]])


def _models(targets):
    return [Model(synth.state_dict(synth.TARGET_SEEDS[t]), shipped_config(), LOG, t) for t in targets]


def test_batched_classifier_float32_vs_oracle(proc):
    reads = synth.raw_reads(5, 64, min_body=3000, max_body=16000, frac_no_polya=0.2, frac_const=0.05)
    rng = np.random.default_rng(1)
    items = []
    for i, (rid, sig) in enumerate(reads):
        scale, offset = [(0.684, 10.0), (1.3, -20.0), (0.1759, 3.2)][i % 3]
        items.append((rid, calibrate(sig[:int(rng.integers(len(sig) // 2, len(sig) + 1))], scale, offset)))
    targets = ["mRNA", "mtRNA", "globin"]
    states = [synth.state_dict(synth.TARGET_SEEDS[t]) for t in targets]
    models = _models(targets)
    clf = BatchedClassifier(models, proc, signal_dtype=np.float32)
    eager = BatchedClassifier(models, proc, signal_dtype=np.float32)
    eager.use_graphs = False
    sigs, ids = [s for _, s in items], [r for r, _ in items]
    for mode in ("deplete", "enrich"):
        dec_o, p_on_o, p_off_o, len_o, cache_o = cref.run_batch_f32(items, states, "RNA002", {}, 0.9, mode)
        cache_g = {}
        res = clf.classify_batch(sigs, ids, cache_g, 0.9, mode)
        assert np.array_equal(res.sig_len, len_o)
        assert cache_g == cache_o
        assessed = len_o > 0
        assert assessed.sum() > 10 and (~assessed).sum() > 3
        assert np.abs(res.p_on[assessed] - p_on_o[assessed]).max() < 1e-3
        assert np.abs(res.p_off[assessed] - p_off_o[assessed]).max() < 1e-3
        near = (np.abs(p_on_o - 0.9).min(axis=1) <= 1e-3) | (np.abs(p_off_o - 0.9).min(axis=1) <= 1e-3)
        assert np.all((res.decisions == dec_o) | near)
        # second pass: the found ends come from the cache (less to upload), same results; this one replays the graph
        res2 = clf.classify_batch(sigs, ids, cache_g, 0.9, mode)
        assert np.array_equal(res2.decisions, res.decisions) and np.array_equal(res2.sig_len, res.sig_len)
        assert np.array_equal(res2.p_on, res.p_on, equal_nan=True) and res2.h2d_bytes < res.h2d_bytes
        assert cache_g == cache_o
        # graph replay and the eager launches give identical results
        for cache in ({}, dict(cache_o)):
            a = clf.classify_batch(sigs, ids, dict(cache), 0.9, mode)
            b = eager.classify_batch(sigs, ids, dict(cache), 0.9, mode)
            for f in ("decisions", "p_on", "p_off", "sig_len", "polya_end"):
                assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=f.startswith("p_")), f
    assert clf._graphs and not eager._graphs
    # refusals: a float32 classifier takes float32 only; the default one still refuses float
    with pytest.raises(TypeError):
        clf.classify_batch([reads[0][1]], [ids[0]], {}, 0.9, "deplete")
    with pytest.raises(TypeError):
        clf.classify_batch([sigs[0], reads[1][1]], ids[:2], {}, 0.9, "deplete")
    with pytest.raises(TypeError):
        BatchedClassifier(models, proc).classify_batch(sigs[:2], ids[:2], {}, 0.9, "deplete")


class OracleProc(SignalProcessor):
    """SignalProcessor whose poly(A) trim and normalisation are numpy's (the oracle's) instead of the GPU's."""
    def trim_polyA(self, signal, read_id, cache):
        return pp.trim_polya(signal, read_id, cache)

    def mad_normalise(self, signal):
        return cref.mad_normalise_f32(signal)


class OracleModel:
    def __init__(self, target):
        self.target = target
        self.state = synth.state_dict(synth.TARGET_SEEDS[target])

    def classify(self, signal):
        return net.classify(self.state, signal)


def _run_control(reads, models, tmp_path, name, mode, warm=()):
    client = sim.SimClient(reads, 3012, 6, first_len=6024)
    assert client.signal_dtype == np.float32
    control = SequencerControl(client, models, SignalProcessor(Kit.create_from_version("RNA002")), LOG,
                               str(tmp_path / name), warm_up_batches=warm)
    control.start()
    control.target(mode, 1, 0.9)
    control.finish()
    with open(tmp_path / f"{name}.csv") as f:
        return [ln.rstrip("\n").split(",", 1)[1].split(",") for ln in f][1:], client, control


def _run_serial(reads, models, proc, tmp_path, name, mode):
    client = sim.SimClient(reads, 3012, 6, first_len=6024)
    client.start_streaming_reads()
    ctl.serial_target(client, models, proc, str(tmp_path / name), mode, 0.9)
    with open(tmp_path / f"{name}.csv") as f:
        return [ln.rstrip("\n").split(",", 1)[1].split(",") for ln in f][1:], client


def _compare_rows(got, want, thr=0.9):
    assert len(got) == len(want) and len(got) > 5
    forgiven = 0
    for a, b in zip(got, want):
        assert a[:4] == b[:4], (a, b)                      # read id, channel, sig_length, models
        pa = np.array([float(x) for x in a[4].split(";")])
        pb = np.array([float(x) for x in b[4].split(";")])
        assert np.abs(pa - pb).max() < 1e-3
        assert a[5:7] == b[5:7]
        if a[7] != b[7]:
            assert np.abs(pb - thr).min() <= 1e-3, (a, b)
            forgiven += 1
    return forgiven


@pytest.mark.parametrize("mode", ["deplete", "enrich"])
def test_sequencer_control_calibrated_client(tmp_path, mode):
    reads = [(rid, calibrate(s, 0.684, 10)) for rid, s in
             synth.raw_reads(77, 48, min_body=3000, max_body=15000, frac_no_polya=0.15, frac_const=0.05)]
    targets = ["mRNA", "mtRNA"]
    got, client, control = _run_control(reads, _models(targets), tmp_path, "live", mode, warm=(48,))
    assert control.classifier_f32 is not None and not control.classifier._graphs      # the int16 one stays idle
    want, ref_client = _run_serial(reads, [OracleModel(t) for t in targets],
                                   OracleProc(Kit.create_from_version("RNA002")), tmp_path, "oracle", mode)
    forgiven = _compare_rows(got, want)
    if not forgiven:
        assert sorted(client.unblocked) == sorted(ref_client.unblocked)
        assert sorted(client.finished) == sorted(ref_client.finished)
    if refshim.available():                # and the reference's own SignalProcessor behind the serial loop
        rp = refshim.load().preprocess
        want, ref_client = _run_serial(reads, [OracleModel(t) for t in targets],
                                       rp.SignalProcessor(rp.Kit.create_from_version("RNA002")), tmp_path, "ref",
                                       mode)
        _compare_rows(got, want)


def test_sequencer_control_refuses_mixed_poll(tmp_path):
    class Mixed(sim.SimClient):
        def get_raw_signal(self, read):
            a = np.frombuffer(read.raw_data, np.int16)
            return a.astype(f32) if read.number == 1 else a
    reads = synth.raw_reads(3, 2, min_body=6000, max_body=8000)
    client = Mixed(reads, 3012, 2, first_len=6024)
    control = SequencerControl(client, _models(["mRNA"]), SignalProcessor(Kit.create_from_version("RNA002")), LOG,
                               str(tmp_path / "mixed"))
    control.start()
    with pytest.raises(TypeError):
        control.target("deplete", 1, 0.9)
