"""GPU: the long-window normalisers (csrc/normalise_long.cu, riser_normalise_long / riser_normalise_f32_long) and the
routing that sends windows above the shared-memory kernels' limits to them.  Every comparison is of bits: fp32 output
arrays for equality, the median / MAD words exactly."""
import logging

import numpy as np
import pytest
import torch

from oracle import convnet_oracle as net
from oracle import preprocess_oracle as pp
from oracle import retrain_oracle as rt
from riser_b200 import Kit, Model, RaggedBatch, SignalProcessor, retrain, synth, _lib
from riser_b200.config import shipped_config
from tests import calibrated_reference as cref

pytestmark = pytest.mark.gpu

LENGTHS = [98305, 250001, 1000000, 2 ** 21 + 3]
SHAPES = ["synth", "full_range", "two_valued", "constant", "end_outliers", "chunk_spikes", "long_run"]


@pytest.fixture(scope="module")
def proc():
    return SignalProcessor(Kit.create_from_version("RNA002"))


def shape(name, n, seed=0):
    """int16 window `name` of n samples."""
    rng = np.random.default_rng([seed, n, SHAPES.index(name)])
    if name == "full_range":
        return rng.integers(-32768, 32768, size=n).astype(np.int16)
    if name == "two_valued":                       # n // 2 of one value, the rest the other: MAD 0 for odd n
        x = np.full(n, 1800, dtype=np.int16)
        x[rng.permutation(n)[:n // 2]] = -250
        return x
    if name == "constant":
        return np.full(n, 321, dtype=np.int16)
    x = synth.body(rng, n).astype(np.int32)
    if name == "end_outliers":
        x[0] += 3000
        x[-1] -= 3000
    elif name == "chunk_spikes":                   # runs of 2..5 spikes at every multiple of 4096 +- 3
        for m in range(4096, n, 4096):
            for a in (m - 3, m + 3):
                r = int(rng.integers(2, 6))
                x[max(a - r // 2, 0):a - r // 2 + r] += 2500 * (1 if rng.random() < 0.5 else -1)
    elif name == "long_run":                       # one run of ~45 % of the window
        a = n // 7
        x[a:a + int(0.45 * n)] += 2500
    return np.clip(x, -32768, 32767).astype(np.int16)


def oracle16(x):
    return np.asarray(pp.mad_normalise(x), dtype=np.float64).astype(np.float32)


def stats16(x):
    med = np.median(x)
    return int(round(2 * med)), int(round(4 * np.median(np.abs(x - med))))


def workspace(B, max_len):
    nbytes = _lib.lib().riser_normalise_long_workspace_bytes(B, max_len)
    return torch.empty(nbytes, dtype=torch.uint8, device="cuda"), nbytes


def long16(sigs, max_len=None, start=None, length=None, ld=None, fill=0.0, batch=None):
    """riser_normalise_long over int16 windows -> (out [B, ld] ndarray, med2_mad4 [B, 2] ndarray)."""
    batch = batch or RaggedBatch(sigs, torch.device("cuda"))
    n = np.array([len(s) for s in sigs], dtype=np.int32) if length is None else np.asarray(length, dtype=np.int32)
    max_len = max_len or int(n.max())
    ld = ld or max_len
    out = torch.full((batch.B, ld), fill, device="cuda")
    stats = torch.full((batch.B, 2), -7, dtype=torch.int32, device="cuda")
    ws, nbytes = workspace(batch.B, max_len)
    st = None if start is None else torch.from_numpy(np.asarray(start, dtype=np.int32)).cuda()
    _lib.check(_lib.lib().riser_normalise_long(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(st),
                                               _lib.ptr(torch.from_numpy(n).cuda()), batch.B, max_len, _lib.ptr(out),
                                               ld, _lib.ptr(stats), _lib.ptr(ws), nbytes, _lib.stream_ptr()),
               "riser_normalise_long")
    return out.cpu().numpy(), stats.cpu().numpy()


def long32(sigs, lim, zero_if_mad0, max_len=None, ld=None, fill=0.0):
    """riser_normalise_f32_long -> (out [B, ld] ndarray, med_mad [B, 2] ndarray)."""
    batch = RaggedBatch(sigs, torch.device("cuda"), dtype=np.float32)
    n = np.array([len(s) for s in sigs], dtype=np.int32)
    max_len = max_len or int(n.max())
    ld = ld or max_len
    out = torch.full((batch.B, ld), fill, device="cuda")
    med_mad = torch.zeros(batch.B, 2, device="cuda")
    ws, nbytes = workspace(batch.B, max_len)
    _lib.check(_lib.lib().riser_normalise_f32_long(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(batch.n),
                                                   batch.B, max_len, lim, zero_if_mad0, _lib.ptr(out), ld,
                                                   _lib.ptr(med_mad), _lib.ptr(ws), nbytes, _lib.stream_ptr()),
               "riser_normalise_f32_long")
    return out.cpu().numpy(), med_mad.cpu().numpy()


def to_pa(x, k):
    return rt.pa_signal(x, scale=0.1 + 0.013 * k, offset=2.5 * k - 9)


@pytest.mark.parametrize("n", LENGTHS)
def test_int16_long_windows_match_oracle(proc, n):
    sigs = [shape(s, n) for s in SHAPES]
    out, stats = long16(sigs)
    for b, (name, x) in enumerate(zip(SHAPES, sigs)):
        assert tuple(stats[b]) == stats16(x), (name, n)
        want = oracle16(x)
        assert np.array_equal(out[b], want), (name, n, np.flatnonzero(out[b] != want)[:8])
    z = proc.mad_normalise(sigs[SHAPES.index("constant")])
    assert z.dtype == np.int64 and not z.any() and len(z) == n


@pytest.mark.parametrize("n", LENGTHS)
def test_float32_long_windows_match_numpy(n):
    sigs = [to_pa(shape(s, n), k) for k, s in enumerate(SHAPES)]
    out, med_mad = long32(sigs, 3.5, 0)                       # retrain: no guard, inf / nan on MAD 0
    for b, (name, x) in enumerate(zip(SHAPES, sigs)):
        want = rt.mad_normalise(x)
        assert np.array_equal(out[b], want, equal_nan=True), (name, n, np.flatnonzero(out[b] != want)[:8])
        med = np.median(x)
        assert med_mad[b, 0] == med and med_mad[b, 1] == np.median(np.abs(x - med)), name
    out, _ = long32(sigs, 3.5, 1)                             # live: zeros on MAD 0
    for b, (name, x) in enumerate(zip(SHAPES, sigs)):
        want = cref.mad_normalise_f32(x).astype(np.float32)
        assert np.array_equal(out[b], want), (name, n, np.flatnonzero(out[b] != want)[:8])
    out, _ = long32(sigs[:1], 2.0, 0)                         # a caller-chosen limit
    assert np.array_equal(out[0], rt.mad_normalise(sigs[0], 2.0))


def test_cabi_windows_inside_reads_ld_and_len0():
    rng = np.random.default_rng(31)
    reads = [synth.body(rng, 260000), synth.body(rng, 150000), synth.body(rng, 9000), synth.body(rng, 130001)]
    start = np.array([1237, 0, 5, 29999], dtype=np.int32)
    length = np.array([200003, 120000, 0, 100002], dtype=np.int32)
    skip = np.array([1000, 0, 0, 29990], dtype=np.int64)      # only part of each read is uploaded: off is virtual
    take = np.array([len(r) for r in reads], dtype=np.int64) - skip
    batch = RaggedBatch(reads, torch.device("cuda"), skip=skip, take=take)
    ld = 200003 + 61
    out, stats = long16(reads, start=start, length=length, ld=ld, fill=-123.0, batch=batch)
    for b, r in enumerate(reads):
        n = int(length[b])
        if n == 0:
            assert np.all(out[b] == -123.0) and tuple(stats[b]) == (-7, -7)
            continue
        w = r[start[b]:start[b] + n]
        assert np.array_equal(out[b, :n], oracle16(w)), b
        assert np.all(out[b, n:] == -123.0), b
        assert tuple(stats[b]) == stats16(w), b
    # a window longer than max_len is processed as its first max_len samples
    out, stats = long16(reads[:2], max_len=140000, ld=140000, fill=5.0)
    assert np.array_equal(out[0], oracle16(reads[0][:140000]))
    assert np.array_equal(out[1, :140000], oracle16(reads[1][:140000]))
    # the same for float32, with rows prefilled
    pa = [to_pa(r, k) for k, r in enumerate(reads[:2])]
    out, _ = long32(pa, 3.5, 0, max_len=140000, ld=140007, fill=9.0)
    assert np.array_equal(out[0, :140000], rt.mad_normalise(pa[0][:140000]))
    assert np.array_equal(out[1, :140000], rt.mad_normalise(pa[1][:140000]))
    assert np.all(out[:, 140000:] == 9.0)


def test_cabi_errors():
    L = _lib.lib()
    sig = torch.zeros(200000, dtype=torch.int16, device="cuda")
    sig32 = torch.zeros(200000, dtype=torch.float32, device="cuda")
    off = torch.zeros(2, dtype=torch.int64, device="cuda")
    ln = torch.full((1,), 150000, dtype=torch.int32, device="cuda")
    out = torch.zeros(1, 150000, device="cuda")
    ws, nbytes = workspace(1, 150000)
    s = _lib.stream_ptr()
    P = _lib.ptr
    assert nbytes > 0
    assert L.riser_normalise_long(P(sig), P(off), None, P(ln), 1, 150000, P(out), 150000, None, P(ws), nbytes - 1, s) == 3
    assert L.riser_normalise_f32_long(P(sig32), P(off), P(ln), 1, 150000, 3.5, 0, P(out), 150000, None, P(ws),
                                      nbytes - 1, s) == 3
    assert L.riser_normalise_long(None, P(off), None, P(ln), 1, 150000, P(out), 150000, None, P(ws), nbytes, s) == 1
    assert L.riser_normalise_long(P(sig), P(off), None, P(ln), 1, 150000, P(out), 150000, None, None, nbytes, s) == 1
    assert L.riser_normalise_f32_long(P(sig32), P(off), P(ln), 1, 150000, 3.5, 0, None, 150000, None, P(ws),
                                      nbytes, s) == 1
    assert L.riser_normalise_long(P(sig), P(off), None, P(ln), 1, 150000, P(out), 149999, None, P(ws), nbytes, s) == 1
    assert L.riser_normalise_long(P(sig), P(off), None, P(ln), 0, 150000, None, 0, None, None, 0, s) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("n", [4096, 12048, 98304])
def test_long_entries_equal_shared_memory_kernels_on_short_windows(n):
    L = _lib.lib()
    rng = np.random.default_rng(n)
    sigs = [synth.body(rng, n - k) for k in range(0, 40, 3)] + [shape("full_range", n), shape("two_valued", n - 1)]
    batch = RaggedBatch(sigs, torch.device("cuda"))
    ld = (n + 3) & ~3
    ref = torch.zeros(batch.B, ld, device="cuda")
    ref_stats = torch.zeros(batch.B, 2, dtype=torch.int32, device="cuda")
    _lib.check(L.riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), None, _lib.ptr(batch.n), batch.B, n,
                                 _lib.ptr(ref), ld, _lib.ptr(ref_stats), _lib.stream_ptr()), "riser_normalise")
    out, stats = long16(sigs, max_len=n, ld=ld, batch=batch)
    assert np.array_equal(out, ref.cpu().numpy()) and np.array_equal(stats, ref_stats.cpu().numpy())
    if n > L.riser_normalise_f32_max_len():
        return
    pa = [to_pa(s, k) for k, s in enumerate(sigs)]
    b32 = RaggedBatch(pa, torch.device("cuda"), dtype=np.float32)
    for lim, live in ((3.5, 1), (3.5, 0), (2.5, 0)):
        ref = torch.zeros(batch.B, n, device="cuda")
        ref_mm = torch.zeros(batch.B, 2, device="cuda")
        if live:
            rc = L.riser_normalise_f32_live(_lib.ptr(b32.sig), _lib.ptr(b32.off), _lib.ptr(b32.n), b32.B, n,
                                            _lib.ptr(ref), n, _lib.ptr(ref_mm), _lib.stream_ptr())
        else:
            rc = L.riser_normalise_f32(_lib.ptr(b32.sig), _lib.ptr(b32.off), _lib.ptr(b32.n), b32.B, n, lim,
                                       _lib.ptr(ref), n, _lib.stream_ptr())
        _lib.check(rc, "riser_normalise_f32")
        out, mm = long32(pa, lim, live, max_len=n)
        assert np.array_equal(out, ref.cpu().numpy(), equal_nan=True), (lim, live)
        if live:
            assert np.array_equal(mm, ref_mm.cpu().numpy())


def test_mixed_batch_routes_by_length(proc):
    rng = np.random.default_rng(33)
    limit = _lib.lib().riser_normalise_max_len()
    sigs = [synth.body(rng, n) for n in (5000, 120000, limit, limit + 1, 16000, 300000, 4096)]
    out, lens, stats = proc.mad_normalise_batch(sigs, return_stats=True)
    out, stats = out.cpu().numpy(), stats.cpu().numpy()
    assert np.array_equal(lens.cpu().numpy(), [len(s) for s in sigs])
    short = [k for k, s in enumerate(sigs) if len(s) <= limit]
    ref, _, ref_stats = proc.mad_normalise_batch([sigs[k] for k in short], return_stats=True)
    ref, ref_stats = ref.cpu().numpy(), ref_stats.cpu().numpy()
    for j, k in enumerate(short):
        n = len(sigs[k])
        assert np.array_equal(out[k, :n], ref[j, :n]) and np.array_equal(stats[k], ref_stats[j]), k
    for k, s in enumerate(sigs):
        n = len(s)
        assert np.array_equal(out[k, :n], oracle16(s)) and tuple(stats[k]) == stats16(s), k
        assert not out[k, n:].any(), k
    # windows (start / length) of reads above the limit
    start = np.array([0, 17, 3, 0, 100, 1001, 0], dtype=np.int32)
    length = np.array([len(s) for s in sigs], dtype=np.int32) - start
    length[0] = 0
    out, _ = proc.mad_normalise_batch(sigs, start=start, length=length)
    out = out.cpu().numpy()
    for k, s in enumerate(sigs[1:], 1):
        assert np.array_equal(out[k, :length[k]], oracle16(s[start[k]:])), k
    assert not out[0].any()


def test_public_entry_points_on_long_reads(proc):
    rng = np.random.default_rng(34)
    x = synth.body(rng, 300000)
    y = proc.mad_normalise(x)
    assert y.dtype == np.float64 and np.array_equal(y.astype(np.float32), oracle16(x))
    f = to_pa(synth.body(rng, 120000), 3)
    y = proc.mad_normalise(f)
    assert y.dtype == np.float32 and np.array_equal(y, cref.mad_normalise_f32(f))
    assert not proc.mad_normalise(np.full(120000, np.float32(7.25))).any()
    reads = [to_pa(synth.body(rng, n), k) for k, n in enumerate((90000, 79999, 80000, 150000))]
    data, dropped = retrain.preprocess_reads(reads, n_secs=20, freq=4000)
    assert data.shape == (3, 80000) and dropped == 1
    for row, r in zip(data, [reads[0], reads[2], reads[3]]):
        assert np.array_equal(row, rt.mad_normalise(r[:80000]))
    state = synth.state_dict(0)
    model = Model(state, shipped_config(), logging.getLogger("test"), "mRNA")
    z = proc.mad_normalise(synth.body(rng, 200000))
    p = model.classify(z)
    want = net.classify(state, z)
    assert abs(p[1].item() - want[1].item()) < 1e-3 and abs(p[0].item() - want[0].item()) < 1e-3


def test_long_path_replays_from_a_cuda_graph():
    rng = np.random.default_rng(35)
    L = _lib.lib()
    sigs = [shape("chunk_spikes", 250001), synth.body(rng, 180000), synth.body(rng, 99000)]
    pa = [to_pa(s, k) for k, s in enumerate(sigs)]
    want, want_stats = long16(sigs)                           # (also loads the kernels before the capture)
    want32, _ = long32(pa, 3.5, 0)
    for k, x in enumerate(pa):
        assert np.array_equal(want32[k, :len(x)], rt.mad_normalise(x)), k
    batch = RaggedBatch(sigs, torch.device("cuda"))
    b32 = RaggedBatch(pa, torch.device("cuda"), dtype=np.float32)
    B, max_len = batch.B, 250001
    out = torch.zeros(B, max_len, device="cuda")
    out32 = torch.zeros(B, max_len, device="cuda")
    stats = torch.zeros(B, 2, dtype=torch.int32, device="cuda")
    ws, nbytes = workspace(B, max_len)
    ws32, _ = workspace(B, max_len)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rc = L.riser_normalise_long(_lib.ptr(batch.sig), _lib.ptr(batch.off), None, _lib.ptr(batch.n), B, max_len,
                                    _lib.ptr(out), max_len, _lib.ptr(stats), _lib.ptr(ws), nbytes, _lib.stream_ptr())
        rc32 = L.riser_normalise_f32_long(_lib.ptr(b32.sig), _lib.ptr(b32.off), _lib.ptr(b32.n), B, max_len, 3.5, 0,
                                          _lib.ptr(out32), max_len, None, _lib.ptr(ws32), nbytes, _lib.stream_ptr())
    assert rc == 0 and rc32 == 0
    for _ in range(2):
        out.fill_(0.0)                                        # (rows past len[b] are not written)
        out32.fill_(0.0)
        stats.fill_(0)
        g.replay()
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(stats.cpu().numpy(), want_stats)
        assert np.array_equal(out32.cpu().numpy(), want32)


def zero_median_window(n, seed):
    """float32 window of n samples whose middle value(s) are -0.0 and whose MAD is 5: 500-sample blocks of 249 x -5,
    2 x -0.0 and 249 x 5 (shuffled), then one more -0.0 when n is odd; every 500-sample window has the same median."""
    rng = np.random.default_rng(seed)
    block = np.float32([-5] * 249 + [-0.0] * 2 + [5] * 249)
    x = np.concatenate([rng.permutation(block) for _ in range(n // 500)] + [np.float32([-0.0] * (n % 500))])
    return x.astype(np.float32)


def test_median_of_negative_zeros_is_positive_zero(proc):
    """numpy's median of two -0.0 (or of one, for an odd count) is +0.0, so every -0.0 sample normalises to
    -0.0 - +0.0 = -0.0; compared as bit patterns, since +0 == -0 as floats."""
    limit = _lib.lib().riser_normalise_f32_max_len()
    lengths = [40000, 40001, 60000, 60001]
    assert lengths[1] < limit < lengths[2]
    sigs = [zero_median_window(n, n) for n in lengths]
    bits = lambda a: np.asarray(a, dtype=np.float32).view(np.uint32)
    for x in sigs:
        assert np.median(x).view(np.uint32) == 0 and np.median(np.abs(x - np.median(x))) == 5
        want = cref.mad_normalise_f32(x)
        assert np.array_equal(bits(want), bits(pp.mad_normalise(x)))
        assert np.array_equal(bits(proc.mad_normalise(x)), bits(want)), len(x)
    out, _ = retrain.mad_normalise_f32_batch(sigs)
    out = out.cpu().numpy()
    out32, med_mad = long32(sigs, 3.5, 0)
    for b, x in enumerate(sigs):
        want = bits(rt.mad_normalise(x))
        assert np.array_equal(bits(out[b, :len(x)]), want), len(x)
        assert np.array_equal(bits(out32[b, :len(x)]), want), len(x)
        assert bits(med_mad[b, 0]) == 0 and med_mad[b, 1] == 5
    batch = RaggedBatch(sigs, torch.device("cuda"), dtype=np.float32)
    _, stats = proc.polya_end_device(batch, return_stats=True)
    stats = stats.cpu().numpy()
    for b, x in enumerate(sigs):
        w = len(x) // 500
        assert np.all(bits(stats[b, :w, 0]) == 0) and np.all(stats[b, :w, 1] == 5), len(x)
