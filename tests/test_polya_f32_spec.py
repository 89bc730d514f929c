"""CPU: the float32 arithmetic riser_polya_end_f32 (csrc/polya_f32.cu) reproduces, pinned against numpy itself --
the pairwise-sum tree of np.mean for 500 and 1,000 elements, the median / MAD rule, the dtype of the mean-change
test -- and a step-by-step restatement of the kernel's window arithmetic against oracle.polya_end on calibrated
reads.  Also: float32 reads go through the native gather (_hostpack) with the 4-sample padding RaggedBatch uses."""
import numpy as np
import pytest

from oracle import preprocess_oracle as pp
from tests import calibrated_reference as cref
from riser_b200 import build, synth
from riser_b200.preprocess import _hostpack

f32 = np.float32
PW_BLOCK = 128


def pw_split(n):
    return n // 2 - (n // 2) % 8


def pw_leaves(n, s=0):
    """Leaves (start, length) of numpy's pairwise sum over [s, s + n), from its recursion (as the kernel derives them
    at compile time)."""
    if n <= PW_BLOCK:
        return [(s, n)]
    n2 = pw_split(n)
    return pw_leaves(n2, s) + pw_leaves(n - n2, s + n2)


def pw_sum(a):
    """The kernel's sum: leaf = 8 interleaved float32 accumulators, combined ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)),
    then the n % 8 tail one by one; leaves combined in the tree's order; the reduction's identity 0 added last."""
    def rec(s, n):
        if n > PW_BLOCK:
            n2 = pw_split(n)
            return f32(rec(s, n2) + rec(s + n2, n - n2))
        body = n - n % 8
        r = a[s:s + body].reshape(-1, 8).copy()
        acc = r[0].copy()
        for row in r[1:]:
            acc = (acc + row).astype(f32)
        res = f32(f32(f32(acc[0] + acc[1]) + f32(acc[2] + acc[3])) + f32(f32(acc[4] + acc[5]) + f32(acc[6] + acc[7])))
        for i in range(s + body, s + n):
            res = f32(res + a[i])
        return res
    return f32(rec(0, len(a)) + f32(0))


def f2key(x):
    u = np.asarray(x, dtype=f32).view(np.uint32)
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def key2f(k):
    k = np.asarray(k, dtype=np.uint32)
    return np.where(k & 0x80000000, k ^ 0x80000000, ~k).astype(np.uint32).view(f32)


def mid_mean(a, b):
    return f32(f32(f32(a + b) + f32(0)) * f32(0.5))


def kernel_median(w):
    """Ranks 249 / 250 on the order-preserving uint32 image, then the two-value rule."""
    k = np.sort(f2key(w))
    return mid_mean(key2f(k[len(w) // 2 - 1]), key2f(k[len(w) // 2]))


def kernel_polya(signal):
    """Restatement of polya_f32_kernel's window loop and scan -> (end or None, [n_windows, 4] stats)."""
    res = 500
    nw = min(len(signal) // res, 512)
    start = end = None
    stats = []
    for w in range(nw):
        x = signal[w * res:(w + 1) * res]
        med = kernel_median(x)
        mad = kernel_median(np.abs((x - med).astype(f32)))
        mean = f32(pw_sum(x) / f32(res))
        rolling = f32(pw_sum(signal[(w - 2) * res:w * res]) / f32(2 * res)) if w > 2 else mean
        change = f32(f32(f32(mean - rolling) / rolling) * f32(100))
        stats.append((med, mad, mean, rolling))
        if not start and w > 0 and change > 20 and mad <= 20:
            start = w * res
        if start and not end and mad > 20:
            end = w * res
    return end, np.array(stats, dtype=np.float64).reshape(-1, 4)


def _same_bits(a, b):
    return np.asarray(a, dtype=f32).view(np.uint32).tolist() == np.asarray(b, dtype=f32).view(np.uint32).tolist()


def test_pairwise_tree_matches_numpy():
    assert pw_leaves(500) == [(0, 120), (120, 128), (248, 120), (368, 64), (432, 68)]
    assert pw_leaves(1000) == [(0, 120), (120, 128), (248, 120), (368, 128), (496, 120), (616, 128), (744, 128),
                               (872, 128)]
    rng = np.random.default_rng(11)
    for t in range(400):
        n = 500 if t % 2 else 1000
        a = (rng.normal(100, 30, n) * rng.uniform(0.1, 3) + rng.uniform(-150, 50)).astype(f32)
        s = np.add.reduce(a)
        assert s.dtype == f32 and _same_bits(pw_sum(a), s)
        m = np.mean(a)
        assert m.dtype == f32 and _same_bits(f32(pw_sum(a) / f32(n)), m)
    # the rolling mean is its own 1000-element tree: the two 500-element sums do not reproduce it in general
    differs = 0
    for _ in range(200):
        a = (rng.normal(90, 20, 1000) * 0.684).astype(f32)
        differs += not _same_bits(f32(pw_sum(a[:500]) + pw_sum(a[500:])), np.add.reduce(a))
    assert differs > 0
    for z in (np.full(500, -0.0, f32), np.zeros(1000, f32)):                # numpy's identity: +0.0
        assert _same_bits(pw_sum(z), np.add.reduce(z)) and _same_bits(pw_sum(z), f32(0))


def test_median_and_mad_rule_matches_numpy():
    rng = np.random.default_rng(12)
    cases = [rng.normal(80, 15, 500).astype(f32) for _ in range(200)]
    cases += [np.round(rng.normal(0, 3, 500)).astype(f32) for _ in range(50)]          # ties, negatives
    cases += [np.full(500, -2.5, f32), np.full(500, -0.0, f32),
              np.concatenate([np.full(250, -0.0, f32), np.full(250, 0.0, f32)])]
    for x in cases:
        med = np.median(x)
        mad = np.median(np.abs(x - med))
        assert med.dtype == f32 and mad.dtype == f32
        assert _same_bits(kernel_median(x), med)
        assert _same_bits(kernel_median(np.abs((x - kernel_median(x)).astype(f32))), mad)
        a, b = np.sort(x)[249:251]
        assert _same_bits(f32(np.float64(f32(a + b)) / 2), med) or (a == 0 and b == 0)


def test_mean_change_stays_float32():
    mean, rolling = f32(121.3), f32(100.7)
    change = (mean - rolling) / rolling * 100                  # preprocess.py:57, NEP 50: float32 throughout
    assert change.dtype == f32
    assert _same_bits(change, f32(f32(f32(mean - rolling) / rolling) * f32(100)))
    # one float32 ulp either side of 20 decides differently
    hi, lo = np.nextafter(f32(20), f32(21)), np.nextafter(f32(20), f32(19))
    assert hi > 20 and not lo > 20 and not f32(20) > 20


@pytest.mark.parametrize("scale,offset", [(0.1759, 3.2), (0.684, 10.0), (1.3, -20.0)])
def test_kernel_restatement_matches_oracle(scale, offset):
    reads = synth.raw_reads(5, 60, min_body=3000, max_body=14000)
    found = 0
    for _, s in reads:
        x = ((s.astype(f32) + f32(offset)) * f32(scale)).astype(f32)
        end, stats = kernel_polya(x)
        want = pp.polya_end(x)
        assert end == want
        found += want is not None
        ref = cref.polya_window_stats(x)
        assert _same_bits(stats, ref)
    if scale == 0.1759:
        assert found == 0          # MAD thresholds are ADC-sized: pA windows never exceed 20
    else:
        assert found > 40


def test_hostpack_packs_float32_reads():
    build.build_hostpack()
    hp = _hostpack()
    rng = np.random.default_rng(4)
    sigs = [rng.normal(90, 20, int(n)).astype(f32) for n in rng.integers(0, 3000, size=50)]
    sigs[7] = np.zeros(0, f32)
    sigs[9] = sigs[9].tobytes()
    as32 = [np.frombuffer(s, f32) if isinstance(s, bytes) else s for s in sigs]
    nbytes = np.zeros(len(sigs), dtype=np.int64)
    hp.lengths(sigs, nbytes)
    n = nbytes // 4
    assert np.array_equal(n, [len(s) for s in as32])
    skip, take = n // 5, n - n // 5 - n // 7
    pos = np.zeros(len(sigs) + 1, dtype=np.int64)
    np.cumsum((take + 3) & ~3, out=pos[1:])                   # 4 float32 samples = 16 bytes (RaggedBatch)
    assert all(p % 4 == 0 for p in pos)
    dst = np.full(int(pos[-1]) + 4, np.nan, dtype=f32)
    want = dst.copy()
    for s, o, a, k in zip(as32, pos[:-1], skip, take):
        want[o:o + k] = s[a:a + k]
    hp.pack(sigs, dst, pos[:-1] * 4, skip * 4, take * 4, 2)
    assert _same_bits(dst, want)


def test_signal_dtype_routing():
    from riser_b200.preprocess import signal_dtype
    assert signal_dtype([np.zeros(3, f32), np.zeros(0, f32)]) == f32
    assert signal_dtype([np.zeros(3, np.int32), np.zeros(2, np.int16)]) == np.int16
    with pytest.raises(TypeError):
        signal_dtype([np.zeros(3, f32), np.zeros(3, np.int16)])


@pytest.mark.skipif(__import__("torch").cuda.is_available(), reason="checks the no-GPU behaviour")
def test_float32_route_needs_a_gpu():
    from riser_b200 import Kit, SignalProcessor, _lib
    p = SignalProcessor(Kit.create_from_version("RNA002"))
    with pytest.raises(_lib.RiserError):
        p.get_polyA_end(np.arange(5000, dtype=f32))
    with pytest.raises(_lib.RiserError):
        p.trim_polyA(np.arange(5000, dtype=f32), "r", {})
