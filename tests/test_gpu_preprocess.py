"""GPU parity: csrc/preprocess.cu through the C ABI against the oracle and the
reference-generated golden fixtures.  Integer statistics are exact; the fp32 output
must equal the reference's float64 result rounded to fp32 (tolerance stated by the
north star: 1e-6 relative -- we assert bit equality, which is stronger)."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import preprocess_oracle as pp
from riser_b200 import Kit, SignalProcessor, synth
from tests.golden import make_golden_params as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def proc():
    return SignalProcessor(Kit.create_from_version("RNA002"))


def sha(a):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def oracle32(x):
    return np.asarray(pp.mad_normalise(x), dtype=np.float64).astype(np.float32)


def check_batch(proc, signals, **kw):
    out, lens, stats = proc.mad_normalise_batch(signals, return_stats=True, **kw)
    out, stats = out.cpu().numpy(), stats.cpu().numpy()
    starts = kw.get("start")
    lengths = kw.get("length")
    for b, s in enumerate(signals):
        st = 0 if starts is None else int(starts[b])
        n = (len(s) - st) if lengths is None else int(lengths[b])
        w = s[st:st + n]
        if n == 0:
            continue
        med = np.median(w)
        mad = np.median(np.abs(w - med))
        assert stats[b, 0] == int(round(2 * med)) and stats[b, 1] == int(round(4 * mad)), b
        want = oracle32(w)
        got = out[b, :n]
        assert np.array_equal(got, want), (b, n, np.abs(got - want).max(), np.flatnonzero(got != want)[:8])


def test_edge_cases_bit_exact(proc, golden_dir):
    g = np.load(os.path.join(golden_dir, "preprocess_edge.npz"))
    sigs = [g[f"norm_in_{n}"] for n in g["norm_names"]]
    out, _ = proc.mad_normalise_batch(sigs)
    out = out.cpu().numpy()
    for b, name in enumerate(g["norm_names"]):
        want = g[f"norm_out_{name}"].astype(np.float64).astype(np.float32)   # reference output
        assert np.array_equal(out[b, :len(want)], want), name
    # single-read drop-in call: the reference's dtype too -- float64, or int64 zeros when MAD == 0 (np.vectorize types
    # its output by the first element, the int 0 of riser/preprocess.py:123)
    for b, name in enumerate(g["norm_names"]):
        y = proc.mad_normalise(sigs[b])
        assert y.dtype == g[f"norm_out_{name}"].dtype, name
        assert np.array_equal(y.astype(np.float32), oracle32(sigs[b])), name
    with pytest.raises(ValueError):
        proc.mad_normalise(np.array([], dtype=np.int16))


def test_realistic_reads_match_reference_sha(proc, golden_dir):
    g = np.load(os.path.join(golden_dir, "normalise_reads.npz"))
    bodies = P.norm_inputs()
    out, _ = proc.mad_normalise_batch(bodies)
    out = out.cpu().numpy()
    for b, x in enumerate(bodies):
        assert np.array_equal(sha(out[b, :len(x)]), g["sha_f32"][b]), b


def test_windows_and_odd_alignment(proc):
    rng = np.random.default_rng(3)
    sigs = [synth.body(rng, int(n)) for n in rng.integers(5000, 20000, size=24)]
    start = rng.integers(0, 900, size=24).astype(np.int32)
    length = np.array([min(len(s) - st, 12048) for s, st in zip(sigs, start)], dtype=np.int32)
    length[3] = 0            # a skipped read writes nothing
    check_batch(proc, sigs, start=start, length=length)


def test_random_stress_wide_ranges(proc):
    rng = np.random.default_rng(11)
    sigs = []
    for k in range(64):
        n = int(rng.integers(1, 16000))
        kind = k % 4
        if kind == 0:
            x = rng.integers(-32768, 32768, size=n)            # full range -> refinement pass
        elif kind == 1:
            x = rng.normal(500, 70, size=n)
            x[rng.random(n) < 0.02] += 5000                    # range > 2048 with a tight core
        elif kind == 2:
            x = rng.integers(0, 3, size=n) * 1000              # few distinct values, heavy ties
        else:
            x = rng.normal(-200, 15, size=n)
        sigs.append(np.clip(np.rint(x), -32768, 32767).astype(np.int16))
    check_batch(proc, sigs)


def test_value_ranges_around_the_histogram_limits(proc):
    """The normalise kernel bins a window by `sample & 2047` before it knows the minimum (fused min / max + histogram
    pass): exact while the range stays below 2,040; between 2,040 and 2,047 the histogram is rebuilt relative to the
    minimum, from 2,048 on it is a shifted histogram with a refinement pass.  Windows on both sides of every limit, with
    minima on both sides of the bins' wrap-around (multiples of 2,048, negative values), outliers included."""
    rng = np.random.default_rng(33)
    sigs = []
    for span in (1, 2, 7, 8, 9, 1000, 2038, 2039, 2040, 2041, 2046, 2047, 2048, 2049, 4095, 4096, 9000):
        for lo in (-2048 - 5, -2048, -1030, -7, 0, 3, 2040, 2047, 2048, 4090, 20000):
            if lo + span > 32767:
                continue
            n = int(rng.integers(4096, 9000))
            x = rng.normal(lo + span / 2.0, max(span / 9.0, 0.6), size=n)
            x = np.clip(np.rint(x), lo, lo + span)
            x[rng.integers(0, n, size=3)] = lo                  # the extremes are attained
            x[rng.integers(0, n, size=3)] = lo + span
            sigs.append(x.astype(np.int16))
    start = rng.integers(0, 9, size=len(sigs)).astype(np.int32)         # every 16-byte phase
    length = np.array([len(s) - st for s, st in zip(sigs, start)], dtype=np.int32)
    check_batch(proc, sigs, start=start, length=length)


def test_polya_end_matches_reference(proc, golden_dir):
    g = np.load(os.path.join(golden_dir, "polya.npz"))
    reads = P.polya_reads()
    sigs, want = [], []
    for r, (_, sig) in enumerate(reads):
        for j, n in enumerate(g["prefixes"]):
            sigs.append(sig[:n])
            want.append(g["ends"][r, j])
    for k in g["hand_names"]:
        sigs.append(g[f"hand_in_{k}"])
        want.append(int(g[f"hand_end_{k}"]))
    ends, stats = proc.get_polyA_end_batch(sigs, return_stats=True)
    assert np.array_equal(ends, np.array(want, dtype=np.int32))
    # window statistics are exact integers
    for b in (0, 7, 100, len(sigs) - 1):
        s = sigs[b]
        for w in range(len(s) // 500):
            win = s[w * 500:(w + 1) * 500].astype(np.int64)
            med = np.median(win)
            mad = np.median(np.abs(win - med))
            assert list(stats[b, w]) == [int(win.sum()), int(round(2 * med)), int(round(4 * mad))]
    # drop-in single calls incl. cache semantics (riser/preprocess.py:87-102)
    rid, sig = reads[0]
    cache, log = {}, []
    for n in (3000, 9000, 12000, 600):
        s, trimmed = proc.trim_polyA(sig[:n], rid, cache)
        log.append([n, len(s), int(trimmed), cache.get(rid, -1)])
    assert np.array_equal(np.array(log), g["cache_log"])


def test_polya_random_vs_oracle(proc):
    rng = np.random.default_rng(5)
    sigs = []
    for k in range(48):
        n = int(rng.integers(0, 25000))
        x = rng.normal(450, 50, size=n)
        for _ in range(3):
            a = int(rng.integers(0, max(n, 1)))
            x[a:a + int(rng.integers(300, 4000))] = rng.normal(rng.choice([620, 700, 300]), rng.choice([5, 12, 30]))
        sigs.append(np.rint(x).astype(np.int16))
    ends = proc.get_polyA_end_batch(sigs)
    want = [(-1 if pp.polya_end(s) is None else pp.polya_end(s)) for s in sigs]
    assert list(ends) == want


def test_polya_decision_only_path_corner_windows(proc):
    """The product path of riser_polya_end (no statistics requested) decides MAD > 20 from one count around the median
    instead of computing the MAD (csrc/preprocess.cu warp_window_fast).  Windows built to sit on its edges -- exactly
    250 samples within 20 of the median with the two middle distances summing to more than 80, MADs of exactly 20 and
    20.5, value ranges of 1,022 .. 1,025 (the histogram's limit), flat and two-valued windows, negative values -- must
    give the same ends as the statistics path and the oracle (riser/preprocess.py:42-79)."""
    rng = np.random.default_rng(11)

    def window(values, counts):
        w = np.repeat(np.array(values, dtype=np.int64), counts)
        assert len(w) == 500
        return rng.permutation(w)

    kinds = [
        window([400, 490, 510, 600], [125, 125, 125, 125]),        # c = 250, d1 + d2 = 40 + 400 -> MAD > 20
        window([475, 490, 510, 525], [125, 125, 125, 125]),        # c = 250, d1 + d2 = 40 + 100 > 80
        window([480, 490, 510, 520], [125, 125, 125, 125]),        # all within 20 of the median: MAD 15
        window([480, 500, 520], [125, 250, 125]),                  # MAD = 10 (c = 500)
        window([460, 479, 521, 540], [125, 125, 125, 125]),        # d1 = 42: c = 0
        window([459, 480, 520, 541], [120, 130, 130, 120]),        # MAD exactly 20 -> not > 20
        window([459, 480, 521, 541], [120, 130, 130, 120]),        # MAD 20.5 -> > 20
        window([0, 500, 1022], [100, 300, 100]),                   # range 1,022: histogram path
        window([0, 500, 1023], [100, 300, 100]),                   # range 1,023: its last bin
        window([0, 500, 1024], [100, 300, 100]),                   # range 1,024: bit-descent path
        window([-300, -280, -260, 725], [200, 100, 100, 100]),     # negative values, wide range
        window([431], [500]),                                      # flat
        window([431, 432], [250, 250]),                            # two values, median between them
        window([431, 432], [249, 251]),
    ]
    sigs = []
    for k in range(40):
        n_win = int(rng.integers(3, 30))
        parts = []
        for _ in range(n_win):
            if rng.random() < 0.5:
                parts.append(kinds[int(rng.integers(len(kinds)))] + int(rng.integers(-3, 4)) * int(rng.random() < 0.3))
            else:
                parts.append(np.rint(rng.normal(rng.choice([450, 620, 700]), rng.choice([4, 14, 27, 60]), size=500)).astype(np.int64))
        tail = np.rint(rng.normal(500, 30, size=int(rng.integers(0, 499)))).astype(np.int64)
        sigs.append(np.clip(np.concatenate(parts + [tail]), -32768, 32767).astype(np.int16))
    ends_fast = proc.get_polyA_end_batch(sigs)
    ends_stats, _ = proc.get_polyA_end_batch(sigs, return_stats=True)
    want = [(-1 if pp.polya_end(s) is None else pp.polya_end(s)) for s in sigs]
    assert list(ends_stats) == want
    assert list(ends_fast) == want
    assert sum(e > 0 for e in want) >= 5 and sum(e < 0 for e in want) >= 5


def test_retrain_float32_normalise_bit_exact(golden_dir):
    """csrc/normalise_f32.cu against the reference's riser/retrain/preprocess.py outputs."""
    from oracle import retrain_oracle as rt
    from riser_b200 import retrain
    g = np.load(os.path.join(golden_dir, "retrain_norm.npz"))
    bodies = synth.ragged_bodies(int(g["seed"]), 16, 4096, 12048)
    sigs = [rt.pa_signal(raw, scale=0.1 + 0.01 * k, offset=3.0 * k - 10) for k, raw in enumerate(bodies)]
    out, _ = retrain.mad_normalise_f32_batch(sigs)
    out = out.cpu().numpy()
    for k, s in enumerate(sigs):
        assert np.array_equal(sha(out[k, :len(s)]), g["sha"][k]), k
    names = [str(n) for n in g["names"]]
    out, _ = retrain.mad_normalise_f32_batch([g[f"in_{n}"] for n in names])
    out = out.cpu().numpy()
    for k, n in enumerate(names):
        want = g[f"out_{n}"]
        assert np.array_equal(out[k, :len(want)], want, equal_nan=True), n
    # retrain/preprocess.py main(): cutoff, discard, stack
    reads = [rt.pa_signal(synth.body(np.random.default_rng(i), 5000 + 900 * i)) for i in range(6)]
    data, dropped = retrain.preprocess_reads(reads, n_secs=2, freq=3012)
    assert data.shape == (4, 6024) and dropped == 2
    assert np.array_equal(data[0], rt.mad_normalise(reads[2][:6024]))


def _spiky(rng, n, every, height, base_sd=10.0):
    x = rng.normal(500, base_sd, size=n)
    x[::every] += height
    return np.clip(np.rint(x), -32768, 32767).astype(np.int16)


def test_outlier_run_paths(proc):
    """The run bookkeeping of the normalise kernel: more run starts than the shared-memory list holds (rescan
    path), with and without the per-value table (range above / below 2048); long runs, runs that touch both ends
    of the window; windows longer than 32 steps of a thread (> 32,768 samples)."""
    rng = np.random.default_rng(21)
    sigs = [
        _spiky(rng, 12000, 10, 1500),                 # 1200 isolated outliers, table path
        _spiky(rng, 12000, 10, 3000),                 # the same above the table's range
        _spiky(rng, 9000, 7, -1200),
    ]
    x = rng.normal(480, 12, size=15000)               # long runs, incl. one at each end of the window
    for a, ln in ((0, 40), (700, 75), (5000, 3), (14960, 40)):
        x[a:a + ln] += 900
    sigs.append(np.rint(x).astype(np.int16))
    x = rng.normal(520, 9, size=70000)                # > 32,768 samples: the per-thread mask is emptied mid-loop
    idx = rng.choice(70000, size=600, replace=False)
    x[idx] += rng.choice([-700, 650], size=600)
    x[40000:40020] -= 800
    sigs.append(np.rint(x).astype(np.int16))
    x = rng.normal(500, 6, size=98304)                # the longest window the kernel stages
    x[rng.random(98304) < 0.004] += 400
    sigs.append(np.rint(x).astype(np.int16))
    check_batch(proc, sigs)


def test_many_short_reads_with_gaps(proc):
    """More reads than resident CTAs, zero-length windows in between: the persistent loop's look-ahead
    (metadata, L2 prefetch) has to stay in step with the reads it skips."""
    rng = np.random.default_rng(22)
    B = 3200
    sigs = [synth.body(rng, int(n)) for n in rng.integers(40, 700, size=B)]
    start = rng.integers(0, 30, size=B).astype(np.int32)
    length = np.array([len(s) - st for s, st in zip(sigs, start)], dtype=np.int32)
    length[rng.random(B) < 0.3] = 0
    length[:5] = 0
    length[-3:] = 0
    check_batch(proc, sigs, start=start, length=length)


def test_normalise_cuts_windows_at_max_len():
    """A len[b] above the max_len the caller states must not run past the staging buffer: the window is processed
    as its first max_len samples (include/riser_b200.h)."""
    from riser_b200 import RaggedBatch, _lib
    rng = np.random.default_rng(9)
    sigs = [synth.body(rng, 9000), synth.body(rng, 5000)]
    batch = RaggedBatch(sigs, torch.device("cuda"))
    max_len = 6000
    out = torch.full((2, max_len), 7.0, device="cuda")
    _lib.check(_lib.lib().riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), None, _lib.ptr(batch.n), 2, max_len,
                                          _lib.ptr(out), out.stride(0), None, _lib.stream_ptr()), "riser_normalise")
    out = out.cpu().numpy()
    assert np.array_equal(out[0], oracle32(sigs[0][:max_len]))
    assert np.array_equal(out[1, :5000], oracle32(sigs[1])) and np.all(out[1, 5000:] == 7.0)
