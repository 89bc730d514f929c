"""Synthetic stand-in for the MinKNOW / ReadUntil client (riser/client.py).

The reference's ``Client`` wraps the third-party ``read_until`` package, which is
out of scope and unavailable offline; the north star says it is "exercised
against synthetic signal".  ``SimClient`` offers the same methods
``SequencerControl`` calls (riser/client.py:33-62, riser/control.py:12,25,31,33,
100,106,119,127,131) and reproduces the AccumulatingCache semantics
(riser/client.py:29-31,44): every poll returns, per channel, the WHOLE prefix of
the current read so far, and the prefix grows by ``chunk`` samples per poll.
"""
import numpy as np


class SimRead:
    """What ``get_read_chunks`` yields: ``.id``, ``.raw_data`` (bytes), ``.number``."""
    __slots__ = ("id", "number", "raw_data")

    def __init__(self, read_id, number, raw_data):
        self.id = read_id
        self.number = number
        self.raw_data = raw_data


class SimClient:
    signal_dtype = np.int16

    def __init__(self, reads, chunk, n_polls, first_len=None, with_number=True):
        """reads: list of (read_id, full signal); channel c (1-based) carries
        reads[c-1].  Each poll exposes ``first_len + k*chunk`` samples (capped at the
        read's length).  After ``n_polls`` polls ``is_running`` turns False.
        ``signal_dtype`` is that of the reads: int16 (raw ADC counts) or float32
        (calibrated pA, what a client run with calibrated signal hands over)."""
        self.reads = reads
        if reads:
            self.signal_dtype = np.asarray(reads[0][1]).dtype
        self.chunk = int(chunk)
        self.first_len = int(first_len if first_len is not None else chunk)
        self.n_polls = int(n_polls)
        self.poll = 0
        self.done = set()          # (channel, id-or-number) passed to stop_receiving
        self.unblocked = []        # every (channel, id) ever passed to unblock
        self.finished = []
        self.messages = []
        self.running = False
        self.with_number = with_number

    # riser/client.py:33-41
    def start_streaming_reads(self):
        self.running = True

    def is_running(self):
        return self.running and self.poll < self.n_polls

    # riser/client.py:43-47
    def get_read_batch(self):
        n = self.first_len + self.poll * self.chunk
        self.poll += 1
        batch = []
        for c, (rid, sig) in enumerate(self.reads, start=1):
            key = (c, c if self.with_number else rid)
            if key in self.done:
                continue
            batch.append((c, SimRead(rid, c if self.with_number else None, sig[:n].tobytes())))
        if not self.with_number:
            for _, r in batch:
                del r.number
        return batch

    def get_raw_signal(self, read):
        return np.frombuffer(read.raw_data, self.signal_dtype)

    # riser/client.py:49-56
    def reject_reads(self, reads, unblock_duration):
        if reads:
            self.unblocked.extend(reads)

    def finish_processing_reads(self, reads):
        if reads:
            self.finished.extend(reads)
            self.done.update(reads)

    def reset(self):
        self.running = False

    def send_warning(self, message):
        self.messages.append(message)


class LiveSimClient(SimClient):
    """Flow-cell-like simulation for latency runs (BASELINE config 5): ``channels``
    pores draw reads from a pool; every poll each active read's prefix grows by ``chunk``
    samples; when a read is finished (unblocked / stop_receiving) or runs out of signal,
    its channel starts the next read of the pool.  Same method surface as ``Client``."""
    def __init__(self, pool, channels, chunk, n_polls, first_len=None):
        super().__init__(pool, chunk, n_polls, first_len=first_len)
        self.channels = int(channels)
        self.next_read = 0
        self.state = {}                       # channel -> [pool index, samples exposed, read number]
        self.read_counter = 0
        for c in range(1, self.channels + 1):
            self._start(c)

    def _start(self, c):
        self.read_counter += 1
        self.state[c] = [self.next_read % len(self.reads), self.first_len, self.read_counter]
        self.next_read += 1

    def get_read_batch(self):
        self.poll += 1
        batch = []
        for c in range(1, self.channels + 1):
            idx, n, number = self.state[c]
            rid, sig = self.reads[idx]
            if (c, number) in self.done or n > len(sig):
                self._start(c)
                idx, n, number = self.state[c]
                rid, sig = self.reads[idx]
            batch.append((c, SimRead(f"{rid}#{number}", number, sig[:n].tobytes())))
            self.state[c][1] = n + self.chunk
        return batch


def calibrate(reads, scale, offset):
    """Calibrated (pA) float32 copies of int16 reads, ``(adc + offset) * scale`` in float32 -- what a ReadUntil client
    run with calibrated signal hands over."""
    s, o = np.float32(scale), np.float32(offset)
    return [(rid, ((sig.astype(np.float32) + o) * s).astype(np.float32)) for rid, sig in reads]


def measure_latency(channels, polls, kit_version="RNA002", targets=("mRNA",), seed=7, skip=5, pool_reads=None,
                    precision=None, calibration=None):
    """BASELINE config 5: ``channels`` pores, every poll each live read's prefix grows by one second of samples
    (AccumulatingCache semantics, riser/client.py:29-31,44); the batched ``SequencerControl`` classifies every
    poll.  Returns p50 / p99 of the time from "batch in hand" to "decisions on host" over the polls after the
    first ``skip`` (the ReadUntil decision budget is ~1 s), with the run's counters.  ``calibration`` = (scale,
    offset): the client hands over calibrated float32 signal, ``(adc + offset) * scale``, instead of int16."""
    import logging
    import os
    import tempfile

    from . import Kit, SignalProcessor, Model, SequencerControl, synth
    from .config import shipped_config
    log = logging.getLogger("riser_b200.sim")
    kit = Kit.create_from_version(kit_version)
    kw = {} if precision is None else {"precision": precision}
    models = [Model(synth.state_dict(synth.TARGET_SEEDS[t]), shipped_config(), log, t, **kw) for t in targets]
    n_pool = int(pool_reads or min(2 * channels, 2048))
    reads = synth.raw_reads(seed, n_pool, min_body=14000, max_body=20000, frac_no_polya=0.05)
    if calibration is not None:
        reads = calibrate(reads, *calibration)
    client = LiveSimClient(reads, channels, chunk=kit.sampling_hz, n_polls=polls, first_len=kit.sampling_hz)
    with tempfile.TemporaryDirectory() as tmp:
        control = SequencerControl(client, models, SignalProcessor(kit), log, os.path.join(tmp, "live"),
                                   warm_up_batches=(channels,))
        control.start()
        control.target("deplete", 1, 0.9)
        control.finish()
        with open(os.path.join(tmp, "live.csv")) as f:
            rows = sum(1 for _ in f) - 1
    lat = np.array(control.batch_latencies) * 1e3
    steady = lat[skip:] if len(lat) > skip + 3 else lat
    out = {"channels": int(channels), "models": len(targets), "kit": kit_version, "polls": int(len(lat)),
            "p50_ms": round(float(np.median(steady)), 3), "p99_ms": round(float(np.percentile(steady, 99)), 3),
            "max_ms": round(float(steady.max()), 3), "batch_size_median": int(np.median(control.batch_sizes)),
            "assessed_rows": rows, "rejected": len(client.unblocked), "finished": len(client.finished)}
    if calibration is not None:
        out["calibration"] = [float(calibration[0]), float(calibration[1])]
    return out
