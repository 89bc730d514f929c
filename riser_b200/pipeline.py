"""Batched trim -> normalise -> classify -> decide pipeline: the additive surface the
rewritten ReadUntil loop calls once per ``get_read_batch()`` (SURVEY.md 8b), replacing
the serial per-read body of riser/control.py:31-93.

Everything between the H2D copy of the packed signals (int16 ADC counts, or float32
calibrated signal with ``signal_dtype=np.float32``) and the D2H copy of the decision
bytes / probabilities runs in the sm_100a kernels behind the C ABI, on the current CUDA
stream, with one host synchronisation per batch.
"""
import os

import numpy as np
import torch

from . import _lib
from .preprocess import RaggedBatch, PinnedArena, _hostpack, signal_dtype as _dtype_of
from .model import decide, DEFAULT_CHUNK

_EMPTY = np.zeros(0, dtype=np.int16)
_EMPTY_F32 = np.zeros(0, dtype=np.float32)

# decision codes (include/riser_b200.h)
TRY_AGAIN, ACCEPT, REJECT, NO_DECISION, SKIPPED = 0, 1, 2, 3, 4
DECISION_NAMES = {TRY_AGAIN: "try_again", ACCEPT: "accept", REJECT: "reject",
                  NO_DECISION: "no_decision", SKIPPED: "skipped"}


def bucket_size(n):
    """Batch sizes are rounded up to 64, 96, 128, 192, 256, 384, ... (powers of two and 1.5 x powers
    of two) so that a live run, whose batch size changes every poll, reuses a handful of plans
    and buffers instead of building new ones; the padding reads have length 0 and cost nothing
    (their tiles are skipped)."""
    b = 64
    while True:
        if n <= b:
            return b
        if n <= b + b // 2:
            return b + b // 2
        b *= 2


def upload_ranges(n, cached_end, min_len, max_len):
    """Which samples of each read the device will look at (int64 skip / take per read).  A read whose poly(A) end
    is cached needs no detection and its window is signal[end + 1 : end + 1 + max_len] when at least min_len
    samples follow the end, nothing otherwise (control.py:36-60 / preprocess.py:87-102 -- the integers
    select_window_kernel computes); a read without a cached end is needed whole (detection, or the fixed trim)."""
    n = np.asarray(n, dtype=np.int64)
    cached_end = np.asarray(cached_end)
    has = cached_end >= 0
    skip = np.where(has, cached_end.astype(np.int64) + 1, 0)
    avail = n - skip
    take = np.where(has, np.where(avail >= min_len, np.minimum(avail, max_len), 0), n)
    return skip, take


class BatchResult:
    """Host-side result of one batch: ``decisions`` uint8 [B], ``p_on`` / ``p_off``
    float32 [B, M], ``sig_len`` int32 [B] (post-trim window length, 0 = skipped),
    ``polya_end`` int32 [B] (-1 = none)."""
    __slots__ = ("decisions", "p_on", "p_off", "sig_len", "polya_end", "h2d_bytes", "d2h_bytes")


class BatchedClassifier:
    def __init__(self, models, processor, chunk=None, signal_dtype=np.int16):
        """``signal_dtype``: what the ReadUntil client hands over (riser/client.py:47).  np.int16 (raw ADC counts,
        the default): integer prefixes are packed as int16, float ones refused.  np.float32 (calibrated signal):
        float32 prefixes only; poly(A) detection and normalisation run in float32 as numpy does for such input
        (riser_polya_end_f32, riser_normalise_f32_live)."""
        self.signal_dtype = np.dtype(signal_dtype)
        if self.signal_dtype not in (np.int16, np.float32):
            raise TypeError(f"BatchedClassifier classifies int16 or float32 signal, not {self.signal_dtype}")
        self.f32 = self.signal_dtype == np.float32
        self.models = list(models)
        self.proc = processor
        self.device = _lib.require_device()
        self.chunk = int(chunk or DEFAULT_CHUNK or 0)
        self.min_len = processor.get_min_length()
        self.max_len = processor.get_max_length()
        self.fixed_trim = processor.get_fixed_trim_length()
        self.ld = (self.max_len + 3) & ~3
        self._bufs = {}
        self._arena = PinnedArena(self.device, dtype=torch.float32 if self.f32 else torch.int16)
        self._graphs = {}
        self.use_graphs = os.environ.get("RISER_LIVE_GRAPHS", "1") != "0"

    # ------------------------------------------------------------------ device stages
    def _buffers(self, B):
        b = self._bufs.get(B)
        if b is None:
            dev, M = self.device, len(self.models)
            b = self._bufs[B] = {
                "x": torch.zeros(B, self.ld, dtype=torch.float32, device=dev),
                "start": torch.zeros(B, dtype=torch.int32, device=dev),
                "len": torch.zeros(B, dtype=torch.int32, device=dev),
                "probs": torch.zeros(M, B, 2, dtype=torch.float32, device=dev),
                "detected": torch.full((B,), -1, dtype=torch.int32, device=dev),
                "out_host": torch.empty(B * (1 + 4 + 4 + 8 * M), dtype=torch.uint8).pin_memory(),
            }
        return b

    def run_windows(self, batch, start, length, threshold, mode, events=None):
        """normalise + classify (every model) + decide for windows already chosen.
        batch: RaggedBatch; start / length: int32 device tensors [B] (length 0 = skip).
        Returns (decisions uint8 [B], probs fp32 [M, B, 2]) on the device."""
        B = batch.B
        buf = self._buffers(B)
        L = _lib.lib()
        if batch.sig.dtype == torch.float32:
            # the float32 normaliser takes each window's own start: off + start
            win_off = batch.off[:B] + start
            _lib.check(L.riser_normalise_f32_live(_lib.ptr(batch.sig), _lib.ptr(win_off), _lib.ptr(length), B,
                                                  self.max_len, _lib.ptr(buf["x"]), buf["x"].stride(0), None,
                                                  _lib.stream_ptr()), "riser_normalise_f32_live")
        else:
            _lib.check(L.riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(start),
                                         _lib.ptr(length), B, self.max_len, _lib.ptr(buf["x"]), buf["x"].stride(0),
                                         None, _lib.stream_ptr()), "riser_normalise")
        for m, model in enumerate(self.models):
            model.classify_batch(buf["x"], length, max_len=self.max_len, probs=buf["probs"][m],
                                 chunk=self.chunk, events=events)
        decisions = decide(buf["probs"], length, threshold, mode, self.max_len)
        return decisions, buf["probs"]

    def select_windows(self, batch, cached_end):
        """poly(A) detection for reads without a cached end + control.py:36-60 gating.
        cached_end: int32 [B] (-1 = not cached), host array or device tensor.  Device tensors out."""
        B = batch.B
        buf = self._buffers(B)
        L = _lib.lib()
        cached = cached_end if torch.is_tensor(cached_end) else torch.from_numpy(
            np.ascontiguousarray(cached_end, dtype=np.int32)).to(self.device, non_blocking=True)
        # detection is only needed where nothing is cached; reads with a cache hit keep -1
        # (their prefix is skipped by giving them length 0 in the detection launch)
        n_detect = torch.where(cached >= 0, torch.zeros_like(batch.n), batch.n)
        fn, name = ((L.riser_polya_end_f32, "riser_polya_end_f32") if batch.sig.dtype == torch.float32 else
                    (L.riser_polya_end, "riser_polya_end"))
        _lib.check(fn(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(n_detect), B, _lib.ptr(buf["detected"]),
                      None, None, 0, _lib.stream_ptr()), name)
        _lib.check(L.riser_select_window(_lib.ptr(batch.n), _lib.ptr(cached), _lib.ptr(buf["detected"]), B,
                                         self.min_len, self.max_len, self.fixed_trim, _lib.ptr(buf["start"]),
                                         _lib.ptr(buf["len"]), _lib.stream_ptr()), "riser_select_window")
        return buf["start"], buf["len"], buf["detected"]

    @staticmethod
    def _as_int16(signals):
        """The batched path packs raw int16 ADC samples (riser/client.py:47: np.frombuffer(raw_data, signal_dtype)
        with the ReadUntil default, uncalibrated signal).  The dtype is looked at once per poll, on the first
        non-empty read: other integer dtypes are converted, a client configured for calibrated (float) signal is
        refused -- packing float bytes as int16 would classify garbage silently."""
        for s in signals:
            if len(s):
                dt = getattr(s, "dtype", None)
                if dt == np.int16:
                    return signals
                if dt is not None and dt.kind in "iu":
                    return [np.ascontiguousarray(x, dtype=np.int16) for x in signals]
                raise TypeError(f"BatchedClassifier.classify_batch needs raw int16 signal, got {dt}: run the "
                                "ReadUntil client with calibrated_signal=False (the default), or use "
                                "SignalProcessor.mad_normalise + Model.classify for float signal")
        return signals

    @staticmethod
    def _as_float32(signals):
        """Calibrated mode: every prefix must be float32 (np.frombuffer(raw_data, float32) of a client run with
        calibrated signal); anything else would be misread."""
        if _dtype_of(signals) != np.float32:
            raise TypeError("this BatchedClassifier was built for calibrated float32 signal: use one with "
                            "signal_dtype=np.int16 for raw signal")
        return signals

    # ------------------------------------------------------------------ public entry
    def classify_batch(self, signals, read_ids, polyA_cache, threshold, mode):
        """One pass of riser/control.py:31-97 over a batch.

        signals: list of int16 (float32 in calibrated mode) arrays (the whole accumulated prefix of each read, as
        ``client.get_raw_signal`` returns it); read_ids: matching ids; polyA_cache: the
        loop's dict (updated here exactly as control.py does: found ends are stored, and
        the dict is cleared when it reaches 1000 entries after an assessed read).
        Returns a BatchResult with host arrays."""
        B = len(signals)
        res = BatchResult()
        M = len(self.models)
        if B == 0:
            res.decisions = np.zeros(0, np.uint8)
            res.p_on = res.p_off = np.zeros((0, M), np.float32)
            res.sig_len = res.polya_end = np.zeros(0, np.int32)
            res.h2d_bytes = res.d2h_bytes = 0
            return res
        n_real = B
        signals = self._as_float32(signals) if self.f32 else self._as_int16(signals)
        B = bucket_size(n_real)                       # pad with empty reads up to the bucket
        cached = np.full(B, -1, dtype=np.int32)
        cached[:n_real] = np.fromiter((polyA_cache.get(r, -1) for r in read_ids), dtype=np.int32, count=n_real)
        if B > n_real:
            signals = list(signals) + [_EMPTY_F32 if self.f32 else _EMPTY] * (B - n_real)
        # size the staging arena once for the longest prefixes the loop can hand over (a read is
        # classified, at the latest, once it exceeds fixed trim + max length: control.py:42-46)
        self._arena.reserve(B * (self.fixed_trim + self.max_len + 8192), B)
        # Upload only what the kernels will look at.  A read whose poly(A) end is cached needs no detection, and its
        # window is known on the host (control.py:36-56, same integers as select_window_kernel): the max_len samples
        # after the end -- or nothing, while fewer than min_len samples follow it.  Reads without a cached end go up
        # whole (detection scans the whole prefix).
        n_all = np.zeros(B, dtype=np.int64)
        _hostpack().lengths(signals, n_all)
        n_all //= self.signal_dtype.itemsize
        skip, take = upload_ranges(n_all, cached, self.min_len, self.max_len)
        batch = RaggedBatch(signals, self.device, arena=self._arena, skip=skip, take=take, trusted=True,
                            extra_i32=cached, dtype=self.signal_dtype)
        # packed pinned result buffer: len | detected | probs | decisions (4-byte fields first)
        buf = self._buffers(B)
        host = buf["out_host"]
        o0, o1, o2 = 4 * B, 8 * B, 8 * B + 8 * M * B

        def device_stage():
            start, length, detected = self.select_windows(batch, batch.extra)
            decisions, probs = self.run_windows(batch, start, length, threshold, mode)
            host[:o0].view(torch.int32).copy_(length, non_blocking=True)
            host[o0:o1].view(torch.int32).copy_(detected, non_blocking=True)
            host[o1:o2].view(torch.float32).view(M, B, 2).copy_(probs, non_blocking=True)
            host[o2:].copy_(decisions, non_blocking=True)

        # Everything between the H2D copies and the host synchronisation is the same kernel sequence on the same
        # buffers for every poll of a batch-size bucket (the arena, the metadata block and the per-bucket buffers
        # keep their addresses; ragged lengths live in device memory): it is captured into a CUDA graph the second
        # time a bucket is seen and replayed from then on -- one launch instead of ~20 per model.
        key = (B, float(threshold), mode, self._arena.generation)
        g = self._graphs.get(key)
        if g is not None:
            g.replay()
        else:
            device_stage()                                   # first poll of a bucket: plans, attributes, buffers
            if self.use_graphs:                              # ... and its graph, so that only this poll is slow
                torch.cuda.current_stream().synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    device_stage()
                if len(self._graphs) > 64:                   # stale arena generations / thresholds
                    self._graphs = {k: v for k, v in self._graphs.items() if k[3] == self._arena.generation}
                self._graphs[key] = g
        torch.cuda.current_stream().synchronize()
        hv = host.numpy()
        res.sig_len = hv[:o0].view(np.int32)[:n_real].copy()
        det = hv[o0:o1].view(np.int32)[:n_real].copy()
        pr = hv[o1:o2].view(np.float32).reshape(M, B, 2)[:, :n_real]
        res.decisions = hv[o2:o2 + n_real].copy()
        res.p_off = np.ascontiguousarray(pr[:, :, 0].T)
        res.p_on = np.ascontiguousarray(pr[:, :, 1].T)
        cached = cached[:n_real]
        B = n_real
        res.polya_end = np.where(cached >= 0, cached, det)
        res.h2d_bytes = batch.h2d_bytes + cached.nbytes
        res.d2h_bytes = host.numel()
        # cache bookkeeping in read order (preprocess.py:93-98, control.py:96-97)
        new = np.flatnonzero((cached < 0) & (det > 0))
        if len(polyA_cache) + len(new) < 1000:
            # the cache cannot reach 1000 entries during this batch: no wipe, order does not matter
            for r in new:
                polyA_cache[read_ids[r]] = int(det[r])
        else:
            for r in range(B):
                if cached[r] < 0 and det[r] > 0:
                    polyA_cache[read_ids[r]] = int(det[r])
                if res.decisions[r] != SKIPPED and len(polyA_cache) >= 1000:
                    polyA_cache.clear()
        return res


def _warm_up(self, batch_sizes, threshold, mode):
    """Build the launch plans, buffers and CUDA graphs of the given batch-size buckets before the run starts, so
    that no live poll pays for them (a 512-read bucket costs ~0.1 s the first time it is seen).  Uses empty
    reads: every window is skipped, the kernels run on zero-length work."""
    for n in sorted(set(bucket_size(int(b)) for b in batch_sizes)):
        self._arena.reserve(n * (self.fixed_trim + self.max_len + 8192), n)
    for n in sorted(set(bucket_size(int(b)) for b in batch_sizes)):
        self.classify_batch([_EMPTY_F32 if self.f32 else _EMPTY] * n, [f"warm-up-{i}" for i in range(n)], {},
                            threshold, mode)


BatchedClassifier.warm_up = _warm_up


class FixedBatchPipeline:
    """Double-buffered host -> device -> host pipeline for fixed-shape batches of
    already-trimmed chunks (BASELINE config 2 / offline throughput): the H2D copy of
    batch k+1 (copy stream) overlaps the kernels of batch k (compute stream); results
    (decision bytes + probabilities) come back through pinned buffers.

        pipe = FixedBatchPipeline(clf, B, L, threshold=0.9, mode="deplete")
        t = pipe.submit(host_int16)          # pinned int16 [B, L]; returns immediately
        decisions, probs = pipe.result(t)    # numpy views, valid until the slot is reused
    """
    def __init__(self, clf, B, L, threshold, mode, slots=2, use_graph=True):
        self.clf, self.B, self.L = clf, int(B), int(L)
        self.use_graph = use_graph
        self.threshold, self.mode = threshold, mode
        dev, M = clf.device, len(clf.models)
        self.copy_stream = torch.cuda.Stream(device=dev)
        padded = (self.L + 7) & ~7
        off = torch.arange(self.B + 1, dtype=torch.int64) * padded
        self.start = torch.zeros(self.B, dtype=torch.int32, device=dev)
        self.length = torch.full((self.B,), self.L, dtype=torch.int32, device=dev)
        self.slots = []
        for _ in range(slots):
            batch = RaggedBatch.__new__(RaggedBatch)
            batch.B = self.B
            batch.n_host = np.full(self.B, self.L, dtype=np.int32)
            batch.sig = torch.zeros(self.B * padded + 8, dtype=torch.int16, device=dev)
            batch.off = off.to(dev)
            batch.n = self.length
            batch.h2d_bytes = self.B * self.L * 2
            self.slots.append({
                "batch": batch, "padded": padded,
                "copied": torch.cuda.Event(), "done": torch.cuda.Event(),
                "dec": torch.empty(self.B, dtype=torch.uint8).pin_memory(),
                "probs": torch.empty(M, self.B, 2, dtype=torch.float32).pin_memory(),
                "busy": False, "graph": None, "g_dec": None, "g_probs": None,
            })
        self.n_submitted = 0
        self.h2d_bytes = self.B * self.L * 2
        self.d2h_bytes = self.B * (1 + 8 * M)

    def submit(self, host):
        slot = self.slots[self.n_submitted % len(self.slots)]
        compute = torch.cuda.current_stream()
        if slot["busy"]:
            self.copy_stream.wait_event(slot["done"])      # the slot's previous batch has been consumed
        with torch.cuda.stream(self.copy_stream):
            dst = slot["batch"].sig[:self.B * slot["padded"]].view(self.B, slot["padded"])[:, :self.L]
            dst.copy_(host, non_blocking=True)
            slot["copied"].record(self.copy_stream)
        compute.wait_event(slot["copied"])
        if self.use_graph:
            decisions, probs = self._replay(slot)
        else:
            decisions, probs = self.clf.run_windows(slot["batch"], self.start, self.length, self.threshold,
                                                    self.mode)
        slot["dec"].copy_(decisions, non_blocking=True)
        slot["probs"].copy_(probs, non_blocking=True)
        slot["done"].record(compute)
        slot["busy"] = True
        self.n_submitted += 1
        return self.n_submitted - 1

    def _replay(self, slot):
        """The fixed-shape kernel sequence (normalise -> network per model -> decide) of a slot,
        captured once into a CUDA graph and replayed: one launch per batch instead of ~15 per
        model."""
        if slot["graph"] is None:
            args = (slot["batch"], self.start, self.length, self.threshold, self.mode)
            self.clf.run_windows(*args)                      # warm-up: plans, smem attributes
            torch.cuda.current_stream().synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                slot["g_dec"], slot["g_probs"] = self.clf.run_windows(*args)
            slot["graph"] = g
        slot["graph"].replay()
        return slot["g_dec"], slot["g_probs"]

    def result(self, ticket):
        slot = self.slots[ticket % len(self.slots)]
        slot["done"].synchronize()
        return slot["dec"].numpy(), slot["probs"].numpy()
