"""Host-side mirror of riser/preprocess.py (Kit, SignalProcessor) backed by the
sm_100a kernels in csrc/preprocess.cu.

The eight methods ``control.py`` calls keep the reference's names, arguments,
return types and error behaviour (riser/preprocess.py:29-115), so the object
drops in behind ``SequencerControl``; the additive ``*_batch`` methods are what
the batched loop (riser_b200/control.py) uses.  All arithmetic that produces
signal values runs on the GPU; there is no CPU fallback.
"""
import os

import numpy as np
import torch

from . import _lib

# riser/preprocess.py:6-12
_MIN_INPUT_SIGNALS = 4096
_MAX_INPUT_NT = 280
_TRIM_RESOLUTION = 500
_TRIM_FIXED_LENGTH_NT = 150.6


class Kit():
    """riser/preprocess.py:15-27."""
    def __init__(self, sampling_hz, transloc_rate):
        self.sampling_hz = sampling_hz
        self.transloc_rate = transloc_rate

    @classmethod
    def create_from_version(cls, version):
        if version == "RNA002":
            return cls(3012, 70)
        elif version == "RNA004":
            return cls(4000, 130)
        else:
            raise Exception(f"Invalid kit version {version}")


class PinnedArena:
    """Grow-only pinned host buffer + device buffer pair reused across batches (pinning and
    cudaMalloc per batch would dominate the latency of a live 512-read batch).  ``dtype``: the
    sample type of the signal buffers (int16 ADC counts, or float32 for calibrated signal)."""
    def __init__(self, device, dtype=torch.int16):
        self.device = device
        self.dtype = dtype
        self.capacity = 0
        self.host = self.dev = self.meta_host = self.meta_dev = None
        self.meta_capacity = 0
        self.generation = 0        # bumped whenever a buffer is re-allocated (captured graphs hold the old pointers)

    def reserve(self, n_samples, n_reads):
        if n_samples > self.capacity:
            self.capacity = int(n_samples * 1.25) + 4096
            self.host = torch.empty(self.capacity, dtype=self.dtype).pin_memory()
            self.dev = torch.empty(self.capacity, dtype=self.dtype, device=self.device)
            self.generation += 1
        if n_reads > self.meta_capacity:
            self.meta_capacity = int(n_reads * 1.25) + 64
            # int64 words: off [B+1], then n [B] and an optional extra int32 [B] (int32 pairs packed)
            self.meta_host = torch.empty(2 * self.meta_capacity + 4, dtype=torch.int64).pin_memory()
            self.meta_dev = torch.empty(2 * self.meta_capacity + 4, dtype=torch.int64, device=self.device)
            self.generation += 1


PACK_THREADS = int(os.environ.get("RISER_PACK_THREADS", max(1, min(4, (os.cpu_count() or 2) // 2))))
_hostpack_mod = None


def _hostpack():
    """The native gather of read prefixes (csrc/hostpack.c), loaded on first use like the CUDA library; there
    is no Python fallback."""
    global _hostpack_mod
    if _hostpack_mod is None:
        try:
            from . import _hostpack as mod
        except ImportError as e:
            raise RuntimeError("riser_b200/_hostpack is not built: run `python -m riser_b200.build`") from e
        _hostpack_mod = mod
    return _hostpack_mod


class RaggedBatch:
    """Reads packed back to back on the device: ``sig`` [total], ``off`` int64
    [B+1], ``n`` int32 [B].  Built from host arrays through one pinned staging
    buffer and one H2D copy (two with metadata); pass a ``PinnedArena`` to reuse buffers.

    The gather into the staging buffer is done by the native ``_hostpack`` module (buffer protocol +
    threads, csrc/hostpack.c).  ``skip`` / ``take`` (int64 sample counts per read, optional) upload only
    ``signal[skip:skip+take]`` of a read; ``off`` then holds the VIRTUAL start of the read (packed position
    - skip), so that ``sig[off[b] + i]`` is still sample i of read b for every i inside the uploaded slice
    and the kernels need not know.  ``n`` is always the full prefix length.
    ``trusted=True`` skips the per-read dtype / contiguity check (the live loop's arrays come straight from
    ``np.frombuffer(raw_data, int16)``).  ``extra_i32`` (arena path only): an int32 [B] host array uploaded with the
    metadata in the same copy, available as ``self.extra``.
    ``dtype``: the sample type, int16 (ADC counts, the default) or float32 (calibrated signal); with an arena it
    must be the arena's.  Every read starts on a 16-byte boundary: 8 int16 or 4 float32 samples."""
    def __init__(self, signals, device, arena=None, skip=None, take=None, trusted=False, extra_i32=None,
                 dtype=np.int16):
        B = len(signals)
        dtype = np.dtype(dtype)
        if dtype not in (np.int16, np.float32):
            raise TypeError(f"RaggedBatch packs int16 or float32 samples, not {dtype}")
        esz = dtype.itemsize
        align = 16 // esz
        tdtype = torch.int16 if dtype == np.int16 else torch.float32
        if arena is not None and arena.dtype != tdtype:
            raise TypeError(f"a {arena.dtype} arena cannot stage {dtype} samples")
        if not trusted:
            signals = [np.ascontiguousarray(s, dtype=dtype) for s in signals]
        nbytes = np.zeros(B, dtype=np.int64)
        hp = _hostpack()
        hp.lengths(signals, nbytes)
        n = nbytes // esz
        if take is None:
            skip = np.zeros(B, dtype=np.int64)
            take = n
        else:
            skip = np.ascontiguousarray(skip, dtype=np.int64)
            take = np.ascontiguousarray(take, dtype=np.int64)
        # keep every packed read 16-byte aligned so the kernels' vector loads need no peeling
        padded = (take + (align - 1)) & ~(align - 1)
        pos = np.zeros(B + 1, dtype=np.int64)
        np.cumsum(padded, out=pos[1:])
        total = int(pos[-1]) + align
        off = pos.copy()
        off[:B] -= skip
        self.B = B
        self.dtype = dtype
        self.n_host = n.astype(np.int32)
        byte_pos = np.ascontiguousarray(pos[:B] * esz)
        if arena is None:
            host = torch.empty(total, dtype=tdtype).pin_memory()
            hp.pack(signals, host.numpy(), byte_pos, skip * esz, take * esz, PACK_THREADS)
            self.sig = host.to(device, non_blocking=True)
            self.off = torch.from_numpy(off).to(device, non_blocking=True)
            self.n = torch.from_numpy(self.n_host).to(device, non_blocking=True)
            self._host = host      # keep the pinned buffer alive until the copy has run
        else:
            arena.reserve(total, B)
            hp.pack(signals, arena.host.numpy(), byte_pos, skip * esz, take * esz, PACK_THREADS)
            self.sig = arena.dev[:total]
            self.sig.copy_(arena.host[:total], non_blocking=True)
            mh = arena.meta_host.numpy()
            mh[:B + 1] = off
            half = (B + 1) // 2
            mh[B + 1:B + 1 + half].view(np.int32)[:B] = self.n_host
            words = B + 1 + half
            if extra_i32 is not None:
                mh[words:words + half].view(np.int32)[:B] = extra_i32
                words += half
            arena.meta_dev[:words].copy_(arena.meta_host[:words], non_blocking=True)
            self.off = arena.meta_dev[:B + 1]
            self.n = arena.meta_dev[B + 1:B + 1 + half].view(torch.int32)[:B]
            self.extra = None if extra_i32 is None else arena.meta_dev[B + 1 + half:B + 1 + 2 * half].view(torch.int32)[:B]
        self.h2d_bytes = total * esz + off.nbytes + self.n_host.nbytes


_F32 = np.dtype(np.float32)


def signal_dtype(signals):
    """The sample type a list of signals is packed as: float32 when every one is float32 (calibrated signal, kept in
    float32 as numpy keeps it), int16 when none is (other integer dtypes are converted); a mix raises TypeError."""
    dtypes = {getattr(s, "dtype", None) for s in signals}
    if _F32 not in dtypes:
        return np.dtype(np.int16)
    if len(dtypes) > 1:
        raise TypeError(f"float32 (calibrated) signal mixed with other dtypes: {sorted(map(str, dtypes))}")
    return _F32


_long_ws = {}       # device -> workspace of the long-window kernels, grown as needed; its users share one stream


def normalise_windows(sig, off, start, len_host, len_dev, out, stats=None, outlier_lim=3.5, live=True):
    """Median / MAD-normalise window b = ``sig[off[b] + start[b]:][:len_host[b]]`` into row b of ``out`` (fp32 [B, ld]),
    for int16 or float32 ``sig``.  ``start``: int32 device tensor (int16 only) or None; ``len_dev``: ``len_host`` on the
    device; ``stats`` (optional): {2 median, 4 MAD} int32 for int16, {median, MAD} float32 for live float32.  float32
    takes ``outlier_lim``, and ``live`` zeros windows whose MAD is 0 (else numpy's inf / nan, as retraining wants).
    Windows above the shared-memory kernels' limit go to ``riser_normalise_long`` / ``riser_normalise_f32_long`` (the
    same results), the rest to ``riser_normalise`` / ``riser_normalise_f32(_live)``; each launch sees the other's
    windows as length 0."""
    L, P = _lib.lib(), _lib.ptr
    f32 = sig.dtype == torch.float32
    assert not f32 or (start is None and (live or stats is None)), "no float32 kernel takes these arguments"
    B = len(len_host)
    max_len = int(len_host.max()) if B else 0
    if max_len <= 0:
        return
    limit = L.riser_normalise_f32_max_len() if f32 else L.riser_normalise_max_len()
    short_len = len_dev
    if max_len > limit:
        is_long = len_host > limit
        short_len = torch.from_numpy(np.where(is_long, 0, len_host).astype(np.int32)).to(sig.device)
        long_len = torch.from_numpy(np.where(is_long, len_host, 0).astype(np.int32)).to(sig.device)
        nbytes = max(L.riser_normalise_long_workspace_bytes(B, max_len), 16)
        ws = _long_ws.get(sig.device)
        if ws is None or ws.numel() < nbytes:
            ws = _long_ws[sig.device] = torch.empty(nbytes, dtype=torch.uint8, device=sig.device)
        if f32:
            _lib.check(L.riser_normalise_f32_long(P(sig), P(off), P(long_len), B, max_len, float(outlier_lim),
                                                  int(live), P(out), out.stride(0), P(stats), P(ws), ws.numel(),
                                                  _lib.stream_ptr()), "riser_normalise_f32_long")
        else:
            _lib.check(L.riser_normalise_long(P(sig), P(off), P(start), P(long_len), B, max_len, P(out),
                                              out.stride(0), P(stats), P(ws), ws.numel(), _lib.stream_ptr()),
                       "riser_normalise_long")
        max_len = limit
    if not f32:
        _lib.check(L.riser_normalise(P(sig), P(off), P(start), P(short_len), B, max_len, P(out), out.stride(0),
                                     P(stats), _lib.stream_ptr()), "riser_normalise")
    elif live:
        _lib.check(L.riser_normalise_f32_live(P(sig), P(off), P(short_len), B, max_len, P(out), out.stride(0),
                                              P(stats), _lib.stream_ptr()), "riser_normalise_f32_live")
    else:
        _lib.check(L.riser_normalise_f32(P(sig), P(off), P(short_len), B, max_len, float(outlier_lim), P(out),
                                         out.stride(0), _lib.stream_ptr()), "riser_normalise_f32")


class SignalProcessor():
    def __init__(self, kit):
        self.kit = kit

    # ------------------------------------------------------------ length gates
    def get_min_length(self):
        return _MIN_INPUT_SIGNALS

    def get_max_length(self):
        return int(_MAX_INPUT_NT / self.kit.transloc_rate * self.kit.sampling_hz)

    def is_max_length(self, signal):
        return len(signal) >= self.get_max_length()

    def get_fixed_trim_length(self):
        return int(_TRIM_FIXED_LENGTH_NT / self.kit.transloc_rate * self.kit.sampling_hz)

    def should_trim_fixed_length(self, signal):
        return len(signal) > self.get_fixed_trim_length() + self.get_max_length()

    def trim_polyA_fixed_length(self, signal):
        return signal[self.get_fixed_trim_length():]

    # ------------------------------------------------------------ poly(A)
    def get_polyA_end(self, signal):
        """riser/preprocess.py:42-79 -> int window-start index or None."""
        end = self.get_polyA_end_batch([signal])[0]
        return None if end < 0 else int(end)

    def trim_polyA(self, signal, read_id, cache):
        """riser/preprocess.py:87-102 (mutates the caller's cache)."""
        trimmed = False
        if read_id in cache:
            polyA_end = cache[read_id]
        else:
            polyA_end = self.get_polyA_end(signal)
            if polyA_end:
                cache[read_id] = polyA_end
        if polyA_end:
            signal = signal[polyA_end + 1:]
            trimmed = True
        return signal, trimmed

    def get_polyA_end_batch(self, signals, return_stats=False):
        """Batched get_polyA_end: list of arrays -> int32 [B] (-1 = None).

        float32 arrays (calibrated signal) go to ``riser_polya_end_f32``, which computes the window statistics in
        float32 as numpy does for them; every other dtype is cast to int16 (``riser_polya_end``).  A list that
        mixes float32 with other dtypes raises TypeError."""
        device = _lib.require_device()
        if not isinstance(signals, RaggedBatch) and len(signals) == 0:
            return np.zeros(0, dtype=np.int32)
        if isinstance(signals, RaggedBatch):
            batch = signals
        else:
            dtype = signal_dtype(signals)
            batch = RaggedBatch([np.ascontiguousarray(s, dtype=dtype) for s in signals], device, dtype=dtype)
        ends = self.polya_end_device(batch, return_stats=return_stats)
        if return_stats:
            return ends[0].cpu().numpy(), ends[1].cpu().numpy()
        return ends.cpu().numpy()

    def polya_end_device(self, batch, return_stats=False, starts=None):
        """Detection on a RaggedBatch already on the device.  stats (``return_stats``): int32 [B, W, 3] =
        {sum, 2 * median, 4 * MAD} per window for int16 reads, float32 [B, W, 4] = {median, MAD, mean,
        rolling mean} for float32 reads."""
        ends = torch.empty(batch.B, dtype=torch.int32, device=batch.sig.device)
        f32 = batch.sig.dtype == torch.float32
        stats, max_w = None, 0
        if return_stats:
            max_w = max(1, int(batch.n_host.max()) // _TRIM_RESOLUTION)
            stats = torch.zeros(batch.B, max_w, 4 if f32 else 3, dtype=torch.float32 if f32 else torch.int32,
                                device=batch.sig.device)
        fn, name = ((_lib.lib().riser_polya_end_f32, "riser_polya_end_f32") if f32 else
                    (_lib.lib().riser_polya_end, "riser_polya_end"))
        _lib.check(fn(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(batch.n), batch.B, _lib.ptr(ends),
                      _lib.ptr(starts), _lib.ptr(stats), max_w, _lib.stream_ptr()), name)
        return (ends, stats) if return_stats else ends

    # ------------------------------------------------------------ normalise
    def mad_normalise(self, signal):
        """riser/preprocess.py:108-115.  Raises ValueError on empty input.

        int16 (what ``client.get_raw_signal`` hands over, riser/client.py:47), any other integer dtype and
        float64 holding integers in the int16 range: numpy works in float64 there and so does ``riser_normalise``
        -- the float64 ndarray returned is the reference's result rounded to fp32 (the cast riser/model.py:25
        applies anyway).  float32 (calibrated signal, the secondary input mode): numpy keeps float32 for the
        median, the MAD, the division and the smoothing, and ``riser_normalise_f32_live`` reproduces that bit
        for bit; a float32 ndarray is returned, as the reference does.  Non-integral float64 takes the float32
        route (1e-7-relative, inside the 1e-6 bar; the reference would stay in float64).  MAD == 0 returns
        int64 zeros like the reference (``np.vectorize`` types its output by the first element, the int 0 of
        preprocess.py:123)."""
        signal = np.asarray(signal)
        if signal.ndim != 1:
            raise ValueError(f"expected a 1-D signal, got shape {signal.shape}")
        n = signal.shape[0]
        if n == 0:
            raise ValueError("Signal must not be empty")
        if signal.dtype != np.int16:
            as16 = None
            if signal.dtype.kind in "iub":
                if signal.min() >= -32768 and signal.max() <= 32767:
                    as16 = signal.astype(np.int16)
            elif signal.dtype == np.float64:
                r = np.rint(signal)
                if np.array_equal(r, signal) and r.min() >= -32768 and r.max() <= 32767:
                    as16 = r.astype(np.int16)
            elif signal.dtype.kind != "f":
                raise TypeError(f"cannot normalise a signal of dtype {signal.dtype}")
            if as16 is None:
                return self._mad_normalise_f32(signal.astype(np.float32))
            signal = as16
        out, _, stats = self.mad_normalise_batch([signal], return_stats=True)
        if int(stats[0, 1]) == 0:                      # 4 * MAD
            return np.zeros(n, dtype=np.int64)
        return out[0, :n].double().cpu().numpy()

    def _mad_normalise_f32(self, signal):
        device = _lib.require_device()
        n = signal.shape[0]
        sig = torch.from_numpy(np.ascontiguousarray(signal)).to(device)
        off = torch.tensor([0, n], dtype=torch.int64, device=device)
        ln = torch.tensor([n], dtype=torch.int32, device=device)
        out = torch.empty(1, n, dtype=torch.float32, device=device)
        med_mad = torch.empty(1, 2, dtype=torch.float32, device=device)
        normalise_windows(sig, off, None, np.array([n], dtype=np.int32), ln, out, med_mad)
        if float(med_mad[0, 1]) == 0.0:
            return np.zeros(n, dtype=np.int64)
        return out[0].cpu().numpy()

    def mad_normalise_batch(self, signals, start=None, length=None, out=None, return_stats=False):
        """Batched mad_normalise over ragged int16 windows.

        signals: list of int16 arrays, or a RaggedBatch already on the device.
        start / length (optional int32 arrays): window of each read
        (``sig[start:start+length]``); default the whole read.
        Returns (out fp32 [B, ld] on the device, lengths int32 device tensor).

        Windows of any length: ``normalise_windows`` routes them by length."""
        device = _lib.require_device()
        batch = signals if isinstance(signals, RaggedBatch) else RaggedBatch(
            [np.ascontiguousarray(s, dtype=np.int16) for s in signals], device)
        if length is None:
            len_host = batch.n_host if start is None else batch.n_host - np.asarray(start, dtype=np.int32)
        else:
            len_host = np.asarray(length, dtype=np.int32)
        max_len = int(len_host.max()) if batch.B else 0
        ld = (max_len + 3) & ~3
        if out is None:
            out = torch.zeros(batch.B, max(ld, 4), dtype=torch.float32, device=device)
        start_t = None if start is None else torch.as_tensor(np.asarray(start, dtype=np.int32)).to(device)
        len_t = batch.n if (length is None and start is None) else torch.from_numpy(len_host).to(device)
        stats = torch.zeros(batch.B, 2, dtype=torch.int32, device=device) if return_stats else None
        normalise_windows(batch.sig, batch.off, start_t, len_host, len_t, out, stats)
        if return_stats:
            return out, len_t, stats
        return out, len_t
