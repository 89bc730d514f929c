"""Training-data preparation with riser/retrain/preprocess.py semantics (SURVEY.md 8f-4):
keep the first ``n_secs * freq`` samples of every pA-scaled (float32) read, discard shorter
reads, median/MAD-normalise and smooth outliers in float32, and stack the results -- the array
``retrain/preprocess.py:97`` saves as ``<name>_<cutoff>.npy`` (fast5 I/O is out of scope: reads
come from any iterable of float32 arrays)."""
import numpy as np
import torch

from . import _lib


def mad_normalise_f32_batch(signals, outlier_lim=3.5):
    """Batched retrain/preprocess.py:8-15 over a list of float32 arrays.  Returns an fp32
    [B, ld] device tensor and the int32 lengths (device).  Reads longer than
    ``riser_normalise_f32_max_len()`` go to ``riser_normalise_f32_long`` (same results), the rest to
    ``riser_normalise_f32``, each launch seeing the other's reads as length 0."""
    device = _lib.require_device()
    B = len(signals)
    n = np.fromiter((len(s) for s in signals), dtype=np.int64, count=B)
    if (n == 0).any():
        raise ValueError("Signal must not be empty")
    off = np.zeros(B + 1, dtype=np.int64)
    np.cumsum(n, out=off[1:])
    host = torch.empty(int(off[-1]), dtype=torch.float32).pin_memory()
    hv = host.numpy()
    for s, o, k in zip(signals, off[:-1], n):
        hv[o:o + k] = np.asarray(s, dtype=np.float32)
    max_len = int(n.max())
    limit = _lib.lib().riser_normalise_f32_max_len()
    sig = host.to(device, non_blocking=True)
    off_d = torch.from_numpy(off).to(device)
    len_d = torch.from_numpy(n.astype(np.int32)).to(device)
    out = torch.zeros(B, max_len, dtype=torch.float32, device=device)
    short_d = len_d
    if max_len > limit:
        is_long = n > limit
        short_d = torch.from_numpy(np.where(is_long, 0, n).astype(np.int32)).to(device)
        long_d = torch.from_numpy(np.where(is_long, n, 0).astype(np.int32)).to(device)
        nbytes = _lib.lib().riser_normalise_long_workspace_bytes(B, max_len)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _lib.check(_lib.lib().riser_normalise_f32_long(_lib.ptr(sig), _lib.ptr(off_d), _lib.ptr(long_d), B, max_len,
                                                       float(outlier_lim), 0, _lib.ptr(out), out.stride(0), None,
                                                       _lib.ptr(ws), nbytes, _lib.stream_ptr()),
                   "riser_normalise_f32_long")
        max_len = limit
    _lib.check(_lib.lib().riser_normalise_f32(_lib.ptr(sig), _lib.ptr(off_d), _lib.ptr(short_d), B, max_len,
                                              float(outlier_lim), _lib.ptr(out), out.stride(0),
                                              _lib.stream_ptr()), "riser_normalise_f32")
    return out, len_d


def preprocess_reads(reads_pA, n_secs, freq, outlier_lim=3.5, batch=512):
    """retrain/preprocess.py:47-99 without the fast5 reader: -> (float32 [N, cutoff] ndarray,
    number of discarded reads)."""
    cutoff = int(freq) * int(n_secs)
    kept = [np.asarray(r, dtype=np.float32)[:cutoff] for r in reads_pA if len(r) >= cutoff]   # :79-83
    n_discarded = sum(1 for r in reads_pA if len(r) < cutoff)
    rows = []
    for lo in range(0, len(kept), batch):
        out, _ = mad_normalise_f32_batch(kept[lo:lo + batch], outlier_lim)
        rows.append(out[:, :cutoff].cpu().numpy())
    data = np.concatenate(rows) if rows else np.zeros((0, cutoff), dtype=np.float32)
    return data, n_discarded
