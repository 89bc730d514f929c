"""numpy reference for calibrated (float32 pA) input, used by the calibrated-signal tests.

With float32 input numpy keeps every step of riser/preprocess.py in float32: the poly(A) window statistics
(42-79) and the normalisation (108-147).  ``oracle.preprocess_oracle`` restates the reference for the int16 path
in float64, so the float32 evaluation lives here, built from the same oracle functions where they apply."""
import numpy as np

from oracle import control_oracle as ctl
from oracle import convnet_oracle as net
from oracle import preprocess_oracle as pp


def polya_window_stats(signal):
    """The per-window values preprocess.py:42-79 compares, as numpy computes them for ``signal``'s dtype: float64
    [n_windows, 4] = median, MAD, mean, rolling mean (the window's own mean for the first three windows).  Holds the
    float32 values exactly for float32 input."""
    res = pp.TRIM_RESOLUTION
    rows = []
    for i in range(0, len(signal) - res + 1, res):
        w = signal[i:i + res]
        med = np.median(w)
        mean = np.mean(w)
        rows.append((med, pp.window_mad(w, med), mean, np.mean(signal[i - 2 * res:i]) if i > 2 * res else mean))
    return np.array(rows, dtype=np.float64).reshape(-1, 4)


def smooth_outliers_f32(arr, lim=pp.OUTLIER_LIMIT):
    """preprocess.py:127-147 on a float32 array: the neighbour mean stays float32, as numpy computes it."""
    idx = np.asarray(np.abs(arr) > lim).nonzero()[0]
    for i in idx:
        if i == 0:
            arr[i] = arr[i + 1]
        elif i == len(arr) - 1:
            arr[i] = arr[i - 1]
        else:
            arr[i] = (arr[i - 1] + arr[i + 1]) / 2
            arr[i] = min(max(arr[i], -lim), lim)
    return arr


def mad_normalise_f32(signal):
    """preprocess.py:108-125 for float32 input: median, MAD, division and smoothing stay float32.  float32 out;
    MAD == 0 gives the reference's int64 zeros."""
    x = np.asarray(signal, dtype=np.float32)
    if x.shape[0] == 0:
        raise ValueError("Signal must not be empty")
    med = np.median(x)
    mad = np.median(np.abs(x - med))
    if mad == 0:
        return np.zeros(x.shape[0], dtype=np.int64)
    return smooth_outliers_f32(((x - med) / (np.float32(pp.SCALING_FACTOR) * mad)).astype(np.float32))


def run_batch_f32(reads, states, version, cache, threshold, mode):
    """``oracle.control_oracle.run_batch`` (control.py:31-97) for float32 reads: the same gating, cache and decision
    rule, with the float32 normaliser above.  Returns decisions, p_on, p_off, sig_len, cache."""
    mx = pp.max_length(version)
    B, M = len(reads), len(states)
    decisions = np.full(B, ctl.SKIPPED, dtype=np.uint8)
    p_on_out = np.zeros((B, M), dtype=np.float32)
    p_off_out = np.zeros((B, M), dtype=np.float32)
    sig_len = np.zeros(B, dtype=np.int32)
    for r, (read_id, raw) in enumerate(reads):
        window, _ = pp.select_window(raw, read_id, cache, version)
        if window is None:
            continue
        x = mad_normalise_f32(window)
        probs = [net.classify(s, x) for s in states]
        p_off = [p[0] for p in probs]
        p_on = [p[1] for p in probs]
        decisions[r] = ctl.decide(p_on, p_off, len(x), mx, threshold, mode)
        p_on_out[r] = [float(p) for p in p_on]
        p_off_out[r] = [float(p) for p in p_off]
        sig_len[r] = len(x)
        if len(cache) >= 1000:
            cache = {}
    return decisions, p_on_out, p_off_out, sig_len, cache
