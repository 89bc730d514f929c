"""Restatement of the per-read body of the ReadUntil loop, riser/control.py:31-93.
Test infrastructure, see oracle/__init__."""
import numpy as np

from . import preprocess_oracle as pp
from . import convnet_oracle as net

# decision codes shared with include/riser_b200.h
TRY_AGAIN, ACCEPT, REJECT, NO_DECISION, SKIPPED = 0, 1, 2, 3, 4
NAMES = {TRY_AGAIN: "try_again", ACCEPT: "accept", REJECT: "reject",
         NO_DECISION: "no_decision", SKIPPED: "skipped"}


def decide(p_on, p_off, sig_len, max_len, threshold, mode):
    """riser/control.py:75-82.  p_on / p_off: per-model torch fp32 scalars (or
    numpy float32): the comparison is done the way torch does it for a 0-dim
    float32 tensor against a Python float."""
    if any(bool(p > threshold) for p in p_on):
        return ACCEPT if mode == "enrich" else REJECT
    if all(bool(p > threshold) for p in p_off):
        return ACCEPT if mode == "deplete" else REJECT
    if sig_len >= max_len:                     # preprocess.py:39-40
        return NO_DECISION
    return TRY_AGAIN


def run_batch(reads, states, version, cache, threshold, mode):
    """One pass of control.py:31-97 over ``reads`` = [(read_id, int16 array)].
    ``states`` = list of state-dicts (one per target model).  Returns per read:
    decision code, p_on per model, post-trim signal length (0 if skipped).
    The polyA cache is wiped when it reaches 1000 entries, after each assessed
    read (control.py:96-97); the (possibly new) dict is returned."""
    mx = pp.max_length(version)
    B, M = len(reads), len(states)
    decisions = np.full(B, SKIPPED, dtype=np.uint8)
    p_on_out = np.zeros((B, M), dtype=np.float32)
    p_off_out = np.zeros((B, M), dtype=np.float32)
    sig_len = np.zeros(B, dtype=np.int32)
    for r, (read_id, raw) in enumerate(reads):
        window, _ = pp.select_window(raw, read_id, cache, version)
        if window is None:
            continue
        x = pp.mad_normalise(window)
        probs = [net.classify(s, x) for s in states]
        p_off = [p[0] for p in probs]
        p_on = [p[1] for p in probs]
        decisions[r] = decide(p_on, p_off, len(x), mx, threshold, mode)
        p_on_out[r] = [float(p) for p in p_on]
        p_off_out[r] = [float(p) for p in p_off]
        sig_len[r] = len(x)
        if len(cache) >= 1000:
            cache = {}
    return decisions, p_on_out, p_off_out, sig_len, cache


CSV_HEADER = 'batch_start,read_id,channel,sig_length,models,prob_targets,threshold,mode,decision\n'   # control.py:146


def serial_target(client, models, proc, out_file, mode, threshold, unblock_duration=0.1):
    """SequencerControl.target of riser/control.py:24-124 run until the client stops, its serial per-read body
    driven through the ``proc`` (SignalProcessor) and ``models`` (Model) objects it is given, as the reference
    calls them (control.py:36-82): poly(A) trim with the run's cache, fixed trim or skip, minimum-length skip,
    cut to the kit's max length, ``mad_normalise``, ``classify`` per model, the decision rule.  One CSV row per
    assessed read (control.py:145-153); rejects are unblocked by read number, rejects + accepts + exhausted
    reads stop being received (control.py:100-106); the cache is wiped at 1000 entries (control.py:96-97)."""
    import time
    names = ";".join(m.target for m in models)
    max_len = proc.get_max_length()
    cache = {}
    with open(f"{out_file}.csv", "a") as sink:
        sink.write(CSV_HEADER)
        while client.is_running():
            batch_start = time.monotonic()
            rejects, done = [], []
            for channel, read in client.get_read_batch():
                signal, trimmed = proc.trim_polyA(client.get_raw_signal(read), read.id, cache)
                if not trimmed:
                    if not proc.should_trim_fixed_length(signal):
                        continue
                    signal = proc.trim_polyA_fixed_length(signal)[:max_len]
                else:
                    if len(signal) < proc.get_min_length():
                        continue
                    signal = signal[:max_len]
                signal = proc.mad_normalise(signal)
                probs = [m.classify(signal) for m in models]
                p_on = [p[1] for p in probs]
                code = decide(p_on, [p[0] for p in probs], len(signal), max_len, threshold, mode)
                sink.write(f"{batch_start:.0f},{read.id},{channel},{len(signal)},{names},"
                           f"{';'.join(str(p.item()) for p in p_on)},{threshold},{mode},{NAMES[code]}\n")
                if code == REJECT:
                    rejects.append((channel, read.number))
                if code in (REJECT, ACCEPT, NO_DECISION):
                    done.append((channel, read.number))
                if len(cache) >= 1000:
                    cache = {}
            client.reject_reads(rejects, unblock_duration)
            client.finish_processing_reads(done)
