"""Device timing of the long-window normalisers (riser_normalise_long / riser_normalise_f32_long, csrc/normalise_long.cu).

  1. 64 reads x 1,000,000 samples, int16 and float32 (retrain mode): the whole-read shape only the long path takes;
  2. 4,096 x 16,000 int16 (bench.py's shape), the long path and riser_normalise alternated in the same process: how
     much the shared-memory kernel gains where both apply.

Every step is timed alone with CUDA events, the L2 overwritten (256 MB) before it; median of the steps.  Achieved
bytes/s count the algorithmic traffic, 6 B / sample for int16 (2 in, 4 out) and 8 B / sample for float32, not the
path's actual passes.  Prints one JSON line per measurement, each with the card's name and power limit.
usage: python tools/time_normalise_long.py [--steps N]"""
import argparse
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from riser_b200 import RaggedBatch, synth, _lib   # noqa: E402
from oracle import retrain_oracle as rt           # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"gpu": name, "power_limit": power}


def timed(fn, steps, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def workspace(B, max_len):
    nbytes = _lib.lib().riser_normalise_long_workspace_bytes(B, max_len)
    return torch.empty(nbytes, dtype=torch.uint8, device="cuda"), nbytes


def int16_long(batch, n, out):
    ws, nbytes = workspace(batch.B, n)
    L = _lib.lib()
    return lambda: _lib.check(L.riser_normalise_long(_lib.ptr(batch.sig), _lib.ptr(batch.off), None, _lib.ptr(batch.n),
                                                     batch.B, n, _lib.ptr(out), out.stride(0), None, _lib.ptr(ws),
                                                     nbytes, _lib.stream_ptr()), "riser_normalise_long")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda")
    info = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    L = _lib.lib()

    def report(what, B, n, ms, bytes_per_sample, **kw):
        print(json.dumps({"what": what, "B": B, "L": n, "ms": round(ms, 4),
                          "GBps": round(bytes_per_sample * B * n / ms / 1e6, 1), "bytes_per_sample": bytes_per_sample,
                          **kw, **info}), flush=True)

    # 1. whole reads
    B, n = 64, 1_000_000
    pool = synth.body_batch(11, 8, n)
    sigs = [pool[i % len(pool)] for i in range(B)]
    batch = RaggedBatch(sigs, dev)
    out = torch.zeros(B, n, device=dev)
    report("normalise_long int16", B, n, timed(int16_long(batch, n, out), args.steps, flush), 6)
    pa = [rt.pa_signal(s, scale=0.1 + 0.01 * (k % 8)) for k, s in enumerate(sigs)]
    b32 = RaggedBatch(pa, dev, dtype=np.float32)
    ws, nbytes = workspace(B, n)
    f32 = lambda: _lib.check(L.riser_normalise_f32_long(_lib.ptr(b32.sig), _lib.ptr(b32.off), _lib.ptr(b32.n), B, n,  # noqa: E731
                                                         3.5, 0, _lib.ptr(out), n, None, _lib.ptr(ws), nbytes,
                                                         _lib.stream_ptr()), "riser_normalise_f32_long")
    report("normalise_f32_long", B, n, timed(f32, args.steps, flush), 8)
    del batch, b32, out, ws

    # 2. bench shape, both paths alternated
    B, n = 4096, 16000
    pool = synth.body_batch(7, 256, n)
    batch = RaggedBatch([pool[i % len(pool)] for i in range(B)], dev)
    ld = (n + 3) & ~3
    out = torch.zeros(B, ld, device=dev)
    long_fn = int16_long(batch, n, out)
    short_fn = lambda: _lib.check(L.riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), None,  # noqa: E731
                                                    _lib.ptr(batch.n), B, n, _lib.ptr(out), ld, None,
                                                    _lib.stream_ptr()), "riser_normalise")
    t_long, t_short = [], []
    for _ in range(4):
        t_long.append(timed(long_fn, args.steps, flush))
        t_short.append(timed(short_fn, args.steps, flush))
    report("normalise_long int16", B, n, float(np.median(t_long)), 6, rounds=[round(t, 4) for t in t_long])
    report("normalise (shared memory) int16", B, n, float(np.median(t_short)), 6, rounds=[round(t, 4) for t in t_short])


if __name__ == "__main__":
    main()
