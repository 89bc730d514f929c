"""Device timing of riser_normalise alone on the bench shape (B x L already-trimmed int16 chunks):
algorithmic bytes = 6 * L per read (int16 in, fp32 out) against the measured HBM copy peak.
usage: python tools/time_normalise.py [B] [L]"""
import json
import os
import sys

import torch

sys.path.insert(0, ".")
from riser_b200 import RaggedBatch, synth, _lib   # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
n = int(sys.argv[2]) if len(sys.argv) > 2 else 16000
pool = synth.body_batch(7, min(B, 256), n)
batch = RaggedBatch([pool[i % len(pool)] for i in range(B)], torch.device("cuda"))
ld = (n + 3) & ~3
out = torch.zeros(B, ld, device="cuda")
length = torch.full((B,), n, dtype=torch.int32, device="cuda")
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
L = _lib.lib()


def run():
    _lib.check(L.riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), None, _lib.ptr(length), B, n,
                                 _lib.ptr(out), ld, None, _lib.stream_ptr()), "normalise")


for _ in range(3):
    run()
torch.cuda.synchronize()
times = []
for _ in range(10):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    run()
    b.record()
    b.synchronize()
    times.append(a.elapsed_time(b))
ms = sorted(times)[len(times) // 2]
peak = 6531.0
if os.path.exists("MEASURED_PEAKS.json"):
    peak = json.load(open("MEASURED_PEAKS.json")).get("hbm_gbs", peak)
gbs = 6 * n * B / ms / 1e6
print(json.dumps({"kernel": "normalise_kernel", "B": B, "L": n, "ms": ms, "algorithmic_GBps": gbs,
                  "hbm_peak_GBps": peak, "frac": gbs / peak}))
