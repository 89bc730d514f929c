"""Device timing of the preprocessing kernels on raw prefixes: poly(A) detection
(riser_polya_end, 2*L algorithmic bytes per read), window selection and normalisation.
usage: python tools/time_preprocess.py [B] [prefix_len] [--f32 [scale,offset]]

--f32: afterwards, the same prefixes calibrated to float32 pA ((adc + offset) * scale, default
0.684,10) through riser_polya_end_f32 (4*L algorithmic bytes per read) and riser_normalise_f32_live."""
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from riser_b200 import Kit, SignalProcessor, RaggedBatch, synth, _lib   # noqa: E402

argv = sys.argv[1:]
f32_cal = None
if "--f32" in argv:
    i = argv.index("--f32")
    f32_cal = (0.684, 10.0)
    if i + 1 < len(argv) and "," in argv[i + 1]:
        f32_cal = tuple(float(v) for v in argv[i + 1].split(","))
        del argv[i + 1]
    del argv[i]
B = int(argv[0]) if len(argv) > 0 else 4096
n = int(argv[1]) if len(argv) > 1 else 18000
proc = SignalProcessor(Kit.create_from_version("RNA002"))
pool = synth.raw_reads(5, 256, min_body=n, max_body=n + 1000)
sigs = [pool[i % len(pool)][1][:n] for i in range(B)]
batch = RaggedBatch(sigs, torch.device("cuda"))


def timed(fn, iters=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


ms = timed(lambda: proc.polya_end_device(batch))
ends = proc.polya_end_device(batch).cpu().numpy()
print(f"polya_end: {ms:.3f} ms for {B} x {n} samples -> {B / ms * 1e3:.0f} reads/s, "
      f"{2 * n * B / ms / 1e6:.0f} GB/s algorithmic (found in {(ends > 0).mean() * 100:.0f}% of reads)")
start = torch.from_numpy(np.where(ends > 0, ends + 1, 0).astype(np.int32)).cuda()
length = torch.from_numpy(np.minimum(n - np.where(ends > 0, ends + 1, 0), 12048).astype(np.int32)).cuda()
out = torch.zeros(B, 12048, device="cuda")
L = _lib.lib()
ms = timed(lambda: _lib.check(L.riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(start),
                                                _lib.ptr(length), B, 12048, _lib.ptr(out), out.stride(0), None,
                                                _lib.stream_ptr()), "normalise"))
tot = int(length.sum().item())
print(f"normalise (trimmed windows, odd alignment): {ms:.3f} ms -> {6 * tot / ms / 1e6:.0f} GB/s algorithmic")

if f32_cal is not None:
    scale, offset = np.float32(f32_cal[0]), np.float32(f32_cal[1])
    sigs32 = [((s.astype(np.float32) + offset) * scale).astype(np.float32) for s in sigs]
    batch32 = RaggedBatch(sigs32, torch.device("cuda"), dtype=np.float32)
    ms = timed(lambda: proc.polya_end_device(batch32))
    ends32 = proc.polya_end_device(batch32).cpu().numpy()
    print(f"polya_end_f32 (scale {float(scale)}, offset {float(offset)}): {ms:.3f} ms for {B} x {n} samples -> "
          f"{B / ms * 1e3:.0f} reads/s, {4 * n * B / ms / 1e6:.0f} GB/s algorithmic "
          f"(found in {(ends32 > 0).mean() * 100:.0f}% of reads)")
    st32 = np.where(ends32 > 0, ends32 + 1, 0)
    len32 = torch.from_numpy(np.minimum(n - st32, 12048).astype(np.int32)).cuda()
    win_off = batch32.off[:B] + torch.from_numpy(st32.astype(np.int64)).cuda()
    ms = timed(lambda: _lib.check(L.riser_normalise_f32_live(_lib.ptr(batch32.sig), _lib.ptr(win_off),
                                                             _lib.ptr(len32), B, 12048, _lib.ptr(out), out.stride(0),
                                                             None, _lib.stream_ptr()), "normalise_f32_live"))
    tot = int(len32.sum().item())
    print(f"normalise_f32_live (trimmed windows): {ms:.3f} ms -> {8 * tot / ms / 1e6:.0f} GB/s algorithmic "
          "(4 bytes in, 4 out per sample)")
