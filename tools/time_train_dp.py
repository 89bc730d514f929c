"""Time data-parallel training (riser_b200.parallel.DataParallelTrainer) across the GPUs of one box: weak scaling of
the shipped ConvNet and of the synthetic ResNet configurations at a fixed per-device batch.

    python tools/time_train_dp.py [--nets cnn,basic,bottleneck] [--gpus 1,2,4,8] [--batches 32,256] [--steps 10]
                                  [--warmup 3] [--length 12048] [--out file.json]

Every read is at the full length.  G = 1 is the plain single-device trainer; G > 1 uses the first G visible devices
(counts above the number visible are skipped).  Prints the GPU name and power limit, and per (network, per-device
batch, G): ms per step (a host clock around `steps` steps ending in a synchronise of every device), reads/s,
weak-scaling efficiency (the G = 1 step time over this one), and the split of a step across the devices (CUDA events
on every device, the mean over devices, per step):
  * exchange: the reduce-scatter and all-gather after the gradients' meeting point, and the bytes each device moves
    in it (its slice from G - 1 peers, then the other slices from their owners);
  * exchange waits / BN waits: how long a device's stream waits for its slowest peer at the exchange's two meeting
    points / at the BatchNorm statistics and backward meeting points (ResNet);
  * host waits: host seconds a worker thread spends at the barrier of the meeting points;
  * enqueue: the host time of step(), which returns once every thread has enqueued its work.
Needs B200s."""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from riser_b200 import _lib, synth, training                       # noqa: E402
from riser_b200.config import CNN_SHIPPED, AttrDict                # noqa: E402
from riser_b200.parallel import DataParallelTrainer                # noqa: E402
from time_train import gpu_info                                    # noqa: E402


def _config(net):
    if net == "cnn":
        return AttrDict({"model": "cnn", "cnn": dict(CNN_SHIPPED), "learning_rate": 1e-4})
    return AttrDict({"model": "resnet", "resnet": dict(synth.RESNET_CONFIGS[net]), "learning_rate": 1e-4})


def _sync_all(G):
    for d in range(G):
        torch.cuda.synchronize(d)


def measure(net, G, B_dev, L, steps, warmup):
    cfg = _config(net)
    B = B_dev * G
    g = torch.Generator(device="cpu").manual_seed(B)
    x = torch.randn(B, L, generator=g).to("cuda:0")
    lens = torch.full((B,), L, dtype=torch.int32, device="cuda:0")
    labels = (torch.arange(B) % 2).to("cuda:0")
    tr = training.make_trainer(cfg, seed=0) if G == 1 else DataParallelTrainer(cfg, list(range(G)), seed=0)
    try:
        for _ in range(warmup):
            tr.step(x, lens, labels)
        _sync_all(G)
        if G > 1:
            tr.group.timing = True
            for rep in tr.replicas:
                rep.ex_times, rep.wait_times, rep.wait_s = [], [], 0.0
        enqueue = 0.0
        t0 = time.perf_counter()
        for _ in range(steps):
            t1 = time.perf_counter()
            tr.step(x, lens, labels)
            enqueue += time.perf_counter() - t1
        _sync_all(G)
        ms = (time.perf_counter() - t0) / steps * 1e3
        row = {"net": net, "G": G, "B_per_device": B_dev, "ms_per_step": ms, "reads_per_s": B / ms * 1e3,
               "host_enqueue_ms_per_step": enqueue / steps * 1e3}
        if G > 1:
            ex = [a.elapsed_time(b) for rep in tr.replicas for a, b in rep.ex_times]
            n = tr.replicas[0].flat.numel()
            row["exchange_ms"] = sum(ex) / len(ex)
            waits = {"exchange": 0.0, "bn": 0.0}
            for rep in tr.replicas:
                for key, a, b in rep.wait_times:
                    waits["exchange" if key in ("gradients", "reduced") else "bn"] += a.elapsed_time(b)
            row["exchange_wait_ms"] = waits["exchange"] / G / steps
            row["bn_wait_ms"] = waits["bn"] / G / steps
            row["exchange_bytes_per_device"] = 2 * (G - 1) * (n * 4 // G)
            row["host_wait_ms_per_step"] = sum(rep.wait_s for rep in tr.replicas) / G / steps * 1e3
            tr.group.timing = False
        return row
    finally:
        if G > 1:
            tr.close()
        del tr
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nets", default="cnn,basic,bottleneck")
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--batches", default="32,256")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--length", type=int, default=12048)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _lib.require_device()
    name, power = gpu_info()
    visible = torch.cuda.device_count()
    print(f"GPU: {name} x {visible} visible; power.limit, clocks.max.sm: {power}")
    gpus = [G for G in (int(v) for v in args.gpus.split(",")) if G <= visible]
    results = {"gpu": name, "visible": visible, "power_limit_max_sm_clock": power, "length": args.length, "rows": []}
    for net in args.nets.split(","):
        for B_dev in (int(b) for b in args.batches.split(",")):
            base = None
            for G in gpus:
                row = measure(net, G, B_dev, args.length, args.steps, args.warmup)
                base = row["ms_per_step"] if G == 1 else base
                row["weak_scaling_efficiency"] = base / row["ms_per_step"] if base else None
                results["rows"].append(row)
                extra = ""
                if G > 1:
                    extra = (f" | exchange {row['exchange_ms']:.3f} ms, {row['exchange_bytes_per_device'] / 1e6:.1f} MB"
                             f"/device | device waits: exchange {row['exchange_wait_ms']:.3f} ms, BN "
                             f"{row['bn_wait_ms']:.3f} ms | host waits {row['host_wait_ms_per_step']:.2f} ms/step")
                eff = row["weak_scaling_efficiency"]
                print(f"{net:10s} B/dev {B_dev:4d} G {G}: {row['ms_per_step']:8.2f} ms/step "
                      f"{row['reads_per_s']:9.1f} reads/s eff {('%.1f %%' % (100 * eff)) if eff else '-':>7s} | "
                      f"enqueue {row['host_enqueue_ms_per_step']:.2f} ms/step{extra}", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)
    return results


if __name__ == "__main__":
    t = time.time()
    main()
    print(f"total {time.time() - t:.1f} s")
