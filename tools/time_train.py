"""Time one training step of the shipped ConvNet shape (riser_b200.training.ConvNetTrainer), or of a synthetic ResNet
configuration (``--net resnet --config basic|bottleneck``, ResNetTrainer), against the same network trained with torch
autograd + torch.optim.Adam on the same GPU (cuDNN; the ResNet's BatchNorm in training mode).

    python tools/time_train.py [--net cnn|resnet] [--config basic] [--steps 10] [--warmup 3] [--batches 32,256]
                               [--length 12048] [--out file.json]

Prints the GPU name and power limit, ms per step and reads/s for both at every batch size (every read at the full
length), and splits the riser_b200 step into forward (convolutions, pools, lengths), BatchNorm forward and backward,
head, wgrad, dgrad, the ReLU / pool backward and Adam (with the weight repacking) from CUDA events around every launch
of an instrumented step.  Needs a B200."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle.convnet_module import ConvNet                         # noqa: E402
from oracle.resnet_module import ResNet                           # noqa: E402
from riser_b200 import _lib                                      # noqa: E402
from riser_b200 import synth, training                            # noqa: E402
from riser_b200.config import CNN_SHIPPED, AttrDict              # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # the query is informational
        out = f"unavailable ({e})"
    return name, out


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


class _Recorder:
    """Stands in for the loaded library: every launch function is bracketed by CUDA events under a category."""

    def __init__(self, lib):
        self.lib, self.spans, self.backward = lib, [], False

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if not name.startswith("riser_") or name.endswith("_bytes"):
            return fn

        def call(*args):
            if name == "riser_conv1d_cl":
                cat = "dgrad" if self.backward else "forward"          # the launches after the head are dgrad
            elif name in ("riser_maxpool1d_pad_cl", "riser_len_chain"):
                cat = "forward"
            elif name in ("riser_bn_stats_cl", "riser_bn_apply_cl"):
                cat = "bn_forward"
            elif name == "riser_bn_bwd_cl":
                cat = "bn_backward"
            elif name == "riser_conv1d_dgrad_cl":
                cat = "dgrad"
            elif name == "riser_gap_linear_ce_bwd":
                cat = "head"
                self.backward = True
            elif name in ("riser_conv1d_wgrad_cl", "riser_conv1d_wgrad_ex"):
                cin = args[5] if name == "riser_conv1d_wgrad_cl" else args[7]
                cat = "wgrad_layer0" if cin == 1 else "wgrad"          # Cin = 1: 2 of the 16 MMA columns are used
            else:
                cat = "relu_pool_bwd"
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = fn(*args)
            b.record()
            self.spans.append((cat, a, b))
            return r
        return call


def breakdown(tr, x, lens, labels):
    rec = _Recorder(_lib.lib())
    orig = _lib.lib
    _lib.lib = lambda: rec
    try:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0 = torch.cuda.Event(enable_timing=True)
        s0.record()
        if isinstance(tr, training.ResNetTrainer):
            tr._run(x, lens, labels, "step")
        else:
            tr._run(x, lens, labels)
        a.record()
        tr.optimizer.step()
        b.record()
        torch.cuda.synchronize()
    finally:
        _lib.lib = orig
    parts = {}
    for cat, e0, e1 in rec.spans:
        parts[cat] = parts.get(cat, 0.0) + e0.elapsed_time(e1)
    parts["adam"] = a.elapsed_time(b)
    total_events = s0.elapsed_time(b)
    parts["repack_and_gaps"] = total_events - sum(parts.values())
    return parts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--net", choices=["cnn", "resnet"], default="cnn")
    ap.add_argument("--config", choices=sorted(synth.RESNET_CONFIGS), default="basic",
                    help="the synthetic ResNet configuration (--net resnet)")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batches", default="32,256")
    ap.add_argument("--length", type=int, default=12048)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = _lib.require_device()
    name, power = gpu_info()
    print(f"GPU: {name}; power.limit, clocks.max.sm: {power}")
    print(f"torch {torch.__version__}; reference convolutions: cudnn.allow_tf32 = {torch.backends.cudnn.allow_tf32}")
    if args.net == "resnet":
        cfg = AttrDict({"model": "resnet", "resnet": dict(synth.RESNET_CONFIGS[args.config]), "learning_rate": 1e-4})
        print(f"ResNet '{args.config}': {cfg.resnet}")
    else:
        cfg = AttrDict({"model": "cnn", "cnn": dict(CNN_SHIPPED), "learning_rate": 1e-4})
    L = args.length
    results = {"gpu": name, "power_limit_max_sm_clock": power, "net": args.net, "length": L, "rows": []}
    if args.net == "resnet":
        results["config"] = args.config
    for B in [int(b) for b in args.batches.split(",")]:
        g = torch.Generator(device="cpu").manual_seed(B)
        x = torch.randn(B, L, generator=g).to(dev)
        lens = torch.full((B,), L, dtype=torch.int32, device=dev)
        labels = (torch.arange(B) % 2).to(dev)
        tr = training.make_trainer(cfg, seed=0)
        ms = timed(lambda: tr.step(x, lens, labels), args.steps, args.warmup)
        parts = breakdown(tr, x, lens, labels)
        del tr
        torch.cuda.empty_cache()
        with torch.random.fork_rng(devices=[]):
            torch.manual_seed(0)
            net = (ResNet(cfg.resnet) if args.net == "resnet" else ConvNet(cfg.cnn)).to(dev).train()
        opt = torch.optim.Adam(net.parameters(), lr=1e-4)

        def ref_step():
            opt.zero_grad(set_to_none=False)
            F.cross_entropy(net(x), labels).backward()
            opt.step()
        ms_ref = timed(ref_step, args.steps, args.warmup)
        del net, opt
        torch.cuda.empty_cache()
        row = {"B": B, "riser_b200_ms_per_step": ms, "riser_b200_reads_per_s": B / ms * 1e3,
               "torch_ms_per_step": ms_ref, "torch_reads_per_s": B / ms_ref * 1e3,
               "split_ms": parts, "split_share": {k: v / sum(parts.values()) for k, v in parts.items()}}
        results["rows"].append(row)
        print(f"B {B:4d}: riser_b200 {ms:9.2f} ms/step ({row['riser_b200_reads_per_s']:8.1f} reads/s) | torch autograd "
              f"{ms_ref:9.2f} ms/step ({row['torch_reads_per_s']:8.1f} reads/s)")
        print("         split (one instrumented step, ms): " +
              ", ".join(f"{k} {v:.2f} ({100 * row['split_share'][k]:.1f} %)" for k, v in parts.items()))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)
    return results


if __name__ == "__main__":
    t = time.time()
    main()
    print(f"total {time.time() - t:.1f} s")
