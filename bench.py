#!/usr/bin/env python
"""Benchmark of the RISER read-classification hot path (contract: see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one pass of the hot path (median/MAD normalise + outlier smoothing ->
12-layer ConvNet -> softmax -> accept/reject decision) over one fixed batch of
synthetic already-trimmed squiggle chunks: BASELINE.json configs[1], RNA004 model shape,
4096 chunks of 4 s at 4 kHz (16,000 int16 samples) per GPU.

  value    reads classified / s, whole job, inputs resident in HBM (device timed, max over ranks)
  e2e      the same through the public API with HOST int16 buffers: pinned H2D copy of the
           batch and D2H of decisions + probabilities inside the timed region
  roofline the tcgen05 conv stack (layers 1..11): algorithmic FLOPs / CUDA-event time of that
           stage, against the measured bf16 peak in MEASURED_PEAKS.json
  cpu_baseline / --impl reference: the reference's OWN CPU path -- SignalProcessor.mad_normalise
           (np.vectorize, riser/preprocess.py:108-147) + Model.classify (riser/model.py:22-28) per read as
           riser/control.py:63-71 -- imported from oracle/_ref (the byte-compiled reference, see
           oracle/build_ref.py; `kind: "reference"`), on the box's host cores, on a bounded sample of the
           same workload.  The oracle port (vectorised numpy normalise) and a 1-thread run are reported beside it.
  torch_cuda_baseline: "PyTorch on B200" -- the reference's Model.classify on cuda at batch 1 (how RISER runs)
           and its ConvNet on the whole batch through cuDNN (TF32, and bf16 autocast), same box, same inputs.
  latency  p50 / p99 per poll of the live loop (BASELINE config 5): 512 channels x 2 models, 3000 x 1.

    python bench.py --reads 1000000 [--gpus N]      BASELINE config 4: R reads of 12,048 samples sharded r mod G

--dump-outputs DIR writes what the last timed step returned (rank 0), as float32: DIR/decisions.npy [B] (decision
codes, include/riser_b200.h) and DIR/probs.npy [M, B, 2] (softmax per model).  The inputs and weights are seeded,
so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import logging
import os
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm (rank 0 alone does the work) is to use all host threads
if "reference" in sys.argv and os.environ.get("RANK", "0") == "0" and os.environ.get("OMP_NUM_THREADS") == "1":
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 4096            # chunks per GPU per step (BASELINE.json configs[1])
LENGTH = 16000          # 4 s at 4 kHz
CHANNELS = [20, 30, 45, 67, 100, 150, 225, 337, 505, 757, 1135, 1702]
METRIC = "reads classified/sec (4 s chunks)"
UNIT = "reads/s"


def flops_per_read(length):
    total, cin, l = 0, 1, int(length)
    for c in CHANNELS:
        total += 2 * 3 * cin * c * l
        cin, l = c, l // 2
    return total + 2 * CHANNELS[-1] * 2


def conv_stack_flops_per_read(length):
    """Layers 1..11 only (what the tcgen05 kernel executes)."""
    return flops_per_read(length) - 2 * 3 * 1 * CHANNELS[0] * length - 2 * CHANNELS[-1] * 2


def workload_name(batch, length):
    return (f"BASELINE configs[1]: RNA004-shape mRNA ConvNet, {batch}-chunk fixed batch per GPU, "
            f"{length} int16 samples per chunk (4 s @ 4 kHz), already trimmed")


def shared_config(batch, length):
    """The `config` object: IDENTICAL in both arms (ours / --impl reference) -- what differs between the arms
    (precision mode, sample sizes, launch counts) lives in other keys of the line."""
    return {"workload": workload_name(batch, length), "batch_per_gpu": batch, "samples_per_chunk": length,
            "network": "ConvNet 12 x [Conv1d k3 + ReLU + MaxPool(2,2)] -> GAP -> Linear(1702, 2) "
                       "(riser/nets/cnn.py, the net riser/model.py:18 builds; BASELINE's metric says ResNet, "
                       "which nothing on the riser.py path instantiates -- SURVEY 0.1)",
            "step": "median/MAD normalise + outlier smoothing -> network -> softmax -> accept/reject decision",
            "flops_per_read": flops_per_read(length),
            "cache": "GPU arm: L2 flushed between timed steps (256 MiB write), inputs 393 MB > L2; CPU arm: n/a"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get("bf16_tflops_sustained", p.get("bf16_tflops")), p.get("hbm_gbs"), "measured"
    return 1400.0, 6650.0, "fallback"


def burst_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("bf16_tflops", 1590.0)
    return 1590.0


def pass_equivalents(length, precision, formats):
    """fp16-pass-equivalents of tensor work executed per algorithmic FLOP of the conv stack (FLOP-weighted over
    layers 1..11): F16 1, F16_W2 2, F16_X3 3; F16_F8: per layer by the row format the plan reports for its input
    (riser_plan_layer_format) -- 3 for hi + lo fp16 planes, 2 for the e4m3 format (fp16 pass + one e4m3 pass of
    twice the K at twice the rate).  1 / this = the structural ceiling of roofline.frac at a perfect tensor pipe."""
    if precision != 3:
        return {0: 1.0, 1: 2.0, 2: 3.0}[precision]
    tot = w = 0.0
    cin, l = 1, int(length)
    for i, c in enumerate(CHANNELS):
        f = 2 * 3 * cin * c * l
        if i >= 1:
            tot += f
            w += f * {1: 2.0, 2: 3.0, 3: 2.0, -1: 3.0}[formats[i]]    # (-1: fused into the previous launch, hi + lo planes)
        cin, l = c, l // 2
    return w / tot


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons (NVML; nvidia-smi as fallback) while the
    timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # torch's device index follows CUDA_VISIBLE_DEVICES; map through the UUID
            uuid = torch.cuda.get_device_properties(index).uuid
            h = None
            for i in range(pynvml.nvmlDeviceGetCount()):
                hi = pynvml.nvmlDeviceGetHandleByIndex(i)
                u = pynvml.nvmlDeviceGetUUID(hi)
                u = u.decode() if isinstance(u, bytes) else u
                if str(uuid) in u:
                    h = hi
            self.handle = h or pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flags = [bool(r & n.nvmlClocksThrottleReasonHwSlowdown), bool(r & n.nvmlClocksThrottleReasonHwThermalSlowdown),
                 bool(r & n.nvmlClocksThrottleReasonSwThermalSlowdown), bool(r & n.nvmlClocksThrottleReasonSwPowerCap)]
        return [str(mhz), str(self.max_mhz)] + ["Active" if f else "Not Active" for f in flags]

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.samples.append(self._sample_nvml())
                    time.sleep(0.005)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                time.sleep(0.05)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def cpu_reads(sample_reads, length, seed=4321):
    """The CPU legs' reads: a pool of 256 synthetic chunks repeated (as the GPU batch repeats its pool of 512)."""
    from riser_b200 import synth
    pool = synth.body_batch(seed, min(sample_reads, 256), length)
    return [pool[i % len(pool)] for i in range(sample_reads)]


class CpuPath:
    """The reference's CPU implementation of one read of the path, riser/control.py:63-71:
    ``signal = proc.mad_normalise(signal); p_off, p_on = model.classify(signal)``.

    kind "reference": the reference's own SignalProcessor / Model (imported from /root/reference in the build
    container, from the byte-compiled oracle/_ref on the GPU box), Model forced onto the CPU, weights loaded through
    its own torch.load path.  kind "port": the oracle restatement (vectorised numpy normalise -- faster than the
    reference's np.vectorize loop -- + torch-CPU ConvNet)."""
    def __init__(self, kind=None):
        from riser_b200 import synth
        from oracle import refshim
        self.kind = kind or ("reference" if refshim.available() else "port")
        if self.kind == "reference":
            import tempfile
            ref = refshim.load()
            ref.model.Model._get_device = lambda self_: torch.device("cpu")      # riser/model.py:30-32
            self.source = refshim.kind()
            with tempfile.TemporaryDirectory() as tmp:
                path = synth.save_state_dict(0, os.path.join(tmp, "mRNA_model_RNA004.pth"))
                self.model = ref.model.Model(path, refshim.cnn_config(), logging.getLogger("reference"), "mRNA")
            self.proc = ref.preprocess.SignalProcessor(ref.preprocess.Kit.create_from_version("RNA004"))
            self.read = lambda x: self.model.classify(self.proc.mad_normalise(x))
        else:
            from oracle import preprocess_oracle as pp
            from oracle import convnet_oracle as net
            self.source = "oracle port"
            state = synth.state_dict(0)
            self.read = lambda x: net.classify(state, pp.mad_normalise(x))

    def rate(self, X, threads):
        torch.set_num_threads(threads)
        for r in range(min(2, len(X))):
            self.read(X[r])
        t0 = time.perf_counter()
        for r in range(len(X)):
            self.read(X[r])
        return len(X) / (time.perf_counter() - t0)


def host_threads():
    cores = os.cpu_count() or 1
    return min(cores, torch.get_num_threads() if torch.get_num_threads() > 1 else cores)


def cpu_baseline(length, n_ref, n_port, n_one):
    """cpu_baseline object of our arm's line: the reference on all host threads (bounded sample), with the port
    and a 1-thread run of the reference beside it."""
    threads = host_threads()
    path = CpuPath()
    out = {"value": path.rate(cpu_reads(n_ref, length), threads), "unit": UNIT, "cores": threads,
           "kind": path.kind, "source": path.source,
           "sample": f"{n_ref} reads of {length} samples, per-read loop (mad_normalise + Model.classify, "
                     f"riser/control.py:63-71), torch threads = {threads}"}
    if n_one:
        out["one_thread"] = {"value": path.rate(cpu_reads(n_one, length), 1), "cores": 1, "sample": f"{n_one} reads"}
    if n_port and path.kind != "port":
        port = CpuPath("port")
        out["port"] = {"value": port.rate(cpu_reads(n_port, length), threads), "cores": threads,
                       "sample": f"{n_port} reads", "note": "oracle restatement, vectorised numpy normalise"}
    torch.set_num_threads(threads)
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on the host cores (rank 0 alone; all host threads)."""
    if rank != 0:
        return
    threads = host_threads()
    path = CpuPath()
    per_step = args.ref_reads
    X = cpu_reads(per_step, args.length)
    for _ in range(args.warmup):
        path.rate(X[:2], threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        path.rate(X, threads)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = (f"{per_step} reads of {args.length} samples per step, per-read loop (mad_normalise + Model.classify, "
              f"riser/control.py:63-71), {path.source}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64+f32", "data": "synthetic",
            "config": shared_config(args.batch, args.length),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": path.kind, "source": path.source,
                             "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


def torch_cuda_baseline(host_i16, dev, B, L, iters=3):
    """"PyTorch on B200" (SURVEY 2.3 / 8d): the reference's own modules on this GPU.
      batch1  : Model.classify per read on cuda (riser/model.py:22-28 -- how RISER runs), normalised input
                resident on the host as float64 like control.py hands it over
      batched : ConvNet(X[B, L]) through cuDNN on the whole batch, TF32 convs (torch's default:
                cudnn.allow_tf32) and bf16 autocast; network only (no normalise, no decision)
    Reads/s; None + a reason when the reference cannot be imported."""
    from oracle import refshim
    from riser_b200 import synth
    if not refshim.available():
        return {"unavailable": "reference not importable (oracle/_ref missing: run python -m oracle.build_ref "
                               "where /root/reference exists)"}
    import tempfile
    out = {"device": torch.cuda.get_device_name(dev), "source": refshim.kind(),
           "cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32)}
    try:
        ref = refshim.load()
        ref.model.Model._get_device = lambda self_: torch.device(dev)
        with tempfile.TemporaryDirectory() as tmp:
            path = synth.save_state_dict(0, os.path.join(tmp, "mRNA_model_RNA004.pth"))
            mdl = ref.model.Model(path, refshim.cnn_config(), logging.getLogger("reference"), "mRNA")
        # --- batch 1, as control.py:69 calls it (float64 numpy in, tensor out, .item() like control.py:152)
        rng = np.random.default_rng(0)
        xs = [rng.standard_normal(L) for _ in range(8)]
        for x in xs[:4]:
            mdl.classify(x)[1].item()
        n1 = 64
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for i in range(n1):
            mdl.classify(xs[i % len(xs)])[1].item()
        torch.cuda.synchronize(dev)
        out["batch1"] = {"value": n1 / (time.perf_counter() - t0), "unit": UNIT,
                         "what": f"reference Model.classify on cuda, one read of {L} samples per call, {n1} calls"}
        # --- whole batch through cuDNN
        X = torch.randn(B, L, device=dev, dtype=torch.float32)
        net = mdl.model

        def timed(fn):
            with torch.no_grad():
                for _ in range(2):
                    fn()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(iters):
                    fn()
                b.record()
                b.synchronize()
            return B * iters / (a.elapsed_time(b) * 1e-3)

        def fwd():
            return torch.nn.functional.softmax(net(X), dim=1)

        def fwd_bf16():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return torch.nn.functional.softmax(net(X), dim=1)

        out["batched_tf32"] = {"value": timed(fwd), "unit": UNIT,
                               "what": f"reference ConvNet(X[{B},{L}]) fp32 input, cuDNN convs with TF32 allowed"}
        out["batched_bf16_autocast"] = {"value": timed(fwd_bf16), "unit": UNIT,
                                        "what": "same under torch.autocast(bfloat16)"}
        del X
        torch.cuda.empty_cache()
    except Exception as e:      # a baseline leg must never take the bench line down
        out["error"] = f"{type(e).__name__}: {e}"[:300]
    return out


def run_reads(args, rank, local_rank, world):
    """BASELINE config 4: R synthetic reads of 12,048 samples (RNA002), read r -> rank r mod G (riser_b200.shard), every
    rank streams its shard through FixedBatchPipeline from HOST buffers in batches of `--batch`; per-read decisions are
    gathered (the only exchange) and checked against decisions computed on ONE GPU for the same reads.  Strong scaling:
    value = R / max-over-ranks device time."""
    import torch.distributed as dist
    from riser_b200 import Kit, SignalProcessor, Model, BatchedClassifier, FixedBatchPipeline, synth, shard
    from riser_b200.config import shipped_config
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    R, B, L = args.reads, args.batch, args.reads_length
    log = logging.getLogger("bench")
    mdl = Model(synth.state_dict(0), shipped_config(), log, "mRNA")
    clf = BatchedClassifier([mdl], SignalProcessor(Kit.create_from_version("RNA002")))
    clf.max_len, clf.ld = L, (L + 3) & ~3
    # read r is pool[(r * 40503) % P]: any rank can name any read without holding a million of them
    P = 509
    pool = synth.body_batch(1234, P, L)
    mine = shard.shard_indices(np.arange(R), rank, world)
    n_batches = (len(mine) + B - 1) // B
    # Three pinned staging batches, refilled from the pool per step INSIDE the timed region: the gather is the native
    # threaded one the live path uses (riser_b200/_hostpack, csrc/hostpack.c: buffer protocol + pthreads, GIL released)
    # and runs one batch ahead in a helper thread, so that the host fill, the H2D copy and the kernels of three
    # consecutive batches overlap.  (A numpy fancy-index fill on the submitting thread held this mode at 0.2 M
    # reads/s per GPU: 20 ms of host work per 4 ms of GPU work.)
    import concurrent.futures
    from riser_b200.preprocess import _hostpack
    n_slots = 3
    hosts = [torch.empty(B, L, dtype=torch.int16).pin_memory() for _ in range(n_slots)]
    pipe = FixedBatchPipeline(clf, B, L, 0.9, "deplete")
    rows = [pool[i] for i in range(P)]                                 # views, one per pool read
    byte_off = np.arange(B, dtype=np.int64) * (2 * L)
    zero_skip = np.zeros(B, dtype=np.int64)
    take = np.full(B, 2 * L, dtype=np.int64)
    pack_threads = max(1, min(8, (os.cpu_count() or 2) // max(1, world) - 1))
    hp = _hostpack()

    def fill(k, host):
        idx = mine[k * B:(k + 1) * B]
        src = ((idx * 40503) % P).tolist()
        hv = host.numpy()
        n = len(src)
        hp.pack([rows[j] for j in src], hv.reshape(-1), byte_off[:n], zero_skip[:n], take[:n], pack_threads)
        if n < B:
            hv[n:] = 0                 # constant reads: classified, ignored at the gather
        return n

    for k in range(2):
        fill(0, hosts[k])
        pipe.result(pipe.submit(hosts[k]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dec_local = np.empty(len(mine), dtype=np.uint8)
    pon_local = np.empty((len(mine), 1), dtype=np.float32)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e0.record()
    pipe.copy_stream.wait_event(e0)
    tickets, counts = [], []
    filler = concurrent.futures.ThreadPoolExecutor(max_workers=1)
    pending = filler.submit(fill, 0, hosts[0]) if n_batches else None
    for k in range(n_batches):
        counts.append(pending.result())
        if k + 1 < n_batches:          # slot (k + 1) % 3 was last submitted as batch k - 2, whose result has been read
            pending = filler.submit(fill, k + 1, hosts[(k + 1) % n_slots])
        tickets.append(pipe.submit(hosts[k % n_slots]))
        if k >= 1:
            d, pr = pipe.result(tickets[k - 1])
            n = counts[k - 1]
            dec_local[(k - 1) * B:(k - 1) * B + n] = d[:n]
            pon_local[(k - 1) * B:(k - 1) * B + n, 0] = pr[0, :n, 1]
    if n_batches:
        d, pr = pipe.result(tickets[-1])
        n = counts[-1]
        dec_local[(n_batches - 1) * B:(n_batches - 1) * B + n] = d[:n]
        pon_local[(n_batches - 1) * B:(n_batches - 1) * B + n, 0] = pr[0, :n, 1]
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    host_s = time.perf_counter() - t_host0
    barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dec_all, pon_all, _ = shard.gather_decisions(mine, dec_local, pon_local, np.zeros(len(mine), np.int32), R)
    else:
        dec_all, pon_all = dec_local, pon_local
    ms = float(t.cpu())
    if rank == 0:
        # single-GPU decisions of the same reads: classify the pool once on this GPU, map through the index rule
        hp = torch.empty(B, L, dtype=torch.int16).pin_memory()
        hp.numpy()[:P] = pool
        hp.numpy()[P:] = 0
        d_pool, _ = pipe.result(pipe.submit(hp))
        expect = d_pool[:P][(np.arange(R) * 40503) % P]
        agree = int((expect == dec_all).sum())
        line = {"metric": METRIC, "value": R / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": n_batches,
                "warmup": 2, "ms_per_step": ms / max(1, n_batches), "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f16+e4m3", "data": "synthetic",
                "config": {"workload": f"BASELINE configs[3]: {R} synthetic reads of {L} samples (RNA002), sharded by read "
                                       f"r mod {world} across {world} B200, batches of {B} from host buffers",
                           "cache": "inputs streamed from host every batch (24 KB per read H2D inside the timed region)"},
                "e2e": {"value": R / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes,
                        "d2h_bytes_per_step": pipe.d2h_bytes},
                "sharding": {"rule": "read r -> rank r mod G (riser_b200.shard.shard_indices)", "collective": "none on the "
                             "data path; decisions gathered once (shard.gather_decisions, 9 B per read)",
                             "decisions_equal_single_gpu": agree, "of": R,
                             "host_gb_per_s_per_rank": len(mine) * L * 2 / host_s / 1e9,
                             "host_note": f"pinned-buffer fill (native gather from the read pool, {pack_threads} threads, one batch ahead) + H2D per rank"},
                "gpu_launches": n_batches * (1 + mdl.launches(B, L) + 1),
                "clocks": sampler.summary()}
        assert agree == R, f"sharded decisions differ from the single-GPU decisions: {agree} of {R} agree"
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def _emit(line):
    """The one JSON line goes to the process's ORIGINAL stdout; everything else that writes to fd 1 during the
    run (NCCL's version banner, library chatter) has been pointed at stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--length", type=int, default=LENGTH)
    ap.add_argument("--precision", type=int, default=None, help="0 F16, 1 F16_W2, 2 F16_X3, 3 F16_F8; default = riser_b200.model.DEFAULT_PRECISION")
    ap.add_argument("--chunk", type=int, default=None)
    ap.add_argument("--ref-reads", type=int, default=128, help="reads per step of the --impl reference arm (~3 s of CPU work)")
    ap.add_argument("--cpu-sample", type=int, default=384, help="reads of the cpu_baseline leg (the reference, all host threads; ~10 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the host-side legs: cpu_baseline, torch_cuda_baseline, latency")
    ap.add_argument("--reads", type=int, default=0, help="BASELINE config 4: this many reads sharded r mod G (separate line)")
    ap.add_argument("--reads-length", type=int, default=12048)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's decisions and probabilities to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.reads):
        ap.error("--dump-outputs applies to the flagship workload (--impl ours, no --reads)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.reads:
        run_reads(args, rank, local_rank, world)
        return

    import torch.distributed as dist
    from riser_b200 import Kit, SignalProcessor, Model, BatchedClassifier, RaggedBatch, synth, _lib, model as rmodel
    from riser_b200.config import shipped_config

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    log = logging.getLogger("bench")
    cfg = shipped_config()
    precision = rmodel.DEFAULT_PRECISION if args.precision is None else args.precision
    mdl = Model(synth.state_dict(0), cfg, log, "mRNA", precision=precision)
    proc = SignalProcessor(Kit.create_from_version("RNA004"))
    clf = BatchedClassifier([mdl], proc, chunk=args.chunk)
    # the bench shape is the 4 s chunk BASELINE names (longer than the live path's 8,615 cap)
    clf.max_len = args.length
    clf.ld = (args.length + 3) & ~3
    B, L = args.batch, args.length

    # synthetic inputs: distinct reads per rank, generated on the host, resident in HBM
    pool = synth.body_batch(100 + rank, min(B, 512), L)
    host = torch.empty(B, L, dtype=torch.int16).pin_memory()
    hv = host.numpy()
    for i in range(B):
        hv[i] = pool[i % len(pool)]
    sigs = [hv[i] for i in range(B)]
    batch = RaggedBatch(sigs, dev)
    start = torch.zeros(B, dtype=torch.int32, device=dev)
    length = torch.full((B,), L, dtype=torch.int32, device=dev)
    # L2 flush buffer (written between timed steps); inputs (131 MB int16 + 262 MB fp32) exceed L2 anyway
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step(events=None):
        return clf.run_windows(batch, start, length, 0.9, "deplete", events=events)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    # ---- device-timed steps (value) with per-stage events for the roofline
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    conv_events = []
    barrier()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record()
        last = step(events=conv_events)
        ev[k][1].record()
    barrier()
    # host copies now: the later legs reuse the classifier's device buffers
    outputs = {"decisions": last[0].cpu().numpy().astype(np.float32),
               "probs": last[1].cpu().numpy().astype(np.float32)} if args.dump_outputs else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    conv_ms = sum(a.elapsed_time(b) for a, b in conv_events) / args.steps
    # the bracket covers layer 0 (CUDA cores) + conv layers 1..11; take layer 0's launches out
    conv_ms -= mdl.time_layer0(clf._buffers(B)["x"], length, L)
    # ---- the HBM-bound stage: riser_normalise alone (6 bytes per sample: int16 in, fp32 out), L2 flushed
    # (a kernel timed alone: the board is first given half a second to leave the power-capped clock the timed
    #  steps drove it into -- the HBM peak it is compared with was measured the same way)
    L_ = _lib.lib()
    xbuf = clf._buffers(B)["x"]
    torch.cuda.synchronize()
    time.sleep(0.5)
    nev = []
    for _ in range(7):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(L_.riser_normalise(_lib.ptr(batch.sig), _lib.ptr(batch.off), _lib.ptr(start), _lib.ptr(length), B, L,
                                      _lib.ptr(xbuf), xbuf.stride(0), None, _lib.stream_ptr()), "riser_normalise")
        b.record()
        nev.append((a, b))
    torch.cuda.synchronize()
    norm_ms = sorted(a.elapsed_time(b) for a, b in nev[2:])[(len(nev) - 2) // 2]      # first two launches: warm-up
    # ---- e2e: the public streaming API with HOST buffers.  Every step copies its 131 MB of
    #      pinned int16 input H2D and brings decisions + probabilities back D2H; the copy of
    #      step k+1 overlaps the kernels of step k (FixedBatchPipeline, two slots).
    from riser_b200 import FixedBatchPipeline
    pipe = FixedBatchPipeline(clf, B, L, 0.9, "deplete")
    hosts = [host, host.clone().pin_memory()]
    for k in range(2):
        pipe.result(pipe.submit(hosts[k % 2]))
    barrier()
    e2e_start, e2e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_start.record()
    pipe.copy_stream.wait_event(e2e_start)
    tickets = []
    for k in range(args.steps):
        tickets.append(pipe.submit(hosts[k % 2]))
        if k >= 1:
            pipe.result(tickets[k - 1])
    dec_np, _ = pipe.result(tickets[-1])
    e2e_end.record()
    e2e_end.synchronize()
    e2e_ms = e2e_start.elapsed_time(e2e_end)
    barrier()
    dec_host = torch.from_numpy(dec_np.copy())
    # ---- the same chunks through the call RISER's loop makes: BatchedClassifier.classify_batch with a list of
    #      UNPINNED numpy arrays (np.frombuffer views in the live run) -> native gather into the pinned arena -> H2D ->
    #      poly(A) detection + gating (control.py:36-60: these 16,000-sample prefixes have no poly(A), so the fixed trim
    #      cuts them to the kit's max length) -> normalise -> network -> decide -> D2H, one host sync per call.
    live_api = None
    if world == 1:
        sig_list = [np.array(hv[i]) for i in range(B)]          # pageable copies
        ids = [f"r{i}" for i in range(B)]
        live_clf = BatchedClassifier([mdl], proc, chunk=args.chunk)
        for _ in range(3):
            r_live = live_clf.classify_batch(sig_list, ids, {}, 0.9, "deplete")
        n_live = args.steps
        t0 = time.perf_counter()
        for _ in range(n_live):
            r_live = live_clf.classify_batch(sig_list, ids, {}, 0.9, "deplete")
        dt_live = time.perf_counter() - t0
        live_api = {"value": B * n_live / dt_live, "unit": UNIT, "ms_per_call": dt_live / n_live * 1e3,
                    "h2d_bytes_per_step": int(r_live.h2d_bytes), "d2h_bytes_per_step": int(r_live.d2h_bytes),
                    "classified_samples_per_read": int(r_live.sig_len.max()),
                    "api": "BatchedClassifier.classify_batch(list of unpinned int16 arrays): host gather + H2D + poly(A) "
                           "detection + gating + normalise + network + decide + D2H; wall clock, no overlap between calls"}
        del live_clf
    sampler.stop_flag = True
    sampler.join(timeout=2)

    t = torch.tensor([total_ms, e2e_ms, conv_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, conv_ms = (float(v) for v in t.cpu())
    n_dec = int((dec_host.numpy() != 4).sum())

    if rank == 0:
        tensor_peak, hbm_peak, peak_src = peaks()
        reads = B * world * args.steps
        value = reads / (total_ms * 1e-3)
        fused = mdl.plan(B, L).fused_layer0       # layer 0 then runs inside the conv kernel
        conv_flops = (conv_stack_flops_per_read(L) + (2 * 3 * CHANNELS[0] * L if fused else 0)) * B
        achieved = conv_flops / (conv_ms * 1e-3) / 1e12
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "conv_stack_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(f"B{B}_L{L}_p{precision}")
        launches_per_step = 1 + mdl.launches(B, L, clf.chunk) + 1
        plan = mdl.plan(B, L)
        formats = {i: plan.layer_format(i) for i in range(1, len(CHANNELS))}
        peq = pass_equivalents(L, precision, formats)
        kern = {}
        for i in range(1, len(CHANNELS)):
            kern.setdefault(plan.layer_kernel(i), []).append(i)
        kern_desc = " + ".join(f"{k} (layer{'s' if len(v) > 1 else ''} {'0+' if k.startswith('fused01') else ''}"
                               f"{','.join(map(str, v))})" for k, v in kern.items())
        f8_layers = [i for i, f in formats.items() if f == 3]
        tsrc = None
        if os.path.exists(tpath):
            with open(tpath) as f:
                tsrc = json.load(f).get("_source")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {0: "f16", 1: "f16", 2: "f16", 3: "f16+e4m3"}[precision],
            "data": "synthetic",
            "config": shared_config(B, L),
            "arm": {"precision_mode": precision,
                    "arithmetic": {0: "f16 operands, f32 accumulate (1 tcgen05 pass)",
                                   1: "f16, weights split hi+lo (2 passes), f32 accumulate",
                                   2: "f16, weights and activations split hi+lo (3 passes), f32 accumulate",
                                   3: "f16 pass + e4m3 correction pass carrying the hi/lo terms (2 pass-equivalents) in "
                                      f"layers {f8_layers[0] if f8_layers else '-'}-11, the other conv layers as mode 2; "
                                      "f32 accumulate; layer 0 and the head in f32, normalise in f64"}[precision],
                    "chunk": clf.chunk, "decisions_made": n_dec},
            "roofline": {"bound": "tensor", "kernel": kern_desc + " -- %d launches per forward" % len({(k, tuple(v)) if k in ("fused01_kernel", "conv_eo2_kernel") else (k, i)
                                                                                      for k, v in kern.items() for i in v}),
                         "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved / tensor_peak,
                         "traffic": traffic, "traffic_source": tsrc, "peak_source": f"bf16_tflops_sustained, {peak_src}",
                         "frac_burst": achieved / burst_peak(), "peak_burst": burst_peak(),
                         "pass_equivalents": peq, "ceiling": 1.0 / peq,
                         "ceiling_note": "1 / fp16-pass-equivalents executed per algorithmic FLOP: what frac would be at a "
                                         "perfect tensor pipe with this precision scheme (single-pass fp16/tf32 misses "
                                         "the 1e-3 probability bar, DESIGN.md section 2)",
                         "executed_tflops": achieved * peq,
                         "share_of_step": conv_ms / (total_ms / args.steps)},
            "roofline_normalise": {"bound": "hbm", "kernel": "normalise_kernel", "achieved": 6 * L * B / norm_ms / 1e6,
                                   "peak": hbm_peak, "unit": "GB/s", "frac": 6 * L * B / norm_ms / 1e6 / hbm_peak,
                                   "ms": norm_ms, "algorithmic_bytes_per_read": 6 * L,
                                   "peak_source": f"hbm_gbs, {peak_src}"},
            "e2e": {"value": reads / (e2e_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes,
                    "overlap": "H2D of step k+1 overlaps kernels of step k (2 slots)",
                    "api": "FixedBatchPipeline.submit / result (pinned [B, L] int16 in, decisions + probabilities out)"},
            "gpu_launches": launches_per_step * args.steps * 2,
            "clocks": sampler.summary(),
        }
        if live_api is not None:
            line["e2e_live_api"] = live_api
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(L, args.cpu_sample, 1024, 48)
            line["torch_cuda_baseline"] = torch_cuda_baseline(host, dev, B, L)
            try:
                from riser_b200 import sim
                line["latency"] = {"what": "ms per poll, batch in hand -> decisions on host (BASELINE config 5; "
                                           "riser_b200.sim.measure_latency, 1 s of new signal per channel and poll)",
                                   "minion_512ch_2models": sim.measure_latency(512, 80, "RNA002", ("mRNA", "mtRNA")),
                                   "promethion_3000ch_1model": sim.measure_latency(3000, 60, "RNA002", ("mRNA",))}
            except Exception as e:
                line["latency"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
