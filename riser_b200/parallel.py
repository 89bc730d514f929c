"""Data-parallel training on the GPUs of one box: ``DataParallelTrainer`` runs a ConvNetTrainer or ResNetTrainer
(riser_b200.training) on every listed device, each on a contiguous slice of every global batch, and keeps them
bitwise equal without NCCL:
  * gradients -- every replica's ``.grad`` tensors are views of one flat fp32 buffer (plus one slot for its share
                 of the mean loss).  The exchange is a reduce-scatter plus an all-gather over peer-to-peer loads
                 (``riser_peer_reduce_f32``): replica d adds slice d of every replica's buffer in device order into
                 its own, then copies the other slices from their owners.  One owner computes each element, so every
                 replica gets the same bits, and a run is repeatable.
  * BatchNorm -- SyncBatchNorm semantics (ResNet): each replica writes float64 partial sums of its rows
                 (``riser_bn_stats_partial_cl`` / ``riser_bn_bwd_partial_cl``), and every replica adds the G
                 partials in device order (``riser_bn_*_finalize_cl``), so statistics, running statistics and
                 sums are those of the global batch.
  * loss      -- ``riser_gap_linear_ce_bwd_ex`` divides by the global batch, so every read's loss, logits and
                 dlogits have the bits of the one-device step.
  * Adam runs on every replica on the same gradients and weights: no broadcast.
A G-device step differs from the one-device step on the same global batch only in the order of sums (the weight
gradients' row sums and the fp32 sum over replicas).

One host thread per device enqueues that replica's work (ctypes releases the GIL during launches).  The threads meet
at every cross-device reduction: each records a CUDA event after writing what its peers will read, a barrier makes
sure every peer's event is recorded, and then each stream waits on its peers' events before the peer reads.  Nothing
is overwritten while a peer may still read it: every BatchNorm layer has its own partial buffers, and each replica's
stream waits for every peer's end-of-exchange event before it starts the next step."""
import ctypes
import operator
import os
import queue
import threading
import time

import torch

from . import _lib
from .training import (BN_EPS, BN_MOMENTUM, ConvNetTrainer, ResNetTrainer, _cnn_config, _resnet_config,
                       default_init_state, model_of, resnet_default_init_state)

MAX_DEVICES = 8                      # RISER_MAX_REPLICAS


def split(B, G):
    """The (lo, hi) read range of each of G replicas in a global batch of B: replica d gets [dB/G, (d+1)B/G)
    (floors), so the ranges are contiguous, in device order, and differ in size by at most one."""
    return [(d * B // G, (d + 1) * B // G) for d in range(G)]


def check_devices(devices):
    """The CUDA device indices of ``devices`` (ints, 'cuda:N' or torch.device) as a list of ints.  ValueError for an
    empty list, a device given twice, more than MAX_DEVICES devices or a non-CUDA / negative entry."""
    out = []
    for d in devices:
        if isinstance(d, (str, torch.device)):
            dv = torch.device(d)
            if dv.type != "cuda" or dv.index is None:
                raise ValueError(f"device {d!r}: name a CUDA device by index ('cuda:N' or N)")
            d = dv.index
        d = operator.index(d)
        if d < 0:
            raise ValueError(f"device {d}: CUDA device indices are >= 0")
        out.append(d)
    if not out:
        raise ValueError("devices: at least one CUDA device")
    if len(set(out)) != len(out):
        raise ValueError(f"devices {out}: a device is listed twice")
    if len(out) > MAX_DEVICES:
        raise ValueError(f"devices {out}: at most {MAX_DEVICES} devices (the peer reduction's limit)")
    return out


class _Group:
    """What the replicas share: the host barrier, the replicas in device order, the slices of the flat gradient."""

    def __init__(self, G):
        self.G = G
        self.barrier = threading.Barrier(G)
        self.replicas = []
        self.batch = 0                   # the global batch of the current step
        self.timing = False              # time every exchange with CUDA events (tools/time_train_dp.py)

    def finish_setup(self):
        n = self.replicas[0].flat.numel()
        chunk = -(-n // (self.G * 32)) * 32          # slice bounds on 128-byte boundaries: vector loads
        self.slices = [(min(n, d * chunk), min(n, (d + 1) * chunk)) for d in range(self.G)]
        self.flat_ptrs = (ctypes.c_void_p * self.G)(*[r.flat.data_ptr() for r in self.replicas])


class _Replica:
    """One replica: its trainer, and its side of the reductions (the trainer's ``reducer``)."""

    def __init__(self, group, rank, trainer):
        self.group, self.rank, self.trainer = group, rank, trainer
        n = sum(p.numel() for p in trainer.params.values())
        self.flat = torch.zeros(n + 1, device=trainer.device)  # every gradient, then this replica's share of the loss
        off = 0
        for p in trainer.params.values():
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()
        self.loss = self.flat[n:]
        self.self_ptr = (ctypes.c_void_p * 1)(self.flat.data_ptr())
        self.parts = {}                  # (kind, BatchNorm key) -> this replica's float64 partial
        self.events, self.keys = [], []  # per meeting point of a step: the event recorded there, and what it is
        self.met = 0
        self.done = torch.cuda.Event()   # recorded when this replica's exchange is finished
        self.finished = torch.cuda.Event()  # recorded when this replica's step is finished
        self.inputs = {}                 # (B, L) -> this replica's copies of its reads, lengths and labels
        self.ex_times = []               # while group.timing: (start, end) events of every exchange after its meeting,
        self.wait_times = []             # and (key, before, after) events around the waits of every meeting point
        self.wait_s = 0.0                # host seconds spent at the barrier
        self.jobs, self.results = queue.Queue(), queue.Queue()
        trainer.reducer = self

    @property
    def batch(self):
        return self.group.batch

    # ------------------------------------------------------------------ meeting points
    def meet(self, key):
        """Every replica's writes so far are visible to this replica's stream from here on."""
        g, i = self.group, self.met
        self.met += 1
        if i == len(self.events):
            self.events.append(torch.cuda.Event())
            self.keys.append(None)
        self.events[i].record()
        self.keys[i] = key
        t0 = time.perf_counter()
        g.barrier.wait()
        self.wait_s += time.perf_counter() - t0
        stream = torch.cuda.current_stream()
        if g.timing:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        for r in g.replicas:
            if r.keys[i] != key:
                raise RuntimeError(f"replica {r.rank} reached {r.keys[i]!r} where replica {self.rank} reached {key!r}")
            if r is not self:
                stream.wait_event(r.events[i])
        if g.timing:
            ev[1].record()
            self.wait_times.append((key,) + ev)

    def _partial(self, kind, cv):
        p = self.parts.get((kind, cv[1]))
        if p is None:
            p = torch.empty(_lib.lib().riser_bn_partial_bytes(cv[3]) // 8, dtype=torch.float64,
                            device=self.trainer.device)
            self.parts[(kind, cv[1])] = p
        return p

    def _peer_parts(self, kind, cv):
        return (ctypes.c_void_p * self.group.G)(*[r.parts[(kind, cv[1])].data_ptr() for r in self.group.replicas])

    # ------------------------------------------------------------------ the trainer's hooks
    def bn_stats(self, cv, y, n, mean, var, run):
        """Batch statistics of BatchNorm cv[1] over the global batch (y None: this replica has no reads)."""
        lib, P, ws = _lib.lib(), _lib.ptr, self.trainer.bn_ws
        B, L = (0, 1) if y is None else y.shape[:2]
        _lib.check(lib.riser_bn_stats_partial_cl(P(y), P(n), B, L, cv[3], P(self._partial("stats", cv)), P(ws),
                                                 ws.numel() * 4, _lib.stream_ptr()), "riser_bn_stats_partial_cl")
        self.meet(("stats", cv[1]))
        _lib.check(lib.riser_bn_stats_finalize_cl(self._peer_parts("stats", cv), self.group.G, cv[3], P(mean), P(var),
                                                  *[P(t) for t in run], BN_MOMENTUM, _lib.stream_ptr()),
                   "riser_bn_stats_finalize_cl")

    def bn_bwd(self, cv, dout, mask, y, n, stats, dx, dy_out):
        """BatchNorm cv[1]'s backward with the global sums; replica 0 owns the weight and bias gradients."""
        lib, P, tr, ws = _lib.lib(), _lib.ptr, self.trainer, self.trainer.bn_ws
        B, L = (0, 1) if y is None else y.shape[:2]
        g, b = tr.params[cv[1] + ".weight"], tr.params[cv[1] + ".bias"]
        _lib.check(lib.riser_bn_bwd_partial_cl(P(dout), P(mask), P(y), P(n), B, L, cv[3], P(stats[0]), P(stats[1]),
                                               BN_EPS, P(self._partial("bwd", cv)), P(ws), ws.numel() * 4,
                                               _lib.stream_ptr()), "riser_bn_bwd_partial_cl")
        self.meet(("bwd", cv[1]))
        _lib.check(lib.riser_bn_bwd_finalize_cl(self._peer_parts("bwd", cv), self.group.G, int(self.rank == 0),
                                                P(dout), P(mask), P(y), P(n), B, L, cv[3], P(stats[0]), P(stats[1]),
                                                P(g), BN_EPS, P(g.grad), P(b.grad), P(dx), P(dy_out), P(ws),
                                                ws.numel() * 4, _lib.stream_ptr()), "riser_bn_bwd_finalize_cl")

    def empty_bn(self, mode):
        """A ResNet replica without reads: zero partials at every BatchNorm, in the order the others meet there."""
        tr = self.trainer
        for cv in tr.convs:
            run = [None] * 3
            if mode == "step":
                run = [tr.buffers[cv[1] + k] for k in (".running_mean", ".running_var", ".num_batches_tracked")]
            self.bn_stats(cv, None, None, *tr.stats[cv[1]], run)
        for cv in tr._bn_backward_order():
            self.bn_bwd(cv, None, None, None, None, tr.stats[cv[1]], None, None)

    def exchange(self):
        """The fixed-order all-reduce of the flat gradient buffers (in place)."""
        g, lib, P = self.group, _lib.lib(), _lib.ptr
        self.meet("gradients")
        if g.timing:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        lo, hi = g.slices[self.rank]
        _lib.check(lib.riser_peer_reduce_f32(g.flat_ptrs, g.G, P(self.flat), lo, hi, _lib.stream_ptr()),
                   "riser_peer_reduce_f32")
        self.meet("reduced")
        for r in g.replicas:
            if r is not self:
                lo, hi = g.slices[r.rank]
                _lib.check(lib.riser_peer_reduce_f32(r.self_ptr, 1, P(self.flat), lo, hi, _lib.stream_ptr()),
                           "riser_peer_reduce_f32 (gather)")
        self.done.record()
        if g.timing:
            ev[1].record()
            self.ex_times.append(ev)

    # ------------------------------------------------------------------ one step of this replica
    def _pull(self, x, lens, labels, lo, hi):
        """This replica's reads [lo, hi) of the global batch (which lies on the first replica's device), copied by
        this replica's own stream with peer loads: the copies neither queue on the first device's stream nor wait for
        its later work.  The first replica uses the slices in place."""
        if self.rank == 0:
            return x[lo:hi], lens[lo:hi], labels[lo:hi]
        key = (hi - lo, x.shape[1])
        bufs = self.inputs.get(key)
        if bufs is None:
            dev = self.trainer.device
            bufs = (torch.empty(*key, device=dev), torch.empty(key[0], dtype=torch.int32, device=dev),
                    torch.empty(key[0], dtype=torch.int64, device=dev))
            self.inputs[key] = bufs
        for src, dst in zip((x[lo:hi], lens[lo:hi], labels[lo:hi]), bufs):
            src, dst = src.view(torch.float32), dst.view(torch.float32)       # one source: a copy of the bits
            _lib.check(_lib.lib().riser_peer_reduce_f32((ctypes.c_void_p * 1)(src.data_ptr()), 1, _lib.ptr(dst), 0,
                                                        dst.numel(), _lib.stream_ptr()), "riser_peer_reduce_f32 (inputs)")
        return bufs

    def run(self, x, lens, labels, ready, mode):
        """mode 'step' (gradients, exchange, Adam) or 'train' (gradients and exchange); ``ready``: recorded after
        the global batch was written."""
        g, tr = self.group, self.trainer
        stream = torch.cuda.current_stream()
        stream.wait_event(ready)
        for r in g.replicas:
            if r is not self:
                stream.wait_event(r.done)          # the peers no longer read this replica's buffers
        self.met = 0
        lo, hi = split(x.shape[0], g.G)[self.rank]
        if hi > lo:
            # the first replica's stream waits on every peer at the first meeting point, after their pulls: the
            # global batch's memory is not reused before they are done
            xs, ls, ys = self._pull(x, lens, labels, lo, hi)
            if isinstance(tr, ResNetTrainer):
                tr._run(xs, ls, ys, mode)
            else:
                tr._run(xs, ls, ys)
        else:
            self.flat.zero_()
            if isinstance(tr, ResNetTrainer):
                self.empty_bn(mode)
        self.exchange()
        if mode == "step":
            tr.optimizer.step()
        self.finished.record()


def _expandable_segments():
    """Whether torch's allocator is configured to map expandable segments (PYTORCH_CUDA_ALLOC_CONF)."""
    for var in ("PYTORCH_CUDA_ALLOC_CONF", "PYTORCH_ALLOC_CONF"):
        for item in os.environ.get(var, "").split(","):
            k, _, v = item.partition(":")
            if k.strip() == "expandable_segments" and v.strip().lower() == "true":
                return True
    return False


def _worker(rep, device):
    torch.cuda.set_device(device)
    while True:
        job = rep.jobs.get()
        if job is None:
            return
        try:
            job(rep)
            rep.results.put(None)
        except BaseException as e:           # noqa: BLE001 -- handed to the caller, the peers are released
            rep.group.barrier.abort()
            rep.results.put(e)
        del job


class DataParallelTrainer:
    """A ConvNetTrainer or ResNetTrainer (by ``config.model``) on each of ``devices`` (at most 8, each once), with
    the surface of the single-device trainers, so ``riser_b200.training.fit`` trains it unchanged.  Every replica is
    built from the same CPU state dict (``state``, or the default init of ``seed``).  A global batch of B reads is
    split with ``split(B, len(devices))``; a replica whose slice is empty (B < G) runs no kernels for the step and
    contributes zero gradient and zero BatchNorm partials.  Lengths and labels are checked on the global batch (the
    ResNet's single-value BatchNorm refusal on the global row count).  ``evaluate`` and ``state_dict`` use the first
    device's replica, which holds the same weights and running statistics as the others.  RiserError for a device
    that is not sm_100 or a pair of devices without peer access, and for torch's expandable_segments allocator
    setting: peer access (cudaDeviceEnablePeerAccess) covers cudaMalloc'ed memory, not the segments that setting maps,
    so the peer loads would fault.  Every method runs on the first device whatever device the caller has current.  The
    replicas' worker threads end with ``close``."""

    def __init__(self, config, devices, state=None, seed=0, logger=None):
        self._threads = []
        self._build(config, check_devices(devices), state, seed, logger)

    def _build(self, config, devices, state, seed, logger):
        """The replicas on ``devices`` in order.  A device listed twice holds two replicas: the same split,
        reductions and ordering on one GPU, which is how the suite checks them on a one-GPU box."""
        self._threads = []
        model = model_of(config)
        for d in devices:
            with torch.cuda.device(d):
                _lib.require_device()
        unique = list(dict.fromkeys(devices))
        if len(unique) > 1:
            if _expandable_segments():
                raise _lib.RiserError("data-parallel training reads peer GPUs' buffers, which needs cudaMalloc'ed "
                                      "memory: unset expandable_segments in PYTORCH_CUDA_ALLOC_CONF")
            _lib.check(_lib.lib().riser_peer_enable((ctypes.c_int * len(unique))(*unique), len(unique)),
                       "riser_peer_enable")
        if state is None:
            state = (resnet_default_init_state(_resnet_config(config), seed) if model == "resnet"
                     else default_init_state(_cnn_config(config), seed))
        state = {k: torch.as_tensor(v).detach().to("cpu") for k, v in state.items()}
        cls = ResNetTrainer if model == "resnet" else ConvNetTrainer
        self.group = _Group(len(devices))
        for rank, d in enumerate(devices):
            with torch.cuda.device(d):
                self.group.replicas.append(_Replica(self.group, rank, cls(config, state=state, seed=seed,
                                                                          logger=logger)))
        self.group.finish_setup()
        self.replicas = self.group.replicas
        self.devices = devices
        self.device = self.replicas[0].trainer.device
        self.logger = logger
        for rep, d in zip(self.replicas, devices):
            t = threading.Thread(target=_worker, args=(rep, d), name=f"riser-dp-{rep.rank}", daemon=True)
            t.start()
            self._threads.append(t)

    # ------------------------------------------------------------------ threads
    def _on_all(self, job):
        if not self._threads:
            raise RuntimeError("DataParallelTrainer is closed")
        for rep in self.replicas:
            rep.jobs.put(job)
        errors = [rep.results.get() for rep in self.replicas]
        failed = [e for e in errors if e is not None]
        if failed:
            self.group.barrier.reset()
            first = next((e for e in failed if not isinstance(e, threading.BrokenBarrierError)), failed[0])
            raise first

    def close(self):
        """Ends and joins the worker threads (after the work they enqueued; the device work may still run)."""
        for rep in getattr(self, "replicas", []):
            rep.jobs.put(None)
        for t in self._threads:
            t.join()
        self._threads = []

    def __del__(self):
        self.close()

    # ------------------------------------------------------------------ the trainers' surface
    def _inputs(self, x, lens, labels):
        """The global batch checked as the single-device trainer checks it, on the first device."""
        return self.replicas[0].trainer._inputs(x, lens, labels)

    def _global(self, x, lens, labels, mode):
        with torch.cuda.device(self.device):
            x, lens, labels = self._inputs(x, lens, labels)
            if x.shape[0] == 0:
                raise ValueError("an empty batch: the loss of 0 reads is undefined")
            self.group.batch = x.shape[0]
            ready = torch.cuda.Event()
            ready.record()
            self._on_all(lambda rep: rep.run(x, lens, labels, ready, mode))
            # the caller's stream: after the first replica's step (its loss, gradients and weights)
            torch.cuda.current_stream().wait_event(self.replicas[0].finished)

    def step(self, x, lens, labels):
        """One Adam step on the global batch on every replica; returns the mean loss as a 0-dim tensor on the first
        device (a view of a buffer the next step overwrites).  Neither allocates nor synchronises after the first
        step at a shape, with the inputs on the first device."""
        self._global(x, lens, labels, "step")
        return self.replicas[0].loss[0]

    def gradients(self, x, lens, labels):
        """The loss gradients of the global batch at the current weights (the first replica's copy)."""
        self._global(x, lens, labels, "train")
        with torch.cuda.device(self.device):
            return {k: p.grad.clone() for k, p in self.replicas[0].trainer.params.items()}

    def evaluate(self, x, lens, labels):
        """(mean loss, number of reads whose argmax class is the label), on the first device."""
        return self.replicas[0].trainer.evaluate(x, lens, labels)

    def state_dict(self):
        """The first replica's state dict (every replica holds the same bits)."""
        with torch.cuda.device(self.device):
            return self.replicas[0].trainer.state_dict()
