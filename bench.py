#!/usr/bin/env python
"""bench.py - GVCNN grouping + fusion shapes/s on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]    # the reference's op graph on host cores

Workload (config.workload, IDENTICAL for both arms): BASELINE.json configs[1] - grouping + fusion FORWARD, 12 views,
D = 2048, G = 8 groups, B = 4096 synthetic shapes per GPU, C_raw = 1024, fp32, in the reference's own mode: ONE
grouping scheme per batch (tf.reduce_mean over the batch, nets/model.py:146; SURVEY.md D5 'batch').  One step = x per
(shape, view) -> per-view batch mean -> one [V] bin row -> pool + fuse of every shape with it, over one batch.
N > 1: one process per GPU (torchrun), shapes sharded by rank ("weak" scaling: 4096 shapes per GPU); the only data-path
exchange is the all-reduce of the V partial sums before binning (SURVEY.md 8e collective (2)), done by the library's
own one-kernel NVLink all-reduce (csrc/comm.cu; --exchange nccl selects torch.distributed/NCCL instead).

The same run also measures, as extra keys: the per-shape mode (`shape_mode`: bins [B, V], the heavier general case
SURVEY.md 8d names, no exchange at all), the training step (`fwd_bwd`, configs[2]: forward with tie mask + backward +
the parameter-gradient all-reduce), the same steps through the Python mirror of the reference's API (`api`), the
host-buffer end-to-end path in both modes (`e2e`), strong scaling at N > 1 (`strong`), the sweep of configs[3]
(`sweep`, N = 1) and the reference's own small shape, configs[0] (`config0`, N = 1).

One JSON line on stdout (rank 0).  `value` = device-resident whole-job shapes/s; `e2e` = the same through the
host-buffer C-ABI entry point (pinned host buffers, H2D + kernels + D2H every step); `roofline` = the pool+fuse
kernel's algorithmic bytes / its CUDA-event duration vs the measured HBM peak; `cpu_baseline` = the reference's op
sequence restated in torch-CPU, timed on this box's cores.

--dump-outputs DIR (CUDA arm) writes what the last timed headline step returned on rank 0 as DIR/<name>.npy:
S [B, D], x [B, V], xsum [V], scores [V] (float32) and bins [V] (float64).  The inputs come from fixed seeds, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "grouping+fusion shapes/s (12-view, D=2048)"
UNIT = "shapes/s"
CFG = dict(B=4096, V=12, D=2048, G=8, C_raw=1024, pool="max", empty_fill=1.0, score_reduce="batch")
NSETS = 3                                                            # rotating input AND output sets (SURVEY.md 8d)
DUMP_LIMIT = 64 << 20                                                # bytes written by one --dump-outputs, all arrays


def bench_config(world, scaling):
    """The `config` object of the JSON line - built by ONE function for both arms, so the driver's comparison of
    the two lines sees the same workload."""
    B, V, D, C, s = CFG["B"], CFG["V"], CFG["D"], CFG["C_raw"], 4
    return {
        "workload": "grouping+fusion forward, 12 views, D=2048, G=8, B=4096 shapes per GPU, C_raw=1024, fp32 "
                    "(BASELINE.json configs[1]); one scheme per batch = the reference's mode (nets/model.py:146)",
        "B_per_gpu": B, "V": V, "D": D, "G": CFG["G"], "C_raw": C, "pool": CFG["pool"], "empty_fill": CFG["empty_fill"],
        "score_reduce": CFG["score_reduce"], "scaling": scaling, "parallelism": "shape-sharded x%d" % world,
        "l2": "inputs larger than L2 (F %.0f MB + R %.0f MB per step vs 126 MB); %d rotating sets of inputs and of "
              "outputs" % (B * V * D * s / 1e6, B * V * C * s / 1e6, NSETS),
    }


# --------------------------------------------------------------------------- helpers
def algorithmic_bytes(B, V, D, C, s):
    """SURVEY.md 8d / BASELINE.md 3: every compulsory tensor counted once."""
    score = B * (V * C * s + 8 * V)
    pool = B * (V * D * s + D * s)
    bwd = B * (D * s + V * D * s)
    return {"score": score, "pool_fwd": pool, "fwd": score + pool, "bwd": bwd, "fwd_bwd": score + pool + bwd}


def dump_outputs(dirname, arrays):
    """Writes each array of {name: ndarray} as dirname/<name>.npy: floating arrays as float32 (float64 kept),
    integer arrays as float64, which holds every int32 exactly.  Refuses more than DUMP_LIMIT bytes in all."""
    import numpy as np
    out = {name: a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in "iub" else np.float32)
           for name, a in arrays.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_LIMIT))
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:                                           # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:                                   # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:                                       # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_to_gpu_numa_node(index):
    """Pin this process to the CPUs NVML reports as local to its GPU, so the pinned host buffers of the
    end-to-end leg are first-touched on the NUMA node whose PCIe root the GPU hangs off (matters when 8
    ranks stream 50 GB/s each from host memory).  Best effort: silently skipped if NVML says nothing."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:                                               # noqa: BLE001
        pass


def synth_inputs(B, V, D, C, seed_base, rank):
    """SURVEY.md 8d: CPU generators with fixed seeds so oracle and GPU see identical bits."""
    import torch
    off = 1000 * rank
    F = torch.randn((B, V, D), generator=torch.Generator().manual_seed(seed_base + 0 + off))
    R = torch.randn((B, V, C), generator=torch.Generator().manual_seed(seed_base + 1 + off))
    lim = math.sqrt(6.0 / (C + 1))                                   # Keras glorot-uniform of Dense(1)
    W = (torch.rand((V, C), generator=torch.Generator().manual_seed(2)) * 2 - 1) * lim
    b = torch.zeros(V)
    dS = torch.randn((B, D), generator=torch.Generator().manual_seed(seed_base + 3 + off))
    return F, R, W, b, dS


def literal_bias(V):
    """Per-view bias U(-4, 4) for the literal batch-mean mode: with b = 0 the mean over 4096 shapes of x ~ N(0, 2) is
    ~0 and every view would land in bin 0 (SURVEY.md 8d).  Same bias in both arms."""
    import torch
    return torch.rand(V, generator=torch.Generator().manual_seed(9)) * 8 - 4


# --------------------------------------------------------------------------- CPU baseline / reference arm
def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_reference_time(B, steps, warmup, V=None, D=None, C=None, G=None):
    """The reference's own op sequence for this path on host cores: oracle/gvcnn_oracle_torch
    .reference_step_cpu (stack views -> per group: where -> gather | ones dummy -> reduce_max ->
    multiply -> add_n -> div, after scores -> host binning -> weights; train.py:270-288,
    nets/model.py:16-102).  Returns (seconds per step list, threads)."""
    import torch
    from oracle import gvcnn_oracle_torch as OT
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    V, D, C, G = V or CFG["V"], D or CFG["D"], C or CFG["C_raw"], G or CFG["G"]
    F, R, W, b, _ = synth_inputs(B, V, D, C, 0, 0)
    b = literal_bias(V)
    views = [F[:, v, :].contiguous() for v in range(V)]              # the reference's list of V view tensors
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        S = OT.reference_step_cpu(views, R, W, b, G, pool=CFG["pool"], empty_fill=CFG["empty_fill"])
        float(S[0, 0])
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return times, threads


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = max(1, args.gpus)
    B = CFG["B"]                                                     # the FULL configs[1] batch every step
    times, threads = cpu_reference_time(B, args.steps, args.warmup)
    total = sum(times)
    value = B * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(world, args.scaling),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "cpu_model": cpu_model(),
                         "sample": "%d steps x the full %d-shape batch (one GPU's share of the job); the reference's op "
                                   "graph (nets/model.py:16-102, train.py:270-288) restated in torch-CPU, all host "
                                   "threads (TensorFlow 1.x is not installable in this image)" % (len(times), B)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------- CUDA arm
def run_cuda_arm(args):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device. The product path is sm_100a CUDA only (no CPU fallback); "
                         "use --impl reference for the host baseline.")
    from gvcnn_tf_b200 import _cabi as C
    from gvcnn_tf_b200 import model, parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # the gradient all-reduce must get SM slots while the dF kernel is running: high-priority NCCL stream
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank if world > 1 else 0)
    torch.cuda.set_device(dev)
    bind_to_gpu_numa_node(dev.index if dev.index is not None else 0)
    L = C.lib()
    C.check(L.gvcnn_check_device(), "gvcnn_check_device")

    Bfull, V, D, G, Cr = CFG["B"], CFG["V"], CFG["D"], CFG["G"], CFG["C_raw"]
    B = Bfull
    if args.scaling == "strong":                                     # SURVEY 8d config 3: B_total fixed at 4096
        if B % world:
            raise SystemExit("bench.py: --scaling strong needs %d %% n_gpus == 0" % B)
        B //= world
    K, Wm = args.steps, max(args.warmup, 3)
    s = 4
    p = lambda t: ctypes.c_void_p(t.data_ptr())

    # ---- the cross-rank exchange: the library's one-kernel NVLink all-reduce, or NCCL through torch.distributed
    comm, exchange_kind, exchange_note = None, "none (1 GPU)", None
    if world > 1:
        exchange_kind = "nccl"
        if args.exchange == "p2p":
            try:
                comm = parallel.P2PComm()
                probe = torch.full((V,), float(rank + 1), device=dev)
                comm.all_reduce_(probe)
                torch.cuda.synchronize()
                comm.check()
                if probe.tolist() != [world * (world + 1) / 2.0] * V:
                    raise RuntimeError("P2PComm self-test gave %s" % probe.tolist())
                exchange_kind = "p2p (gvcnn_comm: one kernel per rank over NVLink peer memory)"
            except Exception as e:                                   # noqa: BLE001
                comm, exchange_note = None, "P2PComm unavailable (%s); using NCCL" % str(e)[:200]
            # every rank must take the same route
            ok = torch.tensor([1 if comm is not None else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0 and comm is not None:
                comm.close()
                comm, exchange_kind = None, "nccl"
    nccl_cb = None
    if world > 1 and comm is None:
        nccl_cb = model.make_exchange(None)
    ex_fn, ex_user = (None, None)
    if comm is not None:
        ex_fn, ex_user = comm.exchange_c
    elif nccl_cb is not None:
        ex_fn, ex_user = ctypes.cast(nccl_cb[0], ctypes.c_void_p), None

    # ---- data: NSETS rotating input sets and NSETS rotating output sets (nothing a step touches can stay in L2)
    sets, host = [], None
    for i in range(NSETS):
        F, R, Wt, bt, dS = synth_inputs(B, V, D, Cr, 10 * i, rank)
        if i == 0:
            host = (F, R, dS)
        sets.append((F.to(dev), R.to(dev), dS.to(dev)))
    Wd, bd = Wt.to(dev), bt.to(dev)
    bias_lit = literal_bias(V).to(dev)
    outs = [dict(S=torch.empty((B, D), dtype=torch.float32, device=dev),
                 mask=torch.empty(((V + 7) // 8, B, D), dtype=torch.uint8, device=dev),
                 dF=torch.empty((B, V, D), dtype=torch.float32, device=dev),
                 scores=torch.empty((B, V), dtype=torch.float32, device=dev),
                 bins=torch.empty((B, V), dtype=torch.int32, device=dev),
                 x=torch.empty((B, V), dtype=torch.float32, device=dev),
                 xsum=torch.empty((V,), dtype=torch.float32, device=dev),
                 sc1=torch.empty((V,), dtype=torch.float32, device=dev),
                 bins1=torch.empty((V,), dtype=torch.int32, device=dev)) for _ in range(NSETS)]
    status = torch.zeros(C.STATUS_WORDS, dtype=torch.int32, device=dev)
    grad_bucket = torch.zeros(V * (Cr + 1), dtype=torch.float32, device=dev)   # FC-score grads (zeros: SURVEY D6)
    stream = torch.cuda.current_stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    pool = C.POOL_MAX if CFG["pool"] == "max" else C.POOL_MEAN
    fill = ctypes.c_float(CFG["empty_fill"])
    global_count = B * world

    # ---- raw C-ABI steps
    def k_score(i):
        o = outs[i % NSETS]
        C.check(L.gvcnn_score_bin_fwd(p(sets[i % NSETS][1]), p(Wd), p(bd), None, p(o["scores"]), p(o["bins"]), None,
                                      p(status), B, V, Cr, G, C.LAYOUT_BVD, C.F32, 0, 1, sp), "score_bin_fwd")

    def k_pool(i, with_mask=False, shared=False):
        o = outs[i % NSETS]
        C.check(L.gvcnn_pool_fuse_fwd(p(sets[i % NSETS][0]), p(o["bins1"] if shared else o["bins"]), 0 if shared else V,
                                      None, 0, p(o["S"]), None, p(o["mask"]) if with_mask else None, p(status),
                                      B, V, D, G, pool, fill, C.LAYOUT_BVD, C.F32, sp), "pool_fuse_fwd")

    def k_bwd(i, shared=False):
        o = outs[i % NSETS]
        C.check(L.gvcnn_pool_fuse_bwd(p(sets[i % NSETS][2]), p(o["bins1"] if shared else o["bins"]), 0 if shared else V,
                                      None, 0, p(o["mask"]), p(o["dF"]), p(status), B, V, D, G, pool, C.LAYOUT_BVD,
                                      C.F32, sp), "pool_fuse_bwd")

    def k_fwd_shape(i, with_mask=False):
        # per-shape forward entry point: score+bin then pool+fuse, chained with programmatic dependent launch
        o = outs[i % NSETS]
        Fd, Rd, _ = sets[i % NSETS]
        C.check(L.gvcnn_grouping_fusion_fwd(p(Rd), p(Wd), p(bd), p(Fd), None, p(o["scores"]), p(o["bins"]), None,
                                            p(o["S"]), p(o["mask"]) if with_mask else None, p(status), B, V, Cr, D, G,
                                            pool, fill, C.LAYOUT_BVD, C.LAYOUT_BVD, C.F32, 0, 1, sp),
                "grouping_fusion_fwd")

    def k_fwd_batch(i, with_mask=False):
        # reference-literal forward entry point: x; column sums + [exchange] + one bin row; pool+fuse (3 launches, PDL)
        o = outs[i % NSETS]
        Fd, Rd, _ = sets[i % NSETS]
        C.check(L.gvcnn_grouping_fusion_batch_fwd(p(Rd), p(Wd), p(bias_lit), p(Fd), p(o["x"]), p(o["xsum"]), None,
                                                  p(o["sc1"]), p(o["bins1"]), None, p(o["S"]),
                                                  p(o["mask"]) if with_mask else None, p(status), B, V, Cr, D, G, 0,
                                                  pool, fill, C.LAYOUT_BVD, C.LAYOUT_BVD, C.F32, 0, 1, global_count,
                                                  ex_fn, ex_user, sp), "grouping_fusion_batch_fwd")

    ar_stream = torch.cuda.Stream(priority=-1) if world > 1 else None   # the bucket's own (high-priority) stream

    def grad_allreduce():
        """sum over ranks * 1/K of the gradient bucket, forked off the step's stream so it overlaps the dF kernel."""
        if world == 1:
            return None
        if comm is not None:                                         # the library's one-kernel NVLink all-reduce
            ar_stream.wait_stream(torch.cuda.current_stream())
            comm.all_reduce_(grad_bucket, 1.0 / world, stream=ar_stream)
            return "join"
        return dist.all_reduce(grad_bucket, op=dist.ReduceOp.AVG, async_op=True)

    def grad_join(work):
        if work == "join":
            torch.cuda.current_stream().wait_stream(ar_stream)
        elif work is not None:
            work.wait()

    def step_train_batch(i):
        k_fwd_batch(i, True)
        work = grad_allreduce()                                      # launched before, and overlapping, the dF kernel
        k_bwd(i, shared=True)
        grad_join(work)

    def step_train_shape(i):
        k_fwd_shape(i, True)
        work = grad_allreduce()
        k_bwd(i, shared=False)
        grad_join(work)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    capturable = (world == 1) or (comm is not None)                  # NCCL collectives stay outside graphs

    def make_graph(step_fn):
        """Captures NSETS consecutive steps (one per rotating set) into a CUDA graph so the timed loop does not
        depend on how fast this box's CPU can issue launches.  Returns None if capture is refused."""
        nonlocal sp
        if args.no_graph or not capturable:
            return None
        saved = sp
        try:
            side = torch.cuda.Stream()
            side.wait_stream(stream)
            g = torch.cuda.CUDAGraph()
            sp = ctypes.c_void_p(side.cuda_stream)
            try:
                with torch.cuda.stream(side):
                    for i in range(NSETS):
                        step_fn(i)                                   # warm the capture stream
                side.synchronize()
                if world > 1:
                    dist.barrier()
                with torch.cuda.graph(g, stream=side):
                    for i in range(NSETS):
                        step_fn(i)
            finally:
                sp = saved
            torch.cuda.synchronize()
            return g
        except Exception:                                            # noqa: BLE001
            sp = saved
            torch.cuda.synchronize()
            return None

    def timed(step_fn, k, graph=None):
        """k steps bracketed by barrier + synchronize; device time by CUDA events; max over ranks.
        With a graph: k // NSETS replays of the NSETS-step graph plus k % NSETS eager steps = exactly k steps."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        if graph is not None:
            for _ in range(k // NSETS):
                graph.replay()
            for i in range(k % NSETS):
                step_fn(i)
        else:
            for i in range(k):
                step_fn(i)
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed_wall(step_fn, k):
        """k calls through the Python API: wall clock (Python, allocator and launches included), max over ranks."""
        barrier()
        t0 = time.perf_counter()
        for i in range(k):
            step_fn(i)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return sec * 1e3

    def per_launch(fns, k):
        """CUDA events around each launch of a sequence; returns the mean ms between consecutive events."""
        barrier()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(fns) + 1)] for _ in range(k)]
        for i in range(k):
            ev[i][0].record(stream)
            for j, fn in enumerate(fns):
                fn(i)
                ev[i][j + 1].record(stream)
        barrier()
        return [statistics.mean(e[j].elapsed_time(e[j + 1]) for e in ev) for j in range(len(fns))]

    sampler = ClockSampler(dev.index if dev.index is not None else 0) if rank == 0 else None

    # ---- sanity before timing: in the literal mode every rank derived the SAME bin row (and, on a small gathered
    #      batch, the row the oracle derives from the global batch)
    literal_check = None
    if world > 1:
        k_fwd_batch(0)
        rows = [torch.empty_like(outs[0]["bins1"]) for _ in range(world)]
        dist.all_gather(rows, outs[0]["bins1"])
        same = all(torch.equal(r, rows[0]) for r in rows)
        Bs = 64                                                      # small global batch through the oracle
        Rs = sets[0][1][:Bs].contiguous()
        xs, xsum_s = torch.empty((Bs, V), device=dev), torch.empty((V,), device=dev)
        sc_s, bn_s = torch.empty((V,), device=dev), torch.empty((V,), dtype=torch.int32, device=dev)
        Ss = torch.empty((Bs, D), device=dev)
        C.check(L.gvcnn_grouping_fusion_batch_fwd(p(Rs), p(Wd), p(bias_lit), p(sets[0][0]), p(xs), p(xsum_s), None,
                                                  p(sc_s), p(bn_s), None, p(Ss), None, p(status), Bs, V, Cr, D, G, 0,
                                                  pool, fill, C.LAYOUT_BVD, C.LAYOUT_BVD, C.F32, 0, 1, Bs * world,
                                                  ex_fn, ex_user, sp), "grouping_fusion_batch_fwd (check)")
        gathered = [torch.empty_like(Rs) for _ in range(world)]
        dist.all_gather(gathered, Rs)
        brow = [torch.empty_like(bn_s) for _ in range(world)]
        dist.all_gather(brow, bn_s)
        oracle_ok = None
        if rank == 0:
            import numpy as np
            from oracle import gvcnn_oracle as O                     # the checker, not the thing measured
            Rg = torch.cat(gathered).cpu().numpy()
            x64, s64 = O.view_scores(Rg, Wt.numpy(), literal_bias(V).numpy(), score_reduce="batch", dtype=np.float64)
            want = O.bins_from_scores(s64.astype(np.float32), G)[0]
            edge = O.edge_ulps_distance(s64.astype(np.float32), G, k=8)[0]
            got = bn_s.cpu().numpy()
            oracle_ok = bool(np.all((got == want) | edge)) and all(torch.equal(r, brow[0]) for r in brow)
        literal_check = {"all_ranks_same_bins": bool(same), "small_global_batch_bins_match_oracle": oracle_ok,
                         "bins": rows[0].tolist()}
        if not same or oracle_ok is False:
            raise SystemExit("bench.py: literal-mode bins differ across ranks or from the oracle: %s" % literal_check)

    # ---- warm-up, then the headline region: exactly K forward steps in the reference's mode
    for i in range(Wm):
        k_fwd_batch(i)
        k_fwd_shape(i)
        step_train_batch(i)
    graph_fwd = make_graph(k_fwd_batch)
    if sampler:
        sampler.start()
    ms_fwd = timed(k_fwd_batch, K, graph_fwd)
    if args.dump_outputs and rank == 0:
        # step i writes output set i % NSETS, in a graph replay or eagerly; later regions overwrite the sets
        o = outs[(K - 1) % NSETS]
        dump_outputs(args.dump_outputs, {"S": o["S"].cpu().numpy(), "x": o["x"].cpu().numpy(),
                                         "xsum": o["xsum"].cpu().numpy(), "scores": o["sc1"].cpu().numpy(),
                                         "bins": o["bins1"].cpu().numpy()})
    # view_score, fused (column sums + exchange + mean/score/bin), pool+fuse; the NCCL route is 5 launches + NCCL's
    fwd_launches = 3 if (world == 1 or comm is not None) else 4

    # ---- the per-shape mode (SURVEY.md 8d's heavier general case; round 1's headline): 2 launches, no exchange
    graph_shape = make_graph(k_fwd_shape)
    ms_shape = timed(k_fwd_shape, K, graph_shape)

    # ---- per-kernel durations, measured live with events around each launch (separate regions so the events do
    #      not sit inside the headline numbers)
    t_score, t_pool = per_launch([k_score, k_pool], K)
    ms_pool_b2b = timed(lambda i: k_pool(i), K)                      # K launches back to back in one event bracket
    t_pool_shared = per_launch([lambda i: k_pool(i, shared=True)], K)[0]

    # ---- training step (configs[2]): fwd with tie mask + bwd (+ grad all-reduce when N > 1)
    graph_train = make_graph(step_train_batch)
    ms_train = timed(step_train_batch, K, graph_train)
    graph_train_s = make_graph(step_train_shape)
    ms_train_shape = timed(step_train_shape, K, graph_train_s)
    _, t_pool_m, t_bwd = per_launch([k_score, lambda i: k_pool(i, True), k_bwd], K)
    us_allreduce, us_allreduce_nccl, us_xsum = None, None, None
    if world > 1:
        def step_allreduce(i):
            grad_join(grad_allreduce())
        for i in range(3):
            step_allreduce(i)
        us_allreduce = timed(step_allreduce, K) / K * 1e3

        def step_allreduce_nccl(i):
            dist.all_reduce(grad_bucket, op=dist.ReduceOp.AVG)
        for i in range(3):
            step_allreduce_nccl(i)
        us_allreduce_nccl = timed(step_allreduce_nccl, K) / K * 1e3
        if comm is not None:
            xs_probe = torch.zeros(V, device=dev)
            us_xsum = timed(lambda i: comm.all_reduce_(xs_probe), K) / K * 1e3

    # ---- the same steps through the Python mirror of the reference's API (gvcnn_tf_b200.model), Python included
    Fl = [t.transpose(0, 1).contiguous() for t, _, _ in sets]         # [V, B, D]: the reference's list of V view tensors
    view_lists = [[fv[v] for v in range(V)] for fv in Fl]
    ex_model = comm.exchange_c if comm is not None else None
    pg = dist.group.WORLD if (world > 1 and comm is None) else None

    def api_shape(i):
        Fd, Rd, _ = sets[i % NSETS]
        return model.grouping_fusion(Rd, Wd, bd, Fd, G, clamp=True)[0]

    def api_batch(i):
        Fd, Rd, _ = sets[i % NSETS]
        return model.grouping_fusion(Rd, Wd, bias_lit, Fd, G, score_reduce="batch", clamp=True, exchange=ex_model,
                                     process_group=pg, global_count=global_count)[0]

    def api_refseq(i, check=True):
        # names and argument order of train.py:270-288 + nets/model.py:154-157
        Rd = sets[i % NSETS][1]
        if world > 1:
            sr = model.score_bin(Rd, Wd, bias_lit, 1, score_reduce="batch", edge_ulps=0, clamp=True, check=False,
                                 exchange=(comm.exchange if comm is not None else None), process_group=pg,
                                 global_count=global_count)
            scores = sr.scores
        else:
            scores = model.view_scores(Rd, Wd, bias_lit)
        scheme = model.group_scheme([scores[0]], G, V, check=check)
        w = model.group_weight(scheme)
        desc = model.view_pooling(view_lists[i % NSETS], scheme)
        return model.group_fusion(desc, w)

    api = {}
    with torch.no_grad():
        for name, fn in (("grouping_fusion(score_reduce='shape')", api_shape),
                         ("grouping_fusion(score_reduce='batch')", api_batch),
                         ("view_scores -> group_scheme -> group_weight -> view_pooling -> group_fusion", api_refseq),
                         ("the same sequence, group_scheme(check='deferred'): exceptions raised one call late, no "
                          "synchronisation inside the step", lambda i: api_refseq(i, "deferred"))):
            for i in range(3):
                fn(i)
            api[name] = timed_wall(fn, K) / K
    model.check_deferred(dev)
    # the reference-shaped sequence gives the one-call literal path's bits
    with torch.no_grad():
        S_seq = api_refseq(0)
        k_fwd_batch(0)
        torch.cuda.synchronize()
        api_same = bool(torch.equal(S_seq.reshape(B, D), outs[0]["S"]))

    # ---- end to end through the host-buffer C-ABI entry point (pinned host memory), both modes
    Ke = max(1, min(K, args.e2e_steps))
    Fh, Rh, dSh = (t.pin_memory() for t in host)
    Sh = torch.empty((B, D), dtype=torch.float32).pin_memory()
    bins_h = torch.empty((B, V), dtype=torch.int32).pin_memory()
    st_h = torch.zeros(C.STATUS_WORDS, dtype=torch.int32)
    chunk = args.e2e_chunk
    pipe = ctypes.c_void_p()
    C.check(L.gvcnn_host_pipeline_create(ctypes.byref(pipe), args.e2e_h2d_streams), "gvcnn_host_pipeline_create")
    ws_bytes = max(L.gvcnn_host_workspace_bytes(B, chunk, V, Cr, D, C.F32, 0, m) for m in (0, 1))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def e2e_step(mode):
        C.check(L.gvcnn_grouping_fusion_host(pipe, p(Rh), p(Fh), p(Wd), p(bias_lit if mode else bd), p(Sh), None, p(bins_h),
                                             None, None, p(st_h), B, V, Cr, D, G, pool, fill, C.F32, mode, global_count,
                                             ex_fn if mode else None, ex_user if mode else None, chunk, p(ws), ws_bytes),
                "gvcnn_grouping_fusion_host")

    def e2e_time(mode):
        for _ in range(2):
            e2e_step(mode)
        barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            e2e_step(mode)                                           # synchronous: returns with S in host memory
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return sec

    e2e_s = e2e_time(C.SCORE_REDUCE_BATCH)
    e2e_same = bool(torch.equal(Sh.to(dev), outs[0]["S"])) if world == 1 else None   # host path == device path (set 0)
    e2e_shape_s = e2e_time(C.SCORE_REDUCE_SHAPE)
    h2d = B * V * (Cr + D) * s
    d2h = B * D * s + V * 4
    d2h_shape = B * D * s + B * V * 4

    # ---- what the box's host->device link can do: one pinned cudaMemcpyAsync of the same bytes, all ranks at once
    Hh = torch.empty(h2d, dtype=torch.uint8).pin_memory()
    Hd = torch.empty(h2d, dtype=torch.uint8, device=dev)
    h2d_ms = []
    for it in range(4):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        Hd.copy_(Hh, non_blocking=True)
        e1.record(stream)
        torch.cuda.synchronize()
        if it:
            h2d_ms.append(e0.elapsed_time(e1))
    h2d_best = min(h2d_ms)
    if world > 1:
        t = torch.tensor([h2d_best], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                      # the slowest rank's link bounds the job
        h2d_best = float(t.item())
    h2d_peak_gbs = h2d / (h2d_best * 1e-3) / 1e9
    del Hh, Hd
    L.gvcnn_host_pipeline_destroy(pipe)

    # ---- strong scaling (configs[2], B_total = 4096 split over the ranks) as an extra key of the weak line
    strong = None
    if world > 1 and args.scaling == "weak" and Bfull % world == 0:
        Bs_ = Bfull // world
        B_saved, gc_saved = B, global_count
        B, global_count = Bs_, Bfull                                 # the step closures read B / global_count
        try:
            for i in range(3):
                k_fwd_batch(i), k_fwd_shape(i), step_train_batch(i)
            g1, g2, g3 = make_graph(k_fwd_batch), make_graph(k_fwd_shape), make_graph(step_train_batch)
            ms1, ms2, ms3 = timed(k_fwd_batch, K, g1), timed(k_fwd_shape, K, g2), timed(step_train_batch, K, g3)
            strong = {"workload": "4096 shapes in total, %d per GPU" % Bs_,
                      "fwd": {"value": Bfull * K / (ms1 * 1e-3), "ms_per_step": ms1 / K},
                      "fwd_shape_mode": {"value": Bfull * K / (ms2 * 1e-3), "ms_per_step": ms2 / K},
                      "fwd_bwd": {"value": Bfull * K / (ms3 * 1e-3), "ms_per_step": ms3 / K}, "unit": UNIT}
        finally:
            B, global_count = B_saved, gc_saved

    clocks = sampler.stop() if sampler else None
    st = status.tolist()
    if any(st[:2]):
        raise SystemExit("bench.py: status words report out-of-range/NaN scores: %s" % st)
    if comm is not None:
        comm.check()

    extra = {}
    if world == 1 and not args.no_sweep:
        extra["sweep"] = run_sweep(torch, C, L, dev, args.sweep_iters)
        extra["config0"] = run_config0(torch, model, dev)

    if rank != 0:
        if comm is not None:
            comm.close()
        if world > 1:
            dist.destroy_process_group()
        return 0

    ab = algorithmic_bytes(B, V, D, Cr, s)
    peak, peak_src = measured_peaks()
    gbps = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9
    value = world * B * K / (ms_fwd * 1e-3)
    ach_pool = gbps(ab["pool_fwd"], t_pool)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")               # ncu dram bytes of the pool kernel, if captured
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get("pool_fuse_fwd_dram_bytes_per_launch")
        except Exception:                                            # noqa: BLE001
            traffic = None
    raw_step = {"shape": ms_shape / K, "batch": ms_fwd / K}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_fwd / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(world, args.scaling),
        "launch": ("CUDA graph of %d steps replayed K/%d times" % (NSETS, NSETS)) if graph_fwd is not None
                  else "stream launches",
        "exchange": {"kind": exchange_kind, "note": exchange_note, "xsum_allreduce_alone_us": us_xsum,
                     "literal_check": literal_check},
        "roofline": {"bound": "hbm", "kernel": "pool_fuse_fwd_ring_kernel", "achieved": ach_pool, "peak": peak,
                     "unit": "GB/s", "frac": ach_pool / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": ab["pool_fwd"], "us_per_launch": t_pool * 1e3,
                     "timing": "CUDA event pair around each launch (includes ~4 us of event/launch gap); "
                               "back_to_back = K launches of this kernel in one event bracket",
                     "back_to_back": {"us_per_launch": ms_pool_b2b / K * 1e3, "achieved": gbps(ab["pool_fwd"], ms_pool_b2b / K),
                                      "frac": gbps(ab["pool_fwd"], ms_pool_b2b / K) / peak},
                     "other_kernels": {
                         "pool_fuse_fwd_ring_kernel (one shared bin row)": {"us_per_launch": t_pool_shared * 1e3,
                                                                           "frac": gbps(ab["pool_fwd"], t_pool_shared) / peak},
                         "view_score_kernel": {"achieved": gbps(ab["score"], t_score), "frac": gbps(ab["score"], t_score) / peak,
                                               "us_per_launch": t_score * 1e3, "algorithmic_bytes_per_launch": ab["score"]},
                         "pool_fuse_bwd_kernel": {"achieved": gbps(ab["bwd"], t_bwd), "frac": gbps(ab["bwd"], t_bwd) / peak,
                                                  "us_per_launch": t_bwd * 1e3, "algorithmic_bytes_per_launch": ab["bwd"]},
                         "pool_fuse_fwd_kernel+mask": {"us_per_launch": t_pool_m * 1e3}},
                     "step": {"fwd_GBps": gbps(ab["fwd"], ms_fwd / K), "fwd_frac": gbps(ab["fwd"], ms_fwd / K) / peak,
                              "fwd_bwd_GBps": gbps(ab["fwd_bwd"], ms_train / K),
                              "fwd_bwd_frac": gbps(ab["fwd_bwd"], ms_train / K) / peak}},
        "shape_mode": {"workload": "same batch, per-shape scores: bins [B, V] (SURVEY.md 8d 'shape'; = the reference at batch "
                                   "size 1 per shape); score+bin and pool+fuse, 2 launches, no exchange",
                       "value": world * B * K / (ms_shape * 1e-3), "unit": UNIT, "ms_per_step": ms_shape / K,
                       "fwd_frac": gbps(ab["fwd"], ms_shape / K) / peak,
                       "fwd_bwd": {"value": world * B * K / (ms_train_shape * 1e-3), "ms_per_step": ms_train_shape / K,
                                   "frac_of_peak": gbps(ab["fwd_bwd"], ms_train_shape / K) / peak}},
        "fwd_bwd": {"workload": "training step (BASELINE.json configs[2]): forward with tie mask, backward dS->dF, %s"
                                % ("all-reduce (x 1/K) of the %d-float FC-score gradient bucket overlapped with the backward"
                                   % grad_bucket.numel() if world > 1 else "no collective at N=1"),
                    "value": world * B * K / (ms_train * 1e-3), "unit": UNIT, "ms_per_step": ms_train / K,
                    "algorithmic_GBps_per_gpu": gbps(ab["fwd_bwd"], ms_train / K),
                    "frac_of_peak": gbps(ab["fwd_bwd"], ms_train / K) / peak,
                    "allreduce_alone_us": us_allreduce, "allreduce_alone_us_nccl": us_allreduce_nccl},
        "api": {"what": "the same step through gvcnn_tf_b200.model (the Python mirror of nets/model.py), wall clock per "
                        "call incl. Python, allocator and launches; ratio = / the raw C-ABI graph-replayed step",
                "ms_per_step": api,
                "ratio_to_raw": {k: v / (raw_step["shape"] if "'shape'" in k else raw_step["batch"]) for k, v in api.items()},
                "reference_sequence_bits_equal_one_call_path": api_same},
        "e2e": {"value": world * B * Ke / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": Ke, "ms_per_step": 1e3 * e2e_s / Ke,
                "api": "gvcnn_grouping_fusion_host (C ABI, pinned host buffers, score_reduce=batch: R pass, batch mean, F "
                       "pass; chunk=%d shapes, 3-deep pipeline, %d copy-in stream(s), persistent gvcnn_host_pipeline)"
                       % (chunk, args.e2e_h2d_streams),
                "h2d_GBps": h2d / (e2e_s / Ke) / 1e9, "h2d_peak_gbs": h2d_peak_gbs,
                "frac": (h2d / (e2e_s / Ke) / 1e9) / h2d_peak_gbs,
                "h2d_peak_how": "one pinned cudaMemcpyAsync of the step's %d input bytes, all %d rank(s) at once, best of 3, "
                                "slowest rank" % (h2d, world),
                "host_path_bits_equal_device_path": e2e_same,
                "shape_mode": {"value": world * B * Ke / e2e_shape_s, "ms_per_step": 1e3 * e2e_shape_s / Ke,
                               "d2h_bytes_per_step": d2h_shape,
                               "frac": (h2d / (e2e_shape_s / Ke) / 1e9) / h2d_peak_gbs}},
        "gpu_launches": fwd_launches * K,
        "clocks": clocks,
    }
    if strong is not None:
        line["strong"] = strong
    line.update(extra)
    if world == 1 and not args.no_cpu_baseline:
        Bc = B                                                       # the full configs[1] batch
        times, threads = cpu_reference_time(Bc, 48, 2)               # ~10-15 s of CPU work
        best = min(times)
        line["cpu_baseline"] = {"value": Bc / best, "unit": UNIT, "cores": threads, "kind": "port", "cpu_model": cpu_model(),
                                "mean_value": Bc * len(times) / sum(times),
                                "sample": "best of %d forward passes over the full %d-shape batch (%.0f ms best, %.1f s of "
                                          "CPU work): the reference's op graph (nets/model.py:16-102) restated in "
                                          "torch-CPU, all host threads" % (len(times), Bc, best * 1e3, sum(times))}
    print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


# --------------------------------------------------------------------------- configs[3] and configs[0] (N = 1 extras)
def run_sweep(torch, C, L, dev, iters):
    """BASELINE.json configs[3]: V x G x D x dtype x pool, B = 4096 - every point timed THE SAME WAY as the headline
    (a CUDA graph of the PDL-chained step, replayed over rotating inputs), summarised as min / median fractions of
    the measured HBM peak.  scripts/sweep.py writes the full table."""
    from scripts import sweep as SW
    rows = SW.sweep(torch, C, L, dev, iters=iters, quick=False)
    peak = measured_peaks()[0]
    fwd = [r["fwd_frac"] for r in rows]
    trn = [r["train_frac"] for r in rows]
    worst = min(rows, key=lambda r: r["train_frac"])
    return {"workload": "configs[3]: V in {6,12,20,80} x G in {2,4,8,16} x D in {1024,2048} x {fp32,bf16} x {max,mean}, "
                        "B=4096, per-shape bins; each point = graph-replayed PDL step",
            "points": len(rows), "peak_GBps": peak,
            "fwd_frac": {"min": min(fwd), "median": statistics.median(fwd)},
            "train_frac": {"min": min(trn), "median": statistics.median(trn),
                           "below_0.70": sum(1 for t in trn if t < 0.70)},
            "worst_train_point": {k: worst[k] for k in ("dtype", "V", "G", "D", "pool", "train_frac", "train_us")}}


def run_config0(torch, model, dev):
    """BASELINE.json configs[0] restated to the head's share (SURVEY.md 8d): the reference's eval batch, 8 shapes x 6
    views of Inception Mixed_7c maps 8x8x2048, C_raw = 1024, num_group = 10, through eval.py's call sequence - the
    CPU port and the CUDA path timed on the same inputs."""
    from oracle import gvcnn_oracle_torch as OT
    B, V, h, w, Cc, Cr, G = 8, 6, 8, 8, 2048, 1024, 10
    g = torch.Generator().manual_seed(77)
    F = torch.randn((V, B, h, w, Cc), generator=g)
    R = torch.randn((B, V, Cr), generator=g)
    lim = math.sqrt(6.0 / (Cr + 1))
    W = (torch.rand((V, Cr), generator=g) * 2 - 1) * lim
    b = literal_bias(V)
    views_cpu = [F[v].reshape(B, -1).contiguous() for v in range(V)]
    torch.set_num_threads(os.cpu_count() or 1)
    cpu = []
    for i in range(12):
        t0 = time.perf_counter()
        S_cpu = OT.reference_step_cpu(views_cpu, R, W, b, G)
        float(S_cpu[0, 0])
        if i >= 2:
            cpu.append(time.perf_counter() - t0)
    Fd = [F[v].to(dev) for v in range(V)]
    Rd, Wd, bd = R.to(dev), W.to(dev), b.to(dev)

    def gpu_step():
        scores = model.view_scores(Rd, Wd, bd)
        scheme = model.group_scheme([scores[0]], G, V)
        return model.group_fusion(model.view_pooling(Fd, scheme), model.group_weight(scheme))
    with torch.no_grad():
        for _ in range(5):
            S_gpu = gpu_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n = 50
        for _ in range(n):
            S_gpu = gpu_step()
        torch.cuda.synchronize()
        gpu_s = (time.perf_counter() - t0) / n
    err = float((S_gpu.reshape(B, -1).cpu() - S_cpu).abs().max())
    return {"workload": "configs[0] head share: B=8, V=6, 8x8x2048 maps (D=131072), C_raw=1024, G=10, eval.py's call "
                        "sequence (scores -> group_scheme -> group_weight -> view_pooling -> group_fusion)",
            "cpu_port_ms": 1e3 * min(cpu), "cpu_cores": os.cpu_count(), "gpu_api_ms": 1e3 * gpu_s,
            "speedup": min(cpu) / gpu_s, "max_abs_diff_vs_cpu_port": err,
            "note": "GPU time is wall clock through the Python API with device-resident inputs, dominated by launch "
                    "latency at this size (25 MB of descriptors)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--e2e-chunk", type=int, default=256)
    ap.add_argument("--e2e-h2d-streams", type=int, default=1, choices=[1, 2])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the configs[3] / configs[0] extras of the N=1 line")
    ap.add_argument("--sweep-iters", type=int, default=6)
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: the library's one-kernel NVLink all-reduce (default) or torch.distributed/NCCL")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 4096 shapes per GPU (default, the contract's line); strong: 4096 shapes in total")
    ap.add_argument("--no-graph", action="store_true", help="time plain stream launches instead of a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed forward step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be >= 1")
    if args.dump_outputs and args.impl != "cuda":
        raise SystemExit("--dump-outputs applies to the CUDA arm only")
    if args.impl == "reference":
        return run_reference_arm(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch ourselves under torchrun, one rank per GPU
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_cuda_arm(args)


if __name__ == "__main__":
    sys.exit(main())
