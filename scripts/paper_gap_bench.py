#!/usr/bin/env python
"""Paper-mode training step at the reference's real geometry (V = 12, num_group = 10, block3 maps [N, 10, 10, 1024] into
the score FC, block4 maps [N, 10, 10, 2048] into the pooling), GAP after the fusion folded (grouping_fusion_paper
(fold_gap=True)) vs unfolded (fused map written, torch mean, gvcnn_pool_fuse_bwd_weights on dS), timed alternately;
the literal-mode folded step (score_bin + pool_fuse_gap) for context; and gvcnn_pool_fuse_gap_bwd_weights alone
against its F bytes, beside a device copy measured in the same run.

Two input sets per configuration, each larger than the 126 MB L2, used in turn, so no timed pass reads its F from L2.

    python scripts/paper_gap_bench.py [--batches 32,128] [--dtypes f32,bf16] [--iters 20]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gvcnn_tf_b200 import _cabi as C, model  # noqa: E402

V, G, HW, CR, CF = 12, 10, 100, 1024, 2048
DT = {"f32": torch.float32, "bf16": torch.bfloat16}


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:                                               # noqa: BLE001
        pl = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "power_limit": pl}


def timed(fns, iters):
    """Median microseconds per call of each fn(i), the fns interleaved call by call (A B A B ...)."""
    for i in range(3):
        for fn in fns:
            fn(i)
    torch.cuda.synchronize()
    ts = [[] for _ in fns]
    for i in range(iters):
        for j, fn in enumerate(fns):
            a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(i)
            c.record()
            c.synchronize()
            ts[j].append(a.elapsed_time(c) * 1e3)
    return [statistics.median(t) for t in ts]


def copy_peak_gbps(iters):
    n = 1 << 28                                                   # 1 GiB per buffer
    src = [torch.empty(n, dtype=torch.float32, device="cuda").fill_(1.0) for _ in range(2)]
    dst = torch.empty(n, dtype=torch.float32, device="cuda")
    (t,) = timed([lambda i: dst.copy_(src[i % 2])], iters)
    return 2 * n * 4 / (t * 1e-6) / 1e9


def bench(B, dname, iters):
    dt = DT[dname]
    es = 4 if dt == torch.float32 else 2
    gen = torch.Generator(device="cuda").manual_seed(B)
    R = [torch.randn(B, V, 10, 10, CR, device="cuda", generator=gen).to(dt).requires_grad_(True) for _ in range(2)]
    F = [torch.relu(torch.randn(B, V, 10, 10, CF, device="cuda", generator=gen)).to(dt).requires_grad_(True)
         for _ in range(2)]
    W = ((torch.rand(V, CR, device="cuda", generator=gen) * 2 - 1) * 0.0765).requires_grad_(True)
    b = torch.zeros(V, device="cuda", requires_grad=True)
    dOut = torch.randn(B, CF, device="cuda", generator=gen).to(dt)

    def clear(i):
        R[i % 2].grad = F[i % 2].grad = W.grad = b.grad = None   # no accumulation kernels in the timed window

    def folded(i):
        clear(i)
        S, *_ = model.grouping_fusion_paper(R[i % 2], W, b, F[i % 2], G, fold_gap=True)
        S.backward(dOut)

    def unfolded(i):
        clear(i)
        S, *_ = model.grouping_fusion_paper(R[i % 2], W, b, F[i % 2], G)
        model._spatial_mean(S).backward(dOut)

    def literal(i):
        clear(i)
        sr = model.score_bin(R[i % 2], W.detach(), b.detach(), G, score_reduce="batch", check=False)
        model.pool_fuse_gap(F[i % 2], sr.bins, G).backward(dOut)

    t_fold, t_unfold, t_lit = timed([folded, unfolded, literal], iters)

    # the weight-gradient kernel alone (+ its finish kernel), on the same F sets
    L = C.lib()
    dc = C.F32 if dt == torch.float32 else C.BF16
    Fd = [f.detach() for f in F]
    bins = torch.randint(0, G, (B, V), dtype=torch.int32, device="cuda", generator=gen)
    wts = torch.rand(B, G, device="cuda", generator=gen)
    S_gap = torch.randn(B, CF, device="cuda", generator=gen).to(dt)
    dw = torch.empty(B, G, device="cuda")
    wsb = L.gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes(B, V, HW, CF, dc)
    ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def kern(i):
        C.check(L.gvcnn_pool_fuse_gap_bwd_weights(Fd[i % 2].data_ptr(), dOut.data_ptr(), S_gap.data_ptr(), bins.data_ptr(),
                                                  V, wts.data_ptr(), G, dw.data_ptr(), ws.data_ptr(), wsb, B, V, HW, CF, G,
                                                  C.POOL_MAX, C.LAYOUT_BVD, dc, st), "gvcnn_pool_fuse_gap_bwd_weights")
    (t_k,) = timed([kern], iters)
    f_bytes = B * V * HW * CF * es
    return {"B": B, "dtype": dname, "V": V, "G": G, "block3": [10, 10, CR], "block4": [10, 10, CF],
            "F_MB_per_set": f_bytes / 1e6, "R_MB_per_set": B * V * HW * CR * es / 1e6,
            "paper_step_folded_us": t_fold, "paper_step_unfolded_us": t_unfold,
            "folded_speedup": t_unfold / t_fold, "literal_step_folded_us": t_lit,
            "bwd_weights_kernel_us": t_k, "bwd_weights_F_read_GBps": f_bytes / (t_k * 1e-6) / 1e9}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--batches", default="32,128")
    ap.add_argument("--dtypes", default="f32,bf16")
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("paper_gap_bench.py measures the GPU: no CUDA device")
    info = card()
    info["copy_peak_GBps"] = copy_peak_gbps(a.iters)      # read + write bytes over time, 1 GiB buffers
    print(json.dumps(info), flush=True)
    for dname in a.dtypes.split(","):
        for B in (int(x) for x in a.batches.split(",")):
            r = bench(B, dname, a.iters)
            r["bwd_weights_share_of_copy_peak"] = r["bwd_weights_F_read_GBps"] / info["copy_peak_GBps"]
            print(json.dumps(r), flush=True)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
