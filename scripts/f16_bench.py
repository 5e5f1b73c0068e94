#!/usr/bin/env python
"""float16 descriptors against bfloat16 (and float32 for reference) on the same kernels:

  * configs[1] (B = 4096, V = 12, D = 2048, C_raw = 1024, G = 8): the literal forward step, the training step, and
    each kernel alone through the C ABI (score + bin, ring forward with and without tie planes, backward);
  * a sweep subset: V in {6, 12, 20}, D in {1024, 2048}, max and mean pooling, training step;
  * the GAP-folded real geometry (V = 12, G = 10, block3 10x10x1024, block4 10x10x2048, B = 32 / 128): the folded
    paper-mode step and the count-mode step (score_bin + pool_fuse_gap);
  * host memory end to end (gvcnn_grouping_fusion_host, literal mode, forward): shapes/s in float16 and float32,
    each timed call alternating with a pinned host-to-device copy that gives the link rate of that moment.

Three input sets per configuration, used in turn; each set's F (R too, from 128 shapes on) is larger than the 126 MB
L2, so no timed pass reads its inputs from L2.  The dtypes of a point are timed call by call in alternation
(f16, bf16, [f32], f16, ...), medians of CUDA-event times, and the whole point is repeated --repeats times so the
run-to-run spread is known.  One JSON line per point on stdout (and in --out).

    python scripts/f16_bench.py [--iters 20] [--repeats 3] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gvcnn_tf_b200 import _cabi as C, model  # noqa: E402

DT = {"f16": torch.float16, "bf16": torch.bfloat16, "f32": torch.float32}
CODE = {"f16": C.F16, "bf16": C.BF16, "f32": C.F32}
NSETS = 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:                                               # noqa: BLE001
        q = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def timed(fns, iters):
    """Median microseconds per call of each fn(i), the fns interleaved call by call (A B A B ...)."""
    for i in range(NSETS):
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


def repeated(names, fns, iters, repeats):
    """{name: {"us": median of the repeats' medians, "spread": [min, max]}}"""
    runs = [timed(fns, iters) for _ in range(repeats)]
    out = {}
    for j, n in enumerate(names):
        v = [r[j] for r in runs]
        out[n] = {"us": statistics.median(v), "spread": [min(v), max(v)]}
    return out


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def head_inputs(B, V, Cr, D, dnames, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    R32 = [torch.randn(B, V, Cr, device="cuda", generator=gen) for _ in range(NSETS)]
    F32 = [torch.relu(torch.randn(B, V, D, device="cuda", generator=gen)) for _ in range(NSETS)]
    W = (torch.rand(V, Cr, device="cuda", generator=gen) * 2 - 1) * (6.0 / (Cr + 1)) ** 0.5
    b = torch.rand(V, device="cuda", generator=gen) * 8 - 4
    dS32 = torch.randn(B, D, device="cuda", generator=gen)
    ins = {}
    for d in dnames:
        ins[d] = ([r.to(DT[d]) for r in R32], [f.to(DT[d]) for f in F32], dS32.to(DT[d]))
    return W, b, ins


def step_fns(W, b, ins, G, pool, fill, train):
    fns = []
    for d, (R, F, dS) in ins.items():
        Fg = [f.clone().requires_grad_(True) for f in F] if train else F

        def fn(i, R=R, Fg=Fg, dS=dS):
            k = i % NSETS
            if train:
                Fg[k].grad = None
                S, _ = model.grouping_fusion(R[k], W, b, Fg[k], G, pool=pool, empty_fill=fill, score_reduce="batch")
                S.backward(dS)
            else:
                model.grouping_fusion(R[k], W, b, Fg[k], G, pool=pool, empty_fill=fill, score_reduce="batch")
        fns.append(fn)
    return fns


def config1(iters, repeats):
    B, V, Cr, D, G = 4096, 12, 1024, 2048, 8
    dnames = ["f16", "bf16", "f32"]
    W, b, ins = head_inputs(B, V, Cr, D, dnames, 1)
    res = {"point": "configs[1]", "B": B, "V": V, "C_raw": Cr, "D": D, "G": G}
    res["forward_step"] = repeated(dnames, step_fns(W, b, ins, G, "max", 1.0, False), iters, repeats)
    res["training_step"] = repeated(dnames, step_fns(W, b, ins, G, "max", 1.0, True), iters, repeats)
    L = C.lib()
    x, sc = torch.empty(B, V, device="cuda"), torch.empty(B, V, device="cuda")
    bins, fl = (torch.empty(B, V, dtype=torch.int32, device="cuda") for _ in range(2))
    st = torch.zeros(4, dtype=torch.int32, device="cuda")
    bins.copy_(torch.randint(0, G, (B, V), dtype=torch.int32, device="cuda"))
    mask = torch.empty((V + 7) // 8, B, D, dtype=torch.uint8, device="cuda")
    kern = {"score": [], "ring_fwd": [], "ring_fwd_tie_planes": [], "bwd": []}
    for d in dnames:
        R, F, dS = ins[d]
        S = torch.empty(B, D, dtype=DT[d], device="cuda")
        dF = [torch.empty_like(f) for f in F]
        c = CODE[d]
        kern["score"].append(lambda i, R=R, c=c: C.check(L.gvcnn_score_bin_fwd(
            _ptr(R[i % NSETS]), _ptr(W), _ptr(b), _ptr(x), _ptr(sc), _ptr(bins), _ptr(fl), _ptr(st), B, V, Cr, G,
            C.LAYOUT_BVD, c, 4, 1, _stream()), "gvcnn_score_bin_fwd"))
        for key, m in (("ring_fwd", None), ("ring_fwd_tie_planes", mask)):
            kern[key].append(lambda i, F=F, S=S, c=c, m=m: C.check(L.gvcnn_pool_fuse_fwd(
                _ptr(F[i % NSETS]), _ptr(bins), V, None, 0, _ptr(S), None, _ptr(m), _ptr(st), B, V, D, G, C.POOL_MAX,
                ctypes.c_float(1.0), C.LAYOUT_BVD, c, _stream()), "gvcnn_pool_fuse_fwd"))
        kern["bwd"].append(lambda i, dS=dS, dF=dF, c=c: C.check(L.gvcnn_pool_fuse_bwd(
            _ptr(dS), _ptr(bins), V, None, 0, _ptr(mask), _ptr(dF[i % NSETS]), _ptr(st), B, V, D, G, C.POOL_MAX,
            C.LAYOUT_BVD, c, _stream()), "gvcnn_pool_fuse_bwd"))
    for k, fns in kern.items():
        res[k + "_kernel"] = repeated(dnames, fns, iters, repeats)
    return res


def sweep_point(V, D, pool, iters, repeats):
    B, Cr, G = 4096, 1024, 8
    fill = 1.0 if pool == "max" else 0.0
    dnames = ["f16", "bf16"]
    W, b, ins = head_inputs(B, V, Cr, D, dnames, V * D)
    return {"point": "sweep", "B": B, "V": V, "D": D, "G": G, "pool": pool,
            "training_step": repeated(dnames, step_fns(W, b, ins, G, pool, fill, True), iters, repeats)}


def gap_point(B, iters, repeats):
    V, G, CR, CF = 12, 10, 1024, 2048
    dnames = ["f16", "bf16"]
    gen = torch.Generator(device="cuda").manual_seed(B)
    R32 = [torch.randn(B, V, 10, 10, CR, device="cuda", generator=gen) for _ in range(NSETS)]
    F32 = [torch.relu(torch.randn(B, V, 10, 10, CF, device="cuda", generator=gen)) for _ in range(NSETS)]
    W = ((torch.rand(V, CR, device="cuda", generator=gen) * 2 - 1) * 0.0765).requires_grad_(True)
    b = torch.zeros(V, device="cuda", requires_grad=True)
    dOut32 = torch.randn(B, CF, device="cuda", generator=gen)
    paper, count = [], []
    for d in dnames:
        R = [r.to(DT[d]).requires_grad_(True) for r in R32]
        F = [f.to(DT[d]).requires_grad_(True) for f in F32]
        dOut = dOut32.to(DT[d])

        def clear(k, R=R, F=F):
            R[k].grad = F[k].grad = W.grad = b.grad = None

        def p(i, R=R, F=F, dOut=dOut, clear=clear):
            k = i % NSETS
            clear(k)
            S, *_ = model.grouping_fusion_paper(R[k], W, b, F[k], G, fold_gap=True)
            S.backward(dOut)

        def c(i, R=R, F=F, dOut=dOut, clear=clear):
            k = i % NSETS
            clear(k)
            sr = model.score_bin(R[k], W.detach(), b.detach(), G, score_reduce="batch", check=False)
            model.pool_fuse_gap(F[k], sr.bins, G).backward(dOut)
        paper.append(p)
        count.append(c)
    return {"point": "gap_folded_real_geometry", "B": B, "V": V, "G": G, "block3": [10, 10, CR], "block4": [10, 10, CF],
            "paper_step_folded": repeated(dnames, paper, iters, repeats),
            "count_step_folded": repeated(dnames, count, iters, repeats)}


def host_point(iters, repeats):
    """gvcnn_grouping_fusion_host, literal mode, forward only, B = 4096 shapes of configs[1] from pinned memory."""
    B, V, Cr, D, G, chunk = 4096, 12, 1024, 2048, 8, 256
    L = C.lib()
    gen = torch.Generator().manual_seed(7)
    W = ((torch.rand(V, Cr, generator=gen) * 2 - 1) * 0.0765).cuda()
    b = (torch.rand(V, generator=gen) * 8 - 4).cuda()
    pipe = ctypes.c_void_p()
    C.check(L.gvcnn_host_pipeline_create(ctypes.byref(pipe), 1), "gvcnn_host_pipeline_create")
    link_src = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
    link_dst = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res = {"point": "host_memory_literal_forward", "B": B, "V": V, "C_raw": Cr, "D": D, "G": G, "chunk_shapes": chunk}
    try:
        calls = {}
        for d in ("f16", "f32"):
            dt = DT[d]
            R = torch.randn(B, V, Cr, generator=gen).to(dt).pin_memory()
            F = torch.relu(torch.randn(B, V, D, generator=gen)).to(dt).pin_memory()
            S = torch.empty(B, D, dtype=dt).pin_memory()
            sc = torch.empty(V).pin_memory()
            bn = torch.empty(V, dtype=torch.int32).pin_memory()
            st = torch.zeros(4, dtype=torch.int32)
            nb = L.gvcnn_host_workspace_bytes(B, chunk, V, Cr, D, CODE[d], 0, C.SCORE_REDUCE_BATCH)
            ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
            calls[d] = (lambda R=R, F=F, S=S, sc=sc, bn=bn, st=st, ws=ws, nb=nb, c=CODE[d]: C.check(
                L.gvcnn_grouping_fusion_host(pipe, _ptr(R), _ptr(F), _ptr(W), _ptr(b), _ptr(S), _ptr(sc), _ptr(bn),
                                             None, None, _ptr(st), B, V, Cr, D, G, C.POOL_MAX, ctypes.c_float(1.0), c,
                                             C.SCORE_REDUCE_BATCH, B, None, None, chunk, _ptr(ws), nb),
                "gvcnn_grouping_fusion_host"), (V * Cr + V * D + D) * (4 if d == "f32" else 2))

        def wall(fn):
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            return time.perf_counter() - t

        def link():
            return link_src.numel() / wall(lambda: link_dst.copy_(link_src, non_blocking=True)) / 1e9
        for d in calls:
            calls[d][0]()                                         # warm-up
        link()
        samples = {d: [] for d in calls}
        links = {d: [] for d in calls}
        for _ in range(repeats):
            for _ in range(max(2, iters // 4)):
                for d, (fn, _) in calls.items():                  # f16, link, f32, link, ...
                    samples[d].append(wall(fn))
                    links[d].append(link())
        for d, (_, shape_bytes) in calls.items():
            t = statistics.median(samples[d])
            lk = statistics.median(links[d])
            res[d] = {"ms_per_call": t * 1e3, "spread_ms": [min(samples[d]) * 1e3, max(samples[d]) * 1e3],
                      "shapes_per_s": B / t, "link_GBps_h2d": lk,
                      "host_bytes_per_shape": shape_bytes, "share_of_link": B * shape_bytes / t / 1e9 / lk}
    finally:
        L.gvcnn_host_pipeline_destroy(pipe)
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("f16_bench.py measures the GPU: no CUDA device")
    out = open(a.out, "w") if a.out else None

    def emit(r):
        line = json.dumps(r)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()
    emit(card())
    emit(config1(a.iters, a.repeats))
    torch.cuda.empty_cache()
    for V in (6, 12, 20):
        for D in (1024, 2048):
            for pool in ("max", "mean"):
                emit(sweep_point(V, D, pool, a.iters, a.repeats))
                torch.cuda.empty_cache()
    for B in (32, 128):
        emit(gap_point(B, a.iters, a.repeats))
        torch.cuda.empty_cache()
    emit(host_point(a.iters, a.repeats))
    if out:
        out.close()


if __name__ == "__main__":
    main()
