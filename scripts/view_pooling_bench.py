#!/usr/bin/env python
"""gvcnn_view_pooling_bwd (the gradient of view_pooling's G group descriptors, dP [G, B, D] -> dF) at configs[1]'s
size and a few neighbours, against what the same run can do otherwise:

  * vp_bwd        gvcnn_view_pooling_bwd through the C ABI, the library's automatic kernel choice;
  * pf_bwd        gvcnn_pool_fuse_bwd (dS [B, D] -> dF) at the same shape and bins;
  * copy          a device-to-device copy of V * D elements per shape (torch copy_): the copy rate of the moment;
  * fwd_groups    the materialising forward, gvcnn_pool_fuse_fwd with group_desc (and the tie planes for max);
  * preload       (when --alt names a library built with -DGVCNN_VP_BWD_PRELOAD=1) vp_bwd with every group row of a
                  shape loaded right after the plan barrier instead of at each group start;
  * chain         model.view_pooling + autograd backward of all G entries (materialise + vp_bwd + torch plumbing);
  * torch_eager   the same through torch eager autograd of the reference graph, oracle/gvcnn_oracle_torch.view_pooling
                  (stack, index_select, amax / sum, per group) on the GPU: what a user writes without this library.

One scheme per batch (the reference's [G, V] scheme), drawn from a fixed seed; M = the non-empty groups.  Three input
and output sets, used in turn, each larger than the 126 MB L2.  The kernels of one point are timed call by call in
alternation (CUDA events, medians), the whole point --repeats times.  Compulsory bytes: vp_bwd reads M rows of dP and
writes V rows of dF per shape, (M + V) * D * s, plus ceil(V / 8) * D bytes of tie planes for max; pf_bwd reads one dS
row: (1 + V) * D * s (+ planes).  One JSON line per point on stdout and in --out.

    python scripts/view_pooling_bench.py [--iters 20] [--repeats 3] [--out FILE] [--alt LIB]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gvcnn_tf_b200 import _cabi as C, model  # noqa: E402
from oracle import gvcnn_oracle_torch as T  # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16}
CODE = {"f32": C.F32, "bf16": C.BF16}
NSETS = 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:                                               # noqa: BLE001
        q = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def timed(fns, iters):
    """Median microseconds per call of each fn(i), the fns interleaved call by call (A B C A B C ...)."""
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
    runs = [timed(fns, iters) for _ in range(repeats)]
    return {n: {"us": statistics.median([r[j] for r in runs]),
                "spread": [min(r[j] for r in runs), max(r[j] for r in runs)]} for j, n in enumerate(names)}


def p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def point(L, alt, dname, pool, B, V, D, G, iters, repeats, eager_iters):
    dt, code = DT[dname], CODE[dname]
    s = torch.finfo(dt).bits // 8
    fill = 1.0 if pool == "max" else 0.0
    gen = torch.Generator(device="cuda").manual_seed(V * 100 + D)
    brow = np.random.default_rng(V).integers(0, G, V).astype(np.int32)
    M = len(set(brow.tolist()))
    bins = torch.as_tensor(brow).cuda()[None]
    scheme = torch.as_tensor((brow[None, :] == np.arange(G)[:, None]).astype(np.int32)).cuda()
    F = [torch.relu(torch.randn(B, V, D, device="cuda", generator=gen)).to(dt) for _ in range(NSETS)]
    dP = [torch.randn(G, B, D, device="cuda", generator=gen).to(dt) for _ in range(NSETS)]
    dS = [torch.randn(B, D, device="cuda", generator=gen).to(dt) for _ in range(NSETS)]
    dF = [torch.empty(B, V, D, device="cuda", dtype=dt) for _ in range(NSETS)]
    S = [torch.empty(B, D, device="cuda", dtype=dt) for _ in range(NSETS)]
    P = [torch.empty(G, B, D, device="cuda", dtype=dt) for _ in range(NSETS)]
    mask = [torch.empty((V + 7) // 8, B, D, device="cuda", dtype=torch.uint8) if pool == "max" else None
            for _ in range(NSETS)]
    pc = C.POOL_MAX if pool == "max" else C.POOL_MEAN
    for k in range(NSETS):                                  # the tie planes the backward reads
        C.check(L.gvcnn_pool_fuse_fwd(p(F[k]), p(bins), 0, None, 0, p(S[k]), p(P[k]), p(mask[k]), None, B, V, D, G, pc,
                                      ctypes.c_float(fill), C.LAYOUT_BVD, code, stream()), "fwd")
    torch.cuda.synchronize()

    def vp(lib):
        def fn(i):
            k = i % NSETS
            C.check(lib.gvcnn_view_pooling_bwd(p(dP[k]), p(bins), 0, p(mask[k]), p(dF[k]), None, B, V, D, G, pc,
                                               C.LAYOUT_BVD, code, stream()), "gvcnn_view_pooling_bwd")
        return fn

    def pf(i):
        k = i % NSETS
        C.check(L.gvcnn_pool_fuse_bwd(p(dS[k]), p(bins), 0, None, 0, p(mask[k]), p(dF[k]), None, B, V, D, G, pc,
                                      C.LAYOUT_BVD, code, stream()), "gvcnn_pool_fuse_bwd")

    def copy(i):
        k = i % NSETS
        dF[k].copy_(F[(k + 1) % NSETS])

    def fwd_groups(i):
        k = i % NSETS
        C.check(L.gvcnn_pool_fuse_fwd(p(F[k]), p(bins), 0, None, 0, p(S[k]), p(P[k]), p(mask[k]), None, B, V, D, G,
                                      pc, ctypes.c_float(fill), C.LAYOUT_BVD, code, stream()), "gvcnn_pool_fuse_fwd")

    names, fns = ["vp_bwd", "pf_bwd", "copy", "fwd_groups"], [vp(L), pf, copy, fwd_groups]
    if alt is not None and pool == "max":
        names.append("preload")
        fns.append(vp(alt))
    res = {"point": "%s %s V=%d D=%d" % (dname, pool, V, D), "dtype": dname, "pool": pool, "B": B, "V": V, "D": D,
           "G": G, "M": M, "bins": brow.tolist()}
    res["kernels"] = repeated(names, fns, iters, repeats)

    planes = (V + 7) // 8 * B * D if pool == "max" else 0
    by_vp = (M + V) * B * D * s + planes
    by_pf = (1 + V) * B * D * s + planes
    by_copy = 2 * V * B * D * s
    kt = res["kernels"]
    res["bytes"] = {"vp_bwd": by_vp, "pf_bwd": by_pf, "copy": by_copy}
    res["GBps"] = {"vp_bwd": by_vp / kt["vp_bwd"]["us"] / 1e3, "pf_bwd": by_pf / kt["pf_bwd"]["us"] / 1e3,
                   "copy": by_copy / kt["copy"]["us"] / 1e3}
    if "preload" in kt:
        res["GBps"]["preload"] = by_vp / kt["preload"]["us"] / 1e3
    res["vp_over_pf_rate"] = res["GBps"]["vp_bwd"] / res["GBps"]["pf_bwd"]
    res["vp_over_copy_rate"] = res["GBps"]["vp_bwd"] / res["GBps"]["copy"]

    # whole chains: the library through autograd, and torch eager on the reference graph (fewer iterations: slow)
    Fg = [f.clone().requires_grad_(True) for f in F]
    Fl = [[f[:, v].contiguous().requires_grad_(True) for v in range(V)] for f in F]

    def chain(i):
        k = i % NSETS
        Fg[k].grad = None
        d = model.view_pooling(Fg[k], scheme, pool=pool, empty_fill=fill)
        torch.autograd.backward([d[g] for g in range(G)], list(dP[k]))

    def eager(i):
        k = i % NSETS
        for v in Fl[k]:
            v.grad = None
        d = T.view_pooling(Fl[k], scheme, pool=pool, empty_fill=fill)
        outs = [(d[g], dP[k][g]) for g in range(G) if d[g].requires_grad]
        torch.autograd.backward([o for o, _ in outs], [g for _, g in outs])

    res["chain"] = repeated(["library", "torch_eager"], [chain, eager], eager_iters, repeats)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--eager-iters", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--alt", default=None, help="a library built with -DGVCNN_VP_BWD_PRELOAD=1 (A/B of the row loads)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    L = C.lib()
    alt = None
    if args.alt:
        alt = ctypes.CDLL(os.path.abspath(args.alt))
        alt.gvcnn_view_pooling_bwd.restype, alt.gvcnn_view_pooling_bwd.argtypes = C.SIGNATURES["gvcnn_view_pooling_bwd"]
    head = {"card": card()}
    print(json.dumps(head), flush=True)
    lines = [head]
    B, G = 4096, 8
    pts = [(d, pool, V, 2048) for d in ("f32", "bf16") for V in (12, 20) for pool in ("max", "mean")]
    pts += [("bf16", pool, V, 1024) for V in (12, 20) for pool in ("max", "mean")]
    for d, pool, V, D in pts:
        r = point(L, alt, d, pool, B, V, D, G, args.iters, args.repeats, args.eager_iters)
        print(json.dumps(r), flush=True)
        lines.append(r)
        torch.cuda.empty_cache()
    lines.append({"card_after": card()})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
