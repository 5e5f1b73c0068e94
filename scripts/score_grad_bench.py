#!/usr/bin/env python
"""The view-score backward (gvcnn_score_bin_bwd + gvcnn_view_score_bwd [+ gvcnn_gap_score_bwd]) and what the
differentiable scores cost a training step:

  * tail_pooled   configs[1] (B = 4096, V = 12, C_raw = 1024), float32 and bfloat16 R, both score modes: the whole score
                  backward from dscores to dW, db, with and without dR.  Compulsory bytes: R read (+ dR written).
  * copy          a device-to-device copy of the same R bytes (torch copy_), in the same run: the copy rate of the moment.
  * tail_maps     the reference geometry (B = 128, V = 12, block3 10 x 10 x 1024), float32 and bfloat16 maps: the score
                  backward with dmaps (dW, db from the pooled float32 R_out; dmaps = dx W / HW).
  * head_step     GVCNNHead count mode on those maps (final maps 10 x 10 x 2048), forward + classifier loss + backward,
                  with the score FC frozen (requires_grad False) and trainable: the latter adds the R_out write to the
                  score kernel (B * V * C_raw * 4 bytes, about 1/HW of the maps' read).

Input sets larger than the 126 MB L2 are rotated (each point uses enough sets to exceed twice the L2).  Calls of one
point are timed in alternation (CUDA events, medians of --iters), the point --repeats times.  One JSON line per point
on stdout and in --out; the first line holds the card's name and power limit.

    python scripts/score_grad_bench.py [--iters 20] [--repeats 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gvcnn_tf_b200 import _cabi as C, model  # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16}
CODE = {"f32": C.F32, "bf16": C.BF16}
L2 = 126 << 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:                                               # noqa: BLE001
        q = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def nsets(nbytes):
    return max(1, -(-2 * L2 // max(nbytes, 1)))


def timed(fns, iters, warm):
    """Median microseconds per call of each fn(i), the fns interleaved call by call."""
    for i in range(warm):
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


def repeated(names, fns, iters, repeats, warm):
    runs = [timed(fns, iters, warm) for _ in range(repeats)]
    return {n: {"us": round(statistics.median([r[j] for r in runs]), 2),
                "spread": [round(min(r[j] for r in runs), 2), round(max(r[j] for r in runs), 2)]}
            for j, n in enumerate(names)}


def p(t):
    return None if t is None else (t.data_ptr() or None)


def s():
    return torch.cuda.current_stream().cuda_stream or None


def tail_point(L, dname, mode, B, V, Cr, HW, iters, repeats):
    """The score backward from dscores [rows, V] on rotated R (or maps) sets."""
    dt, code = DT[dname], CODE[dname]
    es = torch.finfo(dt).bits // 8
    per = B * V * Cr * HW * es
    n = nsets(per)
    g = torch.Generator(device="cuda").manual_seed(B + V + Cr + HW)
    R = [torch.randn((B, V, Cr * HW), device="cuda", generator=g).to(dt) for _ in range(n)]
    dR = [torch.empty_like(r) for r in R]
    R_out = [torch.randn((B, V, Cr), device="cuda", generator=g) for _ in range(n)] if HW > 1 else None
    W = torch.randn((V, Cr), device="cuda", generator=g) * Cr ** -0.5
    rows = 1 if mode == "batch" else B
    ds = torch.randn((rows, V), device="cuda", generator=g)
    xs = torch.randn((rows, V), device="cuda", generator=g)
    sc = xs.abs() / (1 + xs.abs())
    dx, dxm = torch.empty((B, V), device="cuda"), torch.empty(V, device="cuda")
    dW, db = torch.empty_like(W), torch.empty(V, device="cuda")
    ws_bytes = L.gvcnn_view_score_bwd_workspace_bytes(V, Cr)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    red = C.SCORE_REDUCE_BATCH if mode == "batch" else C.SCORE_REDUCE_SHAPE

    def tail():
        C.check(L.gvcnn_score_bin_bwd(p(ds), p(xs), p(sc), p(dxm) if mode == "batch" else None, p(dx), B, V, red,
                                      B if mode == "batch" else 0, None, None, s()), "score_bin_bwd")

    def run(i, want_dr):
        tail()
        if HW > 1:
            C.check(L.gvcnn_view_score_bwd(p(R_out[i % n]), p(dx), p(W), p(dW), p(db), None, p(ws), ws_bytes, B, V, Cr,
                                           C.LAYOUT_BVD, C.F32, s()), "view_score_bwd")
            C.check(L.gvcnn_gap_score_bwd(p(dx), p(W), p(dR[i % n]), B, V, HW, Cr, C.LAYOUT_BVD, code, s()),
                    "gap_score_bwd")
        else:
            C.check(L.gvcnn_view_score_bwd(p(R[i % n]), p(dx), p(W), p(dW), p(db), p(dR[i % n]) if want_dr else None,
                                           p(ws), ws_bytes, B, V, Cr, C.LAYOUT_BVD, code, s()), "view_score_bwd")

    src = [torch.empty(per, dtype=torch.uint8, device="cuda") for _ in range(n)]
    dst = [torch.empty_like(t) for t in src]
    names, fns = [], []
    if HW > 1:
        names += ["bwd_dmaps"]
        fns += [lambda i: run(i, True)]
    else:
        names += ["bwd", "bwd_dR"]
        fns += [lambda i: run(i, False), lambda i: run(i, True)]
    names += ["tail_only", "copy"]
    fns += [lambda i: tail(), lambda i: dst[i % n].copy_(src[i % n])]
    res = repeated(names, fns, iters, repeats, n)
    copy_rate = 2 * per / (res["copy"]["us"] * 1e-6) / 1e9
    out = {"point": "tail_maps" if HW > 1 else "tail_pooled", "dtype": dname, "mode": mode, "B": B, "V": V, "C": Cr,
           "HW": HW, "sets": n, "copy_GBps": round(copy_rate, 1), "timings": res}
    for k in names[:-2]:
        if HW > 1:
            byts = B * V * Cr * 4 + per                         # R_out read, dmaps written
        else:
            byts = per * (2 if k == "bwd_dR" else 1)            # R read (+ dR written)
        gbps = byts / (res[k]["us"] * 1e-6) / 1e9
        out[k] = {"bytes": byts, "GBps": round(gbps, 1), "of_copy_rate": round(gbps / copy_rate, 3)}
    return out


def head_point(dname, mode, B, V, iters, repeats):
    """GVCNNHead count mode on block3 maps: one training step, score FC frozen vs trainable."""
    dt = DT[dname]
    Cr, Cf, HW = 1024, 2048, 100
    per = B * V * HW * (Cr + Cf) * (torch.finfo(dt).bits // 8)
    n = nsets(per)
    g = torch.Generator(device="cuda").manual_seed(17)
    raw = [torch.randn((B, V, 10, 10, Cr), device="cuda", generator=g).to(dt) for _ in range(n)]
    fin = [torch.randn((B, V, 10, 10, Cf), device="cuda", generator=g).to(dt).requires_grad_(True) for _ in range(n)]
    labels = torch.randint(0, 40, (B,), device="cuda", generator=g)
    head = model.GVCNNHead(V, Cr, Cf, 40, score_reduce=mode).cuda()

    def step(i, trainable):
        head.score_kernel.requires_grad_(trainable)
        head.score_bias.requires_grad_(trainable)
        _, _, logits = head(raw[i % n], fin[i % n], fold_gap=True)
        torch.nn.functional.cross_entropy(logits, labels).backward()
        fin[i % n].grad = None

    res = repeated(["frozen_fc", "trainable_fc"], [lambda i: step(i, False), lambda i: step(i, True)], iters, repeats, n)
    return {"point": "head_step", "dtype": dname, "mode": mode, "B": B, "V": V, "maps": [10, 10, Cr], "final": [10, 10, Cf],
            "sets": n, "R_out_bytes": B * V * Cr * 4, "maps_bytes": B * V * HW * Cr * (torch.finfo(dt).bits // 8),
            "timings": res, "trainable_minus_frozen_us": round(res["trainable_fc"]["us"] - res["frozen_fc"]["us"], 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_grad_bench.py needs a CUDA device")
    L = C.lib()
    lines = [card()]
    for dname in ("f32", "bf16"):
        for mode in ("shape", "batch"):
            lines.append(tail_point(L, dname, mode, 4096, 12, 1024, 1, a.iters, a.repeats))
    for dname in ("f32", "bf16"):
        for mode in ("shape", "batch"):
            lines.append(tail_point(L, dname, mode, 128, 12, 1024, 100, a.iters, a.repeats))
    for dname in ("f32", "bf16"):
        lines.append(head_point(dname, "batch", 128, 12, a.iters, a.repeats))
    lines.append(card())
    out = open(a.out, "w") if a.out else None
    for ln in lines:
        js = json.dumps(ln)
        print(js, flush=True)
        if out:
            out.write(js + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
