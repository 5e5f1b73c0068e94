#!/usr/bin/env python
"""What data_format='channels_first' costs against channel-last maps, at the reference geometry (V = 12, block3
10 x 10 x 1024, block4 10 x 10 x 2048), B = 32 and 128, float32 and bfloat16.  Three arms per point:

  a  NCHW maps (contiguous) through the channels-first kernels;
  b  NHWC maps through the channel-last kernels - the ceiling;
  c  NCHW maps through the route a PyTorch user had before: permute(0, 2, 3, 1).contiguous() in, dF permuted back.

Workloads: `gap_score` (score_bin on the block3 maps, per-shape bins), `fgap_fwd` (pool_fuse_gap forward on the block4
maps), `fgap_bwd` (its backward, dF from the [B, C] gradient) and `step` (GVCNNHead count mode with fold_gap: forward,
classifier loss, backward).  Compulsory bytes: the maps read (gap_score, fgap_fwd), dF written (fgap_bwd).  A
device-to-device copy of the block4 maps in the same run gives the copy rate of the moment.  Input sets are rotated
past twice the 126 MB L2.  Calls of the three arms are timed in alternation (CUDA events, medians of --iters).  With
--profile the torch.profiler kernel times of each arm at B = 128 are added.  One JSON line per point in --out
(the first holds the card's name and power limit) and a table in the .md next to it.

    python scripts/channels_first_bench.py [--iters 20] [--out profiles/r08_channels_first_bench.jsonl] [--profile]
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
from gvcnn_tf_b200 import model  # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16}
L2 = 126 << 20
V, G, HW, C3, C4, K = 12, 10, 100, 1024, 2048, 40


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:                                               # noqa: BLE001
        q = "unknown"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def timed(fns, iters, warm=3):
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


def kernel_times(fn, n=5):
    """torch.profiler: CUDA kernel time per call by kernel name (us), over n calls."""
    from torch.profiler import ProfilerActivity, profile
    fn(0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t > 0:
            out[e.key[:90]] = round(t / n, 2)
    return dict(sorted(out.items(), key=lambda kv: -kv[1])[:8])


def nchw_to_nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def point(B, dtn, iters, prof):
    dt = DT[dtn]
    es = torch.empty((), dtype=dt).element_size()
    b3, b4 = B * C3 * HW * es, B * C4 * HW * es
    nset = max(1, -(-2 * L2 // (V * (b3 + b4))))
    gen = torch.Generator(device="cuda").manual_seed(B)
    sets = []
    for _ in range(nset):
        R = [torch.randn(B, C3, 10, 10, device="cuda", generator=gen).to(dt) for _ in range(V)]
        F = [torch.randn(B, C4, 10, 10, device="cuda", generator=gen).to(dt) for _ in range(V)]
        sets.append({"R": R, "F": F, "Rl": [nchw_to_nhwc(t) for t in R], "Fl": [nchw_to_nhwc(t) for t in F]})
    W = torch.randn(V, C3, device="cuda") * 0.03
    bias = torch.zeros(V, device="cuda")
    bins = torch.randint(0, G, (B, V), device="cuda", dtype=torch.int32)
    dOut = torch.randn(B, C4, device="cuda").to(dt)
    rows = []

    def emit(work, arms, nbytes):
        rec = {"work": work, "B": B, "dtype": dtn, "V": V, "sets": nset,
               "us": {k: round(v, 2) for k, v in arms.items()}}
        if nbytes:
            rec["GBps"] = {k: round(nbytes / v / 1e3, 1) for k, v in arms.items()}
        rows.append(rec)

    cf = "channels_first"
    sb = {
        "a": lambda i: model.score_bin(sets[i % nset]["R"], W, bias, G, check=False, data_format=cf),
        "b": lambda i: model.score_bin(sets[i % nset]["Rl"], W, bias, G, check=False),
        "c": lambda i: model.score_bin([nchw_to_nhwc(t) for t in sets[i % nset]["R"]], W, bias, G, check=False),
    }
    emit("gap_score", dict(zip(sb, timed(list(sb.values()), iters))), V * b3)
    fw = {
        "a": lambda i: model.pool_fuse_gap(sets[i % nset]["F"], bins, G, data_format=cf),
        "b": lambda i: model.pool_fuse_gap(sets[i % nset]["Fl"], bins, G),
        "c": lambda i: model.pool_fuse_gap([nchw_to_nhwc(t) for t in sets[i % nset]["F"]], bins, G),
    }
    emit("fgap_fwd", dict(zip(fw, timed(list(fw.values()), iters))), V * b4)

    # backward alone: one forward per arm and set, its graph kept; the timed call is autograd.grad from dOut
    graphs = {}
    for arm in ("a", "b", "c"):
        graphs[arm] = []
        for s in sets:
            leaves = [t.detach().requires_grad_(True) for t in (s["Fl"] if arm == "b" else s["F"])]
            ins = [nchw_to_nhwc(t) for t in leaves] if arm == "c" else leaves
            out = model.pool_fuse_gap(ins, bins, G, data_format=cf if arm == "a" else "channels_last")
            graphs[arm].append((out, leaves))

    def bwd(arm):
        return lambda i: torch.autograd.grad(graphs[arm][i % nset][0], graphs[arm][i % nset][1], dOut,
                                             retain_graph=True)
    bw = {k: bwd(k) for k in ("a", "b", "c")}
    emit("fgap_bwd", dict(zip(bw, timed(list(bw.values()), iters))), V * b4)
    del graphs

    heads = {}
    for arm in ("a", "b", "c"):
        torch.manual_seed(0)
        heads[arm] = model.GVCNNHead(V, C3, C4, K, score_reduce="shape", data_format=cf if arm == "a" else
                                     "channels_last").cuda()

    def step(arm):
        def run(i):
            s = sets[i % nset]
            if arm == "b":
                r, f = [t.detach().requires_grad_(True) for t in s["Rl"]], [t.detach().requires_grad_(True) for t in s["Fl"]]
                ri, fi = r, f
            else:
                r, f = [t.detach().requires_grad_(True) for t in s["R"]], [t.detach().requires_grad_(True) for t in s["F"]]
                ri, fi = (r, f) if arm == "a" else ([nchw_to_nhwc(t) for t in r], [nchw_to_nhwc(t) for t in f])
            _, _, logits = heads[arm](ri, fi, fold_gap=True)
            logits.float().square().mean().backward()
        return run
    st = {k: step(k) for k in ("a", "b", "c")}
    emit("step", dict(zip(st, timed(list(st.values()), iters))), 0)

    src = sets[0]["F"][0]
    dst = torch.empty_like(src)
    t = timed([lambda i: dst.copy_(src)], iters)[0]
    rows.append({"work": "copy", "B": B, "dtype": dtn, "us": round(t, 2), "GBps": round(2 * src.numel() * es / t / 1e3, 1)})
    if prof and B == 128:
        for work, fns in (("gap_score", sb), ("fgap_fwd", fw), ("step", st)):
            rows.append({"work": work + "_kernels", "B": B, "dtype": dtn,
                         "kernels_us": {k: kernel_times(fn) for k, fn in fns.items()}})
    return rows


def write_md(path, head, rows):
    lines = ["# data_format='channels_first': NCHW maps through the channels-first kernels", "",
             "Card: %s (%s).  Written by `scripts/channels_first_bench.py`.  V = 12, block3 10x10x1024, block4 "
             "10x10x2048.  Arms: a = NCHW through the new kernels, b = NHWC through the channel-last kernels (the "
             "ceiling), c = NCHW permuted to NHWC with `.contiguous()` (and dF permuted back).  Medians, us; rates are "
             "compulsory bytes over time." % (head["gpu"], head["nvidia_smi"]), "",
             "| work | B | dtype | a us | b us | c us | a GB/s | b GB/s | a / b rate |", "|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        if "us" in r and isinstance(r["us"], dict):
            g = r.get("GBps", {})
            ratio = "%.3f" % (g["a"] / g["b"]) if g else "%.3f" % (r["us"]["b"] / r["us"]["a"])
            lines.append("| %s | %d | %s | %.1f | %.1f | %.1f | %s | %s | %s |" % (
                r["work"], r["B"], r["dtype"], r["us"]["a"], r["us"]["b"], r["us"]["c"], g.get("a", "-"),
                g.get("b", "-"), ratio))
    lines += ["", "Copy rate in the same run:", ""]
    for r in rows:
        if r["work"] == "copy":
            lines.append("- B = %d %s: %.1f GB/s (device-to-device copy of one view's block4 maps)" % (
                r["B"], r["dtype"], r["GBps"]))
    kern = [r for r in rows if r["work"].endswith("_kernels")]
    if kern:
        lines += ["", "torch.profiler kernel times (us per call), B = 128:", ""]
        for r in kern:
            for arm, ks in r["kernels_us"].items():
                lines.append("- %s %s arm %s: %s" % (r["work"][:-8], r["dtype"], arm,
                                                     ", ".join("%s %.1f" % kv for kv in ks.items())))
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_channels_first_bench.jsonl"))
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--batches", default="32,128")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    head = card()
    rows = []
    for B in [int(x) for x in a.batches.split(",")]:
        for dtn in DT:
            for r in point(B, dtn, a.iters, a.profile):
                print(json.dumps(r), flush=True)
                rows.append(r)
            torch.cuda.empty_cache()
    with open(a.out, "w") as f:
        f.write(json.dumps(head) + "\n")
        for r in rows:
            f.write(json.dumps(r) + "\n")
    write_md(os.path.splitext(a.out)[0] + ".md", head, rows)


if __name__ == "__main__":
    main()
