"""Builds libgvcnn_sm100.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python gvcnn-tf_b200/build.py [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libgvcnn_sm100.so")
SOURCES = ["capi.cu", "host_pipeline.cu", "comm.cu", "score.cu", "gap_score.cu", "scheme.cu", "pool_fwd.cu", "pool_fwd_ring.cu", "pool_fwd_direct.cu", "pool_gap_ring.cu", "pool_bwd.cu", "pool_bwd_fast.cu", "paper_mode.cu", "paper_gap.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "ring_common.cuh"), os.path.join(ROOT, "include", "gvcnn_b200.h")]


def nvcc_path():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libgvcnn_sm100.so cannot be built (there is no fallback path)")


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, defines=(), out=None):
    """Compiles every source to an object file in parallel (one nvcc per file), then links the shared library.
    defines / out: A/B builds of the same sources with -D flags into another path (scripts/_build/)."""
    if out is None and not force and not needs_build():
        return SO
    import concurrent.futures
    import hashlib
    import tempfile
    target = out or SO
    common = [nvcc_path()]
    if os.path.exists("/usr/bin/g++"):      # the image's $CC/$CXX wrappers are not what nvcc should use as host compiler
        common += ["-ccbin", "/usr/bin/g++"]
    common += ["-std=c++17", "-O3", "-lineinfo",
               "-gencode", "arch=compute_100a,code=sm_100a",
               "-fmad=false",                      # one rounding per float32 op unless fmaf() is written
               "-Xcompiler", "-fPIC",
               "-I", os.path.join(ROOT, "include"), "-I", CSRC] + ["-D" + d for d in defines]
    if verbose:
        common.insert(1, "-Xptxas=-v")
    tag = hashlib.sha1((" ".join(defines) + target).encode()).hexdigest()[:10]
    objdir = os.path.join(tempfile.gettempdir(), "gvcnn_build_" + tag)
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        res = subprocess.run(common + ["-c", os.path.join(CSRC, src), "-o", obj], capture_output=True, text=True)
        return src, obj, res

    log = []
    objs = []
    with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        for src, obj, res in ex.map(compile_one, SOURCES):
            log.append(res.stdout + res.stderr)
            if res.returncode != 0:
                sys.stderr.write("".join(log))
                raise RuntimeError("nvcc failed compiling %s" % src)
            objs.append(obj)
    link = common[:1] + (["-ccbin", "/usr/bin/g++"] if os.path.exists("/usr/bin/g++") else []) + \
        ["-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-o", target] + objs
    res = subprocess.run(link, capture_output=True, text=True)
    log.append(res.stdout + res.stderr)
    if res.returncode != 0:
        sys.stderr.write("".join(log))
        raise RuntimeError("nvcc failed linking libgvcnn_sm100.so")
    if verbose:
        sys.stderr.write("".join(log))
    return target


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, defines=defs, out=outs[0] if outs else None))
