"""Restatement of the view-score backward (TF 1.x autodiff of nets/model.py:144-147), float32 one op at a time, for
tests/test_score_grad.py.  TEST INFRASTRUCTURE ONLY.

  1. SigmoidGrad   t = g * s * (1 - s)      association 'scalar': (g * s) * (1 - s), Eigen's scalar functor (what
                                            the library computes); 'packet': g * (s * (1 - s)), its packet path
  2. _LogGrad      u = t * r, r = 1 / |x|   the reciprocal rounded on its own
  3. _AbsGrad      dx = u * sign(x)
  4. _MeanGrad     'batch': dx[b, v] = dx_mean[v] / float(N)
  5. Dense(1)      dR = dx * W (one product, then rounded to R's dtype); dW, db: sums over the batch in
                   gvcnn_view_score_bwd's order (32 slices, ascending) - dW in C (score_grad_oracle.c), as NumPy has
                   no fused multiply-add without double rounding
  6. GAP           dmaps = (dx * W) / HW, rounded once to the maps' dtype
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

f32 = np.float32
NS = 32                                                         # GVCNN_SCORE_BWD_SLICES
_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def view_scores_bwd(g, x, s, score_reduce="shape", global_count=None, batch=None, association="scalar"):
    """dx from the score gradient g.  'shape': g, x, s [B, V] -> dx [B, V].  'batch': g, x (= the batch mean),
    s [V] -> (dx_mean [V], dx [batch, V]) with dx = dx_mean / float(global_count)."""
    g, x, s = (np.asarray(a, dtype=f32) for a in (g, x, s))
    with np.errstate(all="ignore"):
        one_minus = f32(1) - s
        if association == "scalar":
            t = (g * s) * one_minus
        elif association == "packet":
            t = g * (s * one_minus)
        else:
            raise ValueError(association)
        r = f32(1) / np.abs(x)
        u = t * r
        sign = np.where(x > 0, f32(1), np.where(x < 0, f32(-1), f32(0))).astype(f32)
        d = (u * sign).astype(f32)
        if score_reduce == "shape":
            return d
        dx = np.broadcast_to(d.reshape(1, -1) / f32(global_count), (batch, d.size)).astype(f32)
    return d.reshape(-1), dx


def round_to(a, dtype):
    """float32 -> the descriptors' dtype ('f32', 'bf16', 'f16'), nearest even, returned as float32."""
    a = np.ascontiguousarray(a, dtype=f32)
    if dtype == "f32":
        return a
    if dtype == "f16":
        return a.astype(np.float16).astype(f32)
    u = a.view(np.uint32).astype(np.uint64)
    r = (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16).astype(np.uint32).view(f32)
    return np.where(np.isnan(a), a, r)


def dense_dR(dx, W, dtype):
    """dR[b, v, c] = dx[b, v] * W[v, c] in float32, rounded to `dtype`."""
    with np.errstate(all="ignore"):
        return round_to(np.asarray(dx, f32)[:, :, None] * np.asarray(W, f32)[None], dtype)


def gap_dmaps(dx, W, HW, dtype):
    """dmaps[b, v, p, c] = (dx[b, v] * W[v, c]) / HW, rounded to `dtype`: [B, V, HW, C]."""
    with np.errstate(all="ignore"):
        d = (np.asarray(dx, f32)[:, :, None] * np.asarray(W, f32)[None]) / f32(HW)
    d = round_to(d, dtype)
    return np.broadcast_to(d[:, :, None, :], d.shape[:2] + (HW,) + d.shape[2:])


def _slices(B):
    return [(B * sl // NS, B * (sl + 1) // NS) for sl in range(NS)]


def dbias(dx):
    """db[v] = sum over the 32 batch slices (ascending) of the slice's ascending sum of dx[b, v]."""
    dx = np.asarray(dx, f32)
    tot = np.zeros(dx.shape[1], f32)
    for b0, b1 in _slices(dx.shape[0]):
        acc = np.zeros(dx.shape[1], f32)
        for b in range(b0, b1):
            acc = acc + dx[b]
        tot = tot + acc
    return tot


def _c_lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="gvcnn_score_grad_oracle_"), "libscore_grad_oracle.so")
        subprocess.check_call(["cc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", out,
                               os.path.join(_HERE, "score_grad_oracle.c"), "-lm"])
        _lib = ctypes.CDLL(out)
    return _lib


def dW(R, dx):
    """dW[v, c] of gvcnn_view_score_bwd: R float32 [B, V, C] (16-bit R widened exactly), dx [B, V]."""
    R = np.ascontiguousarray(R, dtype=f32)
    dx = np.ascontiguousarray(dx, dtype=f32)
    B, V, C = R.shape
    out = np.empty((V, C), f32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)             # noqa: E731
    _c_lib().score_grad_dw(p(R), p(dx), ctypes.c_int64(B), V, C, p(out))
    return out
