"""Host-side mirror of the reference's ``nets/model.py`` for the grouping + fusion path.

Same function names, positional arguments and error behaviour as the reference
(``group_scheme``, ``group_weight``, ``view_pooling``, ``group_fusion``,
``gvcnn`` head), operating on torch CUDA tensors and calling the sm_100a
kernels of ``libgvcnn_sm100.so`` through ctypes (``_cabi.py``).  torch is used
for device memory, streams and autograd plumbing only; all arithmetic of the
path runs in the library.  There is no CPU path and no fallback: a non-CUDA
tensor or a missing library raises.

Reference map (all in /root/reference):
  group_scheme   nets/model.py:16-25   (caller: train.py:277, eval.py:191)
  group_weight   nets/model.py:28-41   (caller: train.py:278, eval.py:192)
  view_pooling   nets/model.py:44-74   (caller: nets/model.py:154)
  group_fusion   nets/model.py:77-102  (caller: nets/model.py:157)
  view scores    nets/model.py:144-148
  gvcnn head     nets/model.py:143-166
"""
from __future__ import annotations

import collections
import ctypes
import math
from typing import Optional, Sequence

import torch

from . import _cabi as C

__all__ = [
    "group_scheme", "group_weight", "view_pooling", "group_fusion", "view_scores",
    "score_bin", "pool_fuse", "grouping_fusion", "GroupDescriptors", "ScoreResult",
    "GVCNNHead", "gvcnn_head", "basic_pool", "raise_for_status", "grouping_fusion_paper", "pool_fuse_gap",
    "make_exchange", "check_deferred",
]

_POOL = {"max": C.POOL_MAX, "mean": C.POOL_MEAN}
_SCORE_REDUCE = {"shape": C.SCORE_REDUCE_SHAPE, "batch": C.SCORE_REDUCE_BATCH}


def _pool_code(pool: str, variant: int = 0) -> int:
    """`pool` argument of the C ABI; `variant` (tests / A-B runs only) rides in bits 8..11 (GVCNN_POOL_VARIANT)."""
    return C.pool_variant(_POOL[pool], variant)


class _DevArray:
    """A raw device pointer as something torch.as_tensor understands (CUDA array interface), so a C callback
    that receives `float *xsum_dev` can hand it to torch.distributed without a copy."""

    def __init__(self, ptr, n, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def make_exchange(process_group):
    """gvcnn_exchange_fn for a torch.distributed process group: all-reduces (sum) the V per-view partial sums in
    place, ordered on the stream the library is working on (SURVEY.md 8e collective (2)).  Returns
    (ctypes callback, keep-alive) - keep the second value referenced while the callback can still be called."""
    import torch.distributed as dist

    def _exchange(_user, xsum_ptr, n, stream_ptr):
        try:
            t = torch.as_tensor(_DevArray(xsum_ptr, n), device=torch.device("cuda", torch.cuda.current_device()))
            ext = torch.cuda.ExternalStream(stream_ptr) if stream_ptr else torch.cuda.default_stream()
            with torch.cuda.stream(ext):
                dist.all_reduce(t, group=process_group)
            return 0
        except Exception:                                           # noqa: BLE001 - nothing may unwind through C
            import traceback
            traceback.print_exc()
            return 1                                                # cudaErrorInvalidValue: surfaces as GvcnnError
    cb = C.EXCHANGE_FN(_exchange)
    return cb, (_exchange, cb)


# --------------------------------------------------------------------------
# plumbing
# --------------------------------------------------------------------------
# The helpers below sit on every call into the library; they are written for low overhead (the reference-shaped
# five-call sequence is bound by Python time, not GPU time: bench.py `api`).
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    """cudaStream_t of torch's current stream on the current device, as the integer ctypes passes for a void*."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device()) or None
    return torch.cuda.current_stream().cuda_stream or None


def _ptr(t: Optional[torch.Tensor]):
    """Device pointer as a plain int (ctypes converts it for a c_void_p parameter); None stays a null pointer."""
    return None if t is None else (t.data_ptr() or None)


class _NullCtx:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NULL_CTX = _NullCtx()


def _on(dev):
    """`with _on(dev):` - switch the current CUDA device only if it is not already `dev` (torch.cuda.device costs two
    driver calls even when it has nothing to do)."""
    idx = dev.index
    if idx is None or idx == torch.cuda.current_device():
        return _NULL_CTX
    return torch.cuda.device(dev)


def _dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return C.F32
    if dt == torch.bfloat16:
        return C.BF16
    raise TypeError("gvcnn_b200 supports float32 and bfloat16 descriptors, got %s" % dt)


def _require_cuda(t: torch.Tensor, name: str):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if not t.is_cuda:
        raise RuntimeError("%s must live on a CUDA device: gvcnn_b200 has no CPU path" % name)


class _Views:
    """A per-view tensor (R, F or dF) in any accepted layout, reduced to what the
    C ABI wants: (pointer argument, layout code, B, V, D)."""

    def __init__(self, x, layout: Optional[str], name: str):
        self.keep = []
        if isinstance(x, (list, tuple)):                      # the reference's Python list of views
            if len(x) == 0:
                raise ValueError("%s: empty view list" % name)
            first = x[0]
            _require_cuda(first, name)
            shape, dt, dv = first.shape, first.dtype, first.device
            views, ptrs = [], []
            for t in x:                                       # one pass: checks, contiguity, pointer table
                if t is not first:
                    _require_cuda(t, name)
                    if t.shape != shape or t.dtype != dt or t.device != dv:
                        raise ValueError("%s: all views must share shape, dtype and device" % name)
                if not t.is_contiguous():
                    t = t.contiguous()
                views.append(t)
                ptrs.append(t.data_ptr())
            self.keep = views
            self.V = len(views)
            self.B = shape[0] if len(shape) > 0 else 1
            self.D = int(math.prod(shape[1:])) if len(shape) > 0 else 1
            self.view_shape = tuple(shape)
            self.dtype, self.device = dt, dv
            self.layout = C.LAYOUT_PTRS
            self.table = (ctypes.c_void_p * self.V)(*ptrs)
            self.arg = ctypes.addressof(self.table)
            self.kind = "list"
        else:
            _require_cuda(x, name)
            if x.dim() < 3:
                raise ValueError("%s: expected [B, V, ...] or [V, B, ...], got shape %s" % (name, tuple(x.shape)))
            t = x if x.is_contiguous() else x.contiguous()
            self.keep = [t]
            layout = layout or "bvd"
            if layout == "bvd":
                self.B, self.V = t.shape[0], t.shape[1]
                self.layout = C.LAYOUT_BVD
            elif layout == "vbd":
                self.V, self.B = t.shape[0], t.shape[1]
                self.layout = C.LAYOUT_VBD
            else:
                raise ValueError("layout must be 'bvd' or 'vbd'")
            self.D = int(math.prod(t.shape[2:]))
            self.view_shape = (self.B,) + tuple(t.shape[2:])
            self.dtype, self.device = t.dtype, t.device
            self.arg = t.data_ptr() or None
            self.kind = layout
            self.tensor = t
        if self.V <= 0 or self.D <= 0:          # B == 0 (an empty batch) is fine: nothing is launched
            raise ValueError("%s: no views / empty descriptors (B=%d, V=%d, D=%d)" % (name, self.B, self.V, self.D))
        if self.V > C.MAX_VIEWS:
            raise ValueError("%s: at most %d views are supported, got %d" % (name, C.MAX_VIEWS, self.V))

    @classmethod
    def of(cls, tensors, lay, name):
        """From what _view_args returns."""
        return cls(tensors if lay == "list" else tensors[0], lay, name)

    def empty_like(self):
        """Fresh storage of the same layout (for dF)."""
        out = [torch.empty_like(t) for t in self.keep] if self.kind == "list" else torch.empty_like(self.tensor)
        return out, _Views(out, self.kind, "dF")


def _view_args(x, layout):
    """A view argument - the reference's list of V tensors, or one stacked tensor in `layout` - as (tensors, lay):
    the tensors as a tuple (how they travel through autograd.Function.apply) and 'list', 'bvd' or 'vbd'."""
    if isinstance(x, (list, tuple)):
        return tuple(x), "list"
    return (x,), (layout or "bvd")


def _tie_mask(fv, pool, want):
    """Storage for max pooling's tie mask (one bit per view and element: which views the backward routes to)."""
    if not (want and pool == "max"):
        return None
    return torch.empty(((fv.V + 7) // 8, fv.B, fv.D), dtype=torch.uint8, device=fv.device)


def _bin_rows(bins, fv):
    """bins as the pooling kernels read them: int32 [1, V] or [B, V], and the row stride (0: one row for the batch)."""
    if bins.dtype != torch.int32 or not bins.is_contiguous():
        bins = bins.to(torch.int32).contiguous()
    if bins.dim() == 1:
        bins = bins[None]
    return bins, (fv.V if (bins.shape[0] == fv.B and fv.B > 1) else 0)


def _check_score_fc(W, b):
    """The V Dense(1) score layers' kernel and bias."""
    _require_cuda(W, "W"), _require_cuda(b, "b")
    if W.dtype != torch.float32 or b.dtype != torch.float32:
        raise TypeError("W and b must be float32")


def _exchange_forms(exchange):
    """A gvcnn_exchange_fn given as (fn, user) - fn a ctypes function (P2PComm.exchange, an EXCHANGE_FN callback)
    or its address as an int or c_void_p (P2PComm.exchange_c) - as (address, callable, user): the address for the
    C entry points, the callable for score_bin's staged path.  None (no exchange) gives three Nones."""
    if exchange is None:
        return None, None, None
    fn, user = exchange
    if isinstance(fn, (int, ctypes.c_void_p)):
        return fn, C.EXCHANGE_FN(fn if isinstance(fn, int) else fn.value), user
    return ctypes.cast(fn, ctypes.c_void_p), fn, user


def raise_for_status(status: torch.Tensor, num_group: int):
    """Turns the device status words into the reference's exceptions
    (nets/model.py:23): NaN score -> ValueError, bin >= num_group -> IndexError.
    Synchronises (one 16-byte device->host copy)."""
    if status is None:
        raise RuntimeError("no status words were recorded: call with check=True or pass status=")
    st = status.tolist()
    if st[C.STATUS_NAN]:
        raise ValueError("cannot convert float NaN to integer (%d NaN view scores)" % st[C.STATUS_NAN])
    if st[C.STATUS_BIN_RANGE]:
        raise IndexError("index %d is out of bounds for axis 0 with size %d (%d view scores)"
                         % (num_group, num_group, st[C.STATUS_BIN_RANGE]))
    if st[C.STATUS_BAD_SCHEME]:
        raise ValueError("group_scheme columns must be one-hot: every view in exactly one group "
                         "(%d columns are not)" % st[C.STATUS_BAD_SCHEME])


class ScoreResult:
    """x (raw FC output), scores, bins, per-view flags and the status words."""
    __slots__ = ("x", "scores", "bins", "flags", "status", "num_group")

    def __init__(self, x, scores, bins, flags, status, num_group):
        self.x, self.scores, self.bins, self.flags, self.status = x, scores, bins, flags, status
        self.num_group = num_group

    def check(self):
        raise_for_status(self.status, self.num_group)
        return self

    def near_edge(self):
        """bool tensor: views whose score is within edge_ulps of a bin edge."""
        return (self.flags & C.FLAG_NEAR_EDGE) != 0

    def order_edge(self):
        """bool tensor: views whose bin another evaluation ORDER of the same float32 dot product (e.g. the
        reference's own TensorFlow/Eigen GEMV) could legitimately put elsewhere: the a-priori rounding bound
        |dx| <= 2 gamma_n sum |r_c w_c| carried through s = |x| / (1 + |x|) straddles a bin edge.  A superset of
        near_edge(); this, not the 1-ulp flag, is the set to exclude when comparing group indices with TensorFlow.
        (Not computed by the GAP-folded score kernel, whose flags cover the FC's 1-ulp edge only.)"""
        return (self.flags & (C.FLAG_ORDER_EDGE | C.FLAG_NEAR_EDGE)) != 0


# --------------------------------------------------------------------------
# score + bin                                           nets/model.py:143-148, :23
# --------------------------------------------------------------------------
def _new_status(dev):
    return torch.zeros(C.STATUS_WORDS, dtype=torch.int32, device=dev)


def _raw_views(R, layout, c_raw):
    """The raw view descriptors in either form the reference has them in: already pooled ([N, C_raw] per view,
    after GlobalAveragePooling2D, nets/model.py:144) or the block3 maps themselves ([N, h, w, C_raw] per view,
    channel-last) - told apart by the trailing shape against the Dense(1) kernel's C_raw.  Returns (_Views, HW)."""
    rv = _Views(R, layout, "R")
    HW = 1
    if c_raw > 0 and rv.D != c_raw:
        last = rv.view_shape[-1]
        if last != c_raw or rv.D % c_raw:
            raise ValueError("raw view descriptors: trailing dimension %d does not match the score kernel's C_raw = %d"
                             % (last, c_raw))
        HW = rv.D // c_raw
    return rv, HW


def score_bin(R, W, b, num_group, *, score_reduce="shape", layout=None, edge_ulps=4, clamp=False,
              check=True, process_group=None, multiplier=None, status=None, exchange=None,
              global_count=None) -> ScoreResult:
    """Per-view discrimination score and bin.

    R: raw view descriptors after GAP (nets/model.py:144), [B, V, C] ('bvd'),
       [V, B, C] ('vbd') or a list of V [B, C] tensors; float32 or bfloat16.
       Or the raw MAPS before the GAP ([B, V, h, w, C] / [V, B, h, w, C] / list of V [N, h, w, C], channel-last -
       end_points['resnet_v2_50/block3']): the GlobalAveragePooling2D of nets/model.py:144 then runs inside the
       score kernel (gvcnn_gap_score_bin_fwd) and the pooled [B, V, C] tensor is never written.
    W [V, C], b [V]: the V separate Dense(1) layers (nets/model.py:145), float32.
    score_reduce 'shape': one score per (shape, view), bins [B, V] - the
       reference at batch size 1 per shape.  'batch': the literal
       tf.reduce_mean over the batch (nets/model.py:146), bins [1, V]; with a
       torch.distributed ``process_group`` the per-view sums are all-reduced
       first so every rank bins the same global-batch mean (SURVEY.md 8e).
    multiplier: None = num_group; 10 = the reference's hard-coded ``score * 10`` (nets/model.py:23;
       'batch' mode only - the fused per-shape kernel multiplies by num_group).
    edge_ulps: half-width, in float32 ulps of the score, of the band around every bin edge inside which a view is
       flagged NEAR_EDGE (and by which the a-priori ORDER_EDGE band is widened).  Default 4: the reference composes
       float32 log and sigmoid kernels where this library does one IEEE division, and the two can differ by a few ulps.
    status: optional persistent int32[4] device tensor the counters are ADDED to (check it every N steps
       with raise_for_status instead of synchronising every step); with check=False and no status given
       nothing is recorded.
    """
    _check_score_fc(W, b)
    Wc, bc = W.contiguous(), b.contiguous()
    rv, HW = _raw_views(R, layout, int(Wc.shape[-1]) if Wc.dim() == 2 else -1)
    Craw = rv.D // HW
    if tuple(Wc.shape) != (rv.V, Craw) or tuple(bc.shape) != (rv.V,):
        raise ValueError("W must be [V, C] = %s and b [V], got %s and %s"
                         % ((rv.V, Craw), tuple(Wc.shape), tuple(bc.shape)))
    dev = rv.device
    L = C.lib()
    if status is None and check:
        status = _new_status(dev)
    dt = _dtype_code(rv.dtype)
    with _on(dev):
        if score_reduce == "shape":
            if multiplier not in (None, num_group):
                raise ValueError("multiplier is only selectable with score_reduce='batch' or through group_scheme")
            buf = torch.empty((4, rv.B, rv.V), dtype=torch.int32, device=dev)      # x, scores, bins, flags: one allocation
            x, scores, bins, flags = buf[0].view(torch.float32), buf[1].view(torch.float32), buf[2], buf[3]
            if HW > 1:      # raw maps: GlobalAveragePooling2D folded into the score kernel (nets/model.py:144-145)
                C.check(L.gvcnn_gap_score_bin_fwd(rv.arg, _ptr(Wc), _ptr(bc), None, _ptr(x), _ptr(scores), _ptr(bins),
                                                  _ptr(flags), _ptr(status), rv.B, rv.V, HW, Craw, num_group, rv.layout,
                                                  dt, 1, edge_ulps, int(clamp), _stream()), "gvcnn_gap_score_bin_fwd")
            else:
                C.check(L.gvcnn_score_bin_fwd(rv.arg, _ptr(Wc), _ptr(bc), _ptr(x), _ptr(scores), _ptr(bins),
                                              _ptr(flags), _ptr(status), rv.B, rv.V, rv.D, num_group,
                                              rv.layout, dt, edge_ulps, int(clamp), _stream()),
                        "gvcnn_score_bin_fwd")
        elif score_reduce == "batch":
            # x and (pooled-descriptor input only) A = sum |R W| + |b| per (shape, view); column sums of both in one
            # [2, V] buffer, so ONE exchange carries them across the ranks; A feeds the a-priori order-sensitivity flag
            want_bound = HW == 1 and edge_ulps > 0                   # view_scores() asks for scores only
            xb = torch.empty((2 if want_bound else 1, max(rv.B, 1), rv.V), dtype=torch.float32, device=dev)
            if HW > 1:
                C.check(L.gvcnn_gap_score_bin_fwd(rv.arg, _ptr(Wc), _ptr(bc), None, _ptr(xb[0]), None, None, None, None,
                                                  rv.B, rv.V, HW, Craw, 1, rv.layout, dt, 0, 0, 0, _stream()),
                        "gvcnn_gap_score_bin_fwd")
            else:
                C.check(L.gvcnn_view_score_fwd(rv.arg, _ptr(Wc), _ptr(bc), _ptr(xb[0]), _ptr(xb[1]) if want_bound else None,
                                               rv.B, rv.V, rv.D, rv.layout, dt, _stream()), "gvcnn_view_score_fwd")
            sums = torch.empty((2, rv.V), dtype=torch.float32, device=dev)
            buf = torch.empty((4, 1, rv.V), dtype=torch.int32, device=dev)
            x, scores = buf[0].view(torch.float32), buf[1].view(torch.float32)
            bins, flags = buf[2], buf[3]
            ex_ptr, ex_fn, ex_user = _exchange_forms(exchange)
            if not want_bound and process_group is None:
                # no order-sensitivity report asked for: column sums + [exchange] + mean / score / bin in ONE call
                denom = rv.B if global_count is None else int(global_count)
                if denom <= 0:
                    raise ValueError("score_reduce='batch' over an empty (global) batch")
                C.check(L.gvcnn_batch_mean_bin(_ptr(xb[0]), _ptr(sums[0]), _ptr(x), _ptr(scores), _ptr(bins), _ptr(flags),
                                               _ptr(status), rv.B, rv.V, num_group, int(multiplier or 0), edge_ulps,
                                               int(clamp), denom, ex_ptr, ex_user, _stream()), "gvcnn_batch_mean_bin")
                res = ScoreResult(x, scores, bins, flags, status, num_group)
                if check:
                    res.check()
                return res
            nsum = 2 if want_bound else 1                            # rows of `sums` in use: sum x (and sum A)
            if rv.B > 0:
                for j in range(nsum):
                    C.check(L.gvcnn_batch_sum_x(_ptr(xb[j]), _ptr(sums[j]), rv.B, rv.V, _stream()), "gvcnn_batch_sum_x")
            else:
                sums.zero_()
            denom = rv.B if global_count is None else int(global_count)
            if exchange is not None:                                 # a gvcnn_exchange_fn (e.g. parallel.P2PComm)
                C.check(ex_fn(ex_user, _ptr(sums), nsum * rv.V, _stream()), "exchange")
            elif process_group is not None:
                import torch.distributed as dist
                dist.all_reduce(sums[:nsum], group=process_group)
                if global_count is None:
                    cnt = torch.tensor([rv.B], dtype=torch.int64, device=dev)
                    dist.all_reduce(cnt, group=process_group)
                    denom = int(cnt.item())
            if denom <= 0:
                raise ValueError("score_reduce='batch' over an empty (global) batch")
            C.check(L.gvcnn_score_bin(_ptr(sums[0]), ctypes.c_float(float(denom)), _ptr(x), _ptr(scores), _ptr(bins),
                                      _ptr(flags), _ptr(status), rv.V, num_group, int(multiplier or 0), edge_ulps,
                                      int(clamp), _ptr(sums[1]) if want_bound else None, Craw + 2 + denom, _stream()),
                    "gvcnn_score_bin")
        else:
            raise ValueError("score_reduce must be 'shape' or 'batch'")
    res = ScoreResult(x, scores, bins, flags, status, num_group)
    if check:
        res.check()
    return res


def view_scores(raw_view_descriptors, W, b, score_reduce="batch", layout=None, process_group=None):
    """view_discrimination_scores as nets/model.py:144-148 produces them:
    sigmoid(log|mean_n(Dense(1)(raw))|) - [1, V] for the literal 'batch' mode,
    [B, V] for 'shape'."""
    return score_bin(raw_view_descriptors, W, b, 1, score_reduce=score_reduce, layout=layout,
                     edge_ulps=0, clamp=True, check=False, process_group=process_group).scores


# --------------------------------------------------------------------------
# group_scheme / group_weight                           nets/model.py:16-41
# --------------------------------------------------------------------------
# Provenance tags: group_scheme() remembers the bin map its one-hot scheme was made from, group_weight() remembers
# the scheme its weights were counted from.  While the tagged tensors are unmodified (torch's in-place version
# counter), view_pooling / group_weight skip the scheme -> bins conversion and its validation, and group_fusion knows
# the weights ARE 1 + n_g and runs the kernel instantiation that computes them in registers.  Anything else (host
# arrays, edited tensors, hand-made weights) takes the general path - same results, a few more launches.
def _tag(t: torch.Tensor, **kw):
    t._gvcnn_tag = dict(kw, version=t._version)
    return t


def _tag_of(t):
    tag = getattr(t, "_gvcnn_tag", None) if isinstance(t, torch.Tensor) else None
    return tag if (tag is not None and tag["version"] == t._version) else None


class _DeferredStatus:
    """check='deferred': the reference's IndexError / ValueError without a device synchronisation in the middle of
    the step.  The status counters accumulate in one persistent device tensor per device; after every call its 16
    bytes are copied to pinned host memory asynchronously, and the NEXT call (or ``check_deferred()``) raises if the
    last completed copy shows a count - CUDA's own error model: reported at a later call, never lost."""
    _per_device = {}

    def __init__(self, dev):
        self.status = _new_status(dev)
        self.host = torch.zeros(C.STATUS_WORDS, dtype=torch.int32).pin_memory()
        self.event = None
        self.num_group = 0

    @classmethod
    def get(cls, dev):
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        if key not in cls._per_device:
            cls._per_device[key] = cls(dev)
        return cls._per_device[key]

    def poll(self, wait=False):
        if self.event is None:
            return
        if wait:
            self.event.synchronize()
        elif not self.event.query():
            return
        self.event = None
        if int(self.host.sum()) != 0:
            st = self.host.clone()
            self.host.zero_()
            self.status.zero_()
            raise_for_status(st, self.num_group)

    def submit(self, num_group):
        self.num_group = num_group
        self.host.copy_(self.status, non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()


def check_deferred(device=None):
    """Waits for the outstanding deferred status copy (check='deferred') and raises what it reports."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    _DeferredStatus.get(dev).poll(wait=True)


def _bins_from_scores(scores2d: torch.Tensor, num_group: int, clamp=False, check=True, multiplier=None):
    L = C.lib()
    dev = scores2d.device
    deferred = None
    if check == "deferred":
        deferred = _DeferredStatus.get(dev)
        deferred.poll()
        status = deferred.status
    else:
        status = _new_status(dev) if check else None
    bins = torch.empty(scores2d.shape, dtype=torch.int32, device=dev)
    with _on(dev):
        C.check(L.gvcnn_bins_from_scores(_ptr(scores2d), _ptr(bins), None, _ptr(status), scores2d.numel(),
                                         num_group, int(multiplier or 0), 0, int(clamp or deferred is not None),
                                         _stream()), "gvcnn_bins_from_scores")
        if deferred is not None:
            deferred.submit(num_group)
    if check is True:
        raise_for_status(status, num_group)
    return bins


def group_scheme(view_discrimination_score, num_group, num_views, multiplier=None, check=True):
    """One-hot grouping scheme.  Mirrors nets/model.py:16-25.

    view_discrimination_score: what the reference passes - a sequence holding
    ONE sequence of V scores (train.py:270-277, hence the ``[0]``), or a CUDA
    tensor [1, V]; a CUDA tensor [B, V] with B > 1 gives per-shape schemes
    [B, num_group, V].  Returns an int32 CUDA tensor [num_group, num_views].
    Raises IndexError when a score maps to bin >= num_group (score == 1.0) and
    ValueError on NaN, like the reference (one 16-byte device->host read, i.e. a synchronisation in the middle of
    the step - the reference's own host hop; check=False skips it, check='deferred' keeps the exceptions but
    raises them at the NEXT call / ``check_deferred()`` from an asynchronous copy, out-of-range bins clamped meanwhile).
    multiplier: the reference hard-codes ``score * 10`` (model.py:23) and only ever runs num_group == 10;
    None generalises that to ``* num_group`` (identical at 10), ``multiplier=10`` is the literal code for any
    num_group (bins >= num_group then raise IndexError exactly like the reference's out-of-bounds write).
    """
    s = view_discrimination_score
    if isinstance(s, torch.Tensor):
        _require_cuda(s, "view_discrimination_score")
        s2 = s.to(torch.float32).reshape(-1, s.shape[-1]).contiguous()
    else:
        row = s[0]
        if isinstance(row, torch.Tensor):
            _require_cuda(row, "view_discrimination_score")
            s2 = row.to(torch.float32).reshape(1, -1).contiguous()
        else:
            items = [t for t in row]
            if len(items) and isinstance(items[0], torch.Tensor):
                s2 = torch.stack([t.reshape(()) for t in items]).to(torch.float32).reshape(1, -1)
                _require_cuda(s2, "view_discrimination_score")
            else:
                if not torch.cuda.is_available():
                    raise RuntimeError("gvcnn_b200 needs a CUDA device: there is no CPU path")
                s2 = torch.tensor([float(t) for t in items], dtype=torch.float32, device="cuda").reshape(1, -1)
    if s2.shape[1] != num_views:
        raise ValueError("expected %d view scores, got %d" % (num_views, s2.shape[1]))
    bins = _bins_from_scores(s2, num_group, check=check, multiplier=multiplier)
    rows = bins.shape[0]
    scheme = torch.empty((rows, num_group, num_views), dtype=torch.int32, device=bins.device)
    with _on(bins.device):
        C.check(C.lib().gvcnn_bins_to_scheme(_ptr(bins), _ptr(scheme), rows, num_views, num_group, _stream()),
                "gvcnn_bins_to_scheme")
    out = scheme[0] if rows == 1 else scheme
    return _tag(out, kind="scheme", bins=bins, G=num_group, checked=bool(check))  # one-hot by construction


def _small_to_device(x, device, dtype, name):
    """The scheme [G, V] and the weights [G] are small HOST arrays in the reference (NumPy, fed through
    placeholders: train.py:277-288).  Accept them as such and move them next to the descriptors; this is
    an argument transfer of a few hundred bytes, not a CPU compute path."""
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=dtype) if (not x.is_cuda or x.dtype != dtype) else x
    try:
        return torch.as_tensor(x).to(device=device, dtype=dtype)
    except Exception as e:                                          # noqa: BLE001
        raise TypeError("%s must be a tensor or array-like, got %s" % (name, type(x).__name__)) from e


def _scheme_to_bins(g_schemes: torch.Tensor, check=True):
    _require_cuda(g_schemes, "group_scheme")
    tag = _tag_of(g_schemes)
    if tag is not None and tag.get("kind") == "scheme" and (tag["checked"] or not check):
        return tag["bins"], tag["G"]                                 # made by group_scheme and untouched since
    sc = g_schemes.to(torch.int32)
    if sc.dim() == 2:
        sc = sc[None]
    sc = sc.contiguous()
    rows, G, V = sc.shape
    status = _new_status(sc.device) if check else None
    bins = torch.empty((rows, V), dtype=torch.int32, device=sc.device)
    with _on(sc.device):
        C.check(C.lib().gvcnn_scheme_to_bins(_ptr(sc), _ptr(bins), _ptr(status), rows, V, G, _stream()),
                "gvcnn_scheme_to_bins")
    if check:
        raise_for_status(status, G)
    return bins, G


def group_weight(g_schemes):
    """weights[g] = 1 + number of views in group g.  Mirrors nets/model.py:28-41.
    g_schemes: int tensor [G, V] (or [B, G, V]), CUDA or - as in the reference - a host array, which is
    moved to the current CUDA device; returns a float32 CUDA tensor [G] (or [B, G])."""
    if not (isinstance(g_schemes, torch.Tensor) and g_schemes.is_cuda):
        if not torch.cuda.is_available():
            raise RuntimeError("gvcnn_b200 needs a CUDA device: there is no CPU path")
        g_schemes = _small_to_device(g_schemes, torch.device("cuda", torch.cuda.current_device()), torch.int32,
                                     "g_schemes")
    bins, G = _scheme_to_bins(g_schemes)
    rows, V = bins.shape
    w = torch.empty((rows, G), dtype=torch.float32, device=bins.device)
    with _on(bins.device):
        C.check(C.lib().gvcnn_group_weight(_ptr(bins), _ptr(w), rows, V, G, _stream()), "gvcnn_group_weight")
    out = w[0] if g_schemes.dim() == 2 else w
    return _tag(out, kind="weight", bins=bins)


# --------------------------------------------------------------------------
# pooling + fusion                                      nets/model.py:44-102
# --------------------------------------------------------------------------
# What a forward launch ending in pooling + fusion returns: S [B, D], the tie mask, the G pooled groups [G, B, D] (if
# asked for), the status words, and the bins and group weights as the kernel read them, with their row strides (None, 0:
# the kernel computes 1 + n_g) - everything the pooling backward needs.
_Pooled = collections.namedtuple("_Pooled", "S mask P status bins bin_stride weights w_stride")


def _pool_fuse_fwd(fv: _Views, bins: torch.Tensor, G: int, pool: str, empty_fill: float,
                   weights: Optional[torch.Tensor], want_mask: bool, want_groups: bool, want_status: bool = True,
                   variant: int = 0) -> _Pooled:
    dev = fv.device
    dt = _dtype_code(fv.dtype)
    bins, bin_stride = _bin_rows(bins, fv)
    if bins.shape[-1] != fv.V or bins.shape[0] not in (1, fv.B):
        raise ValueError("bins must be [V], [1, V] or [B, V] with V=%d, B=%d; got %s"
                         % (fv.V, fv.B, tuple(bins.shape)))
    w_stride = 0
    if weights is not None:
        _require_cuda(weights, "group_weight")
        weights = weights.to(torch.float32).contiguous()
        if weights.dim() == 1:
            weights = weights[None]
        if weights.shape[-1] != G or weights.shape[0] not in (1, fv.B):
            raise ValueError("group_weight must be [G] or [B, G]")
        w_stride = G if (weights.shape[0] == fv.B and fv.B > 1) else 0
    S = torch.empty((fv.B, fv.D), dtype=fv.dtype, device=dev)
    mask = _tie_mask(fv, pool, want_mask)
    P = torch.empty((G, fv.B, fv.D), dtype=fv.dtype, device=dev) if want_groups else None
    status = _new_status(dev) if want_status else None
    with _on(dev):
        C.check(C.lib().gvcnn_pool_fuse_fwd(fv.arg, _ptr(bins), bin_stride, _ptr(weights), w_stride, _ptr(S), _ptr(P),
                                            _ptr(mask), _ptr(status), fv.B, fv.V, fv.D, G, _pool_code(pool, variant),
                                            ctypes.c_float(empty_fill), fv.layout, dt, _stream()),
                "gvcnn_pool_fuse_fwd")
    return _Pooled(S, mask, P, status, bins, bin_stride, weights, w_stride)


def _pool_fuse_bwd(dS: torch.Tensor, fv_like: _Views, bins, bin_stride, weights, w_stride, mask, G, pool, variant=0):
    dS = dS.contiguous()
    out, gv = fv_like.empty_like()
    with _on(dS.device):
        C.check(C.lib().gvcnn_pool_fuse_bwd(_ptr(dS), _ptr(bins), bin_stride, _ptr(weights), w_stride,
                                            _ptr(mask), gv.arg, None, gv.B, gv.V, gv.D, G,
                                            _pool_code(pool, variant), gv.layout, _dtype_code(gv.dtype), _stream()),
                "gvcnn_pool_fuse_bwd")
    return out


class _PoolFuseFn(torch.autograd.Function):
    """S from `launch(fv, want_mask)` -> (_Pooled, extra outputs): pooling + fusion, on its own or after score + bin
    in the same call into the library; backward = TF autodiff of nets/model.py:62-100 (dF only: no gradient reaches
    scores / weights, train.py:127-128, utils/train_utils.py:203-206).  The extra outputs are non-differentiable."""

    @staticmethod
    def forward(ctx, launch, G, pool, variant, f_lay, *f_t):
        fv = _Views.of(f_t, f_lay, "F")
        out, extras = launch(fv, True)
        ctx.fv, ctx.G, ctx.pool, ctx.variant = fv, G, pool, variant
        ctx.bin_stride, ctx.w_stride = out.bin_stride, out.w_stride
        ctx.save_for_backward(out.bins, out.weights, out.mask)
        ctx.mark_non_differentiable(*[t for t in extras if t is not None])
        return (out.S.reshape(fv.view_shape),) + extras

    @staticmethod
    def backward(ctx, dS, *_unused):
        bins, weights, mask = ctx.saved_tensors
        fv = ctx.fv
        # bins may hold the raw out-of-range value (clamp=False); the backward kernel clamps like the forward did
        out = _pool_fuse_bwd(dS.reshape(fv.B, fv.D), fv, bins, ctx.bin_stride, weights, ctx.w_stride, mask,
                             ctx.G, ctx.pool, ctx.variant)
        return (None,) * 5 + (tuple(out) if isinstance(out, list) else (out,))


def _run_launch(launch, f_t, f_lay, G, pool, variant):
    """(S in the shape of one view,) + the launch's extra outputs.  Through autograd only when a gradient can be asked for;
    otherwise straight into the library (saves the autograd.Function bookkeeping on the inference path)."""
    if torch.is_grad_enabled() and any(t.requires_grad for t in f_t):
        return _PoolFuseFn.apply(launch, G, pool, variant, f_lay, *f_t)
    fv = _Views.of(f_t, f_lay, "F")
    out, extras = launch(fv, False)
    return (out.S.reshape(fv.view_shape),) + extras


def _run_pool_fuse(f_t, f_lay, bins, weights, G, pool, empty_fill, want_status, variant=0):
    """Pooling + fusion from a bin map: (S, status)."""
    def launch(fv, want_mask):
        out = _pool_fuse_fwd(fv, bins, G, pool, empty_fill, weights, want_mask, False, want_status, variant)
        return out, (out.status,)
    return _run_launch(launch, f_t, f_lay, G, pool, variant)


def pool_fuse(final_view_descriptors, bins, num_group, pool="max", empty_fill=1.0, layout=None,
              group_weight=None, check=False, _variant=0):
    """Fused view_pooling + group_fusion (nets/model.py:44-102) from a bin map.

    final_view_descriptors: list of V tensors [N, ...] (the reference's layout),
    or one tensor [B, V, ...] (layout='bvd') / [V, B, ...] (layout='vbd').
    bins: int32 [B, V] (per-shape) or [V] / [1, V] (one scheme for the batch).
    Returns the shape descriptor with the shape of one view, differentiable
    w.r.t. the view descriptors.
    """
    views, lay = _view_args(final_view_descriptors, layout)
    _require_cuda(bins, "bins")
    S, status = _run_pool_fuse(views, lay, bins, group_weight, num_group, pool, empty_fill, check, _variant)
    if check:
        raise_for_status(status, num_group)
    return S


class _PoolFuseGapFn(torch.autograd.Function):
    """Pooling + fusion + the global average pooling that follows it (nets/model.py:154-163) without ever
    writing the fused map: [B, C] out; backward takes the [B, C] gradient."""

    @staticmethod
    def forward(ctx, bins, G, pool, empty_fill, layout, HW, Cch, *views):
        L = C.lib()
        fv = _Views.of(views, layout, "F")
        dev = fv.device
        dt = _dtype_code(fv.dtype)
        bins_c, bstride = _bin_rows(bins, fv)
        out = torch.empty((fv.B, Cch), dtype=fv.dtype, device=dev)
        mask = _tie_mask(fv, pool, any(v.requires_grad for v in views))
        status = _new_status(dev)
        ws_bytes = L.gvcnn_pool_fuse_gap_workspace_bytes(fv.B, Cch, HW, dt)
        ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
        with _on(dev):
            C.check(L.gvcnn_pool_fuse_gap_fwd(fv.arg, _ptr(bins_c), bstride, _ptr(out), _ptr(mask), _ptr(status),
                                              _ptr(ws), ws_bytes, fv.B, fv.V, HW, Cch, G, _POOL[pool],
                                              ctypes.c_float(empty_fill), fv.layout, dt, _stream()),
                    "gvcnn_pool_fuse_gap_fwd")
        ctx.fv, ctx.G, ctx.pool, ctx.HW, ctx.Cch, ctx.bstride = fv, G, pool, HW, Cch, bstride
        ctx.save_for_backward(bins_c, mask)
        ctx.mark_non_differentiable(status)
        return out, status

    @staticmethod
    def backward(ctx, dOut, _dstatus):
        bins_c, mask = ctx.saved_tensors
        fv = ctx.fv
        dOut = dOut.contiguous()
        out, gv = fv.empty_like()
        status = _new_status(dOut.device)
        with _on(dOut.device):
            C.check(C.lib().gvcnn_pool_fuse_gap_bwd(_ptr(dOut), _ptr(bins_c), ctx.bstride, _ptr(mask), gv.arg,
                                                    _ptr(status), gv.B, gv.V, ctx.HW, ctx.Cch, ctx.G, _POOL[ctx.pool],
                                                    gv.layout, _dtype_code(gv.dtype), _stream()),
                    "gvcnn_pool_fuse_gap_bwd")
        grads = tuple(out) if isinstance(out, list) else (out,)
        return (None,) * 7 + grads


def pool_fuse_gap(final_view_descriptors, bins, num_group, pool="max", empty_fill=1.0, layout=None):
    """view_pooling + group_fusion + GlobalAveragePooling2D (nets/model.py:154-163) in one pass: the
    descriptors are channel-last maps ([N, h, w, C] per view, or [B, V, h, w, C] / [V, B, h, w, C]); returns
    the pooled shape descriptor [N, C].  The fused map is never written.  Shapes the specialised kernel does
    not cover (see gvcnn_pool_fuse_gap_fwd) run pool_fuse and average afterwards - same result up to the
    float32 rounding of the mean."""
    views, lay = _view_args(final_view_descriptors, layout)
    shp = tuple(views[0].shape)
    spatial = shp[1:-1] if lay == "list" else shp[2:-1]
    if len(shp) < 3:
        raise ValueError("pool_fuse_gap expects channel-last maps, e.g. [N, h, w, C] per view")
    Cch = shp[-1]
    HW = int(math.prod(spatial)) if len(spatial) else 1
    _require_cuda(bins, "bins")
    try:
        out, _ = _PoolFuseGapFn.apply(bins, num_group, pool, empty_fill, lay, HW, Cch, *views)
        return out
    except C.GvcnnError as e:
        if e.code != C.E_UNSUPPORTED:
            raise
    S = pool_fuse(final_view_descriptors, bins, num_group, pool=pool, empty_fill=empty_fill, layout=layout)
    return S.reshape(S.shape[0], -1, Cch).mean(dim=1)


class GroupDescriptors(dict):
    """What ``view_pooling`` returns: behaves like the reference's
    ``{group index: pooled descriptor}`` dict (nets/model.py:61,72), but lazy -
    the G pooled tensors are only materialised (one kernel writing [G, B, D])
    if somebody indexes or iterates the dict.  ``group_fusion`` recognises an
    UNEDITED object of this type and runs the single-pass fused kernel on the
    original views; once an entry has been assigned or removed it is an
    ordinary dict of tensors and is fused as such."""

    def __init__(self, views, layout, bins, num_group, pool, empty_fill):
        super().__init__()
        self._views, self._layout = views, layout
        self._bins, self._G, self._pool, self._fill = bins, num_group, pool, empty_fill
        self._done = False
        self._edited = False

    def _materialise(self):
        if self._done:
            return
        fv = _Views.of(self._views, self._layout, "F")
        P = _pool_fuse_fwd(fv, self._bins, self._G, self._pool, self._fill, None, want_mask=False, want_groups=True,
                           want_status=False).P
        for g in range(self._G):
            dict.__setitem__(self, g, P[g].reshape(fv.view_shape))
        self._done = True

    def __getitem__(self, k):
        self._materialise()
        return dict.__getitem__(self, k)

    def __iter__(self):
        self._materialise()
        return dict.__iter__(self)

    def __len__(self):
        return dict.__len__(self) if self._edited else self._G

    def __contains__(self, k):
        if self._edited:
            return dict.__contains__(self, k)
        return isinstance(k, int) and 0 <= k < self._G

    def items(self):
        self._materialise()
        return dict.items(self)

    def keys(self):
        self._materialise()
        return dict.keys(self)

    def values(self):
        self._materialise()
        return dict.values(self)

    def get(self, k, default=None):
        self._materialise()
        return dict.get(self, k, default)

    # mutation: from here on this is a plain dict of tensors
    def __setitem__(self, k, v):
        self._materialise()
        self._edited = True
        dict.__setitem__(self, k, v)

    def __delitem__(self, k):
        self._materialise()
        self._edited = True
        dict.__delitem__(self, k)

    def pop(self, *a):
        self._materialise()
        self._edited = True
        return dict.pop(self, *a)

    def update(self, *a, **kw):
        self._materialise()
        self._edited = True
        dict.update(self, *a, **kw)


def view_pooling(final_view_descriptors, group_scheme, pool="max", empty_fill=1.0, layout=None):
    """Intra-group view pooling.  Mirrors nets/model.py:44-74.

    final_view_descriptors: list of V CUDA tensors [N, h, w, C] (as in the
    reference), or a stacked tensor with ``layout``.  group_scheme: int tensor
    [num_group, num_view] (one scheme for the batch, as in the reference) or
    [B, num_group, num_view].  pool='max', empty_fill=1.0 is the shipped
    model.py behaviour (:63,:72); pool='mean', empty_fill=0.0 is unit_test.py's.
    Returns a GroupDescriptors dict {g: pooled descriptor}.
    """
    views, lay = _view_args(final_view_descriptors, layout)
    if len(views) == 0:
        raise ValueError("final_view_descriptors: empty view list")
    _require_cuda(views[0], "final_view_descriptors")
    bins, G = _scheme_to_bins(_small_to_device(group_scheme, views[0].device, torch.int32, "group_scheme"))
    return GroupDescriptors(views, lay, bins, G, pool, empty_fill)


def _fuse_plain_dict(group_descriptors, group_weight):
    """nets/model.py:94-100 on an arbitrary {index: tensor} dict: numerator = sum over the dict's entries of
    group_weight[key] * value, denominator = sum of ALL group weights.  Runs the pooling kernel with every entry
    as a one-member group (max of one value = the value), so the arithmetic is the fused path's:
    acc += w_key * P_key in ascending key order (the reference's dict order for any dict view_pooling built),
    one division.  Differentiable w.r.t. the entries."""
    if len(group_descriptors) == 0:
        raise ValueError("group_fusion: empty group_descriptors")
    keys = sorted(group_descriptors.keys())
    vals = [group_descriptors[k] for k in keys]
    for v in vals:
        _require_cuda(v, "group_descriptors")
    dev = vals[0].device
    w = _small_to_device(group_weight, dev, torch.float32, "group_weight")
    if w.dim() != 1:
        raise ValueError("group_fusion on a plain dict takes one weight per group ([G])")
    G = int(w.shape[0])
    if any((not isinstance(k, int)) or k < 0 or k >= G for k in keys):
        raise IndexError("group_descriptors has a key outside range(len(group_weight)) = range(%d)" % G)
    if len(keys) > C.MAX_VIEWS:
        raise ValueError("at most %d group descriptors" % C.MAX_VIEWS)
    bins = torch.tensor(keys, dtype=torch.int32, device=dev)[None]
    S, _ = _run_pool_fuse(tuple(vals), "list", bins, w, G, "max", 0.0, False)
    return S


def group_fusion(group_descriptors, group_weight):
    """Shape descriptor = sum_g w_g * P_g / sum_g w_g.  Mirrors nets/model.py:77-102.

    With the (unedited) GroupDescriptors returned by ``view_pooling`` this runs the fused
    single-pass kernel over the original views (and is differentiable w.r.t.
    them).  ``group_weight`` is honoured as given ([G] or [B, G] float32), so
    weights other than ``model.group_weight``'s 1 + count also work.  Any other
    ``{index: tensor}`` mapping - the reference's documented argument ("dic {index: group_desc}") - is fused
    entry by entry (``_fuse_plain_dict``).
    """
    if not isinstance(group_descriptors, GroupDescriptors) or group_descriptors._edited:
        if not hasattr(group_descriptors, "keys"):
            raise TypeError("group_fusion expects a {group index: descriptor} mapping")
        return _fuse_plain_dict(group_descriptors, group_weight)
    gd = group_descriptors
    tag = _tag_of(group_weight)
    if tag is not None and tag.get("kind") == "weight" and tag["bins"] is gd._bins:
        w = None       # model.group_weight of this very scheme: the kernel computes 1 + n_g itself
    else:
        w = _small_to_device(group_weight, gd._bins.device, torch.float32, "group_weight")
    S, _ = _run_pool_fuse(gd._views, gd._layout, gd._bins, w, gd._G, gd._pool, gd._fill, False)
    return S


def basic_pool(final_view_descriptors, layout=None):
    """``tf.reduce_max(final_view_descriptors, axis=0)`` - the MVCNN-style
    verification path (nets/model.py:202, :160-161) = all views in one group,
    unit weight."""
    fv = _Views(final_view_descriptors, layout, "F")
    bins = torch.zeros((1, fv.V), dtype=torch.int32, device=fv.device)
    w = torch.ones((1, 1), dtype=torch.float32, device=fv.device)
    return pool_fuse(final_view_descriptors, bins, 1, pool="max", empty_fill=0.0, layout=layout,
                     group_weight=w)


def _grouping_fusion_fwd(rv, fv, want_mask, W, b, G, pool, empty_fill, edge_ulps, clamp, status, variant, literal):
    """Score + bin, then pool + fuse, chained on the device in one call into the library (PDL, no host hop):
    gvcnn_grouping_fusion_fwd per shape, or - `literal` = (multiplier, global_count, exchange address, user) -
    gvcnn_grouping_fusion_batch_fwd (x -> column sums -> [exchange] -> mean -> one bin row -> pool + fuse).
    Extra outputs: (x, scores, bins, flags); x is the batch-mean row in the literal mode."""
    L = C.lib()
    if (rv.B, rv.V) != (fv.B, fv.V) or rv.dtype != fv.dtype:
        raise ValueError("raw and final view descriptors must agree in batch, views and dtype")
    dev = fv.device
    Wc, bc = W.contiguous(), b.contiguous()
    if literal is None:
        buf = torch.empty((4, fv.B, fv.V), dtype=torch.int32, device=dev)      # x, scores, bins, flags: one allocation
        x, scores, bins, flags = buf[0].view(torch.float32), buf[1].view(torch.float32), buf[2], buf[3]
    else:
        xb = torch.empty((max(fv.B, 1), fv.V), dtype=torch.float32, device=dev)
        buf = torch.empty((5, 1, fv.V), dtype=torch.int32, device=dev)           # xsum, x_mean, scores, bins, flags
        xsum, x, scores = (buf[i].view(torch.float32) for i in range(3))
        bins, flags = buf[3], buf[4]
    S = torch.empty((fv.B, fv.D), dtype=fv.dtype, device=dev)
    mask = _tie_mask(fv, pool, want_mask)
    with _on(dev):
        if literal is None:
            C.check(L.gvcnn_grouping_fusion_fwd(rv.arg, _ptr(Wc), _ptr(bc), fv.arg, _ptr(x), _ptr(scores), _ptr(bins),
                                                _ptr(flags), _ptr(S), _ptr(mask), _ptr(status), fv.B, fv.V, rv.D, fv.D,
                                                G, _pool_code(pool, variant), ctypes.c_float(empty_fill), rv.layout,
                                                fv.layout, _dtype_code(fv.dtype), edge_ulps, int(clamp), _stream()),
                    "gvcnn_grouping_fusion_fwd")
        else:
            multiplier, global_count, ex_ptr, ex_user = literal
            C.check(L.gvcnn_grouping_fusion_batch_fwd(rv.arg, _ptr(Wc), _ptr(bc), fv.arg, _ptr(xb), _ptr(xsum), _ptr(x),
                                                      _ptr(scores), _ptr(bins), _ptr(flags), _ptr(S), _ptr(mask),
                                                      _ptr(status), fv.B, fv.V, rv.D, fv.D, G, int(multiplier or 0),
                                                      _pool_code(pool, variant), ctypes.c_float(empty_fill), rv.layout,
                                                      fv.layout, _dtype_code(fv.dtype), edge_ulps, int(clamp),
                                                      int(global_count), ex_ptr, ex_user, _stream()),
                    "gvcnn_grouping_fusion_batch_fwd")
    bin_stride = fv.V if (literal is None and fv.B > 1) else 0
    return _Pooled(S, mask, None, status, bins, bin_stride, None, 0), (x, scores, bins, flags)


def _is_raw_maps(raw, W, layout):
    """True when `raw` holds the un-pooled block3 maps ([..., h, w, C_raw]) rather than [..., C_raw] descriptors."""
    if not (isinstance(W, torch.Tensor) and W.dim() == 2):
        return False
    t = raw[0] if isinstance(raw, (list, tuple)) and len(raw) else raw
    if not isinstance(t, torch.Tensor):
        return False
    lead = 1 if isinstance(raw, (list, tuple)) else 2
    return t.dim() > lead + 1 and t.shape[-1] == W.shape[1]


def grouping_fusion(raw_view_descriptors, W, b, final_view_descriptors, num_group, pool="max",
                    empty_fill=1.0, score_reduce="shape", layout=None, clamp=False, check=False,
                    process_group=None, edge_ulps=4, status=None, multiplier=None, exchange=None,
                    global_count=None, _variant=0):
    """The whole hot path with no host hop (replaces the partial_run split of
    train.py:264-288), one call into the library in either mode: per shape, score + bin
    then pool + fuse, chained on the device; in the literal batch-mean mode, x -> column
    sums -> [exchange] -> mean -> one bin row -> pool + fuse.
    Returns (shape_descriptor, ScoreResult).

    exchange: a gvcnn_exchange_fn (fn, user) - P2PComm.exchange or .exchange_c - carrying the V column sums across
    the ranks; without it, a ``process_group``'s torch.distributed does (called back from inside the library, in
    stream order).

    check=True turns out-of-range / NaN scores into the reference's IndexError / ValueError right away (one
    16-byte device->host read per call, i.e. a synchronisation); the default records nothing.  For a training
    loop pass a persistent ``status`` tensor (int32[4], zeros) - the counters accumulate into it without any
    synchronisation - and call ``raise_for_status(status, num_group)`` every N steps."""
    if status is None and check:
        dev0 = W.device if isinstance(W, torch.Tensor) else None
        status = _new_status(dev0)
    if _is_raw_maps(raw_view_descriptors, W, layout):
        # block3 maps instead of pooled raw descriptors: the GAP of nets/model.py:144 runs inside the score kernel
        # (gvcnn_gap_score_bin_fwd); pooling + fusion follow on the stream, chained with programmatic dependent launch
        sr = score_bin(raw_view_descriptors, W, b, num_group, score_reduce=score_reduce, layout=layout,
                       edge_ulps=edge_ulps, clamp=clamp, check=check, process_group=process_group, status=status,
                       multiplier=multiplier, exchange=exchange, global_count=global_count)
        S = pool_fuse(final_view_descriptors, sr.bins, num_group, pool=pool, empty_fill=empty_fill, layout=layout,
                      _variant=_variant)
        return S, sr
    if score_reduce == "shape":
        if multiplier not in (None, num_group):
            raise ValueError("multiplier is only selectable with score_reduce='batch' or through group_scheme")
    elif score_reduce != "batch":
        raise ValueError("score_reduce must be 'shape' or 'batch'")
    r_t, r_lay = _view_args(raw_view_descriptors, layout)
    f_t, f_lay = _view_args(final_view_descriptors, layout)
    _check_score_fc(W, b)
    literal, keep = None, None
    if score_reduce == "batch":
        B_local = r_t[0].shape[0] if r_lay in ("list", "bvd") else r_t[0].shape[1]
        if exchange is None and process_group is not None:
            cb, keep = make_exchange(process_group)
            exchange = (cb, None)
        ex_ptr, _, ex_user = _exchange_forms(exchange)
        if global_count is None:
            global_count = B_local
            if process_group is not None:
                import torch.distributed as dist
                cnt = torch.tensor([B_local], dtype=torch.int64, device=W.device)
                dist.all_reduce(cnt, group=process_group)
                global_count = int(cnt.item())
        if global_count <= 0:
            raise ValueError("score_reduce='batch' over an empty (global) batch")
        literal = (multiplier, global_count, ex_ptr, ex_user)
    rv = _Views.of(r_t, r_lay, "R")

    def launch(fv, want_mask):
        return _grouping_fusion_fwd(rv, fv, want_mask, W, b, num_group, pool, empty_fill, edge_ulps, clamp, status,
                                    _variant, literal)
    S, x, scores, bins, flags = _run_launch(launch, f_t, f_lay, num_group, pool, _variant)
    del keep
    sr = ScoreResult(x, scores, bins, flags, status, num_group)
    if check:
        sr.check()
    return S, sr


# --------------------------------------------------------------------------
# paper mode: score-derived, differentiable group weights (SURVEY.md 8f n2)
# --------------------------------------------------------------------------
class _PaperModeFn(torch.autograd.Function):
    """S = sum_g w_g P_g / sum_g w_g with w_g = mean score of the group's views (0 for an empty group).
    Unlike the reference (weights fed through placeholders, train.py:127-128), the gradient reaches the
    V Dense(1) score layers: dL/dW, dL/db (and dL/dR if the raw descriptors require grad) besides dL/dF.
    No reference counterpart - checked against float64 autograd of the same formulas."""

    @staticmethod
    def forward(ctx, W, b, G, pool, f_layout, r_layout, n_r, status, *tensors):
        L = C.lib()
        r_t, f_t = tensors[:n_r], tensors[n_r:]
        rv = _Views.of(r_t, r_layout, "R")
        fv = _Views.of(f_t, f_layout, "F")
        # no synchronisation in the training step: out-of-range / NaN scores are clamped for pooling and counted
        # into the caller's persistent `status` tensor (checked every N steps), as in grouping_fusion
        sr = score_bin(r_t if r_layout == "list" else r_t[0], W, b, G, score_reduce="shape", layout=r_layout,
                       edge_ulps=1, clamp=True, check=False, status=status)
        dev = fv.device
        weights = torch.empty((rv.B, G), dtype=torch.float32, device=dev)
        with _on(dev):
            C.check(L.gvcnn_group_weight_from_scores(_ptr(sr.scores), _ptr(sr.bins), _ptr(weights), rv.B, rv.V, G,
                                                     _stream()), "gvcnn_group_weight_from_scores")
        out = _pool_fuse_fwd(fv, sr.bins, G, pool, 0.0, weights, want_mask=True, want_groups=False, want_status=False)
        ctx.rv, ctx.fv, ctx.G, ctx.pool = rv, fv, G, pool
        ctx.bstride, ctx.wstride = out.bin_stride, out.w_stride
        ctx.need_dr = any(t.requires_grad for t in r_t)
        ctx.n_r = n_r
        ctx.save_for_backward(W.contiguous(), sr.x, out.bins, out.weights, out.S, out.mask)
        ctx.mark_non_differentiable(sr.scores, sr.bins, weights)
        return out.S.reshape(fv.view_shape), sr.scores, sr.bins, weights

    @staticmethod
    def backward(ctx, dS, _ds, _db, _dw):
        L = C.lib()
        W, x, bins_c, w_c, S, mask = ctx.saved_tensors
        rv, fv, G, pool = ctx.rv, ctx.fv, ctx.G, ctx.pool
        dS2 = dS.reshape(fv.B, fv.D).contiguous()
        dev = dS2.device
        dF = _pool_fuse_bwd(dS2, fv, bins_c, ctx.bstride, w_c, ctx.wstride, mask, G, pool)
        ws_bytes = L.gvcnn_view_score_bwd_workspace_bytes(rv.V, rv.D)
        n_dw, n_dx, n_W = fv.B * G, fv.B * fv.V, W.numel()
        scratch = torch.empty(n_dw + n_dx + n_W + rv.V + (ws_bytes + 3) // 4, dtype=torch.float32, device=dev)  # one allocation
        dweights = scratch[:n_dw].view(fv.B, G)
        dx = scratch[n_dw:n_dw + n_dx].view(fv.B, fv.V)
        dW = scratch[n_dw + n_dx:n_dw + n_dx + n_W].view_as(W)
        dbias = scratch[n_dw + n_dx + n_W:n_dw + n_dx + n_W + rv.V]
        ws = scratch[n_dw + n_dx + n_W + rv.V:]
        dR_out, dR_views = (rv.empty_like() if ctx.need_dr else (None, None))
        with _on(dev):
            C.check(L.gvcnn_pool_fuse_bwd_weights(fv.arg, _ptr(dS2), _ptr(S), _ptr(bins_c), ctx.bstride, _ptr(w_c),
                                                  ctx.wstride, _ptr(dweights), fv.B, fv.V, fv.D, G, _POOL[pool],
                                                  fv.layout, _dtype_code(fv.dtype), _stream()),
                    "gvcnn_pool_fuse_bwd_weights")
            C.check(L.gvcnn_score_weight_bwd(_ptr(dweights), _ptr(bins_c), _ptr(x), _ptr(dx), fv.B, fv.V, G, _stream()),
                    "gvcnn_score_weight_bwd")
            C.check(L.gvcnn_view_score_bwd(rv.arg, _ptr(dx), _ptr(W), _ptr(dW), _ptr(dbias),
                                           dR_views.arg if dR_views is not None else None, _ptr(ws), ws_bytes,
                                           rv.B, rv.V, rv.D, rv.layout, _dtype_code(rv.dtype), _stream()),
                    "gvcnn_view_score_bwd")
        if dR_out is None:
            gr = (None,) * ctx.n_r
        else:
            gr = tuple(dR_out) if isinstance(dR_out, list) else (dR_out,)
        gf = tuple(dF) if isinstance(dF, list) else (dF,)
        return (dW, dbias, None, None, None, None, None, None) + gr + gf


def grouping_fusion_paper(raw_view_descriptors, W, b, final_view_descriptors, num_group, pool="max", layout=None,
                          status=None):
    """Paper-mode grouping + fusion: group weight = mean discrimination score of the group's views, empty
    groups vanish; differentiable w.r.t. the view descriptors AND the score FC (W, b, optionally the raw
    descriptors).  Returns (shape_descriptor, scores, bins, weights).  Per-shape scores/bins."""
    r_t, r_lay = _view_args(raw_view_descriptors, layout)
    f_t, f_lay = _view_args(final_view_descriptors, layout)
    _check_score_fc(W, b)
    return _PaperModeFn.apply(W, b, num_group, pool, f_lay, r_lay, len(r_t), status, *r_t, *f_t)


def _spatial_mean(S):
    """GlobalAveragePooling2D of the fused map [N, h, w, C] -> [N, C] (nets/model.py:163) for the un-folded path;
    an empty batch (a rank whose shard is exhausted) stays empty."""
    if S.dim() <= 2:
        return S
    return S.reshape(S.shape[0], int(math.prod(S.shape[1:-1])), S.shape[-1]).mean(dim=1)


class GVCNNHead(torch.nn.Module):
    """The trainable state of the path: V separate Dense(1) score layers
    (Keras defaults: glorot-uniform kernel, zero bias; nets/model.py:145 sits
    inside the view loop) and the classifier Dense(num_classes) after global
    average pooling (nets/model.py:163-164)."""

    def __init__(self, num_views, raw_channels, final_channels, num_classes, num_group=10, pool="max",
                 empty_fill=1.0, score_reduce="batch", weight_mode="count"):
        super().__init__()
        self.num_views, self.num_group = num_views, num_group
        self.pool, self.empty_fill, self.score_reduce = pool, empty_fill, score_reduce
        if weight_mode not in ("count", "score"):
            raise ValueError("weight_mode: 'count' (reference, nets/model.py:28-41) or 'score' (paper mode)")
        self.weight_mode = weight_mode
        lim = math.sqrt(6.0 / (raw_channels + 1))
        self.score_kernel = torch.nn.Parameter(torch.empty(num_views, raw_channels).uniform_(-lim, lim))
        self.score_bias = torch.nn.Parameter(torch.zeros(num_views))
        self.classifier = torch.nn.Linear(final_channels, num_classes)
        lim2 = math.sqrt(6.0 / (final_channels + num_classes))
        torch.nn.init.uniform_(self.classifier.weight, -lim2, lim2)
        torch.nn.init.zeros_(self.classifier.bias)

    def forward(self, raw_view_descriptors, final_view_descriptors, process_group=None, check=False, fold_gap=False,
                status=None, global_count=None):
        """raw: post-GAP block3 features [N, V, C_raw] (or list of V [N, C_raw]);
        final: list of V [N, h, w, C] maps or [N, V, h, w, C].  Returns
        (view_discrimination_scores, shape_descriptor, logits) like
        nets/model.py:166.  fold_gap=True (reference-literal weights only) folds the
        GlobalAveragePooling2D of nets/model.py:163 into the pooling kernel: the fused
        map is never written and the second return value is the pooled [N, C] descriptor."""
        if fold_gap and self.weight_mode == "count":
            sr = score_bin(raw_view_descriptors, self.score_kernel.detach(), self.score_bias.detach(),
                           self.num_group, score_reduce=self.score_reduce, process_group=process_group, check=check,
                           status=status, global_count=global_count)
            net = pool_fuse_gap(final_view_descriptors, sr.bins, self.num_group, pool=self.pool,
                                empty_fill=self.empty_fill)
            return sr.scores, net, self.classifier(net.to(self.classifier.weight.dtype))
        if self.weight_mode == "score":
            S, scores, _, _ = grouping_fusion_paper(raw_view_descriptors, self.score_kernel, self.score_bias,
                                                    final_view_descriptors, self.num_group, pool=self.pool,
                                                    status=status)
        else:
            S, sr = grouping_fusion(raw_view_descriptors, self.score_kernel.detach(), self.score_bias.detach(),
                                    final_view_descriptors, self.num_group, pool=self.pool,
                                    empty_fill=self.empty_fill, score_reduce=self.score_reduce,
                                    process_group=process_group, check=check, status=status,
                                    global_count=global_count)
            scores = sr.scores
        net = _spatial_mean(S)
        logits = self.classifier(net.to(self.classifier.weight.dtype))
        return scores, S, logits


def gvcnn_head(raw_view_descriptors, final_view_descriptors, head: GVCNNHead, group_scheme=None,
               group_weight=None):
    """nets/model.py:143-166 from the backbone outputs on: with ``group_scheme``
    / ``group_weight`` given (the reference's placeholders, train.py:127-128) it
    pools and fuses with them; without, it computes them on the device."""
    if group_scheme is None:
        return head(raw_view_descriptors, final_view_descriptors)
    scores = view_scores(raw_view_descriptors, head.score_kernel.detach(), head.score_bias.detach(),
                         score_reduce=head.score_reduce)
    desc = view_pooling(final_view_descriptors, group_scheme, pool=head.pool, empty_fill=head.empty_fill)
    w = group_weight if group_weight is not None else globals()["group_weight"](group_scheme)
    S = group_fusion(desc, w)
    net = _spatial_mean(S)
    return scores, S, head.classifier(net.to(head.classifier.weight.dtype))
