"""PyTorch's NCHW view maps without a transposing copy: data_format='channels_first' on score_bin, pool_fuse_gap,
grouping_fusion(_paper) and GVCNNHead, and the GVCNN_LAYOUT_CHANNELS_FIRST bit of the C ABI.  Contiguous NCHW maps run
the channels-first kernels; maps in torch.channels_last memory run the channel-last kernels through a permuted view.
Either way the bins are those of the channel-last path on the transposed maps, bit for bit.  The GPU tests are marked
one by one; the argument checks need no GPU."""
import ctypes
import importlib.util
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


@pytest.fixture(scope="module")
def cabi():
    from gvcnn_tf_b200 import _cabi
    spec = importlib.util.spec_from_file_location("gvcnn_build", os.path.join(ROOT, "gvcnn-tf_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    b.build()
    return _cabi


@pytest.fixture(scope="module")
def model(cabi):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from gvcnn_tf_b200 import model as m
    assert cabi.lib().gvcnn_check_device() == 0, "libgvcnn_sm100.so needs a compute-capability 10.x device"
    return m


def _hw(HW):
    return {49: (7, 7), 100: (10, 10), 196: (14, 14), 289: (17, 17), 576: (24, 24), 784: (28, 28)}[HW]


def _maps(rng, B, V, C, HW, dt, relu=False):
    """float32 [B, V, C, h, w] values representable in `dt`, on the GPU in `dt` (contiguous NCHW per view)."""
    h, w = _hw(HW)
    a = rng.standard_normal((B, V, C, h, w)).astype(np.float32)
    if relu:                                    # ties: many exact zeros and few distinct values
        a = np.maximum(np.round(a * 2.0) / 2.0, 0.0).astype(np.float32)
    return torch.tensor(a, device="cuda").to(dt)


def _form(x, form, memfmt="contiguous"):
    """[B, V, C, h, w] -> the view argument ('list' of [N, C, h, w], 'bvd', 'vbd'), contiguous or in channel-last memory."""
    def mf(t):
        if memfmt == "contiguous":
            return t.contiguous()
        return t.movedim(-3, -1).contiguous().movedim(-1, -3)       # NHWC memory, NCHW shape
    if form == "list":
        return [mf(x[:, v]) for v in range(x.shape[1])]
    if form == "bvd":
        return mf(x)
    return mf(x.transpose(0, 1))


def _form_cl(x, form):
    """The channel-last twin: permute(...).contiguous() of the same maps."""
    return _form(x.movedim(2, -1), form)


def _leaves(arg):
    ts = arg if isinstance(arg, list) else [arg]
    out = [t.detach().clone(memory_format=torch.preserve_format).requires_grad_(True) for t in ts]
    return out if isinstance(arg, list) else out[0]


def _grad_bvcp(arg, form, cf):
    """Gradient of a view argument back as [B, V, C, h, w] (cf) or [B, V, h, w, C] (channel-last twin)."""
    if form == "list":
        g = torch.stack([t.grad for t in arg], dim=1)
    elif form == "bvd":
        g = arg.grad
    else:
        g = arg.grad.transpose(0, 1)
    return g if cf else g.movedim(-1, 2)


def _fmt(g):
    """'contiguous' / 'channels_last' memory of a [..., C, h, w] gradient."""
    if g.is_contiguous():
        return "contiguous"
    return "channels_last" if g.movedim(-3, -1).is_contiguous() else "other"


def _restated_gap(model, x, bins, G, pool, fill, dt):
    """The fusion-GAP order, restated: pool_fuse's S per position in float32 (float32 widening of the inputs is exact,
    and the kernels round only at the output), summed over the positions in ascending order from 0.0f in float32,
    divided once by HW, rounded once to `dt`.  x: [B, V, C, h, w]."""
    B, V, Cc, h, w = x.shape
    S = model.pool_fuse([x[:, v].float().contiguous() for v in range(V)], bins, G, pool=pool, empty_fill=fill)
    S = S.reshape(B, Cc, h * w).cpu().numpy()
    acc = np.zeros((B, Cc), dtype=np.float32)
    for p in range(h * w):
        acc = (acc + S[:, :, p]).astype(np.float32)
    return torch.tensor(acc / np.float32(h * w)).to(dt)


def _bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


# ----------------------------------------------------------------------------------------------------------------
# score side
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("HW", [49, 100, 196])
@pytest.mark.parametrize("dtn,C", [("f32", 512), ("f32", 1024), ("bf16", 1024), ("bf16", 2048), ("f16", 1024),
                                   ("f16", 2048)])
def test_gap_score_kernel_bit_exact(model, cabi, dtn, C, HW):
    """gvcnn_gap_score_bin_fwd with the channels-first bit: R_out, x, scores, bins, flags and status equal the
    channel-last kernel's on the transposed maps, bit for bit - a score of 1.0 (bin G, clamped and flagged) included."""
    _check_gap_score(model, cabi, DTYPES[dtn], C, HW, 5, 6)


@pytest.mark.gpu
@pytest.mark.parametrize("dtn,C,HW", [("f32", 1024, 289), ("f32", 512, 784), ("bf16", 1024, 576), ("f16", 2048, 784),
                                      ("bf16", 2048, 784)])
def test_gap_score_kernel_large_maps(model, cabi, dtn, C, HW):
    """Maps larger than the register-prefetched chunk (HW > 256 float32, > 512 16-bit: a 17x17 to 28x28 layer3) go
    through the position-blocked kernel: still bit for bit the channel-last kernel's results, through the C ABI and
    through score_bin."""
    dt = DTYPES[dtn]
    _check_gap_score(model, cabi, dt, C, HW, 2, 4)
    rng = np.random.default_rng(HW)
    x = _maps(rng, 2, 4, C, HW, dt)
    W = torch.tensor(rng.uniform(-0.05, 0.05, (4, C)).astype(np.float32), device="cuda")
    bias = torch.tensor(rng.uniform(-1, 1, 4).astype(np.float32), device="cuda")
    a = model.score_bin(_form(x, "bvd"), W, bias, 10, check=False, data_format="channels_first")
    b = model.score_bin(_form_cl(x, "bvd"), W, bias, 10, check=False)
    for u, v in ((a.x, b.x), (a.scores, b.scores), (a.bins, b.bins), (a.flags, b.flags)):
        assert _bits_equal(u, v)


def _check_gap_score(model, cabi, dt, C, HW, B, V):
    rng = np.random.default_rng(HW + C)
    G = 10
    x = _maps(rng, B, V, C, HW, dt)
    W = torch.tensor(rng.uniform(-0.05, 0.05, (V, C)).astype(np.float32), device="cuda")
    bias = torch.tensor(rng.uniform(-2, 2, V).astype(np.float32), device="cuda")
    bias[0] = 1e30                                     # score 1.0 -> bin G: clamped, flagged
    L = cabi.lib()
    outs = {}
    for lay in ("cf", "cl"):
        maps = x.contiguous() if lay == "cf" else x.movedim(2, -1).contiguous()
        R_out = torch.empty((B, V, C), dtype=torch.float32, device="cuda")
        buf = torch.zeros((4, B, V), dtype=torch.int32, device="cuda")
        status = torch.zeros(4, dtype=torch.int32, device="cuda")
        code = cabi.LAYOUT_BVD | (cabi.LAYOUT_CHANNELS_FIRST if lay == "cf" else 0)
        cabi.check(L.gvcnn_gap_score_bin_fwd(maps.data_ptr(), W.data_ptr(), bias.data_ptr(), R_out.data_ptr(),
                                             buf[0].data_ptr(), buf[1].data_ptr(), buf[2].data_ptr(), buf[3].data_ptr(),
                                             status.data_ptr(), B, V, HW, C, G, code, model._dtype_code(dt), 1, 64, 1,
                                             None), "gvcnn_gap_score_bin_fwd")
        outs[lay] = (R_out, buf, status)
    torch.cuda.synchronize()
    for a, b in zip(outs["cf"], outs["cl"]):
        assert _bits_equal(a, b)
    assert int(outs["cf"][2][cabi.STATUS_BIN_RANGE]) >= B          # the clamped view of every shape


@pytest.mark.gpu
@pytest.mark.parametrize("memfmt", ["contiguous", "channels_last"])
@pytest.mark.parametrize("form", ["list", "bvd", "vbd"])
@pytest.mark.parametrize("dtn", list(DTYPES))
def test_score_bin_matches_channel_last(model, dtn, form, memfmt):
    """score_bin(data_format='channels_first') on NCHW maps == score_bin on the permuted channel-last copies, in both
    score_reduce modes: x, scores, bins and flags bit for bit."""
    dt = DTYPES[dtn]
    rng = np.random.default_rng(7)
    B, V, C, G = 4, 8, 1024, 10
    HW = {"list": 49, "bvd": 100, "vbd": 196}[form]
    x = _maps(rng, B, V, C, HW, dt)
    W = torch.tensor(rng.uniform(-0.05, 0.05, (V, C)).astype(np.float32), device="cuda")
    bias = torch.tensor(rng.uniform(-1, 1, V).astype(np.float32), device="cuda")
    for mode in ("shape", "batch"):
        lay = None if form == "list" else form
        a = model.score_bin(_form(x, form, memfmt), W, bias, G, score_reduce=mode, check=False, layout=lay,
                            data_format="channels_first")
        b = model.score_bin(_form_cl(x, form), W, bias, G, score_reduce=mode, check=False, layout=lay)
        for u, v in ((a.x, b.x), (a.scores, b.scores), (a.bins, b.bins), (a.flags, b.flags)):
            assert _bits_equal(u, v), mode


# ----------------------------------------------------------------------------------------------------------------
# fusion GAP
# ----------------------------------------------------------------------------------------------------------------
_FUSE_CASES = [(V, dtn, ("max", "mean")[i % 2], (1.0, 0.0)[(i // 2) % 2], (2, 10, 16)[i % 3], (49, 100, 196)[(i + 1) % 3])
               for i, (V, dtn) in enumerate((V, d) for V in (4, 6, 8, 12, 16, 20) for d in DTYPES)]


@pytest.mark.gpu
@pytest.mark.parametrize("V,dtn,pool,fill,G,HW", _FUSE_CASES)
def test_pool_fuse_gap_forward(model, V, dtn, pool, fill, G, HW):
    """S_gap of contiguous NCHW maps is the restatement bit for bit, and within float32 re-association of the
    channel-last kernel on the transposed maps."""
    dt = DTYPES[dtn]
    rng = np.random.default_rng(V * 100 + HW)
    B, C = 6, 1024 if dt == torch.float32 else 2048
    x = _maps(rng, B, V, C, HW, dt)
    bins = torch.tensor(rng.integers(0, G, (B, V)).astype(np.int32), device="cuda")
    got = model.pool_fuse_gap(_form(x, "list"), bins, G, pool=pool, empty_fill=fill, data_format="channels_first")
    want = _restated_gap(model, x, bins, G, pool, fill, dt)
    assert got.dtype == dt and _bits_equal(got.cpu(), want)
    cl = model.pool_fuse_gap(_form_cl(x, "list"), bins, G, pool=pool, empty_fill=fill)
    tol = 1e-5 if dt == torch.float32 else 1e-2
    torch.testing.assert_close(got.float(), cl.float(), rtol=tol, atol=tol)


@pytest.mark.gpu
@pytest.mark.parametrize("dtn,C", [("f32", 256), ("bf16", 256), ("f16", 512)])
def test_pool_fuse_gap_channels_the_channel_last_kernel_rejects(model, cabi, dtn, C):
    """C = 256 / 512 (ResNet-18/34's last stage) is outside the channel-last GAP kernel (C a multiple of 1024 / 2048)
    but inside the channels-first one: the kernel itself runs, and S_gap is the restatement bit for bit."""
    dt = DTYPES[dtn]
    rng = np.random.default_rng(C)
    B, V, HW, G = 4, 6, 49, 10
    x = _maps(rng, B, V, C, HW, dt)
    bins = torch.tensor(rng.integers(0, G, (B, V)).astype(np.int32), device="cuda")
    maps = x.contiguous()
    out = torch.empty((B, C), dtype=dt, device="cuda")
    cabi.check(cabi.lib().gvcnn_pool_fuse_gap_fwd(maps.data_ptr(), bins.data_ptr(), V, out.data_ptr(), None, None,
                                                  None, 0, B, V, HW, C, G, cabi.POOL_MAX, ctypes.c_float(1.0),
                                                  cabi.LAYOUT_BVD | cabi.LAYOUT_CHANNELS_FIRST, model._dtype_code(dt),
                                                  None), "gvcnn_pool_fuse_gap_fwd")     # no fallback: must be supported
    assert _bits_equal(out.cpu(), _restated_gap(model, x, bins, G, "max", 1.0, dt))
    got = model.pool_fuse_gap(_form(x, "bvd"), bins, G, layout="bvd", data_format="channels_first")
    assert _bits_equal(got, out)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["list", "bvd", "vbd"])
@pytest.mark.parametrize("dtn", ["bf16", "f32"])
def test_pool_fuse_gap_ties_and_forms(model, dtn, form):
    """Tie-heavy relu maps (max pooling writes and reads the tie planes) in every view form: forward bit-exact to the
    restatement, dF bit-exact to the channel-last backward, transposed (C as the channel-last GAP kernel needs it: its
    fallback's torch mean would round dS to 16 bits)."""
    dt = DTYPES[dtn]
    rng = np.random.default_rng(3)
    B, V, HW, G = 4, 12, 100, 10
    C = 1024 if dt == torch.float32 else 2048
    x = _maps(rng, B, V, C, HW, dt, relu=True)
    bins = torch.tensor(rng.integers(0, G, (B, V)).astype(np.int32), device="cuda")
    a = _leaves(_form(x, form))
    b = _leaves(_form_cl(x, form))
    lay = None if form == "list" else form
    ga = model.pool_fuse_gap(a, bins, G, layout=lay, data_format="channels_first")
    gb = model.pool_fuse_gap(b, bins, G, layout=lay)
    assert _bits_equal(ga.cpu(), _restated_gap(model, x, bins, G, "max", 1.0, dt))
    dOut = torch.tensor(rng.standard_normal((B, C)).astype(np.float32), device="cuda").to(dt)
    ga.backward(dOut)
    gb.backward(dOut)
    assert _bits_equal(_grad_bvcp(a, form, True), _grad_bvcp(b, form, False))


@pytest.mark.gpu
def test_pool_fuse_gap_unsupported_falls_back(model):
    """Shapes the channels-first kernel does not cover (V = 5; caller-supplied group weights) take pool_fuse plus the
    mean over the spatial axes: the same values within float32 tolerance."""
    rng = np.random.default_rng(11)
    B, C, HW, G = 3, 256, 49, 4
    for V, weights in ((5, None), (6, torch.rand(G, device="cuda") + 0.5)):
        x = _maps(rng, B, V, C, HW, torch.float32)
        bins = torch.tensor(rng.integers(0, G, (B, V)).astype(np.int32), device="cuda")
        got = model.pool_fuse_gap(_form(x, "list"), bins, G, group_weight=weights, data_format="channels_first")
        S = model.pool_fuse(_form(x, "list"), bins, G, group_weight=weights)
        torch.testing.assert_close(got, S.mean(dim=(-2, -1)), rtol=1e-5, atol=1e-6)


# ----------------------------------------------------------------------------------------------------------------
# backward
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("memfmt", ["contiguous", "channels_last"])
@pytest.mark.parametrize("dtn", list(DTYPES))
@pytest.mark.parametrize("pool", ["max", "mean"])
def test_backward_bit_exact(model, pool, dtn, memfmt):
    """dF of the fusion GAP and dmaps, dW, db of the score side equal the channel-last path's, transposed, bit for bit;
    the gradients come back in the input's memory format."""
    dt = DTYPES[dtn]
    rng = np.random.default_rng(5)
    B, V, Cr, C, HW, G = 4, 6, 1024, 1024 if dt == torch.float32 else 2048, 49, 10
    R = _maps(rng, B, V, Cr, HW, dt)
    F = _maps(rng, B, V, C, HW, dt)
    W0 = torch.tensor(rng.uniform(-0.05, 0.05, (V, Cr)).astype(np.float32), device="cuda")
    b0 = torch.tensor(rng.uniform(-1, 1, V).astype(np.float32), device="cuda")
    dS = torch.tensor(rng.standard_normal((B, C)).astype(np.float32), device="cuda").to(dt)
    ds = torch.tensor(rng.standard_normal((B, V)).astype(np.float32), device="cuda")
    res = {}
    for cf in (True, False):
        r = _leaves(_form(R, "list", memfmt) if cf else _form_cl(R, "list"))
        f = _leaves(_form(F, "list", memfmt) if cf else _form_cl(F, "list"))
        W, bias = W0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
        df = "channels_first" if cf else "channels_last"
        sr = model.score_bin(r, W, bias, G, check=False, data_format=df)
        out = model.pool_fuse_gap(f, sr.bins, G, pool=pool, data_format=df)
        torch.autograd.backward([out, sr.scores], [dS, ds])
        res[cf] = (_grad_bvcp(r, "list", cf), _grad_bvcp(f, "list", cf), W.grad, bias.grad, r, f)
    for a, b in zip(res[True][:4], res[False][:4]):
        assert _bits_equal(a, b)
    for t in res[True][4] + res[True][5]:
        assert _fmt(t.grad) == memfmt


# ----------------------------------------------------------------------------------------------------------------
# head
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fold", [False, True])
@pytest.mark.parametrize("mode", ["count", "score"])
@pytest.mark.parametrize("memfmt", ["contiguous", "channels_last"])
def test_head_matches_channel_last(model, mode, fold, memfmt):
    """GVCNNHead(data_format='channels_first') on NCHW maps == the channel-last head with the same parameters on the
    permuted copies: the scores bit for bit, logits and every gradient within float32 tolerance (the spatial means
    after the fusion may add in another order)."""
    torch.manual_seed(0)
    rng = np.random.default_rng(9)
    B, V, Cr, C, HW, K = 4, 6, 1024, 1024, 49, 5
    R = _maps(rng, B, V, Cr, HW, torch.float32)
    F = _maps(rng, B, V, C, HW, torch.float32)
    h_cl = model.GVCNNHead(V, Cr, C, K, score_reduce="shape", weight_mode=mode).cuda()
    h_cf = model.GVCNNHead(V, Cr, C, K, score_reduce="shape", weight_mode=mode, data_format="channels_first").cuda()
    h_cf.load_state_dict(h_cl.state_dict())
    out = {}
    for cf, head in ((True, h_cf), (False, h_cl)):
        r = _leaves(_form(R, "bvd", memfmt) if cf else _form_cl(R, "bvd"))
        f = _leaves(_form(F, "bvd", memfmt) if cf else _form_cl(F, "bvd"))
        scores, _, logits = head(r, f, fold_gap=fold)
        (logits.square().sum() + (scores.sum() if mode == "count" else 0.0)).backward()
        out[cf] = (scores.detach(), logits.detach(), head.score_kernel.grad, head.score_bias.grad,
                   head.classifier.weight.grad, head.classifier.bias.grad,
                   _grad_bvcp(r, "bvd", cf), _grad_bvcp(f, "bvd", cf))
    assert _bits_equal(out[True][0], out[False][0])
    for a, b in zip(out[True][1:], out[False][1:]):
        torch.testing.assert_close(a, b, rtol=1e-3, atol=1e-5)


# ----------------------------------------------------------------------------------------------------------------
# no copies
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_channels_last_memory_is_not_copied(model):
    """Maps in torch.channels_last memory are handed to the library as they are: the pointer table holds the input's
    own storage, and neither the scores nor the fusion GAP allocate a map-sized buffer."""
    rng = np.random.default_rng(1)
    B, V, C, HW, G = 8, 12, 1024, 100, 10
    x = _maps(rng, B, V, C, HW, torch.float32)
    views = [t.contiguous(memory_format=torch.channels_last) for t in _form(x, "list")]
    W = torch.tensor(rng.uniform(-0.05, 0.05, (V, C)).astype(np.float32), device="cuda")
    bias = torch.zeros(V, device="cuda")
    rv, HW_ = model._raw_views(views, None, C, "channels_first")
    assert HW_ == HW and not rv.cf and [t.data_ptr() for t in rv.keep] == [t.data_ptr() for t in views]
    map_bytes = V * views[0].numel() * 4                 # what a permute(...).contiguous() of the maps would allocate
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    sr = model.score_bin(views, W, bias, G, check=False, data_format="channels_first")
    out = model.pool_fuse_gap(views, sr.bins, G, data_format="channels_first")
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < map_bytes
    assert out.shape == (B, C)


# ----------------------------------------------------------------------------------------------------------------
# no GPU needed
# ----------------------------------------------------------------------------------------------------------------
def test_header_constant_matches_python(cabi):
    with open(os.path.join(ROOT, "include", "gvcnn_b200.h")) as f:
        m = re.search(r"#define\s+GVCNN_LAYOUT_CHANNELS_FIRST\s+(0x[0-9a-fA-F]+|\d+)", f.read())
    assert m and int(m.group(1), 0) == cabi.LAYOUT_CHANNELS_FIRST == 0x10
    for base in (cabi.LAYOUT_BVD, cabi.LAYOUT_VBD, cabi.LAYOUT_PTRS):
        assert base & cabi.LAYOUT_CHANNELS_FIRST == 0


def test_bit_is_rejected_before_any_launch(cabi):
    """Entry points without channel semantics answer GVCNN_E_BAD_LAYOUT for the bit, the weighted GAP-folded ones and
    the GAP weight gradient GVCNN_E_UNSUPPORTED - argument checks only, nothing is launched (no device here)."""
    L = cabi.lib()
    buf = (ctypes.c_uint8 * 4096)()
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf)) % 256      # host memory: never dereferenced by the checks
    cfb = cabi.LAYOUT_BVD | cabi.LAYOUT_CHANNELS_FIRST
    E_BAD_LAYOUT = -3
    assert L.gvcnn_pool_fuse_fwd(p, p, 2, None, 0, p, None, None, None, 2, 2, 64, 2, 0, ctypes.c_float(1.0), cfb, 0,
                                 None) == E_BAD_LAYOUT
    assert L.gvcnn_pool_fuse_bwd(p, p, 2, None, 0, p, p, None, 2, 2, 64, 2, 0, cfb, 0, None) == E_BAD_LAYOUT
    assert L.gvcnn_view_score_fwd(p, p, p, p, None, 2, 2, 64, cfb, 0, None) == E_BAD_LAYOUT
    assert L.gvcnn_view_pooling_bwd(p, p, 2, p, p, None, 2, 2, 64, 2, 0, cfb, 0, None) == E_BAD_LAYOUT
    assert L.gvcnn_pool_fuse_gap_weighted_fwd(p, p, 2, p, 2, p, None, None, p, 4096, 2, 4, 16, 64, 2, 0,
                                              ctypes.c_float(0.0), cfb, 0, None) == cabi.E_UNSUPPORTED
    assert L.gvcnn_pool_fuse_gap_weighted_bwd(p, p, 2, p, 2, p, p, None, 2, 4, 16, 64, 2, 0, cfb, 0,
                                              None) == cabi.E_UNSUPPORTED
    assert L.gvcnn_pool_fuse_gap_bwd_weights(p, p, p, p, 2, p, 2, p, p, 4096, 2, 4, 16, 64, 2, 0, cfb, 0,
                                             None) == cabi.E_UNSUPPORTED
    # the bit on top of an unknown base layout is still a bad layout
    assert L.gvcnn_gap_score_bwd(p, p, p, 2, 2, 16, 64, 7 | cabi.LAYOUT_CHANNELS_FIRST, 0, None) == E_BAD_LAYOUT


def test_data_format_validation():
    from gvcnn_tf_b200 import model as m
    with pytest.raises(ValueError, match="data_format"):
        m.GVCNNHead(4, 16, 16, 3, data_format="NCHW")
    with pytest.raises(ValueError, match="data_format"):
        m.pool_fuse_gap([torch.zeros(2, 8, 3, 3)] * 4, torch.zeros(2, 4, dtype=torch.int32), 2, data_format="nchw")
    with pytest.raises(ValueError, match="C_raw = 16"):
        m._raw_views([torch.zeros(2, 8, 3, 3)] * 4, None, 16, "channels_first")
    with pytest.raises(ValueError, match="C_raw = 16"):
        m._raw_views(torch.zeros(2, 4, 8, 3, 3), "bvd", 16, "channels_first")


def test_restatement_against_float64():
    """The channels-first fusion-GAP order (positions added in order from 0.0f in float32, one division) against the
    float64 mean: within the a-priori bound of a sequential float32 sum, (HW - 1) u sum|S| / HW + u |mean|."""
    rng = np.random.default_rng(0)
    for HW in (49, 100, 196):
        S = (rng.standard_normal((16, 64, HW)) * rng.uniform(0.1, 10, (16, 64, 1))).astype(np.float32)
        acc = np.zeros((16, 64), dtype=np.float32)
        for p in range(HW):
            acc = (acc + S[:, :, p]).astype(np.float32)
        got = (acc / np.float32(HW)).astype(np.float64)
        exact = S.astype(np.float64).mean(axis=2)
        u = 2.0 ** -24
        bound = (HW - 1) * u * np.abs(S.astype(np.float64)).sum(axis=2) / HW + u * np.abs(exact) * 2
        assert np.all(np.abs(got - exact) <= bound)
