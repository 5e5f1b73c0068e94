"""float16 view descriptors (GVCNN_F16) on every entry point.  The contract is bfloat16's: inputs are widened exactly,
the arithmetic is float32 in the reference's op order, and one round-to-nearest-even at the output makes every float16
result equal np.float16(oracle on the float16-rounded inputs), bit for bit.  np.float16 rounds to nearest even and
overflows to inf, as the kernels' cvt.rn.f16 does.  The GPU tests are marked one by one; the binding checks at the top
need no GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import gvcnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def r16(a):
    """float32 -> nearest-even float16 (inf past 65504), returned as float32."""
    with np.errstate(over="ignore"):
        return np.asarray(a, dtype=np.float32).astype(np.float16).astype(np.float32)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t.to(dtype) if dtype is not None else t


def host(t):
    return t.detach().float().cpu().numpy()


# ---------------------------------------------------------------- binding (no GPU)
def test_header_and_binding_agree_on_f16():
    from gvcnn_tf_b200 import _cabi
    with open(os.path.join(ROOT, "include", "gvcnn_b200.h")) as f:
        m = re.search(r"#define\s+GVCNN_F16\s+(\d+)", f.read())
    assert m and int(m.group(1)) == _cabi.F16 == 2
    assert len({_cabi.F32, _cabi.BF16, _cabi.F16}) == 3


def test_dtype_code_maps_float16_and_still_refuses_others():
    from gvcnn_tf_b200 import model, _cabi
    assert model._dtype_code(torch.float16) == _cabi.F16 == 2
    assert model._dtype_code(torch.bfloat16) == _cabi.BF16
    assert model._dtype_code(torch.float32) == _cabi.F32
    for dt in (torch.float64, torch.int8, torch.float8_e4m3fn):
        with pytest.raises(TypeError):
            model._dtype_code(dt)


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def model():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from gvcnn_tf_b200 import model as m, _cabi
    assert _cabi.lib().gvcnn_check_device() == 0, "libgvcnn_sm100.so needs a compute-capability 10.x device"
    return m


def _pool_inputs(seed, B, V, D, G, ties):
    rng = np.random.default_rng(seed)
    F = rng.standard_normal((B, V, D)).astype(np.float32)
    if ties:    # small integers / halves, many exact zeros (+0 only: -0 rounds away in the + 0)
        F = (np.maximum(np.round(F * 2) / 2, 0) + np.float32(0)).astype(np.float32)
    bins = rng.integers(0, G, (B, V)).astype(np.int32)
    dS = rng.standard_normal((B, D)).astype(np.float32)
    return r16(F), bins, r16(dS)


def _variants(V, D):
    """Forced kernel selections that apply: 1 / 2 generic (bulk copy / plain loads), 3 ring (generic where it does not
    apply), 4 the few-view kernel (V = 4, 6, 8, 16-byte rows only: refused otherwise)."""
    return [0, 1, 2, 3] + ([4] if V in (4, 6, 8) and D % 8 == 0 else [])


@gpu
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("mean", 0.0), ("max", 0.0)])
@pytest.mark.parametrize("D", [1024, 2048, 1028, 72])
@pytest.mark.parametrize("V", [4, 6, 8, 12, 16, 20, 5, 33, 80])
def test_pool_fuse_bit_exact_every_variant(model, c_oracle, V, D, pool, fill):
    """S, tie planes and dF equal np.float16 of the float32 oracle, for the ring and few-view sizes, the generic
    view counts (5, 33) and the view-chunked one (80), 16-byte rows of one and two 128-column tiles, unaligned rows
    (1028) and short ones (72); every forced kernel gives the same bits."""
    from gvcnn_tf_b200.model import _Views, _pool_fuse_fwd
    G = 8 if V >= 8 else 5
    B = 3 if V == 80 else 13
    F, bins, dS = _pool_inputs(V * 100 + D, B, V, D, G, ties=(D % 2 == 0))
    want = r16(c_oracle.pool_fuse_fwd(F, bins, G, pool, fill))
    wantg = r16(c_oracle.pool_fuse_bwd(dS, F, bins, G, pool))
    for variant in _variants(V, D):
        x = dev(F, torch.float16).requires_grad_(True)
        S = model.pool_fuse(x, dev(bins), G, pool=pool, empty_fill=fill, _variant=variant)
        assert S.dtype == torch.float16
        S.backward(dev(dS, torch.float16))
        assert x.grad.dtype == torch.float16
        np.testing.assert_array_equal(bits(host(S)), bits(want), err_msg="S, variant %d" % variant)
        np.testing.assert_array_equal(bits(host(x.grad)), bits(wantg), err_msg="dF, variant %d" % variant)
    if pool == "max":
        fv = _Views(dev(F, torch.float16), "bvd", "F")
        mask = _pool_fuse_fwd(fv, dev(bins), G, "max", fill, None, True, False).mask
        np.testing.assert_array_equal(mask.cpu().numpy(), O.tie_mask_planes(F, bins, G))


# float16 value classes: smallest subnormal, subnormals, smallest normal, ordinary values, the largest finite value
F16_MAG = np.array([2.0 ** -24, 3 * 2.0 ** -24, 1e-6, 2.0 ** -14, 1e-3, 0.5, 1.0, 3.0, 1e3, 3e4, 6e4, 65504.0],
                   dtype=np.float32)


@gpu
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("mean", 0.0), ("max", 7e4), ("mean", 7e4), ("max", 0.0)])
@pytest.mark.parametrize("V,D", [(12, 2048), (6, 1024), (20, 1024), (5, 264), (40, 1024)])
def test_special_values(model, c_oracle, V, D, pool, fill):
    """Subnormals, +-0, +-65504, float32 group sums past 65504 (fine: the arithmetic is float32) and results that
    round past 65504 (a fill of 7e4 in the empty groups: S between 65504 and 7e4 becomes 65504 below 65520 and inf
    above).  Everything equals np.float16(oracle) bit for bit, except the one signed-zero case DESIGN §4 documents for
    max pooling: with empty_fill 0 and an empty group, an element where every view holds -0 comes out -0 where the
    reference's sum gives +0.  The test finds every such element and checks it is exactly that case."""
    G = V + 4                                   # empty groups in every shape
    B = 16
    rng = np.random.default_rng(V + D)
    F = rng.choice(F16_MAG, (B, V, D)) * rng.choice(np.array([-1, 1], np.float32), (B, V, D))
    F[:, :, :16] = 0.0
    F[:, ::2, :8] = -0.0
    F[:, :, 16:24] = -0.0                       # every view -0
    F[:, :, 24:32] = 65504.0                    # float32 sums past the float16 range
    F[:, 1::2, 32:40] = -65504.0
    F = r16(F)
    bins = rng.integers(0, G, (B, V)).astype(np.int32)
    bins[:, 0] = 0
    dS = r16(rng.choice(F16_MAG, (B, D)) * rng.choice(np.array([-1, 1], np.float32), (B, D)))
    with np.errstate(over="ignore", invalid="ignore"):
        want = r16(c_oracle.pool_fuse_fwd(F, bins, G, pool, fill))
        wantg = r16(c_oracle.pool_fuse_bwd(dS, F, bins, G, pool))
    assert np.isinf(want).any() or fill != 7e4  # the overflowing case is exercised
    x = dev(F, torch.float16).requires_grad_(True)
    S = model.pool_fuse(x, dev(bins), G, pool=pool, empty_fill=fill)
    S.backward(dev(dS, torch.float16))
    got, gotg = host(S), host(x.grad)
    differ = bits(got) != bits(want)
    if pool == "max" and fill == 0.0:
        all_neg_zero = np.all((F == 0) & np.signbit(F), axis=1)              # [B, D]
        has_empty = np.array([len(np.unique(r)) < G for r in bins])[:, None]
        documented = all_neg_zero & has_empty & (got == 0) & np.signbit(got) & (want == 0) & ~np.signbit(want)
        assert not np.any(differ & ~documented)
    else:
        assert not np.any(differ)
    np.testing.assert_array_equal(bits(gotg), bits(wantg))


@gpu
@pytest.mark.parametrize("pool,fill", [("max", 0.0), ("max", 1.0), ("mean", 0.0)])
@pytest.mark.parametrize("V,D", [(12, 2048), (6, 1024), (4, 2048)])
def test_signed_zeros_follow_bf16(model, V, D, pool, fill):
    """On inputs exact in both 16-bit types (+-0, small integers) float16 and bfloat16 produce zeros at the same
    elements and with the same signs, in the forward and the backward (the non-zero values differ by each type's
    output rounding)."""
    G = V + 2
    rng = np.random.default_rng(V * D)
    F = rng.choice(np.array([0.0, -0.0, -0.0, 1.0, -1.0, 2.0], np.float32), (8, V, D)).astype(np.float32)
    F[:, :, :64] = -0.0
    bins = rng.integers(0, G, (8, V)).astype(np.int32)
    dS = rng.choice(np.array([0.0, -0.0, 1.0, -3.0], np.float32), (8, D)).astype(np.float32)
    out = []
    for td in (torch.float16, torch.bfloat16):
        x = dev(F, td).requires_grad_(True)
        S = model.pool_fuse(x, dev(bins), G, pool=pool, empty_fill=fill)
        S.backward(dev(dS, td))
        out.append([(a == 0, np.signbit(a)) for a in (host(S), host(x.grad))])
    for (z16, s16), (zb, sb) in zip(out[0], out[1]):
        np.testing.assert_array_equal(z16, zb)
        np.testing.assert_array_equal(s16, sb)
    assert out[0][0][0].any() and out[0][0][1].any()


@gpu
@pytest.mark.parametrize("V,D", [(12, 2048), (16, 1024), (5, 100), (40, 1024), (6, 1024), (20, 2048)])
def test_mean_division_shortcuts_are_exact(model, V, D):
    """The float16 mirror of test_gpu_parity's test of the same name: singleton groups skip the division,
    power-of-two sizes multiply by 2^-k, the others divide by a precomputed reciprocal behind a range test.  Group
    sizes 1..V all occur; float16 subnormals, signed zeros, sums past 65504 and the largest values."""
    G, B = V, 2 * V
    rng = np.random.default_rng(V)
    F = rng.choice(F16_MAG, (B, V, D)) * rng.choice(np.array([-1, 1], np.float32), (B, V, D))
    F[:, :, :8] = 0.0
    F[:, ::2, :4] = -0.0
    F[:, :, 8:12] = -0.0
    F = r16(F)
    bins = np.zeros((B, V), dtype=np.int32)
    for i in range(B):
        n = i % V + 1
        bins[i, n:] = np.arange(1, V - n + 1)
    with np.errstate(over="ignore", invalid="ignore"):
        want = r16(O.pool_fuse_fwd(F, bins, G, "mean", 0.0))
    x = dev(F, torch.float16).requires_grad_(True)
    S = model.pool_fuse(x, dev(bins), G, pool="mean", empty_fill=0.0)
    got = host(S)
    ok = ~np.isnan(want)
    np.testing.assert_array_equal(bits(got)[ok], bits(want)[ok])
    assert np.array_equal(np.isnan(got), np.isnan(want))
    dS = r16(rng.choice(F16_MAG, (B, D)) * rng.choice(np.array([-1, 1], np.float32), (B, D)))
    S.backward(dev(dS, torch.float16))
    with np.errstate(over="ignore", invalid="ignore"):
        wantg = r16(O.pool_fuse_bwd(dS, F, bins, G, "mean"))
    gotg = host(x.grad)
    ok = ~np.isnan(wantg)
    np.testing.assert_array_equal(bits(gotg)[ok], bits(wantg)[ok])
    assert np.array_equal(np.isnan(gotg), np.isnan(wantg))


def _score_inputs(seed, B, V, Cr, bias_range):
    rng = np.random.default_rng(seed)
    R = r16(rng.standard_normal((B, V, Cr)))
    W = (rng.uniform(-1, 1, (V, Cr)) * np.sqrt(6.0 / (Cr + 1))).astype(np.float32)
    b = rng.uniform(-bias_range, bias_range, V).astype(np.float32)
    return R, W, b


@gpu
@pytest.mark.parametrize("B,V,Cr,G", [(512, 12, 1024, 8), (64, 6, 1024, 10), (32, 20, 1000, 16), (16, 80, 2048, 4),
                                       (8, 12, 37, 2)])
def test_score_bin(model, c_oracle, B, V, Cr, G):
    """Per shape: x, scores, bins and near-edge flags bit-exact against the kernel-order oracle with the 16-bit lane
    mapping (E = 8; E = 1 for rows that are not 16-byte vectors).  Per batch: the library's batch tail on those x."""
    from gvcnn_tf_b200 import _cabi as Cb
    R, W, b = _score_inputs(B + V + Cr, B, V, Cr, 0.5)
    Rd, Wd, bd = dev(R, torch.float16), dev(W), dev(b)
    sr = model.score_bin(Rd, Wd, bd, G, edge_ulps=1)
    xk = c_oracle.view_score_x_kernel_order(R, W, b, E=8 if Cr % 8 == 0 else 1)
    np.testing.assert_array_equal(sr.x.cpu().numpy(), xk)
    sk = c_oracle.score_f32(xk)
    np.testing.assert_array_equal(sr.scores.cpu().numpy(), sk)
    np.testing.assert_array_equal(sr.bins.cpu().numpy(), O.bins_from_scores(sk, G))
    np.testing.assert_array_equal(sr.near_edge().cpu().numpy(), O.edge_ulps_distance(sk, G, 1))
    # literal batch mode: column sums, mean, score and bin of exactly those x
    srb = model.score_bin(Rd, Wd, bd, G, score_reduce="batch", edge_ulps=0, clamp=True)
    L = Cb.lib()
    xsum, xm, sc = (torch.empty(V, device="cuda") for _ in range(3))
    bn, fl = (torch.empty(V, dtype=torch.int32, device="cuda") for _ in range(2))
    st = torch.zeros(4, dtype=torch.int32, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = L.gvcnn_batch_mean_bin(p(sr.x), p(xsum), p(xm), p(sc), p(bn), p(fl), p(st), B, V, G, 0, 0, 1, B, None, None,
                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, L.gvcnn_strerror(rc)
    assert torch.equal(srb.x[0], xm) and torch.equal(srb.scores[0], sc) and torch.equal(srb.bins[0], bn)


@gpu
@pytest.mark.parametrize("B,V,h,w,Cr,G", [(4, 6, 10, 10, 1024, 10), (8, 6, 8, 8, 1024, 10), (5, 12, 1, 3, 1024, 8),
                                           (2, 20, 7, 7, 2048, 16)])
def test_gap_score_bin(model, c_oracle, B, V, h, w, Cr, G):
    """gvcnn_gap_score_bin_fwd on float16 block3 maps: the pooled R equals the oracle's restatement of the kernel's
    position order, and x / scores / bins follow the E = 8 lane order on that float32 R."""
    from gvcnn_tf_b200 import _cabi as Cb
    rng = np.random.default_rng(B * 1000 + V * 10 + h)
    maps = r16(rng.standard_normal((B, V, h, w, Cr)))
    Wn = rng.uniform(-0.08, 0.08, (V, Cr)).astype(np.float32)
    bn = rng.uniform(-0.5, 0.5, V).astype(np.float32)
    HW = h * w
    R_want = O.gap_mean_kernel_order(maps.reshape(B, V, HW, Cr))
    L = Cb.lib()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    md, Wd, bd = dev(maps, torch.float16), dev(Wn), dev(bn)
    R_out = torch.empty((B, V, Cr), device="cuda")
    x, sc = torch.empty((B, V), device="cuda"), torch.empty((B, V), device="cuda")
    bi, fl = (torch.empty((B, V), dtype=torch.int32, device="cuda") for _ in range(2))
    st = torch.zeros(4, dtype=torch.int32, device="cuda")
    rc = L.gvcnn_gap_score_bin_fwd(p(md), p(Wd), p(bd), p(R_out), p(x), p(sc), p(bi), p(fl), p(st), B, V, HW, Cr, G,
                                   Cb.LAYOUT_BVD, Cb.F16, 1, 1, 0,
                                   ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, L.gvcnn_strerror(rc)
    np.testing.assert_array_equal(R_out.cpu().numpy(), R_want)
    xk = c_oracle.view_score_x_kernel_order(R_want, Wn, bn, E=8)
    np.testing.assert_array_equal(x.cpu().numpy(), xk)
    sk = c_oracle.score_f32(xk)
    np.testing.assert_array_equal(sc.cpu().numpy(), sk)
    np.testing.assert_array_equal(bi.cpu().numpy(), O.bins_from_scores(sk, G))
    sr = model.score_bin(md, Wd, bd, G, edge_ulps=1)        # the Python mirror routes the maps to the same kernel
    assert torch.equal(sr.bins, bi) and torch.equal(sr.x, x)


@gpu
@pytest.mark.parametrize("score_reduce", ["shape", "batch"])
@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("B,V,D", [(300, 12, 2048), (77, 6, 1024), (5, 20, 4096)])
def test_one_call_forward_equals_staged_path(model, B, V, D, pool, score_reduce):
    """grouping_fusion (gvcnn_grouping_fusion_fwd / _batch_fwd) on float16 R and F: the bits of the staged
    score_bin -> pool_fuse path, gradients included; S and dF come back in float16."""
    G, Cr = 8, 1024
    R, W, b = _score_inputs(B + V, B, V, Cr, 2.0)
    F, _, dS = _pool_inputs(B + D, B, V, D, G, ties=True)
    Wd, bd = dev(W), dev(b)
    out = []
    for staged in (False, True):
        x = dev(F, torch.float16).requires_grad_(True)
        if staged:
            sr = model.score_bin(dev(R, torch.float16), Wd, bd, G, score_reduce=score_reduce, clamp=True)
            S = model.pool_fuse(x, sr.bins, G, pool=pool)
        else:
            S, sr = model.grouping_fusion(dev(R, torch.float16), Wd, bd, x, G, pool=pool, score_reduce=score_reduce,
                                          clamp=True)
        S.backward(dev(dS, torch.float16))
        assert S.dtype == x.grad.dtype == torch.float16 and sr.scores.dtype == torch.float32
        out.append((sr.bins.cpu().numpy(), bits(host(S)), bits(host(x.grad))))
    for a, c in zip(out[0], out[1]):
        np.testing.assert_array_equal(a, c)
    assert len(np.unique(out[0][0])) > 2


@gpu
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("mean", 0.0)])
@pytest.mark.parametrize("N,V,h,w,Cc", [(4, 6, 10, 10, 2048), (37, 12, 3, 3, 2048), (2, 8, 5, 4, 4096),
                                        (3, 20, 3, 3, 2048)])
def test_gap_folded_pooling(model, c_oracle, N, V, h, w, Cc, pool, fill):
    """pool_fuse_gap on float16 maps, reference weights and caller weights, forward and backward, at the bf16
    tolerances of test_gpu_parity / test_paper_mode_maps; explicit 1 + n_g weights give the reference-weights bits."""
    G, HW = 8, h * w
    rng = np.random.default_rng(N + V + HW)
    F = r16(np.maximum(rng.standard_normal((N, V, h, w, Cc)), -0.3))
    bins = rng.integers(0, G, (N, V)).astype(np.int32)
    dOut = r16(rng.standard_normal((N, Cc)))
    views = [dev(F[:, v], torch.float16).requires_grad_(True) for v in range(V)]
    out = model.pool_fuse_gap(views, dev(bins), G, pool=pool, empty_fill=fill)
    assert out.dtype == torch.float16 and tuple(out.shape) == (N, Cc)
    S = c_oracle.pool_fuse_fwd(F.reshape(N, V, -1), bins, G, pool, fill).reshape(N, HW, Cc)
    want = S.astype(np.float64).mean(axis=1)
    np.testing.assert_allclose(host(out), want, rtol=1e-2, atol=1e-2 * np.abs(want).max())
    out.backward(dev(dOut, torch.float16))
    dS = np.repeat((dOut / np.float32(HW))[:, None, :], HW, axis=1).reshape(N, -1).astype(np.float32)
    wantg = c_oracle.pool_fuse_bwd(dS, F.reshape(N, V, -1), bins, G, pool).reshape(N, V, h, w, Cc)
    got = np.stack([host(v.grad) for v in views], axis=1)
    np.testing.assert_allclose(got, wantg, rtol=1e-2, atol=1e-2 * np.abs(wantg).max())
    # caller weights 1 + n_g with fill 1: the reference-weights call, bit for bit
    cw = np.stack([1.0 + np.bincount(r, minlength=G) for r in bins]).astype(np.float32)
    Ft = dev(F, torch.float16)
    x0, x1 = Ft.clone().requires_grad_(True), Ft.clone().requires_grad_(True)
    S0 = model.pool_fuse_gap(x0, dev(bins), G, pool=pool, empty_fill=1.0)
    S1 = model.pool_fuse_gap(x1, dev(bins), G, pool=pool, empty_fill=1.0, group_weight=dev(cw))
    assert torch.equal(S0, S1)
    S0.backward(dev(dOut, torch.float16))
    S1.backward(dev(dOut, torch.float16))
    assert torch.equal(x0.grad, x1.grad)


@gpu
@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("fold", [False, True])
def test_paper_mode_maps(model, pool, fold):
    """grouping_fusion_paper on float16 block3 maps and final maps, fold_gap on and off: forward, dF, dW, db and
    dmaps against float64 autograd at the bf16 tolerances of test_paper_mode_maps."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("paper_maps", os.path.join(ROOT, "tests", "test_paper_mode_maps.py"))
    pm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(pm)
    R, W, b, F = pm._paper_inputs(12, 8, 6, 1024, 2, (2, 2, 2048), pool)
    S, _, _ = pm._check_paper_grads(model, R, W, b, F, 8, pool, fold, dtype=torch.float16)
    assert S.dtype == torch.float16


def _host_pipeline(L):
    pipe = ctypes.c_void_p()
    assert L.gvcnn_host_pipeline_create(ctypes.byref(pipe), 1) == 0
    return pipe


def _run_host(L, Cb, pipe, Rh, Fh, Wd, bd, dSh, B, V, Cr, D, G, score_reduce, training, chunk):
    batch = score_reduce == Cb.SCORE_REDUCE_BATCH
    Sh = torch.empty((B, D), dtype=torch.float16).pin_memory()
    dFh = torch.empty((B, V, D), dtype=torch.float16).pin_memory()
    sc = torch.empty((V,) if batch else (B, V)).pin_memory()
    bn = torch.empty((V,) if batch else (B, V), dtype=torch.int32).pin_memory()
    st = torch.zeros(4, dtype=torch.int32)
    nbytes = L.gvcnn_host_workspace_bytes(B, chunk, V, Cr, D, Cb.F16, training, score_reduce)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = L.gvcnn_grouping_fusion_host(pipe, p(Rh), p(Fh), p(Wd), p(bd), p(Sh), p(sc), p(bn),
                                      p(dSh) if training else None, p(dFh) if training else None, p(st),
                                      B, V, Cr, D, G, Cb.POOL_MAX, ctypes.c_float(1.0), Cb.F16, score_reduce, B,
                                      None, None, chunk, p(ws), nbytes)
    assert rc == 0, L.gvcnn_strerror(rc)
    return Sh, dFh, sc, bn


@gpu
@pytest.mark.parametrize("training", [0, 1])
@pytest.mark.parametrize("score_reduce", ["shape", "batch"])
def test_host_pipeline(model, score_reduce, training):
    """gvcnn_grouping_fusion_host with float16 host buffers: the device path's bins, scores, S and dF."""
    from gvcnn_tf_b200 import _cabi as Cb
    B, V, D, G, Cr = 600, 12, 1024, 8, 1024
    R, W, b = _score_inputs(31, B, V, Cr, 2.0)
    F, _, dS = _pool_inputs(32, B, V, D, G, ties=True)
    Rh, Fh, dSh = (torch.tensor(a).to(torch.float16).pin_memory() for a in (R, F, dS))
    Wd, bd = dev(W), dev(b)
    L = Cb.lib()
    red = Cb.SCORE_REDUCE_SHAPE if score_reduce == "shape" else Cb.SCORE_REDUCE_BATCH
    pipe = _host_pipeline(L)
    try:
        Sh, dFh, sc, bn = _run_host(L, Cb, pipe, Rh, Fh, Wd, bd, dSh, B, V, Cr, D, G, red, training, 256)
    finally:
        assert L.gvcnn_host_pipeline_destroy(pipe) == 0
    sr = model.score_bin(dev(R, torch.float16), Wd, bd, G, score_reduce=score_reduce, clamp=True)
    bins = sr.bins if score_reduce == "shape" else sr.bins[0]
    np.testing.assert_array_equal(bn.numpy(), bins.cpu().numpy())
    np.testing.assert_array_equal(sc.numpy(), (sr.scores if score_reduce == "shape" else sr.scores[0]).cpu().numpy())
    x = dev(F, torch.float16).requires_grad_(True)
    S = model.pool_fuse(x, sr.bins, G, pool="max")
    assert torch.equal(Sh, S.detach().cpu())
    if training:
        S.backward(dev(dS, torch.float16))
        assert torch.equal(dFh, x.grad.cpu())


@gpu
@pytest.mark.parametrize("weight_mode", ["count", "score"])
def test_head_trains_under_autocast(model, weight_mode):
    """A GVCNNHead training step under torch.autocast(float16) with float16 backbone features: S comes back float16,
    scores and the score FC's gradients float32, and every gradient is finite."""
    torch.manual_seed(5)
    N, V, Cr, Cf, G = 8, 6, 1024, 2048, 10
    head = model.GVCNNHead(V, Cr, Cf, 5, num_group=G, weight_mode=weight_mode).cuda()
    with torch.no_grad():
        head.score_bias.uniform_(-3, 3)
    raw = torch.randn(N, V, Cr, device="cuda").half()
    final = [torch.relu(torch.randn(N, 4, 4, Cf, device="cuda")).half().requires_grad_(True) for _ in range(V)]
    with torch.autocast("cuda", dtype=torch.float16):
        scores, S, logits = head(raw, final)
        loss = torch.nn.functional.cross_entropy(logits.float(), torch.arange(N, device="cuda") % 5)
    loss.backward()
    assert S.dtype == torch.float16 and scores.dtype == torch.float32
    assert torch.isfinite(loss)
    for f in final:
        assert f.grad is not None and f.grad.dtype == torch.float16 and torch.isfinite(f.grad).all()
    for name, prm in head.named_parameters():
        if prm.grad is not None:
            assert prm.grad.dtype == torch.float32 and torch.isfinite(prm.grad).all(), name
    assert head.classifier.weight.grad is not None
    if weight_mode == "score":
        assert head.score_kernel.grad is not None and head.score_kernel.grad.abs().sum() > 0


@gpu
def test_feature_shard_round_trip(model, tmp_path):
    """float16 shards (NumPy has no bfloat16) -> FeatureShard.batches -> gvcnn_grouping_fusion_host: the device path's
    results for every batch."""
    from gvcnn_tf_b200 import records as rec, _cabi as Cb
    N, V, Cr, D, G = 300, 12, 1024, 2048, 8
    R, W, b = _score_inputs(41, N, V, Cr, 2.0)
    F, _, _ = _pool_inputs(42, N, V, D, G, ties=False)
    prefix = str(tmp_path / "shard16")
    rec.write_feature_shard(prefix, R.astype(np.float16), F.astype(np.float16), np.arange(N) % 40)
    sh = rec.FeatureShard(prefix)
    assert sh.raw.dtype == sh.final.dtype == np.float16
    Wd, bd = dev(W), dev(b)
    L = Cb.lib()
    pipe = _host_pipeline(L)
    seen = 0
    try:
        for r, f, lab in sh.batches(128):
            assert r.dtype == f.dtype == torch.float16
            B = r.shape[0]
            Sh, _, _, bn = _run_host(L, Cb, pipe, r, f, Wd, bd, None, B, V, Cr, D, G, Cb.SCORE_REDUCE_SHAPE, 0, 64)
            sr = model.score_bin(r.cuda(), Wd, bd, G, clamp=True)
            assert torch.equal(bn, sr.bins.cpu())
            assert torch.equal(Sh, model.pool_fuse(f.cuda(), sr.bins, G, pool="max").cpu())
            seen += B
    finally:
        assert L.gvcnn_host_pipeline_destroy(pipe) == 0
    assert seen == N
