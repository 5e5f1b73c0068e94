"""Gradients through view_pooling's group descriptors (gvcnn_view_pooling_bwd).  In the reference the dict that
view_pooling returns is made of graph tensors, so TF autodiff carries the gradient of any use of an entry back to the
view descriptors: max pooling routes dP_g to the views attaining the group max, ties sharing (1 / num_selected) * dP_g;
mean pooling gives every member dP_g / n_g; the empty groups' dummy gets nothing.  float32 gradients equal the
restatement below (view_pooling_bwd) bit for bit, 16-bit ones equal its 16-bit rounding on the widened inputs, up to
the library's one signed-zero convention for max pooling (see `matches`).  The
restatement lives in this file so oracle/ stays as it is.  The GPU tests are marked one by one; the check of the
restatement against torch autograd and the argument checks at the end need no GPU."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import gvcnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
FAST_V = (4, 6, 8, 12, 16, 20)


@pytest.fixture(scope="module")
def model():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from gvcnn_tf_b200 import model as m, _cabi
    assert _cabi.lib().gvcnn_check_device() == 0, "libgvcnn_sm100.so needs a compute-capability 10.x device"
    return m


@pytest.fixture(scope="module")
def cabi():
    from gvcnn_tf_b200 import _cabi
    spec = importlib.util.spec_from_file_location("gvcnn_build", os.path.join(ROOT, "gvcnn-tf_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    b.build()
    return _cabi


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def matches(got, want):
    """Bit for bit, with the library's one signed-zero convention for max pooling (gvcnn_pool_fuse_bwd's too): a view
    that does not attain its group's max gets +0, where TF's (0 / num_selected) * dP_g is -0 for a negative dP_g.
    `want + 0` turns -0 into +0 and leaves every other value as it is; the tests' dP holds no -0 of its own."""
    return np.array_equal(bits(got), bits(np.asarray(want, dtype=np.float32) + np.float32(0)))


def round_to(a, dtype):
    """float32 -> the nearest `dtype` value (round to nearest even), returned as float32."""
    a = np.asarray(a, dtype=np.float32)
    if dtype == torch.bfloat16:
        return O.round_bf16(a)
    if dtype == torch.float16:
        with np.errstate(over="ignore"):
            return a.astype(np.float16).astype(np.float32)
    return a


def scheme_of(bins, G):
    """One-hot int32 scheme from bins: [V] -> [G, V], [B, V] -> [B, G, V]."""
    bins = np.asarray(bins)
    V = bins.shape[-1]
    onehot = (bins[..., None, :] == np.arange(G)[:, None]).astype(np.int32)
    assert onehot.shape[-2:] == (G, V)
    return onehot


def inputs(seed, B, V, D, G, dtype=torch.float32, per_shape=True, ties=True):
    """F with many ties (non-negative halves: relu of a rounded normal, so num_selected > 1 is common), a bin map that
    leaves some groups empty, and a random dP, all already representable in `dtype`."""
    rng = np.random.default_rng(seed)
    F = rng.standard_normal((B, V, D)).astype(np.float32)
    if ties:
        F = (np.maximum(np.round(F * 2) / 2, 0) + np.float32(0)).astype(np.float32)
    bins = rng.integers(0, G, (B, V) if per_shape else (V,)).astype(np.int32)
    dP = rng.standard_normal((G, B, D)).astype(np.float32)
    return round_to(F, dtype), bins, round_to(dP, dtype)


def view_pooling_bwd(dP, F, bins, num_group, pool="max"):
    """The float32 restatement the kernels are held to: dF [B, V, D] from one gradient per group descriptor, dP
    [G, B, D].  TF autodiff of nets/model.py:62-74 alone, in TF's op order - oracle.pool_fuse_bwd with g1 = dP_g:
      reduce_max    dF_v = (indicator / num_selected) * dP_g   (_MinOrMaxGrad: ties share equally)
      reduce_mean   dF_v = dP_g / n_g                          (_MeanGrad)
      cond/gather   empty groups' dummy gets no gradient - their rows of dP are not read;
                    every view is in exactly one group, so every row of dF is written once."""
    dP = np.asarray(dP, dtype=np.float32)
    F = np.asarray(F, dtype=np.float32)
    B, V, D = F.shape
    bins = np.asarray(bins)
    if bins.ndim == 1:
        bins = np.broadcast_to(bins[None, :], (B, V))
    dF = np.zeros_like(F)
    uniq, inv = np.unique(bins, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    for u, brow in enumerate(uniq):
        sel = np.where(inv == u)[0]
        for g in range(num_group):
            ind = np.where(brow == g)[0]
            if ind.size == 0:
                continue
            g1 = dP[g][sel]
            if pool == "max":
                x = F[sel][:, ind, :]                       # [n, k, D]
                y = x.max(axis=1, keepdims=True)
                indicators = (x == y).astype(np.float32)
                num_selected = indicators.sum(axis=1, keepdims=True, dtype=np.float32)
                dF[np.ix_(sel, ind)] = (indicators / num_selected) * g1[:, None, :]
            else:
                dF[np.ix_(sel, ind)] = (g1 / np.float32(ind.size))[:, None, :]
    return dF


def as_layout(F, layout, dtype):
    """[B, V, D] array -> (view argument for view_pooling, leaves whose .grad is dF)."""
    t = torch.as_tensor(F)
    if layout == "list":
        views = [t[:, v].to("cuda", dtype).contiguous().requires_grad_() for v in range(t.shape[1])]
        return views, views
    if layout == "vbd":
        x = t.transpose(0, 1).to("cuda", dtype).contiguous().requires_grad_()
    else:
        x = t.to("cuda", dtype).contiguous().requires_grad_()
    return x, [x]


def grad_bvd(leaves, layout):
    if layout == "list":
        return torch.stack([v.grad for v in leaves], dim=1).float().cpu().numpy()
    g = leaves[0].grad.float().cpu().numpy()
    return g.transpose(1, 0, 2) if layout == "vbd" else g


def view_pooling_grad(model, F, bins, G, pool, fill, layout, dtype, dP, variant=0):
    """dF [B, V, D] (float32) from the gradients dP [G, B, D] of view_pooling's G entries, through autograd."""
    x, leaves = as_layout(F, layout, dtype)
    desc = model.view_pooling(x, torch.as_tensor(scheme_of(bins, G)).cuda(), pool=pool, empty_fill=fill,
                              layout=None if layout == "list" else layout, _variant=variant)
    entries = [desc[g] for g in range(G)]
    assert all(e.requires_grad for e in entries)
    dPt = torch.as_tensor(dP).to("cuda", dtype)
    torch.autograd.backward(entries, [dPt[g] for g in range(G)])
    return grad_bvd(leaves, layout)


# ---------------------------------------------------------------- GPU: kernels against the oracle
@gpu
@pytest.mark.parametrize("D", [2048, 1000, 37])
@pytest.mark.parametrize("V", list(FAST_V) + [5, 33])
@pytest.mark.parametrize("per_shape", [True, False], ids=["BGV", "GV"])
@pytest.mark.parametrize("layout", ["list", "bvd", "vbd"])
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("max", 0.0), ("mean", 0.0), ("mean", 1.0)])
def test_view_pooling_grad_matches_oracle_f32(model, pool, fill, layout, per_shape, V, D):
    """float32, bit for bit: the fast kernel (V in its set, 16-byte rows of >= 1024 elements), the generic vector
    kernel (D = 1000) and the scalar one (D = 37); V = 33 also runs the view-chunked forward."""
    B, G = 6, 8
    F, bins, dP = inputs(V * 1000 + D, B, V, D, G, per_shape=per_shape)
    got = view_pooling_grad(model, F, bins, G, pool, fill, layout, torch.float32, dP)
    want = view_pooling_bwd(dP, F, bins, G, pool)
    assert matches(got, want)


@gpu
@pytest.mark.parametrize("D", [1024, 2048, 36])
@pytest.mark.parametrize("V", list(FAST_V) + [5, 33])
@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "f16"])
def test_view_pooling_grad_16bit_is_rounded_oracle(model, dtype, pool, V, D):
    """bf16 / fp16: dP widened exactly, float32 arithmetic, one rounding: round_T(oracle) bit for bit.  D = 1024 is the
    one-128-thread-tile shape of the fast kernel, D = 36 is not a multiple of the vector width."""
    B, G = 5, 8
    F, bins, dP = inputs(V * 7 + D, B, V, D, G, dtype=dtype)
    for layout in ("bvd", "list"):
        got = view_pooling_grad(model, F, bins, G, pool, 1.0, layout, dtype, dP)
        want = round_to(view_pooling_bwd(dP, F, bins, G, pool), dtype)
        assert matches(got, want), layout


@gpu
@pytest.mark.parametrize("V", FAST_V)
@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("dtype,D", [(torch.float32, 2048), (torch.bfloat16, 1024), (torch.float16, 2048)],
                         ids=["f32", "bf16", "f16"])
def test_forced_generic_equals_forced_fast(model, dtype, D, pool, V):
    B, G = 7, 10
    F, bins, dP = inputs(V + D, B, V, D, G, dtype=dtype)
    generic = view_pooling_grad(model, F, bins, G, pool, 1.0, "bvd", dtype, dP, variant=1)
    fast = view_pooling_grad(model, F, bins, G, pool, 1.0, "bvd", dtype, dP, variant=3)
    assert np.array_equal(bits(generic), bits(fast))


@gpu
def test_forced_fast_is_refused_where_it_does_not_apply(model):
    from gvcnn_tf_b200 import _cabi
    F, bins, dP = inputs(1, 4, 5, 2048, 8)
    with pytest.raises(_cabi.GvcnnError) as e:
        view_pooling_grad(model, F, bins, 8, "max", 1.0, "bvd", torch.float32, dP, variant=3)
    assert e.value.code == _cabi.E_UNSUPPORTED
    F, bins, dP = inputs(2, 4, 12, 37, 8)               # rows not 16-byte aligned
    with pytest.raises(_cabi.GvcnnError) as e:
        view_pooling_grad(model, F, bins, 8, "mean", 0.0, "bvd", torch.float32, dP, variant=4)
    assert e.value.code == _cabi.E_UNSUPPORTED


# ---------------------------------------------------------------- GPU: the whole chain
def _fused_dict_grad(dS, w, G, edit_key, factor):
    """dP [G, B, D] that group_fusion on a plain dict hands back to its entries: g0 = dS / sum_w (left to right),
    g1 = g0 * w_g (then a one-member max group: (1 / 1) * g1), times `factor` for the edited entry."""
    sumw = np.float32(0)
    for x in w:
        sumw = np.float32(sumw + x)
    g0 = dS / sumw
    dP = np.stack([g0 * w[g] for g in range(G)]).astype(np.float32)
    dP[edit_key] = dP[edit_key] * np.float32(factor)
    return dP


@gpu
@pytest.mark.parametrize("V", [12, 20, 5])
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("mean", 0.0)])
def test_edited_dict_through_group_fusion(model, pool, fill, V):
    """view_pooling -> desc[3] = desc[3] * 2 -> group_fusion -> backward: F.grad equals the float32 restatement."""
    B, D, G = 6, 2048, 8
    F, _, _ = inputs(V, B, V, D, G)
    brow = np.random.default_rng(V).integers(0, G, V).astype(np.int32)
    brow[:2] = 3                                        # group 3 is not empty
    dS = np.random.default_rng(V + 1).standard_normal((B, D)).astype(np.float32)
    scheme = torch.as_tensor(scheme_of(brow, G)).cuda()
    x = torch.as_tensor(F).cuda().requires_grad_()
    desc = model.view_pooling(x, scheme, pool=pool, empty_fill=fill)
    desc[3] = desc[3] * 2
    w = model.group_weight(scheme)
    S = model.group_fusion(desc, w)
    S.backward(torch.as_tensor(dS).cuda())
    dP = _fused_dict_grad(dS, w.cpu().numpy(), G, 3, 2.0)
    assert matches(x.grad.cpu().numpy(), view_pooling_bwd(dP, F, brow, G, pool))


@gpu
@pytest.mark.parametrize("layout", ["list", "bvd", "vbd"])
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("mean", 0.0)])
def test_identity_edit_matches_the_fused_path(model, pool, fill, layout):
    """desc[0] = desc[0] turns the dict into a plain one; the op orders coincide (g0 = dS / sum_w, g1 = g0 * w_g,
    (1 / num_selected) * g1 or g1 / n_g), so F.grad is bit-identical to the unedited fused path."""
    B, V, D, G = 8, 12, 2048, 8
    F, _, _ = inputs(3, B, V, D, G)
    brow = np.array([0, 0, 1, 2, 2, 2, 4, 5, 5, 7, 7, 7], dtype=np.int32)
    dS = torch.as_tensor(np.random.default_rng(4).standard_normal((B, D)).astype(np.float32)).cuda()
    scheme = torch.as_tensor(scheme_of(brow, G)).cuda()
    grads = []
    for edit in (False, True):
        x, leaves = as_layout(F, layout, torch.float32)
        lay = None if layout == "list" else layout
        desc = model.view_pooling(x, scheme, pool=pool, empty_fill=fill, layout=lay)
        if edit:
            desc[0] = desc[0]
        S = model.group_fusion(desc, model.group_weight(scheme))
        S.reshape(B, D).backward(dS)
        grads.append(grad_bvd(leaves, layout))
    assert np.array_equal(bits(grads[0]), bits(grads[1]))


@gpu
@pytest.mark.parametrize("pool", ["max", "mean"])
def test_loss_on_one_group_only(model, pool):
    """A loss on one group: the views outside it get exactly zero; the rows of dP that belong to empty groups are not
    read (NaN there changes nothing)."""
    B, V, D, G = 6, 12, 2048, 10
    F, _, _ = inputs(5, B, V, D, G)
    brow = np.array([1, 1, 1, 4, 4, 6, 6, 6, 6, 8, 9, 9], dtype=np.int32)
    scheme = torch.as_tensor(scheme_of(brow, G)).cuda()
    x = torch.as_tensor(F).cuda().requires_grad_()
    desc = model.view_pooling(x, scheme, pool=pool)
    R = torch.as_tensor(np.random.default_rng(6).standard_normal((B, D)).astype(np.float32)).cuda()
    (desc[6] * R).sum().backward()
    dP = np.zeros((G, B, D), dtype=np.float32)
    dP[6] = R.cpu().numpy()
    got = x.grad.cpu().numpy()
    assert matches(got, view_pooling_bwd(dP, F, brow, G, pool))
    assert not np.any(got[:, brow != 6])
    assert np.any(got[:, brow == 6])
    # every entry gets a gradient, the empty groups' one is NaN
    x2 = torch.as_tensor(F).cuda().requires_grad_()
    desc2 = model.view_pooling(x2, scheme, pool=pool)
    empty = [g for g in range(G) if not np.any(brow == g)]
    dPn = dP.copy()
    dPn[empty] = np.nan
    torch.autograd.backward([desc2[g] for g in range(G)], list(torch.as_tensor(dPn).cuda()))
    assert np.array_equal(bits(x2.grad.cpu().numpy()), bits(got))


@gpu
def test_grad_mode_at_the_view_pooling_call(model):
    B, V, D, G = 4, 8, 1024, 6
    F, bins, _ = inputs(7, B, V, D, G)
    scheme = torch.as_tensor(scheme_of(bins, G)).cuda()
    x = torch.as_tensor(F).cuda().requires_grad_()
    with torch.no_grad():
        d = model.view_pooling(x, scheme)
    assert d[0].grad_fn is None and not d[0].requires_grad          # indexed with gradients enabled again
    d2 = model.view_pooling(x, scheme)
    with torch.no_grad():
        e = d2[0]                                                   # indexed under no_grad: still differentiable
    assert e.requires_grad and e.grad_fn is not None
    assert torch.equal(d[1], d2[1].detach())


@gpu
@pytest.mark.parametrize("layout", ["list", "bvd", "vbd"])
def test_empty_batch(model, layout):
    V, D, G = 8, 256, 4
    F = np.zeros((0, V, D), dtype=np.float32)
    x, leaves = as_layout(F, layout, torch.float32)
    desc = model.view_pooling(x, torch.as_tensor(scheme_of(np.arange(V) % G, G)).cuda(),
                              layout=None if layout == "list" else layout)
    sum(desc[g].sum() for g in range(G)).backward()
    assert grad_bvd(leaves, layout).shape == (0, V, D)


# ---------------------------------------------------------------- no GPU
@pytest.mark.parametrize("V", [4, 7, 12])
@pytest.mark.parametrize("pool,fill", [("max", 1.0), ("mean", 0.0)])
def test_restatement_matches_torch_autograd(pool, fill, V):
    """view_pooling_bwd against float64 torch autograd of the graph-literal restatement.  torch's amax backward
    divides by the tie count where TF multiplies by its reciprocal, so the two agree to rounding, not bit for bit."""
    from oracle import gvcnn_oracle_torch as T
    B, D, G = 5, 64, 6
    F, _, dP = inputs(V, B, V, D, G)
    brow = np.random.default_rng(V).integers(0, G, V).astype(np.int32)
    views = [torch.tensor(F[:, v], dtype=torch.float64, requires_grad=True) for v in range(V)]
    desc = T.view_pooling(views, torch.as_tensor(scheme_of(brow, G)), pool=pool, empty_fill=fill)
    outs = [desc[g] for g in range(G) if desc[g].requires_grad]
    grads = [torch.as_tensor(dP[g], dtype=torch.float64) for g in range(G) if desc[g].requires_grad]
    torch.autograd.backward(outs, grads)
    want = torch.stack([v.grad for v in views], dim=1).numpy()
    got = view_pooling_bwd(dP, F, brow, G, pool)
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=0)


def test_view_pooling_bwd_rejects_bad_arguments(cabi):
    """Null dP or dF, max without a tie mask, a misaligned dP, a bad dtype, layout or pool, and a forced fast kernel
    where it does not apply: negative codes, nothing launched."""
    L = cabi.lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.c_void_p((ctypes.cast(buf, ctypes.c_void_p).value + 15) // 16 * 16)
    odd = ctypes.c_void_p(p.value + 2)
    B, V, D, G = 4, 12, 2048, 8
    ptrs = (ctypes.c_void_p * V)(*([p.value] * V))
    null_ptrs = (ctypes.c_void_p * V)()

    def vpb(dP=p, bins=p, mask=p, dF=p, pool=cabi.POOL_MAX, layout=cabi.LAYOUT_BVD, dt=cabi.F32, V=V, D=D, B=B):
        return L.gvcnn_view_pooling_bwd(dP, bins, V, mask, dF, None, B, V, D, G, pool, layout, dt, None)

    assert vpb(dP=None) == -1 and vpb(dF=None) == -1 and vpb(bins=None) == -1
    assert vpb(layout=cabi.LAYOUT_PTRS, dF=ctypes.addressof(null_ptrs)) == -1   # a null view pointer
    assert vpb(mask=None) == -1                                  # max needs the tie mask
    assert vpb(dP=odd) == -6
    assert vpb(dt=7) == -2 and vpb(layout=5) == -3
    assert vpb(pool=3) == -8 and vpb(pool=cabi.pool_variant(cabi.POOL_MEAN, 5)) == -8
    assert vpb(V=0) == -1 and vpb(V=129) == -4 and vpb(D=0) == -1
    assert vpb(B=0) == 0                                         # an empty batch: nothing to do
    # forced V-specialised kernel: V = 5 is not instantiated, D = 37 rows are not 16-byte aligned
    assert vpb(pool=cabi.pool_variant(cabi.POOL_MAX, 3), V=5) == cabi.E_UNSUPPORTED
    assert vpb(pool=cabi.pool_variant(cabi.POOL_MEAN, 4), D=37, mask=None) == cabi.E_UNSUPPORTED
    assert vpb(pool=cabi.pool_variant(cabi.POOL_MEAN, 3), layout=cabi.LAYOUT_PTRS, dF=ctypes.addressof(ptrs),
               dP=ctypes.c_void_p(p.value + 4)) == cabi.E_UNSUPPORTED
