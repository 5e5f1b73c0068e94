"""Paper mode at the reference's real geometry: block3 maps into the trainable score FC and the global average
pooling after the fusion folded into the pooling kernels (pool_fuse_gap with caller weights,
grouping_fusion_paper(fold_gap=True), GVCNNHead(weight_mode="score", fold_gap=True)).  The GPU tests are marked
one by one; the argument checks at the end need no GPU."""
import ctypes
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import gvcnn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def _as_layout(a, layout, dtype=torch.float32, grad=False):
    """[B, V, ...] array -> the view argument in `layout` (fresh leaves)."""
    t = torch.as_tensor(np.asarray(a, dtype=np.float32))
    if layout == "bvd":
        out = [t.to("cuda", dtype).contiguous()]
    elif layout == "vbd":
        out = [t.transpose(0, 1).to("cuda", dtype).contiguous()]
    else:
        out = [t[:, v].to("cuda", dtype).contiguous() for v in range(t.shape[1])]
    for x in out:
        x.requires_grad_(grad)
    return out if layout == "list" else out[0]


def _grad_bvd(x, layout):
    if layout == "bvd":
        return x.grad
    if layout == "vbd":
        return x.grad.transpose(0, 1)
    return torch.stack([v.grad for v in x], dim=1)


def _bins(rng, B, V, G):
    return rng.integers(0, G, (B, V)).astype(np.int32)


def _count_weights(bins, G):
    return np.stack([1.0 + np.bincount(r, minlength=G) for r in bins]).astype(np.float32)


def _weighted_S64(F, bins, w, G, pool):
    """float64 sum_g w_g P_g / sum_g w_g per shape, empty groups contributing 0.  F [B, V, D]."""
    F = F.astype(np.float64)
    B, V, D = F.shape
    S = np.zeros((B, D))
    for b in range(B):
        for g in range(G):
            ind = np.where(bins[b] == g)[0]
            if ind.size:
                P = F[b, ind].max(axis=0) if pool == "max" else F[b, ind].mean(axis=0)
                S[b] += w[b, g] * P
        S[b] /= w[b].astype(np.float64).sum()
    return S


GAP_CASES = [(3, 4, 2, 2, 1024), (2, 6, 3, 1, 2048), (2, 12, 2, 3, 2048), (2, 20, 1, 2, 2048), (4, 4, 10, 10, 2048)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["bvd", "vbd", "list"])
@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,V,h,w,C", GAP_CASES)
def test_weighted_gap_pooling(model, B, V, h, w, C, dtype, pool, layout):
    if dtype == torch.bfloat16 and C % 2048:
        pytest.skip("the bf16 GAP tile is 2048 channels")
    rng = np.random.default_rng(B * 100 + V * 7 + h)
    G = 8
    F = rng.standard_normal((B, V, h, w, C)).astype(np.float32)
    if pool == "max":
        F = np.maximum(np.round(F * 2) / 2, 0)          # ties
    bins = _bins(rng, B, V, G)
    dOut = rng.standard_normal((B, C)).astype(np.float32)
    HW = h * w
    Fq = torch.as_tensor(F).to(dtype).float().numpy()   # what the kernels see
    # explicit 1 + n_g with fill 1 == the reference-weights call, bit for bit
    x0, x1 = _as_layout(F, layout, dtype, True), _as_layout(F, layout, dtype, True)
    bt = torch.as_tensor(bins, device="cuda")
    S0 = model.pool_fuse_gap(x0, bt, G, pool=pool, empty_fill=1.0, layout=None if layout == "list" else layout)
    S1 = model.pool_fuse_gap(x1, bt, G, pool=pool, empty_fill=1.0, layout=None if layout == "list" else layout,
                             group_weight=torch.as_tensor(_count_weights(bins, G), device="cuda"))
    assert torch.equal(S0, S1)
    S0.backward(torch.as_tensor(dOut, device="cuda").to(dtype))
    S1.backward(torch.as_tensor(dOut, device="cuda").to(dtype))
    assert torch.equal(_grad_bvd(x0, layout), _grad_bvd(x1, layout))
    # random weights, fill 0: against float64; one shared row, so the oracle's backward applies too
    wrow = rng.uniform(0.1, 1.0, G).astype(np.float32)
    x2 = _as_layout(F, layout, dtype, True)
    S2 = model.pool_fuse_gap(x2, bt, G, pool=pool, empty_fill=0.0, layout=None if layout == "list" else layout,
                             group_weight=torch.as_tensor(wrow, device="cuda"))
    want = _weighted_S64(Fq.reshape(B, V, HW * C), bins, np.broadcast_to(wrow, (B, G)), G, pool)
    want = want.reshape(B, HW, C).mean(axis=1)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    np.testing.assert_allclose(S2.detach().float().cpu().numpy(), want, rtol=tol, atol=tol * np.abs(want).max())
    S2.backward(torch.as_tensor(dOut, device="cuda").to(dtype))
    if dtype == torch.float32:
        dS = np.repeat((dOut / np.float32(HW))[:, None, :], HW, axis=1).reshape(B, HW * C)
        ref = O.pool_fuse_bwd(dS, F.reshape(B, V, HW * C), bins, G, pool, weights=wrow)
        np.testing.assert_array_equal(_grad_bvd(x2, layout).cpu().numpy().reshape(B, V, -1), ref)


def _paper_inputs(seed, B, V, Cr, hr, F_shape, pool, maps=True):
    rng = np.random.default_rng(seed)
    R = rng.standard_normal((B, V, hr, hr, Cr) if maps else (B, V, Cr)).astype(np.float32)
    W = rng.uniform(-1, 1, (V, Cr)).astype(np.float32) * np.float32(np.sqrt(6.0 / (Cr + 1)))
    b = rng.uniform(-1, 1, V).astype(np.float32)
    F = rng.standard_normal((B, V) + F_shape).astype(np.float32)
    if pool == "max":
        F = np.maximum(F, 0)
    return R, W, b, F


def _paper_ref64(R, W, b, F, G, pool, bins, fold):
    """float64 autograd of the paper-mode formulas with the kernel's bins (no re-binning at edges):
    R maps are pooled first (GlobalAveragePooling2D), x = R.W + b, s = |x| / (1 + |x|), w_g = mean s of the group,
    S = sum_g w_g P_g / sum_g w_g, and with `fold` the mean of S over the positions."""
    B, V = F.shape[:2]
    Rp = R.reshape(B, V, -1, R.shape[-1]).mean(dim=2) if R.dim() > 3 else R
    x = torch.einsum("bvc,vc->bv", Rp, W) + b[None, :]
    s = torch.abs(x) / (1 + torch.abs(x))
    onehot = torch.nn.functional.one_hot(bins, G).to(R.dtype)                  # [B, V, G]
    cnt = onehot.sum(dim=1)
    w = torch.where(cnt > 0, (onehot * s[:, :, None]).sum(dim=1) / cnt.clamp(min=1), torch.zeros_like(cnt))
    Fd = F.reshape(B, V, -1)
    Ps = []
    for g in range(G):
        member = onehot[:, :, g] > 0
        if pool == "max":
            Pg = torch.amax(torch.where(member[:, :, None], Fd, torch.full_like(Fd, -1e300)), dim=1)
        else:
            Pg = (Fd * member[:, :, None]).sum(dim=1) / cnt[:, g].clamp(min=1)[:, None]
        Ps.append(torch.where((cnt[:, g] > 0)[:, None], Pg, torch.zeros_like(Pg)))
    S = (w[:, :, None] * torch.stack(Ps, dim=1)).sum(dim=1) / w.sum(dim=1, keepdim=True)
    if fold:
        S = S.reshape(B, -1, F.shape[-1]).mean(dim=1)
    return S, w


def _check_paper_grads(model, R, W, b, F, G, pool, fold, dtype=torch.float32):
    B = F.shape[0]
    rng = np.random.default_rng(7)
    Rd, Wd, bd, Fd = (torch.as_tensor(a).to("cuda", dtype if a.ndim > 2 else torch.float32).requires_grad_(True)
                      for a in (R, W, b, F))
    S, scores, bins, w = model.grouping_fusion_paper(Rd, Wd, bd, Fd, G, pool=pool, fold_gap=fold)
    dS = torch.as_tensor(rng.standard_normal(tuple(S.shape)).astype(np.float32))
    S.backward(dS.cuda().to(S.dtype))
    R64, W64, b64, F64 = (torch.as_tensor(a).to(dtype if a.ndim > 2 else torch.float32).double().requires_grad_(True)
                          for a in (R, W, b, F))          # the score FC stays float32 whatever the maps' dtype
    S64, w64 = _paper_ref64(R64, W64, b64, F64, G, pool, bins.cpu().long(), fold)
    S64.backward(dS.to(dtype).double().reshape(S64.shape))
    tol = 1e-5 if dtype == torch.float32 else 2e-2
    torch.testing.assert_close(w.cpu().double(), w64.detach(), rtol=tol, atol=tol / 10)
    torch.testing.assert_close(S.detach().cpu().double().reshape(S64.shape), S64.detach(), rtol=tol, atol=tol)
    torch.testing.assert_close(Fd.grad.cpu().double(), F64.grad, rtol=tol, atol=tol / 10)
    for got, ref in ((Wd.grad, W64.grad), (bd.grad, b64.grad), (Rd.grad, R64.grad)):
        scale = float(ref.abs().max())
        assert scale > 0
        torch.testing.assert_close(got.cpu().double(), ref, rtol=1e-3, atol=2e-4 * scale * (1 if dtype == torch.float32 else 50))
    return S, bins, w


@pytest.mark.gpu
@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("fold", [False, True])
@pytest.mark.parametrize("maps", [True, False])
def test_paper_mode_maps_gradients_match_float64_autograd(model, pool, fold, maps):
    """dF, dW, db and dR (dmaps for block3 maps) against float64 autograd, fold on and off."""
    R, W, b, F = _paper_inputs(11, 16, 12, 1024, 3, (3, 3, 1024), pool, maps=maps)
    _check_paper_grads(model, R, W, b, F, 8, pool, fold)


@pytest.mark.gpu
@pytest.mark.parametrize("pool", ["max", "mean"])
def test_paper_mode_maps_bf16(model, pool):
    R, W, b, F = _paper_inputs(12, 8, 6, 1024, 2, (2, 2, 2048), pool)
    _check_paper_grads(model, R, W, b, F, 8, pool, True, dtype=torch.bfloat16)


@pytest.mark.gpu
def test_block3_maps_score_fc_gradient_regression(model):
    """Block3 maps [8, 12, 3, 3, 1024] into the unfolded paper mode: dW and db of the score FC come from the pooled
    R the score kernel writes (they used to be computed with the map size as the channel count)."""
    R, W, b, F = _paper_inputs(5, 8, 12, 1024, 3, (512,), "max")
    _check_paper_grads(model, R, W, b, F, 10, "max", False)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["bvd", "vbd", "list"])
@pytest.mark.parametrize("pool", ["max", "mean"])
def test_folded_paper_mode_matches_unfolded(model, pool, layout):
    """Same inputs: bins and weights equal; float32 dF equals the unfolded dF for dS = dOut / HW bit for bit;
    S_gap within 1e-5 of the spatial mean of the fused map."""
    B, V, h, C, G = 6, 12, 4, 2048, 10
    R, W, b, F = _paper_inputs(3, B, V, 1024, 2, (h, h, C), pool)
    dOut = np.random.default_rng(4).standard_normal((B, C)).astype(np.float32)
    lay = None if layout == "list" else layout
    Wt, bt = torch.as_tensor(W, device="cuda"), torch.as_tensor(b, device="cuda")
    x0, x1 = _as_layout(F, layout, grad=True), _as_layout(F, layout, grad=True)
    Rt = _as_layout(R, layout)
    Sg, s0, b0, w0 = model.grouping_fusion_paper(Rt, Wt, bt, x0, G, pool=pool, layout=lay, fold_gap=True)
    S, s1, b1, w1 = model.grouping_fusion_paper(Rt, Wt, bt, x1, G, pool=pool, layout=lay)
    assert torch.equal(b0, b1) and torch.equal(w0, w1) and torch.equal(s0, s1)
    assert Sg.shape == (B, C)
    torch.testing.assert_close(Sg, model._spatial_mean(S), rtol=1e-5, atol=1e-5)
    d = torch.as_tensor(dOut, device="cuda")
    Sg.backward(d)
    S.backward((d / (h * h))[:, None, None, :].expand(B, h, h, C).contiguous())
    assert torch.equal(_grad_bvd(x0, layout), _grad_bvd(x1, layout))


@pytest.mark.gpu
def test_paper_mode_fallbacks(model):
    """V = 5 (no folded kernel) and C_raw = 96 (no GAP-folded score kernel) take the fallbacks and give the
    unfolded numbers."""
    R, W, b, F = _paper_inputs(8, 4, 5, 1024, 2, (2, 2, 1024), "max")
    args = [torch.as_tensor(a, device="cuda") for a in (R, W, b, F)]
    Sg, _, bins, w = model.grouping_fusion_paper(*args, 6, fold_gap=True)
    S, _, bins1, w1 = model.grouping_fusion_paper(*args, 6)
    assert torch.equal(bins, bins1) and torch.equal(w, w1)
    assert torch.equal(Sg, model._spatial_mean(S))
    R, W, b, F = _paper_inputs(9, 4, 6, 96, 2, (2, 2, 1024), "max")
    Rt = torch.as_tensor(R, device="cuda").requires_grad_(True)
    Wt, bt, Ft = (torch.as_tensor(a, device="cuda") for a in (W, b, F))
    S, _, bins, w = model.grouping_fusion_paper(Rt, Wt, bt, Ft, 6)
    Rp = torch.as_tensor(R, device="cuda").requires_grad_(True)
    S1, _, bins1, w1 = model.grouping_fusion_paper(Rp.reshape(4, 6, -1, 96).mean(dim=2), Wt, bt, Ft, 6)
    assert torch.equal(bins, bins1) and torch.equal(w, w1) and torch.equal(S, S1)
    g = torch.randn_like(S)
    S.backward(g)
    S1.backward(g)
    assert torch.equal(Rt.grad, Rp.grad) and float(Rt.grad.abs().sum()) > 0


@pytest.mark.gpu
def test_head_score_mode_fold_gap(model):
    torch.manual_seed(0)
    B, V, Cr, C = 8, 6, 1024, 2048
    R = torch.randn(B, V, 3, 3, Cr, device="cuda")
    F = torch.relu(torch.randn(B, V, 3, 3, C, device="cuda"))
    head = model.GVCNNHead(V, Cr, C, 5, num_group=10, weight_mode="score", score_reduce="shape").cuda()
    _, S0, logits0 = head(R, F)
    _, Sg, logits = head(R, F.requires_grad_(True), fold_gap=True)
    assert Sg.shape == (B, C)
    torch.testing.assert_close(logits, logits0, rtol=1e-4, atol=1e-4)
    torch.nn.functional.cross_entropy(logits, torch.arange(B, device="cuda") % 5).backward()
    g = head.score_kernel.grad
    assert g is not None and torch.isfinite(g).all() and float(g.abs().sum()) > 0


@pytest.mark.gpu
def test_train_head_score_mode_fold_gap_learns(model, tmp_path):
    spec = importlib.util.spec_from_file_location("train_head", os.path.join(ROOT, "gvcnn-tf_b200", "train_head.py"))
    th = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(th)
    h = th.main(["--num_views", "6", "--raw_channels", "64", "--final_channels", "1024", "--feature_hw", "4",
                 "--train_size", "48", "--val_size", "24", "--batch_size", "8", "--val_batch_size", "8",
                 "--base_learning_rate", "0.05", "--training_number_of_steps", "200", "--weight_mode", "score",
                 "--score_reduce", "shape", "--fold_gap", "--how_many_training_epochs", "3",
                 "--train_logdir", str(tmp_path)])
    assert len(h) == 3 and h[-1][1] < h[0][1], "training loss should go down: %s" % h


def test_new_entry_points_reject_bad_arguments(cabi):
    """Null pointers, a small workspace, V = 5, G = 300 and a misaligned dS_gap: negative codes, nothing launched."""
    L = cabi.lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    p = ctypes.c_void_p((p.value + 15) // 16 * 16)
    odd = ctypes.c_void_p(p.value + 4)
    B, V, HW, C, G = 4, 12, 100, 1024, 10
    ws = L.gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes(B, V, HW, C, cabi.F32)
    assert ws > 0 and ws % (V * 4) == 0
    assert L.gvcnn_pool_fuse_gap_bwd_weights_workspace_bytes(B, V, HW, 96, cabi.F32) == 0

    def gbw(F=p, dS=p, S=p, bins=p, w=p, dw=p, work=p, nbytes=1 << 20, V=V, G=G, pool=0, dt=cabi.F32):
        return L.gvcnn_pool_fuse_gap_bwd_weights(F, dS, S, bins, V, w, G, dw, work, nbytes, B, V, HW, C, G, pool, 0, dt,
                                                 None)
    assert gbw(F=None) == -1 and gbw(dS=None) == -1 and gbw(S=None) == -1 and gbw(w=None) == -1
    assert gbw(dw=None) == -1 and gbw(work=None) == -1
    assert gbw(nbytes=16) == -9
    assert gbw(V=5) == -10 and gbw(G=300) == -10
    assert gbw(dS=odd) == -6
    assert gbw(pool=3) == -8 and gbw(dt=7) == -2
    fwd = L.gvcnn_pool_fuse_gap_weighted_fwd
    assert fwd(p, None, V, p, G, p, None, None, p, 1 << 20, B, V, HW, C, G, 0, 0.0, 0, 0, None) == -1
    assert fwd(p, p, V, p, G, p, None, None, p, 1 << 26, B, 5, HW, C, G, 0, 0.0, 0, 0, None) == -10
    assert fwd(p, p, V, p, 300, p, None, None, p, 1 << 26, B, V, HW, C, 300, 0, 0.0, 0, 0, None) == -10
    assert fwd(p, p, V, p, 65, p, None, None, p, 1 << 26, B, V, HW, C, 65, 0, 1.0, 0, 0, None) == -10
    assert fwd(p, p, V, p, G, p, None, None, p, 16, B, V, HW, C, G, 0, 0.0, 0, 0, None) == -9
    bwd = L.gvcnn_pool_fuse_gap_weighted_bwd
    assert bwd(p, p, V, p, G, None, p, None, B, V, HW, C, G, 0, 0, 0, None) == -1           # max needs the tie mask
    assert bwd(odd, p, V, p, G, p, p, None, B, V, HW, C, G, 0, 0, 0, None) == -10
    sb = L.gvcnn_gap_score_bwd
    assert sb(None, p, p, B, V, HW, C, 0, 0, None) == -1
    assert sb(p, p, None, B, V, HW, C, 0, 0, None) == -1
    assert sb(p, odd, p, B, V, HW, C, 0, 0, None) == -6
