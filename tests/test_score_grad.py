"""Gradient of the view discrimination scores (nets/model.py:144-147): gvcnn_score_bin_bwd and every entry point that
returns scores (view_scores, score_bin, grouping_fusion, GVCNNHead, gvcnn_head), against the float32 restatement in
score_grad_oracle.py (bit for bit) and float64 torch autograd (within tolerance)."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import score_grad_oracle as SO                                  # noqa: E402

from gvcnn_tf_b200 import _cabi as C                            # noqa: E402

f32 = np.float32
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


def _bits_equal(a, b):
    """Bit-identical float32 arrays, any NaN matching any NaN."""
    a = np.ascontiguousarray(a, dtype=f32)
    b = np.ascontiguousarray(b, dtype=f32)
    assert a.shape == b.shape, (a.shape, b.shape)
    both_nan = np.isnan(a) & np.isnan(b)
    bad = (a.view(np.uint32) != b.view(np.uint32)) & ~both_nan
    assert not bad.any(), "%d of %d differ, first at %s: %r vs %r" % (
        bad.sum(), a.size, np.argwhere(bad)[0], a[tuple(np.argwhere(bad)[0])], b[tuple(np.argwhere(bad)[0])])


def _p(t):
    return None if t is None else (t.data_ptr() or None)


def _tail_inputs(rng, n):
    """x with zeros, negatives, large and tiny magnitudes; g with +-0."""
    x = rng.standard_normal(n).astype(f32) * f32(3)
    g = rng.standard_normal(n).astype(f32)
    k = max(n // 8, 1)
    x[:k] = f32(0)
    x[k:2 * k] = rng.choice([f32(1e30), f32(-3e38), f32(1e-30), f32(-1e-38), f32(2.0 ** 25)], k)
    g[2 * k:3 * k] = f32(0)
    g[3 * k:4 * k] = f32(-0.0)
    ax = np.abs(x)
    with np.errstate(all="ignore"):
        s = np.where(np.isinf(ax), f32(1), ax / (f32(1) + ax)).astype(f32)    # the library's forward value
    return g, x, s


# ----------------------------------------------------------------------------------------------------------------------
# CPU: the oracle against float64 autograd and against the other association
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["shape", "batch"])
def test_oracle_vs_float64_autograd(mode):
    rng = np.random.default_rng(1)
    B, V, Cc = 9, 5, 16
    R = rng.standard_normal((B, V, Cc)).astype(f32)
    W = (rng.standard_normal((V, Cc)) * 0.3).astype(f32)
    b = rng.standard_normal(V).astype(f32)
    Rt, Wt, bt = (torch.tensor(a, dtype=torch.float64, requires_grad=True) for a in (R, W, b))
    x = (Rt * Wt[None]).sum(-1) + bt
    if mode == "batch":
        x = x.mean(0)
    s = torch.sigmoid(torch.log(torch.abs(x)))
    g = rng.standard_normal(tuple(s.shape)).astype(f32)
    s.backward(torch.tensor(g, dtype=torch.float64))
    xv, sv = x.detach().numpy().astype(f32), s.detach().numpy().astype(f32)
    if mode == "shape":
        dx = SO.view_scores_bwd(g, xv, sv)
    else:
        _, dx = SO.view_scores_bwd(g, xv, sv, "batch", B, B)
    np.testing.assert_allclose(SO.dW(R, dx), Wt.grad.numpy(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(SO.dbias(dx), bt.grad.numpy(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(SO.dense_dR(dx, W, "f32"), Rt.grad.numpy(), rtol=1e-4, atol=1e-7)


def test_oracle_associations_agree():
    rng = np.random.default_rng(2)
    g, x, s = _tail_inputs(rng, 4096)
    a = SO.view_scores_bwd(g, x, s, association="scalar")
    b = SO.view_scores_bwd(g, x, s, association="packet")
    ok = np.isfinite(a)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    np.testing.assert_allclose(a[ok], b[ok], rtol=4e-7, atol=0)
    assert np.isnan(a[x == 0]).all()                           # 0 * inf, as in TF


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
def _lib():
    return C.lib()


def _tail_bwd(g, x, s, mode, B, V, N=0, exchange=None, user=None):
    dev = "cuda"
    gt, xt, st = (torch.tensor(a, device=dev) for a in (g, x, s))
    dx = torch.full((B, V), float("nan"), device=dev)
    dxm = torch.full((V,), float("nan"), device=dev) if mode == "batch" else None
    rc = _lib().gvcnn_score_bin_bwd(_p(gt), _p(xt), _p(st), _p(dxm), _p(dx), B, V,
                                    C.SCORE_REDUCE_BATCH if mode == "batch" else C.SCORE_REDUCE_SHAPE, N, exchange,
                                    user, None)
    C.check(rc, "gvcnn_score_bin_bwd")
    torch.cuda.synchronize()
    return dx.cpu().numpy(), (dxm.cpu().numpy() if dxm is not None else None)


@pytest.mark.gpu
@pytest.mark.parametrize("V", [4, 6, 12, 20, 33, 80])
@pytest.mark.parametrize("B", [1, 7, 4096])
@pytest.mark.parametrize("mode", ["shape", "batch"])
def test_tail_bit_exact(mode, B, V):
    rng = np.random.default_rng(B * 100 + V)
    if mode == "shape":
        g, x, s = (a.reshape(B, V) for a in _tail_inputs(rng, B * V))
        dx, _ = _tail_bwd(g, x, s, mode, B, V)
        _bits_equal(dx, SO.view_scores_bwd(g, x, s))
    else:
        g, x, s = _tail_inputs(rng, V)
        N = B + 3                                               # a shard of a larger global batch
        dx, dxm = _tail_bwd(g, x, s, mode, B, V, N)
        want_m, want = SO.view_scores_bwd(g, x, s, "batch", N, B)
        _bits_equal(dxm, want_m)
        _bits_equal(dx, want)


@pytest.mark.gpu
def test_tail_packet_association_within_tolerance():
    rng = np.random.default_rng(3)
    g, x, s = _tail_inputs(rng, 4096)
    dx, _ = _tail_bwd(g.reshape(64, 64), x.reshape(64, 64), s.reshape(64, 64), "shape", 64, 64)
    other = SO.view_scores_bwd(g, x, s, association="packet").reshape(64, 64)
    ok = np.isfinite(other)
    np.testing.assert_allclose(dx[ok], other[ok], rtol=4e-7, atol=0)
    assert np.array_equal(np.isnan(dx), np.isnan(other))


def _make_R(rng, B, V, Cc, dtype, layout, HW=1):
    shp = (B, V) + ((HW, Cc) if HW > 1 else (Cc,))
    R = rng.standard_normal(shp).astype(f32)
    R = SO.round_to(R, dtype)
    t = torch.tensor(R, device="cuda").to(DT[dtype])
    if layout == "vbd":
        arg = t.transpose(0, 1).contiguous()
    elif layout == "list":
        arg = [t[:, v].contiguous() for v in range(V)]
    else:
        arg = t.contiguous()
    return R, arg


def _leaf(arg):
    if isinstance(arg, list):
        return [a.clone().requires_grad_(True) for a in arg]
    return arg.clone().requires_grad_(True)


def _grad_bvd(leaf, layout):
    if isinstance(leaf, list):
        return torch.stack([a.grad for a in leaf], 1).float().cpu().numpy()
    g = leaf.grad
    if layout == "vbd":
        g = g.transpose(0, 1)
    return g.float().cpu().numpy()


def _fc(rng, V, Cc):
    W = (rng.standard_normal((V, Cc)) * (1.0 / np.sqrt(Cc))).astype(f32)
    b = rng.uniform(-0.5, 0.5, V).astype(f32)
    return W, b


def _check_entry(model, mode, dtype, layout, B, V, Cc, HW=1, entry="score_bin", N=None):
    rng = np.random.default_rng(B * 7 + V * 3 + Cc + HW)
    R, arg = _make_R(rng, B, V, Cc, dtype, layout, HW)
    W, b = _fc(rng, V, Cc)
    Wt = torch.tensor(W, device="cuda", requires_grad=True)
    bt = torch.tensor(b, device="cuda", requires_grad=True)
    Rl = _leaf(arg)
    lay = None if layout == "list" else layout
    kw = {} if N is None else {"global_count": N}
    if entry == "score_bin":
        sr = model.score_bin(Rl, Wt, bt, 10, score_reduce=mode, layout=lay, check=False, clamp=True, **kw)
    else:
        F = torch.randn((B, V, 64), device="cuda").to(DT[dtype])
        Fa = [F[:, v].contiguous() for v in range(V)] if layout == "list" else \
            (F.transpose(0, 1).contiguous() if layout == "vbd" else F)
        _, sr = model.grouping_fusion(Rl, Wt, bt, Fa, 10, score_reduce=mode, layout=lay, clamp=True, **kw)
    assert sr.scores.requires_grad and not sr.x.requires_grad and not sr.bins.requires_grad
    g = rng.standard_normal(tuple(sr.scores.shape)).astype(f32)
    sr.scores.backward(torch.tensor(g, device="cuda"))
    x, s = sr.x.detach().cpu().numpy(), sr.scores.detach().cpu().numpy()
    if mode == "shape":
        dx = SO.view_scores_bwd(g, x, s)
    else:
        _, dx = SO.view_scores_bwd(g[0], x[0], s[0], "batch", N or B, B)
    if HW > 1:
        # dW, db come from the pooled float32 R the GAP-folded score kernel writes: take it from the library
        rv = model._Views(arg, lay, "R")
        R_out = torch.empty((B, V, Cc), device="cuda")
        xx = torch.empty((B, V), device="cuda")
        C.check(_lib().gvcnn_gap_score_bin_fwd(rv.arg, _p(Wt.detach()), _p(bt.detach()), _p(R_out), _p(xx), None,
                                               None, None, None, B, V, HW, Cc, 1, rv.layout,
                                               model._dtype_code(rv.dtype), 0, 0, 0, None), "gap_score_bin_fwd")
        Rp = R_out.cpu().numpy()
        _bits_equal(_grad_bvd(Rl, layout), SO.gap_dmaps(dx, W, HW, dtype))
    else:
        Rp = R
        _bits_equal(_grad_bvd(Rl, layout), SO.dense_dR(dx, W, dtype))
    if B > 0:
        _bits_equal(Wt.grad.cpu().numpy(), SO.dW(Rp, dx))
        _bits_equal(bt.grad.cpu().numpy(), SO.dbias(dx))
    else:
        assert not Wt.grad.any() and not bt.grad.any()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16", "f16"])
@pytest.mark.parametrize("layout", ["bvd", "vbd", "list"])
@pytest.mark.parametrize("mode", ["shape", "batch"])
@pytest.mark.parametrize("B,V", [(4096, 12), (7, 33), (1, 6), (0, 4), (7, 80), (1, 20)])
def test_score_bin_grad_bit_exact(mode, layout, dtype, B, V):
    from gvcnn_tf_b200 import model
    if mode == "batch" and B == 0:
        pytest.skip("'batch' over an empty batch without an exchange is an error (covered by the exchange test)")
    N = B + 5 if mode == "batch" else None
    _check_entry(model, mode, dtype, layout, B, V, 256 if B < 4096 else 1024, N=N)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("layout", ["bvd", "vbd", "list"])
@pytest.mark.parametrize("mode", ["shape", "batch"])
def test_grouping_fusion_grad_bit_exact(mode, layout, dtype):
    from gvcnn_tf_b200 import model
    _check_entry(model, mode, dtype, layout, 37, 12, 1024, entry="grouping_fusion")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,Cc", [("f32", 512), ("f32", 1024), ("bf16", 1024), ("f16", 2048)])
@pytest.mark.parametrize("layout", ["bvd", "vbd", "list"])
@pytest.mark.parametrize("mode", ["shape", "batch"])
def test_maps_grad_bit_exact(mode, layout, dtype, Cc):
    from gvcnn_tf_b200 import model
    _check_entry(model, mode, dtype, layout, 5, 12, Cc, HW=4)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["shape", "batch"])
def test_entry_points_agree(mode):
    """view_scores, score_bin, grouping_fusion and GVCNNHead: the same W, b and R gradients for the same loss."""
    from gvcnn_tf_b200 import model
    rng = np.random.default_rng(11)
    B, V, Cc, D = 24, 12, 1024, 256
    R = torch.tensor(rng.standard_normal((B, V, Cc)).astype(f32), device="cuda")
    F = torch.tensor(rng.standard_normal((B, V, D)).astype(f32), device="cuda")
    head = model.GVCNNHead(V, Cc, D, 5, score_reduce=mode).cuda()
    rows = 1 if mode == "batch" else B
    G = torch.tensor(rng.standard_normal((rows, V)).astype(f32), device="cuda")

    def run(fn):
        head.zero_grad(set_to_none=True)
        Rl = R.clone().requires_grad_(True)
        s = fn(Rl)
        (s * G).sum().backward()
        return head.score_kernel.grad.clone(), head.score_bias.grad.clone(), Rl.grad.clone()

    W, b = head.score_kernel, head.score_bias
    outs = [run(lambda r: model.view_scores(r, W, b, score_reduce=mode)),
            run(lambda r: model.score_bin(r, W, b, 10, score_reduce=mode, clamp=True).scores),
            run(lambda r: model.grouping_fusion(r, W, b, F, 10, score_reduce=mode, clamp=True)[1].scores),
            run(lambda r: head(r, F)[0])]
    for o in outs[1:]:
        for a, e in zip(o, outs[0]):
            assert torch.equal(a, e)


@pytest.mark.gpu
@pytest.mark.parametrize("maps", [False, True])
@pytest.mark.parametrize("fold_gap", [False, True])
@pytest.mark.parametrize("mode", ["shape", "batch"])
def test_classifier_only_loss_unchanged(mode, fold_gap, maps):
    from gvcnn_tf_b200 import model
    rng = np.random.default_rng(5)
    B, V, Cc, Cf = 16, 12, 1024, 2048
    R = torch.tensor(rng.standard_normal((B, V, 4, Cc) if maps else (B, V, Cc)).astype(f32), device="cuda")
    F = torch.tensor(rng.standard_normal((B, V, 2, 2, Cf)).astype(f32), device="cuda")
    head = model.GVCNNHead(V, Cc, Cf, 5, score_reduce=mode).cuda()
    labels = torch.tensor(rng.integers(0, 5, B), device="cuda")

    def step(detach, score_loss=0.0):
        head.zero_grad(set_to_none=True)
        Fl = F.clone().requires_grad_(True)
        if detach:
            W0, b0 = head.score_kernel, head.score_bias
            head.score_kernel, head.score_bias = (torch.nn.Parameter(W0.detach(), requires_grad=False),
                                                  torch.nn.Parameter(b0.detach(), requires_grad=False))
            try:
                s, S, logits = head(R, Fl, fold_gap=fold_gap)
            finally:
                head.score_kernel, head.score_bias = W0, b0
        else:
            s, S, logits = head(R, Fl, fold_gap=fold_gap)
        loss = torch.nn.functional.cross_entropy(logits, labels)
        if score_loss:
            loss = loss + score_loss * (s ** 2).sum()
        loss.backward()
        return s.detach(), S.detach(), logits.detach(), Fl.grad, head.score_kernel.grad, head.score_bias.grad

    ref = step(True)
    got = step(False)
    for a, e in zip(got[:4], ref[:4]):
        assert torch.equal(a, e)
    assert got[4] is None and got[5] is None                    # what train_head.py's gradient bucket relies on
    both = step(False, 0.5)
    assert torch.equal(both[3], ref[3])                         # the score loss does not touch dF
    head.zero_grad(set_to_none=True)
    s, _, _ = head(R, F, fold_gap=fold_gap)
    (0.5 * (s ** 2).sum()).backward()
    assert torch.equal(both[4], head.score_kernel.grad) and torch.equal(both[5], head.score_bias.grad)
    with torch.no_grad():
        s, _, _ = head(R, F, fold_gap=fold_gap)
    assert not s.requires_grad


@pytest.mark.gpu
def test_gvcnn_head_with_scheme_scores_differentiable():
    from gvcnn_tf_b200 import model
    rng = np.random.default_rng(6)
    B, V, Cc, D = 8, 12, 1024, 256
    R = torch.tensor(rng.standard_normal((B, V, Cc)).astype(f32), device="cuda")
    F = torch.tensor(rng.standard_normal((B, V, D)).astype(f32), device="cuda")
    head = model.GVCNNHead(V, Cc, D, 5).cuda()
    scheme = model.group_scheme(model.view_scores(R, head.score_kernel.detach(), head.score_bias.detach()), 10, V,
                                check=False)
    s, _, _ = model.gvcnn_head(R, F, head, group_scheme=scheme)
    s.sum().backward()
    want_W = head.score_kernel.grad.clone()
    head.zero_grad(set_to_none=True)
    model.view_scores(R, head.score_kernel, head.score_bias).sum().backward()
    assert torch.equal(head.score_kernel.grad, want_W)


class _Exchange:
    """An exchange callback for one simulated rank: its i-th call adds addends[i] (the other rank's buffer of the
    matching call, or None: nothing) to the buffer in place, and records the buffer before and after."""

    def __init__(self, addends=()):
        self.addends, self.calls, self.after = list(addends), [], []
        self.cb = C.EXCHANGE_FN(self._fn)

    def _fn(self, _user, ptr, n, _stream):
        t = torch.as_tensor(_DevArray(ptr, n), device="cuda")
        self.calls.append(t.clone())
        a = self.addends.pop(0) if self.addends else None
        if a is not None:
            t.add_(a)
        self.after.append(t.clone())
        return 0


class _DevArray:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (int(ptr), False), "version": 2}


@pytest.mark.gpu
@pytest.mark.parametrize("B0", [0, 9])
def test_adjoint_exchange_two_ranks_on_one_gpu(B0):
    """A batch split over two simulated ranks: the backward's exchange gives both the same dx_mean, and the two
    ranks' dW add up to the full batch's."""
    from gvcnn_tf_b200 import model
    rng = np.random.default_rng(7)
    V, Cc, B1 = 12, 1024, 23
    N = B0 + B1
    R = rng.standard_normal((N, V, Cc)).astype(f32)
    W, b = _fc(rng, V, Cc)
    g = [rng.standard_normal((1, V)).astype(f32) for _ in range(2)]
    shards = [R[:B0], R[B0:]]

    def rank_pass(r, ex):
        Wt = torch.tensor(W, device="cuda", requires_grad=True)
        bt = torch.tensor(b, device="cuda", requires_grad=True)
        sr = model.score_bin(torch.tensor(shards[r], device="cuda").reshape(-1, V, Cc), Wt, bt, 10,
                             score_reduce="batch", edge_ulps=0, clamp=True, check=False, exchange=(ex.cb, None),
                             global_count=N)
        sr.scores.backward(torch.tensor(g[r], device="cuda"))
        return sr, Wt.grad, bt.grad

    p1 = [_Exchange(), _Exchange()]                             # each rank's own column sums
    for r in range(2):
        rank_pass(r, p1[r])
    assert all(len(e.calls) == 2 for e in p1)                   # forward sums, backward dx_mean: an empty rank too
    xs = [e.calls[0] for e in p1]
    p2 = [_Exchange([xs[1], None]), _Exchange([xs[0], None])]   # global scores; each rank's own dx_mean
    for r in range(2):
        rank_pass(r, p2[r])
    dl = [e.calls[1] for e in p2]
    p3 = [_Exchange([xs[1], dl[1]]), _Exchange([xs[0], dl[0]])]
    res = [rank_pass(r, p3[r]) for r in range(2)]
    assert torch.equal(p3[0].after[1], p3[1].after[1])         # both ranks apply the same global dx_mean
    assert torch.equal(res[0][0].scores, res[1][0].scores)
    x, s = res[0][0].x.cpu().numpy()[0], res[0][0].scores.detach().cpu().numpy()[0]
    _, dx = SO.view_scores_bwd(g[0][0] + g[1][0], x, s, "batch", N, N)
    np.testing.assert_allclose((res[0][1] + res[1][1]).cpu().numpy(), SO.dW(R, dx), rtol=1e-5, atol=1e-7)
    np.testing.assert_allclose((res[0][2] + res[1][2]).cpu().numpy(), SO.dbias(dx), rtol=1e-5, atol=1e-7)


@pytest.mark.gpu
def test_cabi_argument_checks():
    L = _lib()
    V, B = 12, 4
    t = torch.zeros(64, device="cuda")
    p, mis = _p(t), _p(t) + 2
    SH, BA = C.SCORE_REDUCE_SHAPE, C.SCORE_REDUCE_BATCH
    E_ARG, E_MIS = -1, -6
    cb = C.EXCHANGE_FN(lambda *a: 0)
    assert L.gvcnn_score_bin_bwd(None, p, p, None, p, B, V, SH, 0, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, None, None, B, V, SH, 0, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(mis, p, p, None, p, B, V, SH, 0, None, None, None) == E_MIS
    assert L.gvcnn_score_bin_bwd(p, p, p, None, mis, B, V, SH, 0, None, None, None) == E_MIS
    assert L.gvcnn_score_bin_bwd(p, p, p, None, p, B, V, 2, 0, None, None, None) == -8
    assert L.gvcnn_score_bin_bwd(p, p, p, p, p, B, V, SH, 0, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, None, p, B, V, SH, 0, cb, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, p, p, B, V, BA, 0, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, p, p, B, V, BA, -3, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, p, p, B, V, BA, B - 1, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, None, p, B, V, BA, B, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, p, None, B, V, BA, B, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, p, None, 0, V, BA, 1, None, None, None) == E_ARG   # a mean over nothing
    assert L.gvcnn_score_bin_bwd(p, p, p, mis, p, B, V, BA, B, None, None, None) == E_MIS
    assert L.gvcnn_score_bin_bwd(p, p, p, None, p, B, 0, SH, 0, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, None, p, -1, V, SH, 0, None, None, None) == E_ARG
    assert L.gvcnn_score_bin_bwd(p, p, p, None, p, B, C.MAX_VIEWS + 1, SH, 0, None, None, None) == -4
    assert L.gvcnn_score_bin_bwd(None, None, None, None, None, 0, V, SH, 0, None, None, None) == 0
    torch.cuda.synchronize()
