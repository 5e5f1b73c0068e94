"""The Python mirror's own routing (gvcnn_tf_b200.model): the one-call forward in both score modes against the staged
score_bin -> pool_fuse path, for every view layout and with a gradient, and the exchange callback in both of the
forms P2PComm offers.  Run on the B200 box with ``pytest -m gpu``."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def model():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from gvcnn_tf_b200 import model as m, _cabi
    assert _cabi.lib().gvcnn_check_device() == 0, "libgvcnn_sm100.so needs a compute-capability 10.x device"
    return m


def _inputs(seed, B, V, Cr, D):
    rng = np.random.default_rng(seed)
    R = rng.standard_normal((B, V, Cr)).astype(np.float32)
    W = rng.uniform(-0.1, 0.1, (V, Cr)).astype(np.float32)
    b = rng.uniform(-2.0, 2.0, V).astype(np.float32)
    F = np.maximum(np.round(rng.standard_normal((B, V, D)) * 2) / 2, 0).astype(np.float32)   # ties for max pooling
    dS = rng.standard_normal((B, D)).astype(np.float32)
    return R, W, b, F, dS


def _as_layout(a, layout):
    """[B, V, ...] numpy -> the view argument in `layout` (a fresh leaf, so each path gets its own .grad)."""
    if layout == "bvd":
        return torch.tensor(a, device="cuda")
    if layout == "vbd":
        return torch.tensor(np.ascontiguousarray(a.swapaxes(0, 1)), device="cuda")
    return [torch.tensor(np.ascontiguousarray(a[:, v]), device="cuda") for v in range(a.shape[1])]


def _grad_bvd(F, layout):
    if layout == "bvd":
        return F.grad.cpu().numpy()
    if layout == "vbd":
        return F.grad.cpu().numpy().swapaxes(0, 1)
    return np.stack([t.grad.cpu().numpy() for t in F], axis=1)


@pytest.mark.parametrize("pool", ["max", "mean"])
@pytest.mark.parametrize("layout", ["bvd", "vbd", "list"])
@pytest.mark.parametrize("score_reduce", ["shape", "batch"])
def test_grouping_fusion_equals_staged_path_with_gradient(model, score_reduce, layout, pool):
    """grouping_fusion (gvcnn_grouping_fusion_fwd / _batch_fwd, backward through the pooling backward) gives the
    bits of score_bin -> pool_fuse: bins, S and dF."""
    B, V, Cr, D, G = 37, 12, 256, 1024, 8
    R, W, b, F, dS = _inputs(7 + V, B, V, Cr, D)
    Wd, bd, dSd = (torch.tensor(a, device="cuda") for a in (W, b, dS))
    lay = None if layout == "list" else layout

    F1 = _as_layout(F, layout)
    for t in (F1 if layout == "list" else [F1]):
        t.requires_grad_(True)
    S1, sr1 = model.grouping_fusion(_as_layout(R, layout), Wd, bd, F1, G, pool=pool, score_reduce=score_reduce,
                                    layout=lay, clamp=True)
    S1.backward(dSd)

    F2 = _as_layout(F, layout)
    for t in (F2 if layout == "list" else [F2]):
        t.requires_grad_(True)
    sr2 = model.score_bin(_as_layout(R, layout), Wd, bd, G, score_reduce=score_reduce, layout=lay, clamp=True)
    S2 = model.pool_fuse(F2, sr2.bins, G, pool=pool, layout=lay)
    S2.backward(dSd)
    torch.cuda.synchronize()

    assert tuple(S1.shape) == tuple(S2.shape) == (B, D)
    np.testing.assert_array_equal(sr1.bins.cpu().numpy(), sr2.bins.cpu().numpy())
    assert len(np.unique(sr1.bins.cpu().numpy())) > 2                   # the biases spread the views over bins
    np.testing.assert_array_equal(S1.detach().cpu().numpy(), S2.detach().cpu().numpy())
    np.testing.assert_array_equal(_grad_bvd(F1, layout), _grad_bvd(F2, layout))


@pytest.mark.parametrize("form", ["callable", "pointer"])
@pytest.mark.parametrize("edge_ulps", [0, 4])
def test_score_bin_batch_exchange_in_both_forms(model, form, edge_ulps):
    """score_bin(score_reduce='batch', exchange=(fn, user)) with fn an EXCHANGE_FN callback or its address, on the
    one-call path (edge_ulps=0: column sums, exchange and binning inside the library) and on the staged one (the
    order-sensitivity report needs the |R W| sums too, so score_bin calls the exchange itself).  An identity
    exchange (one rank) gives the bins and scores of no exchange."""
    from gvcnn_tf_b200 import _cabi
    B, V, Cr, G = 300, 12, 512, 10
    R, W, b, _, _ = _inputs(3, B, V, Cr, 4)
    Rd, Wd, bd = (torch.tensor(a, device="cuda") for a in (R, W, b))
    calls = []

    def _identity(_user, xsum_ptr, n, _stream):
        calls.append(n)
        return 0
    cb = _cabi.EXCHANGE_FN(_identity)
    fn = cb if form == "callable" else ctypes.cast(cb, ctypes.c_void_p)
    want = model.score_bin(Rd, Wd, bd, G, score_reduce="batch", edge_ulps=edge_ulps, clamp=True)
    got = model.score_bin(Rd, Wd, bd, G, score_reduce="batch", edge_ulps=edge_ulps, clamp=True, exchange=(fn, None))
    torch.cuda.synchronize()
    assert len(calls) == 1
    assert torch.equal(got.bins, want.bins) and torch.equal(got.scores, want.scores)
    assert len(np.unique(got.bins.cpu().numpy())) > 2


@pytest.mark.parametrize("score_reduce", ["shape", "batch"])
def test_grouping_fusion_rejects_score_fc_shape_mismatch(model, score_reduce):
    """A W narrower than R's channels, a b shorter than V, and channel-last maps whose trailing dimension is not C_raw
    raise ValueError before anything is launched, as in score_bin (the score kernel would read past W or b)."""
    B, V, Cr, D, G = 8, 12, 256, 64, 8
    R, W, b, F, _ = _inputs(5, B, V, Cr, D)
    Rd, Wd, bd, Fd = (torch.tensor(a, device="cuda") for a in (R, W, b, F))
    maps = torch.randn((B, V, 2, 2, Cr // 2), device="cuda")          # h * w * C' = 2 C_raw: not descriptors either
    for args in ((Rd, Wd[:, :Cr // 2], bd), (Rd, Wd, bd[:V - 1]), (maps, Wd, bd)):
        with pytest.raises(ValueError):
            model.grouping_fusion(*args, Fd, G, score_reduce=score_reduce)
