"""Multi-process (world_size 2, gloo, CPU) tests of the N>1 host logic: shape sharding, the
parameter-gradient bucket all-reduce, the init broadcast, and the pre-binning all-reduce of the
literal batch-mean score (checked with the oracle, since kernels need a GPU)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gvcnn_tf_b200 import parallel
from oracle import gvcnn_oracle as O


def test_shard_range_partitions_exactly():
    for n in (0, 1, 7, 4096, 2468):
        for k in (1, 2, 3, 4, 8):
            spans = [parallel.shard_range(n, r, k) for r in range(k)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(k - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        parallel.shard_range(4, 2, 2)


def test_every_rank_runs_the_same_number_of_steps():
    """train_size=66, world=4, batch 4 gives shards of 17/17/16/16 shapes = 5/5/4/4 batches: a rank-local loop would
    issue a different number of all-reduces per rank and hang NCCL.  steps_per_epoch is the largest rank's count, and
    global_batch_size says how many shapes the literal batch mean of each step is over."""
    for n, k, bs in ((66, 4, 4), (64, 8, 4), (7, 2, 4), (4096, 8, 512), (3, 4, 2)):
        steps = parallel.steps_per_epoch(n, k, bs)
        per_rank = [-(-(parallel.shard_range(n, r, k)[1] - parallel.shard_range(n, r, k)[0]) // bs) for r in range(k)]
        assert steps == max(per_rank)
        assert sum(parallel.global_batch_size(n, k, bs, st) for st in range(steps)) == n
        assert all(parallel.global_batch_size(n, k, bs, st) > 0 for st in range(steps))
        assert parallel.global_batch_size(n, k, bs, steps) == 0
    assert parallel.steps_per_epoch(66, 4, 4) == 5


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(100 + rank)
        # --- P2PComm construction is collective: without a GPU it must fail on EVERY rank, after both of its
        #     exchanges, instead of leaving a rank waiting in a collective the others skipped
        try:
            parallel.P2PComm()
            raise AssertionError("P2PComm must not come up without a CUDA device")
        except RuntimeError as e:
            assert "could not be set up on every rank" in str(e), str(e)
        dist.barrier()

        # --- init broadcast (utils/_train_helper.py:66-94)
        lin = torch.nn.Linear(5, 3)
        parallel.broadcast_parameters(lin, src=0)
        gathered = [torch.zeros_like(lin.weight) for _ in range(world)]
        dist.all_gather(gathered, lin.weight.data)
        assert all(torch.equal(g, gathered[0]) for g in gathered)

        # --- grad bucket: sum then 1/K (utils/_train_helper.py:17-31); None grads count as zeros
        score_kernel = torch.nn.Parameter(torch.zeros(12, 16))        # no grad in literal mode (D6)
        lin.weight.grad = torch.full_like(lin.weight, float(rank + 1))
        lin.bias.grad = torch.full_like(lin.bias, float(10 * (rank + 1)))
        bucket = parallel.GradBucket([score_kernel, lin.weight, lin.bias])
        bucket.pack()
        work = bucket.all_reduce_mean(async_op=True)
        bucket.finish(work)
        bucket.unpack()
        mean = sum(range(1, world + 1)) / world
        assert torch.allclose(lin.weight.grad, torch.full_like(lin.weight, mean))
        assert torch.allclose(lin.bias.grad, torch.full_like(lin.bias, 10 * mean))
        assert torch.equal(score_kernel.grad, torch.zeros_like(score_kernel))

        # --- sharded forward == unsharded forward (shape independence), via the oracle
        rng = np.random.default_rng(0)                                # same data on every rank
        B, V, D, G, Cr = 11, 6, 16, 10, 32
        F = rng.standard_normal((B, V, D)).astype(np.float32)
        R = rng.standard_normal((B, V, Cr)).astype(np.float32)
        W = rng.uniform(-0.3, 0.3, (V, Cr)).astype(np.float32)
        b = rng.uniform(-3, 3, V).astype(np.float32)
        lo, hi = parallel.shard_range(B, rank, world)
        full = O.grouping_fusion_fwd(R, W, b, F, G, score_reduce="shape")
        mine = O.grouping_fusion_fwd(R[lo:hi], W, b, F[lo:hi], G, score_reduce="shape")
        np.testing.assert_array_equal(mine["S"], full["S"][lo:hi])
        np.testing.assert_array_equal(mine["bins"], full["bins"][lo:hi])

        # --- literal batch-mean score: all-reduce of the V partial sums gives every rank the
        #     global-batch bins (SURVEY 8e collective 2)
        x_local, _ = O.view_scores(R[lo:hi], W, b, "shape", np.float64)
        xsum = torch.tensor(x_local.sum(axis=0))
        cnt = torch.tensor([hi - lo], dtype=torch.int64)
        dist.all_reduce(xsum)
        dist.all_reduce(cnt)
        xbar = (xsum / cnt.item()).numpy()
        bins = O.bins_from_scores(O.score_from_x(xbar).astype(np.float32), G)
        np.testing.assert_array_equal(bins, O.grouping_fusion_fwd(R, W, b, F, G, score_reduce="batch")["bins"][0])
        with open(os.path.join(tmp, "ok_%d" % rank), "w") as f:
            f.write("ok")
    finally:
        dist.destroy_process_group()


def test_world_size_2_gloo(tmp_path, monkeypatch):
    # the workers check the no-GPU behaviour: hide any device, or on a GPU box both ranks would share one and P2PComm
    # would come up
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.path.exists(tmp_path / "ok_0") and os.path.exists(tmp_path / "ok_1")
