#!/usr/bin/env python
"""torchrun check of the score backward on N GPUs, 'batch' mode with a sharded batch: each rank scores its shard
(the forward all-reduces the column sums), puts a DIFFERENT loss on the shared scores, and runs the backward (which
all-reduces the gradient of the batch mean).  Every rank must see the same scores; the ranks' dW and db, summed, must
match one GPU's backward of the whole batch under the summed loss (within float32 tolerance: the order of the sums
differs); the last rank has an empty shard and must still take part.  Run with the exchange of a torch.distributed
process group (NCCL) and with the library's own P2PComm.

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 scripts/score_grad_multi_check.py
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gvcnn_tf_b200 import model, parallel  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
dist.init_process_group("nccl")
V, Cr, per = 12, 1024, 37
N = per * (world - 1)                                               # the last rank's shard is empty
g = torch.Generator(device="cuda").manual_seed(0)
R = torch.randn((N, V, Cr), device="cuda", generator=g)
W0 = torch.randn((V, Cr), device="cuda", generator=g) * Cr ** -0.5
b0 = torch.rand(V, device="cuda", generator=g) - 0.5
G = torch.randn((world, 1, V), device="cuda", generator=g)          # one loss weight row per rank
shard = R[rank * per:(rank + 1) * per] if rank < world - 1 else R[:0]


def rank_grads(**kw):
    W, b = W0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    sr = model.score_bin(shard, W, b, 10, score_reduce="batch", edge_ulps=0, clamp=True, check=False,
                         global_count=N, **kw)
    (sr.scores * G[rank]).sum().backward()
    flat = torch.cat([W.grad.reshape(-1), b.grad, sr.scores.detach().reshape(-1)])
    return flat


# one GPU, the whole batch, the summed loss
W, b = W0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
sr = model.score_bin(R, W, b, 10, score_reduce="batch", edge_ulps=0, clamp=True, check=False)
(sr.scores * G.sum(0)).sum().backward()
want_W, want_b, want_s = W.grad, b.grad, sr.scores.detach().reshape(-1)

comm = parallel.P2PComm()
forms = [("process_group", {"process_group": dist.group.WORLD}), ("P2PComm", {"exchange": comm.exchange})]
for name, kw in forms:
    flat = rank_grads(**kw)
    scores = flat[-V:]
    allg = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(allg, flat)
    assert all(torch.equal(a[-V:], scores) for a in allg), name + ": scores differ across ranks"
    dW = sum(a[:V * Cr] for a in allg).reshape(V, Cr)
    db = sum(a[V * Cr:V * Cr + V] for a in allg)
    torch.testing.assert_close(scores, want_s, rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(dW, want_W, rtol=1e-4, atol=1e-6)
    torch.testing.assert_close(db, want_b, rtol=1e-4, atol=1e-6)
    if rank == 0:
        print("score grad multi-GPU check ok (%s): world %d, empty last shard" % (name, world))
dist.barrier()
comm.close()
dist.destroy_process_group()
