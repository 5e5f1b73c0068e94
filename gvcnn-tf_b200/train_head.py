#!/usr/bin/env python
"""train.py-shaped driver for the grouping + fusion head (SURVEY.md 8f n3).

Mirrors the step structure and flag names of the reference's ``train.py`` for the part of the graph this
repo owns - everything downstream of the backbone (which is out of scope, so the per-view features come
from a feature source; a seeded synthetic one is built in):

    reference (train.py:253-380)                      here
    ------------------------------------------------  ------------------------------------------------
    partial_run #1 -> host group_scheme/group_weight   one device pass: score+bin -> pool+fuse (no host hop)
    -> partial_run #2                                  -> GAP -> Dense(num_classes) -> softmax xent
    MomentumOptimizer(lr, momentum)                    torch.optim.SGD(momentum), same 'poly'/'step' policy
    tf.train.Saver, one ckpt per epoch, resume         torch.save per epoch to train_logdir, --saved_checkpoint_dir
    validation loop + confusion matrix per epoch       same (train.py:319-374)

Multi-GPU: launch with torchrun; shapes are sharded by rank and the head's gradients are all-reduced
in one flat bucket (parallel.GradBucket).  Usage (synthetic features):
    python gvcnn-tf_b200/train_head.py --how_many_training_epochs 2 --num_views 12 --num_group 10
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gvcnn_tf_b200 import _cabi, model, parallel  # noqa: E402

C_COMM_MAX_FLOATS, C_COMM_MAX_WORLD = _cabi.COMM_MAX_FLOATS, _cabi.COMM_MAX_WORLD


def build_flags():
    """Flag names and defaults of train.py:20-103 that concern this path."""
    p = argparse.ArgumentParser()
    p.add_argument("--train_logdir", default="./tfmodels")
    p.add_argument("--ckpt_name_to_save", default="gvcnn.ckpt")
    p.add_argument("--saved_checkpoint_dir", default=None)
    p.add_argument("--learning_policy", default="poly", choices=["poly", "step"])
    p.add_argument("--base_learning_rate", type=float, default=0.001)
    p.add_argument("--learning_rate_decay_factor", type=float, default=1e-3)
    p.add_argument("--learning_rate_decay_step", type=float, default=0.3)
    p.add_argument("--learning_power", type=float, default=0.9)
    p.add_argument("--training_number_of_steps", type=float, default=300000)
    p.add_argument("--momentum", type=float, default=0.9)
    p.add_argument("--slow_start_step", type=int, default=0)
    p.add_argument("--slow_start_learning_rate", type=float, default=1e-4)
    p.add_argument("--how_many_training_epochs", type=int, default=100)
    p.add_argument("--batch_size", type=int, default=4)
    p.add_argument("--val_batch_size", type=int, default=4)
    p.add_argument("--num_views", type=int, default=6)
    p.add_argument("--num_group", type=int, default=10)
    p.add_argument("--labels", default="airplane,bed,bookshelf,toilet,vase")
    # head / feature-source options (no reference counterpart: the backbone is out of scope)
    p.add_argument("--raw_channels", type=int, default=1024)        # block3 depth, nets/resnet_v2.py:242
    p.add_argument("--final_channels", type=int, default=2048)      # block4 depth
    p.add_argument("--feature_hw", type=int, default=1)             # 10 for the reference's 299x299 inputs
    p.add_argument("--train_size", type=int, default=64)
    p.add_argument("--val_size", type=int, default=32)
    p.add_argument("--weight_mode", default="count", choices=["count", "score"])
    p.add_argument("--score_reduce", default="batch", choices=["batch", "shape"])
    p.add_argument("--fold_gap", action="store_true")              # GAP after the fusion folded into the pooling
    p.add_argument("--seed", type=int, default=0)
    return p


def learning_rate(flags, global_step):
    """utils/train_utils.py:65-118 (get_model_learning_rate): 'poly' = tf polynomial_decay with
    end_learning_rate 0, 'step' = staircase exponential decay; slow start for the first steps."""
    if global_step < flags.slow_start_step:
        return flags.slow_start_learning_rate
    if flags.learning_policy == "poly":
        step = min(global_step, flags.training_number_of_steps)
        return flags.base_learning_rate * (1 - step / flags.training_number_of_steps) ** flags.learning_power
    return flags.base_learning_rate * flags.learning_rate_decay_factor ** int(global_step / flags.learning_rate_decay_step)


class SyntheticFeatures:
    """Seeded stand-in for the backbone: class-dependent raw (block3 GAP) and final (block4) features."""

    def __init__(self, n, flags, num_classes, seed, device):
        g = torch.Generator().manual_seed(seed)
        V, Cr, Cf, hw = flags.num_views, flags.raw_channels, flags.final_channels, flags.feature_hw
        self.labels = torch.randint(0, num_classes, (n,), generator=g)
        proto = torch.randn((num_classes, Cf), generator=torch.Generator().manual_seed(1234))
        self.raw = torch.randn((n, V, Cr), generator=g)
        noise = torch.randn((n, V, hw, hw, Cf), generator=g)
        self.final = torch.relu(noise + 1.5 * proto[self.labels][:, None, None, None, :])
        self.device = device

    def batches(self, bs, lo=0, hi=None):
        hi = len(self.labels) if hi is None else hi
        for i in range(lo, hi, bs):
            j = min(i + bs, hi)
            yield (self.raw[i:j].to(self.device), self.final[i:j].to(self.device), self.labels[i:j].to(self.device))

    def empty_batch(self):
        """A zero-shape batch: what a rank whose shard is exhausted contributes to the epoch's last step."""
        return (self.raw[:0].to(self.device), self.final[:0].to(self.device), self.labels[:0].to(self.device))


class _BucketOverlap:
    """Overlaps the flat gradient all-reduce with the rest of the backward pass.  In the reference-literal mode the
    only parameters with a gradient are the classifier's (the score FC gets none, SURVEY D6), and autograd produces
    them FIRST - before the pooling/fusion backward kernel that dominates the step.  A post-accumulate hook on each
    parameter counts the gradients in; when the last expected one has arrived the bucket is packed and the all-reduce
    (the library's one-kernel NVLink all-reduce, or NCCL) is launched on its own stream, while the dF kernel still runs
    on the main one; join() orders the optimizer step behind it."""

    def __init__(self, head, bucket, comm, world):
        self.bucket, self.comm, self.world = bucket, comm, world
        self.stream = torch.cuda.Stream(priority=-1)
        self.fired, self.work, self.pending = False, None, 0
        self.expected = [p for p in bucket.params if p.requires_grad]
        literal = getattr(head, "weight_mode", "count") == "count"
        # parameters that receive a gradient in this mode (the score FC only in paper mode)
        self.with_grad = [p for n, p in head.named_parameters()
                          if p.requires_grad and not (literal and n in ("score_kernel", "score_bias"))]
        for p in self.with_grad:
            p.register_post_accumulate_grad_hook(self._hook)

    def reset(self):
        self.fired, self.work, self.pending = False, None, len(self.with_grad)

    def _hook(self, _param):
        self.pending -= 1
        if self.pending == 0 and not self.fired:
            self.launch()

    def launch(self):
        self.fired = True
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            self.bucket.pack()
            if self.comm is not None:
                self.comm.all_reduce_(self.bucket.flat, 1.0 / self.world, stream=self.stream)   # sum * 1/K, one kernel
            else:
                self.work = self.bucket.all_reduce_mean(async_op=True)

    def join(self):
        if self.work is not None:
            with torch.cuda.stream(self.stream):
                self.bucket.finish(self.work)
        torch.cuda.current_stream().wait_stream(self.stream)


def confusion_matrix(labels, preds, n):
    cm = torch.zeros((n, n), dtype=torch.int64)
    for t, p in zip(labels.tolist(), preds.tolist()):
        cm[t, p] += 1
    return cm


def main(argv=None):
    flags = build_flags().parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("train_head.py needs a CUDA device: the grouping/fusion path has no CPU fallback")
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")   # the small all-reduce must not queue behind dF
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = torch.device("cuda", local_rank if world > 1 else 0)
    labels = flags.labels.split(",")
    num_classes = len(labels)
    torch.manual_seed(flags.seed)
    head = model.GVCNNHead(flags.num_views, flags.raw_channels, flags.final_channels, num_classes,
                           num_group=flags.num_group, score_reduce=flags.score_reduce,
                           weight_mode=flags.weight_mode).to(device)
    if flags.score_reduce == "batch" and flags.weight_mode == "count":
        with torch.no_grad():                       # spread the batch-mean scores over the bins
            head.score_bias.uniform_(-3, 3)
    if world > 1:
        parallel.broadcast_parameters(head, src=0)
    opt = torch.optim.SGD(head.parameters(), lr=flags.base_learning_rate, momentum=flags.momentum)
    bucket = parallel.GradBucket(list(head.parameters()), device=device) if world > 1 else None
    comm, pg = None, None
    if world > 1:
        import torch.distributed as dist
        pg = dist.group.WORLD
        if bucket.flat.numel() <= C_COMM_MAX_FLOATS and world <= C_COMM_MAX_WORLD:
            try:                                    # the library's one-kernel NVLink all-reduce (csrc/comm.cu)
                comm = parallel.P2PComm()
            except Exception as e:                  # noqa: BLE001 - e.g. IPC not permitted: NCCL carries the bucket
                comm = None
                if rank == 0:
                    print("P2PComm unavailable (%s); gradient bucket goes through NCCL" % e)
            ok = torch.tensor([1 if comm is not None else 0], device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0 and comm is not None:
                comm.close()
                comm = None

    overlap = _BucketOverlap(head, bucket, comm, world) if bucket is not None else None

    start_epoch, global_step = 0, 0
    if flags.saved_checkpoint_dir:                  # train.py:229-234: restore the latest checkpoint
        cks = sorted(f for f in os.listdir(flags.saved_checkpoint_dir) if f.startswith(flags.ckpt_name_to_save))
        if cks:
            ck = torch.load(os.path.join(flags.saved_checkpoint_dir, cks[-1]), map_location=device)
            head.load_state_dict(ck["head"])
            opt.load_state_dict(ck["opt"])
            start_epoch, global_step = ck["epoch"] + 1, ck["global_step"]

    train = SyntheticFeatures(flags.train_size, flags, num_classes, flags.seed + 1, device)
    val = SyntheticFeatures(flags.val_size, flags, num_classes, flags.seed + 2, device)
    lo, hi = parallel.shard_range(flags.train_size, rank, world)
    # every rank must issue the SAME number of collectives per epoch: shard sizes differ by up to one shape, so the
    # step count is the largest rank's; a rank that has run out of shapes keeps stepping on an empty batch (zero
    # gradients into the all-reduce, zero shapes into the global batch mean)
    steps_per_epoch = parallel.steps_per_epoch(flags.train_size, world, flags.batch_size)
    status = torch.zeros(4, dtype=torch.int32, device=device)       # out-of-range / NaN score counters, read once per epoch
    history = []
    lr = learning_rate(flags, global_step)
    for epoch in range(start_epoch, flags.how_many_training_epochs):
        head.train()
        tot_loss, n_seen = 0.0, 0
        it = iter(train.batches(flags.batch_size, lo, hi))
        for _step in range(steps_per_epoch):
            batch = next(it, None)
            if batch is None:
                batch = train.empty_batch()
            raw, final, y = batch
            lr = learning_rate(flags, global_step)
            for gparam in opt.param_groups:
                gparam["lr"] = lr
            opt.zero_grad(set_to_none=True)
            if overlap is not None:
                overlap.reset()
            if len(y) > 0 or (world > 1 and flags.score_reduce == "batch"):
                # literal mode on a sharded batch: every rank bins the same GLOBAL batch mean (SURVEY.md 8e (2))
                _, _, logits = head(raw, final, process_group=pg if flags.score_reduce == "batch" else None,
                                    status=status, fold_gap=flags.fold_gap,
                                    global_count=parallel.global_batch_size(flags.train_size, world, flags.batch_size, _step))
            if len(y) > 0:
                loss = torch.nn.functional.cross_entropy(logits, y)
                loss.backward()
                tot_loss += float(loss.detach()) * len(y)
                n_seen += len(y)
            if bucket is not None:                  # one flat all-reduce (utils/_train_helper.py:17-31)
                if not overlap.fired:               # no backward ran on this rank (empty batch): zeros into the sum
                    overlap.launch()
                overlap.join()
                bucket.unpack()
            opt.step()
            global_step += 1
        model.raise_for_status(status, flags.num_group)             # the reference's IndexError / ValueError, once per epoch
        # validation (train.py:319-374)
        head.eval()
        correct, cm = 0, torch.zeros((num_classes, num_classes), dtype=torch.int64)
        with torch.no_grad():
            for raw, final, y in val.batches(flags.val_batch_size):
                _, _, logits = head(raw, final, fold_gap=flags.fold_gap)        # validation runs un-sharded on every rank: local batch mean
                pred = logits.argmax(dim=1)
                correct += int((pred == y).sum())
                cm += confusion_matrix(y.cpu(), pred.cpu(), num_classes)
        acc = correct / flags.val_size
        history.append((epoch, tot_loss / max(n_seen, 1), acc))
        if rank == 0:
            print("Epoch #%d, rate %.6f, train loss %.5f, val top1_acc %.3f%%" % (epoch, lr, history[-1][1], 100 * acc))
            os.makedirs(flags.train_logdir, exist_ok=True)
            torch.save({"head": head.state_dict(), "opt": opt.state_dict(), "epoch": epoch, "global_step": global_step,
                        "flags": vars(flags)},
                       os.path.join(flags.train_logdir, "%s-%04d" % (flags.ckpt_name_to_save, epoch)))
    if rank == 0 and history:
        print("confusion matrix (last epoch):\n%s" % cm)
    main.last_head = head                              # for callers / checks that want the trained module
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return history


if __name__ == "__main__":
    main()
