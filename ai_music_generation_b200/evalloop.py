"""`estimate_loss` of the reference (nanoGPT/train.py:231-244, called at :290-291), rank-sharded (SURVEY.md 8f N4).

The reference evaluates `eval_iters` batches of each split on rank 0 while the other ranks wait at the next collective,
with one `loss.item()` host sync per batch.  Here every rank evaluates ceil(eval_iters / world) batches, the per-rank sums
stay on the device and ONE all-reduce per split combines them (one host sync per split).  With world == 1, or
`shard=False`, it is the reference's loop: `eval_iters` batches on the calling rank, plain mean.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


@torch.no_grad()
def estimate_loss(model, get_batch, eval_iters, device, *, shard=False, group=None, splits=("train", "val")):
    """model(X, Y) -> (logits, loss); get_batch(split) -> (X, Y).  Returns {split: 0-d CPU tensor}, like the reference.

    shard=True: the mean runs over world * ceil(eval_iters / world) batches (every rank draws its own), so with eval_iters a
    multiple of the world size exactly eval_iters batches are evaluated, as in the reference."""
    world = dist.get_world_size(group) if (shard and dist.is_initialized()) else 1
    n_local = -(-eval_iters // world)
    was_training = model.training
    model.eval()
    out = {}
    for split in splits:
        acc = torch.zeros(1, device=device, dtype=torch.float32)
        for _ in range(n_local):
            X, Y = get_batch(split)
            _, loss = model(X, Y)
            acc += loss.detach().float().reshape(1)
        if world > 1:
            dist.all_reduce(acc, group=group)
        out[split] = (acc / (n_local * world)).cpu()[0]
    model.train(was_training)
    return out


@torch.no_grad()
def estimate_tunes_loss(model, batches, device, group=None):
    """Mean loss over every evaluated tune of the hierarchical model: sum_b loss_b * n_b / sum_b n_b, where batch b holds n_b
    tunes and loss_b is the packed forward's mean over them.  `batches` yields (patches, patch_counts) of this rank, in the
    layout of `TunesFormerShaped.forward(patches, patch_counts)`; an empty shard is skipped.  Always without patch sampling.
    The per-rank sums stay on the device, ranks are combined with one all-reduce of the two scalars, and the call
    synchronises with the host once.  Returns a float (nan when no rank evaluated a tune)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    was_training = model.training
    model.eval()
    acc = torch.zeros(2, device=device, dtype=torch.float32)
    for patches, counts in batches:
        if len(counts) == 0:
            continue
        loss = model(patches, counts)
        acc[0] += loss.detach().float() * len(counts)
        acc[1] += len(counts)
    if world > 1:
        dist.all_reduce(acc, group=group)
    model.train(was_training)
    total, n = acc.cpu().tolist()
    return total / n if n > 0 else float("nan")
