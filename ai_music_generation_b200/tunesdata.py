"""ABC tune corpora for the hierarchical model: the JSON list that sample.py reads (records with "abc notation" and "id"),
encoded into bar patches, and the tune-index sampler that cuts each epoch into global batches and per-rank shards.

Both are host-side and touch no device: the training driver packs a shard with `pack_tunes` and uploads it."""
from __future__ import annotations

import json

import numpy as np

from .tunesformer import PATCH_LENGTH, Patchilizer


def load_abc_corpus(path, patch_length=PATCH_LENGTH):
    """Reads a JSON list of {"abc notation": text, "id": key} records.  Returns (keys, patch lists): a record without "id" takes
    its index in the list as key, and every patch list is
    `Patchilizer().encode(text, patch_length, add_special_patches=True)`, so a tune longer than `patch_length` patches
    (the patch-level block_size) is cut there.  A record whose text yields no patch between the start and end patches (empty
    or whitespace-only, or no bar line) is dropped, and the number dropped is printed."""
    with open(path, encoding="utf-8") as f:
        records = json.load(f)
    pz = Patchilizer()
    keys, tunes = [], []
    for i, rec in enumerate(records):
        patches = pz.encode(rec["abc notation"], patch_length=None, add_special_patches=True)
        if len(patches) <= 2:
            continue
        keys.append(rec.get("id", i))
        tunes.append(patches[:patch_length])
    dropped = len(records) - len(tunes)
    if dropped:
        print(f"{path}: dropped {dropped} of {len(records)} tunes with no bar patch")
    return keys, tunes


class TuneBatches:
    """Tune indices of one rank, batch by batch, for one epoch at a time.

    Every epoch shuffles the n_tunes indices with its own permutation, seeded by (seed, epoch), the same on every rank.  The
    permutation is cut into global batches of `batch_size` tunes, and each global batch into `world` contiguous shards of
    batch_size / world tunes; rank `rank` takes shard `rank`.  drop_last=True (training) drops the last incomplete global
    batch, so every rank holds the same number of tunes in every step and the mean over ranks of the per-rank mean loss is
    the mean over tunes.  drop_last=False (evaluation) keeps it: every tune is visited exactly once across the ranks, and a
    rank may get a short or empty last shard."""

    def __init__(self, n_tunes, batch_size, rank=0, world=1, seed=0, drop_last=True):
        if batch_size <= 0 or batch_size % world != 0:
            raise ValueError(f"batch_size ({batch_size}) must be a positive multiple of the number of ranks ({world})")
        if not 0 <= rank < world:
            raise ValueError(f"rank {rank} outside [0, {world})")
        self.n, self.batch_size, self.rank, self.world = int(n_tunes), int(batch_size), int(rank), int(world)
        self.seed, self.drop_last = int(seed), bool(drop_last)

    def __len__(self):
        """Batches per epoch (the same on every rank)."""
        return self.n // self.batch_size if self.drop_last else -(-self.n // self.batch_size)

    def epoch(self, epoch):
        """This rank's shards of the given epoch: a list of int64 index arrays, one per global batch."""
        perm = np.random.default_rng([self.seed, int(epoch)]).permutation(self.n)
        per = self.batch_size // self.world
        out = []
        for b in range(len(self)):
            batch = perm[b * self.batch_size:(b + 1) * self.batch_size]
            out.append(batch[self.rank * per:(self.rank + 1) * per])
        return out
