"""TunesFormer training on tunes of different lengths, one B200: the packed path (TunesFormerShaped.forward(patches,
patch_counts), no pad patches) against the dense path on the same tunes padded with all-pad patches, timed alternately in
one process.  cfg4 widths: patch level 9 layers, character level 3 layers, 768-d, bias, tanh GELU.

Workload: --tunes tunes per step; patch counts uniform on [--min-patches, --max-patches] (seed --seed), and every bar patch
holds bos + 6..30 characters + eos (uniform), padded to 32, like the bars of an IrishMAN tune.  --mixes such batches are drawn
and cycled.  The padded batch of every mix has the longest tune's patch count over all mixes (one dense buffer set: the dense
path keeps one per shape).  The two paths optimise different objectives (the packed loss is the reference's mean over tunes
of each tune's token mean, the padded one a token mean over the batch); both take the same optimizer step work.

One optimizer step = forward + backward + joint clip + AdamW, timed with CUDA events over --steps steps per round, rounds
alternating packed / padded.  Prints one JSON line: ms per step (median and all rounds), real (non-pad) characters per second
(the non-pad characters of the decoded patches 1..P_i-1 of every tune, the same count for both paths), the fraction of
character-level rows that are pad patches in the padded batch, and the card name and power limit read in the same run."""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai_music_generation_b200 import GPTConfig, TunesFormerShaped, pack_tunes  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--tunes", type=int, default=64)
ap.add_argument("--min-patches", type=int, default=16)
ap.add_argument("--max-patches", type=int, default=128)
ap.add_argument("--mixes", type=int, default=8)
ap.add_argument("--steps", type=int, default=8)
ap.add_argument("--rounds", type=int, default=4)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--seed", type=int, default=0)
args = ap.parse_args()

dev = torch.device("cuda", 0)
name = torch.cuda.get_device_name(dev)
try:
    power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"

kw = dict(n_head=12, n_embd=768, dropout=0.0, bias=True, activation="gelu_tanh")
torch.manual_seed(1337)
with contextlib.redirect_stdout(io.StringIO()):
    model = TunesFormerShaped(GPTConfig(block_size=128, vocab_size=1, n_layer=9, **kw),
                              GPTConfig(block_size=32, vocab_size=128, n_layer=3, **kw)).to(dev).train()
    opt = model.configure_optimizers(0.01, 5e-5, (0.9, 0.999))

g = torch.Generator().manual_seed(args.seed)
mixes = []
for _ in range(args.mixes):
    counts = torch.randint(args.min_patches, args.max_patches + 1, (args.tunes,), generator=g).tolist()
    tunes = []
    for n in counts:
        p = torch.randint(3, 128, (n, 32), generator=g)
        lens = torch.randint(8, 33, (n,), generator=g)            # bos + 6..30 characters + eos
        p[:, 0] = 1
        p[torch.arange(n), lens - 1] = 2
        p[torch.arange(32)[None, :] >= lens[:, None]] = 0
        tunes.append(p)
    mixes.append((tunes, counts))
pmax = max(max(c) for _, c in mixes)
batches = []
for tunes, counts in mixes:
    packed, _ = pack_tunes(tunes)
    padded = torch.zeros(len(tunes), pmax, 32, dtype=torch.int64)
    for i, t in enumerate(tunes):
        padded[i, :t.shape[0]] = t
    real = sum(int((t[1:] != 0).sum()) for t in tunes)
    batches.append((packed.to(dev), counts, padded.to(dev), real))


def step(kind, b):
    packed, counts, padded, _ = b
    loss = model(packed, counts) if kind == "packed" else model(padded)
    opt.zero_grad(set_to_none=True)
    loss.backward()
    model.clip_grad_norm_(1.0)
    opt.step()
    return loss


for kind in ("packed", "padded"):
    for i in range(args.warmup):
        step(kind, batches[i % len(batches)])
torch.cuda.synchronize()
times = {"packed": [], "padded": []}
losses = {}
k = 0
for r in range(args.rounds):
    for kind in ("packed", "padded") if r % 2 == 0 else ("padded", "packed"):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            loss = step(kind, batches[(k + i) % len(batches)])
        e1.record()
        torch.cuda.synchronize()
        times[kind].append(e0.elapsed_time(e1) / args.steps)
        losses[kind] = loss.item()
    k += args.steps
real = statistics.mean(b[3] for b in batches)
decoded = statistics.mean(sum(c) - len(c) for _, c, _, _ in batches)
pad_patch_frac = 1.0 - decoded / (args.tunes * (pmax - 1))
ms = {kind: statistics.median(v) for kind, v in times.items()}
print(json.dumps({
    "gpu": name, "power_limit": power,
    "workload": f"TunesFormer cfg4 widths (9L patch + 3L char, 768d), {args.tunes} tunes/step, patch counts uniform "
                f"[{args.min_patches}, {args.max_patches}] seed {args.seed}, {args.mixes} mixes, padded to {pmax} patches",
    "ms_per_step": ms, "ms_per_step_rounds": times,
    "real_chars_per_s": {kind: real / v * 1e3 for kind, v in ms.items()},
    "speedup_packed_over_padded": ms["padded"] / ms["packed"],
    "pad_patch_fraction_of_char_rows": pad_patch_frac,
    "real_chars_per_step": real, "decoded_patches_per_step": decoded, "last_loss": losses,
}))
