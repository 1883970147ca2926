"""Training driver for the hierarchical (TunesFormer-shaped) model on a corpus of ABC tunes, on the B200 kernels.

    python train_tunesformer.py config/tunesformer_irishman.py --batch_size=64
    torchrun --standalone --nproc_per_node=8 train_tunesformer.py config/tunesformer_irishman.py

Settings: the DEFAULTS below, an optional config file and --key=value overrides (configurator.load_settings, as train.py).
Data: `train_data` / `eval_data` are JSON lists of {"abc notation", "id"} records (the format sample.py reads), encoded into
bar patches by tunesdata.load_abc_corpus.  What follows the reference's TunesFormer trainer (SURVEY.md section 2 row 9):
AdamW at lr 5e-5, a cosine schedule with linear warm-up (transformers' get_cosine_schedule_with_warmup, written out in
cosine_lr), evaluation after every epoch, and the best-eval checkpoint saved as `out_dir/weights.pth` whose "model" entry is
the reference's state dict layout.  Everything else is a knob of this driver with the default documented at DEFAULTS.

Each step packs `batch_size` tunes (global; batch_size / world per rank) without pad patches and runs forward, backward,
one global clip_grad_norm_, AdamW and zero_grad; under torchrun the model is wrapped in TunesFormerDDP.  Each epoch ends
with tunes-weighted evaluation (evalloop.estimate_tunes_loss) and one JSON line in `out_dir/logs.jsonl`: epoch, optimizer
steps so far, train loss (mean of the epoch's step losses), eval loss, the lr of the epoch's last step, ms per step and
characters per second.  Both rates cover the epoch's steps up to its one host sync, without evaluation or checkpointing; the
characters are the non-pad codes of every tune's patches 1..P-1, counted before patch sampling.

weights.pth holds the best-eval epoch only, so init_from=resume continues after that epoch, at its schedule step; the records
of any later epochs of the interrupted run are dropped from logs.jsonl, which then describes the run being continued.
"""
from __future__ import annotations

import json
import math
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

from ai_music_generation_b200 import GPTConfig, TunesFormerDDP, TunesFormerShaped, pack_tunes
from ai_music_generation_b200 import evalloop
from ai_music_generation_b200.tunesdata import TuneBatches, load_abc_corpus
from ai_music_generation_b200.tunesformer import CHAR_VOCAB, PATCH_SIZE
from configurator import load_settings

DEFAULTS = dict(
    train_data="data/tunesformer/train.json", eval_data="data/tunesformer/validation.json", out_dir="out-tunesformer",
    num_epochs=32,
    batch_size=8,                  # tunes per optimizer step, over all ranks (the reference: one tune per GPU)
    learning_rate=5e-5,            # the reference's
    weight_decay=0.01, beta1=0.9, beta2=0.999,   # torch.optim.AdamW's defaults; decay applies to the >= 2-D tensors only
    grad_clip=1.0,                 # 0 = no clipping
    warmup_steps=1000,             # optimizer steps of the linear warm-up
    patch_sampling_batch_size=0,   # > 0: decode only this many patches of each longer tune per step (TunesFormerShaped.forward)
    init_from="scratch",           # scratch | resume (out_dir/weights.pth)
    seed=0,                        # weights, the per-epoch tune order and the patch sampling
    dropout=0.0,                   # the packed path has no dropout: > 0 stops at the first step
    # model shape: config/tunesformer_irishman.py holds the full-size one
    patch_num_layers=9, char_num_layers=3, n_embd=768, n_head=12, patch_block_size=128, bias=True, activation="gelu_tanh",
    backend="nccl", device="cuda",
)


def cosine_lr(step, learning_rate, warmup_steps, total_steps):
    """lr of optimizer step `step` (0-based) under transformers.get_cosine_schedule_with_warmup: a linear ramp from 0 over
    warmup_steps, then 0.5 * (1 + cos(pi * progress)) down to 0 at total_steps."""
    if step < warmup_steps:
        return learning_rate * step / max(1, warmup_steps)
    progress = (step - warmup_steps) / max(1, total_steps - warmup_steps)
    return learning_rate * max(0.0, 0.5 * (1.0 + math.cos(math.pi * progress)))


def model_args_from(s):
    common = dict(n_head=s["n_head"], n_embd=s["n_embd"], dropout=s["dropout"], bias=s["bias"], activation=s["activation"])
    return {"patch": dict(n_layer=s["patch_num_layers"], block_size=s["patch_block_size"], vocab_size=1, **common),
            "char": dict(n_layer=s["char_num_layers"], block_size=PATCH_SIZE, vocab_size=CHAR_VOCAB, **common)}


def build_model(model_args, device, checkpoint=None):
    """The model (on `device`) and its optimizer settings come from model_args; a checkpoint's "model" entry (reference layout)
    is loaded through load_reference_state_dict."""
    model = TunesFormerShaped(GPTConfig(**model_args["patch"]), GPTConfig(**model_args["char"]))
    if checkpoint is not None:
        model.load_reference_state_dict(checkpoint["model"])
    return model.to(device).train()


def restore(out_dir, s, device):
    """init_from=resume: (model, optimizer, checkpoint, model_args), the model and optimizer holding the parameters and AdamW
    moments of out_dir/weights.pth.  The shape comes from the checkpoint's model_args, except dropout, which is this run's
    setting."""
    checkpoint = torch.load(os.path.join(out_dir, "weights.pth"), map_location="cpu")
    model_args = {lvl: {**a, "dropout": s["dropout"]} for lvl, a in checkpoint["model_args"].items()}
    model = build_model(model_args, device, checkpoint)
    optimizer = model.configure_optimizers(s["weight_decay"], s["learning_rate"], (s["beta1"], s["beta2"]))
    optimizer.load_state_dict(checkpoint["optimizer"])
    return model, optimizer, checkpoint, model_args


def decoded_chars(tune):
    """Non-pad characters of the patches the character level decodes (1..P-1): the characters/s numerator."""
    return int(np.count_nonzero(np.asarray(tune[1:])))


def main():
    s = load_settings(DEFAULTS, sys.argv[1:])
    config = {k: v for k, v in s.items() if isinstance(v, (int, float, bool, str))}
    if s["init_from"] not in ("scratch", "resume"):
        raise SystemExit(f"unknown init_from {s['init_from']!r} (scratch | resume)")
    ddp = int(os.environ.get("RANK", -1)) != -1
    if ddp:
        dist.init_process_group(backend=s["backend"])
        rank, local_rank, world = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
        device = f"cuda:{local_rank}"
        torch.cuda.set_device(device)
    else:
        rank, world, device = 0, 1, s["device"]
    master = rank == 0
    if "cuda" not in device:
        raise SystemExit("train_tunesformer.py: the sm_100a path needs a CUDA device")
    out_dir = s["out_dir"]
    if master:
        os.makedirs(out_dir, exist_ok=True)
    torch.manual_seed(s["seed"])

    if s["init_from"] == "resume":
        print(f"Resuming training from {out_dir}")
        model, optimizer, checkpoint, model_args = restore(out_dir, s, device)
        start_epoch = checkpoint["epoch"] + 1
        best_epoch, min_eval_loss = checkpoint["best_epoch"], checkpoint["min_eval_loss"]
        checkpoint = None
        log_path = os.path.join(out_dir, "logs.jsonl")
        if master and os.path.exists(log_path):   # epochs after the saved one are trained again
            with open(log_path) as f:
                kept = [line for line in f if line.strip() and json.loads(line)["epoch"] < start_epoch]
            with open(log_path, "w") as f:
                f.writelines(kept)
    else:
        model_args = model_args_from(s)
        model = build_model(model_args, device)
        optimizer = model.configure_optimizers(s["weight_decay"], s["learning_rate"], (s["beta1"], s["beta2"]))
        start_epoch, best_epoch, min_eval_loss = 1, 0, float("inf")
    raw = model
    if ddp:
        model = TunesFormerDDP(model)

    block = model_args["patch"]["block_size"]
    _, train_tunes = load_abc_corpus(s["train_data"], patch_length=block)
    _, eval_tunes = load_abc_corpus(s["eval_data"], patch_length=block)
    # uint8 per tune: pack_tunes widens a batch to int64 on the host, then one pinned copy goes up
    train_tunes = [torch.tensor(t, dtype=torch.uint8) for t in train_tunes]
    eval_tunes = [torch.tensor(t, dtype=torch.uint8) for t in eval_tunes]
    train_chars = np.array([decoded_chars(t) for t in train_tunes], dtype=np.int64)
    train_batches = TuneBatches(len(train_tunes), s["batch_size"], rank, world, s["seed"], drop_last=True)
    eval_batches = TuneBatches(len(eval_tunes), s["batch_size"], rank, world, s["seed"], drop_last=False)
    steps_per_epoch = len(train_batches)
    if steps_per_epoch == 0:
        raise SystemExit(f"{len(train_tunes)} training tunes make no batch of {s['batch_size']}")
    total_steps = s["num_epochs"] * steps_per_epoch
    print(f"{len(train_tunes)} training tunes, {len(eval_tunes)} evaluation tunes, {steps_per_epoch} steps per epoch, "
          f"{world} rank(s)")

    def upload(tunes, ix):
        patches, counts = pack_tunes([tunes[i] for i in ix])
        return patches.pin_memory().to(device, non_blocking=True), counts

    def eval_loss():
        shards = eval_batches.epoch(0)
        return evalloop.estimate_tunes_loss(raw, (upload(eval_tunes, ix) if len(ix) else (None, []) for ix in shards), device)

    log_path = os.path.join(out_dir, "logs.jsonl")
    step = (start_epoch - 1) * steps_per_epoch
    for epoch in range(start_epoch, s["num_epochs"] + 1):
        shards = train_batches.epoch(epoch)
        gen = torch.Generator().manual_seed(int(np.random.SeedSequence([s["seed"], epoch, rank]).generate_state(1)[0]))
        acc = torch.zeros(2, device=device, dtype=torch.float32)   # loss sum, characters before patch sampling (this rank)
        chars = int(sum(int(train_chars[shard].sum()) for shard in shards))
        acc[1] = chars
        t0 = time.time()
        batch = upload(train_tunes, shards[0])
        for b in range(steps_per_epoch):
            lr = cosine_lr(step, s["learning_rate"], s["warmup_steps"], total_steps)
            for group in optimizer.param_groups:
                group["lr"] = lr
            loss = model(*batch, patch_sampling=s["patch_sampling_batch_size"], generator=gen)
            if b + 1 < steps_per_epoch:
                batch = upload(train_tunes, shards[b + 1])   # host work overlaps the asynchronous step
            loss.backward()
            if s["grad_clip"] != 0.0:
                raw.clip_grad_norm_(s["grad_clip"])
            optimizer.step()
            optimizer.zero_grad(set_to_none=True)
            acc[0] += loss.detach()
            step += 1
        if ddp:
            dist.all_reduce(acc)
        train_loss, chars = acc.tolist()   # the epoch's one host sync
        dt = time.time() - t0
        train_loss /= steps_per_epoch * world
        ev = eval_loss()
        rec = {"epoch": epoch, "step": step, "train_loss": train_loss, "eval_loss": ev, "lr": lr,
               "ms_per_step": dt * 1e3 / steps_per_epoch, "chars_per_s": chars / dt}
        print(json.dumps(rec))
        if master:
            with open(log_path, "a") as f:
                f.write(json.dumps(rec) + "\n")
        if ev < min_eval_loss:
            min_eval_loss, best_epoch = ev, epoch   # every rank holds the same all-reduced eval loss
            if master:
                checkpoint = {"model": raw.reference_state_dict(), "optimizer": optimizer.state_dict(), "epoch": epoch,
                              "best_epoch": best_epoch, "min_eval_loss": min_eval_loss, "model_args": model_args,
                              "config": config}
                torch.save(checkpoint, os.path.join(out_dir, "weights.pth"))
                print(f"saved {os.path.join(out_dir, 'weights.pth')} (epoch {epoch}, eval loss {ev:.4f})")
                checkpoint = None
    if ddp:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
