"""Generation driver for the hierarchical (TunesFormer-shaped) model, on the B200 kernels.

    python generate_tunesformer.py --out_dir=out-tunesformer-irishman --num_samples=64
    python generate_tunesformer.py --out_dir=out-tunesformer-irishman --validation_path=data/irishman/validation.json
    torchrun --standalone --nproc_per_node=8 generate_tunesformer.py --out_dir=... --validation_path=...

Weights: `weights` (default out_dir/weights.pth), either what train_tunesformer.py writes or any state dict in the reference
TunesFormer's layout, bare or under a "model" key, loaded through TunesFormerShaped.load_reference_state_dict.  Without
model_args beside it the shape is read from the tensors, except n_head, which is a setting.
Prompts: `num_samples` copies of `start` ("" = the start patch only), or, with `validation_path` set, every tune of that JSON
file cut after its header patches and `n_conditional_bars` bar patches.  All prompts go through
TunesFormerShaped.generate_tunes (nucleus / top-k / temperature sampling on the device) with the integer `seed`; a tune's
random stream is keyed by its index in the whole prompt list, so under torchrun, where every rank takes a contiguous slice of
the prompts, the files do not depend on the number of GPUs.  Output: out_dir/samples/tunesformer_{key}.abc per prompt.
"""
from __future__ import annotations

import os
import re
import sys

import torch

from ai_music_generation_b200 import GPTConfig, Patchilizer, TunesFormerShaped
from ai_music_generation_b200.tunesdata import load_abc_corpus
from ai_music_generation_b200.tunesformer import CHAR_VOCAB
from configurator import load_settings

DEFAULTS = dict(
    out_dir="out-tunesformer", weights="",   # "" = out_dir/weights.pth
    num_samples=1, start="",
    validation_path="", n_conditional_bars=0,
    max_patch=0,        # 0 = the patch decoder's block_size
    top_p=0.8, top_k=8, temperature=1.2, seed=0,
    batch=64,           # tunes that share one pass of the decode loop
    n_head=12,          # for a bare state dict: the head count is not visible in the tensors
    device="cuda",
)


def model_args_from_state_dict(sd, n_head):
    """Shape of a reference-layout TunesFormer state dict: layers, width and block sizes from the tensors."""
    def level(prefix):
        n_layer = len({int(m.group(1)) for k in sd for m in [re.match(re.escape(prefix) + r"h\.(\d+)\.", k)] if m})
        wpe = sd[prefix + "wpe.weight"]
        return dict(n_layer=n_layer, n_head=n_head, n_embd=wpe.shape[1], block_size=wpe.shape[0], dropout=0.0,
                    bias=prefix + "h.0.attn.c_attn.bias" in sd, activation="gelu_tanh")
    patch, char = level("patch_level_decoder.base."), level("char_level_decoder.base.transformer.")
    patch["vocab_size"] = sd["patch_level_decoder.base.wte.weight"].shape[0]
    char["vocab_size"] = CHAR_VOCAB
    return {"patch": patch, "char": char}


def load_model(path, n_head, device):
    ckpt = torch.load(path, map_location="cpu")
    sd = ckpt["model"] if "model" in ckpt else ckpt
    args = ckpt.get("model_args") or model_args_from_state_dict(sd, n_head)
    args = {lvl: {**a, "dropout": 0.0} for lvl, a in args.items()}
    model = TunesFormerShaped(GPTConfig(**args["patch"]), GPTConfig(**args["char"]))
    model.load_reference_state_dict(sd)
    return model.to(device).eval()


def conditional_prompts(path, n_bars):
    """(key, prompt text) per tune of a JSON corpus: its header patches and the first n_bars bar patches, decoded."""
    pz = Patchilizer()
    keys, tunes = load_abc_corpus(path, patch_length=None)
    out = []
    for key, patches in zip(keys, tunes):
        body = patches[1:-1]   # without the start and end patches
        n_head = 0
        while n_head < len(body) and Patchilizer.is_header(pz.patch2bar(body[n_head])):
            n_head += 1
        out.append((key, pz.decode(body[:n_head + n_bars])))
    return out


def main():
    s = load_settings(DEFAULTS, sys.argv[1:])
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    device = s["device"]
    if "LOCAL_RANK" in os.environ:
        device = f"cuda:{os.environ['LOCAL_RANK']}"
        torch.cuda.set_device(device)   # the kernels launch on the current device's stream
    if "cuda" not in device:
        raise SystemExit("generate_tunesformer.py: the sm_100a path needs a CUDA device")
    model = load_model(s["weights"] or os.path.join(s["out_dir"], "weights.pth"), s["n_head"], device)
    if s["validation_path"]:
        prompts = conditional_prompts(s["validation_path"], s["n_conditional_bars"])
    else:
        prompts = [(i, s["start"]) for i in range(s["num_samples"])]
    seen = set()
    for key, _ in prompts:   # the key names the output file
        if str(key) in seen:
            raise SystemExit(f"two prompts share the key {key!r}: their output files would overwrite each other")
        seen.add(str(key))
    max_patch = s["max_patch"] or model.patch_level_decoder.config.block_size
    per = -(-len(prompts) // world)
    ids = list(range(rank * per, min(len(prompts), (rank + 1) * per)))
    tunes = model.generate_tunes([prompts[i][1] for i in ids], max_patch=max_patch, top_p=s["top_p"], top_k=s["top_k"],
                                 temperature=s["temperature"], seed=s["seed"], batch=s["batch"], tune_ids=ids)
    out_dir = os.path.join(s["out_dir"], "samples")
    os.makedirs(out_dir, exist_ok=True)
    for i, tune in zip(ids, tunes):
        with open(os.path.join(out_dir, f"tunesformer_{prompts[i][0]}.abc"), "w", encoding="utf-8") as f:
            f.write(tune)
    print(f"rank {rank}: wrote {len(ids)} tunes to {out_dir}")


if __name__ == "__main__":
    main()
