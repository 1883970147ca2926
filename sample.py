"""Sampling driver with the call surface of the reference's nanoGPT/sample.py, on the B200 kernels.

    python sample.py --out_dir=out-irishman-char --dataset=irishman --tokens_format=char --num_samples=16 --top_k=1

Same settings (reference sample.py:17-42), same checkpoint / meta.pkl contracts (sample.py:55-100), same prompt
construction from a validation set (first `n_conditional_measures` bars; sample.py:108-142), same output normalisation
(cut at '$', trim to the last bar line; sample.py:158-169).  Difference: prompts are decoded in batches through GPT.generate,
also when their lengths differ (prompt_lens; the reference decodes them one at a time through the same batch-generic API,
model.py:305-330).

top_p > 0 draws with TunesFormer's recipe instead of the reference's head (e.g. --top_p=0.8 --top_k=8 --temperature=1.2).
The run's random stream is `seed`, and each prompt draws from its own stream named by its index in the prompt list, so the
files do not depend on `batch` or on how the prompts are grouped.
"""
from __future__ import annotations

import json
import os
import pickle
import re
import sys

import torch

from ai_music_generation_b200 import GPT, GPTConfig
from configurator import load_settings

DEFAULTS = dict(
    dataset="music21_bach", use_validation_prefixes=True, tokens_format="midi", validation_path="",
    n_conditional_measures=4, out_dir="out", init_from="resume", start="$", num_samples=1000, max_new_tokens=500,
    temperature=0.8, top_k=200, seed=1337, device="cuda", dtype="bfloat16", compile=False,
    batch=64,          # new knob: prompts of equal length are decoded together (the reference decodes one at a time)
    early_stop=True,   # new knob: stop a batch once every tune has produced its end symbol '$' (files are cut there anyway)
    top_p=0.0,         # new knob: 0 < top_p <= 1 samples with TunesFormer's nucleus / top-k / temperature chain; 0 = off
)


def build_codec(meta, tokens_format):
    stoi, itos = meta["stoi"], meta["itos"]
    if tokens_format == "char":
        return (lambda text: [stoi[c] for c in text]), (lambda ids: "".join(itos[i] for i in ids))
    return (lambda text: [stoi[t] for t in text.split()]), (lambda ids: " ".join(itos[i] for i in ids))


def prompts_from(s):
    """(key, prompt text) pairs: the bare start symbol, or validation tunes cut after n_conditional_measures bars."""
    start = s["start"]
    if start.startswith("FILE:"):
        with open(start[5:], encoding="utf-8") as f:
            start = f.read()
    if not s["use_validation_prefixes"]:
        return [(i, start) for i in range(s["num_samples"])]
    if s["validation_path"] == "":
        raise ValueError("use_validation_prefixes is True, but validation_path was not set")
    n = s["n_conditional_measures"]
    if s["tokens_format"] == "midi":
        out = []
        for fname in sorted(os.listdir(s["validation_path"])):
            if fname.endswith(".txt"):
                with open(os.path.join(s["validation_path"], fname)) as f:
                    bars = f.read().split("|")[:n]
                out.append((fname[:-4], start + " " + "|".join(bars).strip() + " |"))
        return out
    if s["dataset"] == "irishman" and s["tokens_format"] == "char":
        with open(s["validation_path"]) as f:
            sheets = json.load(f)
        bar = re.compile(r"(:\||::|\s\||\|\])")
        return [(sh.get("id"), start + "".join(bar.split(sh.get("abc notation"))[: n * 2])) for sh in sheets]
    raise NotImplementedError("validation prefixes for this dataset / token format")


def normalise(text, key, abc):
    """sample.py:163-169: keep what follows the first '$'; ABC gets an X: header, token streams end on a bar line."""
    body = text.split("$")[1].strip() if "$" in text else text.strip()
    if abc:
        return f"X:{key}\n" + body
    if not body.endswith("|"):
        body = "|".join(text.split("|")[:-1]).strip() + " |"
    return body


def main():
    s = load_settings(DEFAULTS, sys.argv[1:])
    torch.manual_seed(s["seed"])
    torch.cuda.manual_seed(s["seed"])
    if s["init_from"] == "resume":
        ckpt = torch.load(os.path.join(s["out_dir"], "ckpt.pt"), map_location="cpu")
        model = GPT(GPTConfig(**ckpt["model_args"]))
        model.load_state_dict({k.removeprefix("_orig_mod."): v for k, v in ckpt["model"].items()})
    elif s["init_from"].startswith("gpt2"):
        ckpt = {}   # nanoGPT/sample.py:67-69: a given GPT-2 model (transformers: needs the HF cache or network access)
        model = GPT.from_pretrained(s["init_from"], dict(dropout=0.0))
    else:
        raise SystemExit(f"unknown init_from {s['init_from']!r} (resume | gpt2*)")
    model.eval().to(s["device"])

    meta_path = os.path.join("data", ckpt.get("config", {}).get("dataset", s["dataset"]), "meta.pkl")
    if not os.path.exists(meta_path):
        raise SystemExit(f"{meta_path} not found (the GPT-2 BPE fallback of the reference needs tiktoken + network)")
    print(f"Loading meta from {meta_path}...")
    with open(meta_path, "rb") as f:
        meta = pickle.load(f)
        encode, decode = build_codec(meta, s["tokens_format"])
    stop = meta["stoi"].get("$") if s["early_stop"] else None

    abc = s["tokens_format"] == "char" and s["dataset"] == "irishman"
    out_dir = os.path.join(s["out_dir"], "samples")
    os.makedirs(out_dir, exist_ok=True)
    todo = [(key, text, encode(text), i) for i, (key, text) in enumerate(prompts_from(s))]
    top_k = s["top_k"] if s["top_k"] > 0 else None
    # the nucleus head: one seed per run, each prompt's stream named by its place in prompts_from (before the sort below)
    nucleus = dict(top_p=s["top_p"], seed=s["seed"]) if s["top_p"] > 0 else {}
    block = model.config.block_size
    # prompts sorted by length and cut into batches; a batch of different lengths is decoded together (prompt_lens: rows
    # still inside their prompt are fed its tokens) as long as the longest prompt + max_new_tokens fits the context window,
    # otherwise it falls back to equal-length groups (the window slides: reference-style recompute per group)
    todo.sort(key=lambda item: len(item[2]))
    chunks = []
    for i in range(0, len(todo), s["batch"]):
        chunk = todo[i:i + s["batch"]]
        lens = [len(ids) for _, _, ids, _ in chunk]
        if len(set(lens)) == 1 or max(lens) + s["max_new_tokens"] <= block + 1:
            chunks.append(chunk)
        else:
            by_len = {}
            for item in chunk:
                by_len.setdefault(len(item[2]), []).append(item)
            chunks.extend(group for _, group in sorted(by_len.items()))
    with torch.no_grad():
        for chunk in chunks:
            lens = [len(ids) for _, _, ids, _ in chunk]
            if len(set(lens)) == 1:
                x = torch.tensor([ids for _, _, ids, _ in chunk], dtype=torch.long, device=s["device"])
                if nucleus:
                    nucleus["row_ids"] = [i for _, _, _, i in chunk]
                y = model.generate(x, s["max_new_tokens"], temperature=s["temperature"], top_k=top_k, stop_token=stop,
                                   **nucleus).tolist()
            else:
                x = torch.zeros(len(chunk), max(lens), dtype=torch.long)
                for r, (_, _, ids, _) in enumerate(chunk):
                    x[r, :len(ids)] = torch.tensor(ids, dtype=torch.long)
                if nucleus:
                    nucleus["row_ids"] = [i for _, _, _, i in chunk]
                y = model.generate(x.to(s["device"]), s["max_new_tokens"], temperature=s["temperature"], top_k=top_k,
                                   stop_token=stop, prompt_lens=lens, **nucleus).tolist()
                y = [row[:n + s["max_new_tokens"]] for row, n in zip(y, lens)]
            for (key, text, _, _), ids in zip(chunk, y):
                res = decode(ids)
                print(f"\nPrefix: {text}\nGeneration: {res}\n" + "-" * 50)
                name = f"sample_{key}.abc" if abc else f"sample_{key}.txt"
                with open(os.path.join(out_dir, name), "w") as f:
                    f.write(normalise(res, key, abc))


if __name__ == "__main__":
    main()
