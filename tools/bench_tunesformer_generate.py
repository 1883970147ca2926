"""TunesFormer generation on one GPU: the batched device loop (TunesFormerShaped.generate_tunes) against the host-driven
loop (generate_tune, one prompt at a time).  Results: profiles/r5_tunesformer_generate.md.

Shape: full size (patch level 9 layers, character level 3 layers, 768 wide, 12 heads, biases, tanh GELU, patch block 128,
character block 32), seeded random weights.

  sampled   prompts of a few header patches plus 0-2 bars, the reference's defaults (top_p 0.8, top_k 8, temperature 1.2),
            max_patch 128; at random init eos is rare, so tunes run close to max_patch.  1, 16, 64 and 256 tunes (256 as
            four batches of 64).
  old loop  generate_tune per prompt on a handful of prompts with a small max_patch: time per generated character.
  greedy    both loops with top_k = 1 on the same prompts and max_patch; the character embedding (tied head) is scaled up so
            that the argmax decisions survive bf16 rounding, and the texts must be identical: the time ratio then compares
            equal work.

Every shape is run once before it is timed; times are host clocks closed by a device synchronise.  Prints one JSON line per
measurement, with the card's name and power limit read in the same process.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai_music_generation_b200 import GPTConfig, TunesFormerShaped, ops  # noqa: E402

HEADERS = ["L:1/8", "M:3/4", "M:4/4", "M:6/8", "K:D", "K:G", "K:Ador", "R:reel", "T:tune"]
BARS = ["|: A2 B2 c2 |", " dcBA GFED |", " E2 F G2 A |", " f2 ed cBAG |", " d3 e fga |"]


def prompts(n, seed=0):
    rng = random.Random(seed)
    out = []
    for i in range(n):
        heads = [f"X:{i + 1}"] + rng.sample(HEADERS, rng.randint(2, 4))
        out.append("\n".join(heads) + "\n" + "".join(rng.choice(BARS) for _ in range(rng.randint(0, 2))))
    return out


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # noqa: BLE001 - the numbers are still printed, marked as such
        q = f"unavailable ({e})"
    return name, q


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def new_chars(texts, ps):
    return sum(len(t) - len(p) for t, p in zip(texts, ps))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,16,64,256")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--max-patch", type=int, default=128)
    ap.add_argument("--old-prompts", type=int, default=4)
    ap.add_argument("--old-max-patch", type=int, default=12)
    args = ap.parse_args()
    name, power = card()
    base = {"gpu": name, "power_limit_W, max_sm_clock": power}
    torch.manual_seed(1337)
    pc = GPTConfig(block_size=128, vocab_size=1, n_layer=9, n_head=12, n_embd=768, dropout=0.0, bias=True, activation="gelu_tanh")
    cc = GPTConfig(block_size=32, vocab_size=128, n_layer=3, n_head=12, n_embd=768, dropout=0.0, bias=True, activation="gelu_tanh")
    model = TunesFormerShaped(pc, cc).cuda().eval()
    kw = dict(top_p=0.8, top_k=8, temperature=1.2)

    # ---- sampled arm: the batched device loop
    sizes = [int(s) for s in args.sizes.split(",")]
    for n in sizes:
        ps = prompts(n, seed=n)
        model.generate_tunes(ps, max_patch=8, seed=1, batch=args.batch, **kw)   # warm-up: records every launch list
        texts, dt = timed(lambda: model.generate_tunes(ps, max_patch=args.max_patch, seed=2, batch=args.batch, **kw))
        st = model.last_generate_stats
        chars = new_chars(texts, ps)
        print(json.dumps({**base, "arm": "sampled, device loop", "tunes": n, "batch": args.batch, "max_patch": args.max_patch,
                          "seconds": round(dt, 4), "tunes_per_s": round(n / dt, 3), "chars_per_s": round(chars / dt, 1),
                          "generated_chars": chars, "bars": st["bars"], "ms_per_bar": round(dt / st["bars"] * 1e3, 4),
                          "host_syncs_per_bar": round(st["host_syncs"] / st["bars"], 3),
                          "launches_per_char_step": round(st["char_launches"] / st["char_steps"], 2),
                          "c_calls_per_char_step": round(st["char_calls"] / st["char_steps"], 3),
                          "launches_total": st["launches"]}), flush=True)

    # ---- the host-driven loop, one prompt at a time, against the device loop on the same prompts
    ps = prompts(args.old_prompts, seed=99)
    model.generate_tune(ps[0], max_patch=6, **kw)
    old, dt_old = timed(lambda: [model.generate_tune(p, max_patch=args.old_max_patch, seed=3, **kw) for p in ps])
    model.generate_tunes(ps, max_patch=6, seed=1, **kw)
    new, dt_new = timed(lambda: model.generate_tunes(ps, max_patch=args.old_max_patch, seed=3, **kw))
    c_old, c_new = new_chars(old, ps), new_chars(new, ps)
    print(json.dumps({**base, "arm": "sampled, host loop vs device loop", "tunes": len(ps), "max_patch": args.old_max_patch,
                      "old_seconds": round(dt_old, 4), "old_ms_per_char": round(dt_old / c_old * 1e3, 4),
                      "old_tunes_per_s": round(len(ps) / dt_old, 4),
                      "new_seconds": round(dt_new, 4), "new_ms_per_char": round(dt_new / c_new * 1e3, 5),
                      "new_tunes_per_s": round(len(ps) / dt_new, 4),
                      "ms_per_char_ratio": round((dt_old / c_old) / (dt_new / c_new), 1)}), flush=True)

    # ---- greedy arm: identical texts, so the time ratio compares equal work
    cd = model.char_level_decoder
    with torch.no_grad():
        cd.transformer.wte.weight.mul_(40.0)   # tied with lm_head: sharper logits, argmax decisions that survive bf16
    gkw = dict(top_p=0.8, top_k=1, temperature=1.2)
    model.generate_tune(ps[0], max_patch=6, **gkw)
    old, dt_old = timed(lambda: [model.generate_tune(p, max_patch=args.old_max_patch, **gkw) for p in ps])
    model.generate_tunes(ps, max_patch=6, **gkw)
    new, dt_new = timed(lambda: model.generate_tunes(ps, max_patch=args.old_max_patch, **gkw))
    c_old = new_chars(old, ps)
    print(json.dumps({**base, "arm": "greedy, host loop vs device loop", "tunes": len(ps), "max_patch": args.old_max_patch,
                      "identical_texts": sum(a == b for a, b in zip(old, new)), "generated_chars": c_old,
                      "old_seconds": round(dt_old, 4), "new_seconds": round(dt_new, 4),
                      "time_ratio": round(dt_old / dt_new, 1)}), flush=True)
    print(json.dumps({**base, "launches_counter": ops.LAUNCHES}), flush=True)


if __name__ == "__main__":
    main()
