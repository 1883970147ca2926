"""Nucleus sampling for every vocabulary: the cluster kernel against the top-k head, and generate() with the nucleus head at
the whitespace-model shape.  Source of profiles/r8_nucleus.md.

    python tools/bench_nucleus.py [--quick]

Prints one JSON line per measurement and the GPU name / power limit of the run (both are part of every number).
  * sampler launch alone (CUDA events over 200 back-to-back launches after warm-up, median of 5 such windows) at
    B in {1, 64} and V in {1024, 50 257, 98 465, 786 432}: abcgpt_sample_top_p_cluster (top_p 0.8, top_k 8, temperature 1.2),
    abcgpt_sample_top_p at V = 1024, and abcgpt_sample_topk (temperature 0.8, top_k 200) at the same shapes.  The logits
    (at most 100 MB) stay in L2 across launches, as they do in generate(), where the lm_head GEMM has just written them;
  * generate() of 256 new tokens for B = 64 on the whitespace-shaped model (6 layers, 6 heads, n_embd 384, block 256,
    V = 98 465, KV cache): the nucleus head (top_p 0.8, top_k 8, temperature 1.2) against sample.py's default head
    (temperature 0.8, top_k 200) and greedy, alternated over 5 rounds;
  * the nucleus launch's share of a decode step: sampler time at B = 64 over the measured nucleus-head step time.
"""
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai_music_generation_b200 import GPT, GPTConfig, ops  # noqa: E402
from tools.bench_large_vocab import gpu_info, timed  # noqa: E402

QUICK = "--quick" in sys.argv
V_WS = 98465
CFG = dict(block_size=256, vocab_size=V_WS, n_layer=6, n_head=6, n_embd=384, dropout=0.0, bias=False)
NUCLEUS = dict(top_p=0.8, top_k=8, temperature=1.2)


def bench_sampler():
    res = {}
    seed = torch.tensor([1234], device="cuda", dtype=torch.int64)
    base = torch.tensor([1], device="cuda", dtype=torch.int64)
    for V in (1024, 50257, V_WS, 786432):
        Vpad = (V + 7) // 8 * 8
        for B in (1, 64):
            g = torch.Generator(device="cuda").manual_seed(B)
            logits = (torch.randn(B, Vpad, device="cuda", generator=g) * 3.0).bfloat16()
            out = torch.empty(B, dtype=torch.int64, device="cuda")
            runs = [("sample_top_p_cluster", lambda: ops.sample_top_p_cluster(logits, V, out, 0.8, 8, 1.2, seed, base, 7)),
                    ("sample_topk", lambda: ops.sample_topk(logits, V, out, 0.8, 200, seed, 7))]
            if V <= 1024:
                runs.append(("sample_top_p", lambda: ops.sample_top_p(logits, V, out, 0.8, 8, 1.2, seed, base, 7)))
            for name, fn in runs:
                ms = timed(fn, reps=3 if QUICK else 5)
                res[(name, V, B)] = ms
                print(json.dumps({"bench": name, "V": V, "B": B, "us": round(ms * 1e3, 2)}), flush=True)
            del logits
    return res


def bench_generate(B=64, N=256):
    torch.manual_seed(1337)
    model = GPT(GPTConfig(**CFG)).cuda().eval()
    x = torch.zeros(B, 1, dtype=torch.long, device="cuda")
    heads = {"nucleus_p0.8_k8_t1.2": dict(NUCLEUS, seed=5), "topk200_t0.8": dict(temperature=0.8, top_k=200),
             "greedy": dict(top_k=1)}
    for kw in heads.values():
        model.generate(x, 8, **kw)   # builds the decode state and the replay programs
    times = {name: [] for name in heads}
    for _ in range(2 if QUICK else 5):
        for name, kw in heads.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.generate(x, N, **kw)
            torch.cuda.synchronize()
            times[name].append(time.perf_counter() - t0)
    res = {}
    for name, ts in times.items():
        dt = statistics.median(ts)
        res[name] = dt / N * 1e3
        print(json.dumps({"bench": "generate", **{k: CFG[k] for k in ("n_layer", "n_head", "n_embd", "block_size")}, "V": V_WS,
                          "B": B, "new_tokens": N, "head": name, "ms_per_token_step": round(dt / N * 1e3, 4),
                          "spread_ms_per_token": round((max(ts) - min(ts)) / N * 1e3, 4)}), flush=True)
    del model
    torch.cuda.empty_cache()
    return res


def main():
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    k = bench_sampler()
    g = bench_generate()
    us = k[("sample_top_p_cluster", V_WS, 64)] * 1e3
    step = g["nucleus_p0.8_k8_t1.2"] * 1e3
    print(json.dumps({"bench": "nucleus_share_of_decode_step", "sampler_us": round(us, 2), "step_us": round(step, 1),
                      "share": round(us / step, 4),
                      "step_minus_topk_head_us": round(step - g["topk200_t0.8"] * 1e3, 1)}), flush=True)
    print(json.dumps({"gpu_after": gpu_info()}), flush=True)


if __name__ == "__main__":
    main()
