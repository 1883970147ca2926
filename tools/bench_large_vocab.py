"""Large vocabularies (V = 98 465, the whitespace-tokenised irishman corpus): the sampling head, generate() and the training
step.  Source of profiles/r4_large_vocab.md.

    python tools/bench_large_vocab.py [--quick]

Prints one JSON line per measurement and the GPU name / power limit of the run (both are part of every number).
  * sampler launch alone (CUDA events over >= 200 back-to-back launches after warm-up, median of 5 such windows) at
    B in {1, 64, 256}: V = 98 465 (cluster kernel, top_k 200 and None), V = 50 304 (one-CTA kernel, for reference), and
    argmax at the same shapes.  The logits (at most 50 MB) stay in L2 across launches, as they do in generate(), where the
    lm_head GEMM has just written them;
  * generate() of 255 new tokens for B = 64 on the whitespace-shaped model (6 layers, 6 heads, n_embd 384, block 256,
    V = 98 465, KV cache, one-call compiled decode replay): greedy, and temperature 0.8 / top_k 200;
  * the sampling launch's share of a top-k decode step: sampler time at B = 64 over the measured decode step time;
  * the training step at B = 64, T = 256 of the same model (forward + backward + clip + AdamW), and, from a separate
    instrumented pass (every C-ABI call bracketed by CUDA events), the time of the lm_head GEMMs (the GEMMs with a Vpad
    operand dimension) and of the cross-entropy kernels.  Weight-gradient GEMMs run on a second stream, so the shares are
    of the summed call times, not of the wall-clock step.
"""
import json
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai_music_generation_b200 import GPT, GPTConfig, ops  # noqa: E402

QUICK = "--quick" in sys.argv
V_WS = 98465
CFG = dict(block_size=256, vocab_size=V_WS, n_layer=6, n_head=6, n_embd=384, dropout=0.0, bias=False)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        pl, clk = [s.strip() for s in out.split(",")]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(clk))
    except Exception as e:  # noqa: BLE001
        info["power_limit_w"] = f"unavailable ({type(e).__name__})"
    return info


def timed(fn, reps=5, iters=200, warmup=20):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / iters)
    return statistics.median(out)


def bench_sampler():
    res = {}
    seed = torch.tensor([1234], device="cuda", dtype=torch.int64)
    for V in (V_WS, 50304):
        Vpad = (V + 7) // 8 * 8
        for B in (1, 64, 256):
            g = torch.Generator(device="cuda").manual_seed(B)
            logits = (torch.randn(B, Vpad, device="cuda", generator=g) * 3.0).bfloat16()
            out = torch.empty(B, dtype=torch.int64, device="cuda")
            for top_k in (200, None):
                ms = timed(lambda: ops.sample_topk(logits, V, out, 0.8, top_k, seed, 7))
                res[(V, B, top_k)] = ms
                print(json.dumps({"bench": "sample_topk", "V": V, "B": B, "top_k": top_k,
                                  "kernel": "cluster" if V * 4 > 220 * 1024 else "one_cta", "us": round(ms * 1e3, 2)}),
                      flush=True)
            ms = timed(lambda: ops.argmax(logits, V, out))
            print(json.dumps({"bench": "argmax", "V": V, "B": B, "us": round(ms * 1e3, 2)}), flush=True)
            del logits
    return res


def bench_generate(B=64, N=255):
    torch.manual_seed(1337)
    model = GPT(GPTConfig(**CFG)).cuda().eval()
    x = torch.zeros(B, 1, dtype=torch.long, device="cuda")
    res = {}
    for name, kw in (("greedy", dict(top_k=1)), ("topk200_t0.8", dict(temperature=0.8, top_k=200))):
        model.generate(x, 8, **kw)   # builds the decode state and the replay programs
        times = []
        for _ in range(2 if QUICK else 5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.generate(x, N, **kw)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        dt = statistics.median(times)
        res[name] = dt / N * 1e3   # ms per token step
        print(json.dumps({"bench": "generate", **{k: CFG[k] for k in ("n_layer", "n_head", "n_embd", "block_size")}, "V": V_WS,
                          "B": B, "new_tokens": N, "head": name, "ms_per_token_step": round(dt / N * 1e3, 4),
                          "tokens_per_s": round(B * N / dt)}), flush=True)
    del model
    torch.cuda.empty_cache()
    return res


def bench_train(B=64, T=256):
    torch.manual_seed(0)
    model = GPT(GPTConfig(**CFG)).cuda().train()
    opt = model.configure_optimizers(0.1, 6e-4, (0.9, 0.95), "cuda")
    x = torch.randint(V_WS, (B, T), device="cuda")
    y = torch.randint(V_WS, (B, T), device="cuda")

    def step():
        _, loss = model(x, y)
        loss.backward()
        model.clip_grad_norm_(1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)
    ms = timed(step, reps=3 if QUICK else 5, iters=5 if QUICK else 20, warmup=3)
    # instrumented pass
    sink = []
    ops.set_profile(sink)
    try:
        for _ in range(3):
            step()
        torch.cuda.synchronize()
    finally:
        ops.set_profile(None)
    vpad = (V_WS + 7) // 8 * 8
    per = {"lm_head_gemm": 0.0, "cross_entropy": 0.0, "other": 0.0}
    for name, meta, e0, e1 in sink:
        t = e0.elapsed_time(e1) / 3
        if name == "gemm" and vpad in meta[:3]:
            per["lm_head_gemm"] += t
        elif name.startswith("ce_"):
            per["cross_entropy"] += t
        else:
            per["other"] += t
    total = sum(per.values())
    print(json.dumps({"bench": "train_step", **{k: CFG[k] for k in ("n_layer", "n_head", "n_embd")}, "V": V_WS, "B": B, "T": T,
                      "step_ms": round(ms, 3), "tokens_per_s": round(B * T / ms * 1e3),
                      "instrumented_call_ms": {k: round(v, 3) for k, v in per.items()},
                      "share_of_call_time": {k: round(v / total, 3) for k, v in per.items()}}), flush=True)
    del model, opt
    torch.cuda.empty_cache()


if __name__ == "__main__":
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    samp = bench_sampler()
    gen = bench_generate()
    share = samp[(V_WS, 64, 200)] / gen["topk200_t0.8"]
    print(json.dumps({"bench": "sampling_share_of_topk_decode_step", "B": 64, "sampler_us": round(samp[(V_WS, 64, 200)] * 1e3, 2),
                      "decode_step_us": round(gen["topk200_t0.8"] * 1e3, 2), "share": round(share, 4),
                      "target_le_0.10_met": share <= 0.10}), flush=True)
    bench_train()
    print(json.dumps({"gpu": gpu_info()}), flush=True)
