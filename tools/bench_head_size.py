"""Head sizes 32 / 64 / 128 at the GPT-2-small width (C = 768): attention kernels per layer, the full training step and decode.

    python tools/bench_head_size.py [--quick]

Prints one JSON line per measurement and the GPU name / power limit of the run (both are part of every number).  CUDA events,
medians over repeated timed regions.
  * attention per layer, B = 32, T = 1024, (H, D) = (24, 32), (12, 64), (6, 128): our forward, our backward, and the same shapes
    through torch.nn.functional.scaled_dot_product_attention (bf16, causal) as a bar only;
  * training step (forward + backward + clip + AdamW), 12 layers, n_embd 768, vocab 95, B = 32, T = 1024, n_head 24 / 12 / 6;
  * decode: generate() of 1023 new tokens for 256 sequences (greedy, KV cache), ms per token step.
At equal C the matmul FLOPs of attention are the same for all three head sizes, the exponentials scale with H: D = 32 does twice
the MUFU work of D = 64, D = 128 half of it.
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
SHAPES = [(24, 32), (12, 64), (6, 128)]


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


def timed(fn, reps=5, iters=10, warmup=3):
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


def bench_attention(B=32, T=1024, C=768):
    for H, D in SHAPES:
        torch.manual_seed(0)
        qkv = torch.randn(B * T, 3 * C, device="cuda").bfloat16()
        out = torch.empty(B * T, C, device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(B, H, T, device="cuda")
        dout = torch.randn(B * T, C, device="cuda").bfloat16()
        dqkv = torch.empty_like(qkv)
        delta = torch.empty(B, H, T, device="cuda")
        fwd = timed(lambda: ops.attn_fwd(qkv, out, lse, B, T, H, head_size=D))
        bwd = timed(lambda: ops.attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, head_size=D))
        # torch SDPA (bf16, causal) on [B, H, T, D] views: a bar, not a reference of ours
        q, k, v = (t.view(B, T, H, D).transpose(1, 2).detach().requires_grad_(True) for t in qkv.split(C, dim=1))
        sd_f = timed(lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=True))
        do4 = dout.view(B, T, H, D).transpose(1, 2)

        def sdpa_fb():
            o = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=True)
            o.backward(do4)
        sd_fb = timed(sdpa_fb)
        print(json.dumps({"bench": "attention_per_layer", "B": B, "T": T, "C": C, "H": H, "D": D, "fwd_ms": round(fwd, 4),
                          "bwd_ms": round(bwd, 4), "fwd_bwd_ms": round(fwd + bwd, 4), "sdpa_fwd_ms": round(sd_f, 4),
                          "sdpa_bwd_ms": round(sd_fb - sd_f, 4), "sdpa_fwd_bwd_ms": round(sd_fb, 4)}), flush=True)
        del qkv, out, dout, dqkv, q, k, v


def bench_step(B=32, T=1024):
    for H, D in SHAPES:
        torch.manual_seed(0)
        cfg = GPTConfig(block_size=T, vocab_size=95, n_layer=12, n_head=H, n_embd=768, dropout=0.0, bias=False)
        model = GPT(cfg).cuda().train()
        opt = model.configure_optimizers(0.1, 6e-4, (0.9, 0.95), "cuda")
        x = torch.randint(95, (B, T), device="cuda")
        y = torch.randint(95, (B, T), device="cuda")

        def step():
            _, loss = model(x, y)
            loss.backward()
            model.clip_grad_norm_(1.0)
            opt.step()
            opt.zero_grad(set_to_none=True)
        ms = timed(step, reps=3 if QUICK else 5, iters=5 if QUICK else 10)
        print(json.dumps({"bench": "train_step", "n_layer": 12, "n_embd": 768, "V": 95, "B": B, "T": T, "H": H, "D": D,
                          "step_ms": round(ms, 3), "tokens_per_s": round(B * T / ms * 1e3)}), flush=True)
        del model, opt
        torch.cuda.empty_cache()


def bench_decode(B=256, N=1023):
    for H, D in SHAPES:
        torch.manual_seed(1337)
        model = GPT(GPTConfig(block_size=1024, vocab_size=95, n_layer=12, n_head=H, n_embd=768, dropout=0.0, bias=False)).cuda().eval()
        x = torch.zeros(B, 1, dtype=torch.long, device="cuda")
        model.generate(x, 8, top_k=1)   # builds the decode state and the replay programs
        torch.cuda.synchronize()
        t0 = time.time()
        model.generate(x, N, top_k=1)
        torch.cuda.synchronize()
        dt = time.time() - t0
        print(json.dumps({"bench": "decode", "n_layer": 12, "n_embd": 768, "B": B, "new_tokens": N, "H": H, "D": D,
                          "ms_per_token_step": round(dt / N * 1e3, 4), "tokens_per_s": round(B * N / dt)}), flush=True)
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    bench_attention()
    bench_step()
    bench_decode(N=255 if QUICK else 1023)
    print(json.dumps({"gpu": gpu_info()}), flush=True)
