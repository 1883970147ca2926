"""Headline benchmark: nanoGPT training step on char-level ABC tokens (BASELINE.json metric
"train tokens/s & MFU, GPT-2-124M char-level ABC, 1/2/4/8 B200").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg3|cfg2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one optimizer step of the hot path over one synthetic batch per GPU: forward, cross-entropy,
backward, gradient all-reduce (N > 1), clip_grad_norm_(1.0), AdamW (reference loop: nanoGPT/train.py:335-357,
nanoGPT/bench.py:98-117).  Weak scaling: the per-GPU micro-batch is fixed as N grows.

`value`  : tokens/s with the batch already resident in HBM (CUDA-event timed, max over ranks).
`e2e`    : the same step driven through the public API with pinned-host -> device copies of X, Y and a
           device -> host read of the loss inside every timed step.
`--dump-outputs DIR` : after the timed steps, what the last of them computed goes to DIR as float32 .npy files (dump_outputs).
`roofline`, `kernel_breakdown` : per-kernel-family times from an instrumented pass (CUDA events on the launch
           stream around every C-ABI call), GEMM family against the measured cuBLAS bf16 peak.
`cpu_baseline` / `--impl reference` : the reference step on the host cores (fp32, all host threads, also under torchrun) on a
           bounded sample of the same workload: the UNMODIFIED nanoGPT/model.py from the git-ignored byte-identical
           copy baseline/_ref (tools/vendor_reference.py; kind "reference"), else the oracle port
           (oracle/nanogpt_oracle.py, pinned to the reference by tests/golden; kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[2]: GPT-2 small shape, char-level ABC vocab, B200-sized micro-batch (SURVEY.md 8d)
    "cfg3": dict(name="GPT-2-small-shape 12L/12H/768d block 1024 V=95 (char-level ABC), micro-batch 32x1024 per GPU",
                 cfg=dict(block_size=1024, vocab_size=95, n_layer=12, n_head=12, n_embd=768, dropout=0.0, bias=False),
                 batch=32, lr=6e-4, betas=(0.9, 0.95), cpu_batch=2),
    # BASELINE.json configs[1]: baby GPT of config/irishman_char.py
    "cfg2": dict(name="baby GPT 6L/6H/384d block 256 V=95 (char-level ABC), batch 64x256 per GPU",
                 cfg=dict(block_size=256, vocab_size=95, n_layer=6, n_head=6, n_embd=384, dropout=0.0, bias=False),
                 batch=64, lr=1e-3, betas=(0.9, 0.99), cpu_batch=16),
}
METRIC = "train tokens/s, GPT-2-124M-shape char-level ABC (fwd+bwd+clip+AdamW)"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], burst=p["bf16_tflops"], sustained=p["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, burst=1590.0, sustained=1400.0, source="fallback")


def flops_per_token(c):
    n = 12 * c["n_layer"] * c["n_embd"] ** 2 + c["vocab_size"] * c["n_embd"] + (2 * c["n_layer"] + 1) * c["n_embd"]
    return 6 * n + 12 * c["n_layer"] * c["n_embd"] * c["block_size"]


# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "50", "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------------
def host_threads():
    """All host cores for the CPU arm.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers; the CPU baseline
    runs on rank 0 only, so it takes the whole machine back (otherwise the N > 1 baseline is a one-core number)."""
    import torch
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    torch.set_num_threads(n)
    return torch.get_num_threads()


def cpu_reference_tokens_per_s(wl, steps, warmup, batch=None):
    """One optimizer step of the reference on the host cores, fp32, on a bounded sample (cpu_batch sequences) of the workload.

    kind "reference": the UNMODIFIED nanoGPT/model.py (byte-identical copy under baseline/_ref, tools/vendor_reference.py)
    driven like nanoGPT/train.py:335-357 with device=cpu (forward, backward, stock clip_grad_norm_, torch AdamW from
    configure_optimizers); kind "port": the oracle restatement (oracle/nanogpt_oracle.py), when the copy is absent.
    Returns (tokens/s, s/step, batch, threads, kind)."""
    import contextlib
    import io
    import torch
    threads = host_threads()
    B = batch or wl["cpu_batch"]
    T, V = wl["cfg"]["block_size"], wl["cfg"]["vocab_size"]
    g = torch.Generator().manual_seed(1234)
    x = torch.randint(V, (B, T), generator=g)
    y = torch.randint(V, (B, T), generator=g)
    times = []
    from tools.vendor_reference import import_reference_model
    ref = import_reference_model()
    if ref is not None:
        GPT, GPTConfig = ref
        torch.manual_seed(1337)
        with contextlib.redirect_stdout(io.StringIO()):
            model = GPT(GPTConfig(**wl["cfg"]))
            opt = model.configure_optimizers(0.1, wl["lr"], wl["betas"], "cpu")
        model.train()
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            _, loss = model(x, y)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
            opt.zero_grad(set_to_none=True)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
        kind = "reference"
    else:
        from oracle import nanogpt_oracle as O
        cfg = O.OracleConfig(**wl["cfg"])
        torch.manual_seed(1337)
        sd = {k: torch.randn(s) * 0.02 if len(s) > 1 else torch.ones(s) for k, s in O.param_shapes(cfg).items()}
        state = {}
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            _, _, grads = O.loss_and_grads(sd, cfg, x, y)
            c = O.clip_coef(O.grad_norm(grads), 1.0)
            O.adamw_step(sd, {k: v * c for k, v in grads.items()}, state, lr=wl["lr"], betas=wl["betas"], weight_decay=0.1,
                         step=it + 1)
            if it >= warmup:
                times.append(time.perf_counter() - t0)
        kind = "port"
    dt = sum(times) / len(times)
    return B * T / dt, dt, B, threads, kind


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(1, min(args.warmup, 2))
    tps, dt, B, threads, kind = cpu_reference_tokens_per_s(wl, steps, warmup)
    what = "unmodified reference nanoGPT/model.py" if kind == "reference" else "oracle port"
    sample = f"{steps} timed + {warmup} warm-up optimizer steps of {B}x{wl['cfg']['block_size']} tokens (fp32, CPU, {what})"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": tps, "unit": "tokens/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": {"workload": wl["name"], "global_batch": B,
                                                        "seq_len": wl["cfg"]["block_size"], "parallelism": "cpu"},
        "cpu_baseline": {"value": tps, "unit": "tokens/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": tps, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ----------------------------------------------------------------------------------------------------------------
def gemm_flops(meta):
    M, N, K = meta[0], meta[1], meta[2]
    return 2.0 * M * N * K


def attn_flops(meta, bwd):
    B, T, H = meta
    fwd = 4.0 * B * H * T * T * 64 / 2  # causal half of QK^T and PV
    return 2.5 * fwd if bwd else fwd


# ----------------------------------------------------------------------------------------------------------------
LOGITS_SAMPLE = 1 << 22   # elements; the default cfg3 / cfg2 batches (3.1 M / 1.6 M logits) are written whole
PARAM_SAMPLE = 1 << 16    # elements per parameter tensor; a cfg3 dump (75 tensors + logits) is ~25 MB, well under 64 MB


def _sample(t, limit):
    """t as float32 numpy; above `limit` elements a fixed, seeded sample of `limit` of them (the same positions in every run)."""
    import torch
    t = t.detach()
    if t.numel() > limit:
        idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:limit].sort().values
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu().numpy()


def dump_outputs(out_dir, model, logits, loss, norm):
    """What one training step hands its caller, as DIR/<name>.npy: `logits` and `loss` of the forward, `grad_norm` (the
    pre-clip total norm clip_grad_norm_ returns) and `param.<name>` for every parameter after the optimizer step.  With the
    same bench.py arguments the inputs are identical from run to run, so two builds can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"logits": _sample(logits, LOGITS_SAMPLE), "loss": _sample(loss, 1), "grad_norm": _sample(norm, 1)}
    for name, p in model.named_parameters():
        arrays["param." + name] = _sample(p, PARAM_SAMPLE)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dropout", type=float, default=0.0, help="train with dropout (music configs use 0.2; the headline uses 0 like nanoGPT/bench.py:54)")
    ap.add_argument("--bucket-mb", type=float, default=64.0,
                    help="gradient all-reduce bucket size (N > 1); a huge value = one exposed all-reduce after the backward")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm times a bounded fp32 CPU sample (cpu_batch sequences), not the step of a build of this project
        ap.error("--dump-outputs writes the outputs of the GPU training step; --impl reference has none")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    import torch
    import torch.distributed as dist
    from ai_music_generation_b200 import DDP, GPT, GPTConfig, ops

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch multi-GPU runs with torch.distributed.run (one process per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # rank 0's stdout must carry exactly one JSON line: NCCL_DEBUG=VERSION (set in some images) prints a banner there
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)

    cfg = dict(wl["cfg"], dropout=args.dropout)
    B = args.batch or wl["batch"]
    T, V = cfg["block_size"], cfg["vocab_size"]
    torch.manual_seed(1337)  # same init on every rank (train.py seeds 1337 + rank, then DDP broadcasts rank 0)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        model = GPT(GPTConfig(**cfg)).to(dev)
        opt = model.configure_optimizers(0.1, wl["lr"], wl["betas"], "cuda")
    model.train()
    net = DDP(model, bucket_mb=args.bucket_mb) if world > 1 else model

    g = torch.Generator().manual_seed(1234 + rank)
    n_host = 4
    host = [(torch.randint(V, (B, T), generator=g).pin_memory(), torch.randint(V, (B, T), generator=g).pin_memory())
            for _ in range(n_host)]
    xd, yd = host[0][0].to(dev), host[0][1].to(dev)

    def step_resident():
        logits, loss = net(xd, yd)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        norm = model.clip_grad_norm_(1.0)
        opt.step()
        return logits, loss, norm

    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()
    loss_ready = torch.cuda.Event()

    def step_e2e(i):
        hx, hy = host[i % n_host]
        x = hx.to(dev, non_blocking=True)
        y = hy.to(dev, non_blocking=True)
        _, loss = net(x, y)
        # device -> host read of THIS step's loss, every step: the copy is enqueued right behind the forward (the value
        # exists before the backward starts) and read at the end of the step, so the host never drains the whole step
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        loss_ready.record()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        model.clip_grad_norm_(1.0)
        opt.step()
        loss_ready.synchronize()
        return float(loss_host[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(ms over `steps` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            out = fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, out

    for i in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.LAUNCHES
    ms_total, last = timed(lambda i: step_resident(), args.steps)
    launches = ops.LAUNCHES - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # before the next forward: the logits are a view of the activation buffer that it overwrites
        dump_outputs(args.dump_outputs, model, *last)
    del last
    final_loss = step_resident()[1].item()

    for i in range(2):
        step_e2e(i)
    ms_e2e, _ = timed(step_e2e, args.steps)

    # ---- instrumented pass: CUDA events around every C-ABI call (kernel family shares + GEMM roofline) -----------
    prof = []
    torch.cuda.synchronize()
    ops.set_profile(prof)
    n_prof = 3
    marks = []
    for _ in range(n_prof):
        marks.append(len(prof))
        step_resident()
    marks.append(len(prof))
    torch.cuda.synchronize()
    ops.set_profile(None)
    # per family: the MEDIAN over the instrumented steps of that step's sum (one hiccup in one step — a clock dip, a page
    # fault — must not become the family's number; a two-step mean once showed the wgrad family at 6.0 instead of 4.8 ms)
    per_pass = []
    for a_, b_ in zip(marks[:-1], marks[1:]):
        fp = {}
        for name, meta, e0, e1 in prof[a_:b_]:
            key = name
            if name == "gemm":
                key = {(0, 0): "gemm_fwd", (0, 1): "gemm_dgrad", (1, 1): "gemm_wgrad"}[(meta[3], meta[4])]
            d = fp.setdefault(key, {"ms": 0.0, "calls": 0, "flops": 0.0})
            d["ms"] += e0.elapsed_time(e1)
            d["calls"] += 1
            if name == "gemm":
                d["flops"] += gemm_flops(meta)
            elif name in ("attn_fwd", "attn_bwd"):
                d["flops"] += attn_flops(meta, name == "attn_bwd")
        per_pass.append(fp)
    fam = {}
    for key in per_pass[0]:
        ms_sorted = sorted(fp[key]["ms"] for fp in per_pass if key in fp)
        fam[key] = {"ms": ms_sorted[len(ms_sorted) // 2], "calls": per_pass[0][key]["calls"] * n_prof, "flops": per_pass[0][key]["flops"]}
    prof_total = sum(d["ms"] for d in fam.values())
    for d in fam.values():
        d["calls"] //= n_prof
        d["share"] = round(d["ms"] / prof_total, 4)
        d["ms"] = round(d["ms"], 4)
        if d["flops"]:
            d["tflops"] = round(d["flops"] / d["ms"] / 1e9, 1)
        d.pop("flops")
    gemm_ms = sum(fam[k]["ms"] for k in fam if k.startswith("gemm"))
    gemm_fl = sum(gemm_flops(m) for n, m, _, _ in prof if n == "gemm") / n_prof
    gemm_calls = sum(fam[k]["calls"] for k in fam if k.startswith("gemm"))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    tokens_per_step = world * B * T
    ms_step = ms_total / args.steps
    value = tokens_per_step / (ms_step / 1e3)
    fpt = flops_per_token(cfg)
    achieved_tf = gemm_fl / gemm_ms / 1e9
    out = {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": wl["name"], "global_batch": world * B, "seq_len": T, "parallelism": f"dp{world}",
                   "l2_note": "per-step working set ~11 GB of activations >> 126 MB L2; no explicit flush",
                   "optimizer": "fused clip_grad_norm_(1.0) + AdamW every step, grad accumulation 1", "dropout": args.dropout,
                   "grad_exchange": ("none (1 GPU)" if world == 1 else
                                     ("nvls: one multimem.ld_reduce / multimem.st kernel + norm partials (csrc/nvls.cu)"
                                      if getattr(model._grad_sync, "nvls", None) is not None else "nccl all-reduce buckets overlapped with the backward"))},
        "mfu": {"flops_per_token": fpt, "per_gpu_tflops": value / world * fpt / 1e12,
                "of_nominal_2250": value / world * fpt / 2.25e15,
                "of_measured_burst": value / world * fpt / (pk["burst"] * 1e12),
                "of_measured_sustained": value / world * fpt / (pk["sustained"] * 1e12), "peaks": pk["source"]},
        "loss_after": final_loss,
        "e2e": {"value": tokens_per_step / (ms_e2e / args.steps / 1e3), "unit": "tokens/s",
                "h2d_bytes_per_step": 2 * B * T * 8, "d2h_bytes_per_step": 4},
        "gpu_launches": launches,
        "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "gemm_kernel (tcgen05, all fwd/dgrad/wgrad launches of a step)",
                     "achieved": achieved_tf, "peak": pk["sustained"], "unit": "TFLOP/s", "frac": achieved_tf / pk["sustained"],
                     "peak_kind": f"{pk['source']} sustained cuBLAS bf16", "launches_per_step": gemm_calls,
                     "avg_launch_ms": gemm_ms / gemm_calls, "flops_per_step": gemm_fl,
                     # DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) are NOT measured by this run: the
                     # figure is the launch-weighted mean over the twelve GEMM launches of a block at the cfg3 shapes, seven
                     # roles captured by ncu (profiles/r2b_ncu_gemm.md), the other five from their operand sizes (the captured
                     # roles' traffic equals their algorithmic bytes); null for other workloads
                     "traffic": 240e6 if args.workload == "cfg3" else None,
                     "traffic_source": "profiles/r2b_ncu_gemm.md (ncu capture per role, launch-weighted mean; not re-measured per run)"
                     if args.workload == "cfg3" else None},
        "kernel_breakdown": fam,
    }
    if not args.no_cpu_baseline:
        tps, dt, cb, threads, kind = cpu_reference_tokens_per_s(wl, 2, 1)
        what = "unmodified reference nanoGPT/model.py" if kind == "reference" else "oracle port"
        out["cpu_baseline"] = {"value": tps, "unit": "tokens/s", "cores": threads, "kind": kind,
                               "sample": f"2 timed + 1 warm-up optimizer steps of {cb}x{T} tokens, fp32, {what}"}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
