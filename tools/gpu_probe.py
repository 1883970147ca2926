"""Per-kernel numerical probe + timing on a real B200.  Each case runs in its own subprocess so that a device
trap in one kernel cannot take the others down.  Appends to probe_out/probe.jsonl and prints a summary.

    python tools/gpu_probe.py                # all cases
    python tools/gpu_probe.py gemm attn      # only case groups whose name starts with one of these
    python tools/gpu_probe.py --case NAME    # (internal) run one case in-process
    ABCGPT_PROBE_OUT=DIR python tools/gpu_probe.py ...   # probe.jsonl goes to DIR (tests keep the source tree untouched)
"""
from __future__ import annotations

import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT_DIR = os.path.join(ROOT, "probe_out")


def _timeit(fn, iters=10, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _err(got, ref):
    import torch
    got, ref = got.float(), ref.float()
    d = (got - ref).abs()
    denom = ref.abs().max().item() + 1e-30
    bad = ~torch.isfinite(got)
    return {
        "max_abs": d.max().item() if not bad.any() else float("inf"),
        "max_rel_to_max": (d.max().item() / denom) if not bad.any() else float("inf"),
        "rel_l2": ((got - ref).norm() / (ref.norm() + 1e-30)).item() if not bad.any() else float("inf"),
        "nonfinite": int(bad.sum().item()),
    }


def _mismatch_map(got, ref, tol, rb=8, cb=16, max_r=128, max_c=128):
    """Coarse (row-block x col-block) map of where a 2-D result is wrong, for the first tile."""
    import torch
    g, r = got[:max_r, :max_c].float(), ref[:max_r, :max_c].float()
    wrong = ((g - r).abs() > tol) | ~torch.isfinite(g)
    R, Cc = wrong.shape
    lines = []
    for i in range(0, R, rb):
        lines.append("".join("X" if wrong[i:i + rb, j:j + cb].any().item() else "." for j in range(0, Cc, cb)))
    return lines


# ------------------------------------------------------------------------------------------------------------
def case_gemm(name, M, N, K, a_mn, b_mn, epi, tile_n, splits=0, timing=True, tanh=False):
    import torch
    from ai_music_generation_b200 import ops
    approx = "tanh" if tanh else "none"   # tanh: HF gelu_new (ABCGPT_ACT_TANH)
    act = ops.ACT_TANH if tanh else 0
    torch.manual_seed(0)
    dev = "cuda"
    A = (torch.randn(M, K, device=dev) * 0.5).bfloat16()
    B = (torch.randn(N, K, device=dev) * 0.5).bfloat16()
    a_arg = A.t().contiguous() if a_mn else A
    b_arg = B.t().contiguous() if b_mn else B
    acc = A.float() @ B.float().t()
    res = {"case": name}
    if epi == ops.EPI_BF16:
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        ref = acc
        run = lambda: ops.gemm(a_arg, b_arg, a_mn=a_mn, b_mn=b_mn, epilogue=epi, out=out, tile_n=tile_n)
        outs = [(out, ref, 0.02)]
    elif epi == ops.EPI_GELU:
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        out2 = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        h = acc.bfloat16()
        ref2 = torch.nn.functional.gelu(h.float(), approximate=approx)
        run = lambda: ops.gemm(a_arg, b_arg, a_mn=a_mn, b_mn=b_mn, epilogue=epi | act, out=out, out2=out2, tile_n=tile_n)
        outs = [(out, acc, 0.02), (out2, ref2, 0.02)]
    elif epi == ops.EPI_RESID:
        resid = torch.randn(M, N, device=dev)
        out = torch.zeros(M, N, device=dev)
        ref = resid + acc.bfloat16().float()
        run = lambda: ops.gemm(a_arg, b_arg, a_mn=a_mn, b_mn=b_mn, epilogue=epi, out=out, aux=resid, tile_n=tile_n)
        outs = [(out, ref, 0.02)]
    elif epi == ops.EPI_DGELU:
        hpre = torch.randn(M, N, device=dev).bfloat16()
        out = torch.zeros(M, N, device=dev, dtype=torch.bfloat16)
        hf = hpre.float().requires_grad_(True)
        torch.nn.functional.gelu(hf, approximate=approx).backward(acc.bfloat16().float())
        ref = hf.grad
        run = lambda: ops.gemm(a_arg, b_arg, a_mn=a_mn, b_mn=b_mn, epilogue=epi | act, out=out, aux=hpre, tile_n=tile_n)
        outs = [(out, ref, 0.02)]
    elif epi == ops.EPI_F32_RED:
        out = torch.zeros(M, N, device=dev)
        ref = acc
        def run():
            out.zero_()
            ops.gemm(a_arg, b_arg, a_mn=a_mn, b_mn=b_mn, epilogue=epi, out=out, tile_n=tile_n, splits=splits)
        outs = [(out, ref, 1e-3)]
    else:
        out = torch.zeros(M, N, device=dev)
        ref = acc
        run = lambda: ops.gemm(a_arg, b_arg, a_mn=a_mn, b_mn=b_mn, epilogue=epi, out=out, tile_n=tile_n)
        outs = [(out, ref, 1e-3)]
    run()
    torch.cuda.synchronize()
    scale = math.sqrt(K) * 0.25
    res["errs"] = [_err(o, r) for o, r, _ in outs]
    # bf16 outputs: one rounding step (2^-9 relative) on top of fp32 accumulation; fp32 outputs: accumulation order only
    res["ok"] = all(e["rel_l2"] <= (4e-3 if o.dtype == torch.bfloat16 or epi == ops.EPI_RESID else 1e-4)
                    for e, (o, _, _) in zip(res["errs"], outs))
    if not res["ok"]:
        o, r, tol = outs[0]
        res["map"] = _mismatch_map(o, r, tol * scale)
        res["sample_got"] = o[:2, :8].float().flatten().tolist()
        res["sample_ref"] = r[:2, :8].float().flatten().tolist()
    if timing and res["ok"]:
        ms = _timeit(run)
        res["ms"] = ms
        res["tflops"] = 2.0 * M * N * K / ms / 1e9
    return res


def _attn_ref(qkv, B, T, H, D=64):
    import torch
    C = H * D
    q, k, v = qkv.float().split(C, dim=1)
    q = q.view(B, T, H, D).transpose(1, 2)
    k = k.view(B, T, H, D).transpose(1, 2)
    v = v.view(B, T, H, D).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) * (1.0 / math.sqrt(D))
    mask = torch.ones(T, T, device=qkv.device, dtype=torch.bool).tril()
    s = s.masked_fill(~mask, float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    p = torch.softmax(s, dim=-1)
    o = (p @ v).transpose(1, 2).reshape(B * T, C)
    return o, lse


def case_attn(name, B, T, H, bwd, timing=True, spike=False, D=64):
    """D: head size (64: csrc/attn.cu; 32 / 128: csrc/attn_hd.cu)."""
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(0)
    dev = "cuda"
    C = H * D
    qkv = torch.randn(B * T, 3 * C, device=dev)
    if spike:
        # scores jump by ~2^100 after the first 64 keys: exercises the lazy-rescale path of the forward kernel
        sign = torch.where(torch.arange(C, device=dev) % 2 == 0, 1.0, -1.0)
        qkv[:, :C] = 3.0 * sign
        v3 = qkv.view(B, T, 3 * C)
        v3[:, 64:, C:2 * C] = 3.0 * sign + 0.05 * torch.randn(B, T - 64, C, device=dev)
    qkv = qkv.bfloat16()
    out = torch.zeros(B * T, C, device=dev, dtype=torch.bfloat16)
    lse = torch.zeros(B, H, T, device=dev)
    res = {"case": name}
    ops.attn_fwd(qkv, out, lse, B, T, H, head_size=D)
    torch.cuda.synchronize()
    small = B * H * T * T <= 64 * 1024 * 1024
    if small:
        qkv_f = qkv.float().requires_grad_(True)
        o_ref, lse_ref = _attn_ref(qkv_f, B, T, H, D)
        res["errs"] = [_err(out, o_ref.detach()), _err(lse, lse_ref.detach())]
        res["ok"] = res["errs"][0]["max_abs"] < 0.03 and res["errs"][1]["max_abs"] < 0.01
        if not res["ok"]:
            res["map"] = _mismatch_map(out, o_ref.detach(), 0.03, rb=16, cb=8, max_r=256, max_c=64)
    else:
        res["ok"] = bool(torch.isfinite(out.float()).all().item())
    if bwd:
        dout = torch.randn(B * T, C, device=dev).bfloat16()
        dqkv = torch.zeros(B * T, 3 * C, device=dev, dtype=torch.bfloat16)
        delta = torch.zeros(B, H, T, device=dev)
        ops.attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, head_size=D)
        torch.cuda.synchronize()
        if small:
            o_ref.backward(dout.float())
            g = qkv_f.grad
            e = {"dq": _err(dqkv[:, :C], g[:, :C]), "dk": _err(dqkv[:, C:2 * C], g[:, C:2 * C]),
                 "dv": _err(dqkv[:, 2 * C:], g[:, 2 * C:])}
            res["bwd_errs"] = e
            # T = 1: dQ and dK are exactly zero (softmax over one key), where only an absolute bound is meaningful
            zero = {"dq": g[:, :C].abs().max().item() == 0, "dk": g[:, C:2 * C].abs().max().item() == 0,
                    "dv": g[:, 2 * C:].abs().max().item() == 0}
            res["bwd_ok"] = all(v["rel_l2"] < 0.02 or (zero[k] and v["max_abs"] < 1e-5) for k, v in e.items())
            if not res["bwd_ok"]:
                res["map_dq"] = _mismatch_map(dqkv[:, :64], g[:, :64], 0.05, rb=16, cb=8, max_r=256, max_c=64)
                res["map_dk"] = _mismatch_map(dqkv[:, C:C + 64], g[:, C:C + 64], 0.05, rb=16, cb=8, max_r=256, max_c=64)
                res["map_dv"] = _mismatch_map(dqkv[:, 2 * C:2 * C + 64], g[:, 2 * C:2 * C + 64], 0.05, rb=16, cb=8, max_r=256, max_c=64)
            res["ok"] = res["ok"] and res["bwd_ok"]
    if timing and res["ok"]:
        ms = _timeit(lambda: ops.attn_fwd(qkv, out, lse, B, T, H, head_size=D))
        fl = 4.0 * B * H * T * T * D / 2
        res["fwd_ms"], res["fwd_tflops_causal"] = ms, fl / ms / 1e9
        if bwd:
            ms = _timeit(lambda: ops.attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, head_size=D))
            res["bwd_ms"], res["bwd_tflops_causal"] = ms, 2.5 * fl / ms / 1e9
    return res


def case_layernorm(name, M, C, bias):
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(0)
    dev = "cuda"
    x = torch.randn(M, C, device=dev) * 2 + 0.5
    w = torch.randn(C, device=dev)
    b = torch.randn(C, device=dev) if bias else None
    y = torch.zeros(M, C, device=dev, dtype=torch.bfloat16)
    mean = torch.zeros(M, device=dev)
    rstd = torch.zeros(M, device=dev)
    ops.layernorm_fwd(x, w, b, y, mean, rstd)
    xr = x.clone().requires_grad_(True)
    wr = w.clone().requires_grad_(True)
    br = b.clone().requires_grad_(True) if bias else None
    yr = torch.nn.functional.layer_norm(xr, (C,), wr, br, 1e-5)
    res = {"case": name, "errs": [_err(y, yr.detach())]}
    dy = torch.randn(M, C, device=dev).bfloat16()
    dres = torch.randn(M, C, device=dev)
    dx = torch.zeros(M, C, device=dev)
    dxb = torch.zeros(M, C, device=dev, dtype=torch.bfloat16)
    dw = torch.zeros(C, device=dev)
    db = torch.zeros(C, device=dev) if bias else None
    ops.layernorm_bwd(dy, x, w, mean, rstd, dres, dx, dxb, dw, db)
    yr.backward(dy.float())
    res["errs"] += [_err(dx, xr.grad + dres), _err(dxb, xr.grad + dres), _err(dw, wr.grad)]
    if bias:
        res["errs"].append(_err(db, br.grad))
    res["ok"] = (res["errs"][0]["max_abs"] < 0.05 and res["errs"][1]["rel_l2"] < 1e-5 and res["errs"][2]["rel_l2"] < 5e-3
                 and all(e["rel_l2"] < 1e-4 for e in res["errs"][3:]))
    ms = _timeit(lambda: ops.layernorm_fwd(x, w, b, y, mean, rstd))
    res["fwd_ms"], res["fwd_gbs"] = ms, (4 + 2) * M * C / ms / 1e6
    ms = _timeit(lambda: ops.layernorm_bwd(dy, x, w, mean, rstd, dres, dx, dxb, dw, db))
    res["bwd_ms"], res["bwd_gbs"] = ms, (2 + 4 + 4 + 4 + 2) * M * C / ms / 1e6
    return res


def case_layernorm_resid(name, M, C, bias):
    """x_out = x_in + branch (bf16), y = LN(x_out) in one pass; exact fp32 add, LN against torch."""
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(1)
    dev = "cuda"
    x = torch.randn(M, C, device=dev) * 2 + 0.5
    br = torch.randn(M, C, device=dev).bfloat16()
    w = torch.randn(C, device=dev)
    b = torch.randn(C, device=dev) if bias else None
    xo = torch.zeros(M, C, device=dev)
    y = torch.zeros(M, C, device=dev, dtype=torch.bfloat16)
    mean, rstd = torch.zeros(M, device=dev), torch.zeros(M, device=dev)
    ops.layernorm_fwd_resid(x, br, xo, w, b, y, mean, rstd)
    xs = x + br.float()
    yr = torch.nn.functional.layer_norm(xs, (C,), w, b, 1e-5)
    res = {"case": name, "errs": [_err(xo, xs), _err(y, yr), _err(mean, xs.mean(-1)), _err(rstd, (xs.var(-1, unbiased=False) + 1e-5).rsqrt())]}
    res["ok"] = bool(torch.equal(xo, xs)) and res["errs"][1]["max_abs"] < 0.05 and res["errs"][2]["max_abs"] < 1e-5 and res["errs"][3]["rel_l2"] < 1e-5
    ms = _timeit(lambda: ops.layernorm_fwd_resid(x, br, xo, w, b, y, mean, rstd))
    res["fwd_ms"], res["fwd_gbs"] = ms, (4 + 2 + 4 + 2) * M * C / ms / 1e6
    return res


def case_ce(name, M, V, ldl):
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(0)
    dev = "cuda"
    logits = torch.zeros(M, ldl, device=dev, dtype=torch.bfloat16)
    logits[:, :V] = (torch.randn(M, V, device=dev) * 3).bfloat16()
    logits[:, V:] = 77.0  # poison the padding: must be ignored
    tgt = torch.randint(0, V, (M,), device=dev)
    tgt[::7] = -1
    row_loss = torch.zeros(M, device=dev)
    sc = torch.zeros(2, device=dev)
    loss = torch.zeros(1, device=dev)
    ops.ce_fwd(logits, tgt, row_loss, sc, loss, V)
    lr = logits[:, :V].float().requires_grad_(True)
    ref = torch.nn.functional.cross_entropy(lr, tgt, ignore_index=-1)
    gl = torch.full((1,), 0.5, device=dev)
    dlog = torch.full((M, ldl), 9.0, device=dev, dtype=torch.bfloat16)
    ops.ce_bwd(logits, tgt, sc, gl, dlog, V)
    (ref * 0.5).backward()
    res = {"case": name, "loss": loss.item(), "loss_ref": ref.item(),
           "errs": [_err(dlog[:, :V], lr.grad), {"pad_max": dlog[:, V:].float().abs().max().item() if ldl > V else 0.0}]}
    res["ok"] = abs(loss.item() - ref.item()) < 1e-5 * max(1, abs(ref.item())) and res["errs"][0]["rel_l2"] < 5e-3 \
        and res["errs"][1]["pad_max"] == 0.0
    res["fwd_ms"] = _timeit(lambda: ops.ce_fwd(logits, tgt, row_loss, sc, loss, V))
    res["bwd_ms"] = _timeit(lambda: ops.ce_bwd(logits, tgt, sc, gl, dlog, V))
    return res


def case_colsum(name, M, N, timing=False):
    """Bias gradient: out[n] += sum_m dy[m, n] (bf16 in, fp32 accumulate), on top of a non-zero `out` (gradient accumulation)."""
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(0)
    dy = torch.randn(M, N, device="cuda").bfloat16()
    out = torch.full((N,), 0.5, device="cuda")
    ops.colsum_bf16(dy, out)
    torch.cuda.synchronize()
    ref = 0.5 + dy.double().sum(0)
    err = (out.double() - ref).abs().max().item()
    res = {"case": name, "max_abs": err, "ok": err <= 1e-3 * math.sqrt(M)}
    if timing and res["ok"]:
        ms = _timeit(lambda: ops.colsum_bf16(dy, out))
        res["ms"] = ms
        res["tb_per_s"] = M * N * 2 / ms / 1e9
    return res


def case_adamw(name, n):
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(0)
    dev = "cuda"
    p = torch.randn(n, device=dev)
    g = torch.randn(n, device=dev) * 3
    pr = p.clone().requires_grad_(True)
    opt = torch.optim.AdamW([pr], lr=1e-3, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1)
    m = torch.zeros(n, device=dev)
    v = torch.zeros(n, device=dev)
    sh = torch.zeros(n, device=dev, dtype=torch.bfloat16)
    ss = torch.zeros(1, device=dev)
    for step in range(1, 4):
        gg = g * step
        pr.grad = gg.clone()
        torch.nn.utils.clip_grad_norm_([pr], 1.0)
        opt.step()
        ss.zero_()
        ops.sumsq(gg, ss)
        ops.adamw(p, gg, m, v, sh, lr=1e-3, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.1, step=step, sumsq=ss,
                  max_norm=1.0)
    res = {"case": name, "errs": [_err(p, pr.detach()), _err(sh, pr.detach().bfloat16())],
           "norm": math.sqrt(ss.item()), "norm_ref": (g * 3).norm().item()}
    res["ok"] = res["errs"][0]["max_abs"] < 1e-5 and res["errs"][1]["max_abs"] < 0.04
    gg = g.clone()
    ms = _timeit(lambda: ops.adamw(p, gg, m, v, sh, lr=1e-3, beta1=0.9, beta2=0.95, eps=1e-8, weight_decay=0.1, step=5,
                                   sumsq=ss, max_norm=1.0))
    res["ms"], res["gbs"] = ms, 30.0 * n / ms / 1e6
    ms = _timeit(lambda: ops.sumsq(gg, ss))
    res["sumsq_ms"], res["sumsq_gbs"] = ms, 4.0 * n / ms / 1e6
    return res


def case_embed(name, B, T, C, V):
    import torch
    from ai_music_generation_b200 import ops
    torch.manual_seed(0)
    dev = "cuda"
    idx = torch.randint(0, V, (B, T), device=dev)
    wte = torch.randn(V, C, device=dev, requires_grad=True)
    wpe = torch.randn(T, C, device=dev, requires_grad=True)
    x = torch.zeros(B * T, C, device=dev)
    ops.embed_fwd(idx, wte.detach(), wpe.detach(), x, T)
    ref = wte[idx] + wpe[torch.arange(T, device=dev)]
    dx = torch.randn(B * T, C, device=dev)
    ref.backward(dx.view(B, T, C))
    dwte = torch.zeros(V, C, device=dev)
    dwpe = torch.zeros(T, C, device=dev)
    ops.embed_bwd(idx, dx, dwte, dwpe, T)
    res = {"case": name, "errs": [_err(x, ref.detach().view(B * T, C)), _err(dwte, wte.grad), _err(dwpe, wpe.grad)]}
    res["ok"] = res["errs"][0]["max_abs"] == 0 and res["errs"][1]["rel_l2"] < 1e-5 and res["errs"][2]["rel_l2"] < 1e-5
    res["fwd_ms"] = _timeit(lambda: ops.embed_fwd(idx, wte.detach(), wpe.detach(), x, T))
    res["bwd_ms"] = _timeit(lambda: ops.embed_bwd(idx, dx, dwte, dwpe, T))
    return res


def build_cases():
    from ai_music_generation_b200 import _C
    E = _C
    cases = {}
    # --- GEMM: small single-tile cases first (layout debugging), then production shapes
    for bn in (128, 256):
        cases[f"gemm_nt_small_bn{bn}"] = lambda bn=bn: case_gemm(f"gemm_nt_small_bn{bn}", 128, 256, 64, False, False, E.EPI_BF16, bn, timing=False)
        cases[f"gemm_nt_k256_bn{bn}"] = lambda bn=bn: case_gemm(f"gemm_nt_k256_bn{bn}", 256, 512, 256, False, False, E.EPI_BF16, bn, timing=False)
        cases[f"gemm_nn_small_bn{bn}"] = lambda bn=bn: case_gemm(f"gemm_nn_small_bn{bn}", 128, 256, 128, False, True, E.EPI_BF16, bn, timing=False)
        cases[f"gemm_tn_small_bn{bn}"] = lambda bn=bn: case_gemm(f"gemm_tn_small_bn{bn}", 128, 256, 128, True, True, E.EPI_F32, bn, timing=False)
    cases["gemm2_nt_small"] = lambda: case_gemm("gemm2_nt_small", 256, 256, 64, False, False, E.EPI_BF16, 512, timing=False)
    cases["gemm2_nt_k512"] = lambda: case_gemm("gemm2_nt_k512", 512, 768, 512, False, False, E.EPI_BF16, 512, timing=False)
    cases["gemm2_nn"] = lambda: case_gemm("gemm2_nn", 512, 512, 384, False, True, E.EPI_BF16, 512, timing=False)
    cases["gemm2_tn"] = lambda: case_gemm("gemm2_tn", 512, 512, 1024, True, True, E.EPI_F32, 512, timing=False)
    cases["gemm2_tn_red"] = lambda: case_gemm("gemm2_tn_red", 768, 768, 8192, True, True, E.EPI_F32_RED, 512, timing=False)
    cases["gemm2_ragged"] = lambda: case_gemm("gemm2_ragged", 328, 200, 136, False, False, E.EPI_BF16, 512, timing=False)
    cases["gemm2_gelu"] = lambda: case_gemm("gemm2_gelu", 1024, 1536, 384, False, False, E.EPI_GELU, 512, timing=False)
    cases["gemm2_resid"] = lambda: case_gemm("gemm2_resid", 1024, 384, 1536, False, False, E.EPI_RESID, 512, timing=False)
    cases["gemm2_gelu_tanh"] = lambda: case_gemm("gemm2_gelu_tanh", 1024, 1536, 384, False, False, E.EPI_GELU, 512, timing=False, tanh=True)
    cases["gemm2_dgelu_tanh"] = lambda: case_gemm("gemm2_dgelu_tanh", 1024, 1536, 384, False, True, E.EPI_DGELU, 512, timing=False, tanh=True)
    cases["gemm2_dgelu"] = lambda: case_gemm("gemm2_dgelu", 1024, 1536, 384, False, True, E.EPI_DGELU, 512, timing=False)
    # half tiles of the pair kernel (a short last round of the static schedule is issued as 256 x 128 work items): 10 x 8 = 80 tiles
    # on 74 pairs -> the last 6 tiles become 12 half items, including the ragged M / N edges; every epilogue and operand form
    cases["gemm2_half_nt"] = lambda: case_gemm("gemm2_half_nt", 2500, 2000, 192, False, False, E.EPI_BF16, 512, timing=False)
    cases["gemm2_half_nn"] = lambda: case_gemm("gemm2_half_nn", 2500, 2000, 192, False, True, E.EPI_BF16, 512, timing=False)
    cases["gemm2_half_gelu"] = lambda: case_gemm("gemm2_half_gelu", 2560, 2048, 128, False, False, E.EPI_GELU, 512, timing=False)
    cases["gemm2_half_dgelu"] = lambda: case_gemm("gemm2_half_dgelu", 2500, 2000, 128, False, True, E.EPI_DGELU, 512, timing=False)
    cases["gemm2_half_resid"] = lambda: case_gemm("gemm2_half_resid", 2500, 2000, 192, False, False, E.EPI_RESID, 512, timing=False)
    # automatic tile choice (hint 0) at the baby GPT's shapes, where N = 384 sends the problem to 128 x 128 single-CTA tiles
    cases["gemm_auto_cfg2_resid"] = lambda: case_gemm("gemm_auto_cfg2_resid", 16384, 384, 1536, False, False, E.EPI_RESID, 0, timing=False)
    cases["gemm_auto_cfg2_dgrad"] = lambda: case_gemm("gemm_auto_cfg2_dgrad", 16384, 384, 384, False, True, E.EPI_BF16, 0, timing=False)
    cases["gemm_auto_cfg2_dgelu"] = lambda: case_gemm("gemm_auto_cfg2_dgelu", 16384, 1536, 384, False, True, E.EPI_DGELU, 0, timing=False)
    cases["gemm_auto_cfg2_wgrad"] = lambda: case_gemm("gemm_auto_cfg2_wgrad", 1152, 384, 16384, True, True, E.EPI_F32_RED, 0, timing=False)
    cases["gemm_nt_ragged"] = lambda: case_gemm("gemm_nt_ragged", 200, 96, 136, False, False, E.EPI_BF16, 128, timing=False)
    cases["gemm_nt_f32"] = lambda: case_gemm("gemm_nt_f32", 256, 256, 768, False, False, E.EPI_F32, 256, timing=False)
    cases["gemm_gelu"] = lambda: case_gemm("gemm_gelu", 512, 1536, 384, False, False, E.EPI_GELU, 0, timing=False)
    cases["gemm_resid"] = lambda: case_gemm("gemm_resid", 512, 384, 1536, False, False, E.EPI_RESID, 0, timing=False)
    cases["gemm_dgelu"] = lambda: case_gemm("gemm_dgelu", 512, 1536, 384, False, True, E.EPI_DGELU, 0, timing=False)
    cases["gemm_wgrad_red"] = lambda: case_gemm("gemm_wgrad_red", 1152, 384, 4096, True, True, E.EPI_F32_RED, 0, timing=False)
    M = 32768
    cases["gemm_perf_c_attn"] = lambda: case_gemm("gemm_perf_c_attn", M, 2304, 768, False, False, E.EPI_BF16, 0)
    cases["gemm_perf_c_proj_resid"] = lambda: case_gemm("gemm_perf_c_proj_resid", M, 768, 768, False, False, E.EPI_RESID, 0)
    cases["gemm_perf_c_fc_gelu"] = lambda: case_gemm("gemm_perf_c_fc_gelu", M, 3072, 768, False, False, E.EPI_GELU, 0)
    cases["gemm_perf_mlp_proj_resid"] = lambda: case_gemm("gemm_perf_mlp_proj_resid", M, 768, 3072, False, False, E.EPI_RESID, 0)
    cases["gemm_perf_dgrad_fc"] = lambda: case_gemm("gemm_perf_dgrad_fc", M, 768, 3072, False, True, E.EPI_BF16, 0)
    cases["gemm_perf_dgrad_proj_dgelu"] = lambda: case_gemm("gemm_perf_dgrad_proj_dgelu", M, 3072, 768, False, True, E.EPI_DGELU, 0)
    cases["gemm_perf_wgrad_fc"] = lambda: case_gemm("gemm_perf_wgrad_fc", 3072, 768, M, True, True, E.EPI_F32_RED, 0)
    cases["gemm_perf_wgrad_attn"] = lambda: case_gemm("gemm_perf_wgrad_attn", 2304, 768, M, True, True, E.EPI_F32_RED, 0)
    cases["gemm_perf_lm_head"] = lambda: case_gemm("gemm_perf_lm_head", M, 128, 768, False, False, E.EPI_BF16, 0)
    # --- attention
    cases["attn_t128"] = lambda: case_attn("attn_t128", 2, 128, 2, True, timing=False)
    cases["attn_t256"] = lambda: case_attn("attn_t256", 2, 256, 3, True, timing=False)
    cases["attn_t1024"] = lambda: case_attn("attn_t1024", 2, 1024, 2, True, timing=False)
    cases["attn_t32"] = lambda: case_attn("attn_t32", 3, 32, 2, True, timing=False)
    # short sequences packed 4 / 2 to a 128-row tile (batch fills whole tiles), and a ragged batch that does not pack
    cases["attn_t32_packed"] = lambda: case_attn("attn_t32_packed", 12, 32, 2, True, timing=False)
    cases["attn_t64_packed"] = lambda: case_attn("attn_t64_packed", 6, 64, 3, True, timing=False)
    cases["attn_t64"] = lambda: case_attn("attn_t64", 3, 64, 2, True, timing=False)
    cases["attn_perf_cfg4_char"] = lambda: case_attn("attn_perf_cfg4_char", 8192, 32, 12, True)
    cases["attn_t200"] = lambda: case_attn("attn_t200", 2, 200, 2, True, timing=False)
    # CTA-pair backward (T >= 256): tile counts that leave the pair's second tile partly / entirely past the sequence end
    cases["attn_t300"] = lambda: case_attn("attn_t300", 2, 300, 2, True, timing=False)
    cases["attn_t384"] = lambda: case_attn("attn_t384", 3, 384, 2, True, timing=False)
    cases["attn_t512_many"] = lambda: case_attn("attn_t512_many", 40, 512, 4, True, timing=False)
    cases["attn_spike"] = lambda: case_attn("attn_spike", 2, 320, 2, True, timing=False, spike=True)
    cases["attn_perf_cfg2"] = lambda: case_attn("attn_perf_cfg2", 64, 256, 6, True)
    cases["attn_perf_cfg3"] = lambda: case_attn("attn_perf_cfg3", 32, 1024, 12, True)
    # --- head sizes 32 and 128 (csrc/attn_hd.cu): ragged tails, one position, the rescale path, same tolerances
    for D, H in ((32, 4), (128, 2)):
        for T, B in ((1, 3), (32, 3), (100, 2), (128, 2), (200, 2), (256, 2), (1024, 2)):
            n = f"attn_d{D}_t{T}"
            cases[n] = (lambda n=n, B=B, T=T, H=H, D=D: case_attn(n, B, T, H, True, timing=False, D=D))
        cases[f"attn_d{D}_spike"] = (lambda D=D, H=H: case_attn(f"attn_d{D}_spike", 2, 320, H, True, timing=False, spike=True, D=D))
    for D, H in ((32, 24), (128, 6)):   # the GPT-2-small width (C = 768) at 32 x 1024 tokens
        cases[f"attn_d{D}_perf_c768"] = (lambda D=D, H=H: case_attn(f"attn_d{D}_perf_c768", 32, 1024, H, True, D=D))
    # --- memory-bound kernels
    cases["ln_384"] = lambda: case_layernorm("ln_384", 16384, 384, False)
    cases["ln_768"] = lambda: case_layernorm("ln_768", 32768, 768, False)
    cases["ln_768_bias"] = lambda: case_layernorm("ln_768_bias", 4096, 768, True)
    cases["ln_1000"] = lambda: case_layernorm("ln_1000", 1000, 1000, True)
    cases["ln_resid_768"] = lambda: case_layernorm_resid("ln_resid_768", 32768, 768, False)
    cases["ln_resid_1000_bias"] = lambda: case_layernorm_resid("ln_resid_1000_bias", 1000, 1000, True)
    cases["ce_95"] = lambda: case_ce("ce_95", 32768, 95, 128)
    cases["ce_50304"] = lambda: case_ce("ce_50304", 512, 50304, 50304)
    cases["colsum_768"] = lambda: case_colsum("colsum_768", 5000, 768)
    cases["colsum_narrow_130"] = lambda: case_colsum("colsum_narrow_130", 3001, 130)   # N % 8 != 0: the 4-byte-per-lane kernel
    cases["colsum_perf_cfg4"] = lambda: case_colsum("colsum_perf_cfg4", 262144, 3072, timing=True)
    cases["adamw"] = lambda: case_adamw("adamw", 85813248 // 8 + 3)
    cases["adamw_full"] = lambda: case_adamw("adamw_full", 85813248)
    cases["embed"] = lambda: case_embed("embed", 32, 1024, 768, 95)
    cases["embed_bigv"] = lambda: case_embed("embed_bigv", 4, 256, 384, 5000)
    return cases


def main():
    args = sys.argv[1:]
    if args and args[0] == "--cases":
        import torch  # noqa: F401
        cases = build_cases()
        for n in args[1].split(","):
            print("PROBE_START " + n, flush=True)
            t0 = time.time()
            try:
                res = cases[n]()
            except Exception as e:  # noqa: BLE001
                res = {"case": n, "ok": False, "exception": f"{type(e).__name__}: {e}"}
                if "CUDA" in str(e) or "cuda" in str(e):  # sticky device error: the context is gone
                    res["wall_s"] = round(time.time() - t0, 1)
                    print("PROBE_RESULT " + json.dumps(res), flush=True)
                    sys.exit(3)
            res["wall_s"] = round(time.time() - t0, 1)
            print("PROBE_RESULT " + json.dumps(res), flush=True)
        return
    out_dir = os.environ.get("ABCGPT_PROBE_OUT") or OUT_DIR
    os.makedirs(out_dir, exist_ok=True)
    from ai_music_generation_b200 import _C  # noqa: F401  (no torch import in the parent)
    names = list(build_cases().keys())
    if args:
        names = [n for n in names if any(n.startswith(a) for a in args)]
    results = []
    t00 = time.time()
    remaining = list(names)
    with open(os.path.join(out_dir, "probe.jsonl"), "a") as fout:
        def emit(res):
            results.append(res)
            fout.write(json.dumps(res) + "\n")
            fout.flush()
            print(json.dumps(res), flush=True)
        while remaining:
            try:
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--cases", ",".join(remaining)],
                                   capture_output=True, text=True, timeout=900)
                out, err, rc = p.stdout, p.stderr, p.returncode
            except subprocess.TimeoutExpired as e:
                out = e.stdout.decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
                err, rc = "timeout", -9
            done, started = [], None
            for line in out.splitlines():
                if line.startswith("PROBE_START "):
                    started = line[len("PROBE_START "):]
                elif line.startswith("PROBE_RESULT "):
                    res = json.loads(line[len("PROBE_RESULT "):])
                    emit(res)
                    done.append(res["case"])
                    started = None
            if started is not None:  # the child died inside this case
                emit({"case": started, "ok": False, "crash": True, "rc": rc,
                      "stdout": "\n".join(l for l in out.splitlines() if not l.startswith("PROBE_"))[-1500:],
                      "stderr": err[-1500:]})
                done.append(started)
            if not done:
                emit({"case": remaining[0], "ok": False, "crash": True, "rc": rc, "stderr": err[-1500:]})
                done.append(remaining[0])
            remaining = [n for n in remaining if n not in done]
    nok = sum(1 for r in results if r.get("ok"))
    print(f"PROBE SUMMARY: {nok}/{len(results)} ok in {time.time() - t00:.0f}s; failed: "
          f"{[r['case'] for r in results if not r.get('ok')]}")


if __name__ == "__main__":
    main()
