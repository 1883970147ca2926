"""CPU oracle for the nanoGPT training / sampling step — TEST INFRASTRUCTURE ONLY.

This file is a plain functional restatement (torch CPU tensors, no nn.Module, no CUDA) of the arithmetic on the
reference's hot path.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import it; the product package (ai_music_generation_b200/) never does.

Reference call sites restated (paths relative to /root/reference):
    layer_norm          nanoGPT/model.py:18-27
    attention           nanoGPT/model.py:52-76 (definition = the explicit branch :67-71; SDPA :64 is the same math)
    mlp                 nanoGPT/model.py:87-92 (exact-erf GELU, :83)
    block / forward     nanoGPT/model.py:103-106, :170-193 (tied lm_head :138, ignore_index=-1 :187,
                        last-position logits at inference :190)
    param grouping      nanoGPT/model.py:263-287 (dim >= 2 -> weight decay)
    clip_grad_norm_     nanoGPT/train.py:350-352 (torch/nn/utils/clip_grad.py: coef = max_norm/(norm+1e-6), clamped to 1)
    AdamW               nanoGPT/train.py:354, torch/optim/adam.py single-tensor path with decoupled decay
    generate            nanoGPT/model.py:305-330 (greedy == top_k=1)
    estimate_mfu flops  nanoGPT/model.py:289-298

Pinned (not "parity unpinned"): oracle/make_golden.py imports the UNMODIFIED reference model.py in the build
container, runs it on the inputs below and commits its outputs under tests/golden/; tests/test_oracle_golden.py
checks this restatement against those vectors.  The reference itself ships no tests or golden vectors.

`bf16=True` emulates the dtype flow the reference gets under torch.autocast(bfloat16) (SURVEY.md 3.4): Linear
inputs/weights/outputs rounded to bf16 with fp32 accumulation, attention in bf16, LayerNorm / softmax / loss /
residual stream in fp32.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch
import torch.nn.functional as F


@dataclass
class OracleConfig:
    block_size: int = 1024
    vocab_size: int = 95
    n_layer: int = 12
    n_head: int = 12
    n_embd: int = 768
    dropout: float = 0.0
    bias: bool = False
    activation: str = "gelu"  # "gelu" = nn.GELU() exact erf (nanoGPT/model.py:83); "gelu_tanh" = HF gelu_new (tunesformer/utils.py GPT-2 blocks)


def param_names(cfg: OracleConfig) -> list[str]:
    """state_dict keys in the reference's registration order (lm_head.weight aliases transformer.wte.weight)."""
    names = ["transformer.wte.weight", "transformer.wpe.weight"]
    for i in range(cfg.n_layer):
        p = f"transformer.h.{i}."
        names += [p + "ln_1.weight"] + ([p + "ln_1.bias"] if cfg.bias else [])
        names += [p + "attn.c_attn.weight"] + ([p + "attn.c_attn.bias"] if cfg.bias else [])
        names += [p + "attn.c_proj.weight"] + ([p + "attn.c_proj.bias"] if cfg.bias else [])
        names += [p + "ln_2.weight"] + ([p + "ln_2.bias"] if cfg.bias else [])
        names += [p + "mlp.c_fc.weight"] + ([p + "mlp.c_fc.bias"] if cfg.bias else [])
        names += [p + "mlp.c_proj.weight"] + ([p + "mlp.c_proj.bias"] if cfg.bias else [])
    names += ["transformer.ln_f.weight"] + (["transformer.ln_f.bias"] if cfg.bias else [])
    return names


def param_shapes(cfg: OracleConfig) -> dict[str, tuple[int, ...]]:
    C, V, T = cfg.n_embd, cfg.vocab_size, cfg.block_size
    out = {}
    for n in param_names(cfg):
        if n.endswith("wte.weight"):
            out[n] = (V, C)
        elif n.endswith("wpe.weight"):
            out[n] = (T, C)
        elif "ln_" in n:
            out[n] = (C,)
        elif n.endswith("c_attn.weight"):
            out[n] = (3 * C, C)
        elif n.endswith("c_attn.bias"):
            out[n] = (3 * C,)
        elif n.endswith("attn.c_proj.weight"):
            out[n] = (C, C)
        elif n.endswith("c_fc.weight"):
            out[n] = (4 * C, C)
        elif n.endswith("c_fc.bias"):
            out[n] = (4 * C,)
        elif n.endswith("mlp.c_proj.weight"):
            out[n] = (C, 4 * C)
        else:  # remaining biases of size C
            out[n] = (C,)
    return out


def synthetic_state(cfg: OracleConfig, seed: int = 0) -> dict[str, torch.Tensor]:
    """Closed-form, RNG-free parameters (so fixtures need not store weights): a fixed trigonometric lattice with the
    reference's init scales (std 0.02, residual projections 0.02/sqrt(2L), LayerNorm weights near 1)."""
    sd = {}
    for k, (name, shape) in enumerate(param_shapes(cfg).items()):
        n = math.prod(shape)
        i = torch.arange(n, dtype=torch.float64)
        base = torch.sin(i * (0.37 + 0.011 * k) + 0.5 * k + seed) + 0.5 * torch.cos(i * (1.13 + 0.007 * k) + seed)
        if "ln_" in name and name.endswith("weight"):
            w = 1.0 + 0.1 * base
        elif name.endswith("bias"):
            w = 0.02 * base
        elif name.endswith("c_proj.weight"):
            w = (0.02 / math.sqrt(2 * cfg.n_layer)) * 1.2 * base
        else:
            w = 0.02 * 1.2 * base
        sd[name] = w.to(torch.float32).reshape(shape).clone()
    return sd


def synthetic_tokens(cfg: OracleConfig, batch: int, seqlen: int, seed: int = 0) -> tuple[torch.Tensor, torch.Tensor]:
    """ABC-like token stream without RNG: x from an LCG, y = x shifted by one (next-token targets)."""
    n = batch * (seqlen + 1)
    vals = torch.empty(n, dtype=torch.int64)
    s = 12345 + 7919 * seed
    for i in range(n):
        s = (1103515245 * s + 12345) % 2147483648
        vals[i] = (s >> 8) % cfg.vocab_size
    vals = vals.view(batch, seqlen + 1)
    return vals[:, :-1].contiguous(), vals[:, 1:].contiguous()


# ---------------------------------------------------------------------------------------------------------
def _bf(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(torch.float32)


def _linear(x, w, b, bf16):
    if bf16:  # autocast: operands rounded to bf16, fp32 accumulate, bf16 result
        y = _bf(x) @ _bf(w).t()
        if b is not None:
            y = y + _bf(b)
        return _bf(y)
    y = x @ w.t()
    return y if b is None else y + b


def _layer_norm(x, w, b):
    return F.layer_norm(x, (x.shape[-1],), w, b, 1e-5)


def _drop(x, mask, p, bf16):
    """nn.Dropout with an explicit keep-mask: x * mask / (1 - p), rounded to bf16 when the activation is bf16."""
    if mask is None:
        return x
    y = x * mask.to(x.dtype) / (1.0 - p)
    return _bf(y) if bf16 else y


def _attention(qkv, n_head, bf16, drop_mask=None, p=0.0, key_padding=None):
    B, T, C3 = qkv.shape
    C = C3 // 3
    hs = C // n_head
    q, k, v = qkv.split(C, dim=2)
    q = q.view(B, T, n_head, hs).transpose(1, 2)
    k = k.view(B, T, n_head, hs).transpose(1, 2)
    v = v.view(B, T, n_head, hs).transpose(1, 2)
    if not bf16 and drop_mask is None and key_padding is None:  # same call the reference makes (model.py:64); the explicit form below is its definition (:67-71)
        y = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=True)
        return y.transpose(1, 2).contiguous().view(B, T, C)
    att = (q @ k.transpose(-2, -1)) * (1.0 / math.sqrt(hs))
    mask = torch.ones(T, T, dtype=torch.bool, device=qkv.device).tril()   # qkv's device: the kernel tests run this on the GPU
    att = att.masked_fill(~mask, float("-inf"))
    if key_padding is not None:  # HF attention_mask of TunesFormer's char decoder (tunesformer/utils.py:128-133,152-154): bool [B, T], True = pad key
        att = att.masked_fill(key_padding[:, None, None, :] & ~torch.eye(T, dtype=torch.bool, device=qkv.device)[None, None],
                              float("-inf"))
    att = torch.softmax(att, dim=-1)
    if drop_mask is not None:  # attn_dropout (:70) / SDPA dropout_p (:64) on the probabilities
        att = att * drop_mask.to(att.dtype) / (1.0 - p)
    if bf16:
        att = _bf(att)  # flash kernels feed P to the second matmul in bf16
    y = att @ v
    y = y.transpose(1, 2).contiguous().view(B, T, C)
    return _bf(y) if bf16 else y


def forward(sd, cfg: OracleConfig, idx, targets=None, bf16: bool = False, return_hidden: bool = False, masks=None,
            key_padding=None, inputs_embeds=None, first_embeds=None):
    """(logits, loss) exactly as GPT.forward: full logits with targets, last position only without.

    masks (training with dropout): {'p': float, 'emb': bool [B,T,C], 'attn_p': [L x bool [B,H,T,T]],
    'attn_resid': [L x bool [B,T,C]], 'mlp_resid': [L x bool [B,T,C]]} — the keep-masks nn.Dropout would have drawn."""
    # inputs_embeds [B,T,C]: HF GPT2Model(inputs_embeds=...) (tunesformer/utils.py:102-106); first_embeds [B,C]: the first
    # position's token embedding is replaced (tunesformer/utils.py:146-150)
    B, T = (inputs_embeds.shape[0], inputs_embeds.shape[1]) if inputs_embeds is not None else idx.shape
    assert T <= cfg.block_size
    g = (lambda n: sd.get(n))
    if inputs_embeds is not None:
        tok = inputs_embeds
    else:
        tok = sd["transformer.wte.weight"][idx]
        if first_embeds is not None:
            tok = torch.cat((first_embeds.unsqueeze(1), tok[:, 1:, :]), dim=1)
    x = tok + sd["transformer.wpe.weight"][:T]
    pd = masks["p"] if masks else 0.0
    mk = (lambda name, i=None: None if not masks else (masks[name] if i is None else masks[name][i]))
    x = _drop(x, mk("emb"), pd, False)
    for i in range(cfg.n_layer):
        p = f"transformer.h.{i}."
        h = _layer_norm(x, sd[p + "ln_1.weight"], g(p + "ln_1.bias"))
        qkv = _linear(h, sd[p + "attn.c_attn.weight"], g(p + "attn.c_attn.bias"), bf16)
        a = _attention(qkv, cfg.n_head, bf16, mk("attn_p", i), pd, key_padding)
        x = x + _drop(_linear(a, sd[p + "attn.c_proj.weight"], g(p + "attn.c_proj.bias"), bf16), mk("attn_resid", i), pd, bf16)
        h = _layer_norm(x, sd[p + "ln_2.weight"], g(p + "ln_2.bias"))
        h = _linear(h, sd[p + "mlp.c_fc.weight"], g(p + "mlp.c_fc.bias"), bf16)
        h = F.gelu(h, approximate="tanh") if cfg.activation == "gelu_tanh" else F.gelu(h)
        if bf16:
            h = _bf(h)
        x = x + _drop(_linear(h, sd[p + "mlp.c_proj.weight"], g(p + "mlp.c_proj.bias"), bf16), mk("mlp_resid", i), pd, bf16)
    x = _layer_norm(x, sd["transformer.ln_f.weight"], g("transformer.ln_f.bias"))
    if targets is not None:
        logits = _linear(x, sd["transformer.wte.weight"], None, bf16)
        loss = F.cross_entropy(logits.view(-1, logits.size(-1)).float(), targets.reshape(-1), ignore_index=-1)
    else:
        logits = _linear(x[:, [-1], :], sd["transformer.wte.weight"], None, bf16)
        loss = None
    if return_hidden:
        return logits, loss, x
    return logits, loss


def loss_and_grads(sd, cfg: OracleConfig, idx, targets, bf16: bool = False, loss_scale: float = 1.0, masks=None):
    """loss, logits, {name: grad} via autograd over the functional forward (fp32 master weights)."""
    leaf = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    logits, loss = forward(leaf, cfg, idx, targets, bf16=bf16, masks=masks)
    (loss * loss_scale).backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaf.items()}
    return loss.detach(), logits.detach(), grads


def grad_norm(grads) -> float:
    return math.sqrt(sum(float((g.double() ** 2).sum()) for g in grads.values()))


def clip_coef(total_norm: float, max_norm: float) -> float:
    return min(1.0, max_norm / (total_norm + 1e-6))


def adamw_step(sd, grads, state, *, lr, betas, eps=1e-8, weight_decay=0.1, step: int):
    """In-place AdamW over {name: tensor}; 2-D+ tensors decay, 1-D do not (model.py:270-275)."""
    b1, b2 = betas
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    for k, p in sd.items():
        g = grads[k]
        m = state.setdefault(k + ".m", torch.zeros_like(p))
        v = state.setdefault(k + ".v", torch.zeros_like(p))
        wd = weight_decay if p.dim() >= 2 else 0.0
        p.mul_(1.0 - lr * wd)
        m.lerp_(g, 1.0 - b1)
        v.mul_(b2).addcmul_(g, g, value=1.0 - b2)
        denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
        p.addcdiv_(m, denom, value=-lr / bc1)


def train_steps(sd, cfg, batches, *, lr, betas, weight_decay=0.1, grad_clip=1.0, bf16=False):
    """Runs len(batches) optimizer steps; returns per-step (loss, pre-clip grad norm). Mutates sd."""
    state, out = {}, []
    for step, (x, y) in enumerate(batches, start=1):
        loss, _, grads = loss_and_grads(sd, cfg, x, y, bf16=bf16)
        norm = grad_norm(grads)
        if grad_clip != 0.0:
            c = clip_coef(norm, grad_clip)
            grads = {k: g * c for k, g in grads.items()}
        adamw_step(sd, grads, state, lr=lr, betas=betas, weight_decay=weight_decay, step=step)
        out.append((float(loss), norm))
    return out


@torch.no_grad()
def generate_greedy(sd, cfg: OracleConfig, idx, max_new_tokens: int, bf16: bool = False, return_margins: bool = False):
    """GPT.generate with top_k=1 (argmax), full-context recompute and block_size cropping like the reference."""
    margins = []
    for _ in range(max_new_tokens):
        cond = idx if idx.size(1) <= cfg.block_size else idx[:, -cfg.block_size:]
        logits, _ = forward(sd, cfg, cond, None, bf16=bf16)
        logits = logits[:, -1, :]
        top2 = torch.topk(logits.float(), 2, dim=-1).values
        margins.append(top2[:, 0] - top2[:, 1])
        nxt = torch.argmax(logits, dim=-1, keepdim=True)
        idx = torch.cat((idx, nxt), dim=1)
    if return_margins:
        return idx, torch.stack(margins, dim=1)
    return idx


def sampling_probs(logits: torch.Tensor, temperature: float = 1.0, top_k: int | None = None) -> torch.Tensor:
    """The distribution GPT.generate draws the next token from (model.py:318-324), for last-position logits [B, V] in the
    dtype the model produced them in (bf16 under autocast: the division and the top-k comparison then run in bf16, the
    softmax in fp32 as autocast does).  Returns fp64 probabilities."""
    logits = logits / temperature
    if top_k is not None:
        v, _ = torch.topk(logits, min(top_k, logits.size(-1)))
        logits = logits.clone()
        logits[logits < v[:, [-1]]] = -float("Inf")
    return torch.softmax(logits.double(), dim=-1)


def philox_uniform(seed: int, row: int, counter: int) -> float:
    """Host twin of the uniform csrc/sample.cu draws for (seed, sequence, decode position): Philox4x32-10, key = seed,
    counter = (row, counter lo, counter hi, 0x5A17), first output word >> 8 scaled to [0, 1)."""
    M32 = 0xFFFFFFFF
    k0, k1 = seed & M32, (seed >> 32) & M32
    c0, c1, c2, c3 = row & M32, counter & M32, (counter >> 32) & M32, 0x5A17
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        hi0, lo0, hi1, lo1 = p0 >> 32, p0 & M32, p1 >> 32, p1 & M32
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return (c0 >> 8) / 16777216.0


def inverse_cdf_token(probs: torch.Tensor, u: float, eps: float = 0.0) -> set[int]:
    """Token(s) the inverse-CDF draw may return for the uniform u: the smallest i with cumsum(p)_i > u.  eps > 0 widens the
    comparison by the fp32 rounding of the device's running sum (returns every token whose CDF interval is within eps of u)."""
    cdf = torch.cumsum(probs.double(), dim=-1)
    lo = torch.cat((torch.zeros(1, dtype=torch.float64), cdf[:-1]))
    ok = (probs > 0) & (lo - eps <= u) & (u < cdf + eps)
    return set(torch.nonzero(ok).flatten().tolist())


def num_params(cfg: OracleConfig, non_embedding: bool = True) -> int:
    n = sum(math.prod(s) for s in param_shapes(cfg).values())
    if non_embedding:
        n -= cfg.block_size * cfg.n_embd
    return n


def flops_per_token(cfg: OracleConfig) -> int:
    """6N + 12 L H Q T (model.py:293-296)."""
    return 6 * num_params(cfg) + 12 * cfg.n_layer * cfg.n_head * (cfg.n_embd // cfg.n_head) * cfg.block_size
