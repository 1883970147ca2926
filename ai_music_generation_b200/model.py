"""GPT(GPTConfig) — drop-in for the reference's nanoGPT/model.py on B200 (sm_100a).

Same call surface as the reference (GPTConfig :108-116, GPT.forward :170-193, configure_optimizers :263-287,
generate :305-330, estimate_mfu :289-303, crop_block_size :195-204, get_num_params :150-160) and the same
parameter names / shapes / init RNG consumption, so reference checkpoints load and `train.py` / `sample.py` /
`bench.py` style drivers run unchanged.  What differs is everything underneath:

  * parameters live in ONE flat fp32 arena (and gradients, Adam moments and the bf16 GEMM-operand shadow in
    matching arenas); nn.Parameters are views, so clip + AdamW are single fused launches and DDP buckets are
    plain slices (no copies);
  * GPT.forward / backward are a fixed launch plan of hand-written sm_100a kernels from libabcgpt.so over
    pre-allocated activation buffers (no per-step allocation, CUDA-graph capturable), exposed to autograd as
    one Function: `loss.backward()` fills `.grad` on `model.parameters()` exactly like the reference;
  * the dtype flow is the one the reference gets under torch.autocast(bfloat16) (fp32 residual stream,
    LayerNorm and loss; bf16 GEMM/attention operands with fp32 accumulation), whether or not the caller
    opens an autocast context.

There is no CPU or eager-PyTorch fallback: a missing extension or a non-CUDA tensor raises.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass

import torch
import torch.nn as nn

from . import _C, ops
from .dropout import site_key
from .optim import FusedAdamW


@dataclass
class GPTConfig:
    block_size: int = 1024
    vocab_size: int = 50304
    n_layer: int = 12
    n_head: int = 12
    n_embd: int = 768
    dropout: float = 0.0
    bias: bool = True
    # not in the reference's GPTConfig (model.py:108-116): "gelu" = nn.GELU() exact erf (the reference, default);
    # "gelu_tanh" = HF "gelu_new", the activation of the GPT-2 blocks TunesFormer is built from (tunesformer/utils.py:84-154)
    activation: str = "gelu"


# The sub-modules below only own parameters (names / shapes / init identical to the reference); the arithmetic of
# the whole network is scheduled by GPT._forward_plan / GPT._backward_plan.
class LayerNorm(nn.Module):
    def __init__(self, ndim, bias):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(ndim))
        self.bias = nn.Parameter(torch.zeros(ndim)) if bias else None


class CausalSelfAttention(nn.Module):
    def __init__(self, config):
        super().__init__()
        assert config.n_embd % config.n_head == 0
        self.c_attn = nn.Linear(config.n_embd, 3 * config.n_embd, bias=config.bias)
        self.c_proj = nn.Linear(config.n_embd, config.n_embd, bias=config.bias)
        self.attn_dropout = nn.Dropout(config.dropout)
        self.resid_dropout = nn.Dropout(config.dropout)
        self.n_head, self.n_embd, self.dropout = config.n_head, config.n_embd, config.dropout


class MLP(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.c_fc = nn.Linear(config.n_embd, 4 * config.n_embd, bias=config.bias)
        self.gelu = nn.GELU()
        self.c_proj = nn.Linear(4 * config.n_embd, config.n_embd, bias=config.bias)
        self.dropout = nn.Dropout(config.dropout)


class Block(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.ln_1 = LayerNorm(config.n_embd, bias=config.bias)
        self.attn = CausalSelfAttention(config)
        self.ln_2 = LayerNorm(config.n_embd, bias=config.bias)
        self.mlp = MLP(config)


def _round_up(x, m):
    return (x + m - 1) // m * m


HEAD_SIZES = (32, 64, 128)   # head sizes the sm_100a attention kernels are built for (csrc/attn.cu: 64, csrc/attn_hd.cu: 32, 128)


def head_size_of(cfg: GPTConfig) -> int:
    """n_embd // n_head; raises ValueError unless n_embd splits evenly into heads of a supported size."""
    if cfg.n_head <= 0 or cfg.n_embd % cfg.n_head != 0:
        raise ValueError(f"n_embd ({cfg.n_embd}) must be a multiple of n_head ({cfg.n_head})")
    D = cfg.n_embd // cfg.n_head
    if D not in HEAD_SIZES:
        raise ValueError(f"head size n_embd // n_head = {D} is not supported: the sm_100a attention kernels support head sizes "
                         f"{', '.join(map(str, HEAD_SIZES))}")
    return D


class _Buffers:
    """Activation / scratch buffers for one (B, T) shape, allocated once and reused every step."""

    def __init__(self, cfg: GPTConfig, B: int, T: int, device, keep_activations: bool):
        M, C, L, H = B * T, cfg.n_embd, cfg.n_layer, cfg.n_head
        bf, f32 = torch.bfloat16, torch.float32
        e = lambda *s, dt=bf: torch.empty(*s, device=device, dtype=dt)  # noqa: E731
        nl = L if keep_activations else 1
        self.B, self.T, self.M = B, T, M
        self.keep = keep_activations
        self.Vpad = _round_up(cfg.vocab_size, 128) if cfg.vocab_size <= 1024 else _round_up(cfg.vocab_size, 8)
        self.x = [e(M, C, dt=f32) for _ in range(nl + 1)]        # residual stream at each block input (+ final)
        self.xmid = [e(M, C, dt=f32) for _ in range(nl)]         # after the attention residual
        self.ln1 = [e(M, C) for _ in range(nl)]
        self.ln2 = [e(M, C) for _ in range(nl)]
        self.stat = [e(4, M, dt=f32) for _ in range(nl)]          # mean1, rstd1, mean2, rstd2
        self.qkv = [e(M, 3 * C) for _ in range(nl)]
        self.att = [e(M, C) for _ in range(nl)]
        self.lse = [e(B, H, T, dt=f32) for _ in range(nl)]
        self.h = [e(M, 4 * C) for _ in range(nl)]
        self.g = [e(M, 4 * C) for _ in range(nl)]
        self.lnf = e(M, C)
        self.ybr = e(M, C)                                        # bf16 output of attn.c_proj on its way into the fused add + ln_2
        self.statf = e(2, M, dt=f32)
        self.logits = e(M, self.Vpad)
        self.row_loss = e(M, dt=f32)
        self.sum_count = e(2, dt=f32)
        self.loss = e(1, dt=f32)
        self.last_logits = e(B, self.Vpad)
        self.idx = torch.empty(B, T, device=device, dtype=torch.int64)   # static copies of the inputs: recorded launch plans
        self.tgt = torch.empty(B, T, device=device, dtype=torch.int64)   # hold raw pointers
        self.gl = e(1, dt=f32)
        self.hidden = None   # fp32 ln_f output, allocated on first use by the hierarchical (inputs_embeds) path
        self.plans = {}
        self.gen = 0         # bumped by every forward into these buffers; an autograd node remembers the value it saw
        if keep_activations:
            self.dx = [e(M, C, dt=f32) for _ in range(2)]
            self.dxb = e(M, C)
            self.dxb2 = e(M, C)   # second bf16 stream-gradient buffer: ln_2's output, so that side-stream wgrads of dxb stay valid
            self.dln = e(M, C)
            self.datt = e(M, C)
            self.dqkv = e(M, 3 * C)
            self.dh = e(M, 4 * C)
            self.delta = e(B, H, T, dt=f32)
            self.dlogits = e(M, self.Vpad)


class _DecodeState:
    """Buffers of the single-token decode path: the per-layer head-major cache of c_attn outputs and the [B, *] row buffers of
    one step.  Head size 64: [B, 3H, Tmax, 64] (q | k | v heads, written by the head-strided GEMM); other head sizes:
    [B, 2H, Tmax, D] (k | v heads, appended by the decode kernel from the [B, 3C] row `qkv`)."""

    def __init__(self, cfg: GPTConfig, B: int, Tmax: int, device):
        C, L = cfg.n_embd, cfg.n_layer
        bf, f32 = torch.bfloat16, torch.float32
        e = lambda *s, dt=bf: torch.empty(*s, device=device, dtype=dt)  # noqa: E731
        self.B, self.Tmax = B, Tmax
        self.D = head_size_of(cfg)
        self.Vpad = _round_up(cfg.vocab_size, 128) if cfg.vocab_size <= 1024 else _round_up(cfg.vocab_size, 8)
        self.cache = [e(B, Tmax * (3 if self.D == 64 else 2) * C) for _ in range(L)]
        self.qkv = e(B, 3 * C) if self.D != 64 else None
        self.x = [e(B, C, dt=f32) for _ in range(2)]
        self.ln = e(B, C)
        self.att = e(B, C)
        self.h = e(B, 4 * C)
        self.g = e(B, 4 * C)
        self.stat = e(2, B, dt=f32)
        self.logits = e(B, self.Vpad)
        self.col = torch.zeros(Tmax + 1, B, device=device, dtype=torch.int64)  # token column t = contiguous int64 [B]
        # set by callers of the other input / output modes of GPT._decode_step (hierarchical decoders): fp32 [B, C] input rows
        # (`inp` "first" / "embed"), fp32 [B, C] ln_f output rows (`hidden`), and the (seed, counter base, row ids) device
        # buffers of the ("top_p", ...) sampling head.  Recorded launch lists hold their addresses.
        self.emb = None
        self.hidden = None
        self.sampler = None
        self.plans = {}
        self.affine = {}   # (flags) -> (t0, recorded plan at t0, per-launch argument deltas per position)


def _check_generation(ctx):
    """Activations live in per-(B, T) buffers that every training forward overwrites.  The reference (plain autograd) lets a
    caller run two forwards and differentiate both afterwards (`(l1 + l2).backward()`); here that would differentiate loss 1
    through forward 2's activations, so it raises instead of returning a wrong gradient.  forward/backward pairs in sequence —
    the training loop, gradient accumulation — are unaffected."""
    if ctx.gen != ctx.bufs.gen:
        raise RuntimeError(
            "GPT: backward() of a forward whose activations have been overwritten by a later forward of the same (batch, "
            "sequence) shape.  Call loss.backward() before the next training forward (gradient accumulation does exactly "
            "that), or run the extra forward under torch.no_grad().")


class _GPTStep(torch.autograd.Function):
    """One autograd node for the whole network: forward launches the forward plan, backward the backward plan."""

    @staticmethod
    def forward(ctx, anchor, model, idx, targets):
        bufs = model._forward_plan(idx, targets, keep_activations=True)
        if bufs.drop[0] == 0.0 and model._plan_cache_enabled:
            idx, targets = bufs.idx, bufs.tgt  # the plan staged the inputs into its static buffers
        ctx.model, ctx.bufs, ctx.idx, ctx.targets, ctx.drop = model, bufs, idx, targets, bufs.drop
        ctx.gen = bufs.gen
        B, T = idx.shape
        logits = bufs.logits.view(B, T, -1)[:, :, : model.config.vocab_size]
        ctx.mark_non_differentiable(logits)
        # the loss is returned as its own 4-byte tensor (`losses.append(loss)` across steps keeps every value); the logits
        # stay a view of the per-shape activation buffer: valid until the next forward of the same shape
        return logits, bufs.loss.view(()).clone()

    @staticmethod
    def backward(ctx, _grad_logits, grad_loss):
        _check_generation(ctx)
        ctx.model._backward_plan(ctx.bufs, ctx.idx, ctx.targets, grad_loss, ctx.drop)
        return None, None, None, None


class _GPTEmbedsStep(torch.autograd.Function):
    """The same launch plans for a decoder whose input embeddings come from another network (hierarchical models,
    SURVEY.md 8f N1).  mode 1: x_in = inputs_embeds [B,T,C]; mode 2: x_in = the replacement of the first position's
    embedding [B,C] next to token ids.  Returns (loss, fp32 ln_f output); either may be unused."""

    @staticmethod
    def forward(ctx, anchor, model, x_in, idx, targets, want_hidden, mode):
        bufs = model._forward_plan(idx, targets, keep_activations=True, embeds=x_in if mode == 1 else None,
                                   first=x_in if mode == 2 else None, want_hidden=want_hidden)
        B, T, C = bufs.B, bufs.T, model.config.n_embd
        idx_b = None
        if mode == 2:  # the wte gradient must skip position 0 (its embedding was replaced): abcgpt_embed_bwd skips ids < 0
            idx_b = idx.clone()
            idx_b[:, 0] = -1
        ctx.model, ctx.bufs, ctx.idx, ctx.targets, ctx.drop = model, bufs, idx_b, targets, bufs.drop
        ctx.gen = bufs.gen
        ctx.want_hidden, ctx.mode, ctx.shape = want_hidden, mode, (B, T, C)
        loss = bufs.loss.view(()).clone() if targets is not None else torch.zeros((), device=x_in.device)
        hidden = bufs.hidden.view(B, T, C).clone() if want_hidden else torch.zeros(0, device=x_in.device)
        return loss, hidden

    @staticmethod
    def backward(ctx, grad_loss, grad_hidden):
        B, T, C = ctx.shape
        _check_generation(ctx)
        d_hidden = grad_hidden.reshape(B * T, C).float() if ctx.want_hidden and ctx.targets is None else None
        dx = ctx.model._backward_plan(ctx.bufs, ctx.idx, ctx.targets, grad_loss, ctx.drop, d_hidden=d_hidden, mode=ctx.mode)
        gx = dx.view(B, T, C).clone() if ctx.mode == 1 else dx.view(B, T, C)[:, 0, :].clone()
        return None, None, gx, None, None, None, None


class GPT(nn.Module):
    def __init__(self, config: GPTConfig):
        super().__init__()
        assert config.vocab_size is not None and config.block_size is not None
        self._head_size = head_size_of(config)
        assert config.activation in ("gelu", "gelu_tanh"), config.activation
        self._act = ops.ACT_TANH if config.activation == "gelu_tanh" else 0
        self.config = config
        self.transformer = nn.ModuleDict(dict(
            wte=nn.Embedding(config.vocab_size, config.n_embd),
            wpe=nn.Embedding(config.block_size, config.n_embd),
            drop=nn.Dropout(config.dropout),
            h=nn.ModuleList([Block(config) for _ in range(config.n_layer)]),
            ln_f=LayerNorm(config.n_embd, bias=config.bias),
        ))
        self.lm_head = nn.Linear(config.n_embd, config.vocab_size, bias=False)
        self.transformer.wte.weight = self.lm_head.weight  # weight tying (model.py:138)
        self.apply(self._init_weights)
        for pn, p in self.named_parameters():
            if pn.endswith("c_proj.weight"):
                torch.nn.init.normal_(p, mean=0.0, std=0.02 / math.sqrt(2 * config.n_layer))
        self._arena = None
        self._bufs = {}
        self._shadow_fresh = False
        self._pending_clip = None
        self._plan_cache_enabled = os.environ.get("ABCGPT_PLAN_CACHE", "1") != "0"   # "0": derive every launch afresh (A/B runs)
        # weight-gradient GEMMs on a second stream for steps made of short kernels (see _backward_plan_impl)
        self._wgrad_side = os.environ.get("ABCGPT_WGRAD_SIDE", "auto")   # "0" / "1" force it off / on
        self._next_dropout_seed = None  # tests / reproducibility: force the seed of the next training forward
        self.last_dropout_seed = None
        self.require_backward_grad_sync = True
        self._grad_sync = None  # set by ddp.DDP
        self._flatten()
        print("number of parameters: %.2fM" % (self.get_num_params() / 1e6,))

    # ------------------------------------------------------------------------------------------------------
    # parameter arena
    # ------------------------------------------------------------------------------------------------------
    def _ordered_params(self):
        """decay (dim >= 2) tensors first in layer order, then the 1-D tensors; each start 16-byte aligned."""
        named = list(self.named_parameters())
        return [(n, p) for n, p in named if p.dim() >= 2] + [(n, p) for n, p in named if p.dim() < 2]

    def _flatten(self):
        params = self._ordered_params()
        device = params[0][1].device
        offs, total = [], 0
        for _, p in params:
            offs.append(total)
            total += _round_up(p.numel(), 8)
        n_decay = sum(_round_up(p.numel(), 8) for _, p in params if p.dim() >= 2)
        # the lm_head GEMMs read the vocabulary matrix as a [Vpad, C] operand (V rounded up to the 128-row tile): the rows past
        # V must lie inside the arena (they produce the padding logits columns, which every consumer ignores)
        cfg = self.config
        vpad = _round_up(cfg.vocab_size, 128) if cfg.vocab_size <= 1024 else _round_up(cfg.vocab_size, 8)
        for (_, p), o in zip(params, offs):
            if p is self.lm_head.weight:
                total = max(total, o + vpad * cfg.n_embd)
        flat = torch.zeros(total, device=device, dtype=torch.float32)
        for (_, p), o in zip(params, offs):
            flat[o:o + p.numel()].copy_(p.data.reshape(-1).to(torch.float32))
            p.data = flat[o:o + p.numel()].view(p.shape)
            p.grad = None
        self._arena = {
            "flat": flat, "offs": offs, "names": [n for n, _ in params], "params": [p for _, p in params],
            "n_decay": n_decay, "total": total, "grad": None, "shadow": None,
        }
        self._bufs = {}
        self._shadow_fresh = False

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        if self._arena is not None:
            self._flatten()  # .to()/.cuda()/.float() re-point parameters: rebuild the arena on the new device
        return out

    def load_state_dict(self, state_dict, strict=True, assign=False):
        out = super().load_state_dict(state_dict, strict=strict, assign=False)
        self._shadow_fresh = False
        return out

    def _view(self, which, name):
        a = self._arena
        i = a["names"].index(name)
        p = a["params"][i]
        return a[which][a["offs"][i]:a["offs"][i] + p.numel()].view(p.shape)

    def _ensure_device_state(self):
        a = self._arena
        if not a["flat"].is_cuda:
            raise _C.AbcgptError("GPT: parameters are not on a CUDA device (there is no CPU path; call model.to('cuda'))")
        if a["shadow"] is None:
            a["shadow"] = torch.empty(a["total"], device=a["flat"].device, dtype=torch.bfloat16)
            self._shadow_fresh = False
        if a["grad"] is None:
            a["grad"] = torch.zeros(a["total"], device=a["flat"].device, dtype=torch.float32)
        # The GEMMs read the bf16 shadow.  FusedAdamW rewrites it itself; ANY other in-place edit of a parameter (p.data.copy_,
        # re-initialisation, an EMA swap, a foreign optimizer) bumps that parameter's version counter, which is how a stale
        # shadow is detected here (one recast launch).  Writes through `p.data` carry no version bump in PyTorch: after those
        # call mark_weights_dirty().
        ver = sum(p._version for p in a["params"]) + a["flat"]._version
        if not self._shadow_fresh or ver != a.get("param_versions"):
            ops.cast_bf16(a["flat"], a["shadow"])
            self._shadow_fresh = True
            a["param_versions"] = ver

    def mark_weights_dirty(self):
        """The fp32 parameters were changed behind the module's back: recast the bf16 GEMM-operand copy before the next use."""
        self._shadow_fresh = False

    def _layer_tensors(self):
        """Per-layer (fp32 master, bf16 shadow, grad) views, cached per arena."""
        a = self._arena
        if "layers" in a and a["layers_for"] == (a["shadow"].data_ptr(), a["grad"].data_ptr()):
            return a["layers"]
        cfg = self.config

        def tri(name, need_shadow=True):
            if name not in a["names"]:
                return None
            return (self._view("flat", name), self._view("shadow", name) if need_shadow else None, self._view("grad", name))

        layers = []
        for i in range(cfg.n_layer):
            p = f"transformer.h.{i}."
            layers.append({k: tri(p + k, need_shadow=k.endswith("weight") and "ln_" not in k) for k in (
                "ln_1.weight", "ln_1.bias", "attn.c_attn.weight", "attn.c_attn.bias", "attn.c_proj.weight",
                "attn.c_proj.bias", "ln_2.weight", "ln_2.bias", "mlp.c_fc.weight", "mlp.c_fc.bias", "mlp.c_proj.weight",
                "mlp.c_proj.bias")})
        wte_name = "lm_head.weight" if "lm_head.weight" in a["names"] else "transformer.wte.weight"
        top = {"wte": tri(wte_name), "wpe": tri("transformer.wpe.weight", need_shadow=False),
               "ln_f.weight": tri("transformer.ln_f.weight", False), "ln_f.bias": tri("transformer.ln_f.bias", False)}
        a["layers"], a["top"] = layers, top
        a["layers_for"] = (a["shadow"].data_ptr(), a["grad"].data_ptr())
        return layers

    # ------------------------------------------------------------------------------------------------------
    # launch plans
    # ------------------------------------------------------------------------------------------------------
    def _act_buffers(self, B, T, keep):
        key = (B, T, keep)
        if key not in self._bufs:
            if not keep:  # inference shapes come and go (generate with a growing context): keep only a few of them
                stale = [k for k in self._bufs if len(k) == 3 and k[2] is False]
                for k in stale[:-3]:
                    del self._bufs[k]
            self._bufs[key] = _Buffers(self.config, B, T, self._arena["flat"].device, keep)
        return self._bufs[key]

    # Programmatic dependent launch pays when the kernels of a step are short (baby GPT, 16 k tokens x 384: 3.02 -> 2.88 ms per
    # step) and costs when every kernel fills the GPU for 25-400 us (GPT-2-small shape at 32 k tokens: -1.8 %), see DESIGN 4.5
    _PDL_MAX_WORK = 8 * 1024 * 1024   # tokens x n_embd

    @staticmethod
    def _store_plan(bufs, plan_key, keys, p_drop):
        """Keep a freshly recorded plan; with dropout on it is only reusable if its key sites could be identified."""
        plan = ops.end_record()
        patches = ops.key_patches(plan, keys) if p_drop > 0.0 else []
        if patches is not None:
            bufs.plans[plan_key] = (plan, patches)

    def _forward_plan(self, idx, targets, keep_activations, embeds=None, first=None, want_hidden=False):
        src = idx if idx is not None else embeds
        pdl = src.shape[0] * src.shape[1] * self.config.n_embd <= self._PDL_MAX_WORK
        if not pdl:
            return self._forward_plan_impl(idx, targets, keep_activations, embeds, first, want_hidden)
        ops.set_pdl(True)
        try:
            return self._forward_plan_impl(idx, targets, keep_activations, embeds, first, want_hidden)
        finally:
            ops.set_pdl(False)

    def _backward_plan(self, bufs, idx, targets, grad_loss, drop, d_hidden=None, mode=0):
        pdl = bufs.B * bufs.T * self.config.n_embd <= self._PDL_MAX_WORK
        if not pdl:
            return self._backward_plan_impl(bufs, idx, targets, grad_loss, drop, d_hidden, mode)
        ops.set_pdl(True)
        try:
            return self._backward_plan_impl(bufs, idx, targets, grad_loss, drop, d_hidden, mode)
        finally:
            ops.set_pdl(False)

    def _forward_plan_impl(self, idx, targets, keep_activations, embeds=None, first=None, want_hidden=False):
        """embeds (fp32 [B,T,C]): the decoder is fed embeddings from another network (HF inputs_embeds) instead of token ids;
        first (fp32 [B,C]): token ids, but the first position's embedding is replaced (TunesFormer char decoder);
        want_hidden: also keep the fp32 ln_f output in bufs.hidden (HF last_hidden_state)."""
        cfg = self.config
        # Dropout (model.py:39-40,85,129 + SDPA dropout_p :64): counter-based masks, one key per site, derived from a seed
        # drawn from torch's CPU generator for every forward (reproducible under torch.manual_seed); the backward plan
        # regenerates the masks from the same keys.  site 0 = embedding, block l: 1+3l probs, 2+3l attn resid, 3+3l MLP.
        p_drop = float(cfg.dropout) if self.training else 0.0
        if p_drop > 0.0:
            seed = self._next_dropout_seed if self._next_dropout_seed is not None else int(torch.randint(0, 2 ** 31 - 1, (1,)).item())
            self._next_dropout_seed = None
            keys = [site_key(seed, i) for i in range(1 + 3 * cfg.n_layer)]
        else:
            seed, keys = None, [0] * (1 + 3 * cfg.n_layer)
        src = embeds if embeds is not None else idx
        if not src.is_cuda:
            raise _C.AbcgptError("GPT.forward: inputs must be CUDA tensors (there is no CPU path)")
        self._ensure_device_state()
        layers = self._layer_tensors()
        top = self._arena["top"]
        B, T = src.shape[0], src.shape[1]
        assert T <= cfg.block_size, f"Cannot forward sequence of length {T}, block size is only {cfg.block_size}"
        bufs = self._act_buffers(B, T, keep_activations)
        bufs.gen += 1
        C, H, V = cfg.n_embd, cfg.n_head, cfg.vocab_size
        if idx is not None:
            idx = idx.contiguous()
        bufs.drop = (p_drop, keys, seed)
        self.last_dropout_seed = seed
        # Launch-plan cache: with dropout off every argument of every launch is static (arena views, per-shape buffers,
        # the stream), so the plan is recorded once and replayed; inputs are staged into static buffers.
        plan_key = None
        if self._plan_cache_enabled and embeds is None and first is None and not want_hidden:
            bufs.idx.copy_(idx)
            idx = bufs.idx
            if targets is not None:
                bufs.tgt.copy_(targets)
                targets = bufs.tgt
            # with dropout on, the per-site keys are the only arguments that change between steps: patched at replay
            plan_key = ("fwd", targets is not None, torch.cuda.current_stream().cuda_stream, p_drop)
            plan = bufs.plans.get(plan_key)
            if plan is not None:
                ops.replay(plan[0], plan[1], keys)
                return bufs
            ops.begin_record()
        if embeds is not None:
            if p_drop != 0.0:
                raise _C.AbcgptError("inputs_embeds path: embedding dropout is not implemented (use dropout=0)")
            ops.add_pos(embeds.contiguous().view(B * T, C), top["wpe"][0], bufs.x[0], T)
        else:
            ops.embed_fwd(idx, top["wte"][0], top["wpe"][0], bufs.x[0], T, drop_p=p_drop, drop_key=keys[0])
            if first is not None:
                if p_drop != 0.0:
                    raise _C.AbcgptError("first-embedding path: embedding dropout is not implemented (use dropout=0)")
                ops.set_first_pos(first.contiguous(), top["wpe"][0], bufs.x[0], T)
        for li, lw in enumerate(layers):
            k = li if keep_activations else 0
            x_in, x_out = bufs.x[k], bufs.x[k + 1] if keep_activations else bufs.x[0]
            st = bufs.stat[k]
            b = lambda name: None if lw[name] is None else lw[name][0]  # noqa: E731
            ops.layernorm_fwd(x_in, lw["ln_1.weight"][0], b("ln_1.bias"), bufs.ln1[k], st[0], st[1])
            ops.gemm(bufs.ln1[k], lw["attn.c_attn.weight"][1], epilogue=ops.EPI_BF16, out=bufs.qkv[k], bias=b("attn.c_attn.bias"))
            ops.attn_fwd(bufs.qkv[k], bufs.att[k], bufs.lse[k], B, T, H, drop_p=p_drop, drop_key=keys[1 + 3 * li],
                         head_size=self._head_size)
            # attention branch: the K = 768 projection with the residual add in its epilogue was bound by its fp32 residual
            # loads (0.080 ms against 0.038 ms of HBM time at cfg3); the add rides on the LayerNorm pass that follows instead
            # (x_mid = x + drop(c_proj(att)), ln_2(x_mid) in one kernel; the bf16 branch output mostly stays in L2 in between)
            ops.gemm(bufs.att[k], lw["attn.c_proj.weight"][1], epilogue=ops.EPI_BF16, out=bufs.ybr, bias=b("attn.c_proj.bias"))
            ops.layernorm_fwd_resid(x_in, bufs.ybr, bufs.xmid[k], lw["ln_2.weight"][0], b("ln_2.bias"), bufs.ln2[k], st[2], st[3],
                                    drop_p=p_drop, drop_key=keys[2 + 3 * li])
            ops.gemm(bufs.ln2[k], lw["mlp.c_fc.weight"][1], epilogue=ops.EPI_GELU | self._act, out=bufs.h[k], out2=bufs.g[k],
                     bias=b("mlp.c_fc.bias"))
            ops.gemm(bufs.g[k], lw["mlp.c_proj.weight"][1], epilogue=ops.EPI_RESID, out=x_out, aux=bufs.xmid[k],
                     bias=b("mlp.c_proj.bias"), drop_p=p_drop, drop_key=keys[3 + 3 * li])
        x_last = bufs.x[cfg.n_layer] if keep_activations else bufs.x[0]
        lnf_b = None if top["ln_f.bias"] is None else top["ln_f.bias"][0]
        if want_hidden and bufs.hidden is None:
            bufs.hidden = torch.empty(B * T, C, device=bufs.lnf.device, dtype=torch.float32)
        ops.layernorm_fwd(x_last, top["ln_f.weight"][0], lnf_b, bufs.lnf, bufs.statf[0], bufs.statf[1],
                          y_f32=bufs.hidden if want_hidden else None)
        wte_bf16 = top["wte"][1]
        if want_hidden and targets is None:
            pass  # a decoder without a head (TunesFormer's patch level): the caller reads bufs.hidden
        elif targets is not None:
            ops.gemm(bufs.lnf, wte_bf16, N=bufs.Vpad, epilogue=ops.EPI_BF16, out=bufs.logits)
            ops.ce_fwd(bufs.logits, targets.contiguous().view(-1), bufs.row_loss, bufs.sum_count, bufs.loss, V)
        else:  # last position only (model.py:190): strided A operand, no gather copy
            a = bufs.lnf.view(B, T * C)[:, (T - 1) * C:]
            ops.gemm(a, wte_bf16, M=B, N=bufs.Vpad, K=C, epilogue=ops.EPI_BF16, out=bufs.last_logits)
        if plan_key is not None:
            self._store_plan(bufs, plan_key, keys, p_drop)
        return bufs

    def _backward_plan_impl(self, bufs, idx, targets, grad_loss, drop, d_hidden=None, mode=0):
        """mode 0: token ids in (the reference path); 1: inputs_embeds in (returns the fp32 gradient w.r.t. x[0], which is the
        gradient of the embeddings); 2: token ids with a replaced first embedding (`idx` must carry -1 at position 0 so that
        the wte gradient skips it; returns the same buffer, row 0 of every sequence is the gradient of `first`).
        d_hidden (fp32 [M,C]): gradient of the ln_f output when the decoder has no head."""
        cfg = self.config
        p_drop, keys, _ = drop
        a = self._arena
        layers = self._layer_tensors()
        top = a["top"]
        B, T, M = bufs.B, bufs.T, bufs.M
        C, H, V = cfg.n_embd, cfg.n_head, cfg.vocab_size
        params = a["params"]
        if params[0].grad is None:  # first micro-step after zero_grad(set_to_none=True): start from zero
            a["grad"].zero_()
            for p, o in zip(params, a["offs"]):
                p.grad = a["grad"][o:o + p.numel()].view(p.shape)
        if targets is not None:
            bufs.gl.copy_(grad_loss.reshape(1))
        gl = bufs.gl
        tflat = targets.contiguous().view(-1) if targets is not None else None
        sync = self._grad_sync if (self._grad_sync is not None and self.require_backward_grad_sync) else None
        if self._grad_sync is not None:
            self._grad_sync.norm_fresh = False   # the arena is about to change; a fused exchange at the end sets it again
        # like programmatic dependent launch, the second stream pays where kernels are short (baby GPT 2.66 -> 2.57 ms per step);
        # at the GPT-2-small shape with 32 k tokens the step is energy-bound and it measured neutral (24.54 / 24.61 vs 24.67 / 24.65 ms)
        side = None
        if (self._wgrad_side == "1" or (self._wgrad_side == "auto" and bufs.B * bufs.T * cfg.n_embd <= self._PDL_MAX_WORK)) and not ops.profiling():
            side = ops.side_stream()
        plan_key = None
        if (self._plan_cache_enabled and mode == 0 and d_hidden is None and targets is not None
                and targets.data_ptr() == bufs.tgt.data_ptr()):
            plan_key = ("bwd", sync is not None, torch.cuda.current_stream().cuda_stream, side is not None, p_drop)
            plan = bufs.plans.get(plan_key)
            if plan is not None:
                ops.replay(plan[0], plan[1], keys)
                return
            ops.begin_record()
        wte, wte_bf16, dwte = top["wte"]
        if targets is not None:
            ops.ce_bwd(bufs.logits, tflat, bufs.sum_count, gl, bufs.dlogits, V)
            # lm_head: dW[V,C] += dlogits^T lnf ; d(lnf) = dlogits W
            ops.gemm(bufs.dlogits, bufs.lnf, a_mn=True, b_mn=True, M=V, N=C, K=M, epilogue=ops.EPI_F32_RED, out=dwte)
            ops.gemm(bufs.dlogits, wte_bf16, b_mn=True, M=M, N=C, K=V, epilogue=ops.EPI_BF16, out=bufs.dln)
            if d_hidden is not None:
                raise _C.AbcgptError("backward: a loss head AND a hidden-state gradient on the same decoder is not implemented")
        else:
            ops.cast_bf16(d_hidden.contiguous().view(-1), bufs.dln.view(-1))
        dx, dx_other = bufs.dx[0], bufs.dx[1]
        gw = lambda t: None if t is None else t[2]  # noqa: E731
        # Weight-gradient GEMMs (and bias column sums) depend on nothing downstream of them in the backward: with `side` they go
        # to a second stream and fill the prologue / tail / LayerNorm phases of the dgrad chain.  Ordering (abcgpt_event_*):
        # FORK = the side stream waits for the producer of the wgrad's operand; J0..J3 = the main stream waits, right before it
        # overwrites a buffer, for the side-stream GEMM that read it (dxb, dh, dxb2, dqkv; the overwrite is most of a layer
        # later, so these waits are normally already satisfied).
        FORK, J0, J1, J2, J3 = 0, 1, 2, 3, 4
        # experiment (ABCGPT_DDP_RELEASE=attn): a layer's gradient bucket is released a few kernels later, so that its exchange runs
        # beside the next layer's attention backward instead of beside that layer's first GEMMs
        release_beside_attn = sync is not None and os.environ.get("ABCGPT_DDP_RELEASE", "layer") == "attn"
        held = None
        main_st = torch.cuda.current_stream()

        def wgrad(dy, xin, wname, jslot):
            if side is not None:
                ops.event_record(FORK)
                ops.event_wait(FORK, side)
                with torch.cuda.stream(side):
                    ops.gemm(dy, xin, a_mn=True, b_mn=True, epilogue=ops.EPI_F32_RED, out=lw[wname + ".weight"][2])
                    if lw[wname + ".bias"] is not None:
                        ops.colsum_bf16(dy, lw[wname + ".bias"][2])
                    ops.event_record(jslot)
            else:
                ops.gemm(dy, xin, a_mn=True, b_mn=True, epilogue=ops.EPI_F32_RED, out=lw[wname + ".weight"][2])
                if lw[wname + ".bias"] is not None:
                    ops.colsum_bf16(dy, lw[wname + ".bias"][2])

        def before_overwrite(jslot):
            if side is not None:
                ops.event_wait(jslot, main_st)

        # every bf16 stream gradient `dxb` is produced already masked for the residual-branch dropout of its consumer
        ops.layernorm_bwd(bufs.dln, bufs.x[cfg.n_layer], top["ln_f.weight"][0], bufs.statf[0], bufs.statf[1], None, dx,
                          bufs.dxb, top["ln_f.weight"][2], gw(top["ln_f.bias"]), drop_p=p_drop,
                          drop_key=keys[3 + 3 * (cfg.n_layer - 1)])
        for li in range(cfg.n_layer - 1, -1, -1):
            lw = layers[li]
            st = bufs.stat[li]
            # ---- MLP: x_out = xmid + c_proj(gelu(c_fc(ln_2(xmid))))
            wgrad(bufs.dxb, bufs.g[li], "mlp.c_proj", J0)
            before_overwrite(J1)
            ops.gemm(bufs.dxb, lw["mlp.c_proj.weight"][1], b_mn=True, epilogue=ops.EPI_DGELU | self._act, out=bufs.dh, aux=bufs.h[li])
            wgrad(bufs.dh, bufs.ln2[li], "mlp.c_fc", J1)
            ops.gemm(bufs.dh, lw["mlp.c_fc.weight"][1], b_mn=True, epilogue=ops.EPI_BF16, out=bufs.dln)
            before_overwrite(J2)
            ops.layernorm_bwd(bufs.dln, bufs.xmid[li], lw["ln_2.weight"][0], st[2], st[3], dx, dx_other, bufs.dxb2,
                              lw["ln_2.weight"][2], gw(lw["ln_2.bias"]), drop_p=p_drop, drop_key=keys[2 + 3 * li])
            dx, dx_other = dx_other, dx
            # ---- attention: xmid = x_in + c_proj(attn(c_attn(ln_1(x_in))))
            wgrad(bufs.dxb2, bufs.att[li], "attn.c_proj", J2)
            ops.gemm(bufs.dxb2, lw["attn.c_proj.weight"][1], b_mn=True, epilogue=ops.EPI_BF16, out=bufs.datt)
            before_overwrite(J3)
            if held is not None:   # the previous layer's bucket goes out beside this layer's attention backward (see below)
                ops.record_callback(lambda li_=held: sync.layer_done(li_))
                held = None
            ops.attn_bwd(bufs.qkv[li], bufs.att[li], bufs.datt, bufs.lse[li], bufs.delta, bufs.dqkv, B, T, H,
                         drop_p=p_drop, drop_key=keys[1 + 3 * li], head_size=self._head_size)
            wgrad(bufs.dqkv, bufs.ln1[li], "attn.c_attn", J3)
            ops.gemm(bufs.dqkv, lw["attn.c_attn.weight"][1], b_mn=True, epilogue=ops.EPI_BF16, out=bufs.dln)
            before_overwrite(J0)
            ops.layernorm_bwd(bufs.dln, bufs.x[li], lw["ln_1.weight"][0], st[0], st[1], dx, dx_other, bufs.dxb,
                              lw["ln_1.weight"][2], gw(lw["ln_1.bias"]), drop_p=p_drop if li > 0 else 0.0,
                              drop_key=keys[3 + 3 * (li - 1)] if li > 0 else 0)
            dx, dx_other = dx_other, dx
            if sync is not None:
                before_overwrite(J3)   # the layer's last wgrad (the side stream runs in order): its gradients are complete
                if release_beside_attn and li > 0:
                    held = li          # released right before the NEXT layer's attention backward
                else:
                    ops.record_callback(lambda li=li: sync.layer_done(li))
        before_overwrite(J3)           # join: everything the side stream was given has finished before the backward returns
        if mode == 1:
            ops.pos_bwd(dx, top["wpe"][2], T)
        else:
            ops.embed_bwd(idx.contiguous().view(-1), dx, dwte, top["wpe"][2], T, drop_p=p_drop, drop_key=keys[0])
        if sync is not None:
            ops.record_callback(sync.backward_done)
        if plan_key is not None:
            self._store_plan(bufs, plan_key, keys, p_drop)
        return dx

    # ------------------------------------------------------------------------------------------------------
    # reference call surface
    # ------------------------------------------------------------------------------------------------------
    def get_num_params(self, non_embedding=True):
        n_params = sum(p.numel() for p in self.parameters())
        if non_embedding:
            n_params -= self.transformer.wpe.weight.numel()
        return n_params

    def _init_weights(self, module):
        if isinstance(module, nn.Linear):
            torch.nn.init.normal_(module.weight, mean=0.0, std=0.02)
            if module.bias is not None:
                torch.nn.init.zeros_(module.bias)
        elif isinstance(module, nn.Embedding):
            torch.nn.init.normal_(module.weight, mean=0.0, std=0.02)

    def forward(self, idx, targets=None):
        B, T = idx.size()
        if targets is not None and torch.is_grad_enabled() and self._arena["params"][0].requires_grad:
            anchor = self._anchor_tensor(idx.device)
            logits, loss = _GPTStep.apply(anchor, self, idx, targets)
            return logits, loss
        with torch.no_grad():
            bufs = self._forward_plan(idx, targets, keep_activations=False)
        V = self.config.vocab_size
        if targets is not None:
            return bufs.logits.view(B, T, -1)[:, :, :V], bufs.loss.view(()).clone()
        return bufs.last_logits[:, :V].unsqueeze(1), None

    def forward_hidden(self, inputs_embeds):
        """HF `GPT2Model(inputs_embeds=...)`: position embeddings are added here, returns the fp32 ln_f output
        (`last_hidden_state`), differentiable w.r.t. inputs_embeds (tunesformer/utils.py:96-106)."""
        if not (torch.is_grad_enabled() and self._arena["params"][0].requires_grad):
            with torch.no_grad():
                bufs = self._forward_plan(None, None, keep_activations=False, embeds=inputs_embeds, want_hidden=True)
            return bufs.hidden.view(*inputs_embeds.shape).clone()
        anchor = self._anchor_tensor(inputs_embeds.device)
        _, hidden = _GPTEmbedsStep.apply(anchor, self, inputs_embeds, None, None, True, 1)
        return hidden

    def forward_with_first(self, idx, first_embeds, targets):
        """HF `GPT2LMHeadModel(inputs_embeds=cat(first, wte(idx)[:, 1:]), labels=...)`: token embeddings with the first
        position replaced by `first_embeds` [B, C]; returns the loss over `targets` (already shifted by the caller,
        ignore_index = -1), differentiable w.r.t. first_embeds (tunesformer/utils.py:120-154)."""
        anchor = self._anchor_tensor(idx.device)
        loss, _ = _GPTEmbedsStep.apply(anchor, self, first_embeds, idx, targets, False, 2)
        return loss

    def next_logits_with_first(self, idx, first_embeds):
        """Inference branch of `forward_with_first`: fp32 logits [B, V] of the token that follows `idx` [B, t] when the first
        position's embedding is `first_embeds` [B, C] (tunesformer/utils.py:156-177, CharLevelDecoder.generate)."""
        with torch.no_grad():
            bufs = self._forward_plan(idx, None, keep_activations=False, first=first_embeds)
        return bufs.last_logits[:, :self.config.vocab_size].float()

    def _anchor_tensor(self, device):
        t = getattr(self, "_anchor", None)
        if t is None or t.device != device:
            t = torch.zeros(1, device=device, requires_grad=True)
            object.__setattr__(self, "_anchor", t)
        return t

    _HF_SHAPES = {"gpt2": (12, 12, 768), "gpt2-medium": (24, 16, 1024), "gpt2-large": (36, 20, 1280), "gpt2-xl": (48, 25, 1600)}
    _HF_CONV1D = ("attn.c_attn.weight", "attn.c_proj.weight", "mlp.c_fc.weight", "mlp.c_proj.weight")

    def load_hf_gpt2_state_dict(self, sd_hf):
        """Copies a HuggingFace `GPT2LMHeadModel` state dict into this module (nanoGPT/model.py:236-259): the mask buffers
        (`.attn.bias`, `.attn.masked_bias`) are dropped, the four Conv1D weights per block are stored [in, out] there and are
        transposed here, everything else is copied under the same name.  Shapes must agree exactly."""
        own = self.state_dict()
        src = {k: v for k, v in sd_hf.items() if not (k.endswith(".attn.masked_bias") or k.endswith(".attn.bias"))}
        if len(src) != len(own):
            raise ValueError(f"mismatched keys: {len(src)} != {len(own)}")
        out = {}
        for k, v in src.items():
            if k not in own:
                raise KeyError(f"unexpected key in the GPT-2 checkpoint: {k}")
            v = v.detach()
            if k.endswith(self._HF_CONV1D):
                v = v.t()
            if tuple(v.shape) != tuple(own[k].shape):
                raise ValueError(f"shape mismatch for {k}: {tuple(v.shape)} vs {tuple(own[k].shape)}")
            out[k] = v.contiguous()
        self.load_state_dict(out)
        return self

    @classmethod
    def from_pretrained(cls, model_type, override_args=None):
        """`GPT.from_pretrained('gpt2' | 'gpt2-medium' | 'gpt2-large' | 'gpt2-xl', dict(dropout=...))` as in the reference
        (nanoGPT/model.py:206-261; `train.py:197-205` init_from='gpt2*', `sample.py:67-69`): vocab 50257, block 1024,
        bias=True, weights from `transformers.GPT2LMHeadModel.from_pretrained` (needs the HF cache or network access)."""
        if model_type not in cls._HF_SHAPES:
            raise ValueError(f"unknown GPT-2 checkpoint {model_type!r}")
        override_args = override_args or {}
        if any(k != "dropout" for k in override_args):
            raise ValueError("only dropout can be overridden")
        from transformers import GPT2LMHeadModel
        print("loading weights from pretrained gpt: %s" % model_type)
        n_layer, n_head, n_embd = cls._HF_SHAPES[model_type]
        print("forcing vocab_size=50257, block_size=1024, bias=True")
        args = dict(n_layer=n_layer, n_head=n_head, n_embd=n_embd, vocab_size=50257, block_size=1024, bias=True)
        if "dropout" in override_args:
            print(f"overriding dropout rate to {override_args['dropout']}")
            args["dropout"] = override_args["dropout"]
        model = cls(GPTConfig(**args))
        return model.load_hf_gpt2_state_dict(GPT2LMHeadModel.from_pretrained(model_type).state_dict())

    def crop_block_size(self, block_size):
        assert block_size <= self.config.block_size
        self.config.block_size = block_size
        self.transformer.wpe.weight = nn.Parameter(self.transformer.wpe.weight[:block_size].detach().clone())
        self._flatten()

    def configure_optimizers(self, weight_decay, learning_rate, betas, device_type):
        param_dict = {pn: p for pn, p in self.named_parameters() if p.requires_grad}
        decay_params = [p for n, p in param_dict.items() if p.dim() >= 2]
        nodecay_params = [p for n, p in param_dict.items() if p.dim() < 2]
        optim_groups = [
            {"params": decay_params, "weight_decay": weight_decay},
            {"params": nodecay_params, "weight_decay": 0.0},
        ]
        print(f"num decayed parameter tensors: {len(decay_params)}, with {sum(p.numel() for p in decay_params):,} parameters")
        print(f"num non-decayed parameter tensors: {len(nodecay_params)}, with {sum(p.numel() for p in nodecay_params):,} parameters")
        optimizer = FusedAdamW(optim_groups, lr=learning_rate, betas=betas, model=self)
        print("using fused AdamW: True (sm_100a arena kernel)")
        return optimizer

    def clip_grad_norm_(self, max_norm):
        """Fused counterpart of torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm) (train.py:352): one
        sum-of-squares launch now, the scaling itself is folded into the next optimizer.step().  Returns the total
        gradient norm as a 0-d device tensor (no host sync)."""
        a = self._arena
        if a["grad"] is None or a["params"][0].grad is None:
            raise RuntimeError("clip_grad_norm_: no gradients (call loss.backward() first)")
        if self._grad_sync is not None:
            self._grad_sync.wait()
        ss = a.setdefault("sumsq", torch.zeros(1, device=a["flat"].device, dtype=torch.float32))
        ss.zero_()
        if self._grad_sync is None or not self._grad_sync.fused_sumsq(ss):   # NVLS exchange: the norm came with the gradients
            ops.sumsq(a["grad"], ss)
        self._pending_clip = (ss, float(max_norm))
        return ss.sqrt().view(())

    def estimate_mfu(self, fwdbwd_per_iter, dt, flops_promised=312e12):
        """Same formula as the reference (model.py:289-303); `flops_promised` defaults to the reference's A100
        constant so numbers are comparable, pass 2.25e15 for B200 dense bf16."""
        N = self.get_num_params()
        cfg = self.config
        L, H, Q, T = cfg.n_layer, cfg.n_head, cfg.n_embd // cfg.n_head, cfg.block_size
        flops_per_token = 6 * N + 12 * L * H * Q * T
        flops_per_iter = flops_per_token * T * fwdbwd_per_iter
        return flops_per_iter * (1.0 / dt) / flops_promised

    def _generate_ragged(self, idx, prompt_lens, max_new_tokens, temperature, top_k, stop_token, stop_check_every):
        if not idx.is_cuda:
            raise _C.AbcgptError("GPT.generate: idx must be a CUDA tensor (there is no CPU path)")
        B, Tmax = idx.shape
        lens = torch.as_tensor(prompt_lens, device=idx.device, dtype=torch.int64).view(B)
        lmin, lmax = int(lens.min()), int(lens.max())
        bs = self.config.block_size
        total = lmax + max_new_tokens
        if lmin < 1 or lmax > Tmax:
            raise ValueError(f"prompt_lens must lie in [1, {Tmax}]")
        if total - 1 > bs:
            raise ValueError(f"ragged generation needs max(prompt_lens) + max_new_tokens <= block_size + 1 (got {total} > {bs + 1}); "
                             "group the prompts by length instead")
        fill = 0 if stop_token is None else int(stop_token)
        out = torch.full((B, total), fill, device=idx.device, dtype=torch.int64)
        was_training = self.training
        self.eval()
        try:
            self._ensure_device_state()
            key = ("decode", B, bs)
            if key not in self._bufs:
                self._bufs[key] = _DecodeState(self.config, B, bs, idx.device)
            st = self._bufs[key]
            pos = torch.arange(total, device=idx.device).view(-1, 1)            # [total, 1]
            is_prompt = pos < lens.view(1, -1)                                    # [total, B]
            forced = torch.zeros(total, B, device=idx.device, dtype=torch.int64)
            forced[:lmax] = idx[:, :lmax].t()
            st.col[:lmin].copy_(forced[:lmin])
            head = self._head(temperature, top_k)
            self._reseed_sampler()
            last = total - 1
            ops.set_pdl(True)
            for t in range(last):
                want = t >= lmin - 1
                self._decode_step(st, t, want, head if want else None)
                if want and t + 1 < lmax:   # rows still inside their prompt take the prompt token, the others keep the sampled one
                    st.col[t + 1].copy_(torch.where(is_prompt[t + 1], forced[t + 1], st.col[t + 1]))
                if stop_token is not None and t >= lmin and (t - lmin) % stop_check_every == stop_check_every - 1:
                    seen = ((st.col[:t + 2] == stop_token) & ~is_prompt[:t + 2]).any(dim=0)
                    if bool(seen.all()):
                        last = t + 1
                        break
            ops.set_pdl(False)
            out[:, :last + 1] = st.col[:last + 1].t()
            beyond = pos.view(1, -1) >= (lens + max_new_tokens).view(-1, 1)      # [B, total]
            out.masked_fill_(beyond, fill)
        finally:
            ops.set_pdl(False)
            self.train(was_training)
        return out

    def _decode_step(self, st, t, want_logits, head, inp="tokens", hidden=False):
        """Position t of every sequence (tokens st.col[t]).  Appends this position's q|k|v to the cache and, if
        want_logits, leaves the next-token logits in st.logits and runs the sampling head, which writes token t + 1 of every
        sequence into st.col[t + 1]: head = None (logits only), ("greedy",) = argmax, ("sample", temperature, top_k) = the
        fused temperature / top-k / softmax / multinomial kernel (seeded per generate() call through self._sample_seed),
        ("top_p", top_p, top_k, temperature) = the nucleus / top-k / temperature kernel of the TunesFormer character decoder
        (seed, counter base and row ids from st.sampler; counter = t).
        Input and output modes of a decoder fed by another network (TunesFormer): inp = "tokens" (token ids st.col[t]),
        "first" (t = 0 only: the fp32 row st.emb replaces the token embedding, + wpe[0]) or "embed" (st.emb + wpe[t]);
        hidden = True writes the fp32 ln_f output of the position to st.hidden (HF last_hidden_state) instead of logits.
        Every argument is static per (t, flags), so the launch list is recorded once and replayed afterwards."""
        flags = (want_logits, head, torch.cuda.current_stream().cuda_stream, inp, hidden)
        plan_key = (t,) + flags
        plan = st.plans.get(plan_key) if self._plan_cache_enabled else None
        if plan is not None:
            ops.replay(plan)
            return
        # Every argument of a decode step is affine in the position t (cache rows, token columns, key count): once three
        # consecutive recorded steps confirm constant per-argument differences, later positions replay the recorded launch
        # list with patched arguments instead of re-deriving ~90 launches in Python (the decode loop is launch-bound).
        aff = st.affine.get(flags) if self._plan_cache_enabled and ops._PROFILE is None else None
        if aff is not None:
            if aff[3] is not None:
                ops.replay_compiled(aff[3], t - aff[0])   # the whole step in one C call
            else:
                ops.replay_affine(aff[1], aff[2], t - aff[0])
            return
        if self._plan_cache_enabled:
            ops.begin_record()
        tokens = st.col[t]
        cfg = self.config
        layers = self._layer_tensors()
        top = self._arena["top"]
        B, C, H = st.B, cfg.n_embd, cfg.n_head
        x, y = st.x
        if inp == "tokens":
            ops.embed_fwd(tokens, top["wte"][0], top["wpe"][0][t:t + 1], x, 1)
        elif inp == "first":
            if t != 0 or st.emb is None:
                raise _C.AbcgptError("decode step: the 'first' input mode is position 0 of a state with its emb rows set")
            ops.set_first_pos(st.emb, top["wpe"][0], x, 1)
        elif inp == "embed":
            if st.emb is None:
                raise _C.AbcgptError("decode step: the 'embed' input mode needs the state's emb rows")
            ops.add_pos(st.emb, top["wpe"][0][t:t + 1], x, 1)
        else:
            raise ValueError(f"decode step: unknown input mode {inp!r}")
        for li, lw in enumerate(layers):
            b = lambda name: None if lw[name] is None else lw[name][0]  # noqa: E731
            ops.layernorm_fwd(x, lw["ln_1.weight"][0], b("ln_1.bias"), st.ln, st.stat[0], st.stat[1])
            if st.D == 64:
                # the GEMM writes this position's q | k | v straight into the head-major cache [B, 3H, Tmax, 64]
                qkv_t = st.cache[li].view(B, 3 * H, st.Tmax, 64)[:, 0, t, :]
                ops.gemm(st.ln, lw["attn.c_attn.weight"][1], epilogue=ops.EPI_BF16, out=qkv_t, bias=b("attn.c_attn.bias"),
                         tile_n=128, head_stride=st.Tmax * 64)
                ops.attn_decode(st.cache[li], st.att, B, st.Tmax, t + 1, H)
            else:
                # other head sizes: a plain [B, 3C] row; the decode kernel appends its k | v to the cache [B, 2H, Tmax, D]
                ops.gemm(st.ln, lw["attn.c_attn.weight"][1], epilogue=ops.EPI_BF16, out=st.qkv, bias=b("attn.c_attn.bias"),
                         tile_n=128)
                ops.attn_decode_hd(st.qkv, st.cache[li], st.att, B, st.Tmax, t, H, st.D)
            ops.gemm(st.att, lw["attn.c_proj.weight"][1], epilogue=ops.EPI_RESID, out=y, aux=x, bias=b("attn.c_proj.bias"),
                     tile_n=128)
            ops.layernorm_fwd(y, lw["ln_2.weight"][0], b("ln_2.bias"), st.ln, st.stat[0], st.stat[1])
            ops.gemm(st.ln, lw["mlp.c_fc.weight"][1], epilogue=ops.EPI_GELU | self._act, out=st.h, out2=st.g, bias=b("mlp.c_fc.bias"),
                     tile_n=128)
            ops.gemm(st.g, lw["mlp.c_proj.weight"][1], epilogue=ops.EPI_RESID, out=x, aux=y, bias=b("mlp.c_proj.bias"),
                     tile_n=128)
        if hidden and (want_logits or st.hidden is None):
            raise _C.AbcgptError("decode step: the hidden-state output needs the state's hidden rows and replaces the logits")
        if want_logits or hidden:
            lnf_b = None if top["ln_f.bias"] is None else top["ln_f.bias"][0]
            ops.layernorm_fwd(x, top["ln_f.weight"][0], lnf_b, st.ln, st.stat[0], st.stat[1], y_f32=st.hidden if hidden else None)
        if want_logits:
            ops.gemm(st.ln, top["wte"][1], N=st.Vpad, epilogue=ops.EPI_BF16, out=st.logits, tile_n=128)
            if head is not None and head[0] == "greedy":
                ops.argmax(st.logits, cfg.vocab_size, st.col[t + 1], out_stride=1)
            elif head is not None and head[0] == "top_p":
                seed, counter_base, row_id = st.sampler
                ops.sample_top_p(st.logits, cfg.vocab_size, st.col[t + 1], head[1], head[2], head[3], seed, counter_base, t,
                                 row_id=row_id)
            elif head is not None:
                ops.sample_topk(st.logits, cfg.vocab_size, st.col[t + 1], head[1], head[2], self._seed_buffer(), t)
        if self._plan_cache_enabled:
            plan = st.plans[plan_key] = ops.end_record()
            p1, p2 = st.plans.get((t - 1,) + flags), st.plans.get((t - 2,) + flags)
            if p1 is not None and p2 is not None:
                d1, d2 = ops.plan_deltas(p1, plan), ops.plan_deltas(p2, p1)
                if d1 is not None and d1 == d2:
                    st.affine[flags] = (t, plan, d1, ops.compile_affine(plan, d1))

    def _seed_buffer(self):
        """uint64 device scalar read by the sampling kernel (its address is part of recorded launch lists)."""
        dev = self._arena["flat"].device
        buf = getattr(self, "_sample_seed", None)
        if buf is None or buf.device != dev:
            buf = torch.zeros(1, device=dev, dtype=torch.int64)
            object.__setattr__(self, "_sample_seed", buf)
        return buf

    def _reseed_sampler(self):
        """One draw from torch's CPU generator per generate() call: `torch.manual_seed(seed)` (sample.py:44) makes the sampled
        tunes reproducible, and consecutive calls see different random streams."""
        self._seed_buffer().fill_(int(torch.randint(0, 2 ** 62, (1,)).item()))

    def _head(self, temperature, top_k):
        V = self.config.vocab_size
        if top_k is not None and min(top_k, V) == 1:
            return ("greedy",)   # top_k = 1: the softmax over one surviving token is 1, the draw is its argmax
        k = 0 if top_k is None else min(int(top_k), V)
        return ("sample", float(temperature), 0 if k >= V else k)

    def _sample(self, logits_bf16, out_col, out_stride, head, counter):
        V = self.config.vocab_size
        if head[0] == "greedy":
            ops.argmax(logits_bf16, V, out_col, out_stride=out_stride)
        else:
            ops.sample_topk(logits_bf16, V, out_col, head[1], head[2], self._seed_buffer(), counter, out_stride=out_stride)

    @torch.no_grad()
    def generate(self, idx, max_new_tokens, temperature=1.0, top_k=None, use_cache=True, stop_token=None, stop_check_every=64,
                 prompt_lens=None):
        """Reference semantics (model.py:305-330): feed the sequence back max_new_tokens times, last-position logits,
        temperature, optional top-k, sample, append; the context is cropped to block_size.

        While the context window does not slide (position < block_size) each new token costs ONE single-position step over
        a KV cache instead of the reference's full-context forward; absolute position embeddings make the cache invalid
        once the window slides, so from there on the context is recomputed per token exactly like the reference.
        The sampling head is one fused launch per token writing straight into the pre-allocated token buffer: argmax for
        top_k == 1 (greedy), otherwise temperature / top-k crop / softmax / multinomial (abcgpt_sample_topk) with a Philox
        stream seeded from torch's generator once per call.

        stop_token (extension, default off): sample.py cuts every generated tune at the first end-of-tune symbol
        (sample.py:163-165), so once EVERY sequence of the batch has produced it the remaining steps cannot change the
        written files; checked every `stop_check_every` tokens (one host sync each), the tail is filled with stop_token.

        prompt_lens (extension, default off; SURVEY.md 8f N3 "variable-length prompt batching"): idx is right-padded
        [B, max prompt length] and row i holds prompt_lens[i] real tokens.  Positions are absolute, so all rows advance
        through the same position t together; a row whose prompt is longer than t + 1 takes its next token from the
        prompt instead of the sampler (its prefix is fed through the same single-position steps an equal-length batch
        uses, so each row's tokens are those of generating it alone).  Row i of the result holds its prompt followed by
        max_new_tokens generated tokens; anything after that is filled with stop_token (0 if None).  Needs
        max(prompt_lens) + max_new_tokens <= block_size + 1 (the window may not slide)."""
        if prompt_lens is not None:
            return self._generate_ragged(idx, prompt_lens, max_new_tokens, temperature, top_k, stop_token, stop_check_every)
        if not idx.is_cuda:
            raise _C.AbcgptError("GPT.generate: idx must be a CUDA tensor (there is no CPU path)")
        B, T0 = idx.shape
        bs = self.config.block_size
        total = T0 + max_new_tokens
        out = torch.empty(B, total, device=idx.device, dtype=torch.int64)
        out[:, :T0] = idx
        was_training = self.training
        self.eval()
        try:
            self._ensure_device_state()
            head = self._head(temperature, top_k)
            self._reseed_sampler()
            t = 0
            if use_cache and T0 <= bs:
                key = ("decode", B, bs)
                if key not in self._bufs:
                    self._bufs[key] = _DecodeState(self.config, B, bs, idx.device)
                st = self._bufs[key]
                last = min(total - 1, bs)   # positions 0 .. last-1 can be decoded with the cache
                st.col[:T0].copy_(idx.t())
                stopped = False
                ops.set_pdl(True)   # ~90 small dependent launches per token: overlap each launch / prologue with its predecessor
                for t in range(last):
                    want = t >= T0 - 1
                    self._decode_step(st, t, want, head if want else None)
                    if stop_token is not None and t >= T0 and (t - T0) % stop_check_every == stop_check_every - 1:
                        if bool((st.col[T0:t + 2] == stop_token).any(dim=0).all()):
                            st.col[t + 2:last + 1].fill_(stop_token)
                            stopped = True
                            break
                ops.set_pdl(False)
                out[:, :last + 1].copy_(st.col[:last + 1].t())
                if stopped:
                    out[:, last + 1:].fill_(stop_token)
                    return out
                t = last
            for pos in range(max(t, T0 - 1), total - 1):  # window slides (or cache disabled): reference-style recompute
                lo = max(0, pos + 1 - bs)
                cond = out[:, lo:pos + 1].contiguous()
                bufs = self._forward_plan(cond, None, keep_activations=False)
                self._sample(bufs.last_logits, out[:, pos + 1:], out.stride(0), head, pos)
        finally:
            ops.set_pdl(False)
            self.train(was_training)
        return out
