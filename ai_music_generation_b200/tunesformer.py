"""TunesFormer-shaped hierarchical decoder on the sm_100a kernels (SURVEY.md 8f N1, BASELINE config 4).

Shape donor: tunesformer/utils.py:84-219 (paths relative to /root/reference) — a patch-level GPT-2 (bar patches of
PATCH_SIZE characters, embedded by Linear(PATCH_SIZE*128 -> n_embd) on one-hot rows, `GPT2Model(inputs_embeds=...)`) whose
hidden states become the FIRST input embedding of a character-level GPT-2 LM that spells out the next patch
(`GPT2LMHeadModel(inputs_embeds=cat(encoded_patch, wte(chars)[:, 1:]), labels=chars)`, pad id 0 ignored).

Both decoders are the GPT of model.py (biases, tanh GELU), so every matmul / attention / LayerNorm / loss / AdamW launch is
the same kernel as on the nanoGPT path; the joins are `GPT.forward_hidden` / `GPT.forward_with_first`.  The HF code itself
(third-party arithmetic, single-process DataParallel trainer) is not rebuilt; parameter names follow this package.
"""
from __future__ import annotations

import random
import re

import numpy as np
import torch
import torch.nn as nn

from . import _C, ops
from .model import GPT, GPTConfig, _DecodeState

PATCH_SIZE = 32      # tunesformer/config.py:2
PATCH_LENGTH = 128   # tunesformer/config.py:1
CHAR_VOCAB = 128     # one-hot width per character (utils.py:102)


class Patchilizer:
    """Bar <-> patch codec of the hierarchical model (behaviour of tunesformer/utils.py:9-82; host-side, pure Python).

    A tune is cut at bar lines; every bar (with its closing delimiter) and every header line becomes one patch of PATCH_SIZE
    character codes: bos (1), the characters, eos (2), padded with 0.  (The reference passes the text through `unidecode`
    first; that package is optional here and plain ASCII input is unchanged by it.)"""

    DELIMS = ("|:", "::", ":|", "[|", "||", "|]", "|")
    pad_token_id, bos_token_id, eos_token_id = 0, 1, 2

    def __init__(self):
        self._split = re.compile("(" + "|".join(re.escape(d) for d in self.DELIMS) + ")")

    def split_bars(self, body):
        parts = [x for x in self._split.split("".join(body)) if x]
        if parts and parts[0] in self.DELIMS:       # a leading bar line belongs to the first bar
            parts[1] = parts[0] + parts[1]
            parts = parts[1:]
        return [parts[2 * i] + parts[2 * i + 1] for i in range(len(parts) // 2)]

    def bar2patch(self, bar, patch_size=PATCH_SIZE):
        codes = ([self.bos_token_id] + [ord(c) for c in bar] + [self.eos_token_id])[:patch_size]
        return codes + [self.pad_token_id] * (patch_size - len(codes))

    def patch2bar(self, patch):
        return "".join(chr(t) for t in patch if t > self.eos_token_id)

    def encode(self, abc_code, patch_length=PATCH_LENGTH, patch_size=PATCH_SIZE, add_special_patches=False):
        try:
            from unidecode import unidecode
            abc_code = unidecode(abc_code)
        except ImportError:
            pass
        patches, body = [], ""

        def flush(last_newline):
            bars = self.split_bars(body)
            for i, bar in enumerate(bars):
                patches.append(self.bar2patch(bar + "\n" if (last_newline and i == len(bars) - 1) else bar, patch_size))

        for line in (ln for ln in abc_code.split("\n") if ln):
            header = len(line) > 1 and ((line[0].isalpha() and line[1] == ":") or line.startswith("%%score"))
            if header:
                if body:
                    flush(True)
                    body = ""
                patches.append(self.bar2patch(line + "\n", patch_size))
            else:
                body += line + "\n"
        if body:
            flush(False)
        if add_special_patches:
            patches = ([[self.bos_token_id] * (patch_size - 1) + [self.eos_token_id]] + patches +
                       [[self.bos_token_id] + [self.eos_token_id] * (patch_size - 1)])
        return patches[:patch_length]

    def decode(self, patches):
        return "".join(self.patch2bar(p) for p in patches)


# ---- sampling helpers -------------------------------------------------------------------------------------------------
# The reference draws the next character with the third-party `samplings` package (top_p_sampling, top_k_sampling with
# return_probs=True, then temperature_sampling; tunesformer/utils.py:6,247-250).  The package is not vendored in the reference
# and is absent here, so these are restatements of its documented behaviour, not pinned to it: nucleus filter = keep the most
# probable characters up to and including the one that takes the cumulative probability to top_p, top-k filter = keep the k
# most probable (0 = all), both renormalise; the draw raises the probabilities to 1 / temperature, renormalises and samples
# with numpy's seeded generator.  With top_k = 1 every variant is the argmax, which is what the golden test pins.
def top_p_filter(probs, top_p):
    if top_p >= 1.0:
        return probs
    order = np.argsort(-probs, kind="stable")
    csum = np.cumsum(probs[order])
    keep = order[: int(np.searchsorted(csum, top_p, side="left")) + 1]
    out = np.zeros_like(probs)
    out[keep] = probs[keep]
    return out / out.sum()


def top_k_filter(probs, top_k):
    if top_k <= 0 or top_k >= probs.size:
        return probs
    keep = np.argsort(-probs, kind="stable")[:top_k]
    out = np.zeros_like(probs)
    out[keep] = probs[keep]
    return out / out.sum()


def temperature_draw(probs, temperature, seed=None):
    if temperature <= 0.0 or np.count_nonzero(probs) == 1:
        return int(np.argmax(probs))
    p = np.power(probs.astype(np.float64), 1.0 / temperature)
    p /= p.sum()
    return int(np.random.RandomState(seed).choice(p.size, p=p))


class _PatchEmbed(torch.autograd.Function):
    """out[m,:] = onehot(patch m) W^T + b as a GEMM on the one-hot rows; backward = weight / bias gradients only."""

    @staticmethod
    def forward(ctx, anchor, dec, patches):
        M = patches.shape[0]
        dec._ensure_device_state()
        out = torch.empty(M, dec.config.n_embd, device=patches.device, dtype=torch.float32)
        oh = dec.embed_patches(patches.contiguous(), out)
        ctx.dec, ctx.oh = dec, oh
        return out

    @staticmethod
    def backward(ctx, d_out):
        dec, oh = ctx.dec, ctx.oh
        M, C = d_out.shape
        db16 = torch.empty(M, C, device=d_out.device, dtype=torch.bfloat16)
        ops.cast_bf16(d_out.contiguous().view(-1), db16.view(-1))
        # runs after the stack's backward plan (autograd order), which has zeroed / attached the gradient arena
        ops.gemm(db16, oh, a_mn=True, b_mn=True, epilogue=ops.EPI_F32_RED, out=dec._view("grad", "patch_embedding.weight"))
        ops.colsum_bf16(db16, dec._view("grad", "patch_embedding.bias"))
        sync = dec._grad_sync
        if sync is not None and dec.require_backward_grad_sync:
            sync.finalize()   # this arena's last gradients: wte/wpe, the patch embedding and the 1-D tail go out now
        return None, None, None


class PatchLevelDecoder(GPT):
    """GPT stack + patch embedding in ONE parameter arena (clip / AdamW / DDP buckets cover it without extra code)."""

    def __init__(self, config: GPTConfig):
        super().__init__(config)
        self.patch_embedding = nn.Linear(PATCH_SIZE * CHAR_VOCAB, config.n_embd)
        torch.nn.init.normal_(self.patch_embedding.weight, std=0.02)   # utils.py:94
        torch.nn.init.zeros_(self.patch_embedding.bias)
        self._onehot = {}
        self._flatten()

    def embed_patches(self, patches, out):
        """out fp32 [M, C] = onehot(patches int64 [M, PATCH_SIZE]) W^T + b (one-hot rows, then the GEMM); returns the one-hot
        rows.  The bf16 weight shadow must be current (_ensure_device_state)."""
        M = patches.shape[0]
        oh = self._onehot.get(M)
        if oh is None:
            oh = self._onehot[M] = torch.empty(M, PATCH_SIZE * CHAR_VOCAB, device=patches.device, dtype=torch.bfloat16)
        ops.onehot_bf16(patches, oh, CHAR_VOCAB)
        ops.gemm(oh, self._view("shadow", "patch_embedding.weight"), epilogue=ops.EPI_F32, out=out,
                 bias=self._view("flat", "patch_embedding.bias"))
        return oh

    def encode(self, patches):
        """patches int64 [B, P, PATCH_SIZE] -> fp32 [B, P, C] (last_hidden_state)."""
        B, P, S = patches.shape
        assert S == PATCH_SIZE and P <= self.config.block_size
        emb = _PatchEmbed.apply(self._anchor_tensor(patches.device), self, patches.reshape(B * P, S))
        return self.forward_hidden(emb.view(B, P, -1))


class TunesFormerShaped(nn.Module):
    def __init__(self, patch_config: GPTConfig, char_config: GPTConfig):
        super().__init__()
        assert char_config.vocab_size == CHAR_VOCAB and char_config.block_size >= PATCH_SIZE
        self.patch_level_decoder = PatchLevelDecoder(patch_config)
        self.char_level_decoder = GPT(char_config)
        self.pad_token_id = 0

    def forward(self, patches):
        """patches int64 [B, P, PATCH_SIZE] (pad id 0 at the tail of every patch) -> mean next-character loss over the
        non-pad characters of patches 1..P-1, each decoded from the encoding of the patches before it (utils.py:210-219)."""
        B, P, S = patches.shape
        encoded = self.patch_level_decoder.encode(patches)                  # [B, P, C]
        first = encoded[:, :-1, :].reshape(B * (P - 1), -1)
        chars = patches[:, 1:, :].reshape(B * (P - 1), S)
        y = torch.full_like(chars, -1)
        y[:, :-1] = chars[:, 1:]
        y[y == self.pad_token_id] = -1                                       # labels -100 at pads (utils.py:128-129)
        return self.char_level_decoder.forward_with_first(chars, first, y)

    @torch.no_grad()
    def generate(self, patches, tokens=None, top_p=1.0, top_k=0, temperature=1.0, seed=None):
        """One more patch for every tune of the batch (tunesformer/utils.py:221-255, there for a single tune).

        patches int64 [N, P, PATCH_SIZE] (or [P, PATCH_SIZE]): the tunes so far; `tokens` (optional, int64 [t] starting with
        bos): characters of the new patch that are already fixed (a prompt that ends inside a bar).  The patch-level decoder
        encodes the patches, the character-level decoder then spells the next patch one character at a time from the last
        patch's encoding — every step is one forward of all still-running tunes through the sm_100a kernels; a tune stops at
        eos or after PATCH_SIZE - 1 characters.  Returns (generated patches: one list of character codes per tune — a bare
        list when a single tune was given, like the reference —, the seed to pass to the next call)."""
        single = patches.dim() == 2 or patches.shape[0] == 1
        if patches.dim() == 2:
            patches = patches.unsqueeze(0)
        patches = patches.reshape(patches.shape[0], -1, PATCH_SIZE)
        N = patches.shape[0]
        dev = patches.device
        eos = 2
        first = self.patch_level_decoder.encode(patches)[:, -1, :].contiguous()           # [N, C]
        if tokens is None:
            tokens = torch.tensor([1], device=dev)
        seq = tokens.reshape(1, -1).to(dev).repeat(N, 1)                                    # [N, t]
        out = [[] for _ in range(N)]
        alive = list(range(N))
        rng = random.Random(seed)
        n_seed = None
        while alive:
            if seed is not None:                      # the reference re-seeds Python's generator with every draw
                n_seed = rng.randint(0, 1000000)
                rng.seed(n_seed)
            rows = torch.tensor(alive, device=dev)
            logits = self.char_level_decoder.next_logits_with_first(seq[rows].contiguous(), first[rows].contiguous())
            probs = torch.softmax(logits, dim=-1).cpu().numpy()
            nxt = []
            for j, i in enumerate(alive):
                p = top_k_filter(top_p_filter(probs[j], top_p), top_k)
                tok = temperature_draw(p, temperature, None if n_seed is None else n_seed + j)
                out[i].append(tok)
                nxt.append(tok)
            done = seq.shape[1] >= PATCH_SIZE - 1
            keep = [k for k, tok in enumerate(nxt) if tok != eos and not done]
            if not keep:
                break
            col = torch.zeros(N, 1, dtype=seq.dtype, device=dev)
            col[rows, 0] = torch.tensor(nxt, device=dev, dtype=seq.dtype)
            seq = torch.cat([seq, col], dim=1)
            alive = [alive[k] for k in keep]
        return (out[0] if single else out), n_seed

    @torch.no_grad()
    def generate_tune(self, prompt, max_patch=PATCH_LENGTH, top_p=0.8, top_k=8, temperature=1.2, seed=None):
        """The tune loop of tunesformer/generate.py:128-155 for one prompt (ABC header / opening bars as text): bar patches are
        generated and appended until the model emits an end patch, an empty bar, or `max_patch` patches.  Returns the text."""
        pz = Patchilizer()
        dev = next(self.parameters()).device
        patches = torch.tensor([pz.encode(prompt, add_special_patches=True)[:-1]], device=dev)
        prefix = pz.decode(patches[0].tolist())
        remaining = prompt[len(prefix):]
        tokens = torch.tensor([pz.bos_token_id] + [ord(c) for c in remaining], device=dev) if prompt else None
        tune = prompt
        while patches.shape[1] < max_patch:
            patch, seed = self.generate(patches, tokens, top_p=top_p, top_k=top_k, temperature=temperature, seed=seed)
            tokens = None
            if patch[0] == pz.eos_token_id:
                break
            bar = pz.decode([patch])
            if bar == "":
                break
            tune += bar
            nxt = torch.tensor([[pz.bar2patch(remaining + bar)]], device=dev)
            remaining = ""
            patches = torch.cat([patches, nxt], dim=1)
        return tune

    # ---- generation on the device ------------------------------------------------------------------------------------
    @torch.no_grad()
    def generate_tunes(self, prompts, max_patch=PATCH_LENGTH, top_p=0.8, top_k=8, temperature=1.2, seed=None, batch=64):
        """`generate_tune` for a list of prompt texts, batched and decoded on the device; returns one tune text per prompt.

        Per tune the loop is that of generate_tune: the prompt is encoded with the same Patchilizer, its unfinished last bar
        becomes fixed characters of the first generated bar, each bar is spelled until eos or 31 characters, and a tune stops
        at an end patch, an empty bar or `max_patch` patches.  Both decoders run single-position steps over KV caches
        (generate_patches), the draw is the nucleus / top-k / temperature kernel (abcgpt_sample_top_p), and the host
        synchronises once per bar (plus an early-exit check every 8 characters).

        Seeding differs from `generate` / `generate_tune` on purpose: those reproduce the reference's per-draw reseeding of
        Python's `random` and numpy's generator on the host, which no device kernel can follow.  Here every draw takes a
        Philox uniform of (seed, index of the tune in `prompts`, patch position, character position), so a tune's random
        stream does not depend on the batch it lands in.  An int `seed` makes a call reproducible; seed=None draws one seed
        from torch's CPU generator per call, so `torch.manual_seed` makes it reproducible.  With top_k = 1 every tune equals
        its greedy generate_tune (up to decisions closer than bf16 rounding)."""
        pz = Patchilizer()
        patches, fixed, remaining = [], [], []
        for prompt in prompts:
            enc = pz.encode(prompt, add_special_patches=True)[:-1]
            rest = prompt[len(pz.decode(enc)):]
            patches.append(enc)
            remaining.append(rest)
            fixed.append([ord(c) for c in rest])
        gen = self.generate_patches(patches, fixed, max_patch=max_patch, top_p=top_p, top_k=top_k, temperature=temperature,
                                    seed=seed, batch=batch)
        tunes = []
        for prompt, bars in zip(prompts, gen):
            tune = prompt
            for patch in bars:   # the stop rules of generate_tune: the last patch may be the one that stopped the tune
                if patch[0] == pz.eos_token_id:
                    break
                bar = pz.decode([patch])
                if bar == "":
                    break
                tune += bar
            tunes.append(tune)
        return tunes

    @torch.no_grad()
    def generate_patches(self, prompt_patches, fixed_tokens=None, max_patch=PATCH_LENGTH, top_p=0.8, top_k=8, temperature=1.2,
                         seed=None, batch=64):
        """The bar loop of generate_tune on patches, for many tunes at once.

        prompt_patches: one int [P_i, PATCH_SIZE] tensor (or nested list) per tune, starting with the start patch;
        fixed_tokens: None or one list of character codes per tune that follow bos in the first generated bar (a prompt that
        ends inside a bar).  Returns, per tune, the generated patches as lists of drawn character codes (each ends at its eos
        when one was drawn, like `generate`), the last one possibly the end patch or empty bar that stopped the tune.  The
        patch appended after a bar is bar2patch(fixed + bar) for the first bar and bar2patch(bar) after that.  `batch` tunes
        share one pass of the loop; tunes are grouped by prompt length first, and the result is in input order.  See
        generate_tunes for the seeding."""
        n = len(prompt_patches)
        pbs, cbs = self.patch_level_decoder.config.block_size, self.char_level_decoder.config.block_size
        if max_patch > pbs:
            raise ValueError(f"max_patch ({max_patch}) is above the patch decoder's block_size ({pbs})")
        prompts = [torch.as_tensor(p, dtype=torch.int64).cpu().reshape(-1, PATCH_SIZE).tolist() for p in prompt_patches]
        fixed = [[] for _ in range(n)] if fixed_tokens is None else [[int(c) for c in f] for f in fixed_tokens]
        if len(fixed) != n:
            raise ValueError("fixed_tokens needs one list per tune")
        if any(len(p) == 0 for p in prompts):
            raise ValueError("every prompt needs at least its start patch")
        if any(len(f) + 1 > min(cbs, PATCH_SIZE) for f in fixed):
            raise ValueError(f"at most {min(cbs, PATCH_SIZE) - 1} fixed characters per tune")
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        order = sorted(range(n), key=lambda i: len(prompts[i]))
        out = [None] * n
        # counters of the last call (tools/bench_tunesformer_generate.py): bars spelled (one per batch and patch position),
        # character steps, device->host synchronisations, kernel launches, and launches / C-ABI calls of the character steps
        self.last_generate_stats = stats = {"bars": 0, "char_steps": 0, "host_syncs": 0, "launches": 0, "char_launches": 0,
                                            "char_calls": 0}
        launches0 = ops.LAUNCHES
        for s in range(0, n, max(1, int(batch))):
            idx = order[s:s + max(1, int(batch))]
            res = self._generate_batch([prompts[i] for i in idx], [fixed[i] for i in idx], idx, max_patch, float(top_p),
                                       int(top_k), float(temperature), seed, stats)
            for i, r in zip(idx, res):
                out[i] = r
        stats["launches"] = ops.LAUNCHES - launches0
        return out

    def _decode_states(self, B, device):
        """Per-batch-size decode states of both decoders; the character level's first input rows ARE the patch level's hidden
        rows (no copy between the two)."""
        pd, cd = self.patch_level_decoder, self.char_level_decoder
        key = ("tunes", B)
        sp = pd._bufs.get(key)
        if sp is None:
            sp = pd._bufs[key] = _DecodeState(pd.config, B, pd.config.block_size, device)
            sp.emb = torch.empty(B, pd.config.n_embd, device=device, dtype=torch.float32)
            sp.hidden = torch.empty(B, pd.config.n_embd, device=device, dtype=torch.float32)
        sc = cd._bufs.get(key)
        if sc is None or sc.emb is not sp.hidden:
            sc = cd._bufs[key] = _DecodeState(cd.config, B, cd.config.block_size, device)
            sc.emb = sp.hidden
            sc.sampler = (torch.zeros(1, device=device, dtype=torch.int64), torch.zeros(1, device=device, dtype=torch.int64),
                          torch.zeros(B, device=device, dtype=torch.int64))
        return sp, sc

    def _generate_batch(self, prompts, fixed, row_ids, max_patch, top_p, top_k, temperature, seed, stats):
        pz = Patchilizer()
        eos = pz.eos_token_id
        pd, cd = self.patch_level_decoder, self.char_level_decoder
        dev = pd._arena["flat"].device
        if dev.type != "cuda":
            raise _C.AbcgptError("generate_patches: the model must be on a CUDA device (there is no CPU path)")
        B, S = len(prompts), PATCH_SIZE
        pd._ensure_device_state()
        cd._ensure_device_state()
        sp, sc = self._decode_states(B, dev)
        V = cd.config.vocab_size
        head = ("top_p", top_p, top_k if 0 < top_k < V else 0, temperature)
        seed_t, counter_base, row_id = sc.sampler
        seed_t.fill_(int(seed) & ((1 << 63) - 1))
        row_id.copy_(torch.tensor(row_ids, dtype=torch.int64).pin_memory(), non_blocking=True)
        # patch rows per position, all prompt patches uploaded at once; generated patches land at their position later
        rows = torch.zeros(max_patch, B, S, dtype=torch.int64)
        for i, p in enumerate(prompts):
            k = min(len(p), max_patch)
            rows[:k, i] = torch.tensor(p[:k], dtype=torch.int64)
        patch_rows = rows.pin_memory().to(dev, non_blocking=True)
        tunes = [len(p) for p in prompts]          # patches so far
        done = [len(p) >= max_patch for p in prompts]
        gen = [[] for _ in range(B)]
        pos = torch.arange(S + 1, device=dev).view(-1, 1)
        ops.set_pdl(True)
        try:
            for p in range(max_patch - 1):
                if all(done):
                    break
                pd.embed_patches(patch_rows[p], sp.emb)
                pd._decode_step(sp, p, False, None, inp="embed", hidden=True)
                act = [i for i in range(B) if not done[i] and tunes[i] == p + 1]
                if not act:
                    continue                        # every live tune is still inside its prompt
                # ---- spell one bar for the tunes whose last patch sits at position p
                t0 = [1 + (len(fixed[i]) if not gen[i] else 0) for i in range(B)]   # first drawn position per tune
                forced_rows = [i for i in act if t0[i] > 1]
                n_steps = max(S - 1, max(t0[i] for i in act))
                t0_dev = torch.tensor(t0, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
                if forced_rows:   # a tune whose first bar has fixed characters takes them instead of the draws
                    fx = torch.zeros(S + 1, B, dtype=torch.int64)
                    for i in forced_rows:
                        fx[1:t0[i], i] = torch.tensor(fixed[i], dtype=torch.int64)
                    fx_dev = fx.pin_memory().to(dev, non_blocking=True)
                    is_fixed = pos < t0_dev.view(1, -1)
                    forced_end = max(t0[i] for i in forced_rows)
                live = torch.zeros(B, dtype=torch.bool)
                live[act] = True
                live_dev = live.pin_memory().to(dev, non_blocking=True)
                counter_base.fill_(p * S)
                last = n_steps
                launches0, calls0 = ops.LAUNCHES, ops.CALLS
                for t in range(n_steps):
                    cd._decode_step(sc, t, True, head, inp="first" if t == 0 else "tokens")
                    stats["char_steps"] += 1
                    if forced_rows and t + 1 < forced_end:
                        sc.col[t + 1].copy_(torch.where(is_fixed[t + 1], fx_dev[t + 1], sc.col[t + 1]))
                    if t % 8 == 7 and t + 1 < n_steps:
                        seen = ((sc.col[:t + 2] == eos) & (pos[:t + 2] >= t0_dev.view(1, -1))).any(dim=0) | ~live_dev
                        stats["host_syncs"] += 1
                        if bool(seen.all()):
                            last = t + 1
                            break
                stats["char_launches"] += ops.LAUNCHES - launches0
                stats["char_calls"] += ops.CALLS - calls0
                codes = sc.col[:last + 1].t().cpu().tolist()
                stats["host_syncs"] += 1
                stats["bars"] += 1
                new_rows = {}
                for i in act:
                    drawn = codes[i][t0[i]:max(t0[i], S - 1) + 1]
                    if eos in drawn:
                        drawn = drawn[:drawn.index(eos) + 1]
                    prefix = "".join(chr(c) for c in fixed[i]) if not gen[i] else ""
                    gen[i].append(drawn)
                    bar = pz.decode([drawn])
                    if drawn[0] == eos or bar == "":
                        done[i] = True
                        continue
                    tunes[i] += 1
                    if tunes[i] >= max_patch:
                        done[i] = True
                    else:
                        new_rows[i] = pz.bar2patch(prefix + bar)
                if new_rows:
                    blk = torch.zeros(B, S, dtype=torch.int64)
                    for i, r in new_rows.items():
                        blk[i] = torch.tensor(r, dtype=torch.int64)
                    mask = torch.zeros(B, dtype=torch.bool)
                    mask[list(new_rows)] = True
                    blk_dev = blk.pin_memory().to(dev, non_blocking=True)
                    mask_dev = mask.pin_memory().to(dev, non_blocking=True)
                    patch_rows[p + 1].copy_(torch.where(mask_dev.view(-1, 1), blk_dev, patch_rows[p + 1]))
        finally:
            ops.set_pdl(False)
        return gen

    def load_reference_state_dict(self, sd):
        """Loads a state dict of the reference's `TunesFormer` (tunesformer/utils.py:179-219, HF GPT-2 parameter names): the
        patch level's `GPT2Model` under `patch_level_decoder.base.`, its `patch_embedding` Linear, the character level's
        `GPT2LMHeadModel` under `char_level_decoder.base.` (`transformer.*` and `lm_head.weight`).  Conv1D weights ([in, out]
        there) are transposed, the `attn.bias` / `attn.masked_bias` mask buffers are dropped, the patch level's tied lm_head
        is set from its wte.  Any other missing or unexpected key, or a shape mismatch, raises with the key named (a
        checkpoint with shared weights has another key set and is refused)."""
        conv = GPT._HF_CONV1D
        mask = (".attn.bias", ".attn.masked_bias")
        src = {k: v for k, v in sd.items() if not k.endswith(mask)}
        loads = []
        for dec, own_prefix in ((self.patch_level_decoder, "patch"), (self.char_level_decoder, "char")):
            own = dec.state_dict()
            out = {}
            for name, ref in own.items():
                if name == "lm_head.weight" and own_prefix == "patch":
                    continue   # tied to transformer.wte.weight
                if own_prefix == "patch":
                    key = ("patch_level_decoder." + name if name.startswith("patch_embedding.")
                           else "patch_level_decoder.base." + name.replace("transformer.", "", 1))
                elif name == "lm_head.weight":
                    key = "char_level_decoder.base.lm_head.weight"
                else:
                    key = "char_level_decoder.base." + name
                if key not in src:
                    raise KeyError(f"missing key in the TunesFormer checkpoint: {key}")
                v = src.pop(key).detach()
                if key.endswith(conv):
                    v = v.t()
                if tuple(v.shape) != tuple(ref.shape):
                    raise ValueError(f"shape mismatch for {key}: {tuple(v.shape)} vs {tuple(ref.shape)}")
                out[name] = v.contiguous()
            if own_prefix == "patch":
                out["lm_head.weight"] = out["transformer.wte.weight"]
            else:
                wte = out["transformer.wte.weight"]
                if not torch.equal(out["lm_head.weight"], wte):
                    raise ValueError("char_level_decoder.base.lm_head.weight differs from its tied transformer.wte.weight")
                out["lm_head.weight"] = wte
            loads.append((dec, out))
        if src:
            raise KeyError(f"unexpected key in the TunesFormer checkpoint: {sorted(src)[0]}")
        for dec, out in loads:   # nothing is changed unless the whole checkpoint matches
            dec.load_state_dict(out)
        return self

    def configure_optimizers(self, weight_decay, learning_rate, betas, device_type="cuda"):
        return _Optimizers([self.patch_level_decoder.configure_optimizers(weight_decay, learning_rate, betas, device_type),
                            self.char_level_decoder.configure_optimizers(weight_decay, learning_rate, betas, device_type)])

    def clip_grad_norm_(self, max_norm):
        """One global norm over both decoders, like torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm)."""
        a, b = self.patch_level_decoder, self.char_level_decoder
        na, nb = a.clip_grad_norm_(max_norm), b.clip_grad_norm_(max_norm)
        total = na.square() + nb.square()
        for m in (a, b):   # both AdamW launches read the same device scalar: the squared global norm
            ss, mx = m._pending_clip
            ss.copy_(total.reshape(1))
        return total.sqrt()


class _Optimizers:
    """step / zero_grad / param_groups over the per-decoder FusedAdamW objects."""

    def __init__(self, opts):
        self.opts = opts

    @property
    def param_groups(self):
        return [g for o in self.opts for g in o.param_groups]

    def step(self):
        for o in self.opts:
            o.step()

    def zero_grad(self, set_to_none=True):
        for o in self.opts:
            o.zero_grad(set_to_none=set_to_none)

    def state_dict(self):
        return [o.state_dict() for o in self.opts]

    def load_state_dict(self, sds):
        for o, sd in zip(self.opts, sds):
            o.load_state_dict(sd)
