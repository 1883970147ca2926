"""TunesFormer generation on the device: the nucleus / top-k / temperature kernel (abcgpt_sample_top_p), the KV-cached patch
and character decode steps, and the batched bar loop (TunesFormerShaped.generate_patches / generate_tunes).

  * the sampler, per draw: its uniform is a pure function of (seed, row id, counter base + position) with a host twin
    (oracle.philox_uniform), so every drawn token must lie in the CDF interval of that uniform under the distribution of the
    host restatement (tunesformer.top_p_filter -> top_k_filter -> temperature power) of softmax(float(logits));
  * the sampler, in distribution: chi-square against the restated distribution, support inside the kept set;
  * both caches against the full-forward recompute, relative to the recompute's own error against the fp32 oracle;
  * greedy bars against the unmodified reference's fixture, batched tunes against generate_tune one at a time;
  * reproducibility and the host synchronisations per bar.
"""
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import nanogpt_oracle as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MARGIN = 0.03   # the rule of test_model_gpu.py: compare up to the first reference decision closer than this


def restated(logits_row, top_p, top_k, temperature):
    """(draw distribution, kept set) of the host restatement, applied to softmax(float(logits))."""
    from ai_music_generation_b200 import tunesformer as TF
    probs = torch.softmax(logits_row.float(), dim=-1).numpy()
    p = TF.top_k_filter(TF.top_p_filter(probs, top_p), top_k)
    kept = set(np.nonzero(p)[0].tolist())
    if temperature <= 0.0 or np.count_nonzero(p) == 1:
        q = np.zeros(p.size)
        q[int(np.argmax(p))] = 1.0
    else:
        q = np.power(p.astype(np.float64), 1.0 / temperature)
        q /= q.sum()
    return torch.from_numpy(q), kept


def near_cut(logits_row, top_p):
    """True when a running sum of the sorted probabilities lies within 1e-6 of top_p (the cut may go either way)."""
    if top_p >= 1.0:
        return False
    probs = torch.softmax(logits_row.float(), dim=-1).double()
    csum = torch.cumsum(torch.sort(probs, descending=True).values, 0)
    return bool(((csum - top_p).abs() < 1e-6).any())


def draw(logits, V, top_p, top_k, temperature, seed, base, counter, row_id=None):
    from ai_music_generation_b200 import ops
    dev = logits.device
    out = torch.full((logits.shape[0],), -1, device=dev, dtype=torch.int64)
    ops.sample_top_p(logits, V, out, top_p, top_k, temperature, torch.tensor([seed], device=dev, dtype=torch.int64),
                     torch.tensor([base], device=dev, dtype=torch.int64), counter, row_id=row_id)
    return out.cpu()


def tie_rows(B, V, g):
    """Rows with many exactly equal logits (ties at the top-k boundary) and a nucleus cut that lands inside a tie."""
    rows = (torch.randint(-4, 5, (B, V), generator=g).float() * 0.5).to(torch.bfloat16)
    rows[0] = -1000.0
    rows[0, [5, 9, 17, 40]] = 0.0    # four tokens of p = 1/4: top_p 0.6 keeps 5, 9, 17 and not the tied 40
    return rows


SETTINGS = [  # (top_p, top_k, temperature)
    (0.8, 8, 1.2), (1.0, 0, 1.0), (1.0, 0, 0.7), (0.5, 0, 1.0), (0.95, 20, 2.0), (0.6, 3, 1.0), (0.8, 1, 1.2),
    (0.8, 8, 0.0), (0.9, 0, -1.0), (1.0, 127, 1.0), (0.3, 500, 0.9), (0.0, 0, 1.0),
]


@pytest.mark.parametrize("V,Vpad", [(128, 128), (95, 128), (1024, 1024), (1, 128)])
@pytest.mark.parametrize("top_p,top_k,temperature", SETTINGS)
def test_every_draw_matches_the_restated_cdf(V, Vpad, top_p, top_k, temperature, cuda_device):
    g = torch.Generator().manual_seed(V * 7 + int(top_p * 100) + top_k)
    B = 48
    logits = (torch.randn(B, Vpad, generator=g) * 3.0).to(torch.bfloat16)
    if V >= 64:
        logits[: B // 2, :V] = tie_rows(B // 2, V, g)
    logits[:, V:] = 1e4   # padding columns must never be read
    dev = logits.to(cuda_device)
    row_id = torch.randperm(10_000, generator=g)[:B]
    seed = 0x0F1E_2D3C_4B5A_6978
    for base, counter in ((0, 0), (7 * 32, 5), (123 * 32, 31)):
        toks = draw(dev, V, top_p, top_k, temperature, seed, base, counter, row_id.to(cuda_device))
        for b in range(B):
            q, kept = restated(logits[b, :V], top_p, top_k, temperature)
            tok = int(toks[b])
            if near_cut(logits[b, :V], top_p):
                assert 0 <= tok < V
                continue
            assert tok in kept, (b, tok, sorted(kept))
            u = O.philox_uniform(seed, int(row_id[b]), base + counter)
            assert tok in O.inverse_cdf_token(q, u, eps=2e-6), (b, base, counter, tok, u)


@pytest.mark.parametrize("top_p,top_k", [(0.8, 8), (0.6, 0), (0.95, 20), (0.6, 3)])
def test_kept_set_equals_the_restatement(top_p, top_k, cuda_device):
    """At a temperature of 50 the weights of the kept tokens are nearly equal, so 4096 draws per row reach every one of them."""
    V = 128
    g = torch.Generator().manual_seed(11 + top_k)
    rows = torch.cat([tie_rows(4, V, g), (torch.randn(4, V, generator=g) * 2.0).to(torch.bfloat16)])
    for r in range(rows.shape[0]):
        if near_cut(rows[r], top_p):
            continue
        _, kept = restated(rows[r], top_p, top_k, 50.0)
        dev = rows[r:r + 1].expand(4096, V).contiguous().to(cuda_device)
        seen = set(draw(dev, V, top_p, top_k, 50.0, 5, r, 0).tolist())
        assert seen == kept, (r, sorted(seen), sorted(kept))


def test_distribution_chi_square_streams_and_bounds(cuda_device):
    from ai_music_generation_b200 import _C, ops
    V, top_p, top_k, temperature = 128, 0.95, 24, 1.2
    g = torch.Generator().manual_seed(3)
    row = (torch.randn(1, V, generator=g) * 1.5).to(torch.bfloat16)
    q, kept = restated(row[0], top_p, top_k, temperature)
    assert len(kept) >= 8
    B, rounds = 4096, 50
    dev = row.expand(B, V).contiguous().to(cuda_device)
    ids = torch.arange(B, device=cuda_device)
    counts = torch.zeros(V, dtype=torch.float64)
    for r in range(rounds):   # counter base varied, the row ids name 4096 streams
        counts += torch.bincount(draw(dev, V, top_p, top_k, temperature, 99, 1000 + 32 * r, 3, ids), minlength=V).double()
    n = B * rounds
    assert set(torch.nonzero(counts).flatten().tolist()) <= kept
    exp = q * n
    keep = exp > 5
    chi2 = (((counts - exp) ** 2)[keep] / exp[keep]).sum().item()
    dof = int(keep.sum()) - 1
    z = 3.72   # Wilson-Hilferty bound for p = 1e-4
    bound = dof * (1 - 2 / (9 * dof) + z * (2 / (9 * dof)) ** 0.5) ** 3
    assert chi2 < bound, (chi2, bound, dof)
    # streams
    rows = (torch.randn(256, V, generator=g) * 2.0).to(torch.bfloat16).to(cuda_device)
    a = draw(rows, V, 0.9, 0, 1.5, 42, 64, 3)
    assert torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 64, 3))
    assert torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 64, 3, torch.arange(256, device=cuda_device)))   # NULL = arange
    assert not torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 43, 64, 3))
    assert not torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 96, 3))
    assert not torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 64, 3, torch.arange(256, device=cuda_device) + 1))
    assert torch.equal(draw(rows, V, 0.9, 0, 1.5, 42, 60, 7), draw(rows, V, 0.9, 0, 1.5, 42, 64, 3))   # base + counter
    big = torch.zeros(2, 1152, device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros(2, device=cuda_device, dtype=torch.int64)
    one = torch.zeros(1, device=cuda_device, dtype=torch.int64)
    with pytest.raises(_C.AbcgptError, match="1025"):
        ops.sample_top_p(big, 1025, out, 0.8, 8, 1.0, one, one, 0)
    ops.sample_top_p(big, 1024, out, 0.8, 8, 1.0, one, one, 0)


# ---- models --------------------------------------------------------------------------------------------------------------
def tiny_model(cuda_device, wte_scale=None):
    from ai_music_generation_b200 import GPTConfig, TunesFormerShaped
    from oracle.make_golden_tunesformer import SPEC, inputs
    pc, cc, psd, csd, patches = inputs(SPEC)
    if wte_scale is not None:
        csd = dict(csd)
        csd["transformer.wte.weight"] = csd["transformer.wte.weight"] * wte_scale
    model = TunesFormerShaped(GPTConfig(**SPEC["patch_cfg"]), GPTConfig(**SPEC["char_cfg"]))
    model.patch_level_decoder.load_state_dict({**psd, "lm_head.weight": psd["transformer.wte.weight"]})
    model.char_level_decoder.load_state_dict({**csd, "lm_head.weight": csd["transformer.wte.weight"]})
    return model.to(cuda_device).eval(), (pc, cc, psd, csd), patches


def full_model(cuda_device):
    from ai_music_generation_b200 import GPTConfig, TunesFormerShaped
    pd_ = dict(block_size=128, vocab_size=1, n_layer=9, n_head=12, n_embd=768, dropout=0.0, bias=True, activation="gelu_tanh")
    cd_ = dict(block_size=32, vocab_size=128, n_layer=3, n_head=12, n_embd=768, dropout=0.0, bias=True, activation="gelu_tanh")
    pc, cc = O.OracleConfig(**pd_), O.OracleConfig(**cd_)
    psd, csd = O.synthetic_state(pc, seed=21), O.synthetic_state(cc, seed=22)
    g = torch.Generator().manual_seed(23)
    psd["patch_embedding.weight"] = torch.randn(768, 32 * 128, generator=g) * 0.02
    psd["patch_embedding.bias"] = torch.randn(768, generator=g) * 0.02
    model = TunesFormerShaped(GPTConfig(**pd_), GPTConfig(**cd_))
    model.patch_level_decoder.load_state_dict({**psd, "lm_head.weight": psd["transformer.wte.weight"]})
    model.char_level_decoder.load_state_dict({**csd, "lm_head.weight": csd["transformer.wte.weight"]})
    patches = torch.randint(3, 128, (3, 6, 32), generator=g)
    lens = torch.randint(6, 33, (3, 6), generator=g)
    patches[torch.arange(32)[None, None, :] >= lens[..., None]] = 0
    return model.to(cuda_device).eval(), (pc, cc, psd, csd), patches


@pytest.mark.parametrize("shape", ["tiny", "full"])
@torch.no_grad()
def test_cached_steps_match_the_recompute(shape, cuda_device):
    import torch.nn.functional as F
    if shape == "tiny":
        model, (pc, cc, psd, csd), patches = tiny_model(cuda_device)
        patches = torch.cat([patches[:, :8], patches[:, 2:10], patches[:, 4:12]])   # 3 tunes x 8 patches
    else:
        model, (pc, cc, psd, csd), patches = full_model(cuda_device)
    pd, cd = model.patch_level_decoder, model.char_level_decoder
    B, P, S = patches.shape
    dev_patches = patches.to(cuda_device)
    sp, sc = model._decode_states(B, cuda_device)
    oh = F.one_hot(patches, 128).float().reshape(B, P, S * 128)
    emb = oh @ psd["patch_embedding.weight"].t() + psd["patch_embedding.bias"]
    _, _, truth_h = O.forward(psd, pc, None, None, return_hidden=True, inputs_embeds=emb)
    pd._ensure_device_state()
    for p in range(P):
        pd.embed_patches(dev_patches[:, p].contiguous(), sp.emb)
        pd._decode_step(sp, p, False, None, inp="embed", hidden=True)
        got = sp.hidden.cpu()
        full = pd.encode(dev_patches[:, :p + 1])[:, -1].cpu()
        truth = truth_h[:, p]
        e_got, e_full = (got - truth).abs().max().item(), (full - truth).abs().max().item()
        assert e_got <= 1.5 * e_full + 2e-3 * truth.abs().max().item(), (p, e_got, e_full)
    # character level: first = the patch level's last hidden rows, then characters of the next patch
    first = sp.hidden.clone()
    chars = patches[:, -1].clone()
    chars[:, 0] = 1
    chars[chars == 0] = 2
    sc.col[:S].copy_(chars.t().to(cuda_device))
    cd._ensure_device_state()
    for t in range(S):
        cd._decode_step(sc, t, True, None, inp="first" if t == 0 else "tokens")
        got = sc.logits[:, :128].float().cpu()
        full = cd.next_logits_with_first(chars[:, :t + 1].to(cuda_device), first).cpu()
        truth, _ = O.forward(csd, cc, chars[:, :t + 1], first_embeds=first.cpu())
        truth = truth[:, -1]
        e_got, e_full = (got - truth).abs().max().item(), (full - truth).abs().max().item()
        assert e_got <= 1.5 * e_full + 2e-3 * truth.abs().max().item(), (t, e_got, e_full)


def test_greedy_bars_match_the_reference_fixture(cuda_device):
    with open(os.path.join(GOLDEN, "tunesformer_tiny_generate.json")) as f:
        g = json.load(f)
    model, _, patches = tiny_model(cuda_device, g["char_wte_scale"])
    n0 = g["n_prompt_patches"]
    margins = iter(g["margins"])
    # the loop feeds back its own bars (bar2patch of what it drew), four of them from 5 prompt patches up to max_patch = 9
    gen = model.generate_patches([patches[0, :n0]], max_patch=n0 + 4, top_k=1)[0]
    assert len(gen) == len(g["generated"]) == 4
    compared = 0
    for got, want in zip(gen, g["generated"]):
        ms = [next(margins) for _ in want]
        n_ok = next((i for i, m in enumerate(ms) if m < MARGIN), len(ms))
        assert got[:n_ok] == want[:n_ok] and len(got) == len(want), (got, want)
        compared += n_ok
    assert compared == 124
    # fixed characters after bos: the first bar continues them
    fixed = g["fixed_tokens"][1:]
    got2 = model.generate_patches([patches[0, :n0]], [fixed], max_patch=n0 + 1, top_k=1)[0]
    ms = [next(margins) for _ in g["with_fixed_tokens"]]
    n_ok = next((i for i, m in enumerate(ms) if m < MARGIN), len(ms))
    assert len(got2) == 1 and got2[0][:n_ok] == g["with_fixed_tokens"][:n_ok]
    assert len(got2[0]) == len(g["with_fixed_tokens"])


PROMPTS = [
    "X:1\nL:1/8\nM:3/4\nK:D\n",
    "X:1\nK:G\n",
    "",
    "X:2\nT:a\nM:4/4\nL:1/8\nK:D\n|: A2 B2 | c4 d4 |",
    "X:2\nK:D\n de |\"D\" fa",
    "S:2\nB:9\nE:4\nB:9\nL:1/8\nM:3/4\nK:D\n de |\"D\" ",
    "X:3\nK:A\nabc",
    "X:4\nK:D\n" + "a|" * 12,          # already at max_patch
    "X:5\nM:6/8\nK:Em\n|: E2 F G2 A |",
]


def _host_reference(model, prompt, max_patch, monkeypatch):
    """generate_tune(prompt, top_k=1) plus, per draw, (token, top-2 margin of its probabilities)."""
    from ai_music_generation_b200 import tunesformer as TF
    log = []
    orig_p, orig_d = TF.top_p_filter, TF.temperature_draw

    def top_p(probs, top_p):
        o = np.sort(probs)[::-1]
        log.append([None, float(o[0] - o[1]) if o.size > 1 else 1.0])
        return orig_p(probs, top_p)

    def draw_(probs, temperature, seed=None):
        tok = orig_d(probs, temperature, seed)
        log[-1][0] = tok
        return tok

    monkeypatch.setattr(TF, "top_p_filter", top_p)
    monkeypatch.setattr(TF, "temperature_draw", draw_)
    try:
        text = model.generate_tune(prompt, max_patch=max_patch, top_k=1)
    finally:
        monkeypatch.setattr(TF, "top_p_filter", orig_p)
        monkeypatch.setattr(TF, "temperature_draw", orig_d)
    return text, log


def test_batched_tunes_equal_generating_each_alone(cuda_device, monkeypatch):
    from ai_music_generation_b200.tunesformer import Patchilizer
    with open(os.path.join(GOLDEN, "tunesformer_tiny_generate.json")) as f:
        scale = json.load(f)["char_wte_scale"]
    model, _, _ = tiny_model(cuda_device, scale)
    max_patch = 12
    pz = Patchilizer()
    counts = [len(pz.encode(p, add_special_patches=True)[:-1]) for p in PROMPTS]
    assert len(set(counts)) >= 4 and max(counts) >= max_patch
    refs = [_host_reference(model, prompt, max_patch, monkeypatch) for prompt in PROMPTS]
    # one batch, then batches of 3 (prompts grouped by patch count)
    for batch in (64, 3):
        got = model.generate_tunes(PROMPTS, max_patch=max_patch, top_k=1, batch=batch)
        stats = model.last_generate_stats
        for prompt, text, (want, log) in zip(PROMPTS, got, refs):
            k = next((i for i, (_, m) in enumerate(log) if m < MARGIN), len(log))
            n_chars = sum(1 for tok, _ in log[:k] if tok > 2)   # every drawn code > 2 is one character of the text
            if k == len(log):
                assert text == want, (batch, prompt, text, want)
            else:
                assert text[:len(prompt) + n_chars] == want[:len(prompt) + n_chars], (batch, prompt, text, want)
        assert got[PROMPTS.index("X:4\nK:D\n" + "a|" * 12)] == "X:4\nK:D\n" + "a|" * 12
        assert stats["bars"] > 0 and stats["host_syncs"] <= (1 + math.ceil(31 / 8)) * stats["bars"]


def test_sampled_tunes_are_reproducible(cuda_device):
    model, _, _ = tiny_model(cuda_device, 40.0)
    kw = dict(max_patch=10, top_p=0.8, top_k=8, temperature=1.2)
    a = model.generate_tunes(PROMPTS, seed=1234, **kw)
    assert model.generate_tunes(PROMPTS, seed=1234, **kw) == a
    assert all(t.startswith(p) for t, p in zip(a, PROMPTS))
    assert model.generate_tunes(PROMPTS, seed=1235, **kw) != a
    torch.manual_seed(7)
    b = model.generate_tunes(PROMPTS, **kw)
    torch.manual_seed(7)
    assert model.generate_tunes(PROMPTS, **kw) == b
    stats = model.last_generate_stats
    assert stats["bars"] > 0 and stats["host_syncs"] <= (1 + math.ceil(31 / 8)) * stats["bars"]
    with pytest.raises(ValueError, match="max_patch"):
        model.generate_tunes(PROMPTS[:1], max_patch=17)   # above the patch decoder's block_size (16)
