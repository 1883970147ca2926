"""Large vocabularies on the GPU: the cluster sampling head of csrc/sample.cu (sample_topk_cluster_kernel, V > 56 320) against
the reference's sampling arithmetic, and the model paths a vocabulary of 98 465 whitespace tokens (the irishman corpus with
uint32 token files) runs through: vocabulary padding to a multiple of 8, lm_head GEMMs whose N / M end inside a tile, the
direct embedding-gradient kernel, a logits buffer above 2^31 elements, and train.py / sample.py end to end.

Sampler criteria are those of tests/test_sampling_gpu.py: every drawn token lies in the reference CDF interval of its Philox
uniform (widened by 2e-6 for the fp32 running sums), the drawn support stays inside the reference top-k set (ties at the
threshold included), and a chi-square test against the reference distribution.  Model criteria are those of
tests/test_model_gpu.py: the error against fp32 truth at most 1.5x the emulated bf16 reference's own error."""
import itertools
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import nanogpt_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

V_WS = 98465             # whitespace-tokenised irishman corpus
BOUND = 786432           # largest V of the cluster sampler (include/abcgpt.h abcgpt_sample_topk)
SEED = 0x1234_5678_9ABC_DEF0 & (2 ** 62 - 1)


def round_up(x, m):
    return (x + m - 1) // m * m


def draw(logits, V, temperature, top_k, seed, counter, out_stride=1, sentinel=-1):
    from ai_music_generation_b200 import ops
    B = logits.shape[0]
    out = torch.full((B * out_stride,), sentinel, device=logits.device, dtype=torch.int64)
    seed_t = torch.tensor([seed], device=logits.device, dtype=torch.int64)
    ops.sample_topk(logits, V, out, temperature, top_k, seed_t, counter, out_stride=out_stride)
    return out.cpu()


def check_every_draw(host_logits, dev_logits, V, temperature, top_k, seed, counters):
    probs = O.sampling_probs(host_logits[:, :V], temperature, top_k)
    for counter in counters:
        toks = draw(dev_logits, V, temperature, top_k, seed, counter)
        assert int(toks.min()) >= 0 and int(toks.max()) < V
        for b in range(host_logits.shape[0]):
            u = O.philox_uniform(seed, b, counter)
            assert int(toks[b]) in O.inverse_cdf_token(probs[b], u, eps=2e-6), (b, counter, int(toks[b]), u)
    return probs


def _draw_cases():
    cases = []
    for V in (56321, V_WS, 262144, BOUND):
        for j, (top_k, temperature) in enumerate(itertools.product((None, 1, 200, 4099, V - 1), (0.8, 1.3))):
            B = (1, 5, 64)[j % 3] if V <= 262144 else (1, 5)[j % 2]   # the host reference of 64 x 786 432 is slow, not harder
            # the larger row stride is not a multiple of 8: odd rows are not 16-byte aligned and take the scalar loads
            ldl = round_up(V, 8) + (4 if (j // 2 + j) % 2 else 0)
            cases.append(pytest.param(V, ldl, top_k, temperature, B, id=f"V{V}-ldl{ldl}-k{top_k}-t{temperature}-B{B}"))
    return cases


@pytest.mark.parametrize("V,ldl,top_k,temperature,B", _draw_cases())
def test_every_draw_matches_the_reference_cdf(V, ldl, top_k, temperature, B, cuda_device):
    g = torch.Generator().manual_seed(V + (top_k or 0) + B)
    logits = (torch.randn(B, ldl, generator=g) * 3.0).to(torch.bfloat16)
    logits[:, V:] = 1e4   # padding columns must never be sampled
    check_every_draw(logits, logits.to(cuda_device), V, temperature, top_k, SEED, (0, 1, 1023))


@pytest.mark.parametrize("V", [56321, V_WS, 262144])
def test_ties_at_the_threshold_are_all_kept(V, cuda_device):
    """Rows of a few distinct bf16 values: thousands of tokens tie at the k-th largest value and all of them stay in the
    support; -0.0 and +0.0 are equal values and tie as well."""
    g = torch.Generator().manual_seed(V)
    B, Vpad = 16, round_up(V, 8)
    levels = torch.tensor([-3.0, -1.0, -0.0, 0.0, 0.5, 2.0])
    logits = levels[torch.randint(len(levels), (B, Vpad), generator=g)].to(torch.bfloat16)
    logits[B // 2:] = torch.where(logits[B // 2:] > 0, torch.tensor(-3.0), logits[B // 2:]).to(torch.bfloat16)  # max is +-0
    logits[:, V:] = 1e4
    dev = logits.to(cuda_device)
    for top_k, temperature in ((1, 1.0), (200, 0.8), (V // 3, 1.3)):
        probs = check_every_draw(logits, dev, V, temperature, top_k, SEED, range(8))
        support = probs > 0
        assert int(support.sum(dim=1).min()) >= (top_k if top_k > 200 else top_k + 1)   # the ties were kept
        for c in range(8, 40):
            toks = draw(dev, V, temperature, top_k, SEED, c)
            assert bool(support.gather(1, toks.view(-1, 1)).all())
    # a constant row with top_k = 200 keeps every token: the draws reach the whole row
    const = torch.full((64, Vpad), 0.25).to(torch.bfloat16)
    const[:, V:] = 1e4
    probs = check_every_draw(const, const.to(cuda_device), V, 0.8, 200, SEED, (0, 1, 1023))
    assert bool((probs[:, :V] > 0).all())
    seen = torch.cat([draw(const.to(cuda_device), V, 0.8, 200, SEED, c) for c in range(16)])
    assert int(seen.max()) > V - V // 8 and int(seen.min()) < V // 8


def test_distribution_chi_square_and_support(cuda_device):
    V, Vpad, temperature, top_k = V_WS, round_up(V_WS, 8), 0.8, 200
    g = torch.Generator().manual_seed(5)
    row = (torch.randn(1, Vpad, generator=g) * 2.0).to(torch.bfloat16)
    row[:, V:] = 1e4
    probs = O.sampling_probs(row[:, :V], temperature, top_k)[0]
    support = set(torch.nonzero(probs > 0).flatten().tolist())
    assert len(support) >= top_k
    B, rounds = 4096, 50
    dev = row.expand(B, Vpad).contiguous().to(cuda_device)
    counts = torch.zeros(V, dtype=torch.float64)
    for r in range(rounds):
        toks = draw(dev, V, temperature, top_k, 99, r)
        counts += torch.bincount(toks, minlength=V).double()
    n = B * rounds
    assert set(torch.nonzero(counts).flatten().tolist()) <= support
    exp = probs * n
    keep = exp > 5
    chi2 = (((counts - exp) ** 2)[keep] / exp[keep]).sum().item()
    dof = int(keep.sum()) - 1
    # Wilson-Hilferty bound for p = 1e-4
    z = 3.72
    bound = dof * (1 - 2 / (9 * dof) + z * (2 / (9 * dof)) ** 0.5) ** 3
    assert chi2 < bound, (chi2, bound, dof)
    # two-sample check against torch.multinomial drawing from the reference distribution
    ref = torch.bincount(torch.multinomial(probs.float(), n, replacement=True, generator=g), minlength=V).double()
    tot = counts + ref
    k2 = tot > 10
    chi2_2 = (((counts - ref) ** 2)[k2] / tot[k2]).sum().item()
    dof2 = int(k2.sum()) - 1
    bound2 = dof2 * (1 - 2 / (9 * dof2) + z * (2 / (9 * dof2)) ** 0.5) ** 3
    assert chi2_2 < bound2, (chi2_2, bound2)


def test_determinism_streams_and_out_stride(cuda_device):
    V, Vpad = V_WS, round_up(V_WS, 8)
    g = torch.Generator().manual_seed(2)
    logits = (torch.randn(256, Vpad, generator=g) * 3.0).to(torch.bfloat16).to(cuda_device)
    for top_k in (None, 200):
        x = draw(logits, V, 1.0, top_k, 11, 3)
        assert all(torch.equal(x, draw(logits, V, 1.0, top_k, 11, 3)) for _ in range(5))
        assert not torch.equal(x, draw(logits, V, 1.0, top_k, 12, 3))    # another seed
        assert not torch.equal(x, draw(logits, V, 1.0, top_k, 11, 4))    # another decode position
        s = draw(logits, V, 1.0, top_k, 11, 3, out_stride=3, sentinel=-7)
        assert torch.equal(s[0::3], x)
        assert bool((s[1::3] == -7).all()) and bool((s[2::3] == -7).all())


def test_vocabulary_above_the_bound_is_rejected_before_launch(cuda_device):
    from ai_music_generation_b200 import _C, ops
    V = BOUND + 1
    logits = torch.zeros(1, round_up(V, 8), device=cuda_device, dtype=torch.bfloat16)
    out = torch.full((1,), -1, device=cuda_device, dtype=torch.int64)
    seed = torch.ones(1, device=cuda_device, dtype=torch.int64)
    with pytest.raises(_C.AbcgptError, match=str(BOUND)):
        ops.sample_topk(logits, V, out, 0.8, 200, seed, 0)
    torch.cuda.synchronize()
    assert int(out[0]) == -1   # nothing was written
    # the bound itself still samples
    assert 0 <= int(draw(logits[:, :BOUND], BOUND, 0.8, 200, 1, 0)[0]) < BOUND


# ---- model paths at V = 98 465 ------------------------------------------------------------------------------------------

def cfg_dict(bias, block_size=64, n_layer=2, n_head=2, n_embd=128):
    return dict(block_size=block_size, vocab_size=V_WS, n_layer=n_layer, n_head=n_head, n_embd=n_embd, dropout=0.0, bias=bias)


def make(cfgd, device, seed=1):
    from ai_music_generation_b200 import GPT, GPTConfig
    cfg = O.OracleConfig(**cfgd)
    sd = O.synthetic_state(cfg, seed=seed)
    model = GPT(GPTConfig(**cfgd))
    model.load_state_dict({**sd, "lm_head.weight": sd["transformer.wte.weight"]})
    return cfg, sd, model.to(device)


@pytest.mark.parametrize("bias", [False, True])
def test_forward_backward_match_bf16_oracle(bias, cuda_device):
    cfg, sd, model = make(cfg_dict(bias), cuda_device)
    model.train()
    x, y = O.synthetic_tokens(cfg, 4, 64, seed=0)
    logits, loss = model(x.to(cuda_device), y.to(cuda_device))
    loss.backward()
    torch.set_num_threads(8)
    ref_loss, ref_logits, ref_grads = O.loss_and_grads(sd, cfg, x, y, bf16=True)
    tru_loss, tru_logits, tru_grads = O.loss_and_grads(sd, cfg, x, y, bf16=False)
    assert abs(loss.item() - ref_loss.item()) <= 2e-3, (loss.item(), ref_loss.item(), tru_loss.item())
    assert logits.shape == (4, 64, V_WS)
    ours = (logits.float().cpu() - tru_logits).abs()
    refs = (ref_logits - tru_logits).abs()
    assert ours.max().item() <= 1.5 * refs.max().item() + 1e-2, (ours.max().item(), refs.max().item())
    assert ours.mean().item() <= 1.5 * refs.mean().item() + 1e-3, (ours.mean().item(), refs.mean().item())
    named = dict(model.named_parameters())
    for n, tg in tru_grads.items():
        got = named[n].grad.float().cpu()
        ours_rel = ((got - tg).norm() / tg.norm()).item()
        ref_rel = ((ref_grads[n] - tg).norm() / tg.norm()).item()
        assert ours_rel <= 1.5 * ref_rel + 5e-3, (n, ours_rel, ref_rel)


def test_three_adamw_steps_track_oracle(cuda_device):
    cfg, sd, model = make(cfg_dict(True), cuda_device)
    model.train()
    batches = [O.synthetic_tokens(cfg, 4, 64, seed=s) for s in range(3)]
    opt = model.configure_optimizers(0.1, 1e-3, (0.9, 0.95), "cuda")
    losses = []
    for x, y in batches:
        _, loss = model(x.to(cuda_device), y.to(cuda_device))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        model.clip_grad_norm_(1.0)
        opt.step()
        losses.append(loss.item())
    torch.set_num_threads(8)
    ref_sd = {k: v.clone() for k, v in sd.items()}
    ref = O.train_steps(ref_sd, cfg, batches, lr=1e-3, betas=(0.9, 0.95), bf16=True)
    for step, (got, (want, _)) in enumerate(zip(losses, ref)):
        assert abs(got - want) <= (2e-3 if step == 0 else 1e-2), (step, got, want)
    named = dict(model.named_parameters())
    for n, p in ref_sd.items():
        assert named[n].detach().norm().item() == pytest.approx(p.norm().item(), rel=2e-3), n


def test_greedy_kv_cache_equals_recompute(cuda_device):
    cfg, sd, model = make(cfg_dict(False), cuda_device)
    model.eval()
    prompt, _ = O.synthetic_tokens(cfg, 3, 6, seed=11)
    n_new = 50
    a = model.generate(prompt.to(cuda_device), n_new, top_k=1, use_cache=True).cpu()
    b = model.generate(prompt.to(cuda_device), n_new, top_k=1, use_cache=False).cpu()
    assert a.shape == b.shape == (3, 6 + n_new)
    assert torch.equal(a[:, :6], prompt)
    # identical ids, except after a position where the recompute path's own top-2 logits are within the bf16 tolerance
    for row in range(3):
        diff = (a[row] != b[row]).nonzero()
        if len(diff):
            pos = diff[0].item() - 1
            logits, _ = model(a[row:row + 1, :pos + 1].to(cuda_device))
            top2 = logits[0, -1].float().topk(2).values
            assert (top2[0] - top2[1]).item() <= 6e-2, (row, pos, top2)
    # every token the cached path picked is the argmax of the recompute path's logits for the same context, up to tolerance
    for pos in range(5, a.shape[1] - 1):
        logits, _ = model(a[:, :pos + 1].to(cuda_device))
        lg = logits[:, -1].float().cpu()
        picked = lg.gather(1, a[:, pos + 1:pos + 2]).squeeze(1)
        assert bool((picked >= lg.max(dim=1).values - 6e-2).all()), (pos, picked, lg.max(dim=1).values)


def test_generate_with_sample_py_defaults_is_fused_and_reproducible(cuda_device):
    from ai_music_generation_b200 import ops
    cfg, sd, model = make(cfg_dict(False), cuda_device, seed=4)
    model.eval()
    idx = torch.zeros(8, 1, dtype=torch.int64, device=cuda_device)
    names = []
    orig = ops._call

    def spy(name, *a, **k):
        names.append(name)
        return orig(name, *a, **k)

    ops._call = spy
    try:
        torch.manual_seed(1337)
        a = model.generate(idx, 40, temperature=0.8, top_k=200)
    finally:
        ops._call = orig
    assert "sample_topk" in names and "argmax" not in names
    torch.manual_seed(1337)
    b = model.generate(idx, 40, temperature=0.8, top_k=200)
    c = model.generate(idx, 40, temperature=0.8, top_k=200)
    assert torch.equal(a, b)
    assert not torch.equal(a, c)
    assert a.shape == (8, 41) and int(a.max()) < V_WS and int(a.min()) >= 0
    assert len({tuple(r.tolist()) for r in a}) > 1
    # the window-sliding tail (reference-style recompute, out_stride = out.stride(0)) goes through the same head
    torch.manual_seed(7)
    d = model.generate(idx, 70, temperature=0.8, top_k=200)
    torch.manual_seed(7)
    e = model.generate(idx, 70, temperature=0.8, top_k=200)
    assert torch.equal(d, e)
    assert d.shape == (8, 71) and int(d.max()) < V_WS and int(d.min()) >= 0


def test_ragged_prompts_equal_one_at_a_time(cuda_device):
    cfg, sd, model = make(cfg_dict(True), cuda_device)
    model.eval()
    torch.manual_seed(3)
    lens = [3, 9, 1, 14]
    n_new = 30
    padded = torch.zeros(len(lens), max(lens), dtype=torch.long)
    prompts = []
    for r, n in enumerate(lens):
        prompts.append(torch.randint(1, V_WS, (1, n)))
        padded[r, :n] = prompts[-1][0]
    out = model.generate(padded.to(cuda_device), n_new, top_k=1, prompt_lens=lens).cpu()
    for r, n in enumerate(lens):
        alone = model.generate(prompts[r].to(cuda_device), n_new, top_k=1).cpu()[0]
        assert torch.equal(out[r, :n + n_new], alone), (r, n)


def test_training_step_with_logits_above_two_to_the_31(cuda_device):
    """B * T = 32 768 tokens at V = 98 465: the logits buffer holds 3.2 G elements.  The loss must be the fp32 cross-entropy
    of the returned logits, and every gradient finite."""
    import torch.nn.functional as F
    B, T = 32, 1024
    cfgd = cfg_dict(False, block_size=T, n_layer=1)
    _, _, model = make(cfgd, cuda_device)
    model.train()
    g = torch.Generator().manual_seed(0)
    x = torch.randint(V_WS, (B, T), generator=g).to(cuda_device)
    y = torch.randint(V_WS, (B, T), generator=g).to(cuda_device)
    logits, loss = model(x, y)
    assert logits.shape == (B, T, V_WS)
    assert logits.untyped_storage().nbytes() // 2 > 2 ** 31
    loss.backward()
    with torch.no_grad():
        total = torch.zeros((), dtype=torch.float64, device=cuda_device)
        for b in range(B):   # one sequence (1 024 rows) at a time
            total += F.cross_entropy(logits[b].float(), y[b], reduction="sum").double()
        want = (total / (B * T)).item()
    assert loss.item() == pytest.approx(want, rel=1e-4, abs=1e-4), (loss.item(), want)
    for n, p in model.named_parameters():
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()), n
        assert p.grad.abs().sum().item() > 0, n


def test_train_then_sample_whitespace_tokens_end_to_end(tmp_path, cuda_device):
    """The irishman whitespace recipe: uint32 token files, out_dir out-irishman-whitespace (train.py reads uint32 there, like
    the reference), then sample.py with its default temperature 0.8 and top_k 200 and the whitespace codec."""
    itos = {i: f"t{i}" for i in range(V_WS)}
    itos[0], itos[1] = "$", "|"
    stoi = {s: i for i, s in itos.items()}
    rng = np.random.default_rng(0)
    tune = np.concatenate([[0], rng.integers(2, V_WS, size=40), [1], rng.integers(70000, V_WS, size=20), [1]])
    ids = np.tile(tune, 300).astype(np.uint32)
    assert int(ids.max()) > 65535
    d = tmp_path / "data" / "irishman_whitespace"
    d.mkdir(parents=True)
    ids[: int(0.9 * len(ids))].tofile(d / "train.bin")
    ids[int(0.9 * len(ids)):].tofile(d / "val.bin")
    with open(d / "meta.pkl", "wb") as f:
        pickle.dump({"vocab_size": V_WS, "itos": itos, "stoi": stoi}, f)
    env = dict(os.environ, PYTHONPATH=ROOT)
    common = ["--dataset=irishman_whitespace", "--out_dir=out-irishman-whitespace"]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "train.py"), *common, "--n_layer=2", "--n_head=2", "--n_embd=128",
                        "--block_size=64", "--batch_size=8", "--gradient_accumulation_steps=1", "--max_iters=10",
                        "--eval_interval=5", "--eval_iters=2", "--log_interval=5", "--learning_rate=1e-3",
                        "--warmup_iters=2", "--lr_decay_iters=10", "--min_lr=1e-4"],
                       cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert f"found vocab_size = {V_WS}" in r.stdout
    assert os.path.exists(tmp_path / "out-irishman-whitespace" / "ckpt.pt")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "sample.py"), *common, "--tokens_format=midi",
                        "--use_validation_prefixes=False", "--num_samples=3", "--max_new_tokens=70"],
                       cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    outs = sorted(os.listdir(tmp_path / "out-irishman-whitespace" / "samples"))
    assert outs == ["sample_0.txt", "sample_1.txt", "sample_2.txt"]
    for o in outs:
        text = open(tmp_path / "out-irishman-whitespace" / "samples" / o).read()
        assert all(tok in stoi for tok in text.split()), text[:200]
