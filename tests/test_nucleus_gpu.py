"""Nucleus / top-k / temperature sampling for every vocabulary: the cluster kernel (abcgpt_sample_top_p_cluster), its
agreement with the one-CTA kernel, GPT.generate(top_p=...) on the cached, ragged and slid-window paths, and sample.py --top_p.

  * every draw lies in the CDF interval of its host-regenerated uniform (oracle.philox_uniform) under a restatement of the
    chain: ranks by descending logit (the exact softmax's order) with a stable sort, fp64 running sums, the nucleus cut taken
    either way only where a running sum lies within CUT_TOL of top_p;
  * ties at both cuts keep the lowest indices, also when the tie class spans two CTA slices;
  * the one-CTA and the cluster kernel give the same token on every row whose cut and draw are unambiguous;
  * a row draws the same tokens alone and inside any batch, given the same row id.
"""
import json
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
CUT_TOL = 1e-6       # include/abcgpt.h abcgpt_sample_top_p_cluster: the mass fraction of any prefix is within this of exact
DRAW_EPS = 2e-6      # fp32 exp and the fixed-point weights move a CDF boundary by less than this (relative)
V_WS = 98465         # whitespace tokens of the irishman corpus
SEED = 0x1234_5678_9ABC_DEF


def slice_of(V):
    return ((V + 7) // 8 + 7) // 8 * 8


def make_logits(B, V, ldl, g, ties=True):
    """[B, ldl] bf16: random rows of several widths, half of them with many exactly equal logits; padding = 1e4 (never read)."""
    scale = torch.linspace(0.5, 4.0, B).view(B, 1)
    rows = torch.randn(B, V, generator=g) * scale
    if ties:
        rows[: B // 2] = torch.randint(-6, 7, (B // 2, V), generator=g).float() * 0.5
    out = torch.full((B, ldl), 1e4)
    out[:, :V] = rows
    return out.to(torch.bfloat16)


class Chain:
    """Host restatement of one row: order, fp64 probabilities and running sums, computed once per row."""

    def __init__(self, row_bf16):
        x = row_bf16.double().numpy()
        self.V = x.size
        self.order = np.argsort(-x, kind="stable")       # descending logit, ties by lower index
        p = np.exp(x - x.max())
        self.p = p / p.sum()
        self.csum = np.cumsum(self.p[self.order])
        self.argmax = int(self.order[0])

    def nucleus_sizes(self, top_p, tol=CUT_TOL):
        """Every nucleus size a kernel may pick: the exact one, and its neighbours whose running sums lie within tol of top_p."""
        if top_p >= 1.0:
            return [self.V]
        lo = int(np.searchsorted(self.csum, top_p - tol, side="left"))
        hi = int(np.searchsorted(self.csum, top_p + tol, side="left"))
        return list(range(lo + 1, min(hi, self.V - 1) + 2))

    def kept(self, n):
        return self.order[:n]

    def candidates(self, top_p, top_k, temperature, u, eps=DRAW_EPS):
        """Tokens the draw may return for the uniform u, over every admissible nucleus cut."""
        toks = set()
        for n in self.nucleus_sizes(top_p):
            if 0 < top_k < n:
                n = top_k
            if temperature <= 0.0 or n == 1:
                toks.add(self.argmax)
                continue
            q = np.zeros(self.V)
            k = self.kept(n)
            q[k] = np.power(self.p[k] / self.p[self.argmax], 1.0 / temperature)
            q /= q.sum()
            toks |= O.inverse_cdf_token(torch.from_numpy(q), u, eps=eps)
        return toks

    def ambiguous(self, top_p, top_k, temperature, u, tol=5e-6):
        """True where the two kernels may legitimately differ: a running sum within tol of top_p, or u within tol of a CDF
        boundary of the draw."""
        if top_p < 1.0 and bool((np.abs(self.csum - top_p) < tol).any()):
            return True
        n = self.nucleus_sizes(top_p, 0.0)[0]
        if 0 < top_k < n:
            n = top_k
        if temperature <= 0.0 or n == 1:
            return False
        q = np.zeros(self.V)
        k = self.kept(n)
        q[k] = np.power(self.p[k] / self.p[self.argmax], 1.0 / temperature)
        cdf = np.cumsum(q) / q.sum()
        return bool((np.abs(cdf - u) < tol).any())


def scalars(dev, seed, base):
    return (torch.tensor([seed], device=dev, dtype=torch.int64), torch.tensor([base], device=dev, dtype=torch.int64))


def draw(logits, V, top_p, top_k, temperature, seed, base, counter, row_id=None, cluster=True):
    from ai_music_generation_b200 import ops
    dev = logits.device
    out = torch.full((logits.shape[0],), -1, device=dev, dtype=torch.int64)
    fn = ops.sample_top_p_cluster if cluster else ops.sample_top_p
    s, b = scalars(dev, seed, base)
    fn(logits, V, out, top_p, top_k, temperature, s, b, counter, row_id=row_id)
    return out.cpu()


# ---- 1. the contract -----------------------------------------------------------------------------------------------------
CASES = [  # (V, ldl, B): ragged slices everywhere but 4096 and 786 432; odd strides take the unaligned load path
    (1031, 1037, 64), (4096, 4104, 64), (50257, 50263, 16), (V_WS, 98472, 16), (786432, 786440, 4)]


@pytest.mark.parametrize("V,ldl,B", CASES)
def test_every_draw_lies_in_the_restated_cdf(V, ldl, B, cuda_device):
    g = torch.Generator().manual_seed(V)
    logits = make_logits(B, V, ldl, g)
    dev = logits.to(cuda_device)
    row_id = torch.randperm(100_000, generator=g)[:B]
    chains = [Chain(logits[b, :V]) for b in range(B)]
    temps = (0.0, 0.7, 1.2)
    i = 0
    for top_p in (0.5, 0.8, 0.95, 1.0):
        for top_k in (0, 1, 8, 200, V + 3):
            temperature = temps[i % 3]
            i += 1
            base, counter = 17 * i, 3
            toks = draw(dev, V, top_p, top_k, temperature, SEED, base, counter, row_id.to(cuda_device))
            for b in range(B):
                u = O.philox_uniform(SEED, int(row_id[b]), base + counter)
                ok = chains[b].candidates(top_p, top_k, temperature, u)
                assert int(toks[b]) in ok, (V, b, top_p, top_k, temperature, int(toks[b]), sorted(ok)[:8])


# ---- 2. ties at both cuts ------------------------------------------------------------------------------------------------
def test_ties_keep_the_lowest_indices_across_slices(cuda_device):
    V = 4096
    sl = slice_of(V)                                   # 512: the tie class below straddles slices 0 and 1
    tied = [sl - 12, sl - 7, sl - 2, sl + 3, sl + 8, sl + 30]
    row = torch.full((V,), -30.0)
    row[3000] = 1.0                                    # p = e / (e + 6) = 0.312, each tied token 0.115
    row[tied] = 0.0
    row = row.to(torch.bfloat16)
    chain = Chain(row)
    B = 4096
    dev = row.view(1, V).expand(B, V).contiguous().to(cuda_device)
    ids = torch.arange(B, device=cuda_device)
    # (top_p, top_k) -> kept set: the nucleus cut inside the tie class (0.312 + 0.115 j), the top-k cut inside it, both
    for top_p, top_k, n in ((0.6, 0, 4), (0.7, 0, 5), (1.0, 3, 3), (1.0, 5, 5), (0.9, 4, 4), (0.5, 200, 3)):
        want = {3000, *tied[: n - 1]}
        assert set(chain.kept(n).tolist()) == want
        seen = set(draw(dev, V, top_p, top_k, 50.0, 7, n, 0, ids).tolist())   # nearly equal weights: every kept token shows
        assert seen == want, (top_p, top_k, sorted(seen), sorted(want))
    # a large vocabulary with the tie class at the last slice boundary
    V = V_WS
    sl = slice_of(V)
    tied = [7 * sl - 1, 7 * sl, 7 * sl + 1, 7 * sl + 2]
    row = torch.full((V,), -40.0)
    row[5] = 0.5
    row[tied] = 0.0
    row = row.to(torch.bfloat16)
    dev = row.view(1, V).expand(1024, V).contiguous().to(cuda_device)
    seen = set(draw(dev, V, 0.6, 0, 50.0, 3, 0, 0, torch.arange(1024, device=cuda_device)).tolist())
    want = set(Chain(row).kept(Chain(row).nucleus_sizes(0.6)[0]).tolist())
    assert seen == want == {5, tied[0], tied[1]}, (sorted(seen), sorted(want))


# ---- 3. agreement with the one-CTA kernel --------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [8, 128, 1000, 1024])
def test_agrees_with_the_one_cta_kernel(V, cuda_device):
    g = torch.Generator().manual_seed(100 + V)
    B = 256
    ldl = V + 8
    logits = make_logits(B, V, ldl, g, ties=V >= 128)
    dev = logits.to(cuda_device)
    row_id = torch.randperm(1 << 20, generator=g)[:B]
    rid = row_id.to(cuda_device)
    chains = [Chain(logits[b, :V]) for b in range(B)]
    ambiguous = compared = 0
    for top_p, top_k, temperature in ((0.8, 8, 1.2), (0.5, 0, 1.0), (0.95, 200, 0.7), (1.0, 0, 1.2), (0.9, 3, 0.0),
                                      (1.0, 5, 2.0), (0.3, 0, 0.9)):
        a = draw(dev, V, top_p, top_k, temperature, SEED, 5, 9, rid, cluster=False)
        b = draw(dev, V, top_p, top_k, temperature, SEED, 5, 9, rid, cluster=True)
        for r in range(B):
            u = O.philox_uniform(SEED, int(row_id[r]), 14)
            if chains[r].ambiguous(top_p, top_k, temperature, u):
                ambiguous += 1
                continue
            compared += 1
            assert int(a[r]) == int(b[r]), (V, r, top_p, top_k, temperature, int(a[r]), int(b[r]))
    print(f"V={V}: {compared} rows identical, {ambiguous} ambiguous rows skipped")
    assert compared > 0.9 * (compared + ambiguous)


# ---- 4. distribution, determinism, strides, replay, bounds ---------------------------------------------------------------
def test_distribution_chi_square_at_the_whitespace_vocabulary(cuda_device):
    V, top_p, top_k, temperature = V_WS, 0.95, 24, 1.2
    g = torch.Generator().manual_seed(4)
    row = torch.full((1, V), -8.0)
    hot = torch.randperm(V, generator=g)[:40]         # a peaked row: 40 likely tokens spread over every slice
    row[0, hot] = torch.randn(40, generator=g) * 1.2 + 4.0
    row = row.to(torch.bfloat16)
    chain = Chain(row[0])
    n = min(chain.nucleus_sizes(top_p)[0], top_k)
    assert len(chain.nucleus_sizes(top_p)) == 1 and n >= 8
    kept = set(chain.kept(n).tolist())
    q = np.zeros(V)
    k = chain.kept(n)
    q[k] = np.power(chain.p[k], 1.0 / temperature)
    q /= q.sum()
    B, rounds = 1024, 100
    dev = row.expand(B, V).contiguous().to(cuda_device)
    ids = torch.arange(B, device=cuda_device)
    counts = np.zeros(V)
    for r in range(rounds):
        counts += np.bincount(draw(dev, V, top_p, top_k, temperature, 99, 1000 + r, 3, ids).numpy(), minlength=V)
    assert set(np.nonzero(counts)[0].tolist()) <= kept
    exp = q * B * rounds
    keep = exp > 5
    chi2 = float((((counts - exp) ** 2)[keep] / exp[keep]).sum())
    dof = int(keep.sum()) - 1
    z = 3.72   # Wilson-Hilferty bound for p = 1e-4
    bound = dof * (1 - 2 / (9 * dof) + z * (2 / (9 * dof)) ** 0.5) ** 3
    assert chi2 < bound, (chi2, bound, dof)


def test_determinism_strides_streams_replay_and_bounds(cuda_device):
    from ai_music_generation_b200 import _C, ops
    V = 50257
    g = torch.Generator().manual_seed(5)
    rows = make_logits(64, V, V, g).to(cuda_device)
    a = draw(rows, V, 0.9, 0, 1.5, 42, 64, 3)
    assert torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 64, 3))
    assert torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 64, 3, torch.arange(64, device=cuda_device)))   # NULL = arange
    assert torch.equal(draw(rows, V, 0.9, 0, 1.5, 42, 60, 7), a)                                         # base + counter
    assert not torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 43, 64, 3))
    assert not torch.equal(a, draw(rows, V, 0.9, 0, 1.5, 42, 96, 3))
    perm = torch.randperm(64, generator=g)
    b = draw(rows[perm.to(cuda_device)], V, 0.9, 0, 1.5, 42, 64, 3, perm.to(cuda_device))   # a row's stream follows its id
    assert torch.equal(b, a[perm])
    # out_stride: column 1 of a [64, 3] buffer, the other columns untouched
    buf = torch.full((64, 3), -5, device=cuda_device, dtype=torch.int64)
    s, c = scalars(cuda_device, 42, 64)
    ops.sample_top_p_cluster(rows, V, buf[:, 1], 0.9, 0, 1.5, s, c, 3, out_stride=3)
    assert torch.equal(buf[:, 1].cpu(), a) and bool((buf[:, [0, 2]] == -5).all())
    # a recorded launch, replayed through Python and through the C replay program, reads the device seed and counter base
    out = torch.full((64,), -1, device=cuda_device, dtype=torch.int64)
    ops.begin_record()
    ops.sample_top_p_cluster(rows, V, out, 0.9, 0, 1.5, s, c, 3)
    plan = ops.end_record()
    s.fill_(7)
    c.fill_(100)
    ops.replay(plan)
    want = draw(rows, V, 0.9, 0, 1.5, 7, 100, 3)
    assert torch.equal(out.cpu(), want) and not torch.equal(want, a)
    prog = ops.compile_affine(plan, [[]])
    assert prog is not None and int(prog[0][0]) == _C.FN_IDS["abcgpt_sample_top_p_cluster"] == 9
    s.fill_(42)
    c.fill_(64)
    out.fill_(-1)
    ops.replay_compiled(prog, 0)
    assert torch.equal(out.cpu(), a)
    # bounds: -1 / AbcgptError before any launch
    big = torch.zeros(2, 786440, device=cuda_device, dtype=torch.bfloat16)
    out2 = torch.full((2,), -9, device=cuda_device, dtype=torch.int64)
    for bad in (786433, 7):
        with pytest.raises(_C.AbcgptError, match=str(bad)):
            ops.sample_top_p_cluster(big, bad, out2, 0.8, 8, 1.0, s, c, 0)
        torch.cuda.synchronize()
        assert bool((out2 == -9).all())
    ops.sample_top_p_cluster(big, 786432, out2, 0.8, 8, 1.0, s, c, 0)
    ops.sample_top_p_cluster(big, 8, out2, 0.8, 8, 1.0, s, c, 0)
    assert int(out2.max()) < 8 and int(out2.min()) >= 0


# ---- 5. GPT.generate(top_p=...) ------------------------------------------------------------------------------------------
def tiny_state(V, seed, block_size=64):
    cfgd = dict(block_size=block_size, vocab_size=V, n_layer=2, n_head=2, n_embd=128, dropout=0.0, bias=False)
    return cfgd, O.synthetic_state(O.OracleConfig(**cfgd), seed=seed)


def make_model(V, device, seed=1):
    from ai_music_generation_b200 import GPT, GPTConfig
    cfgd, sd = tiny_state(V, seed)
    model = GPT(GPTConfig(**cfgd))
    model.load_state_dict({**sd, "lm_head.weight": sd["transformer.wte.weight"]})
    return cfgd, sd, model.to(device).eval()


@pytest.mark.parametrize("V", [95, V_WS])
def test_generate_top_p_greedy_and_rows_independent_of_the_batch(V, cuda_device):
    from ai_music_generation_b200 import ops
    cfgd, sd, model = make_model(V, cuda_device)
    g = torch.Generator().manual_seed(V)
    B, T0, n_new, bs = 5, 4, 80, cfgd["block_size"]
    idx = torch.randint(V, (B, T0), generator=g).to(cuda_device)
    kw = dict(top_p=0.8, temperature=1.2, seed=77)
    # top_k = 1 under the nucleus head is greedy
    assert torch.equal(model.generate(idx, n_new, top_p=0.8, top_k=1), model.generate(idx, n_new, top_k=1))
    names = []
    orig = ops._call

    def spy(name, *a, **k):
        names.append(name)
        return orig(name, *a, **k)

    ops._call = spy
    try:
        full = model.generate(idx, n_new, top_k=8, row_ids=[10, 11, 12, 13, 14], **kw).cpu()
    finally:
        ops._call = orig
    kernel = "sample_top_p" if V <= 1024 else "sample_top_p_cluster"
    assert kernel in names and "sample_topk" not in names and "argmax" not in names
    assert torch.equal(full, model.generate(idx, n_new, top_k=8, row_ids=[10, 11, 12, 13, 14], **kw).cpu())
    # cached, then slid: alone, in a batch of 5 and at another batch position, with the same row ids
    perm = [3, 0, 4, 1, 2]
    moved = model.generate(idx[perm], n_new, top_k=8, row_ids=[10 + p for p in perm], **kw).cpu()
    assert torch.equal(moved, full[perm])
    for r in (0, 3):
        alone = model.generate(idx[r:r + 1], n_new, top_k=8, row_ids=[10 + r], **kw).cpu()
        assert torch.equal(alone[0], full[r]), ("cached + slid", r)
    # recompute only (use_cache=False): the whole run slides a window forward
    nc = model.generate(idx, n_new, top_k=8, row_ids=[10, 11, 12, 13, 14], use_cache=False, **kw).cpu()
    nc_alone = model.generate(idx[2:3], n_new, top_k=8, row_ids=[12], use_cache=False, **kw).cpu()
    assert torch.equal(nc_alone[0], nc[2])
    # ragged prompts: each row equals its prompt generated alone
    lens = [3, 7, 1, 12, 5]
    padded = torch.zeros(B, max(lens), dtype=torch.int64)
    prompts = [torch.randint(V, (1, n), generator=g) for n in lens]
    for r, p in enumerate(prompts):
        padded[r, :lens[r]] = p[0]
    rag = model.generate(padded.to(cuda_device), 40, top_k=8, prompt_lens=lens, row_ids=[20, 21, 22, 23, 24], **kw).cpu()
    for r in range(B):
        alone = model.generate(prompts[r].to(cuda_device), 40, top_k=8, row_ids=[20 + r], **kw).cpu()
        assert torch.equal(rag[r, :lens[r] + 40], alone[0]), ("ragged", r)
    # the slid part: every token in the chain's CDF interval under the recompute forward of its window
    for pos in range(bs, T0 + n_new - 1):
        cond = full[:, pos + 1 - bs:pos + 1].to(cuda_device)
        with torch.no_grad():
            logits, _ = model(cond)
        lg = logits[:, -1].cpu()
        for r in range(B):
            u = O.philox_uniform(77, 10 + r, pos + 1)
            ok = Chain(lg[r]).candidates(0.8, 8, 1.2, u)
            assert int(full[r, pos + 1]) in ok, (pos, r, int(full[r, pos + 1]), sorted(ok))
    # errors before any launch
    for bad in (0.0, 1.5, -0.1):
        with pytest.raises(ValueError):
            model.generate(idx, 4, top_p=bad)
    with pytest.raises(ValueError):
        model.generate(idx, 4, top_p=0.8, row_ids=[0, 1])
    with pytest.raises(ValueError):
        model.generate(idx, 4, row_ids=[0, 1, 2, 3, 4])


def test_generate_rejects_vocabularies_above_the_cluster_bound(cuda_device):
    from ai_music_generation_b200 import GPT, GPTConfig
    model = GPT(GPTConfig(block_size=8, vocab_size=786433, n_layer=1, n_head=2, n_embd=64, dropout=0.0, bias=False))
    with pytest.raises(ValueError, match="786432"):
        model.generate(torch.zeros(1, 1, dtype=torch.int64), 2, top_p=0.8)


# ---- 6. sample.py --top_p ------------------------------------------------------------------------------------------------
def write_checkpoint(tmp_path, out_dir, dataset, V, itos):
    cfgd, sd = tiny_state(V, seed=2)
    d = tmp_path / "data" / dataset
    d.mkdir(parents=True, exist_ok=True)
    with open(d / "meta.pkl", "wb") as f:
        pickle.dump({"vocab_size": V, "itos": itos, "stoi": {s: i for i, s in itos.items()}}, f)
    os.makedirs(tmp_path / out_dir, exist_ok=True)
    torch.save({"model_args": cfgd, "model": {**sd, "lm_head.weight": sd["transformer.wte.weight"]},
                "config": {"dataset": dataset}}, tmp_path / out_dir / "ckpt.pt")


def run_sample(tmp_path, out_dir, args):
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "sample.py"), f"--out_dir={out_dir}", *args], cwd=tmp_path, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    d = tmp_path / out_dir / "samples"
    return {name: open(d / name, encoding="utf-8").read() for name in sorted(os.listdir(d))}


# Prompt lengths: with batch 5 the first batch is decoded ragged (longest prompt + 50 fits the window), the second falls
# back to equal-length groups whose window slides; with batch 1 every prompt is decoded alone.
PROMPT_LENS = [9, 3, 21, 5, 5, 21, 26, 7, 26, 31]


def test_sample_py_files_do_not_depend_on_the_batch(tmp_path, cuda_device):
    rng = np.random.default_rng(0)
    # char codec, V = 95: the printable ASCII characters; validation tunes are the whole prompt
    itos = {i: chr(32 + i) for i in range(95)}
    letters = "ABCDEFGabcdefg,'2/"
    tunes = [{"id": f"t{i}", "abc notation": "".join(rng.choice(list(letters), n - 1))} for i, n in enumerate(PROMPT_LENS)]
    (tmp_path / "val.json").write_text(json.dumps(tunes))
    common = ["--dataset=irishman", "--tokens_format=char", f"--validation_path={tmp_path / 'val.json'}",
              "--n_conditional_measures=1000", "--max_new_tokens=50"]
    nucleus = ["--top_p=0.8", "--top_k=8", "--temperature=1.2"]
    write_checkpoint(tmp_path, "out-a", "irishman", 95, itos)
    write_checkpoint(tmp_path, "out-b", "irishman", 95, itos)
    one = run_sample(tmp_path, "out-a", [*common, *nucleus, "--batch=1"])
    five = run_sample(tmp_path, "out-b", [*common, *nucleus, "--batch=5"])
    assert len(one) == len(PROMPT_LENS) and one == five
    default = run_sample(tmp_path, "out-a", [*common, "--batch=5"])
    assert default == run_sample(tmp_path, "out-b", [*common, "--batch=5", "--top_p=0.0"])
    assert default != five
    # whitespace codec above 1024 tokens (the cluster kernel): validation files of bars, tokens t2 .. t{V-1}
    V = 5000
    itos = {i: f"t{i}" for i in range(V)}
    itos[0], itos[1] = "$", "|"
    val = tmp_path / "val_ws"
    val.mkdir()
    for i, n in enumerate(PROMPT_LENS):
        toks = [f"t{t}" for t in rng.integers(2, V, size=n - 1)]
        (val / f"p{i:02d}.txt").write_text(" ".join(toks[:n // 2]) + " | " + " ".join(toks[n // 2:]))
    common = ["--dataset=ws", "--tokens_format=midi", f"--validation_path={val}", "--n_conditional_measures=1000",
              "--max_new_tokens=50"]
    write_checkpoint(tmp_path, "out-c", "ws", V, itos)
    write_checkpoint(tmp_path, "out-d", "ws", V, itos)
    one = run_sample(tmp_path, "out-c", [*common, *nucleus, "--batch=1"])
    five = run_sample(tmp_path, "out-d", [*common, *nucleus, "--batch=5"])
    assert len(one) == len(PROMPT_LENS) and one == five
