"""Head sizes 32 and 128 (csrc/attn_hd.cu) on the GPU: kernel parity against fp32 PyTorch, model parity against the
bf16-emulating oracle (the criteria of test_model_gpu.py / test_dropout_gpu.py), dropout with host-regenerated masks over two
consecutive plan-replayed steps, and generate() (greedy vs the oracle, KV cache vs recompute with a sliding window, ragged
prompts, top-k sampling)."""
import pytest
import torch

from oracle import nanogpt_oracle as O
from tools import gpu_probe

pytestmark = pytest.mark.gpu

HEAD_CASES = [f"attn_d{D}_{s}" for D in (32, 128) for s in ("t1", "t32", "t100", "t128", "t200", "t256", "t1024", "spike")]

# D = 32: 4 heads of 32; D = 128: 2 heads of 128
CFGS = {32: dict(n_layer=2, n_head=4, n_embd=128), 128: dict(n_layer=2, n_head=2, n_embd=256)}


def cfg_dict(D, bias=True, block_size=256, dropout=0.0):
    return dict(block_size=block_size, vocab_size=95, dropout=dropout, bias=bias, **CFGS[D])


def make(cfgd, device, sd=None):
    from ai_music_generation_b200 import GPT, GPTConfig
    cfg = O.OracleConfig(**cfgd)
    sd = O.synthetic_state(cfg, seed=1) if sd is None else sd
    model = GPT(GPTConfig(**cfgd))
    model.load_state_dict({**sd, "lm_head.weight": sd["transformer.wte.weight"]})
    return cfg, sd, model.to(device)


@pytest.mark.parametrize("name", HEAD_CASES)
def test_head_size_kernel_case(name, cuda_device):
    res = gpu_probe.build_cases()[name]()
    assert res["ok"], res


def _compare(model, loss, logits, sd, cfg, x, y, masks=None, loss_tol=2e-3):
    torch.set_num_threads(8)
    ref_loss, ref_logits, ref_grads = O.loss_and_grads(sd, cfg, x, y, bf16=True, masks=masks)
    tru_loss, tru_logits, tru_grads = O.loss_and_grads(sd, cfg, x, y, bf16=False, masks=masks)
    assert abs(loss.item() - ref_loss.item()) <= loss_tol, (loss.item(), ref_loss.item(), tru_loss.item())
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


@pytest.mark.parametrize("D", [32, 128])
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("T", [256, 200])
def test_forward_backward_match_bf16_oracle(D, bias, T, cuda_device):
    cfg, sd, model = make(cfg_dict(D, bias), cuda_device)
    model.train()
    # 8 sequences: with 2 the first layer's ln_1 gradient at D = 128 sat at 2x the emulated reference's own bf16 error (the
    # kernels' dq / dk / dv errors equal those of the head-size-64 kernels, tools/gpu_probe.py attn_d*_t200); more tokens average it
    x, y = O.synthetic_tokens(cfg, 8, T, seed=0)
    logits, loss = model(x.to(cuda_device), y.to(cuda_device))
    loss.backward()
    _compare(model, loss, logits, sd, cfg, x, y)


@pytest.mark.parametrize("D", [32, 128])
def test_three_adamw_steps_track_oracle(D, cuda_device):
    cfgd = cfg_dict(D, True, block_size=128)
    cfg, sd, model = make(cfgd, cuda_device)
    model.train()
    batches = [O.synthetic_tokens(cfg, 4, 128, seed=s) for s in range(3)]
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


def host_masks(cfg, B, T, p, seed):
    from ai_music_generation_b200 import dropout as Dm
    t = torch.from_numpy
    m = {"p": p, "emb": t(Dm.keep_mask(Dm.site_key(seed, 0), B * T, cfg.n_embd, p)).view(B, T, cfg.n_embd),
         "attn_p": [], "attn_resid": [], "mlp_resid": []}
    for l in range(cfg.n_layer):
        m["attn_p"].append(t(Dm.attention_keep_mask(Dm.site_key(seed, 1 + 3 * l), B, cfg.n_head, T, p)))
        m["attn_resid"].append(t(Dm.keep_mask(Dm.site_key(seed, 2 + 3 * l), B * T, cfg.n_embd, p)).view(B, T, cfg.n_embd))
        m["mlp_resid"].append(t(Dm.keep_mask(Dm.site_key(seed, 3 + 3 * l), B * T, cfg.n_embd, p)).view(B, T, cfg.n_embd))
    return m


@pytest.mark.parametrize("D", [32, 128])
def test_dropout_two_consecutive_steps_match_their_masks(D, cuda_device):
    """Step 1 records the launch plans, step 2 replays them with its own keys patched into the attention launches: each step
    must match the oracle run with the masks of its own seed."""
    p, B, T = 0.2, 2, 200
    cfg, sd, model = make(cfg_dict(D, True, dropout=p), cuda_device)
    model.train()
    x, y = O.synthetic_tokens(cfg, B, T, seed=0)
    for seed in (4242, 777):
        model.zero_grad(set_to_none=True)
        model._next_dropout_seed = seed
        logits, loss = model(x.to(cuda_device), y.to(cuda_device))
        assert model.last_dropout_seed == seed
        loss.backward()
        _compare(model, loss, logits, sd, cfg, x, y, masks=host_masks(cfg, B, T, p, seed), loss_tol=3e-3)
    nodrop_loss, _, _ = O.loss_and_grads(sd, cfg, x, y, bf16=True)
    assert abs(nodrop_loss.item() - loss.item()) > 1e-3


@pytest.mark.parametrize("D", [32, 128])
def test_greedy_generation_matches_oracle(D, cuda_device):
    cfg, sd, model = make(cfg_dict(D, True, block_size=64), cuda_device)
    model.eval()
    prompt, _ = O.synthetic_tokens(cfg, 3, 5, seed=7)
    n_new = 30
    out = model.generate(prompt.to(cuda_device), n_new, temperature=1.0, top_k=1).cpu()
    ref, margins = O.generate_greedy(sd, cfg, prompt, n_new, return_margins=True)
    assert out.shape == ref.shape and torch.equal(out[:, :5], prompt)
    for b in range(out.shape[0]):
        diff = (out[b] != ref[b]).nonzero()
        if len(diff):   # only where the reference's own top-2 margin is inside the bf16 logit tolerance
            pos = diff[0].item() - prompt.shape[1]
            assert margins[b, pos].item() <= 6e-2, (b, pos, margins[b, pos].item())


@pytest.mark.parametrize("D", [32, 128])
def test_kv_cache_equals_recompute_with_sliding_window(D, cuda_device):
    cfg, sd, model = make(cfg_dict(D, True, block_size=64), cuda_device)
    model.eval()
    prompt, _ = O.synthetic_tokens(cfg, 3, 6, seed=11)
    n_new = 80                                        # 6 + 80 > 64: the window slides
    a = model.generate(prompt.to(cuda_device), n_new, top_k=1, use_cache=True).cpu()
    b = model.generate(prompt.to(cuda_device), n_new, top_k=1, use_cache=False).cpu()
    ref, margins = O.generate_greedy(sd, cfg, prompt, n_new, return_margins=True)
    for got in (a, b):
        for row in range(got.shape[0]):
            diff = (got[row] != ref[row]).nonzero()
            if len(diff):
                pos = diff[0].item() - prompt.shape[1]
                assert margins[row, pos].item() <= 6e-2, (row, pos, margins[row, pos].item())
    # every token the cached path picked is the argmax of the recompute path's logits for the same context, up to the bf16
    # logit tolerance (a near-tie may go either way, after which the two runs continue from different contexts)
    bs, P0 = cfg.block_size, prompt.shape[1]
    for pos in range(P0 - 1, a.shape[1] - 1):
        logits, _ = model(a[:, max(0, pos + 1 - bs):pos + 1].to(cuda_device))
        lg = logits[:, -1].float().cpu()
        picked = lg.gather(1, a[:, pos + 1:pos + 2]).squeeze(1)
        assert bool((picked >= lg.max(dim=1).values - 6e-2).all()), (pos, picked, lg.max(dim=1).values)
    # the decode loop reached the one-call compiled replay (abcgpt_attn_decode_hd has a replay id)
    st = model._bufs[("decode", 3, 64)]
    assert st.affine and all(v[3] is not None for v in st.affine.values())


@pytest.mark.parametrize("D", [32, 128])
def test_ragged_prompts_equal_one_at_a_time(D, cuda_device):
    cfg, sd, model = make(cfg_dict(D, True, block_size=64), cuda_device)
    model.eval()
    torch.manual_seed(3)
    lens = [3, 9, 1, 14]
    n_new = 30
    padded = torch.zeros(len(lens), max(lens), dtype=torch.long)
    prompts = []
    for r, n in enumerate(lens):
        prompts.append(torch.randint(1, cfg.vocab_size, (1, n)))
        padded[r, :n] = prompts[-1][0]
    out = model.generate(padded.to(cuda_device), n_new, top_k=1, prompt_lens=lens).cpu()
    for r, n in enumerate(lens):
        alone = model.generate(prompts[r].to(cuda_device), n_new, top_k=1).cpu()[0]
        assert torch.equal(out[r, :n + n_new], alone), (r, n)


@pytest.mark.parametrize("D", [32, 128])
def test_top_k_sampling_reproducible_and_in_vocabulary(D, cuda_device):
    cfg, sd, model = make(cfg_dict(D, True, block_size=64), cuda_device)
    model.eval()
    prompt, _ = O.synthetic_tokens(cfg, 4, 6, seed=5)
    torch.manual_seed(0)
    a = model.generate(prompt.to(cuda_device), 40, temperature=0.8, top_k=5).cpu()
    torch.manual_seed(0)
    b = model.generate(prompt.to(cuda_device), 40, temperature=0.8, top_k=5).cpu()
    assert torch.equal(a, b)
    assert a.shape == (4, 46) and int(a.max()) < cfg.vocab_size and int(a.min()) >= 0


def test_unsupported_head_size_is_an_error_at_the_abi(cuda_device):
    from ai_music_generation_b200 import _C, ops
    qkv = torch.zeros(64, 3 * 96, device=cuda_device, dtype=torch.bfloat16)
    out = torch.zeros(64, 96, device=cuda_device, dtype=torch.bfloat16)
    lse = torch.zeros(1, 1, 64, device=cuda_device)
    with pytest.raises(_C.AbcgptError, match="32, 64, 128"):
        ops.attn_fwd(qkv, out, lse, 1, 64, 1, head_size=96)
    with pytest.raises(_C.AbcgptError, match="abcgpt_attn_decode"):
        ops.attn_decode_hd(qkv[:1], out, out[:1], 1, 64, 0, 1, 64)
