"""Host side of the TunesFormer drivers: corpus loading, the per-rank tune sampler, patch-row sampling, the reference-layout
checkpoint export and the learning-rate schedule of train_tunesformer.py."""
import json

import numpy as np
import pytest
import torch

from ai_music_generation_b200 import Patchilizer
from ai_music_generation_b200.tunesdata import TuneBatches, load_abc_corpus
from ai_music_generation_b200.tunesformer import packed_decode_rows, sampled_decode_rows
from oracle.make_golden_tunesformer import SPEC, inputs, to_hf

TUNES = [
    ("a1", "X:1\nL:1/8\nM:6/8\nK:D\n|: A2B c2d | e3 f3 :|\n"),
    ("empty", ""),
    ("b2", "X:2\nK:G\nGAB cde | d2c BAG | A4 z2 |]\n"),
    ("blank", "  \n \n"),
    ("c3", "K:C\n" + "C2E G2c | " * 80 + "\n"),   # longer than a 16-patch block
]


def test_load_abc_corpus_matches_encode_and_drops_empty_tunes(tmp_path, capsys):
    path = tmp_path / "corpus.json"
    path.write_text(json.dumps([{"id": k, "abc notation": t} for k, t in TUNES] + [{"abc notation": TUNES[0][1]}]))
    pz = Patchilizer()
    for block in (128, 16):
        keys, tunes = load_abc_corpus(str(path), patch_length=block)
        assert keys == ["a1", "b2", "c3", 5]      # a record without "id" is keyed by its index
        for key, tune in zip(keys, tunes):
            assert tune == pz.encode(dict(TUNES).get(key, TUNES[0][1]), patch_length=block, add_special_patches=True)
        assert "dropped 2 of 6" in capsys.readouterr().out
    assert len(tunes[2]) == 16


@pytest.mark.parametrize("world", [2, 3])
def test_training_batches_equal_disjoint_and_seeded(world):
    n, bs = 50, 4 * world
    ranks = [TuneBatches(n, bs, r, world, seed=7, drop_last=True) for r in range(world)]
    assert len({len(b) for b in ranks}) == 1 and len(ranks[0]) == n // bs
    epochs = {}
    for e in (1, 2):
        shards = [b.epoch(e) for b in ranks]
        seen = np.concatenate([s for rank in shards for s in rank])
        assert len(set(seen.tolist())) == len(seen) == (n // bs) * bs      # disjoint within the epoch
        for step in zip(*shards):                                          # equal shards in every step
            assert {len(s) for s in step} == {bs // world}
        epochs[e] = [np.concatenate(step).tolist() for step in zip(*shards)]
        again = [TuneBatches(n, bs, r, world, seed=7, drop_last=True).epoch(e) for r in range(world)]
        assert all(np.array_equal(a, b) for x, y in zip(shards, again) for a, b in zip(x, y))
    assert epochs[1] != epochs[2]


@pytest.mark.parametrize("n,bs,world", [(50, 8, 2), (50, 9, 3), (7, 6, 3), (2, 6, 3)])
def test_evaluation_batches_visit_every_tune_once(n, bs, world):
    seen = [i for r in range(world) for s in TuneBatches(n, bs, r, world, seed=1, drop_last=False).epoch(0) for i in s.tolist()]
    assert sorted(seen) == list(range(n))


def test_batch_size_must_divide_by_world():
    with pytest.raises(ValueError):
        TuneBatches(10, 5, 0, 2)
    with pytest.raises(ValueError):
        TuneBatches(10, 4, 2, 3, drop_last=False)


def test_sampled_decode_rows():
    counts = [2, 5, 12, 16, 3]
    src0, tune0 = packed_decode_rows(counts)
    for k in (0, 15, 40):
        src, tune = sampled_decode_rows(counts, k, torch.Generator().manual_seed(0))
        assert np.array_equal(src, src0) and np.array_equal(tune, tune0)
    for k in (1, 2, 4):
        src, tune = sampled_decode_rows(counts, k, torch.Generator().manual_seed(3))
        again = sampled_decode_rows(counts, k, torch.Generator().manual_seed(3))
        assert np.array_equal(src, again[0]) and np.array_equal(tune, again[1])
        assert src.dtype == np.int64 and tune.dtype == np.int32
        for i, c in enumerate(counts):
            rows = src[tune == i]
            full = src0[tune0 == i]
            assert len(rows) == min(k, c - 1)
            assert np.all(np.diff(rows) > 0) and set(rows.tolist()) <= set(full.tolist())
    picks = {tuple(sampled_decode_rows(counts, 2, torch.Generator().manual_seed(s))[0].tolist()) for s in range(8)}
    assert len(picks) > 1


# ---- reference-layout export ------------------------------------------------------------------------------------------
def _model():
    from ai_music_generation_b200 import GPTConfig, TunesFormerShaped
    _, _, psd, csd, _ = inputs(SPEC)
    model = TunesFormerShaped(GPTConfig(**SPEC["patch_cfg"]), GPTConfig(**SPEC["char_cfg"]))
    model.patch_level_decoder.load_state_dict({**psd, "lm_head.weight": psd["transformer.wte.weight"]})
    model.char_level_decoder.load_state_dict({**csd, "lm_head.weight": csd["transformer.wte.weight"]})
    return model, psd, csd


def _hf_modules():
    from transformers import GPT2Config, GPT2LMHeadModel, GPT2Model
    pc, cc = SPEC["patch_cfg"], SPEC["char_cfg"]

    def cfg(c):
        return GPT2Config(num_hidden_layers=c["n_layer"], n_positions=c["block_size"], vocab_size=c["vocab_size"],
                          n_embd=c["n_embd"], n_head=c["n_head"], resid_pdrop=0.0, embd_pdrop=0.0, attn_pdrop=0.0)

    patch, char, top = torch.nn.Module(), torch.nn.Module(), torch.nn.Module()
    patch.patch_embedding = torch.nn.Linear(32 * 128, pc["n_embd"])
    patch.base = GPT2Model(cfg(pc))
    char.base = GPT2LMHeadModel(cfg(cc))
    top.patch_level_decoder, top.char_level_decoder = patch, char
    return top


def test_reference_state_dict_loads_strict_into_hf_and_matches_to_hf():
    model, psd, csd = _model()
    sd = model.reference_state_dict()
    want = to_hf(psd, "patch_level_decoder.base.")
    want["patch_level_decoder.patch_embedding.weight"] = psd["patch_embedding.weight"]
    want["patch_level_decoder.patch_embedding.bias"] = psd["patch_embedding.bias"]
    want.update(to_hf(csd, "char_level_decoder.base.transformer."))
    want["char_level_decoder.base.lm_head.weight"] = csd["transformer.wte.weight"]
    assert sd.keys() == want.keys()
    for k, v in want.items():
        assert torch.equal(sd[k], v.float()), k
    hf = _hf_modules()
    hf.load_state_dict(sd, strict=True)
    assert torch.equal(hf.char_level_decoder.base.lm_head.weight, sd["char_level_decoder.base.transformer.wte.weight"])


def test_reference_state_dict_round_trip_is_bitwise():
    from ai_music_generation_b200 import GPTConfig, TunesFormerShaped
    model, _, _ = _model()
    torch.manual_seed(99)
    fresh = TunesFormerShaped(GPTConfig(**SPEC["patch_cfg"]), GPTConfig(**SPEC["char_cfg"]))
    fresh.load_reference_state_dict(model.reference_state_dict())
    want, got = dict(model.named_parameters()), dict(fresh.named_parameters())
    assert want.keys() == got.keys()
    for k, w in want.items():
        assert torch.equal(got[k].detach(), w.detach()), k


def test_schedule_matches_transformers():
    from transformers import get_cosine_schedule_with_warmup
    import train_tunesformer as T
    base, warmup, total = 5e-5, 7, 50
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.AdamW([p], lr=base)
    sched = get_cosine_schedule_with_warmup(opt, warmup, total)
    for step in range(total + 3):
        assert T.cosine_lr(step, base, warmup, total) == pytest.approx(opt.param_groups[0]["lr"], rel=1e-12, abs=1e-18), step
        opt.step()
        sched.step()
