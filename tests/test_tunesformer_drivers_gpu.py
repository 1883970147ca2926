"""TunesFormer drivers on the GPU: train_tunesformer.py end to end (logs, reference-layout weights, resume) and
generate_tunesformer.py against generate_tunes; tunes-weighted evaluation; patch sampling against the oracle; generation that
does not depend on which other tunes share the batch (tune_ids); a 2-rank torchrun run where two GPUs are present."""
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import nanogpt_oracle as O
from test_tunesformer_packed_gpu import _model, _states, _tunes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TUNE = ("X:1\nL:1/8\nM:6/8\nK:D\n|: A2B c2d | e3 f3 | g2f e2d | c3 A3 :|\n"
        "|: d2e f2g | a3 g3 | f2e d2c | d3 D3 :|\n")
TINY = ["--patch_num_layers=2", "--char_num_layers=2", "--n_embd=128", "--n_head=2", "--patch_block_size=16",
        "--batch_size=8", "--learning_rate=0.002", "--warmup_steps=2", "--seed=3"]


def _corpus(tmp_path):
    train, evl = tmp_path / "train.json", tmp_path / "eval.json"
    train.write_text(json.dumps([{"id": f"t{i}", "abc notation": TUNE} for i in range(64)]))
    evl.write_text(json.dumps([{"id": f"e{i}", "abc notation": TUNE} for i in range(12)]))
    return str(train), str(evl)


def _run(args, nproc=0, env=None):
    cmd = ([sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={nproc}"] if nproc
           else [sys.executable])
    r = subprocess.run(cmd + args, cwd=ROOT, capture_output=True, text=True, timeout=900,
                       env=None if env is None else {**os.environ, **env})
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def _samples(out):
    d = os.path.join(out, "samples")
    files = {}
    for name in sorted(os.listdir(d)):
        with open(os.path.join(d, name), encoding="utf-8") as f:
            files[name] = f.read()
    return files


def _logs(out):
    with open(os.path.join(out, "logs.jsonl")) as f:
        return [json.loads(line) for line in f]


def _settings(**kw):
    import train_tunesformer as T
    return {**T.DEFAULTS, **kw}


def test_train_resume_and_generate_end_to_end(tmp_path, cuda_device):
    import generate_tunesformer as G
    import train_tunesformer as T
    train, evl = _corpus(tmp_path)
    out = str(tmp_path / "run")
    data = [f"--train_data={train}", f"--eval_data={evl}", f"--out_dir={out}"]
    _run(["train_tunesformer.py", *TINY, *data, "--num_epochs=4"])
    logs = _logs(out)
    spe = 64 // 8
    assert [r["epoch"] for r in logs] == [1, 2, 3, 4]
    assert set(logs[0]) >= {"epoch", "train_loss", "eval_loss", "lr", "ms_per_step", "chars_per_s"}
    ev = [r["eval_loss"] for r in logs]
    assert ev[-1] < 0.75 * ev[0], ev              # a memorisable corpus: the eval loss falls by at least a quarter
    for r in logs:
        assert r["lr"] == T.cosine_lr(r["epoch"] * spe - 1, 0.002, 2, 4 * spe)
    ckpt = torch.load(os.path.join(out, "weights.pth"), map_location="cpu")
    best = int(np.argmin(ev)) + 1
    assert ckpt["epoch"] == ckpt["best_epoch"] == best and ckpt["min_eval_loss"] == min(ev)

    # the checkpoint restores parameters and AdamW moments bitwise, through load_reference_state_dict
    s = _settings(learning_rate=0.002)
    model, opt, ck, _ = T.restore(out, s, cuda_device)
    got = model.reference_state_dict()
    assert got.keys() == ckpt["model"].keys()
    for k, v in ckpt["model"].items():
        assert torch.equal(got[k], v), k
    for mine, saved in zip(opt.state_dict(), ckpt["optimizer"]):
        assert len(mine["state"]) == len(saved["state"]) > 0
        for i, st in saved["state"].items():
            for key in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(mine["state"][i][key].cpu(), st[key]), (i, key)
            assert float(mine["state"][i]["step"]) == float(st["step"]) == best * spe

    # resume: continues at the epoch after the saved one, with the lr of an uninterrupted run of the same length
    resumed = str(tmp_path / "resumed")
    shutil.copytree(out, resumed)
    _run(["train_tunesformer.py", *TINY, *data[:2], f"--out_dir={resumed}", "--num_epochs=6", "--init_from=resume"])
    relogs = _logs(resumed)
    assert [r["epoch"] for r in relogs] == list(range(1, 7))   # records after the saved epoch were superseded
    assert relogs[:best] == logs[:best]
    for r in relogs[best:]:
        assert r["step"] == r["epoch"] * spe
        assert r["lr"] == T.cosine_lr(r["epoch"] * spe - 1, 0.002, 2, 6 * spe)

    # generation: one file per prompt, each equal to generate_tunes on the same prompts and settings
    _run(["generate_tunesformer.py", f"--out_dir={out}", f"--validation_path={evl}", "--n_conditional_bars=2",
          "--max_patch=12", "--seed=5"])
    prompts = G.conditional_prompts(evl, 2)
    assert len(prompts) == 12 and prompts[0][1] == "X:1\nL:1/8\nM:6/8\nK:D\n|: A2B c2d | e3 f3 |"
    gm = G.load_model(os.path.join(out, "weights.pth"), 2, cuda_device)
    want = gm.generate_tunes([p for _, p in prompts], max_patch=12, top_p=0.8, top_k=8, temperature=1.2, seed=5)
    files = sorted(os.listdir(os.path.join(out, "samples")))
    assert files == sorted(f"tunesformer_{k}.abc" for k, _ in prompts)
    for (key, _), text in zip(prompts, want):
        with open(os.path.join(out, "samples", f"tunesformer_{key}.abc"), encoding="utf-8") as f:
            assert f.read() == text, key

    # the same run as two ranks of a sharded launch (one after the other on this GPU): each takes a contiguous slice of
    # the prompts with their global ids, and together they write the same files
    sharded = str(tmp_path / "sharded")
    for rank in (0, 1):
        _run(["generate_tunesformer.py", f"--weights={os.path.join(out, 'weights.pth')}", f"--out_dir={sharded}",
              f"--validation_path={evl}", "--n_conditional_bars=2", "--max_patch=12", "--seed=5"],
             env={"RANK": str(rank), "WORLD_SIZE": "2", "LOCAL_RANK": "0"})
    assert _samples(sharded) == _samples(out)


def test_dropout_stops_the_driver(tmp_path):
    train, evl = _corpus(tmp_path)
    r = subprocess.run([sys.executable, "train_tunesformer.py", *TINY, f"--train_data={train}", f"--eval_data={evl}",
                        f"--out_dir={tmp_path / 'drop'}", "--num_epochs=1", "--dropout=0.1"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "packed training does not support dropout" in r.stderr
    assert not os.path.exists(tmp_path / "drop" / "logs.jsonl")


def test_estimate_tunes_loss_is_the_mean_over_tunes(cuda_device):
    from ai_music_generation_b200 import evalloop, pack_tunes
    _, _, psd, csd = _states()
    model = _model(psd, csd, cuda_device)
    tunes = _tunes([2, 5, 12, 16, 3, 7, 9], seed=4)
    with torch.no_grad():
        alone = [model(t.to(cuda_device), [t.shape[0]]).item() for t in tunes]
    batches = [pack_tunes(tunes[0:3]), pack_tunes(tunes[3:6]), pack_tunes(tunes[6:7]), (None, [])]
    got = evalloop.estimate_tunes_loss(model, [(p if p is None else p.to(cuda_device), c) for p, c in batches], cuda_device)
    want = sum(alone) / len(alone)
    # fp32 sums of a few thousand terms per tune: N * eps ~ 1e-4 bounds the reordering
    assert abs(got - want) <= 1e-4 * abs(want), (got, want)
    assert model.training


def _oracle_sampled_loss(pc, cc, psd, csd, tunes, src, tune_of):
    """Mean over tunes of the bf16-emulated character loss over each tune's selected rows, from the oracle's pieces."""
    total, r0 = 0.0, 0
    for i, t in enumerate(tunes):
        P = t.shape[0]
        sel = torch.from_numpy(src[tune_of == i] - r0)
        r0 += P
        oh = torch.nn.functional.one_hot(t[None], 128).float().reshape(1, P, -1)
        emb = O._bf(oh) @ O._bf(psd["patch_embedding.weight"]).t() + psd["patch_embedding.bias"]
        _, _, hidden = O.forward(psd, pc, None, None, bf16=True, return_hidden=True, inputs_embeds=emb)
        first, chars = hidden[0, sel], t[sel + 1]
        y = torch.full_like(chars, -1)
        y[:, :-1] = chars[:, 1:]
        y[y == 0] = -1
        _, loss = O.forward(csd, cc, chars, y, bf16=True, first_embeds=first)
        total += loss.item() / len(tunes)
    return total


def test_patch_sampling(cuda_device):
    from ai_music_generation_b200 import pack_tunes
    from ai_music_generation_b200.tunesformer import sampled_decode_rows
    pc, cc, psd, csd = _states()
    model = _model(psd, csd, cuda_device)
    opt = model.configure_optimizers(0.1, 1e-3, (0.9, 0.95))
    tunes = _tunes([2, 5, 12, 16, 9], seed=6)
    patches, counts = pack_tunes(tunes)
    patches = patches.to(cuda_device)
    with torch.no_grad():
        base = model(patches, counts)
        same = model(patches, counts, patch_sampling=15, generator=torch.Generator().manual_seed(1))
    assert torch.equal(base, same)
    gen = lambda: torch.Generator().manual_seed(11)   # noqa: E731
    loss = model(patches, counts, patch_sampling=2, generator=gen())
    src, tune_of = sampled_decode_rows(counts, 2, gen())
    assert len(src) == 1 + 2 * 4
    torch.set_num_threads(8)
    want = _oracle_sampled_loss(pc, cc, psd, csd, tunes, src, tune_of)
    assert abs(loss.item() - want) <= 2e-3, (loss.item(), want)
    opt.zero_grad(set_to_none=True)
    loss.backward()
    model.clip_grad_norm_(1.0)
    opt.step()
    with torch.no_grad():
        loss2 = model(patches, counts, patch_sampling=2, generator=gen())
    assert loss2.item() < loss.item()


def test_generation_does_not_depend_on_the_batch(cuda_device):
    """Every row of a decode step computes the same bits whatever the batch size: tunes c and d drawn in a batch of four
    equal the same tunes drawn alone as a pair with their global ids."""
    _, _, psd, csd = _states()
    model = _model(psd, csd, cuda_device).eval()
    prompts = ["", "X:1\nK:D\n", "X:2\nL:1/8\nK:G\n|: GAB", "K:C\nC2E G2c |"]
    kw = dict(max_patch=14, top_p=0.8, top_k=8, temperature=1.2, seed=21)
    four = model.generate_tunes(prompts, **kw)
    pair = model.generate_tunes(prompts[2:], tune_ids=[2, 3], **kw)
    assert pair == four[2:]
    assert model.generate_tunes(prompts[2:], **kw) != pair      # the id, not the position in the call, keys the stream


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs (torchrun --nproc_per_node=2)")
def test_two_rank_run_matches_single_process_eval(tmp_path):
    from ai_music_generation_b200 import evalloop, pack_tunes
    from ai_music_generation_b200.tunesdata import load_abc_corpus
    import train_tunesformer as T
    train, evl = _corpus(tmp_path)
    out = str(tmp_path / "ddp")
    _run(["train_tunesformer.py", *TINY, f"--train_data={train}", f"--eval_data={evl}", f"--out_dir={out}", "--num_epochs=2"],
         nproc=2)
    logs = _logs(out)
    assert [r["epoch"] for r in logs] == [1, 2]
    dev = torch.device("cuda:0")
    model, _, ckpt, _ = T.restore(out, _settings(), dev)
    _, tunes = load_abc_corpus(evl, patch_length=16)
    batches = [pack_tunes(tunes[i:i + 8]) for i in range(0, len(tunes), 8)]
    ev = evalloop.estimate_tunes_loss(model, [(p.to(dev), c) for p, c in batches], dev)
    logged = logs[ckpt["epoch"] - 1]["eval_loss"]
    assert abs(ev - logged) <= 1e-4 * abs(logged), (ev, logged)
    # generation on two GPUs writes the files one process writes
    gen = ["generate_tunesformer.py", f"--validation_path={evl}", "--n_conditional_bars=2", "--max_patch=12", "--seed=5",
           f"--weights={os.path.join(out, 'weights.pth')}"]
    _run(gen + [f"--out_dir={tmp_path / 'one'}"])
    _run(gen + [f"--out_dir={tmp_path / 'two'}"], nproc=2)
    assert _samples(str(tmp_path / "two")) == _samples(str(tmp_path / "one"))
    assert len(_samples(str(tmp_path / "one"))) == 12
