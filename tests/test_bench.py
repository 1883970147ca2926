"""bench.py's command line: `--steps` sets the number of timed steps in every arm, and `--dump-outputs DIR` writes what the
last timed training step returned (on the GPU: file set, dtypes, sizes, and that the files belong to one and the same step)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, cwd):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900,
                       cwd=cwd)
    return r, (json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else None)


def test_argument_checks(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r, _ = _bench(*args, cwd=tmp_path)
        assert r.returncode == 2 and "error:" in r.stderr, (args, r.stderr[-500:])
    assert not (tmp_path / "d").exists()


def test_reference_arm_times_the_requested_steps(tmp_path):
    r, out = _bench("--impl", "reference", "--workload", "cfg2", "--steps", "6", "--warmup", "1", cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    assert out["steps"] == 6 and out["cpu_baseline"]["sample"].startswith("6 timed")


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path, cuda_device):
    import bench
    from ai_music_generation_b200 import GPT, GPTConfig
    wl = bench.WORKLOADS["cfg2"]
    B, T, V = wl["batch"], wl["cfg"]["block_size"], wl["cfg"]["vocab_size"]
    dumps = []
    for run in ("a", "b"):
        r, out = _bench("--workload", "cfg2", "--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--dump-outputs",
                        str(tmp_path / run), cwd=tmp_path)
        assert r.returncode == 0, r.stderr[-2000:]
        assert out["steps"] == 3
        dumps.append({f[:-len(".npy")]: np.load(tmp_path / run / f) for f in os.listdir(tmp_path / run)})
    a, b = dumps
    params = dict(GPT(GPTConfig(**wl["cfg"])).named_parameters())     # CPU module: names and sizes only
    assert set(a) == {"logits", "loss", "grad_norm"} | {"param." + n for n in params}
    assert all(x.dtype == np.float32 for x in a.values())
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["logits"].shape == (B, T, V) and a["loss"].shape == () and a["grad_norm"].shape == ()
    for n, p in params.items():
        assert a["param." + n].size == min(p.numel(), bench.PARAM_SAMPLE), n
    assert np.isfinite(a["grad_norm"]) and a["grad_norm"] > 0
    # loss and logits come from the same step: the loss is the cross-entropy of the dumped logits against bench.py's
    # targets (the second draw of its seeded generator)
    g = torch.Generator().manual_seed(1234)
    torch.randint(V, (B, T), generator=g)
    y = torch.randint(V, (B, T), generator=g)
    ce = torch.nn.functional.cross_entropy(torch.from_numpy(a["logits"]).double().view(-1, V), y.view(-1)).item()
    assert abs(ce - float(a["loss"])) <= 1e-4 * ce, (ce, float(a["loss"]))
    # same arguments, same inputs and weights: the runs differ only by the order of the fp32 atomic reductions of the
    # weight-gradient GEMMs (not bitwise, see tests/test_dropin_gpu.py), amplified over the six optimizer steps
    assert float(b["loss"]) == pytest.approx(float(a["loss"]), rel=1e-4)
    assert float(b["grad_norm"]) == pytest.approx(float(a["grad_norm"]), rel=1e-2)
    assert np.abs(a["logits"] - b["logits"]).max() <= 2e-2 * np.abs(a["logits"]).max()
