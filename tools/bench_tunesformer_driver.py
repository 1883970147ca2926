"""train_tunesformer.py against the bare packed step, one B200.

Writes a synthetic ABC corpus (to a temporary directory) whose tunes encode like the mixes of tools/bench_tunesformer_packed.py:
patch counts uniform on [--min-patches, --max-patches] (start patch, one header patch, bars, end patch), every bar 6..30
characters including its bar line, so its patch holds bos + 6..30 characters + eos.  Then it alternates, --rounds times, a run
of train_tunesformer.py at cfg4 widths (64 tunes per step, --epochs epochs of --steps steps) and tools/bench_tunesformer_packed.py,
each in a process of its own.  The driver's steady-state ms/step is the median over its epochs after the first (the first
carries the allocations); characters/s count the non-pad codes of patches 1..P-1 in both.  Prints one JSON line with the card
name and power limit read in the same run."""
import argparse
import json
import os
import random
import shutil
import statistics
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ap = argparse.ArgumentParser()
ap.add_argument("--tunes", type=int, default=64)
ap.add_argument("--min-patches", type=int, default=16)
ap.add_argument("--max-patches", type=int, default=128)
ap.add_argument("--steps", type=int, default=16)
ap.add_argument("--epochs", type=int, default=4)
ap.add_argument("--rounds", type=int, default=2)
ap.add_argument("--seed", type=int, default=0)
args = ap.parse_args()

name = torch.cuda.get_device_name(0)
try:
    power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    power = "unknown"

rng = random.Random(args.seed)
NOTES = "ABCDEFGabcdefgz2345/ "


def tune(i):
    n = rng.randint(args.min_patches, args.max_patches)
    bars = ["".join(rng.choice(NOTES) for _ in range(rng.randint(5, 29))) + "|" for _ in range(n - 3)]
    return {"id": str(i), "abc notation": f"X:{i}\n" + "".join(bars) + "\n"}


# every driver round writes a cfg4 weights.pth of about 1 GB: the directory goes when the script ends
workdir = tempfile.TemporaryDirectory(prefix="bench_tunesformer_driver_")
tmp = workdir.name
train, evl = os.path.join(tmp, "train.json"), os.path.join(tmp, "eval.json")
with open(train, "w") as f:
    json.dump([tune(i) for i in range(args.tunes * args.steps)], f)
with open(evl, "w") as f:
    json.dump([tune(i) for i in range(args.tunes)], f)


def run(cmd):
    r = subprocess.run([sys.executable, *cmd], cwd=ROOT, capture_output=True, text=True, timeout=1200)
    if r.returncode != 0:
        raise SystemExit(r.stdout[-2000:] + r.stderr[-4000:])
    return r.stdout


driver, bare = [], []
for r in range(args.rounds):
    for arm in ("driver", "bare") if r % 2 == 0 else ("bare", "driver"):
        if arm == "bare":
            out = json.loads(run(["tools/bench_tunesformer_packed.py", f"--tunes={args.tunes}",
                                  f"--min-patches={args.min_patches}", f"--max-patches={args.max_patches}"]).strip().splitlines()[-1])
            bare.append({"ms_per_step": out["ms_per_step"]["packed"], "chars_per_s": out["real_chars_per_s"]["packed"]})
        else:
            out_dir = os.path.join(tmp, f"run{r}")
            run(["train_tunesformer.py", "config/tunesformer_irishman.py", f"--train_data={train}", f"--eval_data={evl}",
                 f"--out_dir={out_dir}", f"--batch_size={args.tunes}", f"--num_epochs={args.epochs}", "--warmup_steps=8"])
            with open(os.path.join(out_dir, "logs.jsonl")) as f:
                logs = [json.loads(line) for line in f][1:]
            driver.append({"ms_per_step": statistics.median(x["ms_per_step"] for x in logs),
                           "chars_per_s": statistics.median(x["chars_per_s"] for x in logs),
                           "epochs": [x["ms_per_step"] for x in logs]})
            shutil.rmtree(out_dir)
ms_d = statistics.median(x["ms_per_step"] for x in driver)
ms_b = statistics.median(x["ms_per_step"] for x in bare)
print(json.dumps({
    "gpu": name, "power_limit": power,
    "workload": f"cfg4 widths, {args.tunes} tunes/step, patch counts uniform [{args.min_patches}, {args.max_patches}]; driver: "
                f"{args.tunes * args.steps} tunes, {args.steps} steps/epoch, {args.epochs} epochs",
    "driver_ms_per_step": ms_d, "bare_ms_per_step": ms_b, "driver_over_bare": ms_d / ms_b,
    "driver_chars_per_s": statistics.median(x["chars_per_s"] for x in driver),
    "bare_chars_per_s": statistics.median(x["chars_per_s"] for x in bare),
    "rounds": {"driver": driver, "bare": bare},
}))
