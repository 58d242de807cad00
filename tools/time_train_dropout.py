"""Cost of dropout in the training step: EfficientSATRN train_step at the benchmark's training shape (B = 16, targets
of 231 positions, fp32, default launch plan, CUDA graph of the pass) with dropout off and with p = p_ffn = 0.1
(set_train_dropout), alternating on one model after warm-up, each step timed with CUDA events.  Prints the median ms per
step of both, their ratio, and the GPU name and power limit read in the same run.  The batch is the seeded synthetic
training batch of oracle/train.py (target lengths uniform in [4, 230] tokens, PAD after <EOS>)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from helpers import make_model  # noqa: E402
from oracle import satrn, synth, train  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=16)
ap.add_argument("--positions", type=int, default=231)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--p", type=float, default=0.1)
ap.add_argument("--out", default=None, help="also write the result line (JSON) to this file")
a = ap.parse_args()
assert torch.cuda.is_available(), "time_train_dropout.py measures on the GPU"
dev = torch.device("cuda", 0)


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is reported as unknown rather than guessed
        return "unknown (%s)" % e


spec = satrn.ModelSpec()
model = make_model(synth.synth_state_dict(spec, 0), max_batch=a.batch, max_steps=a.positions).to(dev).train()
x, e = train.synth_batch(spec, a.batch, a.positions, 0)
x, e = x.to(dev), e.to(dev)
settings = {"off": (0.0, 0.0), "on": (a.p, a.p)}


def step(name):
    p, p_ffn = settings[name]
    model.set_train_dropout(p, seed=1, p_ffn=p_ffn)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    loss, _ = model.train_step(x, e, lr=1e-5)
    t1.record()
    t1.synchronize()
    assert torch.isfinite(loss).item(), name
    return t0.elapsed_time(t1)


for _ in range(a.warmup):     # eager pass, graph capture, replay of both settings
    for name in settings:
        step(name)
times = {name: [] for name in settings}
for _ in range(a.reps):
    for name in settings:
        times[name].append(step(name))
med = {name: statistics.median(v) for name, v in times.items()}
res = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(), "batch": a.batch, "positions": a.positions,
       "p": a.p, "reps": a.reps, "ms_per_step_off": round(med["off"], 3), "ms_per_step_on": round(med["on"], 3),
       "ratio_on_off": round(med["on"] / med["off"], 4),
       "spread_ms": {name: [round(min(v), 3), round(max(v), 3)] for name, v in times.items()}}
line = json.dumps(res)
print(line)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")
