"""Full-length greedy decode vs stop-at-<EOS> decode (frx_decode_greedy vs frx_decode_greedy_eos) on one 16-bit
EfficientSATRN handle: images/s of both, the work ratio sum(len) / (B * steps), and a bitwise check of the stop-at-<EOS>
output against the full one under the contract (equal up to the first <EOS>, <PAD> / zero rows after it).

Both calls decode a given encoder output (the encoder is the same for both and is left out).  The memory is the
golden memory of tests/golden tiled over the batch plus seeded noise.  Lengths:
  * forced: forced sequences whose <EOS> position is drawn per image from a seeded normal distribution,
    len = clip(round(N(mean, sd)), 1, steps) (--len-mean / --len-sd; default 40 / 20 tokens);
  * free:   free-running on the synthetic checkpoint with the <EOS> generator bias raised by +1.0 and by +2.0.
The two calls alternate, after warm-up, timed with CUDA events.  B = 256 is one wave of 32 clusters (no refill: a cluster
runs as long as its longest image); larger batches exercise the refill."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from helpers import make_model  # noqa: E402
from oracle import satrn, synth  # noqa: E402

EOS, PAD, V = satrn.EOS_ID, satrn.PAD_ID, 245

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="32,256,2048")
ap.add_argument("--steps", type=int, default=231)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--len-mean", type=float, default=40.0)
ap.add_argument("--len-sd", type=float, default=20.0)
ap.add_argument("--out", default=None, help="also write the result lines (JSON) to this file")
a = ap.parse_args()
assert torch.cuda.is_available(), "time_eos.py measures on the GPU"
dev = torch.device("cuda", 0)
st = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is reported as unknown rather than guessed
        return "unknown (%s)" % e


def model_for(bias):
    spec = satrn.ModelSpec()
    sd = dict(synth.synth_state_dict(spec, 0))
    if bias:
        sd["decoder.generator.bias"] = sd["decoder.generator.bias"].clone()
        sd["decoder.generator.bias"][EOS] += bias
    m = make_model(sd, precision="bf16")
    m.set_option("parts", 2)
    return m.to(dev).eval()


def memory(b, seed):
    base = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "efficientsatrn_seed0.npz"))["memory"])
    g = torch.Generator().manual_seed(seed)
    mem = base.repeat((b + base.size(0) - 1) // base.size(0), 1, 1)[:b]
    return (mem + 0.02 * mem.std() * torch.randn(mem.shape, generator=g)).to(dev).contiguous()


def forced_seqs(b, steps, seed):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(3, V, (b, steps), generator=g)
    n = (torch.randn(b, generator=g) * a.len_sd + a.len_mean).round().clamp(1, steps).long()
    tok[torch.arange(b), n - 1] = EOS
    return tok.to(dev)


def run(model, mem, forced):
    b, steps = mem.size(0), a.steps
    eng = model.engine(dev, b, steps)
    lf = torch.empty(b, steps, V, device=dev)
    tf = torch.empty(b, steps, dtype=torch.int64, device=dev)
    le = torch.empty(b, steps, V, device=dev)
    te = torch.empty(b, steps, dtype=torch.int64, device=dev)
    ln = torch.empty(b, dtype=torch.int32, device=dev)
    fp = forced.data_ptr() if forced is not None else None
    full = lambda: eng.h.call("frx_decode_greedy", mem.data_ptr(), b, steps, lf.data_ptr(), tf.data_ptr(), fp, st())  # noqa: E731
    eos = lambda: eng.h.call("frx_decode_greedy_eos", mem.data_ptr(), b, steps, le.data_ptr(), te.data_ptr(),  # noqa: E731
                             ln.data_ptr(), fp, 0, st())
    for _ in range(a.warmup):
        full()
        eos()
    times = {"full": [], "eos": []}
    for _ in range(a.reps):
        for name, fn in (("full", full), ("eos", eos)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))
    stop = forced if forced is not None else tf
    hit = stop == EOS
    want = torch.where(hit.any(1), hit.int().argmax(1) + 1, torch.full((b,), steps, device=dev))
    keep = torch.arange(steps, device=dev)[None, :] < want[:, None]
    same = (torch.equal(ln.long(), want) and torch.equal(te, torch.where(keep, tf, torch.full_like(tf, PAD)))
            and torch.equal(le, torch.where(keep[..., None], lf, torch.zeros_like(lf))))
    ms_f, ms_e = statistics.median(times["full"]), statistics.median(times["eos"])
    return {"B": b, "steps": steps, "work_ratio": round(want.sum().item() / (b * steps), 4),
            "full_ms": round(ms_f, 3), "eos_ms": round(ms_e, 3),
            "full_img_s": round(b / ms_f * 1e3, 1), "eos_img_s": round(b / ms_e * 1e3, 1),
            "speedup": round(ms_f / ms_e, 3), "bitwise_contract": bool(same),
            "full_ms_min_max": [round(min(times["full"]), 3), round(max(times["full"]), 3)],
            "eos_ms_min_max": [round(min(times["eos"]), 3), round(max(times["eos"]), 3)]}


lines = []
head = {"device": torch.cuda.get_device_name(0), "power_limit": power_limit(), "reps": a.reps, "warmup": a.warmup,
        "forced_lengths": "clip(round(N(%g, %g)), 1, %d)" % (a.len_mean, a.len_sd, a.steps)}
print(json.dumps(head), flush=True)
lines.append(head)
forced_model, free1, free2 = model_for(0.0), model_for(1.0), model_for(2.0)
with torch.no_grad():
    for b in [int(x) for x in a.batches.split(",")]:
        mem = memory(b, seed=b)
        for case, model, forced in (("forced", forced_model, forced_seqs(b, a.steps, seed=b + 1)),
                                    ("free, EOS bias +1.0", free1, None), ("free, EOS bias +2.0", free2, None)):
            r = dict(case=case, **run(model, mem, forced))
            print(json.dumps(r), flush=True)
            lines.append(r)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(json.dumps(x) for x in lines) + "\n")
