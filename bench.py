#!/usr/bin/env python
"""bench.py -- EfficientSATRN greedy-decode images/sec (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port)
    python bench.py --workload {train,beam4,beam8,lite,swin} # the other BASELINE.json configs (3, 4, 5), same contract
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's outputs as DIR/<name>.npy

A "step" is one pass of the hot path (encode + 231-step greedy decode) over one
synthetic batch of 256 images (128x256 grayscale, randn) per GPU.  `value` is
timed with CUDA events with the images already resident in HBM; `e2e` goes
through the host-buffer C-ABI entry (frx_forward_greedy_host): H2D of the pinned
images + compute + D2H of the tokens inside the timed region.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

MAX_SEQUENCE = 230          # inference.py:29 -> expected has 232 ids -> 231 steps
STEPS_PER_IMAGE = MAX_SEQUENCE + 1
METRIC = "EfficientSATRN greedy-decode images/sec"
# SURVEY 8d / BASELINE.md: algorithmic work per image
DECODE_BYTES_PER_IMAGE = {"fp32": 210.5e6, "bf16": 105.4e6}
ENCODE_FLOP_PER_IMAGE = 3.700e9 + 0.207e9
TOTAL_FLOP_PER_IMAGE = 5.54e9


# the decode kernel the library launches for batches of more than 15 clusters (two heads per CTA, clusters of 4)
DECODE_KERNEL = "dec_cluster_bf16_kernel_p2"


def ncu_traffic(kernel, batch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
    (profiles/ncu_traffic.json), or None when no capture matches this kernel / batch -- or when the kernel's source files
    have changed since the capture (the entry carries a hash of them), so the figure can never go stale silently."""
    import hashlib
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None
    for e in json.load(open(path)):
        if e["kernel"] == kernel and e["batch"] == batch:
            h = hashlib.sha256()
            try:
                for f in e.get("kernel_source_files", []):
                    h.update(open(os.path.join(ROOT, "p4-fr-sorry-math-but-love-you_b200", f), "rb").read())
            except OSError:
                return None
            if e.get("kernel_source_sha256_16") != h.hexdigest()[:16]:
                return None
            return e["dram_bytes_per_launch"]
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d["hbm_gbs"], d["bf16_tflops_sustained"], "measured"
    return 6650.0, 1400.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.

    The sampler process is started before the warm-up (nvidia-smi needs a few hundred ms to produce its first
    line on an 8-GPU box); every line is time-stamped on arrival and only the lines that fall inside
    [window_begin(), window_end()] are summarised."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), [c.strip() for c in line.split(",")]))

    def window_begin(self):
        self.t0 = time.monotonic()

    def window_end(self):
        self.t1 = time.monotonic()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in self.rows:
            if self.t0 is not None and not (self.t0 <= t <= self.t1 + 0.02):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_images(batch, seed):
    import torch
    g = torch.Generator().manual_seed(2000 + seed)
    return torch.randn(batch, 1, 128, 256, generator=g)


DUMP_BYTES = 60 * 10**6     # --dump-outputs stays under 64 MB with the .npy headers; the default greedy batch fits whole


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy: floating point as float32, integers (tokens) as float64, which holds them
    exactly.  When they exceed DUMP_BYTES together, the same seeded subset of rows of the leading (batch) dimension is
    kept of every array, so that two builds run with the same arguments still write comparable files."""
    import numpy as np
    arrs = {k: (v.float() if v.is_floating_point() else v.double()).cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_BYTES:
        n = next(iter(arrs.values())).shape[0]
        keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_BYTES // total), replace=False))
        arrs = {k: a[keep] for k, a in arrs.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def workload_config(batch, precision):
    return {"workload": "EfficientSATRN greedy inference, batch %d per GPU, 128x256x1 randn images, "
                        "max_sequence 230 (231 decode steps), seeded synthetic weights with calibrated BatchNorm "
                        "statistics, image batch sharded "
                        "over ranks (no collective)" % batch,
            "batch_per_gpu": batch, "decode_steps": STEPS_PER_IMAGE, "precision": precision,
            "l2": "256 MiB buffer written between timed iterations (L2 flush); per-step working set "
                  "(KV cache + activations) also exceeds the 126 MB L2"}


def checkpoint():
    """The EfficientSATRN weights every EfficientSATRN workload runs: the seeded synthetic checkpoint of the parity
    tests, whose BatchNorm running statistics are calibrated on a seeded batch.  With uncalibrated random-init
    statistics the trunk's activations grow to ~1e7, beyond the fp16 range of the 16-bit encoder, and the 16-bit
    workloads would time a pass whose logits are inf / NaN."""
    from oracle import satrn, synth
    return synth.synth_state_dict(satrn.ModelSpec(), 0)


def build_model(precision, batch):
    import frx
    from helpers import Vocab, flags_dict
    flags = frx.Flags(flags_dict()).get()
    sd = checkpoint()
    model = frx.EfficientSATRN(flags, Vocab(), sd, None, precision=precision, max_batch=batch,
                               max_steps=STEPS_PER_IMAGE)
    return model, sd


def cpu_reference_throughput(sd, sample_batch, runs, as_written=True):
    """The reference's CPU algorithm (oracle port, op for op incl. the per-step
    K/V re-projection) on the host cores.  Returns (images/s, cores, tokens)."""
    import torch
    from oracle import satrn
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    spec = satrn.ModelSpec()
    x = synthetic_images(sample_batch, 0)
    with torch.no_grad():
        satrn.forward_greedy(sd, spec, x[:2], 4, as_written=as_written)  # warm-up
        t0 = time.perf_counter()
        for _ in range(runs):
            logits = satrn.forward_greedy(sd, spec, x, STEPS_PER_IMAGE, as_written=as_written)
        dt = time.perf_counter() - t0
    return sample_batch * runs / dt, cores, logits.argmax(-1), dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    import torch
    sd = checkpoint()
    if args.workload != "greedy":
        wl = args.workload
        if wl == "lite":
            from oracle import satrn as o_satrn, synth as o_synth
            from oracle.make_golden import LITE_SPEC
            sd = o_synth.synth_state_dict(o_satrn.ModelSpec(**LITE_SPEC), 0, calib_batch=4)
        elif wl == "swin":
            from oracle import swin as o_swin
            sd = o_swin.synth_state_dict(o_swin.swin_spec(), 0)
        t0 = time.perf_counter()
        cb = cpu_workload_baseline(wl, args, sd)
        print(json.dumps({"impl": "reference", "metric": wl, "value": cb["value"], "unit": cb["unit"], "n_gpus": args.gpus,
                          "steps": 1, "warmup": 0, "ms_per_step": (time.perf_counter() - t0) * 1e3, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": wl + " (bounded sample, see cpu_baseline.sample)"}, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    sample = args.cpu_sample
    for _ in range(args.warmup):
        pass  # the warm-up happens inside cpu_reference_throughput on a tiny batch
    ips, cores, _, dt = cpu_reference_throughput(sd, sample, max(1, args.steps))
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3,
        "ms_per_step_is": "per bounded sample of %d images (the GPU arm's step is %d images)" % (sample, args.batch),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args.batch, args.precision),
                       reference_arm="the reference's CPU algorithm (oracle port, op for op, fp32) on the host cores; "
                                     "each step is a bounded sample of %d images of the same workload" % sample),
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": "%d step(s) x %d images x 231 decode steps, torch %s CPU fp32, %d threads"
                                   % (max(1, args.steps), sample, torch.__version__, cores)},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_frx(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU for --impl frx (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, T = args.batch, STEPS_PER_IMAGE
    model, sd = build_model(args.precision, B)
    model = model.to(dev).eval()
    model.set_option("timing", 1)
    images_host = synthetic_images(B, rank).pin_memory()
    images = images_host.to(dev)
    logits = torch.empty(B, T, 245, device=dev)
    tokens = torch.empty(B, T, dtype=torch.int64, device=dev)
    tokens_host = torch.empty(B, T, dtype=torch.int64).pin_memory()
    eng = model.engine(dev, B, T)
    stream = torch.cuda.current_stream(dev).cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_device():
        eng.h.call("frx_forward_greedy", images.data_ptr(), B, T, logits.data_ptr(), tokens.data_ptr(), stream)

    def step_host():
        eng.h.call("frx_forward_greedy_host", images_host.data_ptr(), B, T, None, tokens_host.data_ptr(), stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    clocks = ClockSampler(local_rank).start()
    for _ in range(max(args.warmup, 1)):
        step_device()
    torch.cuda.synchronize(dev)
    import ctypes
    ms3 = (ctypes.c_float * 4)()

    # ---- timed region 1: device-resident inputs, CUDA events -------------------
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = eng.launches
    enc_ms, dec_ms, kern_ms = [], [], []
    barrier()
    clocks.window_begin()
    for s, e in ev:
        flush.zero_()            # L2 flush between timed iterations (outside the event pair)
        s.record()
        step_device()
        e.record()
        e.synchronize()
        eng.h.lib.frx_last_timing(eng.h.ptr, ms3)
        enc_ms.append(ms3[0]); dec_ms.append(ms3[1]); kern_ms.append(ms3[3])
    barrier()
    clocks.window_end()
    clocks.stop()
    gpu_launches = eng.launches - launches0
    total_ms = sum(s.elapsed_time(e) for s, e in ev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logits": logits, "tokens": tokens})   # the last timed step's results

    # ---- timed region 2: host buffers through the public entry (e2e) ------------
    # (a) one synchronous call per batch (H2D -> encode -> decode -> D2H -> sync), (b) the pipelined entry: the same
    # per-batch copies, but batch i+1's H2D and batch i-1's D2H run on their own streams under batch i's compute.
    for _ in range(2):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()              # synchronises the stream before returning
    barrier()
    e2e_sync_s = time.perf_counter() - t0
    model.set_option("timing", 0)
    img2 = [images_host, images_host.clone().pin_memory()]
    tok2 = [tokens_host, torch.empty_like(tokens_host).pin_memory()]

    def pipelined(n):
        for i in range(n):
            if i >= 2:
                eng.h.call("frx_forward_greedy_host_wait", i % 2)
            eng.h.call("frx_forward_greedy_host_submit", img2[i % 2].data_ptr(), B, T, tok2[i % 2].data_ptr(), i % 2, stream)
        eng.h.call("frx_forward_greedy_host_wait", 0)
        eng.h.call("frx_forward_greedy_host_wait", 1)
    pipelined(2)
    barrier()
    t0 = time.perf_counter()
    pipelined(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    # the same pipelined entry fed from DEVICE buffers: what the cross-batch overlap (next batch's encoder on the SMs the
    # decode kernel leaves idle) is worth without PCIe in the picture
    img2 = [images, images.clone()]
    tok2 = [tokens, torch.empty_like(tokens)]
    pipelined(2)
    barrier()
    t0 = time.perf_counter()
    pipelined(args.steps)
    barrier()
    overlapped_s = time.perf_counter() - t0
    model.set_option("timing", 1)

    import frx
    total_ms = frx.sharding.max_over_ranks(total_ms, dev)      # the job is as slow as its slowest rank
    e2e_ms = frx.sharding.max_over_ranks(e2e_s * 1e3, dev)
    e2e_sync_ms = frx.sharding.max_over_ranks(e2e_sync_s * 1e3, dev)
    overlapped_ms = frx.sharding.max_over_ranks(overlapped_s * 1e3, dev)
    if rank != 0:
        return
    n_img = B * args.steps * world
    value = n_img / (total_ms / 1e3)
    e2e = n_img / (e2e_ms / 1e3)
    hbm, tflops, how = peaks()
    dec_s = statistics.mean(dec_ms) / 1e3
    enc_s = statistics.mean(enc_ms) / 1e3
    single_kernel = args.precision == "bf16" and statistics.mean(kern_ms) > 0
    if single_kernel:
        dec_s = statistics.mean(kern_ms) / 1e3
    dec_bytes = DECODE_BYTES_PER_IMAGE[args.precision] * B
    achieved = dec_bytes / dec_s / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16",
        "dtype_detail": "fp32" if args.precision == "fp32" else "16-bit operands, fp32 accumulation: fp16 on the encoder side (tcgen05 kind::f16), bf16 weights + KV cache in the decode kernel",
        "data": "synthetic",
        "config": workload_config(B, args.precision),
        "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(images_host.numel() * 4),
                "d2h_bytes_per_step": int(tokens_host.numel() * 8),
                "how": "frx_forward_greedy_host_submit / _wait from pinned host buffers, two batches in flight: every step's "
                       "H2D of its images and D2H of its tokens are inside the timed region, on copy streams under the "
                       "neighbouring steps' compute; the next batch's encoder also overlaps the current batch's decode "
                       "kernel (own stream, the 20 SMs the decode leaves idle), which is why e2e exceeds the "
                       "one-batch-at-a-time `value`",
                "value_one_synchronous_call_per_step": n_img / (e2e_sync_ms / 1e3)},
        "value_overlapped": {"value": n_img / (overlapped_ms / 1e3), "unit": "images/s",
                             "how": "device-resident inputs through the pipelined entry (two batches in flight: batch i+1's "
                                    "encoder runs on its own stream under batch i's decode kernel, which leaves 20 of the 148 SMs "
                                    "idle); `value` is one batch at a time"},
        "gpu_launches": int(gpu_launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                     "traffic": ncu_traffic(DECODE_KERNEL, B) if single_kernel else None,
                     "kernel": DECODE_KERNEL + " (one launch = all 231 decode steps of the batch)" if single_kernel
                     else "greedy decode loop (CUDA graph of the fp32 step kernels)",
                     "algorithmic_bytes_per_launch": dec_bytes,
                     "ms": dec_s * 1e3, "peak_source": how},
        "roofline_encoder": {"bound": "tensor", "achieved": ENCODE_FLOP_PER_IMAGE * B / enc_s / 1e12, "peak": tflops,
                             "unit": "TFLOP/s", "frac": ENCODE_FLOP_PER_IMAGE * B / enc_s / 1e12 / tflops,
                             "ms": enc_s * 1e3, "peak_source": how},
        "clocks": clocks.summary(),
    }
    if world == 1 and not args.no_cpu_baseline:
        # CPU leg: the oracle's op-for-op port of the reference's CPU algorithm, timed on a bounded sample, on the
        # checkpoint the GPU arm runs, and the token agreement of both GPU modes with it on the same images.
        from oracle import satrn as o_satrn
        import frx
        from helpers import Vocab, flags_dict
        ips, cores, cpu_tok, dt = cpu_reference_throughput(sd, args.cpu_sample, args.cpu_runs)
        xs = synthetic_images(args.cpu_sample, 0).to(dev)
        agree = {}
        with torch.no_grad():
            for prec in ("fp32", "bf16"):
                m = frx.EfficientSATRN(frx.Flags(flags_dict()).get(), Vocab(), sd, None, precision=prec,
                                       max_batch=args.cpu_sample, max_steps=T).to(dev).eval()
                _, tok = m.greedy(xs, T)
                agree[prec] = (tok.cpu() == cpu_tok).float().mean().item()
                del m
        # the same port on THIS GPU in eager PyTorch (cuDNN / cuBLAS, TF32 off): what moving the reference to .cuda() gives
        try:
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            sd_gpu = {k: (v.float() if v.is_floating_point() else v).to(dev) for k, v in sd.items()}
            xg = synthetic_images(B, 0).to(dev)
            with torch.no_grad():
                o_satrn.forward_greedy(sd_gpu, o_satrn.ModelSpec(), xg[:8], 8, as_written=True)
                torch.cuda.synchronize(dev)
                g0 = time.perf_counter()
                o_satrn.forward_greedy(sd_gpu, o_satrn.ModelSpec(), xg, T, as_written=True)
                torch.cuda.synchronize(dev)
                gdt = time.perf_counter() - g0
            line["gpu_eager_baseline"] = {"value": B / gdt, "unit": "images/s", "ms_per_batch": gdt * 1e3, "kind": "port",
                                          "sample": "1 batch of %d images x 231 steps, the oracle port of the reference's as-written "
                                                    "algorithm in eager PyTorch %s on this GPU, fp32, TF32 disabled" % (B, torch.__version__)}
            del sd_gpu, xg
        except Exception as exc:  # reported, never fatal: this is a yardstick, not the product
            line["gpu_eager_baseline"] = {"unavailable": repr(exc)[:200]}
        line["cpu_baseline"] = {
            "value": ips, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": "%d batches of %d images x 231 decode steps (%.1f s), oracle port of the reference's "
                      "as-written CPU algorithm, torch %s fp32, BN-calibrated synthetic checkpoint"
                      % (args.cpu_runs, args.cpu_sample, dt, torch.__version__),
            "gpu_fp32_mode_token_agreement": agree["fp32"],
            "gpu_bf16_mode_token_agreement": agree["bf16"]}
    print(json.dumps(line), flush=True)


# =====================================================================================================================
# Other workloads of BASELINE.json.configs: [2] beam search (width 4 / 8), [3] the teacher-forced training step with the
# NCCL gradient all-reduce, [4] LiteSATRN / SwinTRN greedy inference.  Same JSON contract as the headline workload.
# =====================================================================================================================
# training: forward 3.907 GFLOP (trunk + encoder) + teacher-forced decoder over 231 rows (2.815 MMAC per row in the linear
# layers, 41 MMAC self-attention, 11 MMAC cross-attention, 25 MMAC cross K/V) = 5.36 GFLOP; backward = 2x forward
TRAIN_FLOP_PER_IMAGE = 3.0 * (3.907e9 + 2.0 * (231 * 2.815232e6 + 41.0e6 + 11.4e6 + 25.2e6))
# SURVEY A.6: LiteSATRN encoder 0.507 GFLOP / image (ShallowCNN 4 convs + 1 encoder layer at 8x16 tokens); its decode
# (hidden 128, 2 layers, 4 heads) streams sum_t t*2*2*128*2 B of bf16 self K/V + 128 tokens of cross K/V per step
LITE_DECODE_BYTES = sum(t * 2 * 2 * 128 * 2 for t in range(231)) + 231 * 2 * 2 * 128 * 128 * 2 + 231 * 245 * 4
SWIN_ENC_FLOP = 2.0 * 47.1e9 / 2 * 1.0   # Swin-B/384: 47.1 GFLOP (multiply-adds counted as 2) per 384x384 image
SWIN_DECODE_BYTES = sum(t * 4 * 2 * 512 * 4 for t in range(231)) + 231 * 4 * 2 * 144 * 512 * 4 + 231 * 245 * 4   # fp32 step kernels


def _timed(step, steps, warmup, dev, world, flush):
    import torch
    import torch.distributed as dist
    for _ in range(max(warmup, 1)):
        step()
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t_begin = time.monotonic()
    for s, e in ev:
        flush.zero_()
        s.record()
        last = step()
        e.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    return sum(s.elapsed_time(e) for s, e in ev), t_begin, time.monotonic(), last


def run_workload(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import frx
    from helpers import Vocab, flags_dict, make_lite_model, make_swin_model
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    wl, T = args.workload, STEPS_PER_IMAGE
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    hbm, tflops, how = peaks()
    clocks = ClockSampler(local_rank).start()
    extra, roof, cpu = {}, None, None
    g = torch.Generator().manual_seed(2000 + rank)

    if wl == "train":
        B = args.batch or 16                    # configs/EfficientSATRN.yaml: batch_size 16 (per GPU here)
        model, sd = build_model("fp32", B)
        model = model.to(dev).train()
        x_host = torch.randn(B, 1, 128, 256, generator=g).pin_memory()
        e_host = torch.cat([torch.zeros(B, 1, dtype=torch.long), torch.randint(3, 244, (B, MAX_SEQUENCE), generator=g),
                            torch.ones(B, 1, dtype=torch.long)], 1).pin_memory()       # [SOS] + 230 tokens + [EOS]
        x, e = x_host.to(dev), e_host.to(dev)
        eng = model.engine(dev, B, T)
        step_device = lambda: model.train_step(x, e)
        outputs = lambda last: {"loss": last[0], "grad_norm": last[1]}

        def step_host():
            loss, _ = model.train_step(x_host.to(dev, non_blocking=True), e_host.to(dev, non_blocking=True))
            return loss.item()
        h2d, d2h = x_host.numel() * 4 + e_host.numel() * 8, 4
        metric = "EfficientSATRN teacher-forced training images/sec"
        desc = ("EfficientSATRN teacher-forced training step (single_opt, teacher_forcing_ratio 1.0: train-mode BatchNorm, "
                "CrossEntropy ignore PAD, backward, clip_grad_norm 2.0, AdamW), batch %d per GPU, 128x256x1 randn images, "
                "231 target positions, fp32 like the reference, gradients all-reduced over NCCL (%d ranks)" % (B, world))
        dtype = "f32"
    elif wl in ("beam4", "beam8"):
        B, width = args.batch or 256, int(wl[4:])  # the headline batch (the reference's inference.py default is 32)
        model, sd = build_model(args.precision, B)  # 16-bit: every node expansion is one cluster-kernel launch (step mode)
        model = model.to(dev).eval()
        x_host = synthetic_images(B, rank).pin_memory()
        x = x_host.to(dev)
        eng = model.engine(dev, B, T)
        step_device = lambda: model.beam_search(x, None, 1, width, MAX_SEQUENCE)    # returns the tokens on the host
        outputs = lambda last: {"tokens": last}
        step_host = lambda: model.beam_search(x_host.to(dev, non_blocking=True), None, 1, width, MAX_SEQUENCE)
        h2d, d2h = x_host.numel() * 4, B * MAX_SEQUENCE * 8
        metric = "EfficientSATRN beam-search (width %d) images/sec" % width
        desc = ("EfficientSATRN beam_search(topk=1, beam_width=%d, max_sequence=230) through decode(): best-first queue on the "
                "device, batch %d per GPU, %s" % (width, B, "16-bit mode: one cluster-kernel launch per round (step mode)"
                                                  if args.precision == "bf16" else "fp32 step kernels"))
        dtype = "bf16" if args.precision == "bf16" else "f32"
    elif wl == "lite":
        from oracle import satrn as o_satrn, synth as o_synth
        from oracle.make_golden import LITE_SPEC
        B = args.batch or 256
        lspec = o_satrn.ModelSpec(**LITE_SPEC)
        sd = o_synth.synth_state_dict(lspec, 0, calib_batch=4)
        model = make_lite_model(sd, precision=args.precision, max_batch=B, max_steps=T).to(dev).eval()
        x_host = o_synth.synth_images(lspec, B, rank).pin_memory()
        x = x_host.to(dev)
        model.set_option("timing", 1)
        eng = model.engine(dev, B, T)
        tok = torch.empty(B, T, dtype=torch.int64, device=dev)
        step_device = lambda: eng.h.call("frx_forward_greedy", x.data_ptr(), B, T, None, tok.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        outputs = lambda last: {"tokens": tok}
        step_host = lambda: model.greedy(x_host.to(dev, non_blocking=True), T, want_logits=False)[1].cpu()
        h2d, d2h = x_host.numel() * 4, B * T * 8
        metric = "LiteSATRN greedy-decode images/sec"
        desc = "LiteSATRN greedy inference, batch %d per GPU, 128x256x1 images, 231 decode steps, %s mode" % (B, args.precision)
        dtype = "bf16" if args.precision == "bf16" else "f32"
    else:  # swin
        from oracle import swin as o_swin
        B = args.batch or 64
        sd = o_swin.synth_state_dict(o_swin.swin_spec(), 0)
        model = make_swin_model(sd, precision=args.precision, max_batch=B, max_steps=T).to(dev).eval()
        x_host = o_swin.synth_images(B, rank).pin_memory()
        x = x_host.to(dev)
        model.set_option("timing", 1)
        eng = model.engine(dev, B, T)
        tok = torch.empty(B, T, dtype=torch.int64, device=dev)
        step_device = lambda: eng.h.call("frx_forward_greedy", x.data_ptr(), B, T, None, tok.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
        outputs = lambda last: {"tokens": tok}
        step_host = lambda: model.greedy(x_host.to(dev, non_blocking=True), T, want_logits=False)[1].cpu()
        h2d, d2h = x_host.numel() * 4, B * T * 8
        metric = "SwinTRN greedy-decode images/sec"
        desc = ("SwinTRN (Swin-B/384 encoder + 4-layer decoder) greedy inference, batch %d per GPU, 384x384x3 images, 231 decode "
                "steps, %s mode (encoder on tcgen05, decoder on the 512-wide cluster kernel)" % (B, args.precision))
        dtype = "bf16" if args.precision == "bf16" else "f32"

    launches0 = eng.launches
    total_ms, t0, t1, last = _timed(step_device, args.steps, args.warmup, dev, world, flush)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs(last))
    clocks.t0, clocks.t1 = t0, t1
    clocks.stop()
    gpu_launches = eng.launches - launches0
    ms3 = (ctypes.c_float * 4)()
    eng.h.lib.frx_last_timing(eng.h.ptr, ms3)
    # e2e: host buffers, H2D + D2H inside the timed region.  Greedy workloads go through the pipelined host entry (two
    # batches in flight, copies and the next batch's encoder under the current batch's decode); the others are one
    # synchronous call per step.
    e2e_how = "one synchronous call per step (H2D of the inputs, compute, D2H of the result)"
    if wl in ("lite", "swin"):
        model.set_option("timing", 0)
        xh2 = [x_host, x_host.clone().pin_memory()]
        th2 = [torch.empty(B, T, dtype=torch.int64).pin_memory() for _ in range(2)]
        stream = torch.cuda.current_stream(dev).cuda_stream

        def run_pipelined(n):
            for i in range(n):
                if i >= 2:
                    eng.h.call("frx_forward_greedy_host_wait", i % 2)
                eng.h.call("frx_forward_greedy_host_submit", xh2[i % 2].data_ptr(), B, T, th2[i % 2].data_ptr(), i % 2, stream)
            eng.h.call("frx_forward_greedy_host_wait", 0)
            eng.h.call("frx_forward_greedy_host_wait", 1)
        step_all = run_pipelined
        e2e_how = "frx_forward_greedy_host_submit / _wait from pinned host buffers, two batches in flight"
    else:
        def step_all(n):
            for _ in range(n):
                step_host()
    step_all(2)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    w0 = time.perf_counter()
    step_all(args.steps)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    e2e_ms = (time.perf_counter() - w0) * 1e3
    allreduce = None
    if wl == "train" and world > 1:
        grads = eng._train["grads"]
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.all_reduce(grads)
        torch.cuda.synchronize(dev)
        a0.record()
        for _ in range(5):
            dist.all_reduce(grads)
        a1.record()
        torch.cuda.synchronize(dev)
        allreduce = {"bytes": int(grads.numel() * 4), "ms_alone": a0.elapsed_time(a1) / 5,
                     "how": "flat fp32 gradient buffer, one NCCL all-reduce after the CUDA graph of the forward + backward pass "
                            "(train_step's default; overlap=True starts 6 buckets from inside an eagerly launched backward pass "
                            "instead: slower while the exchange is 1 % of the step); ms_alone = that all-reduce timed by itself"}
    total_ms = frx.sharding.max_over_ranks(total_ms, dev)
    e2e_ms = frx.sharding.max_over_ranks(e2e_ms, dev)
    if rank != 0:
        return
    n_img = B * args.steps * world
    step_s = total_ms / args.steps / 1e3
    if wl == "train":
        ach = TRAIN_FLOP_PER_IMAGE * B / step_s / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": tflops, "unit": "TFLOP/s", "frac": ach / tflops, "traffic": None,
                "kernel": "whole step (fp32 FFMA implicit-GEMM forward / dgrad / wgrad kernels; the bf16 tensor-core peak is "
                          "the yardstick the task names, the fp32 FFMA peak of a B200 is ~75 TFLOP/s)",
                "algorithmic_flop_per_step": TRAIN_FLOP_PER_IMAGE * B, "ms": step_s * 1e3, "peak_source": how}
    elif wl in ("beam4", "beam8"):
        by = DECODE_BYTES_PER_IMAGE["fp32" if args.precision == "fp32" else "bf16"] * B
        dec_s = step_s    # whole step (the encoder is ~2 % of it at this batch)
        roof = {"bound": "hbm", "achieved": by / dec_s / 1e9, "peak": hbm, "unit": "GB/s", "frac": by / dec_s / 1e9 / hbm,
                "traffic": None, "kernel": "beam rounds (select + decoder step + push), one node expansion per image and round",
                "algorithmic_bytes_per_launch": by, "ms": dec_s * 1e3, "peak_source": how,
                "note": "upper bound on the useful bytes: an explored chain of 230 nodes reads the fp32 K/V history a greedy pass reads"}
    elif wl == "lite":
        by = LITE_DECODE_BYTES * B
        dec_s = max(ms3[3] if ms3[3] > 0 else ms3[1], 1e-6) / 1e3
        roof = {"bound": "hbm", "achieved": by / dec_s / 1e9, "peak": hbm, "unit": "GB/s", "frac": by / dec_s / 1e9 / hbm,
                "traffic": None, "kernel": "dec_cluster_bf16_kernel_d128 (one launch = all 231 steps)" if args.precision == "bf16" else "fp32 step kernels",
                "algorithmic_bytes_per_launch": by, "ms": dec_s * 1e3, "peak_source": how}
    else:
        enc_s = max(ms3[0], 1e-6) / 1e3
        ach = 47.1e9 * B / enc_s / 1e12
        roof = {"bound": "tensor", "achieved": ach, "peak": tflops, "unit": "TFLOP/s", "frac": ach / tflops, "traffic": None,
                "kernel": "Swin-B/384 encoder (tcgen05 GEMMs + window attention on mma.sync); 47.1 GFLOP per image",
                "ms": enc_s * 1e3, "peak_source": how, "decode_ms": ms3[1]}
    line = {
        "metric": metric, "value": n_img / (total_ms / 1e3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 1), "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": {"workload": desc, "batch_per_gpu": B, "l2": "256 MiB buffer written between timed iterations (L2 flush)"},
        "e2e": {"value": n_img / (e2e_ms / 1e3), "unit": "images/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "how": e2e_how},
        "gpu_launches": int(gpu_launches), "roofline": roof, "clocks": clocks.summary(),
        "timing_ms": {"encode": ms3[0], "decode": ms3[1]},
    }
    if allreduce:
        line["allreduce"] = allreduce
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_workload_baseline(wl, args, sd)
    print(json.dumps(line), flush=True)


def cpu_workload_baseline(wl, args, sd):
    """The oracle's port of the reference's CPU algorithm for the workload, on a bounded sample, all host threads."""
    import torch
    from oracle import satrn as o_satrn
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    spec = o_satrn.ModelSpec()
    if wl == "train":
        from oracle import train as o_train
        tr = o_train.Trainer(sd, spec)
        x, e = o_train.synth_batch(spec, 4, 231, 0)
        tr.step(x[:1], e[:1, :9])
        t0 = time.perf_counter()
        tr.step(x, e)
        dt = time.perf_counter() - t0
        return {"value": 4 / dt, "unit": "images/s", "cores": cores, "kind": "port",
                "sample": "1 training step of 4 images x 231 positions (%.1f s), oracle port (torch %s autograd, fp32)" % (dt, torch.__version__)}
    if wl in ("beam4", "beam8"):
        x = synthetic_images(2, 0)
        with torch.no_grad():
            src = o_satrn.encoder_forward(sd, spec, x)
            t0 = time.perf_counter()
            o_satrn.beam_search(sd, spec, src, int(wl[4:]), MAX_SEQUENCE)
            dt = time.perf_counter() - t0
        return {"value": 2 / dt, "unit": "images/s", "cores": cores, "kind": "port",
                "sample": "beam search of 2 images (%.1f s; the reference processes images one at a time), oracle port, encoder excluded" % dt}
    if wl == "lite":
        from oracle.make_golden import LITE_SPEC
        from oracle import synth as o_synth
        lspec = o_satrn.ModelSpec(**LITE_SPEC)
        x = o_synth.synth_images(lspec, 32, 0)
        with torch.no_grad():
            t0 = time.perf_counter()
            o_satrn.forward_greedy(sd, lspec, x, STEPS_PER_IMAGE, as_written=True)
            dt = time.perf_counter() - t0
        return {"value": 32 / dt, "unit": "images/s", "cores": cores, "kind": "port",
                "sample": "32 images x 231 decode steps (%.1f s), oracle port of the as-written algorithm" % dt}
    from oracle import swin as o_swin
    x = o_swin.synth_images(2, 0)
    with torch.no_grad():
        t0 = time.perf_counter()
        mem = o_swin.encoder_forward(sd, x)
        o_satrn.decode_greedy(o_swin.decoder_view(sd), o_swin.swin_spec(), mem, 24)
        dt = time.perf_counter() - t0
    return {"value": 2 / dt, "unit": "images/s (24 decode steps only)", "cores": cores, "kind": "port",
            "sample": "2 images x 24 decode steps (%.1f s): encoder-dominated sample of the oracle port" % dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="frx", choices=["frx", "reference"])
    ap.add_argument("--workload", default="greedy", choices=["greedy", "train", "beam4", "beam8", "lite", "swin"])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: 256 greedy/lite/beam, 16 train, 64 swin)")
    ap.add_argument("--precision", default=os.environ.get("FRX_PRECISION", "bf16"), choices=["fp32", "bf16"])
    ap.add_argument("--cpu-sample", type=int, default=32)
    ap.add_argument("--cpu-runs", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, under 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl frx")
    if args.workload == "greedy" and not args.batch:
        args.batch = 256
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "greedy":
            run_frx(args, rank, world, local_rank)
        else:
            run_workload(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
