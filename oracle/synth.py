"""Seeded synthetic checkpoint in the reference's state_dict layout.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

There is no network for the pretrained timm weights or trained checkpoints, so
every run uses synthetic weights (BASELINE.json: "random-init weights").  A
plain ``nn.Module`` default init is degenerate for parity purposes (SURVEY F5:
with fresh BatchNorm running stats the 40-block trunk shrinks activations to
1e-7 and every image decodes the same sequence), so the generator below
  1. draws every parameter from a seeded ``torch.Generator`` (CPU, fp32) in the
     order of ``oracle.satrn.param_shapes`` -- variance-preserving normal conv /
     linear weights, NON-zero biases, non-unit norm gains, so that a missing
     bias or a swapped gain shows up in the parity tests;
  2. calibrates every BatchNorm's running statistics with one fp64 forward of
     a seeded batch and rounds them to 10 mantissa bits, which makes the
     resulting state_dict bit-identical on any host (the build container and
     the GPU box generate the same checkpoint from the same seed).
The same dict is loaded by the real reference (``load_state_dict(strict=True)``,
oracle/make_golden.py), by the oracle and by the CUDA library.
"""
from __future__ import annotations

import hashlib
import os
import tempfile
from typing import Dict

import torch

from . import satrn


def _cache_dir() -> str:
    """Per-user directory under the system temporary directory, never inside the repository (which may be
    read-only).  Its name carries a hash of this file and of oracle/satrn.py (the BatchNorm calibration forward), so
    a checkpoint cached by other code is never loaded."""
    h = hashlib.sha256()
    for f in (__file__, satrn.__file__):
        with open(f, "rb") as fh:
            h.update(fh.read())
    return os.path.join(tempfile.gettempdir(), "frx-synth-%d-%s" % (os.getuid(), h.hexdigest()[:16]))


def _draw(name: str, shape: tuple, g: torch.Generator) -> torch.Tensor:
    leaf = name.rsplit(".", 1)[-1]
    if leaf == "num_batches_tracked":
        return torch.ones((), dtype=torch.long)
    if leaf == "running_mean":
        return torch.zeros(shape)
    if leaf == "running_var":
        return torch.ones(shape)
    is_norm = any(t in name for t in (".bn", "norm", "batch_norm"))
    if is_norm and leaf == "weight":
        return torch.rand(shape, generator=g) * 0.8 + 0.6
    if is_norm and leaf == "bias":
        return torch.randn(shape, generator=g) * 0.1
    if leaf == "bias":
        return torch.randn(shape, generator=g) * 0.05
    if name == "decoder.embedding.weight":
        return torch.randn(shape, generator=g) * 0.1
    fan_in = 1
    for d in shape[1:]:
        fan_in *= d
    gain = 2.0 if (len(shape) == 4 and "se." not in name) else 1.0
    if ".q_linear." in name or ".k_linear." in name:
        gain = 4.0  # temperature is sqrt(d_model): keep the softmax non-uniform
    return torch.randn(shape, generator=g) * (gain / fan_in) ** 0.5


def synth_state_dict(spec: satrn.ModelSpec, seed: int = 0, calib_batch: int = 8,
                     cache: bool = True) -> Dict[str, torch.Tensor]:
    tag = "%s_%dx%dx%d_s%d_b%d.pt" % (spec.network, spec.in_ch, spec.height, spec.width, seed, calib_batch)
    cache_dir = _cache_dir()
    path = os.path.join(cache_dir, tag)
    # only a directory this user owns is trusted (the temporary directory is shared)
    if cache and os.path.exists(path) and os.stat(cache_dir).st_uid == os.getuid():
        return torch.load(path)
    g = torch.Generator().manual_seed(1000 + seed)
    sd = {n: _draw(n, s, g) for n, s in satrn.param_shapes(spec).items()}
    # make <EOS> reachable so the best-first search exercises its stop rule
    sd["decoder.generator.bias"][satrn.EOS_ID] += 1.0
    imgs = torch.randn(calib_batch, spec.in_ch, spec.height, spec.width, generator=g, dtype=torch.float64)
    with torch.no_grad():
        satrn.encoder_forward(sd, spec, imgs, calib=satrn._Calib(sd))
    if cache:
        try:
            os.makedirs(cache_dir, mode=0o700, exist_ok=True)
            tmp = path + ".%d.tmp" % os.getpid()
            torch.save(sd, tmp)
            os.replace(tmp, path)
        except OSError:
            pass    # the cache only saves time
    return sd


def synth_images(spec: satrn.ModelSpec, batch: int, seed: int = 0) -> torch.Tensor:
    """SURVEY 8d: images = randn(B, C, H, W) from a seeded CPU generator."""
    g = torch.Generator().manual_seed(2000 + seed)
    return torch.randn(batch, spec.in_ch, spec.height, spec.width, generator=g)
