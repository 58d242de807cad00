"""Counter-based dropout of the training step, restated on the CPU (test infrastructure, like oracle/).

The reference draws its dropout masks from torch's global RNG, which no other implementation can reproduce.  The
library's training step (include/frx.h frx_train_set_dropout) instead keys each mask by its position: Philox4x32-10
(Random123, the generator of curand_Philox4x32_10) with key = the 64-bit seed (low word, high word) and counter
(element index // 4, site + 16 * layer, step, rank); word (index % 4) of the output decides the element.  An element is
kept iff that word is >= min(2^32 - 1, floor(p * 2^32)), p taken as fp32 and the product in float64; kept values are
multiplied by the fp32 scale 1 / (1 - p), dropped ones are 0.

``train_forward`` / ``Trainer`` are oracle/train.py's training step with these masks applied at the reference's sites
(the oracle's own functions, oracle/satrn.py, carry no dropout: they are the parity yardstick and stay as they are).
Torch autograd through them gives the gradients of the masked network.  Sites (the element index runs over the logical
layout given; EfficientSATRN.py line numbers as in oracle/satrn.py):
  0 2-D PE output [B, C, h, w] (:101) | 1 / 2 encoder attention probabilities [B, heads, S, S] / MHA output [B, S, C]
  3 decoder input [B, L, D] (:406) | 4 / 5 decoder self-attention probabilities [B, H, L, L] / output [B, L, D]
  6 / 7 cross-attention probabilities [B, H, L, S] / output [B, L, D] | 8 / 9 after the feed-forward ReLUs (rate p_ffn)
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

from oracle import satrn, train

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF
FFN_SITES = (8, 9)


def philox4x32(ctr, key):
    """Philox4x32-10, vectorised: ctr = four uint32 arrays (or scalars) of one shape, key = two uint32 scalars ->
    four uint32 arrays."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK for x in ctr]
    shape = np.broadcast_shapes(*(x.shape for x in c))
    c = [np.broadcast_to(x, shape).astype(np.uint64) for x in c]
    k0, k1 = np.uint64(key[0] & _MASK), np.uint64(key[1] & _MASK)
    m0, m1, lo = np.uint64(_M0), np.uint64(_M1), np.uint64(_MASK)
    for _ in range(10):
        p0, p1 = m0 * c[0], m1 * c[2]          # < 2^64: exact in uint64
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & lo, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & lo]
        k0, k1 = (k0 + np.uint64(_W0)) & lo, (k1 + np.uint64(_W1)) & lo
    return [x.astype(np.uint32) for x in c]


def keep_threshold(p: float) -> int:
    p32 = float(np.float32(p))
    return min(2 ** 32 - 1, int(np.floor(p32 * 2.0 ** 32)))


def keep_scale(p: float) -> torch.Tensor:
    one = torch.tensor(1.0, dtype=torch.float32)
    return one / (one - torch.tensor(p, dtype=torch.float32))


def keep_mask(n: int, p: float, site: int, layer: int, step: int, rank: int, seed: int) -> np.ndarray:
    """bool [n]: which of the first n elements of a site are kept."""
    calls = (n + 3) // 4
    words = philox4x32((np.arange(calls, dtype=np.uint64), site + 16 * layer, step, rank),
                       (seed & _MASK, (seed >> 32) & _MASK))
    u = np.stack(words, axis=1).reshape(-1)[:n]
    return u >= np.uint32(keep_threshold(p))


class Dropout:
    """The masks of one forward pass (``step``): ``drop(x, site, layer)`` -> x * M * s over x's logical layout."""

    def __init__(self, p: float, p_ffn: float = 0.1, seed: int = 0, rank: int = 0, step: int = 0):
        self.p, self.p_ffn, self.seed, self.rank, self.step = p, p_ffn, seed, rank, step

    def __call__(self, x: torch.Tensor, site: int, layer: int = 0) -> torch.Tensor:
        p = self.p_ffn if site in FFN_SITES else self.p
        keep = keep_mask(x.numel(), p, site, layer, self.step, self.rank, self.seed)
        # the mask in x's own strides, so that the result keeps x's memory layout (and autograd its summation order)
        keep = torch.empty_like(x, dtype=torch.bool).copy_(torch.from_numpy(keep).view(x.shape))
        return torch.where(keep, x * keep_scale(p), torch.zeros((), dtype=x.dtype))


# ---------------------------------------------------------------------------------------------------------------------
# the training oracle's forward pass with the masks (oracle/satrn.py + oracle/train.py, dropout added at each site)
# ---------------------------------------------------------------------------------------------------------------------
def _mha(sd, p, q_in, k_in, v_in, heads, mask, drop, site, layer):
    """satrn.mha with dropout on the attention probabilities (site) and on the output (site + 1)."""
    W = lambda n: sd[p + n].to(q_in.dtype)
    b, ql, kl = q_in.size(0), q_in.size(1), k_in.size(1)
    d = sd[p + ".q_linear.weight"].shape[0]
    hd = d // heads
    q = F.linear(q_in, W(".q_linear.weight"), W(".q_linear.bias")).view(b, ql, heads, hd).transpose(1, 2)
    k = F.linear(k_in, W(".k_linear.weight"), W(".k_linear.bias")).view(b, kl, heads, hd).transpose(1, 2)
    v = F.linear(v_in, W(".v_linear.weight"), W(".v_linear.bias")).view(b, kl, heads, hd).transpose(1, 2)
    attn = torch.matmul(q, k.transpose(2, 3)) / (float(d) ** 0.5)
    if mask is not None:
        attn = attn.masked_fill(mask.unsqueeze(1), float("-inf"))
    attn = drop(torch.softmax(attn, dim=-1), site, layer)
    out = torch.matmul(attn, v).transpose(1, 2).contiguous().view(b, ql, d)
    return drop(F.linear(out, W(".out_linear.weight"), W(".out_linear.bias")), site + 1, layer)


def _encoder_layer(sd, spec, i, x, calib, drop):
    """satrn.encoder_layer_forward with dropout in its attention (sites 1 / 2)."""
    p = "encoder.attention_layers.%d." % i
    W = lambda n: sd[p + n].to(x.dtype)
    b, c, h, w = x.shape
    flat = x.view(b, c, h * w).transpose(1, 2)
    y = F.layer_norm(flat, (c,), W("norm.weight"), W("norm.bias"), 1e-5)
    y = _mha(sd, p + "attention_layer", y, y, y, spec.enc_heads, None, drop, 1, i)
    y = F.layer_norm(y + flat, (c,), W("norm.weight"), W("norm.bias"), 1e-5)
    y = y.reshape(-1, c, h, w)
    y = F.relu(satrn._bn(F.conv2d(y, W("conv0.weight")), sd, p + "norm0", 1e-5, calib))
    y = F.conv2d(y, W("depthwise.weight"), W("depthwise.bias"), 1, 1, 1, y.shape[1])
    y = F.relu(satrn._bn(y, sd, p + "depthwise_norm", 1e-5, calib))
    y = F.relu(satrn._bn(F.conv2d(y, W("conv1.weight")), sd, p + "norm1", 1e-5, calib))
    return y + x


def _decoder_layer(sd, spec, i, tgt, src, tgt_mask, drop):
    """satrn.decoder_layer_as_written (teacher forcing) with dropout at sites 4-9."""
    p = "decoder.attention_layers.%d." % i
    att = _mha(sd, p + "self_attention_layer", tgt, tgt, tgt, spec.dec_heads, tgt_mask, drop, 4, i)
    out = satrn._ln(sd, p + "self_attention_norm", att + tgt)
    att = _mha(sd, p + "attention_layer", out, src, src, spec.dec_heads, None, drop, 6, i)
    out = satrn._ln(sd, p + "attention_norm", att + out)
    f = p + "feedforward_layer"
    ff = drop(F.relu(F.linear(out, sd[f + ".linear0.weight"], sd[f + ".linear0.bias"])), 8, i)
    ff = drop(F.relu(F.linear(ff, sd[f + ".linear1.weight"], sd[f + ".linear1.bias"])), 9, i)
    return satrn._ln(sd, p + "feedforward_norm", ff + out)


def train_forward(sd, spec, images, expected, drop: Dropout, momentum: float = 0.1):
    """oracle.train.train_forward with the masks of one forward pass -> logits [B, L, V]."""
    mode = satrn.TrainMode(momentum)
    x = drop(satrn.pe2d_forward(sd, spec, satrn.trunk_forward(sd, spec, images, mode)), 0)
    for i in range(spec.enc_layers):
        x = _encoder_layer(sd, spec, i, x, mode, drop)
    b, c, h, w = x.shape
    src = x.view(b, c, h * w).transpose(1, 2).contiguous()
    text = expected[:, :-1]                                    # satrn.teacher_forced
    L = text.size(1)
    tgt = drop(satrn._embed(sd, text) + satrn.pe1d_table(spec.dec_hidden, spec.pe1d_len)[:L].unsqueeze(0), 3)
    pad = text == satrn.PAD_ID
    pad[:, 0] = False
    mask = pad.unsqueeze(1) | torch.triu(torch.ones(L, L), diagonal=1).bool().unsqueeze(0)
    for l in range(spec.dec_layers):
        tgt = _decoder_layer(sd, spec, l, tgt, src, mask, drop)
    return F.linear(tgt, sd["decoder.generator.weight"], sd["decoder.generator.bias"])


class Trainer(train.Trainer):
    """oracle.train.Trainer with dropout (p, p_ffn, seed, rank); step = the forward passes it has run."""

    def __init__(self, sd, spec, p, p_ffn=0.1, seed=0, rank=0, **kw):
        super().__init__(sd, spec, **kw)
        self.drop_args, self.passes = (p, p_ffn, seed, rank), 0

    def forward_backward(self, images, expected):
        p, p_ffn, seed, rank = self.drop_args
        drop = Dropout(p, p_ffn, seed, rank, self.passes)
        self.passes += 1
        self.opt.zero_grad()
        with torch.enable_grad():
            loss = train.loss_fn(train_forward(self.sd, self.spec, images, expected, drop), expected)
            loss.backward()
        return loss.item(), {k: v.grad for k, v in self.sd.items() if train.is_param(k)}
