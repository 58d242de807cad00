"""state_dict layout of the networks this package serves -- the checkpoint
contract (SURVEY.md 8b / App. A.2).  ``build_param_tree`` creates an
``nn.Module`` tree whose ``state_dict()`` has exactly the reference's keys,
shapes and dtypes, so reference checkpoints load with ``strict=True`` and
checkpoints saved from this package load into the reference.

Module definitions mirrored (names only, no arithmetic):
networks/EfficientSATRN.py:63-79 (EfficientNet), :90-109 (PositionalEncoding),
:231-257 (EncoderLayer), :175-196 (MultiHeadAttention), :326-337 (Feedforward),
:349-372 (TransformerDecoderLayer), :429-461 (SATRNDecoder); timm 0.4.9
``tf_efficientnetv2_s`` ``.blocks`` (requirements.txt:15, SURVEY App. A.1).
"""
import collections

import torch
import torch.nn as nn

# (block kind, repeats, kernel, stride, expand, out channels, SE ratio)
EFFNETV2_S = (
    ("cn", 2, 3, 1, 1, 24, 0.0),
    ("er", 4, 3, 2, 4, 48, 0.0),
    ("er", 4, 3, 2, 4, 64, 0.0),
    ("ir", 6, 3, 2, 4, 128, 0.25),
    ("ir", 9, 3, 1, 6, 160, 0.25),
    ("ir", 15, 3, 2, 6, 256, 0.25),
)

BUFFER_LEAVES = ("running_mean", "running_var", "num_batches_tracked")


def _bn(s, p, c):
    s[p + ".weight"] = (c,)
    s[p + ".bias"] = (c,)
    s[p + ".running_mean"] = (c,)
    s[p + ".running_var"] = (c,)
    s[p + ".num_batches_tracked"] = ()


def _mha(s, p, q_ch, k_ch, d):
    for name, cin in (("q_linear", q_ch), ("k_linear", k_ch), ("v_linear", k_ch)):
        s["%s.%s.weight" % (p, name)] = (d, cin)
        s["%s.%s.bias" % (p, name)] = (d,)
    s[p + ".out_linear.weight"] = (q_ch, d)
    s[p + ".out_linear.bias"] = (q_ch,)


def _satrn_encoder_tail(s, dims, prefix):
    hidden, filt = dims["enc_hidden"], dims["enc_filter"]
    pe = prefix + "positional_encoding."
    s[pe + "dense0.weight"] = (hidden // 2, hidden)
    s[pe + "dense0.bias"] = (hidden // 2,)
    s[pe + "dense1.weight"] = (hidden * 2, hidden // 2)
    s[pe + "dense1.bias"] = (hidden * 2,)
    for i in range(dims["enc_layers"]):
        p = "%sattention_layers.%d." % (prefix, i)
        s[p + "norm.weight"] = (hidden,)
        s[p + "norm.bias"] = (hidden,)
        _mha(s, p + "attention_layer", hidden, hidden, hidden)
        s[p + "conv0.weight"] = (filt, hidden, 1, 1)
        _bn(s, p + "norm0", filt)
        s[p + "depthwise.weight"] = (filt, 1, 3, 3)
        s[p + "depthwise.bias"] = (filt,)
        _bn(s, p + "depthwise_norm", filt)
        s[p + "conv1.weight"] = (hidden, filt, 1, 1)
        _bn(s, p + "norm1", hidden)


def lite_encoder_shapes(dims, prefix="encoder."):
    """LiteSATRN: ShallowCNN of 4 x (conv3x3 p1, BN, ReLU, maxpool2) (networks/LiteSATRN.py:21-70)
    + the same positional encoding / encoder layers (:266-304)."""
    s = collections.OrderedDict()
    cnn = prefix + "shallow_cnn."
    h = dims["enc_hidden"]
    for i, (ci, co) in enumerate(((dims["in_ch"], h // 2), (h // 2, h), (h, h), (h, h))):
        s["%sconv%d.weight" % (cnn, i)] = (co, ci, 3, 3)
        _bn(s, "%sbatch_norm%d" % (cnn, i), co)
    _satrn_encoder_tail(s, dims, prefix)
    return s


def encoder_shapes(dims, prefix="encoder."):
    s = collections.OrderedDict()
    cnn = prefix + "shallow_cnn."
    hidden, filt = dims["enc_hidden"], dims["enc_filter"]
    s[cnn + "conv_stem.weight"] = (24, dims["in_ch"], 3, 3)
    _bn(s, cnn + "bn1", 24)
    cin = 24
    for si, (kind, reps, k, stride, expand, cout, se) in enumerate(EFFNETV2_S):
        for r in range(reps):
            p = "%seff_block.%d.%d" % (cnn, si, r)
            mid = cin * expand
            if kind == "cn":
                s[p + ".conv.weight"] = (cout, cin, k, k)
                _bn(s, p + ".bn1", cout)
            elif kind == "er":
                s[p + ".conv_exp.weight"] = (mid, cin, k, k)
                _bn(s, p + ".bn1", mid)
                s[p + ".conv_pwl.weight"] = (cout, mid, 1, 1)
                _bn(s, p + ".bn2", cout)
            else:
                red = int(cin * se)
                s[p + ".conv_pw.weight"] = (mid, cin, 1, 1)
                _bn(s, p + ".bn1", mid)
                s[p + ".conv_dw.weight"] = (mid, 1, k, k)
                _bn(s, p + ".bn2", mid)
                s[p + ".se.conv_reduce.weight"] = (red, mid, 1, 1)
                s[p + ".se.conv_reduce.bias"] = (red,)
                s[p + ".se.conv_expand.weight"] = (mid, red, 1, 1)
                s[p + ".se.conv_expand.bias"] = (mid,)
                s[p + ".conv_pwl.weight"] = (cout, mid, 1, 1)
                _bn(s, p + ".bn3", cout)
            cin = cout
    s[cnn + "conv_last.weight"] = (hidden, 256, 1, 1)
    _bn(s, cnn + "bn2", hidden)
    pe = prefix + "positional_encoding."
    s[pe + "dense0.weight"] = (hidden // 2, hidden)
    s[pe + "dense0.bias"] = (hidden // 2,)
    s[pe + "dense1.weight"] = (hidden * 2, hidden // 2)
    s[pe + "dense1.bias"] = (hidden * 2,)
    for i in range(dims["enc_layers"]):
        p = "%sattention_layers.%d." % (prefix, i)
        s[p + "norm.weight"] = (hidden,)
        s[p + "norm.bias"] = (hidden,)
        _mha(s, p + "attention_layer", hidden, hidden, hidden)
        s[p + "conv0.weight"] = (filt, hidden, 1, 1)
        _bn(s, p + "norm0", filt)
        s[p + "depthwise.weight"] = (filt, 1, 3, 3)
        s[p + "depthwise.bias"] = (filt,)
        _bn(s, p + "depthwise_norm", filt)
        s[p + "conv1.weight"] = (hidden, filt, 1, 1)
        _bn(s, p + "norm1", hidden)
    return s


def decoder_shapes(dims, prefix="decoder."):
    s = collections.OrderedDict()
    d, f, src, v = dims["dec_hidden"], dims["dec_filter"], dims["dec_src"], dims["num_classes"]
    s[prefix + "embedding.weight"] = (v + 1, d)
    for i in range(dims["dec_layers"]):
        p = "%sattention_layers.%d." % (prefix, i)
        _mha(s, p + "self_attention_layer", d, d, d)
        s[p + "self_attention_norm.weight"] = (d,)
        s[p + "self_attention_norm.bias"] = (d,)
        _mha(s, p + "attention_layer", d, src, d)
        s[p + "attention_norm.weight"] = (d,)
        s[p + "attention_norm.bias"] = (d,)
        s[p + "feedforward_layer.linear0.weight"] = (f, d)
        s[p + "feedforward_layer.linear0.bias"] = (f,)
        s[p + "feedforward_layer.linear1.weight"] = (d, f)
        s[p + "feedforward_layer.linear1.bias"] = (d,)
        s[p + "feedforward_norm.weight"] = (d,)
        s[p + "feedforward_norm.bias"] = (d,)
    s[prefix + "generator.weight"] = (v, d)
    s[prefix + "generator.bias"] = (v,)
    return s


# SwinTRN encoder is hard-wired in the reference (networks/SWIN.py:1028-1031): Swin-B/384
SWIN_IMG, SWIN_PATCH, SWIN_EMBED, SWIN_WINDOW = 384, 4, 128, 12
SWIN_DEPTHS, SWIN_HEADS, SWIN_HEAD_CLASSES = (2, 2, 18, 2), (4, 8, 16, 32), 21841


def swin_relative_position_index(ws):
    """networks/SWIN.py:116-135"""
    coords = torch.stack(torch.meshgrid([torch.arange(ws), torch.arange(ws)], indexing="ij"))
    cf = torch.flatten(coords, 1)
    rel = (cf[:, :, None] - cf[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += ws - 1
    rel[:, :, 1] += ws - 1
    rel[:, :, 0] *= 2 * ws - 1
    return rel.sum(-1)


def swin_attn_mask(res, ws, shift):
    """networks/SWIN.py:286-310"""
    img = torch.zeros((1, res, res, 1))
    cnt = 0
    for h in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
        for w in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
            img[:, h, w, :] = cnt
            cnt += 1
    mw = img.view(1, res // ws, ws, res // ws, ws, 1).permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, ws * ws)
    m = mw.unsqueeze(1) - mw.unsqueeze(2)
    return m.masked_fill(m != 0, float(-100.0)).masked_fill(m == 0, float(0.0))


def swin_encoder_entries(prefix="encoder."):
    """(name, shape, kind) in the reference's registration order; kind in {"param", "rel_index", "attn_mask"}."""
    out = []
    e = prefix
    r0 = SWIN_IMG // SWIN_PATCH
    out.append((e + "absolute_pos_embed", (1, r0 * r0, SWIN_EMBED), "param"))
    out.append((e + "patch_embed.proj.weight", (SWIN_EMBED, 3, SWIN_PATCH, SWIN_PATCH), "param"))
    out.append((e + "patch_embed.proj.bias", (SWIN_EMBED,), "param"))
    out.append((e + "patch_embed.norm.weight", (SWIN_EMBED,), "param"))
    out.append((e + "patch_embed.norm.bias", (SWIN_EMBED,), "param"))
    for i, (depth, heads) in enumerate(zip(SWIN_DEPTHS, SWIN_HEADS)):
        dim, res = SWIN_EMBED * 2 ** i, r0 // 2 ** i
        for j in range(depth):
            ws, shift = SWIN_WINDOW, (0 if j % 2 == 0 else SWIN_WINDOW // 2)
            if res <= ws:
                ws, shift = res, 0
            p = "%slayers.%d.blocks.%d." % (e, i, j)
            if shift > 0:
                out.append((p + "attn_mask", (res, ws, shift), "attn_mask"))
            for n, s in (("norm1.weight", (dim,)), ("norm1.bias", (dim,)),
                         ("attn.relative_position_bias_table", ((2 * ws - 1) ** 2, heads))):
                out.append((p + n, s, "param"))
            out.append((p + "attn.relative_position_index", (ws,), "rel_index"))
            for n, s in (("attn.qkv.weight", (3 * dim, dim)), ("attn.qkv.bias", (3 * dim,)),
                         ("attn.proj.weight", (dim, dim)), ("attn.proj.bias", (dim,)),
                         ("norm2.weight", (dim,)), ("norm2.bias", (dim,)),
                         ("mlp.fc1.weight", (4 * dim, dim)), ("mlp.fc1.bias", (4 * dim,)),
                         ("mlp.fc2.weight", (dim, 4 * dim)), ("mlp.fc2.bias", (dim,))):
                out.append((p + n, s, "param"))
        if i < len(SWIN_DEPTHS) - 1:
            p = "%slayers.%d.downsample." % (e, i)
            out.append((p + "reduction.weight", (2 * dim, 4 * dim), "param"))
            out.append((p + "norm.weight", (4 * dim,), "param"))
            out.append((p + "norm.bias", (4 * dim,), "param"))
    out.append((e + "norm.weight", (SWIN_EMBED * 8,), "param"))
    out.append((e + "norm.bias", (SWIN_EMBED * 8,), "param"))
    out.append((e + "head.weight", (SWIN_HEAD_CLASSES, SWIN_EMBED * 8), "param"))
    out.append((e + "head.bias", (SWIN_HEAD_CLASSES,), "param"))
    return out


def build_swin_encoder_tree():
    tree = ParamTree()
    for name, shape, kind in swin_encoder_entries():
        short = name[len("encoder."):]
        if kind == "rel_index":
            tree.add(short, swin_relative_position_index(shape[0]), True)
        elif kind == "attn_mask":
            tree.add(short, swin_attn_mask(*shape), True)
        else:
            tree.add(short, _init_tensor(name, shape), False)
    return tree


def swin_decoder_shapes(dims, prefix="decoder."):
    """SWIN's Feedforward is an nn.Sequential (networks/SWIN.py:827-841): layers.0 / layers.3."""
    s = collections.OrderedDict()
    for k, v in decoder_shapes(dims, prefix).items():
        s[k.replace("feedforward_layer.linear0", "feedforward_layer.layers.0")
           .replace("feedforward_layer.linear1", "feedforward_layer.layers.3")] = v
    return s


def dims_from_flags(FLAGS, num_classes):
    """The fields the constructors read (networks/EfficientSATRN.py:667-688)."""
    enc, dec = FLAGS.SATRN.encoder, FLAGS.SATRN.decoder
    return dict(
        height=FLAGS.input_size.height, width=FLAGS.input_size.width, in_ch=FLAGS.data.rgb,
        enc_hidden=enc.hidden_dim, enc_filter=enc.filter_dim, enc_layers=enc.layer_num, enc_heads=enc.head_num,
        dec_src=dec.src_dim, dec_hidden=dec.hidden_dim, dec_filter=dec.filter_dim,
        dec_layers=dec.layer_num, dec_heads=dec.head_num, num_classes=num_classes)


def dropout_rate_from_flags(FLAGS):
    """FLAGS.dropout_rate (configs/*.yaml), the rate the reference hands its encoder and decoder; 0 when the flags carry
    none."""
    return float(getattr(FLAGS, "dropout_rate", 0.0) or 0.0)


class ParamTree(nn.Module):
    """A module that only holds parameters/buffers under reference names."""

    def add(self, dotted, tensor, is_buffer):
        head, _, rest = dotted.partition(".")
        if rest:
            if head not in self._modules:
                self.add_module(head, ParamTree())
            self._modules[head].add(rest, tensor, is_buffer)
        elif is_buffer:
            self.register_buffer(head, tensor)
        else:
            self.register_parameter(head, nn.Parameter(tensor))

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("ParamTree holds weights only; compute runs in libfrx.so")


def _init_tensor(name, shape):
    leaf = name.rsplit(".", 1)[-1]
    if leaf == "num_batches_tracked":
        return torch.zeros((), dtype=torch.long)
    if leaf == "running_mean":
        return torch.zeros(shape)
    if leaf == "running_var":
        return torch.ones(shape)
    is_norm = any(t in name for t in (".bn", "norm"))
    if is_norm:
        return torch.ones(shape) if leaf == "weight" else torch.zeros(shape)
    if leaf == "bias":
        return torch.zeros(shape)
    t = torch.empty(shape)
    if name.endswith("embedding.weight"):
        return nn.init.normal_(t)
    if t.dim() >= 2:
        return nn.init.xavier_normal_(t)  # :193-196,:255-257,:336-337
    return t.zero_()


def build_param_tree(shapes, strip_prefix):
    tree = ParamTree()
    for name, shape in shapes.items():
        assert name.startswith(strip_prefix)
        leaf = name.rsplit(".", 1)[-1]
        tree.add(name[len(strip_prefix):], _init_tensor(name, shape), leaf in BUFFER_LEAVES)
    return tree
