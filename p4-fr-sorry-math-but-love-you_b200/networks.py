"""Drop-in ``nn.Module`` front-ends for the reference's ``networks/`` constructors.

Same constructor signatures, attribute tree, ``state_dict`` layout and method
contracts as /root/reference/networks/EfficientSATRN.py:664-952; the arithmetic
runs in ``lib/libfrx.so`` through the C ABI of include/frx.h.  PyTorch is only
the plumbing here (parameter storage, device memory, the CUDA stream).
"""
import ctypes
import math
import random

import torch
import torch.nn as nn

from . import _lib, layout, sharding

START, END, PAD = "<SOS>", "<EOS>", "<PAD>"  # data/dataset.py:12-14

_PRECISIONS = {"fp32": 0, "bf16": 1}


def pe2d_table(length, hidden):
    """Host-built 2-D positional table, computed exactly like
    PositionalEncoding.get_position_encoding (EfficientSATRN.py:111-127):
    fp32 torch ops on the CPU, sin||cos concatenated."""
    position = torch.arange(length).float()
    n_ts = hidden // 2
    log_inc = math.log(1.0e4 / 1.0) / (torch.FloatTensor([n_ts]) - 1)
    inv = 1.0 * torch.exp(torch.arange(n_ts) * -log_inc)
    scaled = position.unsqueeze(1) * inv.unsqueeze(0)
    return torch.cat((torch.sin(scaled), torch.cos(scaled)), dim=1).contiguous()


def pe1d_table(channels, max_len=500):
    """PositionEncoder1D.generate_encoder (EfficientSATRN.py:408-418)."""
    pos = torch.arange(max_len).float().unsqueeze(1)
    i = torch.arange(channels).float().unsqueeze(0)
    table = pos * (1 / torch.pow(10000, (2 * (i // 2)) / channels))
    table[:, 0::2] = torch.sin(table[:, 0::2])
    table[:, 1::2] = torch.cos(table[:, 1::2])
    return table.contiguous()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p()


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class _TrainForward(torch.autograd.Function):
    """EfficientSATRN.forward under model.train(): the library's train-mode forward as an autograd node, so that the
    reference's own loop -- ``loss = criterion(output.transpose(1, 2), expected[:, 1:]); loss.backward()``
    (train_modules/train_single_opt.py:79-92) -- drives the library's backward pass.  ``anchor`` is any parameter that
    requires grad (autograd only runs nodes with a differentiable input); the parameter gradients are written to
    ``.grad`` directly (accumulating, like autograd)."""

    @staticmethod
    def forward(ctx, module, x, expected, anchor):
        ctx.module, ctx.x, ctx.e = module, x, expected
        return module._train_forward(x, expected)

    @staticmethod
    def backward(ctx, grad_logits):
        ctx.module._train_backward(ctx.x, ctx.e, grad_logits.contiguous().float())
        return None, None, None, None


class _Engine:
    """One frx handle bound to (device, max_batch, max_steps, precision)."""

    def __init__(self, dims, ids, device, max_batch, max_steps, precision, parts, network=0):
        cfg = _lib.FrxConfig()
        cfg.network = network
        self.network = network
        self.down = 16 if network == 1 else 32
        for k in ("height", "width", "in_ch", "enc_hidden", "enc_filter", "enc_layers", "enc_heads",
                  "dec_src", "dec_hidden", "dec_filter", "dec_layers", "dec_heads", "num_classes"):
            setattr(cfg, k, int(dims[k]))
        cfg.sos_id, cfg.eos_id, cfg.pad_id = ids
        cfg.max_batch, cfg.max_steps = int(max_batch), int(max_steps)
        cfg.precision = _PRECISIONS[precision]
        cfg.device = device.index if device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", cfg.device)
        self.max_batch, self.max_steps, self.precision = int(max_batch), int(max_steps), precision
        self.dims = dims
        self.h = _lib.Handle(cfg)
        self.h.call("frx_set_option", b"parts", parts)

    def load(self, state_dict):
        def put(name, t):
            if t.dtype == torch.int64:
                t, dt = t.detach().contiguous(), 1
            else:
                t, dt = t.detach().float().contiguous(), 0
            shape = (ctypes.c_int64 * max(t.dim(), 1))(*t.shape)
            self.h.call("frx_load_tensor", name.encode(), _ptr(t), shape, t.dim(), dt)

        skip = ("num_batches_tracked", "relative_position_index", "attn_mask")  # derived constants, recomputed in-kernel
        for name, t in state_dict.items():
            if name.endswith(skip) or name.startswith("encoder.head."):  # Swin's classification head is never used
                continue
            # SWIN names its FFN linears layers.0 / layers.3 (networks/SWIN.py:831-838); the C side uses one naming
            put(name.replace("feedforward_layer.layers.0", "feedforward_layer.linear0")
                    .replace("feedforward_layer.layers.3", "feedforward_layer.linear1"), t)
        d = self.dims
        if self.network != 2:
            put("pe2d.h", pe2d_table(d["height"] // self.down, d["enc_hidden"]))
            put("pe2d.w", pe2d_table(d["width"] // self.down, d["enc_hidden"]))
        put("pe1d", pe1d_table(d["dec_hidden"]))
        self.h.call("frx_finalize_weights")

    def option(self, key, value):
        self.h.call("frx_set_option", key.encode(), int(value))

    @property
    def launches(self):
        return int(self.h.lib.frx_launch_count(self.h.ptr))

    @property
    def device_bytes(self):
        return int(self.h.lib.frx_device_bytes(self.h.ptr))


class _FrxModule(nn.Module):
    """Shared engine management (lazy creation, weight re-sync when dirty)."""

    _parts = 3  # bit0 encoder, bit1 decoder
    _network = 0  # FRX_NET_EFFICIENT_SATRN
    _down = 32

    def _setup(self, FLAGS, train_dataset, precision, max_batch, max_steps):
        self._dims = layout.dims_from_flags(FLAGS, len(train_dataset.id_to_token))
        self._flags_dropout = layout.dropout_rate_from_flags(FLAGS)
        self._train_dropout = None   # (p, p_ffn, seed) of set_train_dropout
        t2i = train_dataset.token_to_id
        self._ids = (int(t2i[START]), int(t2i.get(END, 1)), int(t2i[PAD]))
        self._precision = precision
        self._max_batch = max_batch
        self._max_steps = max_steps
        self._engine = None
        self._dirty = True
        self._options = {}

    # --- keep the device copy of the weights coherent with the nn.Parameters ---
    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self._dirty = True
        return out

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._dirty = True
        return out

    def refresh(self):
        """Call after mutating parameters in place (e.g. an optimizer step)."""
        self._dirty = True

    def set_option(self, key, value):
        self._options[key] = int(value)
        if self._engine is not None:
            self._engine.option(key, value)

    def engine(self, device, batch, steps):
        if device.type != "cuda":
            raise RuntimeError("frx runs on a CUDA device (B200) only; there is no CPU fallback "
                               "(input is on %s)" % device)
        e = self._engine
        need_b = max(batch, self._max_batch or 0)
        need_t = max(steps, self._max_steps or 0)
        if e is None or e.device != torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device()) \
                or e.max_batch < batch or e.max_steps < steps:
            if e is not None:
                need_b, need_t = max(need_b, e.max_batch), max(need_t, e.max_steps)
                e.h.close()
            e = _Engine(self._dims, self._ids, device, need_b, need_t, self._precision, self._parts, self._network)
            for k, v in self._options.items():
                e.option(k, v)
            self._engine = e
            self._dirty = True
        if self._dirty:
            e.load(self.state_dict())
            self._dirty = False
        return e


class EfficientSATRN(_FrxModule):
    """networks/EfficientSATRN.py:664-867.

    Extra keyword-only arguments (not in the reference): ``precision``
    ("fp32" | "bf16"), ``max_batch`` / ``max_steps`` to pre-size the workspaces
    (they grow on demand otherwise)."""

    def __init__(self, FLAGS, train_dataset, checkpoint=None, decoding_manager=None, *,
                 precision="fp32", max_batch=None, max_steps=None):
        super().__init__()
        self._setup(FLAGS, train_dataset, precision, max_batch, max_steps)
        self.encoder = layout.build_param_tree(layout.encoder_shapes(self._dims), "encoder.")
        self.decoder = layout.build_param_tree(layout.decoder_shapes(self._dims), "decoder.")
        d = self.decoder
        d.hidden_dim, d.filter_dim = self._dims["dec_hidden"], self._dims["dec_filter"]
        d.num_classes, d.layer_num = self._dims["num_classes"], self._dims["dec_layers"]
        d.pad_id, d.st_id = self._ids[2], self._ids[0]
        d.manager = decoding_manager
        self.criterion = nn.CrossEntropyLoss(ignore_index=self._ids[2])
        if checkpoint:
            self.load_state_dict(checkpoint)

    def _attach_manager(self, eng):
        """Upload the DecodingManager's rule tables (postprocessing/postprocessing.py:182-405) once per engine."""
        if getattr(eng, "_rules_of", None) is not self.decoder.manager:
            from .decoding import compile_decoding_rules
            flags, limit, ids6 = compile_decoding_rules(self.decoder.manager)
            n = len(flags)
            eng.h.call("frx_set_decoding_rules", (ctypes.c_int32 * n)(*flags), (ctypes.c_int32 * n)(*limit), n,
                       (ctypes.c_int32 * 6)(*ids6))
            eng._rules_of = self.decoder.manager

    def forward(self, input, expected, is_train, teacher_forcing_ratio):
        """:697-706 -> logits [B, expected.size(1)-1, num_classes] fp32 on input's device."""
        if self.training:
            # model.train(): BatchNorm batch statistics (and running-statistics updates) like the reference's modules.  The
            # teacher-forced branch (:488-495) is the one the training loop takes (teacher_forcing_ratio 1.0); it returns
            # logits that carry a grad_fn, so criterion(...).backward() fills every parameter's .grad (compatibility path:
            # parameters / gradients cross the host; EfficientSATRN.train_step is the fused fast path).  Dropout: off
            # unless set_train_dropout enabled it.
            if not (is_train and random.random() < teacher_forcing_ratio):
                raise NotImplementedError("train mode runs the teacher-forced branch only (teacher_forcing_ratio 1.0, "
                                          "configs/EfficientSATRN.yaml); call .eval() for greedy decoding")
            x = input.detach().float().contiguous()
            e = expected.to(device=x.device, dtype=torch.int64).contiguous()
            anchor = next(p for p in self.parameters() if p.requires_grad)
            return _TrainForward.apply(self, x, e, anchor)
        b, steps = input.size(0), expected.size(1) - 1
        eng = self.engine(input.device, b, steps)
        x = input.detach().float().contiguous()
        v = self._dims["num_classes"]
        if is_train and random.random() < teacher_forcing_ratio:  # :488-495 (consumes the RNG like the reference)
            text = expected[:, :-1].to(device=x.device, dtype=torch.int64).contiguous()
            memory = torch.empty(b, self.memory_tokens, self._dims["enc_hidden"], device=x.device)
            logits = torch.empty(b, steps, v, device=x.device)
            st = _stream(x.device)
            eng.h.call("frx_encode", _ptr(x), b, _ptr(memory), st)
            eng.h.call("frx_decode_teacher_forced", _ptr(memory), _ptr(text), b, steps, _ptr(logits), st)
            return logits
        logits = torch.empty(b, steps, v, device=x.device)
        # :536-564: with a manager every row is its masked softmax, not logits -- inference branch only; the is_train
        # branch that lost the teacher-forcing draw (:496-525) never consults the manager and returns raw greedy logits
        if not is_train and self.decoder.manager is not None:
            self._attach_manager(eng)
            eng.h.call("frx_forward_greedy_managed", _ptr(x), b, steps, _ptr(logits), None, _stream(x.device))
            return logits
        eng.h.call("frx_forward_greedy", _ptr(x), b, steps, _ptr(logits), None, _stream(x.device))
        return logits

    # ------------------------------------------------------------------------------------------------------------
    # training step (train_modules/train_single_opt.py:72-112)
    # ------------------------------------------------------------------------------------------------------------
    def _trainer(self, device, batch, length):
        """Lazily create the library's training state (parameters, gradients, Adam moments, activation tape)."""
        eng = self.engine(device, batch, max(length, 1))
        tr = getattr(eng, "_train", None)
        if tr is None or tr["max_batch"] < batch or tr["max_len"] < length:
            if tr is not None:
                raise RuntimeError("training state was sized for batch %d / length %d; create the model with larger "
                                   "max_batch / max_steps" % (tr["max_batch"], tr["max_len"]))
            mb, ml = max(batch, self._max_batch or 0), max(length, min(self._max_steps or 0, 256))
            n = int(eng.h.lib.frx_train_param_count(eng.h.ptr))
            if n <= 0:
                raise RuntimeError("frx_train_param_count: " + eng.h.lib.frx_last_error(eng.h.ptr).decode())
            grads = torch.zeros(n, dtype=torch.float32, device=eng.device)   # flat gradient buffer, all-reduced over NCCL
            eng.h.call("frx_train_create", mb, ml, _ptr(grads))
            tr = eng._train = {"max_batch": mb, "max_len": ml, "grads": grads, "works": [],
                               "scalars": torch.zeros(4, dtype=torch.float32, device=eng.device)}
            self._apply_train_dropout(eng)
        return eng, tr

    def set_train_dropout(self, p=None, seed=0, p_ffn=0.1):
        """Train with the reference's dropout (off by default): rate ``p`` (None: FLAGS.dropout_rate) at the 2-D PE
        output, the attention probabilities and MHA outputs of every encoder / decoder layer and the decoder input;
        ``p_ffn`` after each decoder feed-forward ReLU (the reference builds Feedforward with its default 0.1 whatever the
        flag says, EfficientSATRN.py:327, :368-370).  The masks are counter-based (Philox4x32-10 keyed by ``seed``,
        include/frx.h frx_train_set_dropout), so a run is reproducible; under torch.distributed each rank draws its own.
        They are not torch's masks.  ``set_train_dropout(0, p_ffn=0)`` turns dropout off again.  Applies to train_step
        and to the train-mode forward; inference never drops."""
        p = self._flags_dropout if p is None else float(p)
        p_ffn = float(p_ffn)
        for name, r in (("p", p), ("p_ffn", p_ffn)):
            if not 0.0 <= r < 1.0:
                raise ValueError("set_train_dropout: %s = %r outside [0, 1)" % (name, r))
        seed = int(seed)
        if not 0 <= seed < 1 << 64:
            raise ValueError("set_train_dropout: seed must fit in 64 unsigned bits")
        self._train_dropout = (p, p_ffn, seed)
        eng = self._engine
        if eng is not None and getattr(eng, "_train", None) is not None:
            self._apply_train_dropout(eng)

    def _apply_train_dropout(self, eng):
        if self._train_dropout is None:
            return
        import torch.distributed as dist
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        p, p_ffn, seed = self._train_dropout
        eng.h.call("frx_train_set_dropout", p, p_ffn, seed, rank)

    def train_step(self, input, expected, lr=5e-4, weight_decay=1e-6, max_grad_norm=2.0, process_group=None,
                   overlap=False, enc_lr=None, dec_lr=None):
        """One iteration of the reference's single-optimizer loop (train_single_opt.py:72-112) with teacher forcing 1.0:
        train-mode forward (BatchNorm batch statistics), CrossEntropyLoss(ignore_index=PAD), backward,
        clip_grad_norm_(max_grad_norm), AdamW(lr, weight_decay) -- all inside the library, fp32.  Returns
        (loss, grad_norm) as 0-dim device tensors (no host synchronisation).

        Data parallel: when torch.distributed is initialised (one process per GPU, NCCL) the flat gradient buffer is
        all-reduced (sum, then 1 / world inside the optimiser kernel) before the update; with ``overlap`` each bucket's
        all-reduce starts as soon as the backward pass has produced it (trunk stages last), under the rest of the pass --
        which then runs eagerly instead of as one CUDA graph.  The default is the graph + one all-reduce of the whole
        buffer: on NVLink the 108.9 MB exchange takes 0.23 ms of a 25 ms step, less than the graph saves (2 x B200:
        26.3 vs 29.7 ms per step, profiles/r2_train_dp_2gpu.txt).
        ``expected`` is [B, L + 1] int64 with -1 already replaced by PAD (:77-78).

        ``enc_lr`` / ``dec_lr`` (both given): the dual-optimizer loop (train_modules/train_dual_opt.py:95-112) -- gradient
        clipping and AdamW run separately over the encoder and the decoder parameters; returns
        (loss, enc_grad_norm, dec_grad_norm)."""
        import torch.distributed as dist
        b, lp1 = input.size(0), expected.size(1)
        eng, tr = self._trainer(input.device, b, lp1 - 1)
        x = input.detach().float().contiguous()
        e = expected.to(device=x.device, dtype=torch.int64).contiguous()
        st = _stream(x.device)
        world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        reducer = tr.get("reducer")
        if world > 1 and (reducer is None or reducer.group is not process_group):
            reducer = tr["reducer"] = sharding.GradBucketReducer(tr["grads"], process_group)
        if world > 1 and overlap:
            reducer.begin()
            cb = _lib.BUCKET_CALLBACK(lambda _ctx, off, count: reducer.on_bucket(off, count))
        else:
            cb = _lib.BUCKET_CALLBACK()   # NULL: no callback
        eng.h.call("frx_train_set_bucket_callback", cb, None)
        sc = tr["scalars"]
        eng.h.call("frx_train_fwd_bwd", _ptr(x), _ptr(e), b, lp1, _ptr(sc), st)
        if world > 1:
            if not overlap:
                reducer.begin()
            reducer.finish()      # the current stream waits for the NCCL stream; no host synchronisation
        self._trained, self._train_path = True, "fused"
        if enc_lr is not None and dec_lr is not None:
            eng.h.call("frx_train_apply_dual", float(enc_lr), float(dec_lr), float(weight_decay), float(max_grad_norm), 1.0 / world,
                       ctypes.c_void_p(sc.data_ptr() + 4), ctypes.c_void_p(sc.data_ptr() + 8), st)
            return sc[0], sc[1], sc[2]
        eng.h.call("frx_train_apply", float(lr), float(weight_decay), float(max_grad_norm), 1.0 / world,
                   ctypes.c_void_p(sc.data_ptr() + 4), st)
        return sc[0], sc[1]

    # -- compatibility path: forward / backward as separate calls around the caller's own criterion and optimiser --------
    def _param_signature(self):
        return tuple(p._version for p in self.parameters())

    def _train_forward(self, x, e):
        b, lp1 = x.size(0), e.size(1)
        eng, tr = self._trainer(x.device, b, lp1 - 1)
        sig = self._param_signature()
        if tr.get("sig") is not None and tr["sig"] != sig:
            # an external optimiser stepped the nn.Parameters: push them into the library's training state
            with torch.no_grad():
                for name, p in self.named_parameters():
                    eng.h.call("frx_train_import", name.encode(), _ptr(p.detach().float().contiguous()))
        tr["sig"] = sig
        logits = torch.empty(b, lp1 - 1, self._dims["num_classes"], device=x.device)
        eng.h.call("frx_train_forward", _ptr(x), _ptr(e), b, lp1, _ptr(logits), None, _stream(x.device))
        self._trained, self._train_path = True, "compat"
        self._compat_steps = getattr(self, "_compat_steps", 0) + 1
        return logits

    def _train_backward(self, x, e, grad_logits):
        eng = self._engine
        b, lp1 = x.size(0), e.size(1)
        eng.h.call("frx_train_backward", _ptr(x), _ptr(grad_logits), b, lp1, _stream(x.device))
        with torch.no_grad():
            for name, p in self.named_parameters():
                if not p.requires_grad:
                    continue
                g = torch.empty_like(p, dtype=torch.float32).contiguous()
                eng.h.call("frx_train_read_grad", name.encode(), _ptr(g))
                p.grad = g if p.grad is None else p.grad + g

    def sync_trained_weights(self, buffers_only=None):
        """Copy the library's trained parameters and BatchNorm running statistics back into this module's
        nn.Parameters / buffers (state_dict layout) -- before saving a checkpoint (utils/checkpoint.py:28-32) or
        running inference with the trained weights.  After the compatibility path (forward + loss.backward() + a torch
        optimiser) the nn.Parameters are the master copy, so only the buffers are pulled (``buffers_only`` defaults to
        that case); ``state_dict()`` calls this automatically."""
        eng = self._engine
        if eng is None or getattr(eng, "_train", None) is None:
            return
        if buffers_only is None:
            buffers_only = getattr(self, "_train_path", "fused") == "compat"
        steps = int(eng.h.lib.frx_train_step_count(eng.h.ptr)) if not buffers_only else getattr(self, "_compat_steps", 0)
        params = {n for n, _ in self.named_parameters()}
        self._syncing = True
        try:
            with torch.no_grad():
                for name, t in super().state_dict().items():
                    if name.endswith("num_batches_tracked"):
                        t.fill_(int(t) + steps - getattr(self, "_synced_steps", 0))
                        continue
                    if buffers_only and name in params:
                        continue
                    buf = torch.empty_like(t, dtype=torch.float32).contiguous()
                    eng.h.call("frx_train_export", name.encode(), _ptr(buf))
                    t.copy_(buf)
        finally:
            self._syncing = False
        self._synced_steps = steps
        self._trained = False
        self._dirty = True

    def state_dict(self, *args, **kwargs):
        if getattr(self, "_trained", False) and not getattr(self, "_syncing", False):
            self.sync_trained_weights()
        return super().state_dict(*args, **kwargs)

    def read_grad(self, name):
        """Gradient of one parameter (state_dict name) from the last train_step / frx_train_fwd_bwd, state_dict layout."""
        eng = self._engine
        t = self.state_dict()[name]
        buf = torch.empty_like(t, dtype=torch.float32).contiguous()
        eng.h.call("frx_train_read_grad", name.encode(), _ptr(buf))
        return buf

    def read_train_tap(self, name):
        """Named buffer of the last training step's activation / gradient tape (frx_train_read_tap), flat fp32."""
        eng = self._engine
        n = int(eng.h.lib.frx_train_read_tap(eng.h.ptr, name.encode(), None, 0))
        if n < 0:
            raise RuntimeError("frx_train_read_tap: " + eng.h.lib.frx_last_error(eng.h.ptr).decode())
        buf = torch.empty(n, dtype=torch.float32, device=eng.device)
        eng.h.lib.frx_train_read_tap(eng.h.ptr, name.encode(), _ptr(buf), n)
        return buf

    @property
    def memory_tokens(self):
        return (self._dims["height"] // self._down) * (self._dims["width"] // self._down)

    def encode(self, input):
        """SATRNEncoder.forward :311-323 -> src [B, h*w, C]."""
        b = input.size(0)
        eng = self.engine(input.device, b, 1)
        x = input.detach().float().contiguous()
        memory = torch.empty(b, self.memory_tokens, self._dims["enc_hidden"], device=x.device)
        eng.h.call("frx_encode", _ptr(x), b, _ptr(memory), _stream(x.device))
        return memory

    def submit_host(self, images_host, tokens_host, steps, slot):
        """Pipelined host entry (frx_forward_greedy_host_submit): enqueue H2D of ``images_host`` (CPU fp32, ideally
        pinned) -> encode + greedy decode -> D2H of the tokens into ``tokens_host`` (CPU int64 [B, steps]) for ``slot``
        0 / 1 and return at once; ``wait_host(slot)`` blocks until the tokens have arrived.  With both slots in flight
        the copies of the neighbouring batches run under the current batch's compute."""
        b = images_host.size(0)
        dev = torch.device("cuda", torch.cuda.current_device()) if self._engine is None else self._engine.device
        eng = self.engine(dev, b, steps)
        eng.h.call("frx_forward_greedy_host_submit", _ptr(images_host), b, steps, _ptr(tokens_host), int(slot), _stream(dev))

    def wait_host(self, slot):
        self._engine.h.call("frx_forward_greedy_host_wait", int(slot))

    def greedy(self, input, steps, forced=None, want_logits=True):
        """Encode + greedy loop returning (logits | None, tokens [B, steps] int64)
        on the input's device; ``forced`` feeds given tokens (forced decoding)."""
        b = input.size(0)
        eng = self.engine(input.device, b, steps)
        x = input.detach().float().contiguous()
        dev = x.device
        memory = self.encode(x)
        logits = torch.empty(b, steps, self._dims["num_classes"], device=dev) if want_logits else None
        tokens = torch.empty(b, steps, dtype=torch.int64, device=dev)
        f = forced.to(device=dev, dtype=torch.int64).contiguous() if forced is not None else None
        eng.h.call("frx_decode_greedy", _ptr(memory), b, steps, _ptr(logits), _ptr(tokens), _ptr(f), _stream(dev))
        return logits, tokens

    def greedy_until_eos(self, input, max_steps, forced=None, want_logits=False):
        """Encode + greedy decode that stops each image at its first <EOS> (frx_decode_greedy_eos): returns
        (logits | None, tokens [B, max_steps] int64, lengths [B] int32) on the input's device.  Up to lengths[b] the
        logits and tokens are the full greedy decode's (bitwise); after it tokens are <PAD> and logits rows 0.  With a
        DecodingManager attached the rows are its masked probabilities and the tokens its picks.  ``forced`` feeds given
        tokens; row b then stops after the step where forced[b, t] is <EOS>."""
        b = input.size(0)
        eng = self.engine(input.device, b, max_steps)
        x = input.detach().float().contiguous()
        dev = x.device
        managed = self.decoder.manager is not None
        if managed:
            self._attach_manager(eng)
        memory = self.encode(x)
        logits = torch.empty(b, max_steps, self._dims["num_classes"], device=dev) if want_logits else None
        tokens = torch.empty(b, max_steps, dtype=torch.int64, device=dev)
        lengths = torch.empty(b, dtype=torch.int32, device=dev)
        f = forced.to(device=dev, dtype=torch.int64).contiguous() if forced is not None else None
        eng.h.call("frx_decode_greedy_eos", _ptr(memory), b, max_steps, _ptr(logits), _ptr(tokens), _ptr(lengths), _ptr(f),
                   int(managed), _stream(dev))
        return logits, tokens, lengths

    def greedy_host(self, images_host, steps, tokens_host=None, logits_host=None):
        """End-to-end call with HOST buffers (frx_forward_greedy_host): H2D of the
        images, encode, decode, D2H of the tokens; returns the host token tensor."""
        b = images_host.size(0)
        dev = torch.device("cuda", torch.cuda.current_device())
        eng = self.engine(dev, b, steps)
        if tokens_host is None:
            tokens_host = torch.empty(b, steps, dtype=torch.int64).pin_memory()
        eng.h.call("frx_forward_greedy_host", _ptr(images_host), b, steps, _ptr(logits_host), _ptr(tokens_host),
                   _stream(dev))
        return tokens_host

    def beam_search(self, input, data_loader=None, topk=1, beam_width=5, max_sequence=230):
        """:708-867 (topk=1) -> LongTensor [B, max_sequence] on the CPU."""
        if topk != 1:
            raise NotImplementedError("only topk=1 (what decode() uses, postprocessing/decoding.py:43-48)")
        b = input.size(0)
        eng = self.engine(input.device, b, max_sequence)
        memory = self.encode(input)
        out = torch.empty(b, max_sequence, dtype=torch.int64, device=input.device)
        eng.h.call("frx_beam_search", _ptr(memory), b, beam_width, max_sequence, _ptr(out), _stream(input.device))
        return out.cpu()

    def read_tap(self, name):
        eng = self._engine
        n, shape = ctypes.c_int64(), (ctypes.c_int32 * 4)()
        eng.h.call("frx_read_tap", name.encode(), None, 0, ctypes.byref(n), shape, None)
        out = torch.empty(tuple(shape), device=eng.device)
        eng.h.call("frx_read_tap", name.encode(), _ptr(out), n.value, ctypes.byref(n), shape, _stream(eng.device))
        return out  # NHWC


class LiteSATRN(EfficientSATRN):
    """networks/LiteSATRN.py:548-590 -- the knowledge-distillation student: a 4-conv ShallowCNN trunk (1/16
    resolution, :21-70) in front of the same SATRN encoder / decoder classes; greedy decoding only (the
    reference's LiteSATRN has no beam_search).  precision="bf16" keeps the fp32 ShallowCNN / encoder layer and runs the
    whole greedy loop in the persistent cluster kernel (128-wide geometry: clusters of 4 CTAs, one per head)."""

    _network = 1
    _down = 16

    def __init__(self, FLAGS, train_dataset, checkpoint=None, decoding_manager=None, *,
                 precision="fp32", max_batch=None, max_steps=None):
        nn.Module.__init__(self)
        self._setup(FLAGS, train_dataset, precision, max_batch, max_steps)
        self.encoder = layout.build_param_tree(layout.lite_encoder_shapes(self._dims), "encoder.")
        self.decoder = layout.build_param_tree(layout.decoder_shapes(self._dims), "decoder.")
        d = self.decoder
        d.hidden_dim, d.filter_dim = self._dims["dec_hidden"], self._dims["dec_filter"]
        d.num_classes, d.layer_num = self._dims["num_classes"], self._dims["dec_layers"]
        d.pad_id, d.st_id = self._ids[2], self._ids[0]
        d.manager = decoding_manager
        self.criterion = nn.CrossEntropyLoss(ignore_index=self._ids[2])
        if checkpoint:
            self.load_state_dict(checkpoint)

    def beam_search(self, *a, **k):
        raise AttributeError("LiteSATRN has no beam_search (networks/LiteSATRN.py defines none)")


class SWIN(EfficientSATRN):
    """networks/SWIN.py:1024-1063 -- Swin-B/384 encoder (patch 4, window 12, depths 2-2-18-2, absolute position
    embedding; hard-wired in the reference, the yaml's SATRN.encoder block is ignored) + the transformer decoder
    of configs/SWIN.yaml.  Input [B, 3, 384, 384]; greedy decoding only.  precision="bf16" runs the encoder's linear
    layers on the tcgen05 GEMM (the 512-wide, 4-layer decoder keeps the fp32 step kernels).  Unlike the reference the
    constructor does not download ImageNet weights (there is no network): pass a checkpoint dict."""

    _network = 2
    _down = 32

    def __init__(self, FLAGS, train_dataset, checkpoint=None, *, precision="fp32", max_batch=None, max_steps=None):
        nn.Module.__init__(self)
        self._setup(FLAGS, train_dataset, precision, max_batch, max_steps)
        self._dims.update(height=layout.SWIN_IMG, width=layout.SWIN_IMG, in_ch=3, enc_hidden=layout.SWIN_EMBED * 8,
                          enc_filter=0, enc_layers=0, enc_heads=0)
        self.encoder = layout.build_swin_encoder_tree()
        self.decoder = layout.build_param_tree(layout.swin_decoder_shapes(self._dims), "decoder.")
        d = self.decoder
        d.hidden_dim, d.filter_dim = self._dims["dec_hidden"], self._dims["dec_filter"]
        d.num_classes, d.layer_num = self._dims["num_classes"], self._dims["dec_layers"]
        d.pad_id, d.st_id = self._ids[2], self._ids[0]
        d.manager = None
        self.criterion = nn.CrossEntropyLoss(ignore_index=self._ids[2])
        if isinstance(checkpoint, dict):
            self.load_state_dict(checkpoint)

    def beam_search(self, *a, **k):
        raise AttributeError("SWIN has no usable beam_search (the reference's is dead code, SURVEY App. A.6)")


class EfficientSATRN_encoder(_FrxModule):
    """:870-894 -- the ensemble driver's encoder half (utils/ensemble_utils.py:168-176)."""

    _parts = 1

    def __init__(self, FLAGS, train_dataset, checkpoint=None, *, precision="fp32", max_batch=None):
        super().__init__()
        self._setup(FLAGS, train_dataset, precision, max_batch, 1)
        self.encoder = layout.build_param_tree(layout.encoder_shapes(self._dims), "encoder.")
        if checkpoint:
            self.load_state_dict(checkpoint)

    def forward(self, input):
        b = input.size(0)
        eng = self.engine(input.device, b, 1)
        x = input.detach().float().contiguous()
        s = (self._dims["height"] // 32) * (self._dims["width"] // 32)
        memory = torch.empty(b, s, self._dims["enc_hidden"], device=x.device)
        eng.h.call("frx_encode", _ptr(x), b, _ptr(memory), _stream(x.device))
        return memory


class EfficientSATRN_decoder(_FrxModule):
    """:897-952 -- stateful ``step_forward`` / ``reset_status`` used by the
    ensemble driver (utils/ensemble_utils.py:83-118)."""

    _parts = 2

    def __init__(self, FLAGS, train_dataset, checkpoint=None, *, precision="fp32", max_batch=None, max_steps=231):
        super().__init__()
        self._setup(FLAGS, train_dataset, precision, max_batch, max_steps)
        self.decoder = layout.build_param_tree(layout.decoder_shapes(self._dims), "decoder.")
        self.decoder.layer_num = self._dims["dec_layers"]
        self.decoder.st_id, self.decoder.pad_id = self._ids[0], self._ids[2]
        self.step_idx = 0
        self.features = [None] * self._dims["dec_layers"]  # kept for API compatibility; state lives in the handle
        if checkpoint:
            self.load_state_dict(checkpoint)

    def step_forward(self, src, target):
        """:932-948  src [b, S, C], target [b] int64 -> logits [b, 1, V]."""
        b = src.size(0)
        eng = self.engine(src.device, b, self._max_steps or 231)
        st = _stream(src.device)
        if self.step_idx == 0:
            eng.h.call("frx_decode_begin", _ptr(src.detach().float().contiguous()), b, st)
        tgt = target.to(device=src.device, dtype=torch.int64).contiguous()
        out = torch.empty(b, 1, self._dims["num_classes"], device=src.device)
        eng.h.call("frx_decode_step", _ptr(tgt), _ptr(out), st)
        self.step_idx += 1
        return out

    def reset_status(self):
        """:950-952"""
        self.step_idx = 0
        self.features = [None] * self._dims["dec_layers"]
