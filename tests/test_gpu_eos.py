"""Greedy decoding that stops at <EOS> (frx_decode_greedy_eos, EfficientSATRN.greedy_until_eos, decode(...,
stop_at_eos=True)) against the full-length decode of the same handle: for each image, everything up to its first <EOS>
is bit-identical, <PAD> / zero rows after it, and lengths = first <EOS> + 1 (or max_steps)."""
import numpy as np
import pytest
import torch

from conftest import load_golden, load_manager_golden
from helpers import make_lite_model, make_model, make_swin_model
from oracle import manager, satrn, swin, synth
from oracle.make_golden import LITE_SPEC

pytestmark = pytest.mark.gpu

SOS, EOS, PAD = satrn.SOS_ID, satrn.EOS_ID, satrn.PAD_ID
V = 245


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _memory(model, b, seed):
    """Seeded encoder output [b, S, C]: the golden memory tiled over the batch for EfficientSATRN (each row scaled and
    perturbed, so that the rows differ), a seeded normal tensor for the other networks."""
    g = torch.Generator().manual_seed(seed)
    s, c = model.memory_tokens, model._dims["dec_src"]
    if model._network == 0:
        base = torch.from_numpy(load_golden(0)["memory"])
        mem = base.repeat((b + base.size(0) - 1) // base.size(0), 1, 1)[:b]
        mem = mem * (1 + 0.1 * torch.randn(b, 1, 1, generator=g)) + 0.05 * mem.std() * torch.randn(mem.shape, generator=g)
    else:
        mem = torch.randn(b, s, c, generator=g)
    return mem.cuda().contiguous()


def _forced(b, steps, seed):
    """Seeded forced sequences: random non-special tokens, <EOS> at a random step -- at step 0 (length 1) in row 0, at
    the last step in row 1 -- and no <EOS> at all in every fifth row."""
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(3, V, (b, steps), generator=g)
    at = torch.randint(0, steps, (b,), generator=g)
    at[0] = 0
    if b > 1:
        at[1] = steps - 1
    for i in range(b):
        if i % 5 != 2:
            tok[i, at[i]] = EOS
    return tok.cuda()


def _full(model, mem, steps, forced=None, managed=False):
    b = mem.size(0)
    eng = model.engine(mem.device, b, steps)
    logits = torch.empty(b, steps, V, device="cuda")
    tokens = torch.empty(b, steps, dtype=torch.int64, device="cuda")
    if managed:
        eng.h.call("frx_decode_greedy_managed", mem.data_ptr(), b, steps, logits.data_ptr(), tokens.data_ptr(), _stream())
    else:
        eng.h.call("frx_decode_greedy", mem.data_ptr(), b, steps, logits.data_ptr(), tokens.data_ptr(),
                   forced.data_ptr() if forced is not None else None, _stream())
    return logits, tokens


def _eos(model, mem, steps, forced=None, managed=False, want_logits=True):
    b = mem.size(0)
    eng = model.engine(mem.device, b, steps)
    logits = torch.full((b, steps, V), float("nan"), device="cuda") if want_logits else None
    tokens = torch.full((b, steps), -7, dtype=torch.int64, device="cuda")
    lengths = torch.full((b,), -7, dtype=torch.int32, device="cuda")
    eng.h.call("frx_decode_greedy_eos", mem.data_ptr(), b, steps, logits.data_ptr() if logits is not None else None,
               tokens.data_ptr(), lengths.data_ptr(), forced.data_ptr() if forced is not None else None, int(managed),
               _stream())
    return logits, tokens, lengths


def _expected_lengths(stop):
    b, steps = stop.shape
    hit = stop == EOS
    first = hit.int().argmax(1) + 1
    return torch.where(hit.any(1), first, torch.full_like(first, steps))


def _check(full, out, stop):
    """The stop-at-<EOS> contract: out equals full up to the first <EOS> of `stop` (inclusive), <PAD> / 0 after it."""
    full_logits, full_tokens = full
    logits, tokens, lengths = out
    torch.cuda.synchronize()
    want = _expected_lengths(stop)
    assert torch.equal(lengths.long(), want)
    keep = torch.arange(stop.size(1), device=stop.device)[None, :] < want[:, None]
    assert torch.equal(tokens, torch.where(keep, full_tokens, torch.full_like(full_tokens, PAD)))
    if logits is not None:
        ref = torch.where(keep[..., None], full_logits, torch.zeros_like(full_logits))
        bad = (logits != ref).any(-1).nonzero()
        assert bad.numel() == 0, (
            "%d logits rows differ; first (image, step, length): %s; NaN rows in full / stop-at-<EOS>: %d / %d; max diff %s"
            % (bad.size(0), [(int(b), int(t), int(want[b])) for b, t in bad[:8].tolist()],
               int(full_logits.isnan().any(-1).sum()), int(logits.isnan().any(-1).sum()),
               (logits - ref)[bad[:, 0], bad[:, 1]].abs().max().item()))
    return want


def _decoder_only(model):
    model.set_option("parts", 2)   # the decode runs on a given memory: no encoder workspaces for a 1000-image batch
    return model


@pytest.fixture(scope="module")
def geometries(ckpt0):
    """One 16-bit handle per decode-kernel geometry: 256-wide with one and two heads per CTA, 128-wide, 512-wide."""
    hpc1 = _decoder_only(make_model(ckpt0, precision="bf16").cuda().eval())
    hpc1.set_option("dec_hpc", 1)
    hpc2 = _decoder_only(make_model(ckpt0, precision="bf16").cuda().eval())
    hpc2.set_option("dec_hpc", 2)
    lite_sd = synth.synth_state_dict(satrn.ModelSpec(**LITE_SPEC), 0, calib_batch=4)
    lite = _decoder_only(make_lite_model(lite_sd, precision="bf16").cuda().eval())
    sw = _decoder_only(make_swin_model(swin.synth_state_dict(swin.swin_spec(), 0), precision="bf16").cuda().eval())
    return {"hpc1": hpc1, "hpc2": hpc2, "lite": lite, "swin": sw}


@pytest.mark.parametrize("geometry", ["hpc1", "hpc2", "lite", "swin"])
# 9, 100, 250: the last cluster is partial (slots past the batch exist and any cluster may claim any image)
@pytest.mark.parametrize("b", [1, 7, 9, 100, 250, 300, 1000])
def test_forced_lengths_every_geometry(geometries, geometry, b):
    model = geometries[geometry]
    steps = 50
    mem = _memory(model, b, seed=b)
    forced = _forced(b, steps, seed=b + 1)
    with torch.no_grad():
        full = _full(model, mem, steps, forced)
        out = _eos(model, mem, steps, forced)
    lengths = _check(full, out, forced)
    assert lengths.min().item() == 1 and (b < 2 or lengths.max().item() == steps)


def _eos_biased(ckpt, bias):
    sd = dict(ckpt)
    sd["decoder.generator.bias"] = sd["decoder.generator.bias"].clone()
    sd["decoder.generator.bias"][EOS] += bias
    return sd


# <EOS> generator-bias increments tried in turn (cumulative: +1.0, +1.1, ..., +1.5, +2.0, +3.0).  The contract is
# checked bitwise at every setting.  +1.0 stops only a few percent of the rows of this memory (on a B200: 7 of 256, 41 of
# 1000); the larger biases stop most or all of them, so that rows are refilled at every step of the decode.  Batches of
# 256 and more must be mixed at +1.0 already (rows that stop early and rows that run to max_steps); a small batch must be
# mixed at one setting at least.
BIASES = (1.0, 0.1, 0.1, 0.1, 0.1, 0.1, 0.5, 1.0)


def _free_running_sweep(model, mem, steps, managed=False):
    mixed = []
    for add in BIASES:
        with torch.no_grad():
            model.decoder.generator.bias[EOS] += add
        model.refresh()
        model.engine(mem.device, mem.size(0), steps)   # re-finalize with the new bias
        if managed:
            model._attach_manager(model._engine)
        with torch.no_grad():
            full = _full(model, mem, steps, managed=managed)
            out = _eos(model, mem, steps, managed=managed)
        lengths = _check(full, out, full[1])
        early = int((lengths < steps).sum())
        print("bias +%.1f: %d of %d rows stop early, mean length %.1f of %d"
              % (model.decoder.generator.bias[EOS].item() - model._eos_bias0, early, mem.size(0),
                 lengths.float().mean().item(), steps))
        mixed.append(0 < early < mem.size(0))
    assert any(mixed)
    return mixed


@pytest.fixture(scope="module")
def free_model(ckpt0):
    return _decoder_only(make_model(_eos_biased(ckpt0, 1.0), precision="bf16").cuda().eval())


@pytest.mark.parametrize("b,hpc", [(256, 0), (1000, 0)] + [(b, hpc) for b in (9, 100, 250) for hpc in (1, 2)])
def test_free_running_stops_at_emitted_eos(ckpt0, b, hpc):
    model = _decoder_only(make_model(ckpt0, precision="bf16").cuda().eval())
    if hpc:
        model.set_option("dec_hpc", hpc)
    model._eos_bias0 = model.decoder.generator.bias[EOS].item()
    mixed = _free_running_sweep(model, _memory(model, b, seed=10 + b), 231)
    if b >= 256:
        assert mixed[0]   # bias +1.0


def test_managed_probabilities_and_tokens(ckpt0):
    g = load_manager_golden()
    rules = manager.Rules([str(t) for t in g["vocab"]], g["flags"], g["limit"])
    model = _decoder_only(make_model(ckpt0, precision="bf16").cuda().eval())
    model._eos_bias0 = model.decoder.generator.bias[EOS].item()
    model.decoder.manager = rules.as_manager()
    b, steps = 300, 231
    mem = _memory(model, b, seed=3)
    _free_running_sweep(model, mem, steps, managed=True)
    with pytest.raises(RuntimeError):
        _eos(model, mem, steps, forced=_forced(b, steps, 0), managed=True)


def test_fp32_mode_applies_the_contract(ckpt0, spec):
    model = make_model(_eos_biased(ckpt0, 1.0)).cuda().eval()
    b, steps = 7, 60
    mem = _memory(model, b, seed=4)
    forced = _forced(b, steps, seed=5)
    with torch.no_grad():
        _check(_full(model, mem, steps), _eos(model, mem, steps), _full(model, mem, steps)[1])
        _check(_full(model, mem, steps, forced), _eos(model, mem, steps, forced), forced)


def test_repeatable_counter_reset_and_graph_capture(free_model):
    steps = 231
    mem = _memory(free_model, 1000, seed=6)
    with torch.no_grad():
        a = _eos(free_model, mem, steps)
        c = _eos(free_model, mem, steps)
        torch.cuda.synchronize()
        assert all(torch.equal(x, y) for x, y in zip(a, c))
        small = mem[:5].contiguous()
        out = _eos(free_model, small, steps)       # after a 1000-image call: the work counter starts at 0 again
        full = _full(free_model, small, steps)
        _check(full, out, full[1])
        # captured in a CUDA graph and replayed
        logits = torch.empty(1000, steps, V, device="cuda")
        tokens = torch.empty(1000, steps, dtype=torch.int64, device="cuda")
        lengths = torch.empty(1000, dtype=torch.int32, device="cuda")
        eng = free_model.engine(mem.device, 1000, steps)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, capture_error_mode="relaxed"):
            eng.h.call("frx_decode_greedy_eos", mem.data_ptr(), 1000, steps, logits.data_ptr(), tokens.data_ptr(),
                       lengths.data_ptr(), None, 0, _stream())
        logits.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(logits, a[0]) and torch.equal(tokens, a[1]) and torch.equal(lengths, a[2])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_decode_stop_at_eos(ckpt0, spec, precision):
    from frx import decode
    model = make_model(_eos_biased(ckpt0, 2.0), precision=precision).cuda().eval()
    x = synth.synth_images(spec, 5, 3).cuda()
    expected = satrn.expected_tokens(5, 39).cuda()
    with torch.no_grad():
        full = decode(model, x, expected=expected)
        short = decode(model, x, expected=expected, stop_at_eos=True)
    assert short.dtype == torch.int64 and short.shape == full.shape == (5, 40)
    keep = torch.arange(40, device=full.device)[None, :] < _expected_lengths(full)[:, None]
    assert torch.equal(short, torch.where(keep, full, torch.full_like(full, PAD)))
    assert (~keep).any()
