"""Dropout in the training step (set_train_dropout / frx_train_set_dropout) against the train-step oracle applying the same
counter-based masks (tests/dropout_oracle.py): the generator on the GPU, loss / gradients / optimiser steps of EfficientSATRN
and LiteSATRN through train_step, the reference-style loop, the split-K plan, reproducibility, and that neither the
default pass nor inference changes."""
import ctypes

import pytest
import torch

import dropout_oracle
from helpers import make_lite_model, make_model
from oracle import satrn, synth, train
from test_gpu_train import EXACT, EXACT_TOL, GLOBAL_TOL, GRAD_TOL, LOSS_TOL, NORM_TOL, SPLITK_GLOBAL_TOL, SPLITK_NORM_TOL
from test_oracle_dropout import KNOWN_ANSWERS

pytestmark = pytest.mark.gpu
P = 0.1           # FLAGS.dropout_rate of tests/helpers.py, and the decoder feed-forward's fixed rate
# EfficientSATRN's global gradient norm at step 0: measured 1.7e-4 / 3.1e-4 off the oracle (seeds 1 / 0) with dropout
# against < 1e-4 without.  The loss (1e-6), the tensors above every ReLU (EXACT_TOL) and the whole gradient (< GLOBAL_TOL)
# agree; the worst tensors sit below the encoder layers' ReLU feed-forward, where units flip across their kink (see
# test_gpu_train.py GRAD_TOL).  A wrong mask would move the norm by percents, not by 1e-4.
DROP_NORM_TOL = 1e-3


def _grad_errors(model, grads, names, exact=()):
    worst, worst_name, num, den = 0.0, "", 0.0, 0.0
    for n in names:
        got, want = model.read_grad(n).cpu(), grads[n]
        err = (got - want).norm().item() / max(want.norm().item(), 1e-12)
        if want.norm().item() < 1e-5:     # pure round-off (biases in front of a train-mode BatchNorm): absolute scale
            err = (got - want).norm().item() / 1e-3
        num += (got - want).norm().item() ** 2
        den += want.norm().item() ** 2
        if n in exact:
            assert err <= EXACT_TOL, (n, err)
        if err > worst:
            worst, worst_name = err, n
    return (num / den) ** 0.5, worst, worst_name


def _three_steps(model, tr, spec, seed, label, norm_tol=NORM_TOL):
    """Three train_steps against the oracle Trainer with the same masks; steps 1-2 replay the captured CUDA graph."""
    names = [k for k in tr.sd if train.is_param(k)]
    for it in range(3):
        x, e = train.synth_batch(spec, 4, 24, 10 * seed + it)
        loss, gn = model.train_step(x.cuda(), e.cuda())
        loss, gn = loss.item(), gn.item()
        if it == 0:
            ref_loss, grads = tr.forward_backward(x, e)
            glob, worst, worst_name = _grad_errors(model, grads, names, EXACT if label == "EfficientSATRN" else ())
            ref_gn = float(torch.nn.utils.clip_grad_norm_(tr.params, max_norm=tr.max_grad_norm))
            tr.opt.step()
            print("%s dropout seed %d step 0: loss %.6f (oracle %.6f), grad norm %.5f (oracle %.5f), whole-gradient rel-L2 "
                  "%.2e, worst tensor %.2e at %s" % (label, seed, loss, ref_loss, gn, ref_gn, glob, worst, worst_name))
            assert abs(loss - ref_loss) <= LOSS_TOL * abs(ref_loss)
            assert abs(gn - ref_gn) <= norm_tol * ref_gn
            assert glob <= GLOBAL_TOL, glob
            assert worst <= GRAD_TOL, (worst_name, worst)
        else:
            ref_loss, ref_gn = tr.step(x, e)
            print("%s dropout seed %d step %d: loss %.6f (oracle %.6f), grad norm %.5f (oracle %.5f)"
                  % (label, seed, it, loss, ref_loss, gn, ref_gn))
            assert abs(loss - ref_loss) <= 2e-3 * abs(ref_loss), (it, loss, ref_loss)
            assert abs(gn - ref_gn) <= 3e-2 * ref_gn, (it, gn, ref_gn)


def test_philox_on_the_gpu_matches_random123():
    import frx
    lib = frx._lib.load_library()
    u32 = ctypes.c_uint32
    for ctr, key, want in KNOWN_ANSWERS:
        out = (u32 * 4)()
        assert lib.frx_philox4x32((u32 * 4)(*ctr), (u32 * 2)(*key), out) == 0
        assert tuple(out) == want, ["%08x" % w for w in out]


@pytest.mark.parametrize("seed", [0, 1])
def test_train_step_with_dropout_matches_oracle(spec, seed):
    sd = synth.synth_state_dict(spec, seed)
    model = make_model(sd, max_batch=4, max_steps=24).cuda().train()
    model.set_option("train_splitk", 0)
    model.set_train_dropout(seed=1000 + seed)          # p = FLAGS.dropout_rate (0.1), p_ffn = 0.1
    tr = dropout_oracle.Trainer(sd, spec, P, P, 1000 + seed)
    _three_steps(model, tr, spec, seed, "EfficientSATRN", DROP_NORM_TOL)


def test_lite_train_step_with_dropout_matches_oracle():
    from oracle.make_golden import LITE_SPEC
    lspec = satrn.ModelSpec(**LITE_SPEC)
    sd = synth.synth_state_dict(lspec, 0, calib_batch=4)
    model = make_lite_model(sd, max_batch=4, max_steps=24).cuda().train()
    model.set_option("train_splitk", 0)
    model.set_train_dropout(P, seed=7)
    tr = dropout_oracle.Trainer(sd, lspec, P, P, 7)
    _three_steps(model, tr, lspec, 0, "LiteSATRN")


def test_reference_style_loop_with_dropout(spec, ckpt0):
    """output = model(input, expected, True, 1.0); loss.backward(); clip; torch AdamW -- the compatibility path's backward
    regenerates the masks of the forward it continues."""
    model = make_model(ckpt0, max_batch=4, max_steps=24).cuda().train()
    model.set_option("train_splitk", 0)
    model.set_train_dropout(P, seed=11)
    opt = torch.optim.AdamW(model.parameters(), lr=5e-4, weight_decay=1e-6)
    crit = torch.nn.CrossEntropyLoss(ignore_index=2)
    tr = dropout_oracle.Trainer(ckpt0, spec, P, P, 11)
    for it in range(3):
        x, e = train.synth_batch(spec, 4, 24, 40 + it)
        opt.zero_grad()
        out = model(x.cuda(), e.cuda(), True, 1.0)
        loss = crit(out.transpose(1, 2), e[:, 1:].cuda())
        loss.backward()
        gn = torch.nn.utils.clip_grad_norm_(model.parameters(), 2.0)
        opt.step()
        ref_loss, ref_gn = tr.step(x, e)
        print("reference-style loop with dropout, step %d: loss %.6f (oracle %.6f), grad norm %.5f (oracle %.5f)"
              % (it, loss.item(), ref_loss, gn.item(), ref_gn))
        assert abs(loss.item() - ref_loss) <= (LOSS_TOL if it == 0 else 2e-3) * abs(ref_loss)
        assert abs(gn.item() - ref_gn) <= (NORM_TOL if it == 0 else 3e-2) * ref_gn


@pytest.mark.parametrize("seed", [0, 1])
def test_train_step_with_dropout_default_split_k_plan(spec, seed):
    sd = synth.synth_state_dict(spec, seed)
    tr = dropout_oracle.Trainer(sd, spec, P, P, 5)
    names = [k for k in tr.sd if train.is_param(k)]
    x, e = train.synth_batch(spec, 4, 24, 10 * seed)
    ref_loss, grads = tr.forward_backward(x, e)
    ref_gn = sum(grads[n].norm().item() ** 2 for n in names) ** 0.5
    res = []
    for rep in range(2):
        model = make_model(sd, max_batch=4, max_steps=24).cuda().train()
        model.set_train_dropout(P, seed=5)
        loss, gn = model.train_step(x.cuda(), e.cuda())
        res.append((loss.item(), gn.item()))
    loss, gn = res[0]
    num = sum((model.read_grad(n).cpu() - grads[n]).norm().item() ** 2 for n in names)
    glob = (num / ref_gn ** 2) ** 0.5
    print("split-K plan with dropout, seed %d: loss %.6f (oracle %.6f), grad norm %.5f (oracle %.5f), whole-gradient "
          "rel-L2 %.2e" % (seed, loss, ref_loss, gn, ref_gn, glob))
    assert abs(loss - ref_loss) <= LOSS_TOL * abs(ref_loss)
    assert abs(gn - ref_gn) <= SPLITK_NORM_TOL * ref_gn
    assert glob <= SPLITK_GLOBAL_TOL
    assert abs(res[0][0] - res[1][0]) <= 1e-6 * abs(res[0][0]) and abs(res[0][1] - res[1][1]) <= 1e-5 * res[0][1]


def _run(model, spec, steps, seed0=60, lr=5e-4):
    """train_steps on seeded batches -> [(loss, flat gradient buffer)], and the launches they made."""
    out = []
    before = model._engine.launches if model._engine is not None else 0
    for it in range(steps):
        x, e = train.synth_batch(spec, 4, 24, seed0 + it)
        loss, _ = model.train_step(x.cuda(), e.cuda(), lr=lr, weight_decay=0.0 if lr == 0 else 1e-6)
        out.append((loss.item(), model._engine._train["grads"].clone()))
    return out, model._engine.launches - before


def test_rates_zero_restore_the_pass_without_dropout(ckpt0, spec):
    """set_train_dropout(0, p_ffn=0) after passes with dropout (one of them a graph replay) runs the same kernels as a model
    that never enabled it -- equal launch counts over an eager, a captured and a replayed step -- with the same loss and
    gradients up to the run-to-run spread of the pass: the weight-gradient and BatchNorm reductions add per-CTA partials
    with atomics, so two runs of one pass agree to ~1e-7, not bitwise.  lr = 0 keeps the parameters of both models equal."""
    plain = make_model(ckpt0, max_batch=4, max_steps=24).cuda().train()
    toggled = make_model(ckpt0, max_batch=4, max_steps=24).cuda().train()
    toggled.set_train_dropout(P, seed=3)
    with_drop, _ = _run(toggled, spec, 3, lr=0.0)
    toggled.set_train_dropout(0, p_ffn=0)
    got, n_toggled = _run(toggled, spec, 3, lr=0.0)
    want, n_plain = _run(plain, spec, 3, lr=0.0)
    assert n_toggled == n_plain
    for (l0, g0), (l1, g1) in zip(got, want):
        assert abs(l0 - l1) <= 1e-6 * abs(l1), (l0, l1)
        assert (g0 - g1).norm().item() <= 1e-5 * g1.norm().item()
    assert abs(with_drop[0][0] - want[0][0]) > 1e-4 * abs(want[0][0])   # the step with dropout was a different pass


def test_dropout_is_reproducible_and_keyed_by_seed_and_rank(ckpt0, spec):
    def losses(seed, rank=None):
        m = make_model(ckpt0, max_batch=4, max_steps=24).cuda().train()
        m.set_train_dropout(P, seed=seed)
        if rank is not None:
            eng, _ = m._trainer(torch.device("cuda"), 4, 24)
            eng.h.call("frx_train_set_dropout", P, P, seed, rank)
        res, _ = _run(m, spec, 3)
        return res
    # step 0 to the run-to-run spread of the pass (atomics, see above); later steps start from parameters that Adam's
    # first, sign-like update has moved by that spread, and a ReLU unit may flip: their losses only
    a, b = losses(21), losses(21)
    assert abs(a[0][0] - b[0][0]) <= 1e-6 * abs(b[0][0])
    assert (a[0][1] - b[0][1]).norm().item() <= 1e-5 * b[0][1].norm().item()
    for (l0, _), (l1, _) in zip(a[1:], b[1:]):
        assert abs(l0 - l1) <= 1e-4 * abs(l1)
    assert a[0][0] != a[1][0]                                   # each step draws new masks
    for other in (losses(22), losses(21, rank=1)):
        assert abs(other[0][0] - a[0][0]) > 1e-4 * abs(a[0][0])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_inference_never_drops(ckpt0, spec, precision):
    x, e = train.synth_batch(spec, 4, 24, 8)
    outs = []
    for configure in (False, True):
        m = make_model(ckpt0, precision=precision, max_batch=4, max_steps=24).cuda()
        if configure:
            m.set_train_dropout(0.5, seed=9, p_ffn=0.5)
            if precision == "fp32":
                m._trainer(torch.device("cuda"), 4, 24)          # the handle's training state carries the setting
        with torch.no_grad():
            outs.append(m.eval()(x.cuda(), e.cuda(), False, 0.0).cpu())
    assert torch.equal(outs[0], outs[1])


def test_rates_outside_the_unit_interval_are_rejected(ckpt0):
    m = make_model(ckpt0, max_batch=4, max_steps=24).cuda().train()
    for p in (-0.1, 1.0):
        with pytest.raises(ValueError):
            m.set_train_dropout(p)
    eng, _ = m._trainer(torch.device("cuda"), 4, 24)
    with pytest.raises(RuntimeError, match="rates must lie"):
        eng.h.call("frx_train_set_dropout", 1.0, 0.0, 0, 0)
    fresh = make_model(ckpt0).cuda().engine(torch.device("cuda"), 1, 1)   # a handle without training state
    with pytest.raises(RuntimeError, match="frx_train_create"):
        fresh.h.call("frx_train_set_dropout", 0.1, 0.1, 0, 0)
