"""The CPU restatement of the training step's counter-based dropout (tests/dropout_oracle.py): the Philox4x32-10
generator against Random123's known-answer vectors, the keep rule's statistics, and the dropout training oracle, which
with all-keep masks must compute exactly what the oracle without dropout computes."""
import numpy as np
import torch

import dropout_oracle as dropout
from oracle import synth, train

KNOWN_ANSWERS = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


def test_philox_known_answers():
    for ctr, key, want in KNOWN_ANSWERS:
        got = tuple(int(w) for w in dropout.philox4x32(ctr, key))
        assert got == want, ["%08x" % w for w in got]
    # vectorised: the same vectors as one batch of counters under one key
    ctr = np.array([[0, 0, 0, 0], [0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344]], dtype=np.uint64).T
    got = dropout.philox4x32(list(ctr), (0, 0))
    assert [int(w[0]) for w in got] == list(KNOWN_ANSWERS[0][2])


def test_keep_fraction_and_scale_over_a_large_site():
    n, p = 1 << 20, 0.1
    x = torch.randn(n, generator=torch.Generator().manual_seed(5)) + 3.0   # no exact zeros among the inputs
    y = dropout.Dropout(p, seed=0x123456789, step=7)(x, 5, 2)
    kept = y != 0
    frac = kept.float().mean().item()
    sigma = (p * (1 - p) / n) ** 0.5
    assert abs(frac - (1 - p)) <= 6 * sigma, frac
    s = torch.tensor(1.0) / (torch.tensor(1.0) - torch.tensor(p, dtype=torch.float32))
    assert torch.equal(y[kept], x[kept] * s)
    # another site, layer, step, rank or seed draws another mask
    for kw, site, layer in ((dict(seed=0x123456789, step=8), 5, 2), (dict(seed=0x123456789, step=7, rank=1), 5, 2),
                            (dict(seed=0x123456788, step=7), 5, 2), (dict(seed=0x123456789, step=7), 5, 3),
                            (dict(seed=0x123456789, step=7), 7, 2)):
        other = dropout.Dropout(p, **kw)(x, site, layer) != 0
        assert (other != kept).float().mean().item() > 0.1


def test_threshold_uses_the_fp32_rate():
    assert dropout.keep_threshold(0.0) == 0
    assert dropout.keep_threshold(0.1) == int(np.floor(float(np.float32(0.1)) * 2.0 ** 32))
    assert dropout.keep_threshold(np.nextafter(np.float32(1), np.float32(0))) <= 2 ** 32 - 1


def test_all_keep_masks_change_nothing(spec):
    """p = p_ffn = 0 runs every site's mask (all kept, scale 1): loss and gradients bitwise equal to the oracle without
    dropout."""
    sd = synth.synth_state_dict(spec, 0)
    x, e = train.synth_batch(spec, 2, 8, 4)
    plain = train.Trainer(sd, spec)
    masked = dropout.Trainer(sd, spec, 0.0, 0.0, 3, 0)
    loss0, g0 = plain.forward_backward(x, e)
    loss1, g1 = masked.forward_backward(x, e)
    assert loss0 == loss1
    for k in g0:
        assert torch.equal(g0[k], g1[k]), k
    # and a real rate changes the loss
    dropped = dropout.Trainer(sd, spec, 0.1, 0.1, 3, 0)
    assert dropped.forward_backward(x, e)[0] != loss0
