"""The host plan of the fused policy pretraining (engine.plan_xent) against the reference's loss restated in
oracle/ref_port.policy_xent_loss: row lengths from the first <END>, the clamp to L-1 positions, the per-position weights
with the unclamped caplen, the number of decode steps S, and the error for a row without <END>.  No GPU needed."""
import numpy as np
import pytest
import torch

from oracle import ref_port, synth


def _plan(caps):
    from icrl_b200.engine import plan_xent
    return plan_xent(caps)


def _caps(rows, L=17):
    """Captions of the given END columns (None: no END); <START> first, words in between, <NULL> after END."""
    rs = np.random.RandomState(7)
    caps = rs.randint(4, 50, size=(len(rows), L)).astype(np.int64)
    caps[:, 0] = 1
    for i, e in enumerate(rows):
        if e is not None:
            caps[i, e] = 2
            caps[i, e + 1:] = 0
    return caps


def test_lengths_weights_and_steps():
    caps = _caps([1, 5, 16, 9])
    n, w, S = _plan(caps)
    B, L = caps.shape
    caplen = np.array([2, 6, 17, 10])
    assert n.tolist() == [2, 6, 16, 10]                      # END in the last column: clamped to L-1 positions
    assert S == 16
    np.testing.assert_array_equal(w, caplen / (B * np.minimum(caplen, L - 1)))
    assert w[2] == 17 / (4 * 16)                             # the unclamped caplen in the weight


def test_steps_follow_the_longest_row():
    n, w, S = _plan(_caps([1, 3, 2]))
    assert n.tolist() == [2, 4, 3] and S == 4


def test_first_end_of_the_row_counts():
    caps = _caps([12, 12])
    caps[0, 4] = 2                                           # a stray <END> mid-row ends that row
    n, w, S = _plan(caps)
    assert n.tolist() == [5, 13] and S == 13


def test_row_without_end_raises():
    caps = _caps([3, None, 6])
    with pytest.raises(ValueError, match="row 1"):
        _plan(caps)
    with pytest.raises(ValueError):
        _plan(caps[:, :1])


def test_plan_reproduces_the_reference_loss():
    """sum_b w_b sum_{s < n_b} CE(b, s) with the plan's n and w equals the reference's loss (float64 port) on rows with
    END at column 1, mid-row, as a stray token and in the last column."""
    w_ = synth.make_weights(3, vocab=64)
    nets = ref_port.Nets(w_, dtype=torch.float64)
    f = np.random.RandomState(3).standard_normal((6, 512)).astype(np.float32)
    caps = _caps([1, 7, 16, 16, 3, 10])
    caps[3, 5] = 2
    loss, logits = ref_port.policy_xent_loss(nets, f, caps)
    n, w, S = _plan(caps)
    z = logits.detach()
    t = torch.as_tensor(caps[:, 1:])
    ce = torch.logsumexp(z, dim=2) - z.gather(2, t.unsqueeze(2)).squeeze(2)        # (B, L-1)
    mask = torch.arange(caps.shape[1] - 1)[None, :] < torch.as_tensor(n)[:, None]
    mine = float((torch.as_tensor(w)[:, None] * ce * mask).sum())
    ref = float(loss.detach())
    assert abs(mine - ref) <= 1e-12 * abs(ref)
    assert not bool(mask[:, S:].any())
