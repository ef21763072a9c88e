"""CPU checks of the sample-weighted update restatement (tests/prio_oracle.py) that the prioritized replay's weighted fit is
compared with on the GPU."""
import pytest
import torch

from oracle import policy_torch as po
from oracle import policy_train_torch as pt
from tests import prio_oracle as wo


def _small_batch(B=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    img = (torch.rand((B, 400, 400, 2), generator=g) < 0.02).float()
    vec = torch.rand((B, 8), generator=g) * 400
    ta = torch.randn((B, 2), generator=g)
    tp = torch.randn((B, 400, 400), generator=g) * 0.1
    return img, vec, ta, tp


def test_unit_weights_are_the_unweighted_oracle_exactly():
    w = po.init_weights(3, randomize_bn=True)
    img, vec, ta, tp = _small_batch()
    l0, g0, s0 = pt.loss_and_grads(w, img, vec, ta, tp)
    l1, g1, s1 = wo.loss_and_grads(w, img, vec, ta, tp, torch.ones(3))
    assert l0 == l1
    assert all(torch.equal(g0[k], g1[k]) for k in g0)
    assert all(torch.equal(s0[k][0], s1[k][0]) and torch.equal(s0[k][1], s1[k][1]) for k in s0)
    # one step from the same state ends at the same weights
    wa, wb = dict(w), dict(w)
    pt.fit(wa, pt.KerasAdam(), img, vec, ta, tp)
    wo.fit(wb, pt.KerasAdam(), img, vec, ta, tp, torch.ones(3))
    assert all(torch.equal(wa[k], wb[k]) for k in wa)


def test_one_hot_weight_is_one_over_b_of_that_samples_loss():
    w = po.init_weights(5)
    B = 3
    img, vec, ta, tp = _small_batch(B, seed=1)
    act, ptr, _ = pt.forward_train(w, img, vec)
    for k in range(B):
        hot = torch.zeros(B)
        hot[k] = 1.0
        (tot, la, lp), _, _ = wo.loss_and_grads(w, img, vec, ta, tp, hot)
        want_a = float(((act[k] - ta[k]) ** 2).mean()) / B
        want_p = float(((ptr[k] - tp[k]) ** 2).mean()) / B
        assert la == pytest.approx(want_a, rel=1e-5) and lp == pytest.approx(want_p, rel=1e-5)
        assert tot == pytest.approx(want_a + want_p, rel=1e-5)


def test_weighted_gradients_against_central_finite_differences():
    """As test_train_oracle's check of the unweighted loss: float64 copy of the model, w in (0, 2]."""
    wd = {k: v.double() for k, v in po.init_weights(2).items()}
    img, vec, ta, tp = [t.double() for t in _small_batch(3, seed=4)]
    sw = torch.tensor([0.25, 2.0, 0.7], dtype=torch.float64)
    _, grads, _ = wo.loss_and_grads(wd, img, vec, ta, tp, sw)
    for name, idx in (("upconv4/kernel", (1, 1, 3, 0)), ("dense2/bias", (7,)), ("norm2/gamma", (5,)), ("output1/kernel", (4, 1))):
        eps = 1e-5
        vals = []
        for s in (+1, -1):
            w2 = {k: v.clone() for k, v in wd.items()}
            w2[name][idx] += s * eps
            a, p, _ = pt.forward_train(w2, img, vec)
            la, lp = wo.weighted_losses(a, p, ta, tp, sw)
            vals.append(float(la + lp))
        fd = (vals[0] - vals[1]) / (2 * eps)
        assert abs(fd - float(grads[name][idx])) <= 1e-5 + 1e-3 * abs(fd), (name, fd, float(grads[name][idx]))
