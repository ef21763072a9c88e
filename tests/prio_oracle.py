"""Sample-weighted restatement of the Q-learning update for the prioritized-replay tests -- TEST INFRASTRUCTURE.

``model.fit(..., sample_weight=w)`` in tf.keras under SUM_OVER_BATCH_SIZE: each head's loss is (1/B) sum_b w_b mse_b.  It is
written as the mean over every element of w_b * error^2, on the forward of oracle/policy_train_torch.py, so that w = 1
repeats that oracle's arithmetic exactly.  BatchNormalization keeps its unweighted batch statistics, as in Keras."""
import torch

from oracle import policy_train_torch as pt


def weighted_losses(act, ptr, target_act, target_ptr, sample_weight):
    sw = torch.as_tensor(sample_weight).to(act.dtype)
    la = (((act - target_act) ** 2) * sw[:, None]).mean()
    lp = (((ptr - target_ptr) ** 2) * sw[:, None, None]).mean()
    return la, lp


def loss_and_grads(w, image, vector, target_act, target_ptr, sample_weight):
    """pt.loss_and_grads with per-sample weights -> (total, mse_act, mse_ptr), {name: grad}, BN batch stats."""
    wt = {k: v.clone().detach().requires_grad_(k in pt.trainable_names(w)) for k, v in w.items()}
    act, ptr, stats = pt.forward_train(wt, image, vector)
    la, lp = weighted_losses(act, ptr, target_act, target_ptr, sample_weight)
    (la + lp).backward()
    grads = {k: (wt[k].grad.detach() if wt[k].grad is not None else torch.zeros_like(wt[k])) for k in pt.trainable_names(w)}
    return (float((la + lp).detach()), float(la.detach()), float(lp.detach())), grads, stats


def fit(w, opt, image, vector, target_act, target_ptr, sample_weight):
    """pt.fit with per-sample weights: one step in place on ``w``; returns the weighted pre-update losses."""
    losses, grads, stats = loss_and_grads(w, image, vector, target_act, target_ptr, sample_weight)
    for bn, (mean, var, _) in stats.items():
        w[bn + "/mean"] = w[bn + "/mean"] * pt.BN_MOMENTUM + mean * (1.0 - pt.BN_MOMENTUM)
        w[bn + "/var"] = w[bn + "/var"] * pt.BN_MOMENTUM + var * (1.0 - pt.BN_MOMENTUM)
    opt.step(w, grads)
    return losses
