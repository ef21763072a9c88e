"""Double DQN targets of ``ofb_trainer_td_targets_double`` (include/ofb_train.h) and the target network's soft update,
restated on the host -- TEST INFRASTRUCTURE.

The online network's predictions on the next observation select, the target network's evaluate:
  a* = 1 if act_online[1] > act_online[0] else 0                      (ties to 0)
  p* = the first flat index of the online map's maximum over its non-NaN entries, 0 when it has none.
The selected target values then go through ``oracle.policy_train_torch.td_targets`` -- the single-network targets, whose max
over a map holding only the selected value is that value -- one sample at a time, so that a per-sample discount can stand in
for gamma.  Every rounding is fp32 and one at a time, as on the device."""
import numpy as np
import torch

from oracle import policy_train_torch as ptt


def select_act(act_online):
    """-> a* int [B] of act_online [B, 2]."""
    a = torch.as_tensor(act_online, dtype=torch.float32)
    return (a[:, 1] > a[:, 0]).to(torch.int64)


def select_ptr(ptr_online):
    """-> p* int [B]: the first flat index (row-major, as stored) of each map's maximum over its non-NaN entries."""
    m = np.asarray(torch.as_tensor(ptr_online, dtype=torch.float32).reshape(ptr_online.shape[0], -1))
    out = []
    for row in m:
        ok = ~np.isnan(row)
        if not ok.any():
            out.append(0)
            continue
        out.append(int(np.flatnonzero(ok & (row == row[ok].max()))[0]))
    return torch.tensor(out, dtype=torch.int64)


def td_targets_double(act_obs, ptr_obs, act_on, ptr_on, act_tg, ptr_tg, iaction, pointer, reward, done, gamma=ptt.GAMMA,
                      discount=None):
    """-> (t_act [B,2], t_ptr [B,400,400], td_act [B], td_ptr [B]); every input a CPU tensor in the ABI's layout."""
    B = act_obs.shape[0]
    a_star, p_star = select_act(act_on), select_ptr(ptr_on)
    v_act = act_tg[torch.arange(B), a_star]
    v_ptr = ptr_tg.reshape(B, -1)[torch.arange(B), p_star]
    t_act, t_ptr = act_obs.clone(), ptr_obs.clone()
    for b in range(B):
        g = float(discount[b]) if discount is not None else gamma
        ta, tp = ptt.td_targets(act_obs[b:b + 1], ptr_obs[b:b + 1], v_act[b].repeat(1, 2), v_ptr[b].reshape(1, 1),
                                iaction[b:b + 1], pointer[b:b + 1], reward[b:b + 1], done[b:b + 1], gamma=g)
        t_act[b], t_ptr[b] = ta[0], tp[0]
    rows = torch.arange(B)
    ia, px, py = iaction.long(), pointer[:, 0].long(), pointer[:, 1].long()
    td_act = t_act[rows, ia] - act_obs[rows, ia]
    td_ptr = t_ptr[rows, px, py] - ptr_obs[rows, px, py]
    return t_act, t_ptr, td_act, td_ptr


def blend(weights, target, tau):
    """theta- <- tau * theta + (1 - tau) * theta- in numpy fp32, tau and 1 - tau rounded to fp32 once."""
    a, b = np.float32(tau), np.float32(1.0 - float(tau))
    return {k: a * np.asarray(weights[k], dtype=np.float32) + b * np.asarray(target[k], dtype=np.float32) for k in weights}
