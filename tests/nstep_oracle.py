"""N-step transitions of the device replay memory (include/ofb_replay.h, "N-step returns"), restated on the host -- TEST
INFRASTRUCTURE.

Input: what a run records frame by frame for frames 0..T (T = the newest pushed frame): ``alive`` bool [F, A, P], the arenas'
``episode`` counters [F, A] and the ships' pending ``reward`` [F, A, P] (obs_vec[0]).  From them the one-step fields of frame t:
valid1[t] = alive at t and the same episode at t and t+1, r[t] = the pending reward at t+1, done1[t] = dead at t+1.  The window of
transition (t, a, p) walks j = 0, 1, ...: a death at t+j ends it with done = 1 after k = j + 1 frames; j + 1 = n ends it at
k = n; otherwise the end of the episode after frame t+j+1 ends it at k = j + 1 (a truncation: bootstrap from s_{t+j+1}).
R and the discount are computed in np.float32 one rounding at a time, as the device does without fma."""
import numpy as np


def one_step_fields(alive, episode, reward):
    """-> valid1, r, done1 of frames 0..F-2, each [F-1, A, P]."""
    alive = np.asarray(alive, dtype=bool)
    episode = np.asarray(episode)
    reward = np.asarray(reward, dtype=np.float32)
    valid1 = alive[:-1] & (episode[:-1] == episode[1:])[:, :, None]
    return valid1, reward[1:], ~alive[1:]


def window(valid1, r, done1, t, a, p, n, gamma):
    """-> (k, done, R, discount) of transition (t, a, p); frames t .. t+n-1 must have their one-step fields."""
    k, done = n, 0
    for j in range(n):
        if done1[t + j, a, p]:
            k, done = j + 1, 1
            break
        if j + 1 == n:
            break
        if not valid1[t + j + 1, a, p]:
            k = j + 1
            break
    g = np.float32(gamma)
    R = np.float32(r[t + k - 1, a, p])
    for j in range(k - 2, -1, -1):
        R = np.float32(r[t + j, a, p] + np.float32(g * R))
    d = g
    for _ in range(1, k):
        d = np.float32(d * g)
    return k, done, R, d


def expected(alive, episode, reward, n, gamma, depth=None):
    """[(t, a, p, R, done, discount, k)] of an n-step memory after frames 0..T were pushed, in its order (oldest frame first,
    then arena, then ship).  ``depth``: the ring's, which keeps the frames [T - depth + 1, T - n] (default: all of them)."""
    valid1, r, done1 = one_step_fields(alive, episode, reward)
    T = len(alive) - 1
    first = 0 if depth is None else max(0, T - depth + 1)
    A, P = valid1.shape[1], valid1.shape[2]
    out = []
    for t in range(first, T - n + 1):
        for a in range(A):
            for p in range(P):
                if valid1[t, a, p]:
                    k, done, R, d = window(valid1, r, done1, t, a, p, n, gamma)
                    out.append((t, a, p, R, done, d, k))
    return out


def td_target(reward, discount, done, max_next):
    """The discounted target's fp32 expression, one rounding at a time: r + (discount * max) * keep."""
    keep = np.float32(0.0 if done else 1.0)
    return np.float32(np.float32(reward) + np.float32(np.float32(np.float32(discount) * np.float32(max_next)) * keep))
