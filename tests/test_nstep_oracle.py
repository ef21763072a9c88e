"""The n-step oracle (tests/nstep_oracle.py) pinned on hand-built scenes -- CPU only.

Frames 0..T of one or a few arenas are written out by hand (alive, episode, pending reward), and the expected windows are
stated from the rules of include/ofb_replay.h: a death ends a window with done = 1, a restart (full or masked) truncates it
and bootstraps from the episode's last observation, the ring and the newest n - 1 frames bound the candidates."""
import numpy as np
import pytest
import torch

from tests import nstep_oracle as no

G = 0.9


def _scene(T, A=1, P=1, deaths=(), restarts=(), rewards=None):
    """alive / episode / reward for frames 0..T.  deaths: (frame, a, p) = dead from that frame on (until its arena's next
    restart); restarts: (frame, arenas or None) = the episode counter increments at that frame and the ships live again."""
    alive = np.ones((T + 1, A, P), dtype=bool)
    episode = np.zeros((T + 1, A), dtype=np.int64)
    for f, arenas in sorted(restarts):
        for a in (range(A) if arenas is None else arenas):
            episode[f:, a] += 1
    for f, a, p in deaths:
        for t in range(f, T + 1):
            if t > f and episode[t, a] != episode[f, a]:
                break
            alive[t, a, p] = False
    reward = np.zeros((T + 1, A, P), dtype=np.float32) if rewards is None else np.asarray(rewards, dtype=np.float32)
    return alive, episode, reward


def _one_step_expected(alive, episode, reward, frames):
    """test_gpu_replay._expected restated on arrays: [(t, a, p, reward, done)] for t in `frames`."""
    out = []
    for t in frames:
        for a in range(alive.shape[1]):
            for p in range(alive.shape[2]):
                if alive[t, a, p] and episode[t, a] == episode[t + 1, a]:
                    out.append((t, a, p, float(reward[t + 1, a, p]), 0 if alive[t + 1, a, p] else 1))
    return out


def _by_t(exp):
    return {(t, a, p): (R, done, d, k) for t, a, p, R, done, d, k in exp}


@pytest.mark.parametrize("n", [2, 3, 5])
def test_a_death_at_each_j_ends_the_window_there(n):
    T = 20
    for j in range(n):
        t0 = 4
        alive, episode, reward = _scene(T, deaths=[(t0 + j + 1, 0, 0)])    # dead at t0+j+1: done1[t0+j]
        reward[t0 + j + 1, 0, 0] = 2.0
        got = _by_t(no.expected(alive, episode, reward, n, G))
        R, done, d, k = got[(t0, 0, 0)]
        assert (k, done) == (j + 1, 1)
        assert d == np.float32(G) ** np.float32(k) or abs(float(d) - G ** k) < 1e-6
        assert float(R) == pytest.approx(2.0 * G ** j, rel=1e-6)
        # no transition from a dead ship
        assert all(t <= t0 + j for (t, _, _) in got)


@pytest.mark.parametrize("n", [3, 5])
def test_full_and_masked_restarts_truncate_and_bootstrap(n):
    T, A = 30, 2
    alive, episode, reward = _scene(T, A=A, restarts=[(10, None), (20, [0])])
    reward[:, :, 0] = 1.0
    got = _by_t(no.expected(alive, episode, reward, n, G))
    # full restart at frame 10: frame 9 has no transition; frame 9 - j's window ends at s_9 after k = j frames
    assert (9, 0, 0) not in got and (9, 1, 0) not in got
    for j in range(1, n):
        for a in range(A):
            R, done, d, k = got[(9 - j, a, 0)]
            assert (k, done) == (j, 0), (j, a)
    # masked restart of arena 0 at frame 20: only arena 0 is truncated
    assert (19, 0, 0) not in got and (19, 1, 0) in got
    assert got[(18, 0, 0)][3] == 1 and got[(18, 1, 0)][3] == n
    assert got[(19 - n, 0, 0)][3] == n and got[(19 - n, 0, 0)][1] == 0 and got[(20 - n, 0, 0)][3] == n - 1
    # the window never spans a restart
    for (t, a, p), (_, _, _, k) in got.items():
        assert episode[t, a] == episode[t + k, a]


def test_ring_and_newest_frames_bound_the_candidates():
    T = 15
    alive, episode, reward = _scene(T, A=2, P=2)
    for n, D in [(3, 4), (3, 6), (1, 2), (2, 16)]:
        exp = no.expected(alive, episode, reward, n, G, depth=D)
        frames = sorted({e[0] for e in exp})
        assert frames == list(range(max(0, T - D + 1), T - n + 1)), (n, D)
        assert [e[:3] for e in exp] == sorted(e[:3] for e in exp)                 # oldest frame first, then arena, ship
    # a window cut by the ring: its frames still exist (t + k <= T), only t is bounded
    exp = no.expected(alive, episode, reward, 3, G, depth=4)
    assert all(t + k <= T for t, *_, k in exp)


def test_n1_is_the_one_step_memory():
    rng = np.random.default_rng(3)
    T, A, P = 25, 3, 2
    alive, episode, reward = _scene(T, A=A, P=P, deaths=[(5, 0, 1), (12, 2, 0), (18, 1, 1)], restarts=[(9, None), (16, [1])],
                                    rewards=rng.integers(0, 3, size=(26, 3, 2)))
    exp = no.expected(alive, episode, reward, 1, G)
    one = _one_step_expected(alive, episode, reward, range(T))
    assert [(t, a, p, float(R), done) for t, a, p, R, done, _, _ in exp] == one
    assert all(d == np.float32(G) and k == 1 for *_, d, k in exp)
    # and with a ring of depth D: the last D - 1 frames
    exp = no.expected(alive, episode, reward, 1, G, depth=6)
    assert [(t, a, p, float(R), done) for t, a, p, R, done, _, _ in exp] == _one_step_expected(alive, episode, reward, range(T - 5, T))


def test_return_is_the_fp32_loop_and_the_discounted_sum():
    rng = np.random.default_rng(7)
    T, n = 40, 5
    rewards = rng.standard_normal((T + 1, 4, 1)).astype(np.float32) * 3
    alive, episode, reward = _scene(T, A=4, deaths=[(17, 1, 0), (30, 3, 0)], restarts=[(25, [0, 2])], rewards=rewards)
    valid1, r, done1 = no.one_step_fields(alive, episode, reward)
    g = np.float32(0.97)
    kinds = set()
    for t, a, p, R, done, d, k in no.expected(alive, episode, reward, n, 0.97):
        loop = r[t + k - 1, a, p]
        for j in range(k - 2, -1, -1):
            loop = np.float32(r[t + j, a, p] + np.float32(g * loop))
        assert np.float32(R).view(np.uint32) == np.float32(loop).view(np.uint32)
        exact = sum(float(g) ** j * float(r[t + j, a, p]) for j in range(k))
        scale = sum(abs(float(g) ** j * float(r[t + j, a, p])) for j in range(k))
        assert abs(float(R) - exact) <= 4 * k * np.finfo(np.float32).eps * scale + 1e-30
        assert abs(float(d) - float(g) ** k) <= k * np.finfo(np.float32).eps * float(g) ** k
        kinds.add("death" if done else ("full" if k == n else "truncated"))
    assert kinds == {"death", "full", "truncated"}


def test_discounted_target_with_gamma_is_the_oracles_target():
    from oracle import policy_train_torch as pt
    g = torch.Generator().manual_seed(4)
    B = 6
    act_o, act_n = torch.randn((B, 2), generator=g), torch.randn((B, 2), generator=g)
    ptr_o, ptr_n = torch.randn((B, 400, 400), generator=g), torch.randn((B, 400, 400), generator=g)
    ia = torch.tensor([0, 1, 1, 0, 1, 0], dtype=torch.int32)
    pointer = torch.tensor([[10, 20], [399, 0], [7, 7], [0, 399], [200, 123], [55, 301]], dtype=torch.int32)
    reward = torch.tensor([2.0, 0.0, 3.5, -1.0, 0.0, 1.0])
    done = torch.tensor([0, 1, 0, 1, 0, 0], dtype=torch.uint8)
    ta, tp = pt.td_targets(act_o, ptr_o, act_n, ptr_n, ia, pointer, reward, done, gamma=pt.GAMMA)
    for b in range(B):
        x, y = int(pointer[b, 0]), int(pointer[b, 1])
        want_a = no.td_target(reward[b].item(), pt.GAMMA, int(done[b]), act_n[b].max().item())
        want_p = no.td_target(reward[b].item(), pt.GAMMA, int(done[b]), ptr_n[b].max().item())
        assert np.float32(ta[b, int(ia[b])].item()).view(np.uint32) == want_a.view(np.uint32)
        assert np.float32(tp[b, x, y].item()).view(np.uint32) == want_p.view(np.uint32)
