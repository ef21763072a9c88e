"""N-step returns of the device replay memory (include/ofb_replay.h, ofb_train.h; replay.py, trainer.py) -- runs on the B200 box.

Every check compares with what the run itself produced, kept aside frame by frame by tests/test_gpu_replay.py's recording
driver (the maps the frame kernel wrote, bg.obs_vec, the played actions, ship_alive and episode), through the host restatement
of tests/nstep_oracle.py: which transitions exist, their window length k, done, the return R and the discount, bit for bit."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

from tests import nstep_oracle as no
from tests.test_gpu_replay import _drive

pytestmark = pytest.mark.gpu

G = 0.9


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _oracle(rec, n, gamma=G, depth=None):
    alive = np.stack([r["alive"].numpy() for r in rec])
    episode = np.stack([r["episode"].numpy() for r in rec])
    reward = np.stack([r["vec"][:, :, 0].cpu().numpy() for r in rec])
    return no.expected(alive, episode, reward, n, gamma, depth=depth)


def _bits(x):
    return np.asarray(x, dtype=np.float32).view(np.uint32)


def _check(mem, rec, exp, positions=None):
    """gather of `positions` (default: all) against the oracle's transitions and the run's own maps and fields."""
    positions = list(range(len(exp))) if positions is None else positions
    for lo in range(0, len(positions), 512):
        pos = positions[lo:lo + 512]
        g = mem.gather(pos)
        sel = [exp[i] for i in pos]
        assert torch.equal(g.maps_obs, torch.stack([rec[t]["maps"][a] for t, a, *_ in sel])), "maps_obs differ from frame t's"
        assert torch.equal(g.maps_next, torch.stack([rec[t + k]["maps"][a] for t, a, *_, k in sel])), "maps_next differ from t+k's"
        assert torch.equal(g.vec_obs, torch.stack([rec[t]["vec"][a, p] for t, a, p, *_ in sel]))
        assert torch.equal(g.vec_next, torch.stack([rec[t + k]["vec"][a, p] for t, a, p, *_, k in sel]))
        assert torch.equal(g.iaction, torch.stack([rec[t]["iact"][a, p] for t, a, p, *_ in sel]))
        assert torch.equal(g.pointer, torch.stack([rec[t]["xy"][a, p] for t, a, p, *_ in sel]))
        assert np.array_equal(_bits(g.reward.cpu().numpy()), _bits([e[3] for e in sel])), "R differs from the oracle's"
        assert np.array_equal(_bits(g.discount.cpu().numpy()), _bits([e[5] for e in sel]))
        assert g.done.cpu().tolist() == [e[4] for e in sel]
        assert g.steps.cpu().tolist() == [e[6] for e in sel]


def _bg(layout, N=64):
    from ofighters_b200 import ArenaConfig, BatchedBattleground
    if layout == "P1":
        return BatchedBattleground(N, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=3), 1
    return BatchedBattleground(N, ships={"QlearnIA": 7}, config=ArenaConfig(laser_cap=512), seed=4), 7


# ---------------------------------------------------------------------------------------------- 1. windows, maps, returns
@pytest.mark.parametrize("layout", ["P1", "policy7"])
@pytest.mark.parametrize("n", [3, 5])
def test_nstep_windows_gather_the_runs_own_frames(n, layout):
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    N, T = 64, 40
    bg, P = _bg(layout, N)
    pol = PolicyB200.random_init(max_ships=N * P, seed=1)
    mem = DeviceReplayMemory(bg, depth=T + 2, n_step=n)
    mask = torch.arange(N) % 2 == 0
    rec = _drive(bg, mem, pol, T, restarts={15: None, 27: mask})
    exp = _oracle(rec, n)
    assert len(mem) == len(exp) and mem.frames == T
    assert max(t for t, *_ in exp) == T - 1 - n                       # the newest n frames are not candidates yet
    kinds = set()
    for t, a, p, R, done, d, k in exp:
        if done:
            kinds.add("death")
        elif k == n:
            kinds.add("full")
        elif t + k == 14:
            kinds.add("full restart")
        elif t + k == 26 and a % 2 == 0:
            kinds.add("masked restart")
    assert kinds == {"death", "full", "full restart", "masked restart"}, kinds
    _check(mem, rec, exp)


# ---------------------------------------------------------------------------------------------- 2. ring wrap
@pytest.mark.parametrize("extra", [1, 3])
def test_ring_keeps_frames_t_minus_depth_plus_one_to_t_minus_n(extra):
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    n = 3
    D, T = n + extra, 14
    bg = BatchedBattleground(16, ships={"QlearnIA": 1, "turret": 6}, seed=8)
    mem = DeviceReplayMemory(bg, depth=D, n_step=n)
    rec = _drive(bg, mem, PolicyB200.random_init(max_ships=16), T, restarts={9: None})
    exp = _oracle(rec, n, depth=D)
    assert len(mem) == len(exp) > 0
    assert {t for t, *_ in exp} <= set(range(T - D, T - n))
    _check(mem, rec, exp)


# ---------------------------------------------------------------------------------------------- 3. n = 1, refusal
def test_gather_nstep_on_a_one_step_memory_is_gather():
    from ofighters_b200 import BatchedBattleground, OfbError, _lib
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    bg = BatchedBattleground(32, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=5)
    mem = DeviceReplayMemory(bg, depth=12)
    _drive(bg, mem, PolicyB200.random_init(max_ships=32), 16, restarts={7: None})
    n = len(mem)
    g = mem.gather(range(n))
    lib = _lib.load()
    ids = mem._ids[:n].contiguous()
    out = {k: torch.empty_like(getattr(g, k)) for k in ("maps_obs", "vec_obs", "maps_next", "vec_next", "iaction", "pointer",
                                                          "reward", "done")}
    disc = torch.empty(n, dtype=torch.float32, device="cuda")
    steps = torch.empty(n, dtype=torch.int32, device="cuda")
    _lib.check(lib.ofb_replay_gather_nstep(mem._h, _p(ids), n, G, *[_p(out[k]) for k in ("maps_obs", "vec_obs", "maps_next",
                                           "vec_next", "iaction", "pointer", "reward", "done")], _p(disc), _p(steps), None))
    torch.cuda.synchronize()
    for k, v in out.items():
        assert torch.equal(v, getattr(g, k)), k
    assert bool((disc == np.float32(G)).all()) and bool((steps == 1).all())
    # an n-step handle refuses the one-step gather
    mem3 = DeviceReplayMemory(bg, depth=6, n_step=3)
    with pytest.raises(OfbError, match="gather_nstep"):
        _lib.check(lib.ofb_replay_gather(mem3._h, _p(ids), 1, None, None, None, None, None, None, None, None, None))


# ---------------------------------------------------------------------------------------------- 4. discounted TD kernels
def test_discounted_td_kernels():
    from ofighters_b200 import _lib
    lib = _lib.load()
    B = 64
    g = torch.Generator().manual_seed(13)
    act_o, act_n = torch.randn((B, 2), generator=g), torch.randn((B, 2), generator=g)
    ptr_o, ptr_n = torch.randn((B, 400, 400), generator=g), torch.randn((B, 400, 400), generator=g)
    ia = torch.randint(0, 2, (B,), generator=g, dtype=torch.int32)
    pointer = torch.randint(0, 400, (B, 2), generator=g, dtype=torch.int32)
    reward = torch.randn((B,), generator=g) * 2
    done = (torch.rand((B,), generator=g) < 0.3).to(torch.uint8)
    d = [t.cuda() for t in (act_o, ptr_o, act_n, ptr_n, ia, pointer, reward, done)]
    args = [_p(t) for t in d]

    def run(disc):
        ta, tp = torch.empty_like(d[0]), torch.empty_like(d[1])
        ea, ep = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
        if disc is None:
            _lib.check(lib.ofb_trainer_td_errors(*args, G, B, _p(ea), _p(ep), None))
            _lib.check(lib.ofb_trainer_td_targets(*args, G, B, _p(ta), _p(tp), None))
        else:
            _lib.check(lib.ofb_trainer_td_errors_discounted(*args, _p(disc), B, _p(ea), _p(ep), None))
            _lib.check(lib.ofb_trainer_td_targets_discounted(*args, _p(disc), B, _p(ta), _p(tp), None))
        torch.cuda.synchronize()
        return ta.cpu(), tp.cpu(), ea.cpu(), ep.cpu()

    scalar = run(None)
    same = run(torch.full((B,), G, dtype=torch.float32, device="cuda"))
    for x, y in zip(scalar, same):
        assert torch.equal(x, y)
    disc = torch.rand((B,), generator=g) ** 3
    ta, tp, ea, ep = run(disc.cuda())
    for b in range(B):
        x, y, i = int(pointer[b, 0]), int(pointer[b, 1]), int(ia[b])
        want_a = no.td_target(reward[b].item(), disc[b].item(), int(done[b]), act_n[b].max().item())
        want_p = no.td_target(reward[b].item(), disc[b].item(), int(done[b]), ptr_n[b].max().item())
        assert _bits(ta[b, i].item()) == want_a.view(np.uint32) and _bits(tp[b, x, y].item()) == want_p.view(np.uint32)
        assert torch.equal(ea[b], ta[b, i] - act_o[b, i]) and torch.equal(ep[b], tp[b, x, y] - ptr_o[b, x, y])
        # the untouched entries are the predictions
        assert ta[b, 1 - i] == act_o[b, 1 - i]


# ---------------------------------------------------------------------------------------------- 5. prioritized + n-step
def test_prioritized_nstep_draws_candidates_and_sets_entry_masses():
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import PrioritizedReplayMemory
    from tests.test_gpu_prioritized_replay import _age_positions
    n, N, D, T = 3, 64, 12, 30
    bg = BatchedBattleground(N, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=3)
    mem = PrioritizedReplayMemory(bg, depth=D, alpha=0.6, seed=2, n_step=n)
    pol = PolicyB200.random_init(max_ships=N, seed=1)
    # entry masses: frame T - n gets the maximum mass of the push of T, while updates keep raising it
    maps = bg.raster("bits")
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(T):
        if t in (12, 21):
            bg.restart()
            bg.raster("bits", out=maps)
        mx = float(mem.max_mass())
        mem.push(*pol.act(bg, maps, epsilon=0.5))
        if t >= n:
            s = (t - n) % D
            assert bool((mem.masses()[s * N:(s + 1) * N] == mx).all()), t
        if len(mem) > 0:
            smp = mem.sample_prioritized(8, 0.5)
            mem.update_priorities(smp.ids, torch.rand(8, device="cuda", generator=gen) * (t + 2), torch.zeros(8, device="cuda"))
        bg.frame(maps=maps)
    assert float(mem.max_mass()) > 1.0
    # draws: only oracle transitions, never a frame newer than T - n
    rec = _drive(bg, mem, pol, D + 4, restarts={6: None})
    exp = _oracle(rec, n, depth=D)
    pos, ids = _age_positions(mem)
    assert len(mem) == len(exp) == ids.numel()
    newest = (mem.frames - 1) % D
    too_new = {(newest - i) % D for i in range(n)}
    for k in range(20):
        s = mem.sample_prioritized(256, 0.4)
        assert int(mem._n_valid.item()) == len(mem)
        p = pos[s.ids.long()]
        assert bool((p >= 0).all()), "a drawn id is not a candidate"
        assert not any(int(i) // N in too_new for i in s.ids.tolist())
        if k == 0:
            _check_sample(s, rec, [exp[i] for i in p.tolist()])


def _check_sample(g, rec, sel):
    assert torch.equal(g.maps_next, torch.stack([rec[t + k]["maps"][a] for t, a, *_, k in sel]))
    assert np.array_equal(_bits(g.reward.cpu().numpy()), _bits([e[3] for e in sel]))
    assert g.steps.cpu().tolist() == [e[6] for e in sel] and g.done.cpu().tolist() == [e[4] for e in sel]


# ---------------------------------------------------------------------------------------------- 6. replay == hand pipeline
def test_replay_on_an_nstep_memory_is_the_hand_pipeline():
    from oracle import policy_torch as po
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    from ofighters_b200.trainer import TrainerB200
    bg = BatchedBattleground(32, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=21)
    mem = DeviceReplayMemory(bg, depth=40, n_step=3)
    rec = _drive(bg, mem, PolicyB200.random_init(max_ships=32, seed=2), 36, restarts={24: None})
    exp = _oracle(rec, 3)
    n = len(mem)
    assert n == len(exp) > 8
    w = po.init_weights(6, randomize_bn=True)
    a, b = TrainerB200(weights=w, learning_rate=1e-4, batch_size=8), TrainerB200(weights=w, learning_rate=1e-4, batch_size=8)
    random.seed(7)
    ha = a.replay(8, memory=mem)
    random.seed(7)
    pos = random.sample(range(n), 8)
    g = mem.gather(pos)
    act_o, ptr_o = b.predict(g.maps_obs, g.vec_obs)
    act_n, ptr_n = b.predict(g.maps_next, g.vec_next)
    ta, tp = act_o.cpu().clone(), ptr_o.cpu().clone()
    an, pn = act_n.cpu(), ptr_n.cpu()
    for i, e in enumerate(exp[q] for q in pos):
        _, _, _, R, done, d, _ = e
        x, y = g.pointer[i].tolist()
        ta[i, int(g.iaction[i])] = float(no.td_target(R, d, done, an[i].max().item()))
        tp[i, x, y] = float(no.td_target(R, d, done, pn[i].max().item()))
    dev = [t.clone() for t in (act_o, ptr_o)]
    b._td_targets(dev[0], dev[1], act_n, ptr_n, g.iaction, g.pointer, g.reward, g.done, g.discount, 8)
    assert torch.equal(dev[0].cpu(), ta) and torch.equal(dev[1].cpu(), tp)            # the device targets are the oracle's
    lb = b.fit(g.maps_next, g.vec_next, ta.cuda(), tp.cuda()).cpu().tolist()
    assert ha.history["loss"][0] == pytest.approx(lb[0], rel=1e-5)
    wa, wb = a.get_weights(), b.get_weights()
    for k in wa:                                          # tolerances of test_transitions_equal_qlearners_memory_and_replay_matches
        noise_driven = k.endswith("/bias") and "conv" in k and k != "upconv4/bias"
        diff = (wa[k] - wb[k]).abs()
        assert float(diff.max()) <= 2.2e-4, k
        if not noise_driven:
            assert float((diff <= 2e-6 + 1e-5 * float(wb[k].abs().max())).float().mean()) >= 0.999, k


# ---------------------------------------------------------------------------------------------- 7. BatchedQLearner
@pytest.mark.parametrize("prioritized", [False, True])
def test_batched_qlearner_with_an_nstep_memory(prioritized):
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory
    from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200
    random.seed(1)
    bg = BatchedBattleground(64, ships={"QlearnIA": 1, "random": 6}, seed=21)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=8, max_ships=64)
    mem = PrioritizedReplayMemory(bg, depth=16, n_step=3, seed=4) if prioritized else DeviceReplayMemory(bg, depth=16, n_step=3)
    bq = BatchedQLearner(tr, mem, replay_every=20, collecting_steps=20, snapshot=0)
    maps = bg.raster("bits")
    replays = []
    for t in range(120):
        if t == 70:
            bg.restart()
            bg.raster("bits", out=maps)
            bq.reset()
        _, _, rep = bq.act(bg, maps)
        bg.frame(maps=maps)
        if rep:
            replays.append(bq.total_steps)
    assert replays == list(range(20, 121, 20)) and tr.steps == 6
    assert len(bq.losses) == 6 and all(np.isfinite(bq.losses))


# ---------------------------------------------------------------------------------------------- 8. bad arguments
def test_bad_arguments_raise():
    from ofighters_b200 import BatchedBattleground, OfbError, _lib
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory
    from ofighters_b200.trainer import TrainerB200
    bg = BatchedBattleground(8, ships={"QlearnIA": 1, "random": 6}, seed=2)
    for kw in (dict(n_step=0), dict(depth=3, n_step=3), dict(depth=2, n_step=2)):
        with pytest.raises(Exception, match="Invalid n_step"):
            DeviceReplayMemory(bg, **kw)
    with pytest.raises(Exception, match="Invalid n_step"):
        PrioritizedReplayMemory(bg, depth=4, n_step=4)
    lib = _lib.load()
    plain = DeviceReplayMemory(bg, depth=4)
    with pytest.raises(OfbError, match="depth - 1"):
        _lib.check(lib.ofb_replay_set_n_step(plain._h, 4))
    with pytest.raises(OfbError, match="depth - 1"):
        _lib.check(lib.ofb_replay_set_n_step(plain._h, 0))
    pol = PolicyB200.random_init(max_ships=8)
    maps = bg.raster("bits")
    plain.push(*pol.act(bg, maps))
    with pytest.raises(OfbError, match="first push"):
        _lib.check(lib.ofb_replay_set_n_step(plain._h, 2))
    mem = DeviceReplayMemory(bg, depth=8, n_step=3, gamma=0.99)
    for _ in range(6):
        mem.push(*pol.act(bg, maps))
        bg.frame(maps=maps)
    assert len(mem) > 0
    tr = TrainerB200(batch_size=8, max_ships=8)
    with pytest.raises(Exception, match="Invalid memory"):
        tr.replay(4, memory=mem)
    pmem = PrioritizedReplayMemory(bg, depth=8, n_step=2, gamma=0.5)
    with pytest.raises(Exception, match="Invalid memory"):
        tr.replay(4, memory=pmem, beta=0.5)
