"""Device-resident replay memory (include/ofb_replay.h, ofighters_b200/replay.py) and BatchedQLearner -- runs on the B200 box.

Every check compares with what the run itself produced, kept aside frame by frame: the maps the fused frame kernel wrote,
bg.obs_vec, the actions act() played, the ship_alive / episode fields of the state.  From those the host derives the expected
transitions with QlearnIA.play's rules (agents/qlearnIA_V2.py:372-401): one per policy ship alive at t whose arena is still in
the same episode at t+1, reward = the head's reward at t+1, done = dead at t+1; oldest frame first, then arena, then ship."""
import random

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _drive(bg, mem, actor, frames, restarts=(), eps=0.5, keep_maps=None):
    """Run `frames` frames: [restart] -> keep the observation -> act -> push -> fused frame.  `restarts`: {t: mask or None}.
    keep_maps: arena indices whose maps are kept (default: all)."""
    ships = mem.ships
    policy = [i for i, b in enumerate(bg.behaviors) if b in ("QlearnIA", "external")]
    cols = [policy.index(s) for s in ships]
    maps = bg.raster("bits")
    rec = []
    for t in range(frames):
        if t in restarts:
            bg.restart(mask=restarts[t])
            bg.raster("bits", out=maps)
        st = bg.state(("ship_alive", "episode"))
        kept = maps.clone() if keep_maps is None else maps.index_select(0, keep_maps)
        r = dict(maps=kept, vec=bg.obs_vec[:, ships, :].clone(), alive=st["ship_alive"][:, ships].cpu(),
                 episode=st["episode"].cpu())
        iact, xy = actor.act(bg, maps, epsilon=eps)
        mem.push(iact, xy)
        n, P = bg.n_arenas, len(policy)
        r["iact"] = iact.reshape(n, P)[:, cols].clone()
        r["xy"] = xy.reshape(n, P, 2)[:, cols].clone()
        rec.append(r)
        bg.frame(maps=maps)
    return rec


def _expected(rec, track, frames):
    """[(t, a, p, reward, done)] for t in `frames` (each must have a successor in rec), in the memory's order."""
    out = []
    for t in frames:
        alive, nxt = rec[t]["alive"], rec[t + 1]
        P = alive.shape[1]
        same = (rec[t]["episode"] == nxt["episode"]).tolist()
        al, al1 = alive.tolist(), nxt["alive"].tolist()
        rew = nxt["vec"][:, :, 0].cpu().tolist()
        for a in range(track):
            for p in range(P):
                if al[a][p] and same[a]:
                    out.append((t, a, p, rew[a][p], 0 if al1[a][p] else 1))
    return out


def _check(mem, rec, exp, positions=None, map_row=None):
    """Gather `positions` (default: all) and compare with the expected transitions exp[positions]."""
    positions = list(range(len(exp))) if positions is None else positions
    map_row = map_row or (lambda a: a)
    for lo in range(0, len(positions), 512):
        pos = positions[lo:lo + 512]
        g = mem.gather(pos)
        sel = [exp[i] for i in pos]
        mo = torch.stack([rec[t]["maps"][map_row(a)] for t, a, p, _, _ in sel])
        mn = torch.stack([rec[t + 1]["maps"][map_row(a)] for t, a, p, _, _ in sel])
        vo = torch.stack([rec[t]["vec"][a, p] for t, a, p, _, _ in sel])
        vn = torch.stack([rec[t + 1]["vec"][a, p] for t, a, p, _, _ in sel])
        ia = torch.stack([rec[t]["iact"][a, p] for t, a, p, _, _ in sel])
        pt = torch.stack([rec[t]["xy"][a, p] for t, a, p, _, _ in sel])
        assert torch.equal(g.maps_obs, mo), "maps_obs differ from the frame's maps"
        assert torch.equal(g.maps_next, mn), "maps_next differ from the frame's maps"
        assert torch.equal(g.vec_obs, vo) and torch.equal(g.vec_next, vn)
        assert torch.equal(g.iaction, ia) and torch.equal(g.pointer, pt)
        assert g.reward.cpu().tolist() == [e[3] for e in sel]
        assert g.done.cpu().tolist() == [e[4] for e in sel]


@pytest.mark.parametrize("layout", ["P1", "policy7"])
def test_snapshots_rasterise_to_the_frames_maps_and_follow_the_rules(layout):
    from ofighters_b200 import ArenaConfig, BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    N, T = 64, 30
    if layout == "P1":
        bg = BatchedBattleground(N, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=3)
    else:
        bg = BatchedBattleground(N, ships={"QlearnIA": 7}, config=ArenaConfig(laser_cap=512), seed=4)
    P = len(bg.behaviors) if layout == "policy7" else 1
    pol = PolicyB200.random_init(max_ships=N * P, seed=1)
    mem = DeviceReplayMemory(bg, depth=T + 2)
    assert mem.ships == list(range(P)) and len(mem) == 0
    mask = torch.arange(N) % 2 == 0
    rec = _drive(bg, mem, pol, T, restarts={12: None, 21: mask})
    exp = _expected(rec, N, range(T - 1))
    assert len(mem) == len(exp) and mem.frames == T
    # no transition spans a restart (the full one at 12, the masked one at 21 for the even arenas only)
    assert not any(t == 11 for t, *_ in exp) and not any(t == 20 and a % 2 == 0 for t, a, *_ in exp)
    assert any(t == 20 and a % 2 == 1 for t, a, *_ in exp)
    # each death once, done = 1; none from a dead ship
    deaths = sum(1 for t in range(T - 1) for a in range(N) for p in range(P)
                 if rec[t]["alive"][a, p] and not rec[t + 1]["alive"][a, p] and rec[t]["episode"][a] == rec[t + 1]["episode"][a])
    assert deaths > 0 and sum(e[4] for e in exp) == deaths
    _check(mem, rec, exp)


def test_ring_keeps_the_last_depth_minus_one_frames():
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    bg = BatchedBattleground(16, ships={"QlearnIA": 1, "turret": 6}, seed=8)
    mem = DeviceReplayMemory(bg, depth=3)
    rec = _drive(bg, mem, PolicyB200.random_init(max_ships=16), 10)
    exp = _expected(rec, 16, [7, 8])
    assert len(mem) == len(exp) > 0
    _check(mem, rec, exp)


def test_transitions_equal_qlearners_memory_and_replay_matches():
    """QLearner(track=4) and DeviceReplayMemory(track=4) fed with the same played actions hold the same transitions in the same
    order; a replay drawn from each with the same `random` state reports the same loss and ends at the same weights."""
    from collections import deque
    from oracle import policy_torch as po
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.replay import DeviceReplayMemory
    from ofighters_b200.trainer import Epsilon_cos, QLearner, TrainerB200
    random.seed(1)
    bg = BatchedBattleground(32, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=21)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=8, max_ships=32, memory_size=100000)
    ql = QLearner(tr, track=4, replay_every=50, collecting_steps=20, snapshot=0)
    mem = DeviceReplayMemory(bg, depth=64, track=4)
    maps = bg.raster("bits")
    for t in range(60):
        if t == 40:
            bg.restart()
            bg.raster("bits", out=maps)
            ql.reset()
        iact, xy, _ = ql.act(bg, maps)
        mem.push(iact, xy)
        bg.frame(maps=maps)
    n = len(tr.memory)
    assert len(mem) == n > 40
    g = mem.gather(range(n))
    m = list(tr.memory)
    assert torch.equal(g.maps_obs, torch.stack([e[0][0] for e in m])) and torch.equal(g.vec_obs, torch.stack([e[0][1] for e in m]))
    assert g.iaction.tolist() == [e[1] for e in m] and [tuple(p) for p in g.pointer.tolist()] == [tuple(e[2]) for e in m]
    assert g.reward.tolist() == [float(e[3]) for e in m]
    assert torch.equal(g.maps_next, torch.stack([e[4][0] for e in m])) and torch.equal(g.vec_next, torch.stack([e[4][1] for e in m]))
    assert g.done.tolist() == [1 if e[5] else 0 for e in m]

    w = po.init_weights(6, randomize_bn=True)
    a, b = TrainerB200(weights=w, learning_rate=1e-4, batch_size=8), TrainerB200(weights=w, learning_rate=1e-4, batch_size=8)
    b.memory = deque(m)
    random.seed(7)
    ha = a.replay(8, memory=mem)
    random.seed(7)
    hb = b.replay(8)
    assert ha.history["loss"][0] == pytest.approx(hb.history["loss"][0], rel=1e-5)
    wa, wb = a.get_weights(), b.get_weights()
    for k in wa:                                          # tolerances of test_replay_is_the_references_sequence_of_calls
        noise_driven = k.endswith("/bias") and "conv" in k and k != "upconv4/bias"
        diff = (wa[k] - wb[k]).abs()
        assert float(diff.max()) <= 2.2e-4, k
        if not noise_driven:
            assert float((diff <= 2e-6 + 1e-5 * float(wb[k].abs().max())).float().mean()) >= 0.999, k


def test_full_size_ring_above_2_31_bytes():
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    N = 65536
    bg = BatchedBattleground(N, ships={"QlearnIA": 1, "random": 6}, seed=0x0F16)
    mem = DeviceReplayMemory(bg, depth=16)
    assert 16 * N * bg.state_stride > 2 ** 31 and mem.device_bytes > 16 * N * bg.state_stride
    g = torch.Generator().manual_seed(5)
    keep = torch.randperm(N, generator=g)[:2048].sort().values
    row = {a: i for i, a in enumerate(keep.tolist())}
    rec = _drive(bg, mem, PolicyB200.random_init(max_ships=N), 16, keep_maps=keep.cuda())
    exp = _expected(rec, N, range(15))
    assert len(mem) == len(exp)
    random.seed(3)
    kept = [i for i, e in enumerate(exp) if e[1] in row]
    _check(mem, rec, exp, positions=random.sample(kept, 256), map_row=lambda a: row[a])
    # heads, actions, rewards and done at random positions anywhere in the ring (the maps of all arenas are not kept)
    pos = random.sample(range(len(exp)), 256)
    got = mem.gather(pos)
    sel = [exp[i] for i in pos]
    assert torch.equal(got.vec_obs, torch.stack([rec[t]["vec"][a, 0] for t, a, *_ in sel]))
    assert torch.equal(got.vec_next, torch.stack([rec[t + 1]["vec"][a, 0] for t, a, *_ in sel]))
    assert torch.equal(got.pointer, torch.stack([rec[t]["xy"][a, 0] for t, a, *_ in sel]))
    assert got.done.tolist() == [e[4] for e in sel]


def test_batched_qlearner_loop():
    import tempfile
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.replay import DeviceReplayMemory
    from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200
    random.seed(1)
    bg = BatchedBattleground(32, ships={"QlearnIA": 1, "random": 6}, seed=21)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=8, max_ships=32, name="b")
    mem = DeviceReplayMemory(bg, depth=16)
    bq = BatchedQLearner(tr, mem, replay_every=50, collecting_steps=20, snapshot=1, snapshot_folder=tempfile.mkdtemp())
    w0 = tr.get_weights()
    maps = bg.raster("bits")
    replays, outside = [], 0
    for t in range(120):
        if t == 100:
            bg.restart()
            bg.raster("bits", out=maps)
            bq.reset()
        outside += 0 if bq.collecting else 1
        if t == 61:                                       # a frame without a replay never waits for the device
            torch.cuda.synchronize()
            torch.cuda.set_sync_debug_mode("error")
            try:
                _, _, rep = bq.act(bg, maps)
                bg.frame(maps=maps)
            finally:
                torch.cuda.set_sync_debug_mode(0)
        else:
            _, _, rep = bq.act(bg, maps)
            bg.frame(maps=maps)
        if rep:
            replays.append(bq.total_steps)
    assert replays == [50, 100] and tr.steps == 2 and len(bq.losses) == 2 and all(np.isfinite(bq.losses))
    assert tr.epsilon.t == outside == 120 - 19
    w1 = tr.get_weights()
    assert not torch.equal(w0["upconv4/kernel"], w1["upconv4/kernel"])
    assert torch.equal(tr.model.weights["dense2/kernel"], w1["dense2/kernel"])      # the inference engine holds the trained weights
    assert len(bq.saved) == 1 and bq.epsilons and bq.episode == 1


def test_bad_arguments_raise():
    from ofighters_b200 import BatchedBattleground, OfbError
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory
    from ofighters_b200.trainer import BatchedQLearner, TrainerB200
    bg = BatchedBattleground(8, ships={"QlearnIA": 1, "random": 6}, seed=2)
    other = BatchedBattleground(8, ships={"QlearnIA": 1, "random": 6}, seed=2)
    mem = DeviceReplayMemory(bg, depth=4)
    with pytest.raises(Exception, match="empty"):
        mem.sample(1)
    pol = PolicyB200.random_init(max_ships=8)
    maps = bg.raster("bits")
    iact, xy = pol.act(bg, maps)
    with pytest.raises(Exception, match="Invalid iaction"):
        mem.push(iact[:7], xy)
    with pytest.raises(Exception, match="Invalid iaction"):
        mem.push(iact.long(), xy)
    with pytest.raises(Exception, match="Invalid xy"):
        mem.push(iact, xy.reshape(-1))
    with pytest.raises(Exception, match="Invalid battleground"):
        mem.push(iact, xy, bg=other)
    mem.push(iact, xy)
    with pytest.raises(Exception, match="empty"):
        mem.sample(1)                                     # the newest frame has no successor yet
    for _ in range(3):
        bg.frame(maps=maps)
        mem.push(*pol.act(bg, maps))
    assert len(mem) >= 9
    tr = TrainerB200(batch_size=8, max_ships=8)
    with pytest.raises(Exception, match="Invalid batch"):
        tr.replay(9, memory=mem)
    bq = BatchedQLearner(tr, mem, snapshot=0)
    with pytest.raises(Exception, match="Invalid battleground"):
        bq.act(other, maps)
    with pytest.raises(Exception, match="Invalid positions"):
        mem.gather([len(mem)])
    with pytest.raises(OfbError, match="depth"):
        DeviceReplayMemory(bg, depth=1)
    with pytest.raises(Exception, match="Invalid ships"):
        DeviceReplayMemory(bg, ships=[1])
