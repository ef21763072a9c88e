"""Prioritized replay on the device (include/ofb_replay.h, ofb_train.h; replay.PrioritizedReplayMemory) -- runs on the B200 box.

The weighted fit is compared with the fp64 autograd restatement of tests/prio_oracle.py under the tolerances of
test_gpu_train.py; the sampler with the masses it was given (read back), the candidates of ofb_replay_index and the run's
own maps and fields, as test_gpu_replay.py does for the uniform path."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.test_gpu_replay import _drive, _expected
from tests.test_gpu_train import _arena_batch, _dense_image

pytestmark = pytest.mark.gpu


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _age_positions(mem):
    """transition id -> position in age order (ofb_replay_index's order), -1 for ids that are not valid candidates."""
    n = len(mem)
    ids = mem._ids[:n].long()
    pos = torch.full((mem.depth * mem.track * len(mem.ships),), -1, dtype=torch.long, device=mem.device)
    pos[ids] = torch.arange(n, device=mem.device)
    return pos, ids


def _compare(g, rec, sel):
    """The gathered namespace g against the run's own record for the expected transitions sel = [(t, a, p, reward, done)]."""
    assert torch.equal(g.maps_obs, torch.stack([rec[t]["maps"][a] for t, a, p, _, _ in sel]))
    assert torch.equal(g.maps_next, torch.stack([rec[t + 1]["maps"][a] for t, a, p, _, _ in sel]))
    assert torch.equal(g.vec_obs, torch.stack([rec[t]["vec"][a, p] for t, a, p, _, _ in sel]))
    assert torch.equal(g.vec_next, torch.stack([rec[t + 1]["vec"][a, p] for t, a, p, _, _ in sel]))
    assert torch.equal(g.iaction, torch.stack([rec[t]["iact"][a, p] for t, a, p, _, _ in sel]))
    assert torch.equal(g.pointer, torch.stack([rec[t]["xy"][a, p] for t, a, p, _, _ in sel]))
    assert g.reward.cpu().tolist() == [e[3] for e in sel]
    assert g.done.cpu().tolist() == [e[4] for e in sel]


def _small_memory(alpha, depth=3, frames=6, seed=8, eps=0.0):
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import PrioritizedReplayMemory
    bg = BatchedBattleground(16, ships={"QlearnIA": 1, "turret": 6}, seed=seed)
    mem = PrioritizedReplayMemory(bg, depth=depth, alpha=alpha, eps=eps, seed=5)
    rec = _drive(bg, mem, PolicyB200.random_init(max_ships=16), frames)
    return bg, mem, rec


def _td_of(ids, scale=1.0):
    """TD errors that are a function of the transition id, as those of one forward are."""
    x = ids.double()
    return (torch.sin(x) * 4 * scale).float(), (torch.cos(3 * x) * scale).float()


def _set_masses(mem, values):
    """Masses of the valid transitions (age order) := values, through update_priorities (td_act = value, td_ptr = 0)."""
    _, ids = _age_positions(mem)
    mem.sample_prioritized(1, 0.0)                        # the ids must come after the last push
    td = torch.as_tensor(values, dtype=torch.float32, device=mem.device)
    mem.update_priorities(ids.int().contiguous(), td, torch.zeros_like(td))
    return ids


# ---------------------------------------------------------------------------------------------- 1. weighted fit
@pytest.mark.parametrize("B", [8, 3])
def test_fit_weighted_matches_the_weighted_oracle(B):
    from oracle import policy_torch as po
    from oracle import policy_train_torch as pt
    from ofighters_b200.trainer import TrainerB200
    from tests import prio_oracle as wo
    w = po.init_weights(4, randomize_bn=True)
    _, maps, vec = _arena_batch(B)
    g = torch.Generator().manual_seed(10 + B)
    ta = torch.randn((B, 2), generator=g) * 3
    tp = torch.randn((B, 400, 400), generator=g) * 0.5
    sw = 2.0 * (1.0 - torch.rand((B,), generator=g))                        # (0, 2]
    tr = TrainerB200(weights=w, learning_rate=1e-4, batch_size=8)
    img, vec_h = _dense_image(maps), vec.cpu()
    wd = {k: v.double() for k, v in w.items()}
    imgd, vecd, tad, tpd, swd = img.double(), vec_h.double(), ta.double(), tp.double(), sw.double()
    opt = pt.KerasAdam(lr=1e-4)
    olosses, ograds, _ = wo.loss_and_grads(wd, imgd, vecd, tad, tpd, swd)
    loss = tr.fit(maps, vec, ta.cuda(), tp.cuda(), sample_weight=sw.cuda()).cpu()
    wo.fit(wd, opt, imgd, vecd, tad, tpd, swd)
    assert np.allclose(loss.numpy(), np.array(olosses), rtol=2e-4)
    grads = tr.get_grads()
    zero_grad = [k for k in ograds if k.endswith("/bias") and "conv" in k and k != "upconv4/bias"]
    for k, og in ograds.items():
        scale = max(float(og.abs().max()), float(ograds[k.replace("/bias", "/kernel")].abs().max()) if k in zero_grad else 0.0)
        err = float((grads[k].double() - og).abs().max())
        assert err <= 2e-3 * scale + 1e-9, (k, err, scale)
    for _ in range(2):
        tr.fit(maps, vec, ta.cuda(), tp.cuda(), sample_weight=sw.cuda())
        wo.fit(wd, opt, imgd, vecd, tad, tpd, swd)
    got = tr.get_weights()
    assert tr.steps == 3
    for k in wd:
        if k.endswith("/mean") or k.endswith("/var"):
            assert float((got[k].double() - wd[k]).abs().max()) <= 1e-5, k
            continue
        diff = ((got[k].double() - w[k].double()) - (wd[k] - w[k].double())).abs()
        assert float(diff.max()) <= 2.2e-4 * 3, (k, float(diff.max()))
        if k not in zero_grad:
            assert float((diff <= 5e-6 * 3).float().mean()) >= 0.99, k

    # w = 1: the unweighted fit, within the same tolerances (the weight gradients' fp32 atomics are not bit-reproducible)
    a, b = TrainerB200(weights=w, learning_rate=1e-4, batch_size=8), TrainerB200(weights=w, learning_rate=1e-4, batch_size=8)
    la = a.fit(maps, vec, ta.cuda(), tp.cuda(), sample_weight=torch.ones(B, device="cuda")).cpu()
    lb = b.fit(maps, vec, ta.cuda(), tp.cuda()).cpu()
    assert np.allclose(la.numpy(), lb.numpy(), rtol=2e-4)
    ga, gb = a.get_grads(), b.get_grads()
    for k in ga:
        scale = max(float(gb[k].abs().max()), float(gb[k.replace("/bias", "/kernel")].abs().max()) if k in zero_grad else 0.0)
        assert float((ga[k] - gb[k]).abs().max()) <= 2e-3 * scale + 1e-9, k


# ---------------------------------------------------------------------------------------------- 2. TD errors
def test_td_errors_are_target_minus_prediction_exactly():
    from ofighters_b200 import _lib
    lib = _lib.load()
    B = 6
    g = torch.Generator().manual_seed(12)
    act_o, act_n = torch.randn((B, 2), generator=g), torch.randn((B, 2), generator=g)
    ptr_o, ptr_n = torch.randn((B, 400, 400), generator=g), torch.randn((B, 400, 400), generator=g)
    ia = torch.tensor([0, 1, 1, 0, 1, 0], dtype=torch.int32)
    pointer = torch.tensor([[10, 20], [399, 0], [7, 7], [0, 399], [200, 123], [55, 301]], dtype=torch.int32)
    reward = torch.tensor([2.0, 0.0, 3.0, -1.0, 0.0, 1.0])
    done = torch.tensor([0, 1, 0, 1, 1, 0], dtype=torch.uint8)
    d = [t.cuda() for t in (act_o, ptr_o, act_n, ptr_n, ia, pointer, reward, done)]
    td_a, td_p = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
    _lib.check(lib.ofb_trainer_td_errors(*[_p(t) for t in d], 0.9, B, _p(td_a), _p(td_p), None))
    ta, tp = torch.empty_like(d[0]), torch.empty_like(d[1])
    _lib.check(lib.ofb_trainer_td_targets(*[_p(t) for t in d], 0.9, B, _p(ta), _p(tp), None))
    torch.cuda.synchronize()
    ta, tp = ta.cpu(), tp.cpu()
    for b in range(B):
        x, y = int(pointer[b, 0]), int(pointer[b, 1])
        assert torch.equal(td_a.cpu()[b], ta[b, int(ia[b])] - act_o[b, int(ia[b])])
        assert torch.equal(td_p.cpu()[b], tp[b, x, y] - ptr_o[b, x, y])          # the reference's [x][y] entry


# ---------------------------------------------------------------------------------------------- 3. distribution
def test_draws_follow_the_masses_and_are_stratified():
    from scipy.stats import chisquare
    _, mem, _ = _small_memory(alpha=1.0)
    pos, ids = _age_positions(mem)
    n = ids.numel()
    assert n >= 16
    masses = 0.05 + 0.1 * torch.arange(n, dtype=torch.float32).flip(0)          # distinct, |td| + 0 with alpha = 1
    _set_masses(mem, masses)
    got = mem.masses()[ids]
    assert torch.equal(got.cpu(), masses)
    counts = torch.zeros(n, dtype=torch.long, device="cuda")
    for _ in range(2000):
        s = mem.sample_prioritized(64, 0.5)
        p = pos[s.ids.long()]
        assert bool((p >= 0).all()) and bool((p[1:] >= p[:-1]).all()), "draws of one sample are not in age order"
        counts += torch.bincount(p, minlength=n)
    exp = (masses.double() / masses.double().sum() * 2000 * 64).numpy()
    assert chisquare(counts.cpu().numpy(), exp).pvalue > 1e-3


def test_alpha_zero_is_uniform_with_unit_weights():
    from scipy.stats import chisquare
    _, mem, _ = _small_memory(alpha=0.0, seed=9)
    pos, ids = _age_positions(mem)
    n = ids.numel()
    _set_masses(mem, torch.linspace(0.1, 5.0, n))
    assert bool((mem.masses()[ids] == 1.0).all())
    counts = torch.zeros(n, dtype=torch.long, device="cuda")
    for _ in range(2000):
        s = mem.sample_prioritized(64, 0.8)
        assert bool((s.weight == 1.0).all())
        counts += torch.bincount(pos[s.ids.long()], minlength=n)
    assert chisquare(counts.cpu().numpy()).pvalue > 1e-3


# ---------------------------------------------------------------------------------------------- 4. validity
def test_sampled_transitions_are_valid_and_gather_the_runs_own_fields():
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import PrioritizedReplayMemory
    N, T, D = 64, 30, 12
    bg = BatchedBattleground(N, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=3)
    mem = PrioritizedReplayMemory(bg, depth=D, alpha=0.6, seed=1)
    mask = torch.arange(N) % 2 == 0
    rec = _drive(bg, mem, PolicyB200.random_init(max_ships=N, seed=1), T, restarts={12: None, 21: mask, 25: None})
    exp = _expected(rec, N, range(T - D, T - 1))                           # the ring wrapped: the last D - 1 frames
    assert len(mem) == len(exp) and mem.frames == T
    assert not any(t == 24 for t, *_ in exp) and not any(t == 20 and a % 2 == 0 for t, a, *_ in exp)
    assert sum(e[4] for e in exp) > 0                                       # deaths are among them
    pos, ids = _age_positions(mem)
    cP = N
    newest = (T - 1) % D
    for k in range(4):
        s = mem.sample_prioritized(256, 0.4)
        p = pos[s.ids.long()]
        assert bool((p >= 0).all()), "a drawn id is not one of ofb_replay_index's"
        assert not bool((s.ids.long() // cP == newest).any())
        _compare(s, rec, [exp[i] for i in p.tolist()])
        if k == 1:                                                          # skewed masses: still only valid candidates
            g = torch.Generator(device="cuda").manual_seed(2)
            mem.update_priorities(s.ids, torch.rand(256, device="cuda", generator=g) * 50, torch.zeros(256, device="cuda"))


# ---------------------------------------------------------------------------------------------- 5. weights, priorities
def test_weights_and_priority_updates():
    bg, mem, _ = _small_memory(alpha=0.6, eps=1e-6, frames=5, seed=11)
    pos, ids = _age_positions(mem)
    n = ids.numel()
    s = mem.sample_prioritized(min(n, 16), 0.0)
    da, dp = _td_of(s.ids)
    dup_ids = torch.cat([s.ids, s.ids[:4]])               # duplicates carry identical errors
    dup_a, dup_p = torch.cat([da, da[:4]]), torch.cat([dp, dp[:4]])
    mem.update_priorities(dup_ids, dup_a, dup_p)
    m = mem.masses()
    want = ((da.double().abs() + dp.double().abs() + 1e-6) ** 0.6).float()
    assert torch.allclose(m[s.ids.long()], want, rtol=1e-6, atol=0)
    mx = float(mem.max_mass())
    assert mx == float(m[s.ids.long()].max()) and mx > 1.0
    # weights against numpy fp64 from the read-back masses
    for beta in (0.4, 1.0):
        t = mem.sample_prioritized(64, beta)
        mv = mem.masses()[ids].double().cpu().numpy()
        mmin = mv[mv > 0].min()
        w = (m[t.ids.long()].double().cpu().numpy() / mmin) ** (-beta)
        assert np.allclose(t.weight.cpu().numpy(), w, rtol=1e-5, atol=0) and float(t.weight.max()) <= 1.0
    # the next push's new transitions enter with the new maximum
    newest = (mem.frames - 1) % mem.depth
    from ofighters_b200.policy import PolicyB200
    maps = bg.raster("bits")
    mem.push(*PolicyB200.random_init(max_ships=16).act(bg, maps))
    cP = mem.track * len(mem.ships)
    assert bool((mem.masses()[newest * cP:(newest + 1) * cP] == mx).all())
    # duplicate ids in any order give the same masses
    s = mem.sample_prioritized(32, 0.5)
    ids2 = torch.cat([s.ids, s.ids])
    a2, p2 = _td_of(ids2, 0.5)
    mem.update_priorities(ids2, a2, p2)
    m1 = mem.masses()
    mem.sample_prioritized(1, 0.5)
    mem.update_priorities(ids2.flip(0).contiguous(), a2.flip(0).contiguous(), p2.flip(0).contiguous())
    assert torch.equal(mem.masses(), m1)


# ---------------------------------------------------------------------------------------------- 6. full size
def test_full_size_sample_and_update():
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.replay import PrioritizedReplayMemory
    N, P, D = 65536, 7, 16
    bg = BatchedBattleground(N, ships={"QlearnIA": P}, seed=0x0F16)
    mem = PrioritizedReplayMemory(bg, depth=D, alpha=0.6, seed=3)
    assert D * N * P > 7.3e6
    g = torch.Generator(device="cuda").manual_seed(6)
    maps = bg.raster("bits")
    for _ in range(D + 1):                                # the ring wraps once
        iact = torch.randint(0, 2, (N * P,), dtype=torch.int32, device="cuda", generator=g)
        xy = torch.randint(0, 400, (N * P, 2), dtype=torch.int32, device="cuda", generator=g)
        mem.push(iact, xy)
        bg.frame(maps=maps)
    pos, ids = _age_positions(mem)
    assert ids.numel() > 0.5 * (D - 1) * N * P
    for k in range(3):
        s = mem.sample_prioritized(256, 0.5)
        p = pos[s.ids.long()]
        assert bool((p >= 0).all()) and bool((p[1:] >= p[:-1]).all())
        total = float(mem.last_total())
        want = mem.masses()[ids].double().cpu().numpy().sum()
        assert abs(total - want) <= 1e-12 * want, (total, want)
        g = torch.Generator(device="cuda").manual_seed(k)
        mem.update_priorities(s.ids, torch.randn(256, device="cuda", generator=g) * 10, torch.randn(256, device="cuda", generator=g))


# ---------------------------------------------------------------------------------------------- 7. end to end
def test_batched_qlearner_with_prioritized_memory():
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.replay import PrioritizedReplayMemory
    from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200
    bg = BatchedBattleground(256, ships={"QlearnIA": 1, "random": 6}, seed=21)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=8, max_ships=256)
    mem = PrioritizedReplayMemory(bg, depth=16, alpha=0.6, eps=1e-6, seed=7)
    bq = BatchedQLearner(tr, mem, replay_every=10, collecting_steps=20, snapshot=0, beta0=0.4, beta_frames=100)
    updates = []
    orig = mem.update_priorities

    def spy(ids, td_act, td_ptr):
        updates.append((ids.clone(), td_act.clone(), td_ptr.clone()))
        orig(ids, td_act, td_ptr)

    mem.update_priorities = spy
    maps = bg.raster("bits")
    replays = []
    for t in range(120):
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
    assert replays == list(range(10, 121, 10)) and tr.steps == 12
    assert all(np.isfinite(bq.losses)) and len(bq.losses) == 12
    assert bq.betas == pytest.approx([min(1.0, 0.4 + 0.6 * t / 100) for t in replays], rel=1e-12)
    ids, da, dp = updates[-1]
    want = ((da.double().abs() + dp.double().abs() + 1e-6) ** 0.6).float()
    assert torch.allclose(mem.masses()[ids.long()], want, rtol=1e-6, atol=0)


# ---------------------------------------------------------------------------------------------- 8. bad arguments
def test_bad_arguments_raise():
    from ofighters_b200 import BatchedBattleground, OfbError, _lib
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import DeviceReplayMemory, EmptyReplayMemory, PrioritizedReplayMemory
    from ofighters_b200.trainer import TrainerB200
    bg = BatchedBattleground(8, ships={"QlearnIA": 1, "random": 6}, seed=2)
    with pytest.raises(Exception, match="Invalid priorities"):
        PrioritizedReplayMemory(bg, alpha=-0.1)
    lib = _lib.load()
    plain = DeviceReplayMemory(bg, depth=4)
    cfg = _lib.OfbReplayPrioConfig(alpha=-1.0, eps=0.0, seed=0)
    with pytest.raises(OfbError, match="alpha"):
        _lib.check(lib.ofb_replay_enable_priorities(plain._h, C.byref(cfg)))
    pol = PolicyB200.random_init(max_ships=8)
    maps = bg.raster("bits")
    plain.push(*pol.act(bg, maps))
    cfg.alpha = 0.5
    with pytest.raises(OfbError, match="first push"):
        _lib.check(lib.ofb_replay_enable_priorities(plain._h, C.byref(cfg)))

    mem = PrioritizedReplayMemory(bg, depth=4)
    with pytest.raises(EmptyReplayMemory, match="empty"):
        mem.sample_prioritized(1, 0.5)
    for _ in range(3):
        mem.push(*pol.act(bg, maps))
        bg.frame(maps=maps)
    with pytest.raises(Exception, match="Invalid beta"):
        mem.sample_prioritized(4, -0.5)
    with pytest.raises(Exception, match="Invalid batch"):
        mem.sample_prioritized(0, 0.5)
    tr = TrainerB200(batch_size=8, max_ships=8)
    with pytest.raises(Exception, match="Invalid batch"):
        tr.replay(9, memory=mem, beta=0.5)
    with pytest.raises(Exception, match="Invalid batch"):
        tr.replay(0, memory=mem, beta=0.5)
    s = mem.sample_prioritized(4, 0.5)
    z = torch.zeros(4, device="cuda")
    with pytest.raises(Exception, match="outside"):
        mem.update_priorities(torch.tensor([0, 1, 2, 4 * 8], dtype=torch.int32, device="cuda"), z, z)
    with pytest.raises(Exception, match="Invalid td_act"):
        mem.update_priorities(s.ids, z[:3], z)
    mem.push(*pol.act(bg, maps))
    with pytest.raises(Exception, match="push happened"):
        mem.update_priorities(s.ids, z, z)
    with pytest.raises(Exception, match="Invalid sample_weight"):
        tr.fit(s.maps_next, s.vec_next, torch.zeros(4, 2), torch.zeros(4, 400, 400), sample_weight=torch.ones(3))
