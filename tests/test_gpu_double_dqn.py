"""Target network and Double DQN (include/ofb_train.h ofb_trainer_td_targets_double; trainer.py) -- runs on the B200 box.

The kernel is checked bit for bit against the host restatement of tests/double_oracle.py, on random maps and on maps built to
catch a wrong selection: equal maxima in different blocks of a sample's cluster, the maximum in the first and the last 16
bytes, NaNs, -inf and constant maps.  With the target's maps equal to the online ones it must give the single-network kernels'
results.  The trainer's target network is checked through its refresh cadence and blend, the replay paths through the targets
they hand to fit, and the learner end to end."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

from tests import double_oracle as do

pytestmark = pytest.mark.gpu

G = 0.9
N = 400 * 400
SLICE = N // 8                                            # floats per block of a sample's 8-block cluster


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _same(a, b):
    """Bit equality, NaN matching any NaN (the device returns the canonical NaN, the host propagates payloads)."""
    a, b = a.detach().cpu().contiguous(), b.detach().cpu().contiguous()
    if a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a.masked_fill(na, 0).view(torch.int32), b.masked_fill(nb, 0).view(torch.int32))


def _adversarial(m, b, kind, g):
    """Overwrite the online map m [400*400] of sample b with a map of `kind`."""
    if kind == "slice_tie":                               # equal maxima in blocks 6, 2 and 5: block 2's wins
        m[6 * SLICE] = 9.0
        m[2 * SLICE + SLICE - 1] = 9.0
        m[5 * SLICE + 4 * 17 + 1] = 9.0
    elif kind == "thread_tie":                            # equal maxima in one block, different threads and float4 lanes
        m[3 * SLICE + 4 * 700 + 3] = 8.0
        m[3 * SLICE + 4 * 5 + 2] = 8.0
        m[3 * SLICE + 4 * 2000] = 8.0
    elif kind == "first16":
        m[int(torch.randint(0, 4, (1,), generator=g))] = 7.0
    elif kind == "last16":
        m[N - 4 + int(torch.randint(0, 4, (1,), generator=g))] = 7.0
        m[N - 1 - 4] = 6.999
    elif kind == "nan":
        idx = torch.randint(0, N, (2000,), generator=g)
        m[idx] = float("nan")
        m[0] = float("nan")
        top = int(m.nan_to_num(-1e30).argmax())
        m[top - 1 if top > 0 else top + 1] = float("nan")
    elif kind == "neg_inf":
        m[:] = -float("inf")
        m[int(torch.randint(0, N, (1,), generator=g))] = float("nan")
    elif kind == "constant":
        m[:] = 0.25
    elif kind == "all_nan":
        m[:] = float("nan")


KINDS = ["slice_tie", "random", "first16", "last16", "nan", "neg_inf", "constant", "all_nan", "thread_tie"]


def _case(B, seed):
    g = torch.Generator().manual_seed(seed)
    c = dict(act_obs=torch.randn((B, 2), generator=g), ptr_obs=torch.randn((B, 400, 400), generator=g),
             act_on=torch.randn((B, 2), generator=g), ptr_on=torch.randn((B, 400, 400), generator=g),
             act_tg=torch.randn((B, 2), generator=g), ptr_tg=torch.randn((B, 400, 400), generator=g),
             iaction=torch.randint(0, 2, (B,), generator=g, dtype=torch.int32),
             pointer=torch.randint(0, 400, (B, 2), generator=g, dtype=torch.int32),
             reward=torch.randn((B,), generator=g) * 2, done=(torch.rand((B,), generator=g) < 0.25).to(torch.uint8))
    c["act_on"][::3, 1] = c["act_on"][::3, 0]             # act ties
    for b in range(B):
        _adversarial(c["ptr_on"][b].view(-1), b, KINDS[b % len(KINDS)], g)
    for b in range(0, B, 7):                              # NaNs in some target maps: whatever is selected is taken as is
        c["ptr_tg"][b].view(-1)[::9973] = float("nan")
    c["ptr_tg"][1::7] = -float("inf")
    return c


def _kernel(lib, d, disc, inplace, with_td):
    """Runs ofb_trainer_td_targets_double on device copies d -> (t_act, t_ptr, td_act, td_ptr) on the host."""
    from ofighters_b200 import _lib
    B = d["act_obs"].shape[0]
    a_obs, p_obs = d["act_obs"].clone(), d["ptr_obs"].clone()
    t_act, t_ptr = (a_obs, p_obs) if inplace else (torch.full_like(a_obs, 5.0), torch.full_like(p_obs, 5.0))
    td_a = torch.full((B,), 3.0, device="cuda") if with_td else None
    td_p = torch.full((B,), 3.0, device="cuda") if with_td else None
    _lib.check(lib.ofb_trainer_td_targets_double(
        *[_p(d[k]) if k not in ("act_obs", "ptr_obs") else _p(a_obs if k == "act_obs" else p_obs)
          for k in ("act_obs", "ptr_obs", "act_on", "ptr_on", "act_tg", "ptr_tg", "iaction", "pointer", "reward", "done")],
        G, _p(disc), B, _p(t_act), _p(t_ptr), _p(td_a), _p(td_p), None))
    torch.cuda.synchronize()
    if not inplace:                                       # out of place leaves the predictions untouched
        assert torch.equal(a_obs, d["act_obs"]) and torch.equal(p_obs, d["ptr_obs"])
    return t_act.cpu(), t_ptr.cpu(), (td_a.cpu() if with_td else None), (td_p.cpu() if with_td else None)


# ---------------------------------------------------------------------------------------------- 1. kernel == oracle
@pytest.mark.parametrize("B", [1, 5, 8, 64, 256])
@pytest.mark.parametrize("discounted", [False, True])
def test_kernel_matches_the_oracle_bit_for_bit(B, discounted):
    from ofighters_b200 import _lib
    lib = _lib.load()
    c = _case(B, seed=B * 10 + discounted)
    disc = (torch.rand((B,), generator=torch.Generator().manual_seed(B)) ** 2) if discounted else None
    want = do.td_targets_double(c["act_obs"], c["ptr_obs"], c["act_on"], c["ptr_on"], c["act_tg"], c["ptr_tg"], c["iaction"],
                                c["pointer"], c["reward"], c["done"], gamma=G, discount=disc)
    d = {k: v.cuda() for k, v in c.items()}
    ddisc = disc.cuda() if disc is not None else None
    for inplace in (True, False):
        for with_td in (True, False):
            t_act, t_ptr, td_a, td_p = _kernel(lib, d, ddisc, inplace, with_td)
            assert _same(t_act, want[0]), (inplace, with_td)
            assert _same(t_ptr, want[1]), (inplace, with_td)
            if with_td:
                assert _same(td_a, want[2]) and _same(td_p, want[3])
                rows = torch.arange(B)
                ia, px, py = c["iaction"].long(), c["pointer"][:, 0].long(), c["pointer"][:, 1].long()
                assert _same(td_a, t_act[rows, ia] - c["act_obs"][rows, ia])
                assert _same(td_p, t_ptr[rows, px, py] - c["ptr_obs"][rows, px, py])
    # the selections the adversarial maps were built for
    p_star = do.select_ptr(c["ptr_on"]).tolist()
    for b in range(B):
        kind = KINDS[b % len(KINDS)]
        if kind == "slice_tie":
            assert p_star[b] == 2 * SLICE + SLICE - 1
        elif kind in ("constant", "all_nan", "neg_inf"):
            assert p_star[b] == 0 or (kind == "neg_inf" and p_star[b] == 1)


# ---------------------------------------------------------------------------------------------- 2. synced identity
def _real_predictions(B=64):
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from oracle import policy_torch as po
    bg = BatchedBattleground(B, ships={"QlearnIA": 1, "random": 6}, seed=11)
    pol = PolicyB200(po.init_weights(3, randomize_bn=True), max_ships=B)
    maps = bg.raster("bits")
    obs = pol.forward(maps, bg.obs_vec[:, 0, :].contiguous(), 1, want_ptr=True)
    for _ in range(3):
        iact, xy = pol.act(bg, maps, epsilon=0.5)
        bg.frame(maps=maps)
    nxt = pol.forward(maps, bg.obs_vec[:, 0, :].contiguous(), 1, want_ptr=True)
    g = torch.Generator(device="cuda").manual_seed(2)
    return dict(act_obs=obs["act"], ptr_obs=obs["ptr"], act_next=nxt["act"], ptr_next=nxt["ptr"],
                iaction=torch.randint(0, 2, (B,), device="cuda", generator=g, dtype=torch.int32),
                pointer=torch.randint(0, 400, (B, 2), device="cuda", generator=g, dtype=torch.int32),
                reward=torch.randn((B,), device="cuda", generator=g),
                done=(torch.rand((B,), device="cuda", generator=g) < 0.2).to(torch.uint8))


def test_synced_maps_give_the_single_network_kernels_results():
    from ofighters_b200 import _lib
    lib = _lib.load()
    r = _real_predictions()
    B = r["act_obs"].shape[0]
    assert not bool(torch.isnan(r["ptr_next"]).any())
    flat = r["ptr_next"].reshape(B, -1)
    mx = flat.max(dim=1, keepdim=True).values
    assert not bool(((flat == mx) & (flat.view(torch.int32) != mx.view(torch.int32))).any())     # no +0 / -0 tie
    fields = [_p(r[k]) for k in ("iaction", "pointer", "reward", "done")]
    single = [_p(r[k]) for k in ("act_obs", "ptr_obs", "act_next", "ptr_next")]
    for disc in (None, torch.rand((B,), device="cuda") ** 2, torch.full((B,), G, device="cuda")):
        sa, sp = torch.empty_like(r["act_obs"]), torch.empty_like(r["ptr_obs"])
        ea, ep = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
        if disc is None:
            _lib.check(lib.ofb_trainer_td_targets(*single, *fields, G, B, _p(sa), _p(sp), None))
            _lib.check(lib.ofb_trainer_td_errors(*single, *fields, G, B, _p(ea), _p(ep), None))
        else:
            _lib.check(lib.ofb_trainer_td_targets_discounted(*single, *fields, _p(disc), B, _p(sa), _p(sp), None))
            _lib.check(lib.ofb_trainer_td_errors_discounted(*single, *fields, _p(disc), B, _p(ea), _p(ep), None))
        da, dp = r["act_obs"].clone(), r["ptr_obs"].clone()
        xa, xp = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
        _lib.check(lib.ofb_trainer_td_targets_double(
            _p(da), _p(dp), _p(r["act_next"]), _p(r["ptr_next"]), _p(r["act_next"]), _p(r["ptr_next"]), *fields, G, _p(disc), B,
            _p(da), _p(dp), _p(xa), _p(xp), None))
        torch.cuda.synchronize()
        assert torch.equal(da.view(torch.int32), sa.view(torch.int32)) and torch.equal(dp.view(torch.int32), sp.view(torch.int32))
        assert torch.equal(xa.view(torch.int32), ea.view(torch.int32)) and torch.equal(xp.view(torch.int32), ep.view(torch.int32))


# ---------------------------------------------------------------------------------------------- 3. refresh cadence
def _fit_batch(B=8, seed=5):
    from ofighters_b200 import BatchedBattleground
    bg = BatchedBattleground(B, ships={"QlearnIA": 1, "random": 6}, seed=seed)
    maps = bg.raster("bits")
    for _ in range(2):
        bg.frame(maps=maps)
    g = torch.Generator(device="cuda").manual_seed(seed)
    return maps, bg.obs_vec[:, 0, :].contiguous(), torch.randn((B, 2), device="cuda", generator=g), \
        torch.randn((B, 400, 400), device="cuda", generator=g) * 0.1


def test_target_refresh_cadence_and_blend():
    from oracle import policy_torch as po
    from ofighters_b200.trainer import TrainerB200
    w0 = po.init_weights(4, randomize_bn=True)
    maps, vec, ta, tp = _fit_batch()
    tr = TrainerB200(weights=w0, learning_rate=1e-3, batch_size=8, max_ships=8, target_update=3, target_tau=1.0)

    def target_pred():
        r = tr.target_model.forward(maps, vec, 1, want_ptr=True)
        return torch.cat([r["act"].reshape(-1), r["ptr"].reshape(-1)]).cpu()

    p0 = target_pred()
    for k in (1, 2):
        tr.fit(maps, vec, ta, tp)
        assert torch.equal(target_pred().view(torch.int32), p0.view(torch.int32)), k
        assert tr.target_updates == 0
    tr.fit(maps, vec, ta, tp)
    assert tr.target_updates == 1 and not torch.equal(target_pred(), p0)
    w, wt = tr.get_weights(), tr.get_target_weights()
    for k in w:
        assert torch.equal(w[k], wt[k]), k
    assert any("norm" in k and k.endswith("/mean") and not torch.equal(w[k], torch.as_tensor(w0[k]).float()) for k in w)
    # tau = 0.25: the numpy fp32 blend, refresh after refresh
    tr = TrainerB200(weights=w0, learning_rate=1e-3, batch_size=8, max_ships=8, target_update=3, target_tau=0.25)
    want = {k: torch.as_tensor(v).float().numpy() for k, v in w0.items()}
    for step in range(1, 7):
        tr.fit(maps, vec, ta, tp)
        if step % 3 == 0:
            want = do.blend({k: v.numpy() for k, v in tr.get_weights().items()}, want, 0.25)
        got = tr.get_target_weights()
        for k in got:
            assert np.array_equal(got[k].numpy().view(np.uint32), want[k].view(np.uint32)), (step, k)
    assert tr.target_updates == 2


# ---------------------------------------------------------------------------------------------- 4. replay plumbing
def _memory(kind, bg):
    from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory
    if kind == "uniform":
        return DeviceReplayMemory(bg, depth=12)
    if kind == "nstep":
        return DeviceReplayMemory(bg, depth=12, n_step=3)
    if kind == "prioritized":
        return PrioritizedReplayMemory(bg, depth=12, seed=3)
    if kind == "prioritized_nstep":
        return PrioritizedReplayMemory(bg, depth=12, seed=3, n_step=3)
    return None


@pytest.mark.parametrize("kind", ["deque", "uniform", "nstep", "prioritized", "prioritized_nstep"])
def test_replay_paths_build_the_single_network_targets_when_synced(kind):
    from oracle import policy_torch as po
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.trainer import TrainerB200
    from tests.test_gpu_replay import _drive
    bg = BatchedBattleground(32, ships={"QlearnIA": 1, "random": 3, "turret": 3}, seed=17)
    tr = TrainerB200(weights=po.init_weights(8, randomize_bn=True), learning_rate=1e-4, batch_size=8, max_ships=32,
                     target_update=1, target_tau=1.0, double_dqn=True)
    mem = _memory(kind, bg)
    pol = PolicyB200.random_init(max_ships=32, seed=2)
    if mem is None:                                       # the reference's deque, filled from the first four arenas
        maps = bg.raster("bits")
        for t in range(10):
            obs = [(maps[a].clone(), bg.obs_vec[a, 0].clone()) for a in range(4)]
            iact, xy = pol.act(bg, maps, epsilon=0.5)
            bg.frame(maps=maps)
            for a in range(4):
                tr.remember(obs[a], int(iact[a]), tuple(xy[a].tolist()), float(bg.obs_vec[a, 0, 0]),
                            (maps[a].clone(), bg.obs_vec[a, 0].clone()), t == 4 and a == 0)
    else:
        _drive(bg, mem, pol, 12, restarts={6: None})
    prio = kind.startswith("prioritized")
    kw = dict(memory=mem, beta=0.5) if prio else dict(memory=mem)
    random.seed(3)
    tr.replay(8, **kw)                                    # a real fit: its refresh makes theta- = theta
    assert tr.target_updates == 1
    for k, v in tr.get_target_weights().items():
        assert torch.equal(v, tr.get_weights()[k])

    got, tds = {}, {}
    if mem is not None:                                   # the same minibatch for every path
        name = "sample_prioritized" if prio else "sample"
        orig, cache = getattr(mem, name), []

        def once(*a):
            if not cache:
                cache.append(orig(*a))
            return cache[0]
        setattr(mem, name, once)
        if prio:
            orig_up = mem.update_priorities
            mem.update_priorities = lambda ids, da, dp: (tds.__setitem__(mode, (da.clone(), dp.clone())), orig_up(ids, da, dp))
    steps = tr.steps
    tr.fit = lambda maps, vec, a, p, **k: (got.__setitem__(mode, (a.clone(), p.clone())), torch.zeros(3, device="cuda"))[1]
    target_model = tr.target_model
    for mode in ("double", "target", "single"):
        tr.double_dqn = mode == "double"
        tr.target_model = None if mode == "single" else target_model
        random.seed(5)
        tr.replay(8, **kw)
    assert tr.steps == steps
    for mode in ("double", "target"):
        assert torch.equal(got[mode][0].view(torch.int32), got["single"][0].view(torch.int32)), mode
        assert torch.equal(got[mode][1].view(torch.int32), got["single"][1].view(torch.int32)), mode
        if prio:
            assert torch.equal(tds[mode][0].view(torch.int32), tds["single"][0].view(torch.int32)), mode
            assert torch.equal(tds[mode][1].view(torch.int32), tds["single"][1].view(torch.int32)), mode


# ---------------------------------------------------------------------------------------------- 5. end to end
@pytest.mark.parametrize("prioritized", [False, True])
def test_batched_qlearner_with_double_dqn(prioritized):
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory
    from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200
    random.seed(1)
    bg = BatchedBattleground(64, ships={"QlearnIA": 1, "random": 6}, seed=21)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=8, max_ships=64,
                     target_update=2, target_tau=0.5, double_dqn=True)
    mem = PrioritizedReplayMemory(bg, depth=16, alpha=0.6, eps=1e-6, seed=7) if prioritized else \
        DeviceReplayMemory(bg, depth=16, n_step=3)
    bq = BatchedQLearner(tr, mem, replay_every=20, collecting_steps=20, snapshot=0)
    updates = []
    if prioritized:
        orig = mem.update_priorities

        def spy(ids, td_act, td_ptr):
            updates.append((ids.clone(), td_act.clone(), td_ptr.clone()))
            orig(ids, td_act, td_ptr)
        mem.update_priorities = spy
    maps = bg.raster("bits")
    replays = []
    for t in range(120):
        if t == 70:
            bg.restart()
            bg.raster("bits", out=maps)
            bq.reset()
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
    assert replays == list(range(20, 121, 20)) and tr.steps == 6 and tr.target_updates == 3
    assert len(bq.losses) == 6 and all(np.isfinite(bq.losses))
    if prioritized:
        assert len(updates) == 6
        ids, da, dp = updates[-1]
        assert bool(torch.isfinite(da).all()) and bool(torch.isfinite(dp).all())
        want = ((da.double().abs() + dp.double().abs() + 1e-6) ** 0.6).float()
        assert torch.allclose(mem.masses()[ids.long()], want, rtol=1e-6, atol=0)


# ---------------------------------------------------------------------------------------------- 6. bad arguments
def test_bad_arguments_raise():
    from ofighters_b200 import _lib
    from ofighters_b200.trainer import TrainerB200
    for kw in (dict(double_dqn=True), dict(target_update=0), dict(target_update=-2), dict(target_update=1.5),
               dict(target_update=3, target_tau=0.0), dict(target_update=3, target_tau=1.5), dict(target_update=3, target_tau=-1)):
        with pytest.raises(Exception, match="Invalid"):
            TrainerB200(batch_size=2, max_ships=2, **kw)
    with pytest.raises(Exception, match="no target network"):
        TrainerB200(batch_size=2, max_ships=2).get_target_weights()
    lib = _lib.load()
    B = 2
    a = torch.zeros((B, 2), device="cuda")
    m = torch.zeros((B, 400, 400), device="cuda")
    ia = torch.zeros(B, dtype=torch.int32, device="cuda")
    pt = torch.zeros((B, 2), dtype=torch.int32, device="cuda")
    r = torch.zeros(B, device="cuda")
    dn = torch.zeros(B, dtype=torch.uint8, device="cuda")
    td = torch.zeros(B, device="cuda")

    def call(**over):
        args = dict(ao=a, po=m, an=a, pn=m, at=a, pt_=m, ia=ia, ptr=pt, r=r, d=dn, disc=None, B=B, ta=a, tp=m, tda=td, tdp=td)
        args.update(over)
        return lib.ofb_trainer_td_targets_double(
            *[_p(args[k]) for k in ("ao", "po", "an", "pn", "at", "pt_", "ia", "ptr", "r", "d")], G, _p(args["disc"]), args["B"],
            *[_p(args[k]) for k in ("ta", "tp", "tda", "tdp")], None)

    assert call() == 0
    torch.cuda.synchronize()
    for over in (dict(pn=None), dict(pt_=None), dict(at=None), dict(ta=None), dict(B=0), dict(tda=None), dict(tdp=None)):
        assert call(**over) == -1, over                   # OFB_E_ARG
    assert call(tda=None, tdp=None) == 0
    mis = torch.zeros(B * N + 1, device="cuda")[1:]       # 4 bytes off the 16-byte grid
    assert call(pn=mis) == -1 and call(po=mis, tp=mis) == -1
    assert "aligned" in lib.ofb_last_error().decode()
    torch.cuda.synchronize()
