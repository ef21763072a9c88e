"""Data-parallel fit and replay (ofb_trainer_fit_shard, ofb_replay_rescale_weights, TrainerB200(reducer=...)) on ONE device.

``ThreadReducer(world)`` gives W virtual ranks: W trainer handles on W streams driven by W threads.  A reduce call synchronises
its rank's stream and waits at a barrier; rank 0 sums the W slices on the device (in rank order) and every rank copies the
sum back.  No process and no NCCL are involved, so these tests check the arithmetic of the sharded fit and the collective
protocol of the sharded replay; scripts/dp_check.py runs the same fit over NCCL on several GPUs.

Tolerances: a sharded fit's losses and batch statistics equal the one-GPU fit of the concatenated batch up to the order of
fp64 sums (losses 1e-6 relative at the first step and 2e-5 at the next two, whose weights carry the fp32 atomics' noise;
statistics 1e-5); gradients, Adam trajectories and moving statistics are held to tests/test_gpu_train.py's bounds against the
fp64 torch oracle run on the concatenated batch.  The one-GPU fit of that batch is held to the same gradient bound: at
B = 64 it covers the element-wise kernels past the 2 368 blocks blocks_for allows (from B = 61 dense1's input gradient has
more elements than one pass of the capped grid), which must stride over the grid.
"""
import math
import random
import threading

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


class _RankReducer:
    """Rank ``rank``'s view of a ThreadReducer: the ``reducer`` interface TrainerB200 takes."""

    def __init__(self, hub, rank):
        self.hub, self.rank, self.world = hub, rank, hub.world
        self.calls = 0
        self.fail_at = None                               # raise on this call (error-path test)

    def _exchange(self, tensor, combine):
        hub = self.hub
        torch.cuda.current_stream().synchronize()
        hub.slots[self.rank] = tensor
        hub.barrier.wait()
        if self.rank == 0:
            hub.out = combine(hub.slots)
            torch.cuda.current_stream().synchronize()
        hub.barrier.wait()
        tensor.copy_(hub.out)
        torch.cuda.current_stream().synchronize()
        hub.barrier.wait()                                # nobody reuses the slots before every rank has copied

    def all_reduce(self, tensor, op="sum"):
        self.calls += 1
        if self.fail_at is not None and self.calls == self.fail_at:
            raise RuntimeError("reducer failure injected at call %d" % self.calls)

        def combine(slots):
            acc = slots[0].clone()
            for t in slots[1:]:
                acc = acc + t if op == "sum" else (torch.minimum(acc, t) if op == "min" else torch.maximum(acc, t))
            return acc
        self._exchange(tensor, combine)

    def broadcast(self, tensor, src=0):
        self._exchange(tensor, lambda slots: slots[src].clone())


class ThreadReducer:
    def __init__(self, world, timeout=120.0):
        self.world = world
        self.barrier = threading.Barrier(world, timeout=timeout)
        self.slots = [None] * world
        self.out = None
        self.ranks = [_RankReducer(self, r) for r in range(world)]


def run_ranks(world, fn, timeout=600.0):
    """fn(rank) on W threads, each on its own stream; re-raises the first failure."""
    results, errors = [None] * world, []
    streams = [torch.cuda.Stream() for _ in range(world)]

    def body(r):
        try:
            with torch.cuda.stream(streams[r]):
                results[r] = fn(r)
                torch.cuda.current_stream().synchronize()
        except BaseException as e:                        # noqa: B902
            errors.append(e)
    threads = [threading.Thread(target=body, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout)
    assert not any(t.is_alive() for t in threads), "a virtual rank hung"
    if errors:
        raise errors[0]
    return results


# ------------------------------------------------------------------------------------------------ data
def _dense_image(maps):
    b = maps.cpu().numpy().view(np.uint32)
    n = b.shape[0]
    img = np.unpackbits(b.view(np.uint8).reshape(n, 2, -1), axis=2, bitorder="little").reshape(n, 2, 400, 400)
    return torch.from_numpy(img.transpose(0, 2, 3, 1).astype(np.float32))


def _batch(B, seed=11):
    from ofighters_b200 import BatchedBattleground
    bg = BatchedBattleground(B, ships={"random": 7}, seed=seed)
    for _ in range(35):
        bg.frame()
    maps = bg.raster("bits")
    vec = bg.obs_vec[:, 0, :].contiguous()
    g = torch.Generator().manual_seed(B)
    ta = torch.randn((B, 2), generator=g) * 3
    tp = torch.randn((B, 400, 400), generator=g) * 0.5
    sw = torch.rand((B,), generator=g) * 0.9 + 0.1
    return maps, vec, ta, tp, sw


def _oracle_fit(wd, opt, img, vec, ta, tp, sw):
    """One fp64 step of oracle/policy_train_torch.py on the concatenated batch, with tf.keras' sample_weight when sw is given:
    each head's loss (1/B) sum_b w_b mse_b.  -> losses, grads, BN batch stats."""
    from oracle import policy_train_torch as pt
    names = pt.trainable_names(wd)
    wt = {k: v.clone().detach().requires_grad_(k in names) for k, v in wd.items()}
    act, ptr, stats = pt.forward_train(wt, img, vec)
    if sw is None:
        la, lp = ((act - ta) ** 2).mean(), ((ptr - tp) ** 2).mean()
    else:
        la, lp = (sw[:, None] * (act - ta) ** 2).mean(), (sw[:, None, None] * (ptr - tp) ** 2).mean()
    (la + lp).backward()
    grads = {k: wt[k].grad.detach() for k in names}
    for bn, (mean, var, n) in stats.items():
        wd[bn + "/mean"] = wd[bn + "/mean"] * pt.BN_MOMENTUM + mean * (1.0 - pt.BN_MOMENTUM)
        wd[bn + "/var"] = wd[bn + "/var"] * pt.BN_MOMENTUM + var * (1.0 - pt.BN_MOMENTUM)
    opt.step(wd, grads)
    return (float((la + lp).detach()), float(la.detach()), float(lp.detach())), grads, stats


def _shards(sizes):
    lo, out = 0, []
    for n in sizes:
        out.append((lo, lo + n))
        lo += n
    return out


def _make_ranks(world, w, batch_size, **kw):
    from ofighters_b200.trainer import TrainerB200
    hub = ThreadReducer(world)
    trainers = run_ranks(world, lambda r: TrainerB200(weights=w, learning_rate=1e-4, batch_size=batch_size, max_ships=8,
                                                      reducer=hub.ranks[r], **kw))
    return hub, trainers


def _bn_stats_from_exchange(tr, n_global):
    """Batch mean / biased variance of each BN layer from the reduced forward sums of the last sharded fit."""
    from ofighters_b200 import _lib
    from oracle import policy_train_torch as pt
    s = tr._xstats.cpu()
    sizes = [400, 200, 100, 50, 50, 100, 200]
    chans = [8, 8, 8, 8, 2, 4, 8]
    out = {}
    for l, bn in enumerate(pt.BN_LAYERS):
        o = _lib.TRAIN_STATS_FWD + 16 * l
        n = n_global * sizes[l] * sizes[l]
        c = chans[l]
        m = s[o:o + c] / n
        out[bn] = (m, (s[o + 8:o + 8 + c] / n - m * m).clamp_min(0.0))
    return out


FIT_CASES = [[8], [3, 5], [1, 7], [2, 2, 2, 2], [64], [32, 32], [16, 16, 16, 16], [1, 63]]


@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("sizes", FIT_CASES, ids=["+".join(map(str, s)) for s in FIT_CASES])
def test_sharded_fit_equals_the_fit_of_the_concatenated_batch(sizes, weighted):
    from oracle import policy_torch as po
    from oracle import policy_train_torch as pt
    from ofighters_b200.trainer import TrainerB200
    W, B = len(sizes), sum(sizes)
    w = po.init_weights(4, randomize_bn=True)
    maps, vec, ta, tp, sw = _batch(B)
    if not weighted:
        sw = None
    hub, trainers = _make_ranks(W, w, max(sizes))
    single = TrainerB200(weights=w, learning_rate=1e-4, batch_size=B, max_ships=8)
    dev = torch.device("cuda")
    wd = {k: v.double().to(dev) for k, v in w.items()}
    img, vecd, tad, tpd = _dense_image(maps).double().to(dev), vec.double(), ta.double().to(dev), tp.double().to(dev)
    swd = sw.double().to(dev) if sw is not None else None
    opt = pt.KerasAdam(lr=1e-4)
    parts = _shards(sizes)
    zero_grad = None
    for step in (1, 2, 3):
        def fit_rank(r):
            lo, hi = parts[r]
            kw = {} if sw is None else {"sample_weight": sw[lo:hi].cuda()}
            return trainers[r].fit(maps[lo:hi].contiguous(), vec[lo:hi], ta[lo:hi].cuda(), tp[lo:hi].cuda(), **kw).cpu()
        losses = run_ranks(W, fit_rank)
        ref = single.fit(maps, vec, ta.cuda(), tp.cuda(), sample_weight=None if sw is None else sw.cuda()).cpu()
        olosses, ograds, ostats = _oracle_fit(wd, opt, img, vecd, tad, tpd, swd)
        # every rank reports the global batch's loss; equal to the single fit's up to fp64 summation order
        for r in range(W):
            assert torch.equal(losses[r], losses[0])
        tol = 1e-6 if step == 1 else 2e-5
        assert np.allclose(losses[0].numpy(), ref.numpy(), rtol=tol, atol=0), (step, losses[0], ref)
        assert np.allclose(losses[0].numpy(), np.array(olosses), rtol=2e-4), (step, losses[0], olosses)
        # the replicas are bit-identical
        wts = [t.get_weights() for t in trainers]
        for r in range(1, W):
            assert trainers[r].steps == trainers[0].steps == step
            for k in wts[0]:
                assert torch.equal(wts[r][k], wts[0][k]), (r, k)
        if step == 1:
            # batch statistics (from the reduced forward sums) against the oracle's
            got_stats = _bn_stats_from_exchange(trainers[0], B)
            for bn, (m, v) in got_stats.items():
                om, ov, _ = ostats[bn]
                assert float((m - om.cpu()).abs().max()) <= 1e-5, bn
                assert float((v - ov.cpu()).abs().max()) <= 1e-5 * max(1.0, float(ov.abs().max())), bn
            # gradients (the reduced ones, on every rank, and the one-GPU fit's) against the fp64 oracle on the concatenated batch
            grads, gref = trainers[0].get_grads(), single.get_grads()
            zero_grad = [k for k in ograds if k.endswith("/bias") and "conv" in k and k != "upconv4/bias"]
            for k, og in ograds.items():
                og = og.cpu()
                scale = max(float(og.abs().max()),
                            float(ograds[k.replace("/bias", "/kernel")].abs().max()) if k in zero_grad else 0.0)
                err = float((grads[k].double() - og).abs().max())
                err_single = float((gref[k].double() - og).abs().max())
                assert err <= 2e-3 * scale + 1e-9, (k, err, scale)
                assert err_single <= 2e-3 * scale + 1e-9, ("one-GPU fit", k, err_single, scale)
            g1 = trainers[W - 1].get_grads()
            for k in grads:
                assert torch.equal(grads[k], g1[k]), k
        # Adam trajectory and moving statistics (tests/test_gpu_train.py's bounds)
        got = wts[0]
        for k in wd:
            ref_k = wd[k].cpu()
            if k.endswith("/mean") or k.endswith("/var"):
                assert float((got[k].double() - ref_k).abs().max()) <= 1e-5, (step, k)
                continue
            diff = (got[k].double() - ref_k).abs()
            assert float(diff.max()) <= 2.2e-4 * step, (step, k, float(diff.max()))
            if k not in zero_grad:
                assert float((diff <= 5e-6 * step).float().mean()) >= 0.99, (step, k)


def test_one_rank_with_a_reducer_equals_the_plain_fit():
    """W = 1 with a reducer against ofb_trainer_fit without one.  The weight gradients add with fp32 atomics in an order that
    changes from run to run, so the comparison is within the fit's own run-to-run noise, not bit for bit: two plain fits
    set the noise, and the reducer's fit must stay within a small multiple of it (or 1e-6 of the tensor's scale)."""
    from oracle import policy_torch as po
    from ofighters_b200.trainer import TrainerB200
    w = po.init_weights(5, randomize_bn=True)
    maps, vec, ta, tp, _ = _batch(8, seed=3)
    plain = [TrainerB200(weights=w, learning_rate=1e-4, batch_size=8, max_ships=8) for _ in range(2)]
    hub, (shard,) = _make_ranks(1, w, 8)
    lp = [t.fit(maps, vec, ta.cuda(), tp.cuda()).cpu() for t in plain]
    ls = run_ranks(1, lambda r: shard.fit(maps, vec, ta.cuda(), tp.cuda()).cpu())[0]
    assert hub.ranks[0].calls == 17                       # batch_global + 16 stages
    assert np.allclose(ls.numpy(), lp[0].numpy(), rtol=1e-6, atol=0)
    g0, g1, gs = plain[0].get_grads(), plain[1].get_grads(), shard.get_grads()
    for k in g0:
        scale = float(g0[k].abs().max())
        noise = float((g0[k] - g1[k]).abs().max())
        assert float((gs[k] - g0[k]).abs().max()) <= max(4.0 * noise, 1e-6 * scale, 1e-12), k
    w0, ws = plain[0].get_weights(), shard.get_weights()
    for k in w0:
        assert float((ws[k] - w0[k]).abs().max()) <= 2.2e-4, k


def test_sharded_fit_refuses_bad_batches_and_a_failing_reducer():
    from oracle import policy_torch as po
    from ofighters_b200 import _lib
    from ofighters_b200.trainer import TrainerB200
    w = po.init_weights(6, randomize_bn=True)
    maps, vec, ta, tp, _ = _batch(4, seed=5)
    plain = TrainerB200(weights=w, learning_rate=1e-4, batch_size=4, max_ships=8)
    with pytest.raises(_lib.OfbError, match="smaller than batch_local"):
        plain.fit(maps, vec, ta.cuda(), tp.cuda(), batch_global=3)
    with pytest.raises(_lib.OfbError, match="needs a reducer"):
        plain.fit(maps, vec, ta.cuda(), tp.cuda(), batch_global=8)
    assert plain.steps == 0
    hub, (tr,) = _make_ranks(1, w, 4)
    hub.ranks[0].fail_at = hub.ranks[0].calls + 5     # the batch size, then FWD_BN 0..2 pass, FWD_BN 3 fails
    with pytest.raises(_lib.OfbError, match="reducer failed at stage 3") as ei:
        run_ranks(1, lambda r: tr.fit(maps, vec, ta.cuda(), tp.cuda()))
    assert isinstance(ei.value.__cause__, RuntimeError) and "injected" in str(ei.value.__cause__)
    assert tr.steps == 0


# ------------------------------------------------------------------------------------------------ sharded replay
def _drive_shards(world, n_total, frames, make_memory, seed=21):
    """Per rank: its shard of n_total arenas, a memory, a few frames of eps-greedy play pushed."""
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.sharding import make_sharded_battleground
    from oracle import policy_torch as po
    out = []
    for r in range(world):
        bg = make_sharded_battleground(n_total, rank=r, world=world, ships={"QlearnIA": 1, "random": 6}, seed=seed)
        mem = make_memory(bg)
        pol = PolicyB200(po.init_weights(3, randomize_bn=True), max_ships=bg.n_arenas)
        maps = bg.raster("bits")
        for _ in range(frames[r]):
            iact, xy = pol.act(bg, maps, epsilon=0.5)
            mem.push(iact, xy)
            bg.frame(maps=maps)
        out.append((bg, mem, maps))
    return out


def test_uniform_draws_are_per_rank_and_from_the_ranks_own_arenas():
    from oracle import policy_torch as po
    from ofighters_b200.replay import DeviceReplayMemory
    shards = _drive_shards(2, 16, [6, 6], lambda bg: DeviceReplayMemory(bg, depth=8))
    assert [bg.arena0 for bg, _, _ in shards] == [0, 8]
    hub, trainers = _make_ranks(2, po.init_weights(2, randomize_bn=True), 4)
    draws = [[tr._rng.random() for _ in range(8)] for tr in trainers]
    assert draws[0] != draws[1]                           # rank-specific streams
    for r, (bg, mem, _) in enumerate(shards):
        n = len(mem)
        a = mem.sample(4, rng=random.Random(99))
        b = mem.gather(random.Random(99).sample(range(n), 4))
        for f in ("maps_obs", "maps_next", "vec_obs", "iaction", "pointer", "reward", "done"):
            assert torch.equal(getattr(a, f), getattr(b, f)), f
    # the two shards hold different arenas: the same positions gather different observations
    pos = list(range(4))
    assert not torch.equal(shards[0][1].gather(pos).maps_obs, shards[1][1].gather(pos).maps_obs)


def test_rescaled_weights_are_schauls_over_the_union_of_the_memories():
    from ofighters_b200.replay import PrioritizedReplayMemory
    shards = _drive_shards(3, 24, [7, 7, 7], lambda bg: PrioritizedReplayMemory(bg, depth=8, alpha=0.6, eps=1e-3,
                                                                                 seed=bg.arena0 + 1))
    beta = 0.7
    g = torch.Generator(device="cuda").manual_seed(4)
    for r, (bg, mem, _) in enumerate(shards):               # spread the masses differently on every rank
        mb = mem.sample_prioritized(8, beta)
        scale = [0.5, 3.0, 20.0][r]
        mem.update_priorities(mb.ids, torch.rand(8, device="cuda", generator=g) * scale,
                              torch.rand(8, device="cuda", generator=g) * scale)
    samples, stats = [], []
    for bg, mem, _ in shards:
        mb = mem.sample_prioritized(8, beta)
        samples.append(mb)
        stats.append(mem.sample_stats())
    ratio = torch.stack([s[1:2] / s[0:1] for s in stats]).min(dim=0).values.contiguous()
    local_w = [mb.weight.clone() for mb in samples]
    for (bg, mem, _), mb, st in zip(shards, samples, stats):
        mem.rescale_weights(mb.weight, beta, st, ratio)
    # host formula over the union: w_i = ((m_i / M_r) / g)^-beta, g = min_r m_min,r / M_r, from masses() of the valid ids
    host = []
    for bg, mem, _ in shards:
        n = len(mem)
        m = mem.masses().double().cpu()[mem._ids[:n].long().cpu()]
        host.append((float(m.sum()), float(m[m > 0].min())))
    g_host = min(mn / tot for tot, mn in host)
    for r, ((bg, mem, _), mb) in enumerate(zip(shards, samples)):
        tot, mn = host[r]
        assert math.isclose(float(stats[r][0]), tot, rel_tol=1e-12) and float(stats[r][1]) == mn
        m = mem.masses().double().cpu()[mb.ids.long().cpu()]
        want = ((m / tot) / g_host) ** -beta
        got = mb.weight.double().cpu()
        assert float(((got - want).abs() / want).max()) <= 1e-6, (r, got, want)
        assert float(got.max()) <= 1.0 + 1e-6
        assert bool((got <= local_w[r].double().cpu() * (1 + 1e-6)).all())
    # the rank holding the smallest normalised mass keeps its local weights (factor 1)
    r_min = min(range(3), key=lambda r: host[r][1] / host[r][0])
    assert torch.allclose(samples[r_min].weight, local_w[r_min], rtol=1e-6, atol=0)


@pytest.mark.parametrize("kind", ["uniform", "prioritized"])
def test_a_rank_with_an_empty_memory_makes_every_rank_skip(kind):
    from oracle import policy_torch as po
    from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory
    mk = (lambda bg: DeviceReplayMemory(bg, depth=8)) if kind == "uniform" else \
        (lambda bg: PrioritizedReplayMemory(bg, depth=8, seed=1))
    shards = _drive_shards(2, 16, [5, 1], mk)                # rank 1 pushed one frame: no transition yet
    assert len(shards[0][1]) > 0 and len(shards[1][1]) == 0
    hub, trainers = _make_ranks(2, po.init_weights(2, randomize_bn=True), 4)
    res = run_ranks(2, lambda r: trainers[r].replay(4, memory=shards[r][1], beta=0.5))
    assert res == [None, None]
    assert [t.steps for t in trainers] == [0, 0]
    assert hub.ranks[0].calls == hub.ranks[1].calls == 1    # the decision only


@pytest.mark.parametrize("kind", ["uniform", "prioritized", "nstep", "double"])
def test_batched_qlearner_runs_on_two_shards(kind):
    from oracle import policy_torch as po
    from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory
    from ofighters_b200.sharding import make_sharded_battleground
    from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos
    W, n_total = 2, 48
    w = po.init_weights(8, randomize_bn=True)
    kw = dict(target_update=2, target_tau=0.5, double_dqn=True) if kind == "double" else {}
    hub = ThreadReducer(W)

    def run(r):
        from ofighters_b200.trainer import TrainerB200
        bg = make_sharded_battleground(n_total, rank=r, world=W, ships={"QlearnIA": 1, "random": 6}, seed=31)
        tr = TrainerB200(weights=w, learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=4,
                         max_ships=bg.n_arenas, reducer=hub.ranks[r], **kw)
        if kind == "uniform":
            mem = DeviceReplayMemory(bg, depth=12)
        elif kind == "nstep":
            mem = DeviceReplayMemory(bg, depth=12, n_step=3)
        else:
            mem = PrioritizedReplayMemory(bg, depth=12, seed=7 + r, n_step=3 if kind == "double" else 1)
        bq = BatchedQLearner(tr, mem, replay_every=10, collecting_steps=5, snapshot=0)
        maps = bg.raster("bits")
        for t in range(120):
            if t == 70:
                bg.restart()
                bg.raster("bits", out=maps)
                bq.reset()
            bq.act(bg, maps)
            bg.frame(maps=maps)
        return tr.get_weights(), tr.steps, list(bq.losses)
    res = run_ranks(W, run)
    (w0, s0, l0), (w1, s1, l1) = res
    assert s0 == s1 == len(l0) == len(l1) >= 10
    assert l0 == l1 and all(math.isfinite(x) for x in l0)
    for k in w0:
        assert torch.equal(w0[k], w1[k]), k
