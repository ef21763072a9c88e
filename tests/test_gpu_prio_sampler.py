"""The prioritized sampler (ofb_replay_sample_prioritized, csrc/ofb_replay.cu) draw by draw against the exact inverse CDF of
tests/prio_sample_oracle.py -- runs on the B200 box.

Scenes of policy ships only, pushed with iaction = 1 and idle in the frame: nobody fires, so every candidate is valid and
candidate c (ofb_replay_index's order) is the c-th transition in age order, in tile c // 2048 of the sampler.  The masses are
set with alpha = 1, eps = 0 and td_ptr = 0, so each one is exactly |td_act|.  The shapes run the tile search over one, two,
42 and thousands of tiles, the scan's chunks of per = 1 .. 4 tiles per thread, and masses that are equal, spread, span
1e-42 .. 3e38, leave whole tiles empty, or single out one candidate."""
import math
import zlib

import numpy as np
import pytest
import torch

from tests import prio_sample_oracle as so
from tests.test_gpu_prioritized_replay import _age_positions, _p, _set_masses
from tests.test_gpu_replay import _drive

pytestmark = pytest.mark.gpu

TILE = 2048
TINY = 2.0 ** -126
FLT_MAX = float(np.finfo(np.float32).max)
B_CYCLE = (1, 7, 256, 4096)
BETAS = (0.4, 1.0, 0.0, 0.7, 2.5)

# name: (arenas, policy ships, tracked arenas, depth, frames pushed, n_step) -> n_tiles
SHAPES = {
    "t1_2047": (2047, 1, 2047, 2, 2, 1),            # 1 partial tile
    "t1_2048": (2048, 1, 2048, 2, 2, 1),            # 1 full tile
    "t2_2049": (2049, 1, 2049, 2, 2, 1),            # the last tile holds one candidate
    "t42": (4096, 7, 4096, 4, 6, 1),                # 42 tiles, per = 1, the ring wrapped
    "t1024": (65536, 8, 65536, 5, 5, 1),            # per = 1, every scan thread busy
    "t1025": (65536, 8, 32800, 9, 9, 1),            # per = 2
    "t2240": (65536, 7, 65536, 11, 11, 1),          # per = 3, the trailing scan threads empty
    "t3360": (65536, 7, 65536, 16, 17, 1),          # the workload's memory (per = 4), the ring wrapped
    "t42_n3": (4096, 7, 4096, 6, 8, 3),             # an n-step memory: candidates up to frame T - 3
}
LARGEST = ("t1025", "t2240", "t3360")
REPORT = []


def _battleground(N, P):
    from ofighters_b200 import BatchedBattleground
    return BatchedBattleground(N, ships={"QlearnIA": P}, seed=0x5A + N + P)


class _Scene:
    """A prioritized memory of one shape, its candidates and its sampler counter (the calls that had candidates)."""

    def __init__(self, name, bgs):
        from ofighters_b200.replay import PrioritizedReplayMemory
        N, P, track, depth, frames, n_step = SHAPES[name]
        if (N, P) not in bgs:
            bgs[(N, P)] = _battleground(N, P)
        bg = bgs[(N, P)]
        self.mem = mem = PrioritizedReplayMemory(bg, depth=depth, track=track, alpha=1.0, eps=0.0, seed=0x1234 + depth,
                                                 n_step=n_step)
        iact = torch.ones(N * P, dtype=torch.int32, device="cuda")
        xy = torch.zeros((N * P, 2), dtype=torch.int32, device="cuda")
        for _ in range(frames):
            mem.push(iact, xy)
            bg.frame()
        cP = track * P
        self.n_cand = (min(frames, depth) - n_step) * cP
        self.n_tiles = -(-self.n_cand // TILE)
        assert len(mem) == self.n_cand, "a candidate is not valid: the scene must not fire"
        self.pos, self.ids = _age_positions(mem)
        newest = (frames - 1) % depth
        oldest = (newest - (min(frames, depth) - 1)) % depth
        c = torch.arange(self.n_cand, device="cuda")
        assert torch.equal(self.ids, ((oldest + c // cP) % depth) * cP + c % cP)     # candidate c = age position c
        self.calls = 0

    def set_masses(self, values):
        values = np.asarray(values, dtype=np.float32)
        _set_masses(self.mem, values)                     # one sample_prioritized call
        self.calls += 1
        assert np.array_equal(self.mem.masses()[self.ids].cpu().numpy(), values)


@pytest.fixture(scope="module")
def scenes():
    bgs, cache = {}, {}

    def get(name):
        if name not in cache:
            cache.clear()                                 # one large memory at a time
            torch.cuda.empty_cache()
            cache[name] = _Scene(name, bgs)
        return cache[name]

    yield get
    cache.clear()
    bgs.clear()
    for line in REPORT:
        print(line)


def _sample(scene, B, beta):
    """One ofb_replay_sample_prioritized call (no gather) -> ids, weights, its counter, the kernel's total, sample_stats."""
    mem = scene.mem
    ids = torch.empty((B,), dtype=torch.int32, device="cuda")
    w = torch.empty((B,), dtype=torch.float32, device="cuda")
    from ofighters_b200 import _lib
    _lib.check(mem._lib.ofb_replay_sample_prioritized(mem._h, B, beta, _p(ids), _p(w), _p(mem._n_valid), mem._stream()))
    counter = scene.calls
    scene.calls += 1
    return ids, w, counter, float(mem.last_total()), mem.sample_stats().cpu().numpy()


def _check_draws(scene, masses, label, calls=20):
    """`calls` samples of B in B_CYCLE against the reference of `masses` (age order) -> (draws, ambiguous draws)."""
    ref = so.Reference(masses)
    n_draws = n_amb = 0
    for k in range(calls):
        B, beta = B_CYCLE[k % len(B_CYCLE)], BETAS[k % len(BETAS)]
        ids, w, counter, total, stats = _sample(scene, B, beta)
        assert int(scene.mem._n_valid.item()) == ref.n_valid, label
        assert abs(total - ref.total) <= so.WINDOW * ref.total, (label, total, ref.total)
        assert stats[0] == total and stats[1] == ref.m_min, (label, stats, ref.m_min)
        got = scene.pos[ids.long()].cpu().numpy()
        assert (got >= 0).all(), (label, "a draw is not a candidate")
        d = ref.draw(total, so.uniforms(scene.mem.seed, counter, B), B)
        wrong = np.flatnonzero(~d.ambiguous & (got != d.pos))
        assert wrong.size == 0, (label, k, B, [(int(b), int(got[b]), int(d.pos[b]), float(d.u[b])) for b in wrong[:8]])
        assert ((got >= d.lo) & (got <= d.hi)).all(), (label, k, "an ambiguous draw left its window")
        assert (ref.m[got] > 0).all() and (np.diff(got) >= 0).all(), label
        wg, wr = w.cpu().numpy().astype(np.float64), ref.weights(got, beta)
        assert (wg <= 1.0).all(), (label, float(wg.max()))
        normal = wr >= TINY
        bad = np.flatnonzero(normal & ~np.isclose(wg, wr, rtol=1e-5, atol=0))
        assert bad.size == 0, (label, beta, [(float(ref.m[got[b]]), float(wg[b]), float(wr[b])) for b in bad[:8]])
        assert (wg[~normal] <= TINY).all(), label
        n_draws += B
        n_amb += int(d.ambiguous.sum())
    REPORT.append("{}: {} draws, {} ambiguous".format(label, n_draws, n_amb))
    assert n_amb <= 1e-3 * n_draws, (label, n_amb, n_draws)
    return n_draws, n_amb


def _pattern(name, n, T, rng):
    """Masses of n candidates (T tiles) in candidate order."""
    if name == "a":
        return np.full(n, 1.5, dtype=np.float32)
    if name == "b":
        return rng.uniform(0.5, 2.0, n).astype(np.float32)
    if name == "c":
        m = (10.0 ** rng.uniform(-30.0, 30.0, n)).astype(np.float32)
        m[rng.choice(n, 5, replace=False)] = 1e-42                        # subnormal
        m[rng.choice(n, 5, replace=False)] = 3e38
        return m
    if name == "d":
        empty = np.zeros(T, dtype=bool)
        empty[0] = True                                                   # the first tile
        for start, run in ((2, 1), (5, 2), (10, 5), (T // 3, 2)):         # interior runs, across scan chunks
            empty[start:start + run] = True
        empty[T // 2:(3 * T) // 4:2] = True                               # every other tile
        empty[T - max(1, T // 8):] = True                                 # every tile after last_tile
        if T == 2:
            empty[:] = [True, False]
        m = rng.uniform(0.5, 2.0, n).astype(np.float32)
        m[empty[np.arange(n) // TILE]] = 0
        assert m.any() and (T < 3 or not m[-1])
        return m
    raise ValueError(name)


_CASES = [(s, p) for s in SHAPES if s != "t42_n3" for p in "abcd"
          if not (p == "b" and s in LARGEST) and not (p == "d" and s.startswith("t1_"))]


@pytest.mark.parametrize("shape, pattern", _CASES)
def test_draws_match_the_exact_inverse_cdf(scenes, shape, pattern):
    sc = scenes(shape)
    rng = np.random.default_rng(zlib.crc32((shape + pattern).encode()))
    m = _pattern(pattern, sc.n_cand, sc.n_tiles, rng)
    sc.set_masses(m)
    _check_draws(sc, m, "{} ({} tiles) {}".format(shape, sc.n_tiles, pattern))


@pytest.mark.parametrize("shape", [s for s in SHAPES if s != "t42_n3"])
def test_a_single_non_zero_candidate_takes_every_draw(scenes, shape):
    sc = scenes(shape)
    for c in sorted({0, 2047, 2048, sc.n_cand - 1} & set(range(sc.n_cand))):
        m = np.zeros(sc.n_cand, dtype=np.float32)
        m[c] = 3.7
        sc.set_masses(m)
        for B in B_CYCLE:
            ids, w, _, total, _ = _sample(sc, B, 0.6)
            assert (sc.pos[ids.long()] == c).all() and (w == 1.0).all(), (shape, c, B)
            assert int(sc.mem._n_valid.item()) == 1 and total == np.float32(3.7)
        _check_draws(sc, m, "{} single candidate {}".format(shape, c), calls=4)


@pytest.mark.parametrize("shape", [s for s in SHAPES if s != "t42_n3"])
def test_all_zero_masses_draw_nothing(scenes, shape):
    from ofighters_b200.replay import EmptyReplayMemory
    sc = scenes(shape)
    sc.set_masses(np.zeros(sc.n_cand, dtype=np.float32))
    with pytest.raises(EmptyReplayMemory):
        sc.mem.sample_prioritized(8, 0.5)
    sc.calls += 1                                          # an all-zero memory still counts
    assert int(sc.mem._n_valid.item()) == 0 and float(sc.mem.last_total()) == 0.0
    one = torch.ones(sc.n_cand, device="cuda")
    sc.mem.update_priorities(sc.ids.int().contiguous(), one, torch.zeros_like(one))   # the counter goes on
    _check_draws(sc, np.ones(sc.n_cand, dtype=np.float32), "{} after all-zero".format(shape), calls=2)


@pytest.mark.parametrize("pattern", ["b", "d"])
def test_n_step_memory_draws_from_its_reduced_range(scenes, pattern):
    sc = scenes("t42_n3")
    assert sc.n_cand == 3 * 4096 * 7 and sc.n_tiles == 42
    m = _pattern(pattern, sc.n_cand, sc.n_tiles, np.random.default_rng(31))
    sc.set_masses(m)
    _check_draws(sc, m, "t42_n3 {}".format(pattern))


def test_a_real_scene_with_invalid_candidates():
    """Deaths, a masked restart and a ring wrap: the reference draws over the valid transitions in age order, the invalid
    candidates between them carry no mass."""
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.policy import PolicyB200
    from ofighters_b200.replay import PrioritizedReplayMemory
    N, D, T = 4096, 8, 14
    bg = BatchedBattleground(N, ships={"QlearnIA": 3, "random": 2, "turret": 2}, seed=17)
    mem = PrioritizedReplayMemory(bg, depth=D, alpha=1.0, eps=0.0, seed=99)
    mask = torch.arange(N) % 3 == 0
    _drive(bg, mem, PolicyB200.random_init(max_ships=N, seed=2), T, restarts={4: None, 9: mask},
           keep_maps=torch.zeros(1, dtype=torch.long, device="cuda"))
    n = len(mem)
    n_cand = (D - 1) * N * 3
    assert 0.5 * n_cand < n < n_cand, (n, n_cand)                          # invalid candidates are among them
    pos, ids = _age_positions(mem)

    class Sc:
        pass

    sc = Sc()
    sc.mem, sc.pos, sc.ids, sc.calls = mem, pos, ids, 0
    rng = np.random.default_rng(5)
    m = rng.uniform(0.5, 2.0, n).astype(np.float32)
    m[rng.random(n) < 0.2] = 0
    m[: n // 50] = 0
    _set_masses(mem, m)
    sc.calls += 1
    assert np.array_equal(mem.masses()[ids].cpu().numpy(), m)
    _check_draws(sc, m, "real scene ({} valid of {} candidates)".format(n, n_cand))


def test_update_priorities_edges():
    from ofighters_b200.replay import PrioritizedReplayMemory
    bg = _battleground(64, 7)
    iact = torch.ones(64 * 7, dtype=torch.int32, device="cuda")
    xy = torch.zeros((64 * 7, 2), dtype=torch.int32, device="cuda")
    sub = float(np.float32(1e-40))
    vals = [0.0, -0.0, sub, -sub, 1e-45, 1e-30, 1e30, -1e30, math.inf, -math.inf, math.nan, 1.0, -2.5, 3e38, 1e-20, 7.0]
    da = np.array([a for a in vals for _ in vals], dtype=np.float32)
    dp = np.array([p for _ in vals for p in vals], dtype=np.float32)
    for alpha in (0.0, 0.6, 1.0, 2.5):
        for eps in (0.0, 1e-6):
            mem = PrioritizedReplayMemory(bg, depth=3, alpha=alpha, eps=eps, seed=3)
            for _ in range(3):
                mem.push(iact, xy)
                bg.frame()
            pos, ids = _age_positions(mem)
            assert ids.numel() == 2 * 64 * 7 >= da.size
            mem.sample_prioritized(1, 0.0)
            sel = ids[:da.size].int().contiguous()
            mem.update_priorities(sel, torch.from_numpy(da).cuda(), torch.from_numpy(dp).cuda())
            with np.errstate(over="ignore", invalid="ignore"):
                x = (np.abs(da.astype(np.float64)) + np.abs(dp.astype(np.float64)) + float(np.float32(eps))) ** \
                    float(np.float32(alpha))                              # the memory keeps alpha and eps in fp32
                want = x.astype(np.float32)
            want[~(want <= FLT_MAX)] = FLT_MAX                             # non-finite errors (and overflow) clamp
            got = mem.masses()[sel.long()].cpu().numpy()
            ulp = np.spacing(want)
            assert (np.abs(got.astype(np.float64) - want) <= ulp).all(), (alpha, eps, got[got != want][:8], want[got != want][:8])
            assert float(mem.max_mass()) == max(1.0, float(got.max()))
            zero = np.flatnonzero(got == 0)
            if eps == 0.0 and alpha > 0:
                assert zero.size > 0                                      # 0 and underflowing errors
                if alpha == 2.5:
                    assert (np.flatnonzero((want == 0) & (x > 0)).size > 0)   # (1e-30)^2.5 underflows to 0
            else:
                assert zero.size == 0
            drawn = torch.zeros(ids.numel(), dtype=torch.bool, device="cuda")
            for _ in range(6):
                s = mem.sample_prioritized(4096, 0.4)
                drawn[pos[s.ids.long()]] = True
                assert bool((s.weight <= 1.0).all()) and bool((s.weight >= 0.0).all())
            assert not drawn[torch.from_numpy(zero).cuda()].any(), "a zero mass was drawn"
