"""The reference-bot bridge (ofighters_b200/refbridge.py): its Observation fields equal the reference's own
Observation (build container), and a play(obs)-style bot can drive ships of one arena on the GPU."""
import numpy as np
import pytest

from oracle import ref_shim
from tests import trace_util as tu


@pytest.mark.parametrize("name", ["default_s7_seed0", "default_s7_seed1"])
def test_observation_fields_equal_the_reference_traces(name):
    """At every frame of a stored trace of the reference that keeps its full maps, the bridge's Observation built from the
    batch formats (the C restatement's observation heads, bit maps and alive flags) equals what the reference recorded:
    the 8-value head its bots were shown, its ship_map / laser_map arrays, the ships' positions, pointings and rewards,
    and done = not playable.  The vector is the head followed by both maps, row by row."""
    from ofighters_b200.refbridge import observation_fields
    from oracle.step_c import ArenasC
    gold = tu.load_golden(tu.GOLDEN_DIR + "/" + name + ".npz")
    spawn, actions = gold["spawn"], gold["actions"]
    E, T, S, _ = actions.shape
    frames = list(gold["map_frames"])
    c = ArenasC(spawn[:1])
    n_checked = n_done = 0
    for e in range(E):
        if e > 0:
            c.reset(spawn[e:e + 1])
        for t in range(T):
            c.step(actions[e, t][None])
            if t not in frames or t + 1 == T:             # the head of frame t + 1 shows the state after frame t
                continue
            heads, bits, alive = c.obs_vec()[0], c.raster_bits()[0], c.arr["ship_alive"][0]
            ref_maps = np.unpackbits(gold["maps"][e, frames.index(t)], axis=-1, bitorder="little").reshape(2, 400, 400)
            for i in range(S):
                got = observation_fields(heads[i], bits[0], bits[1], alive[i])
                assert got.vector.shape == (320008, 1) and got.vector.dtype == np.float64
                assert np.array_equal(got.vector[:8, 0].astype(np.float32), gold["obs_vec"][e, t + 1, i])
                assert np.array_equal(got.vector[8:, 0], ref_maps.reshape(-1))
                assert np.array_equal(got.ship_map, ref_maps[0]) and np.array_equal(got.laser_map, ref_maps[1])
                assert (got.pos.x, got.pos.y) == (gold["ship_x"][e, t, i], gold["ship_y"][e, t, i])
                assert (got.pointing.x, got.pointing.y) == (gold["ship_px"][e, t, i], gold["ship_py"][e, t, i])
                assert (got.dim.x, got.dim.y) == (400, 400) and got.can_shoot == gold["obs_vec"][e, t + 1, i, 1]
                assert got.reward == gold["ship_reward"][e, t, i] and got.done == (not gold["ship_alive"][e, t, i])
                n_checked += 1
                n_done += got.done
    assert n_checked >= 6 * S and 0 < n_done < n_checked      # frames with both playable ships and wreckage


@pytest.mark.reference
def test_observation_fields_equal_the_reference_observation():
    """After 30 frames of the real reference, every ship's Observation (vector, maps, head fields, done) equals what
    the bridge builds from the batch formats (8-value head + bit-packed maps + alive flag)."""
    import contextlib
    import io
    from ofighters_b200.refbridge import observation_fields
    from oracle.step_py import ArenaPy
    from oracle.traces import make_tapes
    ref = ref_shim.load()
    spawn, actions = make_tapes(3, 1, 30, 7, "random")
    arena = ref_shim.ReferenceArena(7, spawn[0], [actions[0, :, i] for i in range(7)])
    py = ArenaPy(spawn[0])
    for t in range(30):
        arena.frame()
        py.step(actions[0, t])
    bg = arena.bg

    def pack(m):
        return np.packbits(np.asarray(m, dtype=np.uint8).ravel(), bitorder="little").view(np.uint32)

    sm, lm = py.maps()
    heads = py.obs_vec()
    n_done = 0
    for i, ship in enumerate(bg.ships):
        with contextlib.redirect_stdout(io.StringIO()):
            want = ref.Observation(battleground=bg, ship=ship)          # what Ship.get_action is shown (lib/ship.py:253-258)
        got = observation_fields(heads[i].astype(np.float32), pack(sm), pack(lm), py.alive[i])
        assert got.vector.shape == (320008, 1) == want.vector.shape and got.vector.dtype == np.float64
        assert np.array_equal(got.vector, np.asarray(want.vector, dtype=np.float64))
        assert np.array_equal(got.ship_map, want.ship_map) and np.array_equal(got.laser_map, want.laser_map)
        assert (got.pos.x, got.pos.y) == (want.pos.x, want.pos.y)
        assert (got.pointing.x, got.pointing.y) == (want.pointing.x, want.pointing.y)
        assert (got.dim.x, got.dim.y) == (want.dim.x, want.dim.y)
        assert got.done == want.done and got.can_shoot == want.can_shoot and got.reward == want.reward
        n_done += got.done
    assert 0 < n_done < 7                                               # the trace has both playable ships and wreckage


def test_action_row_follows_the_reference_action_semantics():
    from types import SimpleNamespace as NS
    from ofighters_b200.refbridge import action_row
    assert action_row(None, (5, 6)).tolist() == [0, 0, 5, 6]                    # dead ship's agent returns None
    a = NS(shoot=True, thrust=True, pointing=NS(x=300, y=333))                   # both flags may be set (lib/action.py:24-41)
    assert action_row(a, (0, 0)).tolist() == [1, 1, 300, 333]
    assert action_row(NS(shoot=False, thrust=True, pointing=None), (7, 8)).tolist() == [0, 1, 7, 8]


@pytest.mark.gpu
def test_reference_style_bot_drives_one_arena():
    """A play(obs) bot plugged into arena 3 gives the same trajectory as the C restatement fed the same actions."""
    import torch
    from types import SimpleNamespace as NS
    from oracle.step_c import ArenasC
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.refbridge import ArenaView

    class ChaseBot:                                     # written against the reference's Observation / Action fields only
        def __init__(self):
            self.seen = []
        def play(self, obs):
            assert obs.vector.shape == (320008, 1) and obs.ship_map.shape == (400, 400)
            # own disk is drawn at [row=y, col=x] -- while the ship flies: a wreck is still asked (lib/ship.py:253-262) but not drawn
            assert obs.done or obs.ship_map[obs.pos.y, obs.pos.x] == 1.0 or not (0 <= obs.pos.x < 400)
            self.seen.append((obs.pos.x, obs.pos.y, obs.reward))
            ys, xs = np.nonzero(obs.ship_map)
            if xs.size == 0:
                return None
            far = np.argmax((xs - obs.pos.x) ** 2 + (ys - obs.pos.y) ** 2)
            return NS(shoot=len(self.seen) % 2 == 0, thrust=True, pointing=NS(x=int(xs[far]), y=int(ys[far])))

    N, S, k = 6, 7, 3
    c0 = ArenasC(np.zeros((N, S, 2), np.int32))
    spawn = c0.random_spawn(11, 0)
    bg = BatchedBattleground(N, ships={"external": S}, spawn_xy=torch.from_numpy(spawn))
    c = ArenasC(spawn, lcap=bg.laser_cap)
    view, bots = ArenaView(bg, k), {i: ChaseBot() for i in range(S)}
    for t in range(25):
        view.play(bots)
        acts = bg.actions.cpu().numpy().copy()
        bg.generate_frame()
        c.step(acts)
        st = bg.state(("ship_x", "ship_y", "ship_alive", "ship_score", "n_lasers"))
        for name in st:
            assert np.array_equal(st[name].cpu().numpy().astype(np.int64), c.arr[name].astype(np.int64)), (name, t)
    assert len(bots[0].seen) >= 1 and any(r != 0 for b in bots.values() for (_, _, r) in b.seen)
    assert all(len(b.seen) == 25 for b in bots.values())          # wrecks are asked too (their answer is discarded)
