"""Parity of the CUDA arena path (K1 step, K2 raster, bots, reset) -- runs on the B200 box.

Everything goes through libofb.so's C ABI (via ofighters_b200.BatchedBattleground) and is
compared bit-for-bit with (a) the committed traces of the real reference and (b) the C
restatement on the same seeded inputs.
"""
import numpy as np
import pytest
import torch

from tests import trace_util as tu

pytestmark = pytest.mark.gpu

STATE_CMP = ("time", "n_lasers", "kills", "deaths", "shots", "overflow", "ship_x", "ship_y", "ship_px", "ship_py",
             "ship_alive", "ship_hull", "ship_reward", "ship_score", "ship_steps")


def _gpu():
    from tests.gpu_util import GpuEngine
    return GpuEngine


@pytest.mark.parametrize("path", tu.golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_cuda_path_matches_reference_trace(path):
    gold = tu.load_golden(path)
    bad = tu.run_engine(_gpu(), gold, n_copies=5)
    assert bad == []


@pytest.mark.parametrize("path", tu.golden_files(), ids=lambda p: p.split("/")[-1][:-4])
def test_fused_frame_matches_reference_trace(path):
    """The fused frame kernel (ofb_frame: step + observation maps in one launch) against the real reference's traces."""
    from tests.gpu_util import GpuEngineFused
    gold = tu.load_golden(path)
    bad = tu.run_engine(GpuEngineFused, gold, n_copies=5)
    assert bad == []


@pytest.mark.parametrize("N,S,kind,T,lcap", [(4096, 7, "random", 230, 0), (20000, 7, "random", 60, 0), (700, 7, "turret", 120, 0),
                                             (333, 12, "random", 90, 0), (150, 32, "stress", 40, 2048),
                                             (3000, 32, "stress", 40, 0), (5, 1, "random", 30, 0)])
def test_fused_frame_equals_step_then_raster(N, S, kind, T, lcap):
    _fused_vs_split(N, S, kind, T, lcap)
    from ofighters_b200 import _lib
    assert _lib.load().ofb_debug_last_frame_fused() == 1      # every shape here fits the ring: one launch per frame


@pytest.mark.parametrize("knobs", [dict(OFB_FRAME_K="19"), dict(OFB_FRAME_K="9"), dict(OFB_FRAME_LPA="32", OFB_FRAME_SW="8"),
                                   dict(OFB_FRAME_LPA="16", OFB_FRAME_SW="4", OFB_FRAME_NG="3", OFB_FRAME_NBUF="1"),
                                   dict(OFB_FRAME_LPA="16", OFB_FRAME_SW="8", OFB_FRAME_NG="1", OFB_FRAME_NBUF="3"),
                                   dict(OFB_FRAME_LPA="8", OFB_FRAME_SW="8", OFB_FRAME_NG="1", OFB_FRAME_NBUF="3"),
                                   dict(OFB_FRAME_LPA="32", OFB_FRAME_SW="12", OFB_FRAME_NG="1", OFB_FRAME_NBUF="3"),
                                   dict(OFB_FRAME_LPA="8", OFB_FRAME_SW="8", OFB_FRAME_NG="2", OFB_FRAME_NBUF="1"), dict(OFB_FRAME_POSTCAP="8"), dict(OFB_FRAME_SPLIT="1")],
                         ids=lambda d: ",".join("%s=%s" % (k[10:], v) for k, v in d.items()))
def test_fused_frame_ring_geometries(knobs, monkeypatch):
    """The shared-memory ring of the fused kernel under other geometries (slots, stepper warps, raster groups)."""
    monkeypatch.setenv("OFB_FRAME_TUNE", "1")            # the knobs are only read when tuning is switched on
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    _fused_vs_split(9000, 7, "random", 50, 0)
    from ofighters_b200 import _lib
    # the geometry is instantiated: this was the fused kernel (OFB_FRAME_SPLIT forces the two-launch form of ofb_frame)
    assert _lib.load().ofb_debug_last_frame_fused() == (0 if "OFB_FRAME_SPLIT" in knobs else 1)


@pytest.mark.parametrize("N", [1, 2, 31, 147, 148, 149, 443])
@pytest.mark.parametrize("S", [2, 7, 20])
def test_fused_frame_ragged_batches(N, S):
    """Arena counts around the SM count (one CTA per SM: ranges of 0, 1, 2 and 3 arenas) and other ship counts."""
    _fused_vs_split(N, S, "turret", 25, 0)


def _fused_vs_split(N, S, kind, T, lcap):
    """ofb_frame_bots == ofb_step_bots + ofb_raster bit for bit (state, observation heads, maps), incl. the episode
    restart, arena ranges longer than the shared-memory ring, saturated laser lists (overflow counted identically) and
    laser lists longer than a ring slot (read back from the arena block)."""
    from ofighters_b200 import ArenaConfig, BatchedBattleground
    mk = lambda: BatchedBattleground(N, ships={kind: S}, config=ArenaConfig(laser_cap=lcap), seed=4242, arena0=17)
    a, b = mk(), mk()
    maps_a = a.raster("bits")
    maps_b = torch.zeros_like(maps_a)
    for t in range(T):
        if t == 200 or (T < 200 and t == T // 2):
            a.restart()
            b.restart()
        a.frame()
        a.raster("bits", out=maps_a)
        b.frame(maps=maps_b)
        if t % 9 == 0 or t == T - 1:
            assert torch.equal(maps_a, maps_b), "maps t %d" % t
            assert torch.equal(a.obs_vec, b.obs_vec), "obs t %d" % t
    sa, sb = a.state(), b.state()
    live = torch.arange(a.laser_cap, device=a.device)[None, :] < sa["n_lasers"].long()[:, None]
    for k in sa:
        if k.startswith("laser_"):
            assert torch.equal(torch.where(live, sa[k], torch.zeros_like(sa[k])),
                               torch.where(live, sb[k], torch.zeros_like(sb[k]))), k
        else:
            assert torch.equal(sa[k], sb[k]), k


def _compare_states(g, c, tag):
    from oracle.step_c import ArenasC  # noqa: F401  (oracle = checker only)
    ga = g.arrays()
    for k in STATE_CMP:
        assert np.array_equal(ga[k].astype(np.int64), c.arr[k].astype(np.int64)), "%s %s" % (k, tag)
    n = c.arr["n_lasers"]
    L = min(ga["laser_x"].shape[1], c.arr["laser_x"].shape[1])
    live = np.arange(L)[None, :] < n[:, None]
    for k in ("laser_x", "laser_y", "laser_owner", "laser_destroyed"):
        assert np.array_equal(np.where(live, ga[k][:, :L], 0), np.where(live, c.arr[k][:, :L], 0)), "%s %s" % (k, tag)


@pytest.mark.parametrize("N,S,kind,T", [(1500, 7, "random", 200), (300, 32, "stress", 60), (257, 12, "turret", 120),
                                        (64, 1, "random", 50), (33, 16, "runner", 80)])
def test_cuda_path_matches_c_restatement_on_device_bots(N, S, kind, T):
    """Device bots + step + reset + raster vs the C restatement, same Philox stream."""
    from oracle.step_c import ArenasC
    from ofighters_b200 import _lib
    GpuEngine = _gpu()
    seed = 0xC0FFEE + N
    c0 = ArenasC(np.zeros((N, S, 2), np.int32))
    spawn = c0.random_spawn(seed, 0, arena0=1000)
    g = GpuEngine(spawn, lcap=64 * S if kind in ("turret", "shoot") else 0, seed=seed, arena0=1000)
    bg = g.bg
    c = ArenasC(spawn, lcap=bg.laser_cap)
    # device-side spawn draws must equal the oracle's
    bg._draw_spawn(0)
    assert np.array_equal(bg._spawn.cpu().numpy(), spawn)
    kinds = torch.full((S,), _lib.BOT_KINDS[kind], dtype=torch.uint8, device=bg.device)
    for ep in range(2):
        for t in range(T):
            step = ep * T + t
            bg._lib.ofb_bot_actions(bg._h, 0, kinds.data_ptr(), seed, 1000, step, bg.actions.data_ptr(), None)
            torch.cuda.synchronize()
            acts = c.bot_actions(kind, seed, step, arena0=1000)
            assert np.array_equal(bg.actions.cpu().numpy(), acts), "bot actions step %d" % step
            assert np.array_equal(g.obs_vec(), c.obs_vec()), "obs step %d" % step
            bg.generate_frame()
            c.step(acts)
            if t % 7 == 0 or t == T - 1:
                _compare_states(g, c, "ep %d t %d" % (ep, t))
            if t % 25 == 3:
                assert np.array_equal(g.raster_bits(), c.raster_bits()), "raster ep %d t %d" % (ep, t)
        sp = c.random_spawn(seed, ep + 1, arena0=1000)
        g.reset(sp)
        c.reset(sp)
        assert np.array_equal(bg.stats.cpu().numpy(), c.arr["stats"])
    assert int(g.arrays()["overflow"].sum()) == 0


def test_raster_dense_formats_agree_with_bits():
    from oracle.step_c import ArenasC
    GpuEngine = _gpu()
    N, S = 48, 7
    c = ArenasC(np.zeros((N, S, 2), np.int32))
    spawn = c.random_spawn(5, 0)
    g = GpuEngine(spawn)
    c = ArenasC(spawn, lcap=g.bg.laser_cap)
    for t in range(40):
        a = c.bot_actions("random", 5, t)
        g.step(a)
        c.step(a)
    bits = g.raster_bits()
    assert np.array_equal(bits, c.raster_bits())
    dense = np.unpackbits(bits.view(np.uint8).reshape(N, 2, -1), axis=2, bitorder="little").reshape(N, 2, 400, 400)
    dense = dense.transpose(0, 2, 3, 1)                                   # NHWC
    u8 = g.bg.raster("u8").cpu().numpy()
    assert np.array_equal(u8, dense)
    bf = g.bg.raster("bf16").float().cpu().numpy()
    assert np.array_equal(bf, dense.astype(np.float32))


def test_partial_reset_mask_and_arena_view():
    from oracle.step_c import ArenasC
    GpuEngine = _gpu()
    N, S = 40, 7
    c = ArenasC(np.zeros((N, S, 2), np.int32))
    spawn = c.random_spawn(9, 0)
    g = GpuEngine(spawn)
    c = ArenasC(spawn, lcap=g.bg.laser_cap)
    for t in range(30):
        a = c.bot_actions("random", 9, t)
        g.step(a)
        c.step(a)
    mask = (np.arange(N) % 3 == 0)
    sp = c.random_spawn(9, 1)
    g.bg.restart(mask=torch.from_numpy(mask), spawn_xy=torch.from_numpy(sp))
    c.reset(sp, mask=mask)
    _compare_states(g, c, "after masked reset")
    view = g.bg.arena(3)
    assert view.ships[2].body.x == int(c.arr["ship_x"][3, 2])
    assert len(view.lasers) == int(c.arr["n_lasers"][3])
    assert view.ships[0].state in ("flying", "destroyed")


def test_running_stats_equal_the_episode_end_stats():
    """ofb_stats mid-episode == what ofb_reset adds at the episode's end (plus the rewards still pending)."""
    from ofighters_b200 import BatchedBattleground
    bg = BatchedBattleground(300, ships={"turret": 7}, seed=12)
    for _ in range(80):
        bg.frame()
    run = bg.running_stats().cpu()
    st = bg.state()
    assert int(run[0]) == int(st["ship_score"].sum() + st["ship_reward"].sum())
    assert run[1:].tolist() == [int(st["kills"].sum()), int(st["deaths"].sum()), int(st["shots"].sum()), 300 * 7, 300]
    bg.restart()
    end = bg.stats.cpu()
    assert end[1:].tolist() == run[1:].tolist() and int(end[0]) == int(st["ship_score"].sum())
    a = bg.absolute_state
    assert tuple(a.maps.shape) == (300, 2, 5000) and a.obs_vec is bg.obs_vec


def test_errors_are_loud():
    from ofighters_b200 import BatchedBattleground
    with pytest.raises(Exception, match="ships argument must be int or dict"):
        BatchedBattleground(4, ships="seven")
    bg = BatchedBattleground(4, ships=3)
    with pytest.raises(Exception, match="Invalid actions"):
        bg.generate_frame(torch.zeros((4, 3, 5), dtype=torch.int16, device=bg.device))
    with pytest.raises(Exception):
        BatchedBattleground(4, ships=33)


def test_sharded_arenas_equal_the_unsharded_run():
    """Arena-level sharding (SURVEY 8(e)): slices keyed by global arena id reproduce the whole batch."""
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.sharding import shard_range
    N, T = 101, 45
    whole = BatchedBattleground(N, ships={"random": 7}, seed=77)
    parts = []
    for r in range(3):
        lo, hi = shard_range(N, r, 3)
        parts.append(BatchedBattleground(hi - lo, ships={"random": 7}, seed=77, arena0=lo))
    for t in range(T):
        whole.frame()
        for p in parts:
            p.frame()
    whole.restart()
    for p in parts:
        p.restart()
    w = whole.state()
    ps = [p.state() for p in parts]
    for k in ("ship_x", "ship_y", "ship_px", "ship_py", "ship_alive", "ship_reward", "ship_score", "n_lasers", "kills"):
        assert torch.equal(torch.cat([q[k] for q in ps]), w[k]), k
    assert torch.equal(sum(p.stats for p in parts), whole.stats)
    assert torch.equal(torch.cat([p.raster("bits") for p in parts]), whole.raster("bits"))


@pytest.mark.parametrize("wait", [True, False], ids=["sync", "pipelined"])
def test_host_tape_replay_matches_c_restatement(wait):
    """ofb_step_host / ofb_step_host_async: a HOST action tape replayed frame by frame gives the oracle's state,
    and every frame's observation heads land in the host buffer they were queued for."""
    from oracle.step_c import ArenasC
    GpuEngine = _gpu()
    N, S, T = 211, 7, 60
    c = ArenasC(np.zeros((N, S, 2), np.int32))
    spawn = c.random_spawn(21, 0)
    g = GpuEngine(spawn)
    bg = g.bg
    c = ArenasC(spawn, lcap=bg.laser_cap)
    tape = torch.empty((T, N, S, 4), dtype=torch.int16).pin_memory()
    obs = torch.full((T, N, S, 8), float("nan"), dtype=torch.float32).pin_memory()
    want_obs = np.empty((T, N, S, 8), np.float32)
    for t in range(T):
        a = c.bot_actions("random", 21, t)
        tape[t].copy_(torch.from_numpy(a))
        c.step(a)
        want_obs[t] = c.obs_vec()
    maps = bg.raster("bits")
    for t in range(T):
        if wait:
            bg.step_host(tape[t], obs[t], wait=True)
            bg.raster("bits", out=maps)
        else:                                            # pipelined copies around the fused frame kernel
            bg.step_host(tape[t], obs[t], wait=False, maps=maps)
    bg.wait_host()
    torch.cuda.synchronize()
    _compare_states(g, c, "after host tape")
    assert np.array_equal(obs.numpy(), want_obs)
    assert np.array_equal(maps.cpu().numpy().view(np.uint32), c.raster_bits())


def test_record_replay_roundtrip(tmp_path):
    """BatchedRecord (lib/record.py counterpart): a device-bot run recorded from frame 0 and again from mid-episode,
    saved to .orec, loaded and replayed through the host-buffer path reproduces the run bit for bit -- and the
    C restatement fed the same tape agrees."""
    from oracle.step_c import ArenasC
    from ofighters_b200 import BatchedBattleground
    from ofighters_b200.record import BatchedRecord
    N, S = 37, 7
    bg = BatchedBattleground(N, ships={"random": S}, seed=99)
    c = ArenasC(bg._spawn.cpu().numpy(), lcap=bg.laser_cap)
    rec, mid = BatchedRecord(bg, capacity=8), None
    for t in range(40):
        if t == 17:
            mid = BatchedRecord(bg)                      # initial state with live lasers and dead ships
        if t == 25:
            bg.restart()
            c.reset(bg._spawn.cpu().numpy())
            for r in (rec, mid):
                r.saveReset(bg._spawn)
        acts = bg.request_actions()
        for r in (rec, mid):
            if r is not None:
                r.saveFrame(acts)
        c.step(acts.cpu().numpy())
        bg.generate_frame()
    want = {k: v.cpu() for k, v in bg.state().items()}
    for k in ("ship_x", "ship_y", "ship_alive", "ship_score", "ship_steps", "n_lasers", "kills"):
        assert np.array_equal(want[k].numpy().astype(np.int64), c.arr[k].astype(np.int64)), k
    for r, frames, tag in ((rec, 40, "full"), (mid, 23, "mid")):
        path = r.save(str(tmp_path / tag))
        assert path.endswith(".orec")
        r2 = BatchedRecord.load(path)
        assert r2.n_frames == frames and str(r2).startswith("BatchedRecord(%d frames" % frames)
        game = None
        for _ in range(frames):
            game = r2.nextFrame()
        game.wait_host()
        torch.cuda.synchronize()
        got = {k: v.cpu() for k, v in game.state().items()}
        for k in want:
            if k.startswith("laser_"):
                live = torch.arange(want[k].shape[1])[None, :] < want["n_lasers"].long()[:, None]
                assert torch.equal(torch.where(live, got[k], torch.zeros_like(got[k])),
                                   torch.where(live, want[k], torch.zeros_like(want[k]))), (tag, k)
            elif k != "episode":
                assert torch.equal(got[k], want[k]), (tag, k)
        assert np.array_equal(r2.obs_host.numpy(), bg.obs_vec.cpu().numpy()), tag
        with pytest.raises(Exception, match="end of record"):
            r2.nextFrame()


def test_compact_observation_heads_roundtrip_and_pipelined_host_path():
    """lib/observation.py:119-123: can_shoot is always 1 and dim is the map size, so the 5 remaining entries of a head (exact
    small integers) travel to the host as int16 [N,S,5] (ofb_obs_pack_i16): expanding them gives the float32 heads back, and the
    pipelined host loop (ofb_frame_host_async_i16) delivers exactly what the float32 path delivers."""
    import torch
    from ofighters_b200 import BatchedBattleground
    N, S, T = 300, 7, 24
    a = BatchedBattleground(N, ships={"random": S}, seed=9)
    b = BatchedBattleground(N, ships={"external": S}, seed=9)
    c = BatchedBattleground(N, ships={"external": S}, seed=9)
    maps_b, maps_c = b.raster("bits"), c.raster("bits")
    tape = torch.empty((T, N, S, 4), dtype=torch.int16).pin_memory()
    obs16 = [torch.empty((N, S, 5), dtype=torch.int16).pin_memory() for _ in range(2)]
    obs32 = [torch.empty((N, S, 8), dtype=torch.float32).pin_memory() for _ in range(2)]
    for t in range(T):
        tape[t].copy_(a.request_actions())
        a.generate_frame()
        assert torch.equal(a.expand_obs(a.obs_compact()), a.obs_vec)
    for t in range(T):
        b.step_host(tape[t], obs16[t & 1], wait=False, maps=maps_b)
        c.step_host(tape[t], obs32[t & 1], wait=False, maps=maps_c)
    b.wait_host()
    c.wait_host()
    torch.cuda.synchronize()
    assert torch.equal(b.expand_obs(obs16[(T - 1) & 1]), obs32[(T - 1) & 1])
    assert torch.equal(obs32[(T - 1) & 1], a.obs_vec.cpu()) and torch.equal(maps_b, maps_c)
    with pytest.raises(Exception, match="compact"):
        b.step_host(tape[0], obs16[0], wait=True)


def test_host_wait_covers_the_action_copy_without_observation_buffer():
    """ADVICE r1: step_host(obs_host=None, wait=False) followed by wait_host() must mean that the pinned action buffer has been
    consumed: overwriting it afterwards may not change the replay."""
    import torch
    from ofighters_b200 import BatchedBattleground
    N, S, T = 20000, 7, 12
    src = BatchedBattleground(N, ships={"random": S}, seed=4)
    tape = []
    for t in range(T):
        tape.append(src.request_actions().cpu().clone())
        src.generate_frame()
    rep = BatchedBattleground(N, ships={"external": S}, seed=4)
    buf = torch.empty((N, S, 4), dtype=torch.int16).pin_memory()
    for t in range(T):
        buf.copy_(tape[t])
        rep.step_host(buf, None, wait=False)
        rep.wait_host()
        buf.fill_(-1)                                    # scribble over the tape: the frame must already have its copy
    want, got = src.state(("ship_x", "ship_y", "ship_score", "n_lasers")), rep.state(("ship_x", "ship_y", "ship_score", "n_lasers"))
    assert all(torch.equal(want[k], got[k]) for k in want)


def _bench_dump(out_dir, workload, steps):
    """Runs bench.py --dump-outputs (3 warm-up steps, without the extra measurements) and loads what it wrote."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", workload, "--steps", str(steps), "--warmup", "3",
                    "--dump-outputs", str(out_dir)], check=True, timeout=900, stdout=subprocess.DEVNULL,
                   env=dict(os.environ, OFB_BENCH_NO_EXTRA="1"))
    d = {f[:-4]: np.load(os.path.join(str(out_dir), f)) for f in os.listdir(str(out_dir))}
    assert all(v.dtype in (np.float32, np.float64) for v in d.values())
    assert sum(v.nbytes for v in d.values()) <= 64 * 2 ** 20
    return d


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs on arena4096 with 4 timed steps: the pre-roll puts the episode restart inside them, so the last
    step is frame 2 of episode 1 (202 frames in all).  The sampled arenas' state, observation heads and maps equal the C
    restatement's after the same 202 seeded frames, and every file is float32 / float64, 64 MB at most in all."""
    from oracle.step_c import ArenasC
    d = _bench_dump(tmp_path, "arena4096", 4)
    ids = d["arena_ids"].astype(np.int64)
    assert len(ids) == 512 and np.all(np.diff(ids) > 0) and ids[-1] < 4096
    assert np.all(d["time"] == 2)
    N, S, seed = 4096, 7, 0x0F16
    c = ArenasC(ArenasC(np.zeros((N, S, 2), np.int32)).random_spawn(seed, 0))
    for it in range(202):
        if it == 200:
            c.reset(c.random_spawn(seed, 1))
        c.step(c.bot_actions("random", seed, it))
    for k in ("time", "ship_x", "ship_y", "ship_px", "ship_py", "ship_alive", "ship_hull", "ship_score", "n_lasers", "kills", "deaths"):
        assert np.array_equal(d[k], c.arr[k][ids]), k
    n = int(d["n_lasers"].max())
    live = np.arange(n)[None, :] < d["n_lasers"][:, None]
    assert np.array_equal(d["laser_x"][:, :n], np.where(live, c.arr["laser_x"][ids, :n], 0))
    assert np.array_equal(d["obs_vec"], c.obs_vec()[ids])
    assert np.array_equal(d["maps"], c.raster_bits()[ids[:128]])
    assert np.array_equal(d["stats"], c.arr["stats"])
    assert d["actions"].shape == (512, S, 4) and not d["actions"].any()     # scripted bots draw their actions in the frame kernel
    assert "policy_iaction" not in d


def test_bench_dump_outputs_carry_the_played_policy_actions(tmp_path):
    """bench.py --dump-outputs on policy7 (all 7 ships driven by the policy forward): policy_iaction / policy_xy hold one
    played action per sampled arena and ship, and the dumped action rows are exactly those actions, [iaction == 0 (shoot),
    iaction == 1 (thrust), x, y] (QlearnIA.play's action vector)."""
    d = _bench_dump(tmp_path, "policy7", 2)
    ia, xy, act = d["policy_iaction"], d["policy_xy"], d["actions"]
    assert ia.shape == (512, 7) and xy.shape == (512, 7, 2) and act.shape == (512, 7, 4)
    assert np.isin(ia, (0, 1)).all() and ((xy >= 0) & (xy < 400)).all()
    assert np.array_equal(act[..., 0], ia == 0) and np.array_equal(act[..., 1], ia == 1) and np.array_equal(act[..., 2:], xy)
    assert xy.any()                                      # rows were really written (a zero buffer would agree with zeros)
