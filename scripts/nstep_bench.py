"""Cost and effect of n-step returns in the device replay memory (DeviceReplayMemory / PrioritizedReplayMemory with n_step) at
configs[2]: 65 536 arenas x 7 ships, ship 0 policy-driven, depth 16.
  * gather_nstep at n = 1, 3, 5 against the one-step gather at B = 8 / 256 (rings full and wrapped, the same frames pushed into
    each memory; CUDA events around the C calls alone, outputs preallocated, 50 calls per figure);
  * td_targets_discounted against td_targets at B = 256;
  * BatchedQLearner per frame over 400 frames (the restart at frame 200 inside), n = 1 against n = 3, uniform and prioritized,
    trainer batch 8, two runs per arm with the arms alternated; beside each, the share of transitions with R != 0 or done = 1
    among those replayed and among all the transitions the memory holds at the end of the run (the indicator DESIGN.md §5
    reports for n = 1; not a pass criterion).
The card's name and power limit are read in the same run.
Usage: python scripts/nstep_bench.py [--frames 400] [--out FILE]  -> one JSON line (and FILE)."""
import argparse
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from learn_bench import card, events_ms  # noqa: E402
from ofighters_b200 import ArenaConfig, BatchedBattleground, _lib  # noqa: E402
from ofighters_b200.policy import PolicyB200  # noqa: E402
from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory  # noqa: E402
from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200  # noqa: E402

SEED, MAX_TIME, DEPTH, N, GAMMA = 0x0F16, 200, 16, 65536, 0.9
SHIPS = {"QlearnIA": 1, "random": 6}
NS = (1, 3, 5)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _outputs(B, words):
    z = lambda shape, dt: torch.empty(shape, dtype=dt, device="cuda")      # noqa: E731
    return [z((B, 2, words), torch.int32), z((B, 8), torch.float32), z((B, 2, words), torch.int32), z((B, 8), torch.float32),
            z((B,), torch.int32), z((B, 2), torch.int32), z((B,), torch.float32), z((B,), torch.uint8), z((B,), torch.float32),
            z((B,), torch.int32)]


def rare_fraction(lib, mem, s):
    """Share of the memory's transitions with R != 0 or done = 1: their scalar fields gathered without the maps."""
    n = len(mem)
    ids = mem._ids[:n].contiguous()
    R = torch.empty(n, dtype=torch.float32, device="cuda")
    d = torch.empty(n, dtype=torch.uint8, device="cuda")
    if mem.n_step > 1:
        _lib.check(lib.ofb_replay_gather_nstep(mem._h, _p(ids), n, GAMMA, *[None] * 6, _p(R), _p(d), None, None, s))
    else:
        _lib.check(lib.ofb_replay_gather(mem._h, _p(ids), n, *[None] * 6, _p(R), _p(d), s))
    return float(((R != 0) | (d != 0)).double().mean()), n


def gather_costs(lib, s):
    bg = BatchedBattleground(N, ships=SHIPS, config=ArenaConfig(), seed=SEED)
    pol = PolicyB200.random_init(seed=0, max_ships=N)
    mems = {n: DeviceReplayMemory(bg, depth=DEPTH, n_step=n) for n in NS}
    maps = bg.raster("bits")
    for _ in range(DEPTH + 2):                           # rings full and wrapped
        iact, xy = pol.act(bg, maps, epsilon=0.5)
        for m in mems.values():
            m.push(iact, xy)
        bg.frame(maps=maps)
    words = bg.config.width * bg.config.height // 32
    out = {"arenas": N, "depth": DEPTH, "transitions": {str(n): len(m) for n, m in mems.items()},
           "rare_fraction_in_memory": {str(n): rare_fraction(lib, m, s)[0] for n, m in mems.items()}}
    g = torch.Generator().manual_seed(1)
    for B in (8, 256):
        row = {}
        o = _outputs(B, words)
        for n, m in mems.items():
            ids = m._ids[torch.randint(0, len(m), (B,), generator=g).cuda()].contiguous()
            if n == 1:
                row["gather"] = 1e3 * events_ms(lambda: _lib.check(lib.ofb_replay_gather(m._h, _p(ids), B, *[_p(t) for t in o[:8]], s)), 50)
            row["gather_nstep_n%d" % n] = 1e3 * events_ms(
                lambda: _lib.check(lib.ofb_replay_gather_nstep(m._h, _p(ids), B, GAMMA, *[_p(t) for t in o], s)), 50)
        row["maps_bytes_written"] = B * 2 * 2 * words * 4
        out["gather_us_B%d" % B] = row
    return out


def td_costs(lib, s, B=256):
    g = torch.Generator(device="cuda").manual_seed(0)
    a = [torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)]
    n = [torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)]
    ia = torch.randint(0, 2, (B,), dtype=torch.int32, device="cuda")
    pt = torch.randint(0, 400, (B, 2), dtype=torch.int32, device="cuda")
    r = torch.zeros(B, device="cuda")
    d = torch.zeros(B, dtype=torch.uint8, device="cuda")
    disc = torch.full((B,), GAMMA ** 3, device="cuda")
    ta, tp = torch.empty_like(a[0]), torch.empty_like(a[1])
    args = [_p(t) for t in (a[0], a[1], n[0], n[1], ia, pt, r, d)]
    res = {}
    for rep in range(2):                                  # the two forms alternated
        res.setdefault("td_targets_us", []).append(
            1e3 * events_ms(lambda: _lib.check(lib.ofb_trainer_td_targets(*args, GAMMA, B, _p(ta), _p(tp), s)), 50))
        res.setdefault("td_targets_discounted_us", []).append(
            1e3 * events_ms(lambda: _lib.check(lib.ofb_trainer_td_targets_discounted(*args, _p(disc), B, _p(ta), _p(tp), s)), 50))
    return res


def learn_loop(lib, s, frames, policy, prioritized, n_step, batch=8):
    """BatchedQLearner at configs[2] -> (ms per frame, replayed rare share, memory rare share, replays)."""
    bg = BatchedBattleground(N, ships=SHIPS, config=ArenaConfig(), seed=SEED)
    maps = bg.raster("bits")
    if prioritized:
        mem = PrioritizedReplayMemory(bg, depth=DEPTH, alpha=0.6, seed=1, n_step=n_step)
    else:
        mem = DeviceReplayMemory(bg, depth=DEPTH, n_step=n_step)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=batch, max_ships=max(16, batch))
    learner = BatchedQLearner(tr, mem, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    hits = torch.zeros(2, dtype=torch.float64, device="cuda")
    name = "sample_prioritized" if prioritized else "sample"
    orig = getattr(mem, name)

    def counted(*a, **k):
        g = orig(*a, **k)
        hits[0] += ((g.reward != 0) | (g.done != 0)).sum()
        hits[1] += g.reward.numel()
        return g

    setattr(mem, name, counted)
    replays = 0
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(st)
    for _ in range(frames):
        if bg.time >= MAX_TIME:
            bg.restart()
            bg.raster("bits", out=maps)
            learner.reset()
        replays += 1 if learner.act(bg, maps)[2] else 0
        bg.frame(maps=maps)
    e1.record(st)
    torch.cuda.synchronize()
    h = hits.tolist()
    in_mem, _ = rare_fraction(lib, mem, s)
    return e0.elapsed_time(e1) / frames, h[0] / max(h[1], 1.0), in_mem, replays


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nstep_bench.py measures the GPU path and needs a CUDA device")
    lib = _lib.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {"card": card(), "depth": DEPTH, "arenas": N, "gamma": GAMMA}
    out["gather"] = gather_costs(lib, s)
    torch.cuda.empty_cache()
    out["td_B256"] = td_costs(lib, s)
    policy = PolicyB200.random_init(seed=0, max_ships=N)
    learn_loop(lib, s, 5, policy, True, 3)                # warm-up of every kernel on this shape
    learn = {}
    for rep in range(2):
        for prio in (False, True):
            for n in (1, 3):
                ms, frac, in_mem, k = learn_loop(lib, s, args.frames, policy, prio, n)
                arm = learn.setdefault("%s_n%d" % ("prioritized" if prio else "uniform", n),
                                       {"frame_ms": [], "rare_fraction_replayed": [], "rare_fraction_in_memory": [], "replays": k})
                arm["frame_ms"].append(ms)
                arm["rare_fraction_replayed"].append(frac)
                arm["rare_fraction_in_memory"].append(in_mem)
                torch.cuda.empty_cache()
    out["learn_%d_frames_B8" % args.frames] = learn
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
