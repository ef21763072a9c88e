"""Cost of prioritized replay (replay.PrioritizedReplayMemory) against the uniform DeviceReplayMemory, on two layouts at depth 16:
  * P1:      65 536 arenas x 7 ships, ship 0 policy-driven (the bench's policy workload);
  * policy7: 16 384 arenas x 7 policy ships.
For each: push with and without priorities (each push timed alone after a 512 MB memset, so the arena state comes from HBM and
not the 126 MB L2, the two memories alternated), sample_prioritized at B = 8 / 256 with its algorithmic bytes (the valid +
mass pass over every candidate, plus one 2048-candidate tile per draw), update_priorities and td_errors at B = 256 -- CUDA
events around the C calls alone, outputs preallocated.
Then, on P1, BatchedQLearner per frame over 400 frames (the restart at frame 200 inside), uniform against prioritized at
trainer batch 8 and 256, two runs per arm with the arms alternated; beside each, the fraction of the replayed transitions
with reward != 0 or done = 1 (an indicator of where the fit budget goes, not a pass criterion).
The card's name and power limit are read in the same run.
Usage: python scripts/prio_bench.py [--frames 400] [--out FILE]  -> one JSON line (and FILE)."""
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

SEED, MAX_TIME, DEPTH = 0x0F16, 200, 16
LAYOUTS = {"P1": (65536, {"QlearnIA": 1, "random": 6}), "policy7": (16384, {"QlearnIA": 7})}


def _p(t):
    return C.c_void_p(t.data_ptr())


def push_us(mems, iact, xy, reps=60):
    """Median push time of each memory, each push alone after an L2-clearing memset, the memories alternated."""
    flush = torch.empty(512 * 2 ** 20, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream()
    samples = {k: [] for k in mems}
    for i in range(reps):
        for k, m in mems.items():
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            m.push(iact, xy)
            e1.record(st)
            samples[k].append((e0, e1))
    torch.cuda.synchronize()
    out = {}
    for k, s in samples.items():
        ts = sorted(a.elapsed_time(b) for a, b in s[10:])
        out[k] = {"median_us": 1e3 * ts[len(ts) // 2], "min_us": 1e3 * ts[0], "max_us": 1e3 * ts[-1]}
    return out


def layout_costs(name, lib, s):
    N, ships = LAYOUTS[name]
    bg = BatchedBattleground(N, ships=ships, config=ArenaConfig(), seed=SEED)
    P = sum(1 for b in bg.behaviors if b == "QlearnIA")
    pol = PolicyB200.random_init(seed=0, max_ships=N * P)
    uni, pri = DeviceReplayMemory(bg, depth=DEPTH), PrioritizedReplayMemory(bg, depth=DEPTH, alpha=0.6, seed=1)
    maps = bg.raster("bits")
    for _ in range(DEPTH + 2):                           # both rings full and wrapped
        iact, xy = pol.act(bg, maps, epsilon=0.5)
        uni.push(iact, xy)
        pri.push(iact, xy)
        bg.frame(maps=maps)
    out = {"arenas": N, "policy_ships": P, "depth": DEPTH, "uniform_ring_device_bytes": uni.device_bytes,
           "prioritized_ring_device_bytes": pri.device_bytes}
    iact, xy = pol.act(bg, maps, epsilon=0.5)
    out["push"] = push_us({"uniform": uni, "prioritized": pri}, iact, xy)
    n_cand = (DEPTH - 1) * N * P
    out["candidates"] = n_cand
    out["valid_transitions"] = len(pri)
    nv = torch.zeros(1, dtype=torch.int32, device="cuda")
    for B in (8, 256):
        ids = torch.empty(B, dtype=torch.int32, device="cuda")
        w = torch.empty(B, dtype=torch.float32, device="cuda")
        ms = events_ms(lambda: _lib.check(lib.ofb_replay_sample_prioritized(pri._h, B, 0.5, _p(ids), _p(w), _p(nv), s)), 50)
        nbytes = n_cand * (1 + 4) + B * 2048 * (1 + 4)
        out["sample_B%d" % B] = {"us": 1e3 * ms, "bytes": nbytes, "GBps": nbytes / (ms * 1e-3) / 1e9}
    B = 256
    td_a = torch.randn(B, device="cuda")
    td_p = torch.randn(B, device="cuda")
    out["update_priorities_us_B256"] = 1e3 * events_ms(
        lambda: _lib.check(lib.ofb_replay_update_priorities(pri._h, _p(ids), _p(td_a), _p(td_p), B, s)), 50)
    return out


def td_errors_us(lib, s, B=256):
    g = torch.Generator(device="cuda").manual_seed(0)
    a = [torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)]
    n = [torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)]
    ia = torch.randint(0, 2, (B,), dtype=torch.int32, device="cuda")
    pt = torch.randint(0, 400, (B, 2), dtype=torch.int32, device="cuda")
    r = torch.zeros(B, device="cuda")
    d = torch.zeros(B, dtype=torch.uint8, device="cuda")
    oa, op = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
    args = [_p(t) for t in (a[0], a[1], n[0], n[1], ia, pt, r, d)]
    return 1e3 * events_ms(lambda: _lib.check(lib.ofb_trainer_td_errors(*args, 0.9, B, _p(oa), _p(op), s)), 50)


def learn_loop(frames, policy, prioritized, batch):
    """BatchedQLearner on P1 -> (ms per frame, fraction of replayed transitions with reward != 0 or done = 1, replays)."""
    N, ships = LAYOUTS["P1"]
    bg = BatchedBattleground(N, ships=ships, config=ArenaConfig(), seed=SEED)
    maps = bg.raster("bits")
    mem = PrioritizedReplayMemory(bg, depth=DEPTH, alpha=0.6, seed=1) if prioritized else DeviceReplayMemory(bg, depth=DEPTH)
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=batch, max_ships=max(16, batch))
    learner = BatchedQLearner(tr, mem, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    hits = torch.zeros(2, dtype=torch.float64, device="cuda")    # (rare transitions, transitions) replayed, summed on the device
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
    return e0.elapsed_time(e1) / frames, h[0] / max(h[1], 1.0), replays


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prio_bench.py measures the GPU path and needs a CUDA device")
    lib = _lib.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {"card": card(), "depth": DEPTH}
    for name in LAYOUTS:
        out[name] = layout_costs(name, lib, s)
        torch.cuda.empty_cache()
    out["td_errors_us_B256"] = td_errors_us(lib, s)
    policy = PolicyB200.random_init(seed=0, max_ships=LAYOUTS["P1"][0])
    learn_loop(5, policy, True, 8)                        # warm-up of every kernel on this shape
    learn = {}
    for rep in range(2):
        for batch in (8, 256):
            for prio in (False, True):
                ms, frac, n = learn_loop(args.frames, policy, prio, batch)
                arm = learn.setdefault("%s_B%d" % ("prioritized" if prio else "uniform", batch),
                                       {"frame_ms": [], "rare_fraction": [], "replays": n})
                arm["frame_ms"].append(ms)
                arm["rare_fraction"].append(frac)
                torch.cuda.empty_cache()
    out["learn_%d_frames" % args.frames] = learn
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
