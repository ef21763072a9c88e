"""Cost of the data-parallel learner (TrainerB200(reducer=sharding.DistReducer()), BatchedQLearner on every rank).

    python -m torch.distributed.run --nproc-per-node W scripts/dp_bench.py [--frames 400] [--out FILE]

Measured on every rank, reported by rank 0 (the min / median / max over ranks of each rank's median where it says so):
  (a) one sharded fit at global batch G = 64 / 256 / 1024, split evenly (G / W per rank): CUDA events around
      TrainerB200.fit (the all-reduce of the batch size, the 96 kernels, the 16 reduce stages), each fit alone after a
      512 MB memset that evicts L2; beside it the 17 collectives of a fit alone (the int32 batch size, 7 x 16 + 2 + 7 x 16
      fp64 statistics, 571 730 fp32 gradients) on the same stream.  The two arms alternate.
  (b) BatchedQLearner per frame at 131 072 arenas per GPU (7 ships, ship 0 policy-driven), depth 16, a replay every 50
      frames, trainer batch 8 per rank, uniform and prioritized memories, over --frames frames with a restart every 200;
      and, for comparison, today's learner: rank 0's QLearner on the policy ships of its first 8 arenas, every rank's actor
      refreshed by a weight broadcast every 50 frames.  Beside each, the share of replayed transitions with reward != 0
      or done = 1.  Two runs per arm, the arms alternated.
The card's name and power limit are read in the same run."""
import argparse
import datetime
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from learn_bench import card  # noqa: E402
from ofighters_b200 import ArenaConfig, BatchedBattleground, _lib, sharding  # noqa: E402
from ofighters_b200.policy import PolicyB200  # noqa: E402
from ofighters_b200.replay import DeviceReplayMemory, PrioritizedReplayMemory  # noqa: E402
from ofighters_b200.trainer import (BatchedQLearner, Epsilon_cos, QLearner, TrainerB200, flatten_weights,  # noqa: E402
                                    unflatten_weights)

SEED, MAX_TIME, DEPTH, N = 0x0F16, 200, 16, 131072


def _stats(ts):
    ts = sorted(ts)
    return {"median": ts[len(ts) // 2], "min": ts[0], "max": ts[-1]}


def fit_costs(dev, rank, world, reps=12):
    """(a): per global batch, the sharded fit and its collectives alone, in ms (this rank's median / min / max)."""
    red = sharding.DistReducer()
    flush = torch.empty(512 * 2 ** 20, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev)
    out = {}
    for G in (64, 256, 1024):
        b = G // world
        bg = BatchedBattleground(b, ships={"random": 7}, seed=SEED, device=dev, arena0=rank * b)
        for _ in range(20):
            bg.frame()
        maps = bg.raster("bits")
        vec = bg.obs_vec[:, 0, :].contiguous()
        g = torch.Generator(device=dev).manual_seed(rank)
        ta = torch.randn((b, 2), device=dev, generator=g)
        tp = torch.randn((b, 400, 400), device=dev, generator=g) * 0.5
        tr = TrainerB200(learning_rate=1e-4, batch_size=b, device=dev, max_ships=8, reducer=red)
        slices = [torch.zeros(16, dtype=torch.float64, device=dev) for _ in range(14)] + \
            [torch.zeros(2, dtype=torch.float64, device=dev), torch.zeros(571730, dtype=torch.float32, device=dev)]
        nb = torch.zeros(1, dtype=torch.int32, device=dev)

        def collectives():
            red.all_reduce(nb)
            for s in slices:
                red.all_reduce(s)
        for _ in range(3):                               # warm-up of both arms
            tr.fit(maps, vec, ta, tp, sync_model=False)
            collectives()
        fit_ms, coll_ms = [], []
        for _ in range(reps):
            for arm, fn, acc in (("fit", lambda: tr.fit(maps, vec, ta, tp, sync_model=False), fit_ms),
                                 ("coll", collectives, coll_ms)):
                flush.zero_()
                dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                fn()
                e1.record(st)
                torch.cuda.synchronize(dev)
                acc.append(e0.elapsed_time(e1))
        out["G%d" % G] = {"per_rank_batch": b, "fit_ms": _stats(fit_ms), "collectives_ms": _stats(coll_ms)}
        del tr, bg
        torch.cuda.empty_cache()
    return out


def learn_loop(dev, rank, world, frames, mode, policy):
    """(b): ms per frame on this rank and (rare transitions, transitions) replayed on this rank."""
    bg = BatchedBattleground(N, ships={"QlearnIA": 1, "random": 6}, config=ArenaConfig(), seed=SEED, device=dev,
                             arena0=rank * N)
    maps = bg.raster("bits")
    hits = torch.zeros(2, dtype=torch.float64, device=dev)
    schedule = Epsilon_cos(period=110 * 400)

    def count(g):
        hits[0] += ((g.reward != 0) | (g.done != 0)).sum()
        hits[1] += g.reward.numel()

    learner = trainer = None
    if mode in ("dp_uniform", "dp_prioritized"):
        trainer = TrainerB200(learning_rate=1e-4, epsilon=schedule, batch_size=8, device=dev, max_ships=16, seed=0,
                              reducer=sharding.DistReducer())
        mem = PrioritizedReplayMemory(bg, depth=DEPTH, alpha=0.6, seed=1 + rank) if mode == "dp_prioritized" else \
            DeviceReplayMemory(bg, depth=DEPTH)
        name = "sample_prioritized" if mode == "dp_prioritized" else "sample"
        orig = getattr(mem, name)

        def counted(*a, **k):
            g = orig(*a, **k)
            count(g)
            return g
        setattr(mem, name, counted)
        learner = BatchedQLearner(trainer, mem, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    elif rank == 0:                                        # today's learner: rank 0's QLearner on its first 8 arenas
        trainer = TrainerB200(learning_rate=1e-4, epsilon=schedule, batch_size=8, device=dev, max_ships=16, seed=0)
        learner = QLearner(trainer, track=8, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    n_len = 571730
    st = torch.cuda.current_stream(dev)
    torch.cuda.synchronize(dev)
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for t in range(frames):
        if bg.time >= MAX_TIME:
            bg.restart()
            bg.raster("bits", out=maps)
            if learner is not None:
                learner.reset()
        if mode.startswith("dp_"):
            _, _, replayed = learner.act(bg, maps)
            if replayed:                                   # the actor follows the rank's own replica
                policy.load_weights(trainer.get_weights())
        else:
            if learner is not None:
                learner.act(bg, maps)
            else:
                policy.act(bg, maps, epsilon=schedule, collecting=t + 1 < 20)
                if t + 1 >= 20:
                    schedule.next()
            if (t + 1) % 50 == 0:                          # every rank's actor <- rank 0's weights
                flat = flatten_weights(trainer.get_weights()).to(dev) if rank == 0 else \
                    torch.empty(n_len, dtype=torch.float32, device=dev)
                sharding.broadcast_weights(flat, src=0)
                policy.load_weights(unflatten_weights(flat.cpu()))
        bg.frame(maps=maps)
    e1.record(st)
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / frames, hits.tolist()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dp_bench.py measures the GPU path and needs a CUDA device")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=600), device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    try:
        _lib.load()
        out = {"world": world, "card": card(), "arenas_per_gpu": N, "depth": DEPTH, "replay_every": 50,
               "trainer_batch_per_rank": 8}
        out["fit"] = fit_costs(dev, rank, world)
        torch.cuda.empty_cache()
        policy = PolicyB200.random_init(device=dev, seed=0, max_ships=N)
        learn_loop(dev, rank, world, 5, "dp_prioritized", policy)      # warm-up of every kernel on this shape
        learn = {}
        for rep in range(2):
            for mode in ("rank0_qlearner", "dp_uniform", "dp_prioritized"):
                ms, hits = learn_loop(dev, rank, world, args.frames, mode, policy)
                t = torch.tensor([ms, ms, hits[0], hits[1]], dtype=torch.float64, device=dev)
                lo, hi = t[:1].clone(), t[1:2].clone()
                dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                dist.all_reduce(hi, op=dist.ReduceOp.MAX)
                h = t[2:].clone()
                dist.all_reduce(h)
                arm = learn.setdefault(mode, {"frame_ms_min_over_ranks": [], "frame_ms_max_over_ranks": [],
                                              "rare_fraction": []})
                arm["frame_ms_min_over_ranks"].append(float(lo))
                arm["frame_ms_max_over_ranks"].append(float(hi))
                hh = h.tolist()
                arm["rare_fraction"].append(hh[0] / max(hh[1], 1.0) if hh[1] else None)
                torch.cuda.empty_cache()
        out["learn_%d_frames" % args.frames] = learn
        out["card_after"] = card()
        if rank == 0:
            line = json.dumps(out)
            print(line)
            if args.out:
                with open(args.out, "w") as f:
                    f.write(line + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
