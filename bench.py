"""bench.py -- env-steps/s of the Ofighters hot path on B200 (contract: see README / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one lockstep frame of every arena in the batch: scripted-bot actions -> fused arena
step (K1) -> observation raster (K2) [-> policy forward for the policy workloads], with the
MAX_TIME=200 episode restart when due.  One process per GPU; arenas are sharded with no data-path
collective (weak scaling: the per-GPU batch is fixed), NCCL only all-reduces the per-episode stats.

Workloads (BASELINE.json configs):
    policy       configs[2]: 65536 arenas, ship 0 policy-driven (conv+dense bi-head forward, bf16)   [default at --gpus 1]
    sharded1m    configs[4]: 131072 arenas per GPU, policy forward, learning, per-episode score/loss all-reduce
                 and weight broadcast                                                                 [default at --gpus N > 1]
    arena4096    configs[1]: 4096 default arenas (7 ships), random bots, step + raster
    stress       configs[3]: 16384 arenas x 32 ships, max fire rate, step + raster
    policy7      configs[2] variant: 16384 arenas, all 7 ships policy-driven (trunk once per arena, heads x7)

The metric BASELINE.json names is "env-steps/sec (batched arenas + policy fwd)", so the default workload is the one
with the forward.  The un-timed pre-roll places the MAX_TIME=200 episode restart -- `restart()`, the per-episode
all-reduces and (when learning) a replay + weight broadcast -- INSIDE the K timed steps.

Timing: CUDA events on the launching stream around every step, L2 flushed (256 MiB memset)
between steps when the working set is smaller than L2, barrier + synchronize on both sides of the
timed region, max over ranks.  `--impl reference` times the CPU restatement of the reference
(oracle/step_c.c, OpenMP over all host cores) on the same workload; the reference itself is pure
Python and is not part of this repository.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step computed (observation heads, arena state,
the policy ships' played actions, bit maps) as DIR/<name>.npy in float32 / float64, for a fixed seeded sample of arenas
(rank 0's when several GPUs run), so that two builds can be compared output for output on identical inputs.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 0x0F16

WORKLOADS = {
    # name: (arenas per GPU, ships, bot kind, laser_cap, policy ships, description)
    "arena4096": dict(n=4096, ships=7, bot="random", lcap=0, policy=0,
                      desc="configs[1]: 4096 default arenas (400x400, 7 ships), random-action bots, "
                           "step + observation raster (bit-packed maps)"),
    "stress": dict(n=16384, ships=32, bot="stress", lcap=32 * 64, policy=0,
                   desc="configs[3]: 16384 arenas x 32 ships, every ship shoots every frame, step + raster"),
    "policy": dict(n=65536, ships=7, bot="random", lcap=0, policy=1,
                   desc="configs[2]: 65536 default arenas, ship 0 driven by the bi-head policy forward (bf16), "
                        "ships 1-6 random bots"),
    "policy7": dict(n=16384, ships=7, bot="random", lcap=512, policy=7,      # (seven ships that all shoot: more lasers in flight than the default 128 slots)
                    desc="configs[2] variant of SURVEY 8(d): 16384 default arenas, ALL 7 ships policy-driven "
                         "(trunk once per arena, heads x7 -> 114688 forwards per frame), bf16"),
    "sharded1m": dict(n=131072, ships=7, bot="random", lcap=0, policy=1,
                      desc="configs[4]: 131072 arenas per GPU (1M over 8), policy forward, per-episode stats all-reduce"),
}


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        if os.environ.get("OFB_BENCH_NO_SAMPLER"):        # diagnostic: is the NVML polling visible in the step times?
            return
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ----------------------------------------------------------------------------- L2 flush
class L2Flush:
    """Evicts the working set from the 126 MB L2 between timed iterations: a 256 MiB memset (the write the
    timing rules ask for) followed by a 256 MiB read of a second buffer.  The read pass matters: L2 is
    write-back, so a bare memset leaves ~100 MB of DIRTY lines behind and their write-back would be charged
    to the next timed kernel (measured: see profiles/r01_flush_study.md)."""

    def __init__(self, dev, mode="write+read"):
        import torch
        self.mode = mode
        self.w = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
        self.r = torch.zeros(64 * 2 ** 20, dtype=torch.float32, device=dev) if mode == "write+read" else None
        self.acc = torch.empty((), dtype=torch.float32, device=dev)
        self.torch = torch

    def __call__(self):
        self.w.zero_()
        if self.r is not None:
            self.torch.sum(self.r, dim=0, out=self.acc)

    def describe(self):
        return "flushed between steps (256 MiB memset%s, outside the per-step events)" % (
            " + 256 MiB read so no dirty lines remain" if self.r is not None else "")


# ----------------------------------------------------------------------------- CPU arm
def cpu_arm(wl, steps, warmup, n_cap=4096):
    """The reference's algorithm on the host cores: oracle/step_c.c (bots + step + raster, OpenMP).
    Returns (env_steps_per_s, ms_per_step, cores, sample description)."""
    import ctypes
    import numpy as np
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ["OMP_NUM_THREADS"] = str(cores)          # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses every core
    from oracle.step_c import ArenasC
    try:
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)   # in case the OpenMP runtime was initialised already
    except OSError:
        pass
    N = min(wl["n"], n_cap)
    S = wl["ships"]
    c0 = ArenasC(np.zeros((N, S, 2), np.int32))
    spawn = c0.random_spawn(SEED, 0)
    c = ArenasC(spawn, lcap=wl["lcap"] or None)
    out_t = 0.0
    t_ep, ep = 0, 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        if t_ep >= 200:
            ep += 1
            c.reset(c.random_spawn(SEED, ep))
            t_ep = 0
        c.step(c.bot_actions(wl["bot"], SEED, it))
        c.raster_bits()
        t_ep += 1
        if it >= warmup:
            out_t += time.perf_counter() - t0
    return N * steps / out_t, out_t / steps * 1e3, cores, \
        "%d arenas x %d frames of bots+step+raster, oracle/step_c.c (gcc -O2 -fopenmp, %d threads)" % (N, steps, cores)


def cpu_policy_rate(cores, batch=8, reps=3):
    """The policy forward on the host cores: the torch-fp32 restatement of the Keras model (oracle/policy_torch.py, the same
    arithmetic as model.predict) on a bounded sample of `batch` forwards per call.  -> ship-forwards per second."""
    import numpy as np  # noqa: F401
    import torch
    from oracle import policy_torch as po
    torch.set_num_threads(cores)
    w = po.init_weights(0)
    g = torch.Generator().manual_seed(0)
    img = (torch.rand((batch, 400, 400, 2), generator=g) < 0.01).float()
    vec = torch.rand((batch, 8), generator=g) * 400
    with torch.no_grad():
        po.forward(w, img, vec)
        t0 = time.perf_counter()
        for _ in range(reps):
            act, ptr = po.forward(w, img, vec)
            po.decode(act, ptr)
    return batch * reps / (time.perf_counter() - t0)


def cpu_arm_with_policy(wl, steps, warmup):
    """cpu_arm for the policy workloads: the arena rate and the forward rate are measured separately on bounded samples and
    combined per frame (1 frame = 1 arena step + `policy` ship-forwards per arena), since one full-size CPU frame of 65 536
    forwards would take minutes."""
    v, ms, cores, sample = cpu_arm(wl, steps, warmup)
    if not wl["policy"]:
        return v, ms, cores, sample, None
    fwd = cpu_policy_rate(cores)
    combined = 1.0 / (1.0 / v + wl["policy"] / fwd)
    sample += "; policy forward: oracle/policy_torch.py (torch fp32, %d threads) on batches of 8 = %.1f ship-forwards/s; " \
              "combined per frame as 1 / (1 / arena rate + %d / forward rate)" % (cores, fwd, wl["policy"])
    return combined, 1e3 * min(wl["n"], 4096) / combined, cores, sample, fwd


def python_port_rate(ships, frames=100):
    """The pure-Python restatement (same language and structure as the reference) on one core."""
    import numpy as np
    from oracle.step_py import ArenaPy
    from oracle.traces import make_tapes
    spawn, actions = make_tapes(1, 1, frames, ships, "random")
    a = ArenaPy(spawn[0])
    t0 = time.perf_counter()
    for t in range(frames):
        a.step(actions[0, t])
        a.maps()
    return frames / (time.perf_counter() - t0)


# ----------------------------------------------------------------------------- shared by both arms
METRIC = "env-steps/sec (batched arenas: bots + fused step + observation raster%s)"


def resolve_workload(args):
    """No --workload: the metric's own config -- configs[2] on one GPU, configs[4] (1M arenas over 8 GPUs: 131072 each,
    learning + per-episode all-reduce) on several."""
    name = args.workload
    if name == "auto":
        name = "policy" if args.gpus <= 1 else "sharded1m"
    return name, WORKLOADS[name]


def workload_config(name, wl, world, learn):
    """The `config` object: identical in the `ours` and the `reference` arm (only static facts of the workload)."""
    return {"workload": name, "desc": wl["desc"], "arenas_per_gpu": wl["n"], "arenas_total": wl["n"] * world,
            "ships_per_arena": wl["ships"], "policy_ships_per_arena": wl["policy"], "bots": wl["bot"],
            "map_format": "bits u32[N,2,5000]", "max_time": 200, "learning": bool(learn),
            "episode": "the un-timed pre-roll ends half of the timed steps before frame 200, so the MAX_TIME restart (restart + "
                       "per-episode all-reduces%s) runs inside the timed region" %
                       (" + replay / weight broadcast" if learn else "")}


def wants_learning(args, name, wl):
    return bool(wl["policy"]) and (args.learn == "on" or (args.learn == "auto" and name == "sharded1m"))


# --dump-outputs: 512 sampled arenas, the bit maps of the first 128 of them.  At the largest laser list of any workload
# (stress: 2048 slots x 32 ships) that is 54 MB, under the 64 MB the dump may take.
DUMP_ARENAS, DUMP_MAP_ARENAS, DUMP_MAX_BYTES = 512, 128, 64 * 2 ** 20


def dump_outputs(out_dir, bg, maps, played):
    """Writes the outputs of the last step as out_dir/<name>.npy: `arena_ids` (global ids of a sample of DUMP_ARENAS arenas
    drawn with SEED), for those arenas the observation heads `obs_vec`, every field of `bg.state()` (laser slots past an
    arena's live count are zeroed, the laser columns cut at the sample's largest live count), the batch's action buffer
    `actions` (the rows the policy wrote; scripted bots draw their actions inside the frame kernel and leave their rows
    zero), the policy ships' played `policy_iaction` / `policy_xy` (policy workloads), the bit maps `maps` (u32 words, first
    DUMP_MAP_ARENAS sampled arenas); and the batch's episode statistics `stats`.  Integers become float64 (float32 when
    16 bits or fewer), so every value is exact."""
    import numpy as np
    import torch
    N = bg.n_arenas
    ids = np.sort(np.random.Generator(np.random.PCG64(SEED)).choice(N, size=min(N, DUMP_ARENAS), replace=False))
    sel = torch.from_numpy(ids).to(bg.device)
    pick = lambda t: t.index_select(0, sel).cpu().numpy()
    st = {k: pick(v) for k, v in bg.state().items()}
    width = max(1, int(st["n_lasers"].max()))
    live = np.arange(width)[None, :] < st["n_lasers"][:, None]
    for k in st:
        if k.startswith("laser_"):
            st[k] = np.where(live, st[k][:, :width], 0).astype(st[k].dtype)
    out = {"arena_ids": ids + bg.arena0, "obs_vec": pick(bg.obs_vec), **st, "actions": pick(bg.actions),
           "maps": maps.index_select(0, sel[:DUMP_MAP_ARENAS]).cpu().numpy().view(np.uint32), "stats": bg.stats.cpu().numpy()}
    if played is not None:
        iact, xy = played
        out["policy_iaction"] = pick(iact.reshape(N, -1))
        out["policy_xy"] = pick(xy.reshape(N, -1, 2))
    for k, v in out.items():
        out[k] = v.astype(np.float32 if v.dtype == np.float32 or (v.dtype.kind in "iub" and v.dtype.itemsize <= 2) else np.float64)
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# ----------------------------------------------------------------------------- GPU arm
def gpu_arm(args, name, wl):
    import torch
    import torch.distributed as dist
    from ofighters_b200 import ArenaConfig, BatchedBattleground
    from ofighters_b200 import _lib, sharding  # noqa: F401

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N, S = wl["n"], wl["ships"]
    steps, warmup = args.steps, max(args.warmup, 3)
    max_time = 200

    ships = {wl["bot"]: S} if not wl["policy"] else {"QlearnIA": wl["policy"], wl["bot"]: S - wl["policy"]}
    ships = {k: v for k, v in ships.items() if v > 0}
    bg = BatchedBattleground(N, ships=ships, config=ArenaConfig(laser_cap=wl["lcap"]), device=dev, seed=SEED,
                             arena0=rank * N)
    policy = None
    learner = trainer = None
    learn = wants_learning(args, name, wl)
    loss_stats = torch.zeros(2, dtype=torch.float64, device=dev)
    # ships per launch of the forward's kernels: the whole batch by default (measured at 65 536 arenas: 21.2 ms per forward as one
    # chunk, 22.8 ms in chunks of 8 192 -- fewer partial waves; the workspace is 0.18 MB per ship)
    max_ships = int(os.environ.get("OFB_BENCH_MAX_SHIPS", str(min(N * max(wl["policy"], 1), 131072))))
    if wl["policy"]:
        from ofighters_b200.policy import PolicyB200
        policy = PolicyB200.random_init(device=dev, seed=0, max_ships=max_ships)       # the actor of every rank
    if learn:
        # ONE shared trainer (agents/qlearnIA_V2.py:308): rank 0 learns from the policy ships of its first 8 arenas
        # (QlearnIA.play's bookkeeping: collecting phase, eps-greedy with the trainer's schedule, replay at deaths and every
        # 50 steps); every rank's actor takes the trainer's weights at common points (every 50 frames and at the episode
        # end), the episode's [sum loss, replays] rides the K7 all-reduce
        from ofighters_b200.trainer import Epsilon_cos, QLearner, TrainerB200, flatten_weights, unflatten_weights
        schedule = Epsilon_cos(period=110 * 400)
        if rank == 0:
            trainer = TrainerB200(learning_rate=1e-4, epsilon=schedule, batch_size=8, device=dev, seed=0, max_ships=16)
            learner = QLearner(trainer, track=8, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    trainer_len = 571730
    maps = torch.empty((N, 2, 400 * 400 // 32), dtype=torch.int32, device=dev)
    bg.raster("bits", out=maps)
    state_bytes = N * bg.state_stride
    flush_needed = state_bytes + maps.numel() * 4 < 2 * 126 * 2 ** 20
    flush_buf = L2Flush(dev, args.flush) if flush_needed else None
    launches = [0]
    coll = {"all_reduce": 0, "broadcast": 0, "restarts": 0, "replays": 0}
    frame_no = [0]                                        # frames since construction (identical on every rank)
    weights_dirty = [False]
    played = [None]                                       # (iaction, xy) the policy ships played in the last step

    def n_launched():
        return bg.launch_count + (policy.launch_count if policy is not None else 0) + \
            (trainer.launch_count + trainer.model.launch_count if trainer is not None else 0)

    def sync_actor_weights():
        """Every rank's actor <- the shared trainer's weights (a broadcast over NCCL when there are several ranks)."""
        if world > 1:
            # the shared trainer's weights + the step of its epsilon schedule (exact in fp32: t < 44000)
            flat = torch.cat([flatten_weights(trainer.get_weights()), torch.tensor([trainer.epsilon.t])]).to(dev) if rank == 0 else \
                torch.empty(trainer_len + 1, dtype=torch.float32, device=dev)
            sharding.broadcast_weights(flat, src=0)
            coll["broadcast"] += 1
            host = flat.cpu()
            policy.load_weights(unflatten_weights(host[:trainer_len]))
            if rank != 0:
                schedule.t = float(host[-1])
        elif weights_dirty[0]:
            policy.load_weights(trainer.get_weights())
        weights_dirty[0] = False

    def one_step():
        n0 = n_launched()
        if bg.time >= max_time:
            bg.restart()
            coll["restarts"] += 1
            if learner is not None:
                loss_stats[0] += sum(learner.losses)
                loss_stats[1] += len(learner.losses)
                learner.losses.clear()
                learner.reset()
            if world > 1:
                sharding.reduce_episode_stats(bg.stats)   # K7: per-episode [score, kills, deaths, shots, ships, arenas]
                coll["all_reduce"] += 1
                if learn:
                    sharding.reduce_loss_stats(loss_stats)     # ... and [sum of replay losses, replays]
                    coll["all_reduce"] += 1
            if learn:
                sync_actor_weights()
            if policy is not None:
                bg.raster("bits", out=maps)        # Battleground.restart builds a fresh Observation
        if policy is not None:
            if learn:
                sched = learner.trainer.epsilon if learner is not None else schedule
                collecting = frame_no[0] + 1 < 20
                if learner is not None:
                    iact, xy, replayed = learner.act(bg, maps)     # choose (collecting / eps-greedy), write rows, remember / replay
                    played[0] = (iact, xy)
                    coll["replays"] += 1 if replayed else 0
                    weights_dirty[0] |= replayed
                else:                                          # the other ranks follow the shared schedule between broadcasts
                    played[0] = policy.act(bg, maps, epsilon=sched, collecting=collecting)
                    if not collecting:
                        sched.next()
                if (frame_no[0] + 1) % 50 == 0:
                    sync_actor_weights()
            else:
                played[0] = policy.act(bg, maps)   # forward on the current maps -> the policy ship's ("external") action row
        bg.frame(maps=maps)                        # scripted bots + step + observation maps: one fused launch (ofb_frame_bots)
        frame_no[0] += 1
        launches[0] += n_launched() - n0

    stream = torch.cuda.current_stream(dev)
    # un-timed pre-roll: the episode is advanced so that frame 200 (the restart) falls in the middle of the timed steps
    preroll = max(0, max_time - steps // 2 - warmup) if steps < 2 * max_time else 0
    for _ in range(preroll + warmup):
        one_step()
    torch.cuda.synchronize(dev)
    time_at_start = bg.time

    # ---- timed region: exactly K steps, per-step CUDA events, optional L2 flush between steps
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sampler = ClockSampler(physical_gpu_index(local_rank))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    sampler.start()
    launches[0] = 0
    for k in coll:
        coll[k] = 0
    wall0 = time.perf_counter()
    for k in range(steps):
        if flush_buf is not None:
            flush_buf()
        ev[k][0].record(stream)
        one_step()
        ev[k][1].record(stream)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    coll_timed = dict(coll)
    time_at_end = bg.time
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    per_rank_ms = [total_ms / steps]
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_ms = [float(x.item()) / steps for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    st = bg.state(("overflow", "near_ties", "n_lasers"))
    counters = torch.stack([st["overflow"].sum(), st["near_ties"].sum(), st["n_lasers"].sum()]).to(torch.int64)
    if world > 1:
        dist.all_reduce(counters, op=dist.ReduceOp.SUM)
    overflow, near_ties, live_lasers = [int(x) for x in counters.tolist()]
    bg.check_overflow()
    value = N * world * steps / (total_ms * 1e-3)
    episode_stats = sharding.stats_dict(bg.stats)
    if args.dump_outputs and rank == 0:                   # before the measurements below restart and step the batch
        dump_outputs(args.dump_outputs, bg, maps, played[0])

    # ---- dominant kernel alone, same events + flush
    roof = kernel_roofline(bg, maps, flush_buf, wl, dev, policy)

    # ---- end-to-end through the public API with HOST buffers
    def make_bg():
        return BatchedBattleground(N, ships=ships, config=ArenaConfig(laser_cap=wl["lcap"]), device=dev, seed=SEED,
                                   arena0=rank * N)

    e2e = e2e_arm(bg, maps, wl, dev, min(steps, 400 if policy is None else 20), world, policy, make_bg)

    extra = {"ship_steps_per_s": value * S,
             "l2": (flush_buf.describe() if flush_needed else "working set %.0f MB > L2" % ((state_bytes + maps.numel() * 4) / 1e6)),
             "wall_s_timed_region": wall, "ms_per_step_by_rank": per_rank_ms,
             "frames_timed": "episode frames %d..%d, restart, frames 0..%d" % (time_at_start, max_time - 1, time_at_end - 1)
                             if coll_timed["restarts"] else "episode frames %d..%d" % (time_at_start, time_at_end - 1),
             "ms_per_step_min_median_max": [min(step_ms), sorted(step_ms)[len(step_ms) // 2], max(step_ms)],
             "preroll_frames": preroll, "live_lasers_at_end": live_lasers, "episode_stats_reduced": episode_stats}
    if learn:
        extra["learning"] = {
            "replays_in_timed_region_rank0": coll_timed["replays"], "replays_reduced": float(loss_stats[1].item()),
            "mean_replay_loss": ((float(loss_stats[0].item()) + (sum(learner.losses) if learner is not None else 0.0))
                                 / max(1.0, float(loss_stats[1].item()) + (len(learner.losses) if learner is not None else 0))),
            "trainer_steps": trainer.steps if trainer is not None else None,
            "epsilon": learner.trainer.epsilon.get() if learner is not None else None,
            "what": "rank 0 runs QlearnIA.play's bookkeeping for the policy ships of its first 8 arenas (20 random collecting steps, "
                    "eps-greedy with Epsilon_cos(110*400) evaluated on the device, Trainer.replay = batch 8, Adam 1e-4, at "
                    "every tracked death and every 50 steps of bot 1); every rank's actor takes the trainer's weights every 50 "
                    "frames and at the episode end (NCCL broadcast of 571730 floats); [sum loss, replays] all-reduced with the "
                    "episode statistics"}
    if wl["policy"] and rank == 0 and world == 1 and not os.environ.get("OFB_BENCH_NO_EXTRA"):
        extra["other_workloads"] = side_workloads(dev)
    out = {
        "metric": METRIC % (" + policy fwd" if wl["policy"] else ""),
        "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 laser physics / i32 ship state / u32 bit maps" + (" / bf16 policy" if wl["policy"] else ""),
        "data": "synthetic (Philox-seeded spawns and bot actions)",
        "config": workload_config(name, wl, world, learn),
        "gpu_launches": launches[0], "collectives_in_timed_region": coll_timed["all_reduce"] + coll_timed["broadcast"],
        "collectives": coll_timed, "near_ties": near_ties, "overflow": overflow,
        "clocks": clocks, "e2e": e2e, "roofline": roof, "extra": extra,
    }
    if rank == 0:
        if world == 1:
            v, ms, cores, sample, fwd = cpu_arm_with_policy(wl, 100, 5)
            try:
                py = python_port_rate(S)
            except Exception:
                py = None
            out["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                   "sample": sample, "python_port_env_steps_per_s_1core": py}
            if fwd is not None:
                out["cpu_baseline"]["policy_ship_forwards_per_s"] = fwd
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def side_workloads(dev):
    """configs[1] and configs[3] (the forward-less arena workloads) in short form, for the `extra` of the default line:
    event-timed fused frame kernel with the L2 flushed between launches."""
    import torch
    from ofighters_b200 import ArenaConfig, BatchedBattleground
    res = {}
    for wname in ("arena4096", "stress"):
        w = WORKLOADS[wname]
        b = BatchedBattleground(w["n"], ships={w["bot"]: w["ships"]}, config=ArenaConfig(laser_cap=w["lcap"]), device=dev, seed=SEED)
        m = torch.empty((w["n"], 2, 5000), dtype=torch.int32, device=dev)
        fl = L2Flush(dev)
        st = torch.cuda.current_stream(dev)
        for _ in range(12 if wname == "stress" else 30):
            b.frame(maps=m)
        ts = []
        for _ in range(20 if wname == "arena4096" else 8):
            fl()
            a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            b.frame(maps=m)
            c.record(st)
            ts.append((a, c))
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(c) for a, c in ts) / len(ts)
        res[wname] = {"env_steps_per_s": w["n"] / (ms * 1e-3), "ms_per_step": ms, "arenas": w["n"], "ships": w["ships"],
                      "frames": "%d..%d of an episode" % (b.time - len(ts), b.time - 1)}
        del b, m, fl
    return res


def _ncu_traffic():
    """DRAM bytes per launch / per item of the dominant kernels, from the committed `ncu --set full` captures (profiles/)."""
    out = {}
    for fn in ("r01_traffic.json", "r02_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", fn)) as f:
                out.update(json.load(f))
        except Exception:
            pass
    return out


# Forward layers: kernel, what bounds it, algorithmic bytes and FLOPs per item (DESIGN.md section 4; Appendix B MACs x 2).
# "per": the trunk runs once per ARENA, the heads once per policy SHIP.
POLICY_LAYERS = {
    "trunk12": dict(kernel_sparse="k_st_trunk12 (conv1 + conv2)", kernel_dense="k_tz_trunk12", per="arena", bytes=40000 + 160000,
                    flops=2 * (23.04e6 + 23.04e6)),
    # the default: conv1 .. conv4 + pools in one sparse tensor-core kernel, bit maps in, flat (25 x 25 x 8 bf16) out
    "trunk": dict(kernel="k_st_trunk12 (fused conv1..conv4)", per="arena", bytes=40000 + 10240, flops=2 * (23.04e6 + 23.04e6 + 5.76e6 + 1.44e6)),
    "conv3": dict(kernel="k_tc_conv_pool", per="arena", bytes=160000 + 40000, flops=2 * 5.76e6),
    "conv4": dict(kernel="k_tc_conv_pool", per="arena", bytes=40000 + 10240, flops=2 * 1.44e6),
    "dense1": dict(kernel="k_tc_dense1", per="arena", bytes=10240 + 400, flops=2 * 0.5e6),
    "heads": dict(kernel="k_heads", per="ship", bytes=400 + 32 + 80000, flops=2 * (5.1e3 + 62.5e3 + 45e3 + 720e3 + 800)),
    "up3": dict(kernel="k_tz_up3", per="ship", bytes=80000 + 640000, flops=2 * 11.52e6),
    "up4": dict(kernel="k_tz_up4", per="ship", bytes=640000 + 8, flops=2 * 11.52e6),
    "tail": dict(kernel="k_tz_tail", per="ship", bytes=80000 + 8, flops=2 * (11.52e6 + 11.52e6)),
    "argmax": dict(kernel="k_argmax_final", per="ship", bytes=8, flops=0.0),
}
TENSOR_LAYERS = ("conv3", "conv4", "up3", "up4", "tail")      # tcgen05 kernels: reported against the tensor peak


def time_frame_kernel(bg, maps, flush_buf, dev, iters):
    """k_frame alone (CUDA events, flush or queued work before every launch) -> (mean us, algorithmic bytes per launch)."""
    import torch
    stream = torch.cuda.current_stream(dev)
    map_bytes = maps.numel() * 4
    ts = []
    for _ in range(3):
        bg.frame(maps=maps)
    for _ in range(iters):
        nb = bg.algorithmic_step_bytes() + map_bytes
        if flush_buf is not None:
            flush_buf()
        torch.cuda._sleep(2000000)                        # ~1 ms of queued work: the timed launch is enqueued before the GPU gets to it
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        bg.frame(maps=maps)
        b.record(stream)
        ts.append((a, b, nb))
    torch.cuda.synchronize(dev)
    return sum(a.elapsed_time(b) for a, b, _ in ts) / iters * 1e3, sum(x[2] for x in ts) / iters


def kernel_roofline(bg, maps, flush_buf, wl, dev, policy=None, iters=50):
    """Arena workloads: the dominant kernel is the fused frame kernel (step + raster; the maps are >95 % of its bytes):
    achieved = algorithmic bytes (88 B/ship + 64 B/live laser + the maps it must produce: N * 2 * W*H/8) / mean launch time.
    Policy workloads: the forward's slowest kernel, each kernel against the roofline that really bounds it -- the tcgen05
    kernels as algorithmic FLOPs (Appendix B MACs x 2) / time against the measured bf16 peak, the CUDA-core kernels as
    algorithmic bytes / time against the measured HBM peak (with a note when the kernel is issue-bound rather than
    HBM-bound) -- with the per-layer table, the whole forward in dense-equivalent FLOPs and the frame kernel (HBM) at this
    arena count beside it."""
    import torch
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s"
    stream = torch.cuda.current_stream(dev)
    if policy is not None:
        tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        P = wl["policy"]                                  # policy ships per arena: the trunk runs once per arena, the heads P times
        n = bg.n_arenas
        traffic = _ncu_traffic().get("policy_per_item", {})
        dense_trunk = bool(os.environ.get("OFB_POLICY_DENSE_TRUNK"))

        def profile_now():
            vec = bg.obs_vec[:, :P, :].contiguous().reshape(-1, 8)
            policy.profile(True)
            for _ in range(3):
                policy.forward_argmax(maps, vec, P)
            prof = policy.profile(False)                  # {layer: ms per forward of the whole batch}
            if getattr(policy, "fused_trunk", False) and prof.get("conv3", 0.0) == 0.0:
                prof["trunk"] = prof.pop("trunk12")       # the fused trunk kernel is timed in the first slot
            layers = {}
            for k, ms in prof.items():
                if ms <= 0 or k not in POLICY_LAYERS:
                    continue
                L = POLICY_LAYERS[k]
                items = n * (P if L["per"] == "ship" else 1)
                kern = L.get("kernel") or (L["kernel_dense"] if dense_trunk else L["kernel_sparse"])
                tens = k in TENSOR_LAYERS or (k == "trunk12" and dense_trunk)
                ent = {"kernel": kern, "ms": ms, "bound": "tensor" if tens else "hbm",
                       "alg_tflops": L["flops"] * items / (ms * 1e-3) / 1e12, "alg_gbs": L["bytes"] * items / (ms * 1e-3) / 1e9}
                ent["frac"] = ent["alg_tflops"] / tpeak if tens else ent["alg_gbs"] / peak
                if kern in traffic:
                    ent["ncu_dram_bytes_per_item"] = traffic[kern]
                layers[k] = ent
            return prof, layers

        prof, layers = profile_now()
        dom = max(layers, key=lambda k: layers[k]["ms"])
        total = sum(prof.values())
        D = layers[dom]
        chunks = max(1, -(-n * P // policy.max_ships))
        items_per_launch = min(n * (P if POLICY_LAYERS[dom]["per"] == "ship" else 1), policy.max_ships)
        fus, fbytes = time_frame_kernel(bg, maps, flush_buf, dev, 10)
        ftr = _ncu_traffic().get("arena%d" % n, {})
        roof = {"bound": D["bound"], "kernel": D["kernel"],
                "achieved": D["alg_tflops"] if D["bound"] == "tensor" else D["alg_gbs"],
                "peak": tpeak if D["bound"] == "tensor" else peak, "unit": "TFLOP/s" if D["bound"] == "tensor" else "GB/s",
                "frac": D["frac"],
                "peak_source": ("MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16 GEMM loop)" if D["bound"] == "tensor" else hbm_src)
                               if peaks else "fallback",
                "traffic": traffic[D["kernel"]] * items_per_launch if D["kernel"] in traffic else None,
                "us_per_launch": D["ms"] * 1e3 / chunks,
                "note": "slowest kernel of the forward at the state the timed region ended in; tcgen05 kernels = algorithmic FLOPs "
                        "(Appendix B MACs x 2) / device time vs the measured bf16 peak; CUDA-core kernels = algorithmic bytes / device "
                        "time vs the measured HBM peak (the sparse trunk k_st_trunk12 and k_heads are issue- / latency-bound, not HBM-bound: "
                        "the fraction says how far above their HBM floor they run; the fused tail k_tz_tail is bound by the shared-memory "
                        "port: an SS-mode tcgen05.mma below N = 128 costs max(N/2, 32 + N/4) cycles (measured, profiles/r02_mma_pace.md), "
                        "ncu: tensor-operand + LSU wavefronts = 94 % of the shared-memory data pipe, tensor pipe 57 % active; see DESIGN.md)",
                "whole_forward": {"ms": total, "forwards_per_s": n * P / (total * 1e-3), "policy_ships_per_arena": P,
                                  "dense_equiv_tflops": 155.3e6 * n * P / (total * 1e-3) / 1e12,
                                  "frac_of_peak": 155.3e6 * n * P / (total * 1e-3) / 1e12 / tpeak,
                                  "pointer_head_floor_ms": 47.7e6 * n * P / (tpeak * 1e12) * 1e3,
                                  "note": "dense-equivalent = 155.3 MFLOP per ship-forward (Appendix B), the trunk counted once per SHIP "
                                          "as the reference's batch-1 predict does; the library runs it once per arena; "
                                          "pointer_head_floor_ms = 47.7 MFLOP x ships / measured bf16 peak (SURVEY 8(d))"},
                "layers": layers,
                "frame_kernel": {"bound": "hbm", "kernel": "k_frame", "us_per_launch": fus, "algorithmic_bytes_per_launch": fbytes,
                                 "achieved": fbytes / (fus * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": fbytes / (fus * 1e-6) / 1e9 / peak, "traffic": ftr.get("k_frame"), "peak_source": hbm_src}}
        # the same table at the laser peak of an episode (around frame 30), where the sparse trunk is at its slowest
        if not os.environ.get("OFB_BENCH_NO_EXTRA"):
            bg.restart()
            bg.raster("bits", out=maps)
            for _ in range(30):
                bg.frame(maps=maps)
            prof30, layers30 = profile_now()
            roof["at_laser_peak_frame30"] = {"ms": sum(prof30.values()), "layers_ms": {k: v["ms"] for k, v in layers30.items()}}
        return roof
    res = {}
    map_bytes = maps.numel() * 4
    bg.restart()
    for _ in range(40):                                   # back to the steady-state laser population of a running episode
        bg.frame(maps=maps)
    for name, fn, nbytes in (("k_frame", lambda: bg.frame(maps=maps), lambda: bg.algorithmic_step_bytes() + map_bytes),
                             ("k_raster", lambda: bg.raster("bits", out=maps), map_bytes),
                             ("k_step", lambda: bg.generate_frame(), bg.algorithmic_step_bytes)):
        ts = []
        for _ in range(5):                                # warm-up (module load, clocks)
            fn()
        for _ in range(iters):
            nb = nbytes() if callable(nbytes) else nbytes    # (reads the live laser count: a host sync -- before the flush, so
            if flush_buf is not None:                        #  that the timed launch is queued behind it like in the step loop)
                flush_buf()
            else:
                torch.cuda._sleep(200000)                    # ~100 us of queued work for the same reason
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            ts.append((a, b, nb))
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b, _ in ts) / iters
        nb = sum(x[2] for x in ts) / iters
        res[name] = {"us": ms * 1e3, "bytes": nb, "gbs": nb / (ms * 1e-3) / 1e9}
    dom = "k_frame"
    tr = _ncu_traffic().get("arena%d" % bg.n_arenas, {}) if bg.ships_number == 7 else {}
    return {"bound": "hbm", "kernel": dom, "achieved": res[dom]["gbs"], "peak": peak, "unit": "GB/s",
            "frac": res[dom]["gbs"] / peak,
            "peak_source": hbm_src,
            "traffic": tr.get(dom),
            "traffic_note": "ncu dram__bytes_read+write per launch (profiles/r01_ncu_full_frame*_v4.md): below the algorithmic bytes "
                            "at 4096 arenas because the last ~50 MB of the maps are still dirty in the 126 MB L2 when the kernel ends", "us_per_launch": res[dom]["us"], "algorithmic_bytes_per_launch": res[dom]["bytes"],
            "what": "k_frame = fused step + raster (one persistent launch per frame); algorithmic bytes = 88 B/ship + 64 B/live laser "
                    "+ the 2 x W*H/8-byte maps it must produce, per arena (SURVEY 8(d))",
            "other_kernels": {"k_step": res["k_step"], "k_raster": res["k_raster"]}}


def _max_over_ranks(dt, world, dev):
    if world > 1:
        import torch
        import torch.distributed as dist
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    return dt


def e2e_policy_tape(wl, dev, steps, world, policy, make_bg):
    """Policy workloads end to end with HOST buffers: every frame the scripted ships' action rows come from a pinned host tape
    (H2D on a copy stream), the policy ship's row from the forward on the device, the fused frame kernel steps and rasterises,
    and the compact int16 [N,S,5] observation heads (ofb_obs_pack_i16) go back to pinned host memory (D2H on a third
    stream).  Copies of frame k +- 1 overlap the kernels of frame k.  Wall clock, max over ranks."""
    import torch
    twin = make_bg()
    N, S = twin.n_arenas, twin.ships_number
    T = steps + 3
    tape = torch.empty((T, N, S, 4), dtype=torch.int16).pin_memory()
    for k in range(T):                                     # what the device bots would play on a twin of the batch
        tape[k].copy_(twin.request_actions())
        twin.generate_frame()
    del twin
    torch.cuda.synchronize(dev)
    main = torch.cuda.current_stream(dev)

    def run(pipelined):
        bg = make_bg()
        maps = bg.raster("bits")
        act_dev = [torch.empty((N, S, 4), dtype=torch.int16, device=dev) for _ in range(2)]
        obs_dev = [torch.empty((N, S, 5), dtype=torch.int16, device=dev) for _ in range(2)]
        obs_host = [torch.empty((N, S, 5), dtype=torch.int16).pin_memory() for _ in range(2)]
        s_h2d, s_d2h = (torch.cuda.Stream(dev), torch.cuda.Stream(dev)) if pipelined else (main, main)
        ev_h2d = [torch.cuda.Event() for _ in range(2)]
        ev_frame = [torch.cuda.Event() for _ in range(2)]
        ev_d2h = [torch.cuda.Event() for _ in range(2)]

        def step(k):
            i = k & 1
            if k >= 2:
                s_h2d.wait_event(ev_frame[i])              # frame k - 2 has consumed act_dev[i]
            with torch.cuda.stream(s_h2d):
                act_dev[i].copy_(tape[k], non_blocking=True)
                ev_h2d[i].record(s_h2d)
            decided = policy.decide(bg, maps)              # the forward does not need the tape's rows: it overlaps the copy
            main.wait_event(ev_h2d[i])
            bg.actions = act_dev[i]
            policy.write(bg, *decided)                     # the policy ship's row
            if k >= 2:
                main.wait_event(ev_d2h[i])                 # obs_dev[i] has left for the host
            bg.generate_frame(act_dev[i], maps=maps)       # fused step + maps with every row taken from the buffer
            bg.obs_compact(out=obs_dev[i])
            ev_frame[i].record(main)
            s_d2h.wait_event(ev_frame[i])
            with torch.cuda.stream(s_d2h):
                obs_host[i].copy_(obs_dev[i], non_blocking=True)
                ev_d2h[i].record(s_d2h)

        for k in range(3):
            step(k)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for k in range(3, T):
            step(k)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        st = {k: v.cpu() for k, v in bg.state(("ship_x", "ship_y", "ship_score", "ship_alive", "n_lasers", "kills")).items()}
        return dt, st, obs_host[(T - 1) & 1].clone(), bg.obs_vec.cpu()

    dt, st, last16, last_obs = run(True)
    dt = _max_over_ranks(dt, world, dev)
    _, st_sync, _, _ = run(False)                          # the same tape without the copy streams: the pipelining changes nothing
    same = all(torch.equal(st[k], st_sync[k]) for k in st)
    if not same:
        raise SystemExit("e2e: the pipelined run diverged from the synchronous run of the same tape")
    if not torch.equal(last16.to(torch.float32), last_obs[..., [0, 2, 3, 6, 7]]):
        raise SystemExit("e2e: the compact observation heads on the host differ from the device's")
    return {"unit": "env-steps/s", "h2d_bytes_per_step": N * S * 4 * 2, "d2h_bytes_per_step": N * S * 5 * 2,
            "value": N * world * steps / dt, "steps": steps, "pipelined_equals_synchronous": same,
            "what": "pinned host tape int16[N,S,4] of the scripted ships' actions -> H2D (copy stream) | policy forward + action row of the "
                    "policy ship + fused step + raster (maps stay in HBM) | compact int16[N,S,5] observation heads -> D2H into pinned host "
                    "memory (third stream), every frame; final state equal to a synchronous run of the same tape; wall clock"}


def e2e_arm(bg, maps, wl, dev, steps, world, policy=None, make_bg=None):
    """Same metric through BatchedBattleground with HOST buffers, wall clock, max over ranks.

    Headline `value`: replay of a HOST-resident action tape (the reference's record/replay use, lib/record.py:32-39, and
    the parity mode of the tests): every frame the frame's int16 [N,S,4] actions are copied from pinned host memory, step +
    raster run (+ the policy forward for the policy ship of the policy workloads), and the observation heads (what every bot
    is shown next, incl. its reward; compact int16 [N,S,5] form) are copied back to pinned host memory.  The copies are
    pipelined against the kernels of neighbouring frames.  `closed_loop`: a host-side numpy bot that reads frame k's
    observations before it sends frame k+1 (the numpy bot's CPU time is inside the timed region)."""
    import numpy as np
    import torch
    N, S = bg.n_arenas, bg.ships_number
    out = {"unit": "env-steps/s", "h2d_bytes_per_step": N * S * 4 * 2, "d2h_bytes_per_step": N * S * 5 * 2}

    # ---------------- closed loop (host numpy bot inside the timed region)
    rng = np.random.Generator(np.random.PCG64(7))
    T = 64 if policy is None else 16
    kind = rng.integers(0, 3, size=(T, N, S), dtype=np.int16)
    newp = rng.integers(0, 401, size=(T, N, S, 2), dtype=np.int16)
    act_host = torch.empty((N, S, 4), dtype=torch.int16).pin_memory()
    obs_host = torch.empty((N, S, 8), dtype=torch.float32).pin_memory()
    act_np, obs_np = act_host.numpy(), obs_host.numpy()
    obs_host.copy_(bg.obs_vec)
    torch.cuda.synchronize(dev)

    def host_step(k):
        t = k % T
        decided = None
        if policy is not None:
            if bg.time >= 200:
                bg.restart()
                bg.raster("bits", out=maps)
            decided = policy.decide(bg, maps)               # the forward is queued first: the host bot below overlaps it
        if wl["bot"] == "stress":
            act_np[..., 0] = 1
            act_np[..., 1] = kind[t] & 1
            act_np[..., 2:] = np.minimum(newp[t], 399)
        else:                                               # agents/agent.py:123-133 on the host
            act_np[..., 0] = kind[t] == 0
            act_np[..., 1] = kind[t] == 1
            rep = (kind[t] == 2)[..., None]
            act_np[..., 2:] = np.where(rep, newp[t], obs_np[..., 2:4].astype(np.int16))
        if policy is None:
            if bg.time >= 200:
                bg.restart()
            bg.step_host(act_host, obs_host)                # H2D actions, K1, D2H obs heads (synchronises)
            bg.raster("bits", out=maps)
        else:
            bg.actions.copy_(act_host, non_blocking=True)   # host bots' rows (stream-ordered behind the forward)
            policy.write(bg, *decided)                      # policy ship's row from the forward
            bg.generate_frame(maps=maps)                    # fused step + maps
            obs_host.copy_(bg.obs_vec, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()

    cl_steps = min(steps, 100 if policy is None else 10)
    for k in range(3):
        host_step(k)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(cl_steps):
        host_step(k)
    torch.cuda.synchronize(dev)
    dt = _max_over_ranks(time.perf_counter() - t0, world, dev)
    closed = {"value": N * world * cl_steps / dt, "steps": cl_steps, "h2d_bytes_per_step": N * S * 4 * 2, "d2h_bytes_per_step": N * S * 8 * 4,
              "what": "host numpy bot reads frame k's float32 obs heads before sending frame k+1: pinned actions -> H2D -> "
                      "step -> D2H obs heads -> sync -> raster (maps stay in HBM)%s; bot CPU time inside the timed "
                      "region; wall clock" % (" [policy workloads: the forward of the policy ship is queued first and the host "
                                              "bot's numpy runs while it executes; step + raster fused]" if policy is not None else "")}
    if make_bg is None:
        out.update(value=closed["value"], steps=cl_steps, what=closed["what"], d2h_bytes_per_step=N * S * 8 * 4)
        return out
    if policy is not None:
        out = e2e_policy_tape(wl, dev, steps, world, policy, make_bg)
        out["closed_loop"] = closed
        return out

    # ---------------- action-tape replay, pipelined
    # the tape: what the device bots of this workload play on a twin of the batch (same seed -> same episode)
    steps = max(10, min(steps, (512 * 2 ** 20) // (N * S * 8)))     # keep the pinned tape under 512 MiB
    twin = make_bg()
    tape = torch.empty((steps + 3, N, S, 4), dtype=torch.int16).pin_memory()
    for k in range(steps + 3):
        if twin.time >= 200:
            twin.restart()
        tape[k].copy_(twin.request_actions())
        twin.generate_frame()
    want = {k: v.cpu() for k, v in twin.state(("ship_x", "ship_y", "ship_score", "ship_alive", "n_lasers", "kills")).items()}
    want_obs = twin.obs_vec.cpu()
    del twin
    rep = make_bg()
    obs2 = [torch.empty((N, S, 5), dtype=torch.int16).pin_memory() for _ in range(2)]

    def tape_step(k):
        if rep.time >= 200:
            rep.restart()
        rep.step_host(tape[k], obs2[k & 1], wait=False, maps=maps)   # queue H2D(k) | fused step + raster (k) | pack + D2H(k) on three streams

    for k in range(3):
        tape_step(k)
    rep.wait_host()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for k in range(3, steps + 3):
        tape_step(k)
    rep.wait_host()
    torch.cuda.synchronize(dev)
    dt = _max_over_ranks(time.perf_counter() - t0, world, dev)
    got = {k: v.cpu() for k, v in rep.state(tuple(want)).items()}
    same = all(torch.equal(got[k], want[k]) for k in want)
    if not same:
        raise SystemExit("e2e: the tape replay diverged from the device-bot run it was recorded from")
    last = obs2[(steps + 2) & 1]
    if not torch.equal(last.to(torch.float32), want_obs[..., [0, 2, 3, 6, 7]]):
        raise SystemExit("e2e: the observation heads that arrived on the host differ from the recorded run's")
    out.update(value=N * world * steps / dt, steps=steps, closed_loop=closed, replay_matches_device_run=same,
               what="action-tape replay: pinned host int16[N,S,4] -> H2D -> fused step + raster (ofb_frame_host_async_i16; maps stay in HBM) -> "
                    "the 5 non-constant entries of every observation head as int16[N,S,5] (ofb_obs_pack_i16) -> D2H into pinned host "
                    "memory, every frame; copies on their own streams overlap neighbouring frames' kernels; final state and last heads "
                    "checked against the device-bot run the tape was recorded from; wall clock")
    return out


# ----------------------------------------------------------------------------- main
_JSON_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout: libraries print there too (NCCL's version banner, torchrun notices), so
    everything but the final line is sent to stderr at the file-descriptor level."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        os.write(1, line)
    else:
        os.write(_JSON_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="auto", choices=["auto"] + sorted(WORKLOADS),
                    help="auto = the metric's config: policy (configs[2]) on one GPU, sharded1m (configs[4]) on several")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--learn", default="auto", choices=["auto", "on", "off"],
                    help="policy workloads: QlearnIA.play's learning loop on rank 0 (replay = fit at tracked deaths and every 50 "
                         "frames), weights broadcast, loss in the per-episode reduction (auto = on for sharded1m)")
    ap.add_argument("--flush", default="write+read", choices=["write", "write+read"],
                    help="L2 flush between timed steps when the working set is L2-sized")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, "
                         "a seeded sample of arenas, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    name, wl = resolve_workload(args)
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) != 0:
            return
        steps = args.steps
        v, ms, cores, sample, fwd = cpu_arm_with_policy(wl, steps, min(max(args.warmup, 3), 10))
        emit(({
            "impl": "reference", "metric": METRIC % (" + policy fwd" if wl["policy"] else ""),
            "value": v, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 laser physics / i32 ship state / u32 bit maps" + (" / fp32 policy" if wl["policy"] else ""),
            "data": "synthetic (Philox-seeded)",
            "config": workload_config(name, wl, max(1, args.gpus), wants_learning(args, name, wl)),
            "reference_class": "cpu-port",
            "note": "CPU restatement of the reference's algorithm on a bounded sample of the workload (the reference is pure "
                    "Python and is not part of this repository)" +
                    ("; policy forward = torch-fp32 restatement of the Keras model; learning is not part of the CPU sample"
                     if wl["policy"] else ""),
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    gpu_arm(args, name, wl)


if __name__ == "__main__":
    main()
