"""Cost of learning from every arena: the policy workload (65 536 arenas x 7 ships, ship 0 driven by the policy forward) over
400 frames (the MAX_TIME restart at frame 200 falls inside), per frame in ms from CUDA events:
  (a) act + fused frame, no learning;
  (b) the same + DeviceReplayMemory.push of all arenas (depth 16);
  (c) BatchedQLearner (push, a replay every 50 frames) with trainer batch 8 and 256.
All arms play the same game: the same actor weights (the learner trains its own trainer, not the actor), the same
20-frame collecting phase and the same eps-greedy schedule, so the arms differ only by the learning work.  Each arm runs
twice, in alternation, to show the spread.
Beside it: push in us with its bytes against the measured HBM copy rate, gather at B = 256, fit at B = 8 / 64 / 256, and the
device memory of the ring and of the trainer's workspace.  The card's name and power limit are read in the same run.
Usage: python scripts/learn_bench.py [--frames 400] [--out FILE]  -> one JSON line (and FILE)."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ofighters_b200 import ArenaConfig, BatchedBattleground, _lib  # noqa: E402
from ofighters_b200.policy import PolicyB200  # noqa: E402
from ofighters_b200.replay import DeviceReplayMemory  # noqa: E402
from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200  # noqa: E402

N, SEED, MAX_TIME, DEPTH = 65536, 0x0F16, 200, 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q[torch.cuda.current_device()] if q else None}


def events_ms(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    st = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(st)
    for _ in range(iters):
        fn()
    b.record(st)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def make_bg():
    return BatchedBattleground(N, ships={"QlearnIA": 1, "random": 6}, config=ArenaConfig(), seed=SEED)


def run_loop(frames, policy, mode, batch=None):
    """-> (ms per frame, extras).  mode: "none" | "push" | "learn"."""
    bg = make_bg()
    maps = bg.raster("bits")
    mem = DeviceReplayMemory(bg, depth=DEPTH) if mode != "none" else None
    learner = None
    extras = {}
    if mode == "learn":
        free0 = torch.cuda.mem_get_info()[0]
        tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=batch, max_ships=max(16, batch))
        torch.cuda.synchronize()
        extras["trainer_device_bytes"] = free0 - torch.cuda.mem_get_info()[0]
        learner = BatchedQLearner(tr, mem, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    if mem is not None:
        extras["ring_device_bytes"] = mem.device_bytes
    replays = [0]
    sched = Epsilon_cos(period=110 * 400)
    k = [0]

    def frame():
        if bg.time >= MAX_TIME:
            bg.restart()
            bg.raster("bits", out=maps)
            if learner is not None:
                learner.reset()
        if learner is not None:
            replays[0] += 1 if learner.act(bg, maps)[2] else 0
        else:                                             # BatchedQLearner's choice of actions, without the learning
            collecting = k[0] + 1 < 20
            iact, xy = policy.act(bg, maps, epsilon=sched, collecting=collecting)
            if mem is not None:
                mem.push(iact, xy)
            if not collecting:
                sched.next()
        bg.frame(maps=maps)
        k[0] += 1

    st = torch.cuda.current_stream()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(st)
    for _ in range(frames):
        frame()
    b.record(st)
    torch.cuda.synchronize()
    extras["replays"] = replays[0]
    if mem is not None:
        extras["valid_transitions_at_end"] = len(mem)
    return a.elapsed_time(b) / frames, extras, (bg, maps, mem)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("learn_bench.py measures the GPU path and needs a CUDA device")
    out = {"workload": "policy: %d arenas x 7 ships, ship 0 policy-driven, %d frames, restart at frame %d" % (N, args.frames, MAX_TIME),
           "card": card(), "depth": DEPTH}
    policy = PolicyB200.random_init(seed=0, max_ships=N)
    run_loop(5, policy, "push")                           # warm-up of every kernel on this shape

    out["frame_ms_no_learning"] = [run_loop(args.frames, policy, "none")[0]]
    out["frame_ms_push"] = [run_loop(args.frames, policy, "push")[0]]
    out["frame_ms_no_learning"].append(run_loop(args.frames, policy, "none")[0])
    ms, ex, (bg, maps, mem) = run_loop(args.frames, policy, "push")
    out["frame_ms_push"].append(ms)
    out["ring_device_bytes"] = ex["ring_device_bytes"]
    out["push_valid_transitions_at_end"] = ex["valid_transitions_at_end"]

    # push alone, on the state the loop ended in; its bytes from the live laser counts
    iact, xy = policy.act(bg, maps)
    # each push timed alone after a 512 MB memset, so that the arena state is read from HBM and not from the 126 MB L2
    flush = torch.empty(512 * 2 ** 20, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream()
    samples = []
    for i in range(60):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        mem.push(iact, xy)
        e1.record(st)
        samples.append((e0, e1))
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in samples[10:])
    out["push_us"] = 1e3 * ts[len(ts) // 2]
    out["push_us_min_max"] = [1e3 * ts[0], 1e3 * ts[-1]]
    del flush
    n_l = bg.state(("n_lasers",))["n_lasers"].long()
    lay_off_laser = 32 + 16 * 8
    snap = int((lay_off_laser + (n_l + 7) // 8 * 288).sum())
    meta = N * (4 + 8 + 1) + N * (16 + 4 + 4 + 1 + 1 + 4)   # new slot's action/pointer/valid; previous slot's ship+header reads, valid/reward/done
    out["push_bytes"] = {"snapshot_read": snap, "snapshot_write": snap, "fields": meta, "total": 2 * snap + meta,
                         "mean_snapshot_bytes_per_arena": snap / N}
    buf = torch.empty(2 * 2 ** 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(buf)
    copy_ms = events_ms(lambda: dst.copy_(buf), 20)
    out["hbm_copy_peak_GBps"] = 2 * buf.numel() / (copy_ms * 1e-3) / 1e9
    out["push_GBps"] = out["push_bytes"]["total"] / (out["push_us"] * 1e-6) / 1e9
    out["push_share_of_copy_peak"] = out["push_GBps"] / out["hbm_copy_peak_GBps"]
    del buf, dst

    # gather at B = 256 (the C call alone, outputs preallocated)
    n = len(mem)
    B = 256
    pos = torch.randperm(n)[:B].cuda()
    ids = mem._ids.index_select(0, pos).contiguous()
    o = [torch.empty((B, 2, 5000), dtype=torch.int32, device="cuda"), torch.empty((B, 8), device="cuda"),
         torch.empty((B, 2, 5000), dtype=torch.int32, device="cuda"), torch.empty((B, 8), device="cuda"),
         torch.empty((B,), dtype=torch.int32, device="cuda"), torch.empty((B, 2), dtype=torch.int32, device="cuda"),
         torch.empty((B,), device="cuda"), torch.empty((B,), dtype=torch.uint8, device="cuda")]
    lib = _lib.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out["gather_us_B256"] = 1e3 * events_ms(lambda: _lib.check(lib.ofb_replay_gather(
        mem._h, C.c_void_p(ids.data_ptr()), B, *[C.c_void_p(t.data_ptr()) for t in o], s)), 50)
    out["gather_bytes_B256"] = 2 * B * 40000
    g = mem.sample(256)
    del mem, bg

    # fit at B = 8, 64, 256 on sampled transitions
    free0 = torch.cuda.mem_get_info()[0]
    tr = TrainerB200(learning_rate=1e-4, batch_size=256, max_ships=256)
    torch.cuda.synchronize()
    out["trainer_device_bytes_B256"] = free0 - torch.cuda.mem_get_info()[0]
    gen = torch.Generator().manual_seed(1)
    ta = (torch.randn((256, 2), generator=gen) * 3).cuda()
    tp = (torch.randn((256, 400, 400), generator=gen) * 0.5).cuda()
    out["fit_ms"] = {}
    for b in (8, 64, 256):
        out["fit_ms"][str(b)] = events_ms(lambda: tr.fit(g.maps_next[:b].contiguous(), g.vec_next[:b], ta[:b].contiguous(),
                                                        tp[:b].contiguous(), sync_model=False), 10)
    del tr, ta, tp

    for rep in range(2):
        for b in (8, 256):
            ms, ex, _ = run_loop(args.frames, policy, "learn", batch=b)
            out.setdefault("frame_ms_learn_B%d" % b, []).append(ms)
            out["learn_B%d" % b] = ex
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
