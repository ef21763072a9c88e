"""Cost of the target network and Double DQN (TrainerB200(target_update=..., double_dqn=True)) at configs[2]: 65 536 arenas x 7
ships, ship 0 policy-driven, depth 16.
  * ofb_trainer_td_targets_double against ofb_trainer_td_targets and against ofb_trainer_td_errors + ofb_trainer_td_targets (the
    prioritized path's two passes) at B = 8 / 64 / 256, in place as replay calls them.  Each call is timed alone with CUDA
    events after a 512 MB write that evicts the 126 MB L2, the arms alternated call by call, 40 calls per arm; the median and
    the spread (min, max) are reported, with the bytes the kernel must move over the median time, against the copy rate
    measured in the same run (a 2 GB device-to-device copy: bytes read + written over its time);
  * one target refresh: get_weights (the host copy sync_model already makes), the fp32 blend and the target engine's
    load_weights (BN fold + upload), host clock around synchronised work;
  * BatchedQLearner per frame over 400 frames (the restart at frame 200 inside) at trainer batch 8 and 256, with
    DeviceReplayMemory, Double DQN with a refresh after every fit (target_update=1, the most refreshes) against no target
    network, two runs per arm with the arms alternated;
  * an INDICATOR, not a pass criterion: over the replays of a Double DQN run (batch 256, target_update=2), the mean over
    sampled next observations of max Q_online(s') - Q_target(s', p*) of the pointer head, p* the online argmax.
The card's name and power limit are read in the same run.
Usage: python scripts/double_bench.py [--frames 400] [--out FILE]  -> one JSON line (and FILE)."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from learn_bench import card  # noqa: E402
from ofighters_b200 import ArenaConfig, BatchedBattleground, _lib  # noqa: E402
from ofighters_b200.policy import PolicyB200  # noqa: E402
from ofighters_b200.replay import DeviceReplayMemory  # noqa: E402
from ofighters_b200.trainer import BatchedQLearner, Epsilon_cos, TrainerB200, blend_weights  # noqa: E402

SEED, MAX_TIME, DEPTH, N, GAMMA = 0x0F16, 200, 16, 65536, 0.9
SHIPS = {"QlearnIA": 1, "random": 6}
MAP_BYTES = 400 * 400 * 4


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _median(x):
    x = sorted(x)
    return x[len(x) // 2]


def copy_rate():
    """Device-to-device copy of 2 GB: (read + written bytes) / time, GB/s."""
    a = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * a.numel() * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9


def kernel_costs(lib, s, B, calls=40):
    g = torch.Generator(device="cuda").manual_seed(B)
    act_o, ptr_o = torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)
    act_n, ptr_n = torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)
    act_t, ptr_t = torch.randn((B, 2), device="cuda", generator=g), torch.randn((B, 400, 400), device="cuda", generator=g)
    ia = torch.randint(0, 2, (B,), dtype=torch.int32, device="cuda", generator=g)
    pt = torch.randint(0, 400, (B, 2), dtype=torch.int32, device="cuda", generator=g)
    r = torch.zeros(B, device="cuda")
    d = torch.zeros(B, dtype=torch.uint8, device="cuda")
    tda, tdp = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
    single = [_p(t) for t in (act_o, ptr_o, act_n, ptr_n, ia, pt, r, d)]
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    arms = {
        "td_targets": lambda: _lib.check(lib.ofb_trainer_td_targets(*single, GAMMA, B, _p(act_o), _p(ptr_o), s)),
        "td_errors+td_targets": lambda: (_lib.check(lib.ofb_trainer_td_errors(*single, GAMMA, B, _p(tda), _p(tdp), s)),
                                         _lib.check(lib.ofb_trainer_td_targets(*single, GAMMA, B, _p(act_o), _p(ptr_o), s))),
        "td_targets_double": lambda: _lib.check(lib.ofb_trainer_td_targets_double(
            *[_p(t) for t in (act_o, ptr_o, act_n, ptr_n, act_t, ptr_t, ia, pt, r, d)], GAMMA, None, B, _p(act_o), _p(ptr_o),
            None, None, s)),
        "td_targets_double+td": lambda: _lib.check(lib.ofb_trainer_td_targets_double(
            *[_p(t) for t in (act_o, ptr_o, act_n, ptr_n, act_t, ptr_t, ia, pt, r, d)], GAMMA, None, B, _p(act_o), _p(ptr_o),
            _p(tda), _p(tdp), s)),
    }
    times = {k: [] for k in arms}
    st = torch.cuda.current_stream()
    for k in range(calls + 3):
        for name, fn in arms.items():                     # the arms alternated call by call
            flush.fill_(k & 0xff)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            fn()
            e1.record(st)
            e1.synchronize()
            if k >= 3:
                times[name].append(1e3 * e0.elapsed_time(e1))
    # bytes each arm must move: the map(s) read, in place (the obs maps' copy is not made)
    need = {"td_targets": B * MAP_BYTES, "td_errors+td_targets": 2 * B * MAP_BYTES, "td_targets_double": B * MAP_BYTES,
            "td_targets_double+td": B * MAP_BYTES}
    out = {}
    for name, t in times.items():
        med = _median(t)
        out[name] = {"us_median": med, "us_min": min(t), "us_max": max(t), "bytes": need[name],
                     "GB_per_s": need[name] / (med * 1e-6) / 1e9}
    return out


def refresh_cost(reps=5):
    tr = TrainerB200(learning_rate=1e-4, batch_size=8, max_ships=16, target_update=1)
    res = {"get_weights_ms": [], "blend_ms": [], "target_load_weights_ms": []}
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        w = tr.get_weights()
        t1 = time.perf_counter()
        wt = blend_weights(w, tr.get_target_weights(), 0.5)
        t2 = time.perf_counter()
        tr.target_model.load_weights(wt)
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        res["get_weights_ms"].append(1e3 * (t1 - t0))
        res["blend_ms"].append(1e3 * (t2 - t1))
        res["target_load_weights_ms"].append(1e3 * (t3 - t2))
    return res


def learn_loop(frames, policy, batch, double, target_update=1, gaps=None):
    """BatchedQLearner at configs[2] -> (ms per frame, replays)."""
    bg = BatchedBattleground(N, ships=SHIPS, config=ArenaConfig(), seed=SEED)
    maps = bg.raster("bits")
    mem = DeviceReplayMemory(bg, depth=DEPTH)
    kw = dict(target_update=target_update, double_dqn=True) if double else {}
    tr = TrainerB200(learning_rate=1e-4, epsilon=Epsilon_cos(period=110 * 400), batch_size=batch, max_ships=max(16, batch), **kw)
    learner = BatchedQLearner(tr, mem, replay_every=50, collecting_steps=20, snapshot=0, actor=policy)
    if gaps is not None:                                  # indicator: max Q_online(s') - Q_target(s', p*) of the pointer head
        orig = tr._td_targets_double

        def spy(act_o, ptr_o, maps_n, vec_n, *a, **k):
            on = tr.predict(maps_n, vec_n)[1].reshape(maps_n.shape[0], -1)
            tg = tr.target_model.forward(maps_n, vec_n, 1, want_ptr=True)["ptr"].reshape(maps_n.shape[0], -1)
            mx, p = on.max(dim=1)
            gaps.append(float((mx - tg.gather(1, p[:, None])[:, 0]).double().mean()))
            return orig(act_o, ptr_o, maps_n, vec_n, *a, **k)
        tr._td_targets_double = spy
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
    return e0.elapsed_time(e1) / frames, replays, tr.target_updates


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=400)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("double_bench.py measures the GPU path and needs a CUDA device")
    lib = _lib.load()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = {"card": card(), "depth": DEPTH, "arenas": N, "l2_flush": "512 MB write before every timed call"}
    out["copy_GB_per_s"] = copy_rate()
    torch.cuda.empty_cache()
    for B in (8, 64, 256):
        out["td_B%d" % B] = kernel_costs(lib, s, B)
        torch.cuda.empty_cache()
    out["refresh"] = refresh_cost()
    policy = PolicyB200.random_init(seed=0, max_ships=N)
    learn_loop(5, policy, 8, True)                        # warm-up of every kernel on this shape
    learn = {}
    for batch in (8, 256):
        for rep in range(2):
            for double in (False, True):
                ms, k, ups = learn_loop(args.frames, policy, batch, double)
                arm = learn.setdefault("B%d_%s" % (batch, "double_C1" if double else "single"),
                                       {"frame_ms": [], "replays": k, "target_updates": ups})
                arm["frame_ms"].append(ms)
                torch.cuda.empty_cache()
    out["learn_%d_frames" % args.frames] = learn
    gaps = []
    learn_loop(args.frames, policy, 256, True, target_update=2, gaps=gaps)
    out["indicator_ptr_gap_online_max_minus_target_at_argmax"] = {"batch": 256, "target_update": 2, "per_replay": gaps,
                                                                 "mean": sum(gaps) / max(len(gaps), 1)}
    out["card_after"] = card()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
