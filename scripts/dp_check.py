"""Data-parallel fit over NCCL (TrainerB200(reducer=sharding.DistReducer())): a check to run on 1 to 8 GPUs of one box.

    python -m torch.distributed.run --nproc-per-node 8 scripts/dp_check.py [--fits 20] [--out FILE]

Every rank holds an uneven shard (3, 4 or 5 samples by rank) of one global batch and takes --fits sharded fits on it:
  * after every fit the weights of every rank hash identically (an all-reduce MIN of the hash equals the MAX);
  * rank 0 gathers the shards, runs a one-GPU trainer from the same initial weights on the concatenated batch and compares:
    the first fit's losses (1e-6 relative) and gradients (2e-3 of each tensor's largest gradient), every later fit's losses
    (2e-5 relative: the two fp32 runs part slowly, as Adam turns gradient noise into +-lr steps), and the weights after the
    last fit (within 2.2e-4 per step; the share of each tensor's elements within 5e-6 per step is reported, not checked:
    over 20 steps that share is set by the noise, not by the sharding);
  * the process group has a timeout and is destroyed before the script exits on every rank.
Rank 0 prints one JSON line (and writes it to FILE).  Exit code 0 when every check holds."""
import argparse
import datetime
import hashlib
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ofighters_b200 import BatchedBattleground, sharding  # noqa: E402
from ofighters_b200.trainer import TrainerB200, flatten_weights  # noqa: E402
from oracle import policy_torch as po  # noqa: E402


def weights_hash(tr):
    b = flatten_weights(tr.get_weights()).numpy().tobytes()
    return int.from_bytes(hashlib.sha256(b).digest()[:7], "little")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fits", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=300), device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    try:
        sizes = [3 + (r % 3) for r in range(world)]
        lo = sum(sizes[:rank])
        bg = BatchedBattleground(sizes[rank], ships={"random": 7}, seed=11, device=dev, arena0=lo)
        for _ in range(35):
            bg.frame()
        maps = bg.raster("bits")
        vec = bg.obs_vec[:, 0, :].contiguous()
        g = torch.Generator().manual_seed(1000 + rank)
        ta = (torch.randn((sizes[rank], 2), generator=g) * 3).to(dev)
        tp = (torch.randn((sizes[rank], 400, 400), generator=g) * 0.5).to(dev)
        w = po.init_weights(4, randomize_bn=True)
        tr = TrainerB200(weights=w, learning_rate=1e-4, batch_size=max(sizes), device=dev, max_ships=8,
                         reducer=sharding.DistReducer())
        losses, hashes_ok, grads1 = [], True, None
        for i in range(args.fits):
            losses.append(tr.fit(maps, vec, ta, tp).cpu())
            if i == 0:
                grads1 = tr.get_grads()
            h = torch.tensor([weights_hash(tr)], dtype=torch.int64, device=dev)
            hmin, hmax = h.clone(), h.clone()
            dist.all_reduce(hmin, op=dist.ReduceOp.MIN)
            dist.all_reduce(hmax, op=dist.ReduceOp.MAX)
            hashes_ok &= int(hmin.item()) == int(hmax.item())
        final = tr.get_weights()
        shard = {"maps": maps.cpu(), "vec": vec.cpu(), "ta": ta.cpu(), "tp": tp.cpu()}
        gathered = [None] * world if rank == 0 else None
        dist.gather_object(shard, gathered, dst=0)
        result = {"world": world, "sizes": sizes, "fits": args.fits, "hashes_identical": bool(hashes_ok)}
        ok = bool(hashes_ok)
        if rank == 0:
            cat = {k: torch.cat([s[k] for s in gathered]).to(dev).contiguous() for k in shard}
            single = TrainerB200(weights=w, learning_rate=1e-4, batch_size=sum(sizes), device=dev, max_ships=8)
            ref_losses, ref_grads1 = [], None
            for i in range(args.fits):
                ref_losses.append(single.fit(cat["maps"], cat["vec"], cat["ta"], cat["tp"]).cpu())
                if i == 0:
                    ref_grads1 = single.get_grads()
            loss_err = [float(((a - b).abs() / b.abs()).max()) for a, b in zip(losses, ref_losses)]
            zero_grad = [k for k in ref_grads1 if k.endswith("/bias") and "conv" in k and k != "upconv4/bias"]
            grad_err = {}
            for k, rg in ref_grads1.items():
                scale = max(float(rg.abs().max()),
                            float(ref_grads1[k.replace("/bias", "/kernel")].abs().max()) if k in zero_grad else 0.0)
                grad_err[k] = float((grads1[k] - rg).abs().max()) / max(scale, 1e-30)
            ref_final = single.get_weights()
            traj_ok, traj_bad, share_min = True, [], 1.0
            for k in ref_final:
                diff = (final[k].double() - ref_final[k].double()).abs()
                if float(diff.max()) > 2.2e-4 * args.fits:
                    traj_ok = False
                    traj_bad.append(k)
                if k not in zero_grad and not (k.endswith("/mean") or k.endswith("/var")):
                    share_min = min(share_min, float((diff <= 5e-6 * args.fits).float().mean()))
            result.update({"loss_rel_err_first": loss_err[0], "loss_rel_err_max": max(loss_err),
                           "grad_err_max_over_scale": max(grad_err.values()), "trajectory_within_bounds": bool(traj_ok),
                           "trajectory_out_of_bounds": traj_bad, "min_share_within_5e-6_per_step": share_min,
                           "loss_first": losses[0].tolist(), "loss_last": losses[-1].tolist(),
                           "card": torch.cuda.get_device_name(dev)})
            ok &= loss_err[0] <= 1e-6 and max(loss_err) <= 2e-5 and max(grad_err.values()) <= 2e-3 and traj_ok
            result["ok"] = bool(ok)
            line = json.dumps(result)
            print(line)
            if args.out:
                with open(args.out, "w") as f:
                    f.write(line + "\n")
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.broadcast(flag, src=0)
        ok = bool(flag.item())
    finally:
        dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
