"""Arena-level sharding over the GPUs of one box (SURVEY 8(e)).

Arenas never read each other (lib/battleground.py:32-44 holds all of an arena's state), so the
hot path shards with no data-path collective: rank g of G owns the contiguous global arena ids
``[g*N/G, (g+1)*N/G)`` and keys its device RNG by GLOBAL arena id (``arena0``), which makes every
arena's trajectory independent of G.  The only exchange is the per-episode statistics vector
``[sum score, kills, deaths, shots, ships, arenas]`` (what the reference accumulates in
``agent.scores`` / ``last_x_time_rewards``): one all-reduce(sum) of 6 int64 per 200-frame episode -- plus, when a rank
learns (trainer.QLearner), the episode's [sum of replay losses, replays] pair and a broadcast of the single shared
trainer's weights (572 k floats) after each scheduled replay.
Works with any ``torch.distributed`` backend: NCCL over NVLink on the GPU box, gloo in CPU tests.
"""
import torch
import torch.distributed as dist

STAT_NAMES = ("score", "kills", "deaths", "shots", "ships", "arenas")


def shard_range(n_total, rank, world):
    """Global arena ids [lo, hi) owned by ``rank``; sizes differ by at most one, lower ranks first."""
    if world < 1 or not 0 <= rank < world:
        raise Exception("Invalid rank {} for world size {}.".format(rank, world))
    base, extra = divmod(int(n_total), world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def reduce_episode_stats(stats, group=None, async_op=False):
    """In-place sum of the 6-entry int64 statistics tensor over all ranks (no-op without a process group)."""
    if stats.dtype != torch.int64 or stats.numel() != len(STAT_NAMES):
        raise Exception("Invalid statistics tensor : expected int64 [{}].".format(len(STAT_NAMES)))
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None
    return dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group, async_op=async_op)


def reduce_loss_stats(loss_stats, group=None):
    """In-place sum over all ranks of the float64 [sum of replay losses, replays] pair of an episode -- the "loss" half of
    the per-episode score/loss reduction (only ranks that learn contribute non-zero entries)."""
    if loss_stats.dtype != torch.float64 or loss_stats.numel() != 2:
        raise Exception("Invalid loss statistics tensor : expected float64 [2].")
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None
    return dist.all_reduce(loss_stats, op=dist.ReduceOp.SUM, group=group)


def broadcast_weights(flat, src=0, group=None):
    """The reference has ONE trainer shared by every bot (agents/qlearnIA_V2.py:308, "All bots share the same trainer" :362):
    the learning rank's flat fp32 weights (include/ofb_train.h order) replace everyone's, in place.  No-op without a group."""
    if flat.dtype != torch.float32 or flat.dim() != 1:
        raise Exception("Invalid weights tensor : expected flat float32.")
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return None
    return dist.broadcast(flat, src=src, group=group)


class DistReducer:
    """The reducer of a data-parallel ``TrainerB200`` (``reducer=``) over a ``torch.distributed`` process group: every rank
    of ``group`` builds its trainer with one.  ``all_reduce`` sums (or takes the minimum / maximum) in place, ordered after
    the work queued on the current stream -- what the trainer's reduce hook needs, since the fit's kernels run on that
    stream.  NCCL gives every rank the same bits.  Create the group with a ``timeout``, so that a rank that stops calling
    fails the others instead of hanging them.

        dist.init_process_group("nccl", timeout=datetime.timedelta(seconds=120))
        trainer = TrainerB200(weights, batch_size=8, reducer=DistReducer())
    """

    _OPS = {"sum": "SUM", "min": "MIN", "max": "MAX"}

    def __init__(self, group=None):
        if not (dist.is_available() and dist.is_initialized()):
            raise Exception("DistReducer needs an initialised torch.distributed process group.")
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)

    def all_reduce(self, tensor, op="sum"):
        if op not in self._OPS:
            raise Exception("Invalid op {} : expected one of {}.".format(op, sorted(self._OPS)))
        dist.all_reduce(tensor, op=getattr(dist.ReduceOp, self._OPS[op]), group=self.group)

    def broadcast(self, tensor, src=0):
        """``tensor`` of group rank ``src`` to every rank, in place."""
        g_src = src if self.group is None else dist.get_global_rank(self.group, src)
        dist.broadcast(tensor, src=g_src, group=self.group)


def stats_dict(stats):
    v = stats.detach().cpu().tolist()
    return dict(zip(STAT_NAMES, v))


def make_sharded_battleground(n_total, rank=None, world=None, **kw):
    """``BatchedBattleground`` for this rank's slice of ``n_total`` arenas (needs a GPU)."""
    from .battleground import BatchedBattleground
    if world is None:
        world = dist.get_world_size() if dist.is_initialized() else 1
    if rank is None:
        rank = dist.get_rank() if dist.is_initialized() else 0
    lo, hi = shard_range(n_total, rank, world)
    return BatchedBattleground(hi - lo, arena0=lo, **kw)
