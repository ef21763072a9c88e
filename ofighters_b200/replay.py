"""Device-resident replay memory: the ``Trainer.memory`` of the reference (agents/qlearnIA_V2.py:237-238) for every arena of a
batch, through include/ofb_replay.h.

``Trainer.memory`` is a deque of (obs, iaction, ipointer, reward, next_obs, done) whose observations are a pair of 400x400
maps.  Kept like that for a batch, every arena would cost 40 KB of bit maps per frame.  ``DeviceReplayMemory`` keeps a ring
of arena state snapshots on the device instead -- header, ships and the live laser list, about 1 KB per arena at the
default workload -- and rasterises only the transitions a replay samples, with the frame kernel's raster code, so a
gathered map is bit for bit the map the frame wrote.  Transitions follow ``QlearnIA.play`` (:372-401): one per policy ship
that is alive at t, none across a restart (masked restarts included), a death once with done = 1.

    memory = DeviceReplayMemory(bg, depth=16)     # all arenas, the battleground's QlearnIA / external ships
    iact, xy = policy.act(bg, maps, ...)          # the PLAYED actions
    memory.push(iact, xy)                         # before bg.frame(): the snapshot is the observation acted on
    bg.frame(maps=maps)
    trainer.replay(trainer.batch_size, memory=memory)

``push`` never synchronises the host.  ``len()`` does (it compacts the valid transitions and reads their number), and so does
``sample``.  The order of the transitions -- oldest frame first, then arena, then ship -- is the order in which ``QLearner``
appends to ``trainer.memory``, and ``sample`` draws ``random.sample(range(len), batch_size)`` with Python's ``random`` as
``Trainer.replay`` does on its deque, so the same ``random`` state picks the same minibatch.

``PrioritizedReplayMemory`` adds prioritized replay on the device: masses from the TD errors, a stratified proportional sampler
and importance weights for ``TrainerB200.fit(..., sample_weight=...)``.

Either memory takes ``n_step``: with n > 1 a transition is an n-step window, gathered on the device with its discounted return
R = sum_j gamma^j r_{t+j} over k <= n frames, its bootstrap observation s_{t+k} and discount = gamma^k (include/ofb_replay.h
states the rules).  A shot bonus then reaches back n frames per fit instead of one.

    memory = DeviceReplayMemory(bg, depth=16, n_step=3)       # gamma = trainer.gamma = 0.9
    learner = BatchedQLearner(trainer, memory)
"""
import ctypes as C
import random
from types import SimpleNamespace

import torch

from . import _lib

_POLICY_BEHAVIORS = ("QlearnIA", "external")


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


class DeviceReplayMemory:
    def __init__(self, bg, depth=16, track=None, ships=None, n_step=1, gamma=0.9):
        """``bg``: the BatchedBattleground whose arenas are remembered.  ``depth``: frames in the ring (>= 2); it holds the
        transitions of the last ``depth - 1`` pushed frames.  ``track``: the first ``track`` arenas (default: all).
        ``ships``: ship indices to remember, among the battleground's QlearnIA / external ships (default: all of them);
        ``push`` takes the actions of all those ships, as ``PolicyB200.act`` returns them.
        ``n_step``: frames of a transition's return (1 <= n_step <= depth - 1); with n_step > 1 the ring holds the
        transitions of the frames [T - depth + 1, T - n_step] (T = the newest), ``gather`` returns the n-step return R in
        ``reward`` with ``discount`` = gamma^k and ``steps`` = k, and ``gamma`` discounts the rewards inside the window (it
        must be the trainer's)."""
        if not torch.cuda.is_available():
            raise _lib.OfbError("DeviceReplayMemory needs a CUDA device: the ring lives in HBM and has no CPU fallback")
        policy = [i for i, b in enumerate(bg.behaviors) if b in _POLICY_BEHAVIORS]
        if not policy:
            raise Exception("no policy-driven ship in this battleground")
        ships = list(policy) if ships is None else [int(s) for s in ships]
        if not ships or len(set(ships)) != len(ships) or any(s not in policy for s in ships):
            raise Exception("Invalid ships {} : expected distinct policy-driven ships among {}.".format(ships, policy))
        track = bg.n_arenas if track is None else int(track)
        if not 1 <= track <= bg.n_arenas:
            raise Exception("Invalid track {} : the batch holds {} arenas.".format(track, bg.n_arenas))
        n_step, gamma = int(n_step), float(gamma)
        if n_step < 1 or (n_step > 1 and int(depth) < n_step + 1):      # (a one-step memory's depth is ofb_replay_create's)
            raise Exception("Invalid n_step {} : need 1 <= n_step <= depth - 1 = {}.".format(n_step, int(depth) - 1))
        if not 0.0 <= gamma < float("inf"):
            raise Exception("Invalid gamma {} : expected a finite value >= 0.".format(gamma))
        self.bg = bg
        self.device = bg.device
        self.depth = int(depth)
        self.track = track
        self.ships = ships
        self.n_step, self.gamma = n_step, gamma
        self.n_policy = len(policy)                      # policy ships per arena in the actions push() takes
        self._cols = None if ships == policy else torch.tensor([policy.index(s) for s in ships], dtype=torch.long,
                                                               device=self.device)
        self._lib = _lib.load()
        idx = (C.c_int32 * len(ships))(*ships)
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.ofb_replay_create(bg._h, 0, track, idx, len(ships), self.depth, C.byref(h)))
        self._h = h
        if n_step > 1:
            _lib.check(self._lib.ofb_replay_set_n_step(h, n_step))
        self._ids = torch.empty(max(1, (self.depth - 1) * track * len(ships)), dtype=torch.int32, device=self.device)
        self._count = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._n = 0
        self._stale = False
        self.launch_count = 0

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                self._lib.ofb_replay_destroy(h)
            except Exception:
                pass
            self._h = None

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def device_bytes(self):
        """HBM the memory owns: the ring of snapshots, the per-transition fields and the index scratch."""
        return int(self._lib.ofb_replay_device_bytes(self._h))

    @property
    def frames(self):
        """Frames pushed so far."""
        return int(self._lib.ofb_replay_pushes(self._h))

    # ------------------------------------------------------------------ write
    def push(self, iaction, xy, bg=None):
        """Remember the current state of the tracked arenas with the actions their policy ships PLAY from it: ``iaction``
        int32 [A*P] and ``xy`` int32 [A*P, 2] as ``PolicyB200.act`` returns them (A arenas, P policy ships).  Call it after
        the actions were chosen and before ``bg.frame``.  Asynchronous: no host synchronisation."""
        if bg is not None and bg is not self.bg:
            raise Exception("Invalid battleground : this memory remembers another battleground's arenas.")
        N, P = self.bg.n_arenas, self.n_policy
        for name, t, shapes in (("iaction", iaction, ((N * P,), (N, P))), ("xy", xy, ((N * P, 2), (N, P, 2)))):
            if not isinstance(t, torch.Tensor) or t.dtype != torch.int32 or t.device != self.device or \
                    tuple(t.shape) not in shapes:
                raise Exception("Invalid {} : expected an int32 tensor of shape {} on {}.".format(name, shapes[0], self.device))
        iaction, xy = iaction.reshape(N, P), xy.reshape(N, P, 2)
        if self._cols is not None:
            iaction, xy = iaction.index_select(1, self._cols), xy.index_select(1, self._cols)
        iaction, xy = iaction.contiguous(), xy.contiguous()
        _lib.check(self._lib.ofb_replay_push(self._h, self.bg._h, _ptr(iaction), _ptr(xy), self._stream()))
        self.launch_count += 1
        self._stale = True

    # ------------------------------------------------------------------ read
    def __len__(self):
        """Number of valid transitions (synchronises with the device)."""
        if self._stale:
            _lib.check(self._lib.ofb_replay_index(self._h, _ptr(self._ids), _ptr(self._count), self._stream()))
            self.launch_count += 3
            self._n = int(self._count.item())
            self._stale = False
        return self._n

    def gather(self, positions):
        """The transitions at ``positions`` (0 = oldest) -> SimpleNamespace of device tensors: maps_obs / maps_next int32
        [B, 2, W*H/32] bit maps, vec_obs / vec_next float32 [B, 8], iaction int32 [B], pointer int32 [B, 2] = (x, y),
        reward float32 [B], done uint8 [B] -- the inputs of ``TrainerB200.replay``'s targets and fit.  An n-step memory
        (n_step > 1) puts the return R in ``reward``, s_{t+k} in maps_next / vec_next and adds ``discount`` float32 [B]
        (gamma^k) and ``steps`` int32 [B] (k)."""
        n = len(self)
        pos = torch.as_tensor(positions, dtype=torch.int64).reshape(-1)
        if pos.numel() < 1:
            raise Exception("gather of no transition")
        if int(pos.min()) < 0 or int(pos.max()) >= n:
            raise Exception("Invalid positions : the memory holds {} transitions.".format(n))
        return self._gather_ids(self._ids.index_select(0, pos.to(self.device)).contiguous())

    def _gather_ids(self, ids):
        """``gather`` of transition ids (int32 [B] on the device, valid until the next push)."""
        B = ids.numel()
        words = self.bg.config.width * self.bg.config.height // 32
        dev = self.device
        out = SimpleNamespace(
            maps_obs=torch.empty((B, 2, words), dtype=torch.int32, device=dev),
            vec_obs=torch.empty((B, 8), dtype=torch.float32, device=dev),
            maps_next=torch.empty((B, 2, words), dtype=torch.int32, device=dev),
            vec_next=torch.empty((B, 8), dtype=torch.float32, device=dev),
            iaction=torch.empty((B,), dtype=torch.int32, device=dev),
            pointer=torch.empty((B, 2), dtype=torch.int32, device=dev),
            reward=torch.empty((B,), dtype=torch.float32, device=dev),
            done=torch.empty((B,), dtype=torch.uint8, device=dev))
        if self.n_step > 1:
            out.discount = torch.empty((B,), dtype=torch.float32, device=dev)
            out.steps = torch.empty((B,), dtype=torch.int32, device=dev)
            _lib.check(self._lib.ofb_replay_gather_nstep(
                self._h, _ptr(ids), B, self.gamma, _ptr(out.maps_obs), _ptr(out.vec_obs), _ptr(out.maps_next), _ptr(out.vec_next),
                _ptr(out.iaction), _ptr(out.pointer), _ptr(out.reward), _ptr(out.done), _ptr(out.discount), _ptr(out.steps),
                self._stream()))
            self.launch_count += 1
            return out
        _lib.check(self._lib.ofb_replay_gather(self._h, _ptr(ids), B, _ptr(out.maps_obs), _ptr(out.vec_obs), _ptr(out.maps_next),
                                               _ptr(out.vec_next), _ptr(out.iaction), _ptr(out.pointer), _ptr(out.reward),
                                               _ptr(out.done), self._stream()))
        self.launch_count += 1
        return out

    def sample(self, batch_size, rng=None):
        """``random.sample(range(len(self)), batch_size)`` -- the draw ``Trainer.replay`` makes on its deque -- gathered.
        ``rng``: a ``random.Random`` to draw with instead of the module's shared state (each rank of a data-parallel trainer
        keeps its own)."""
        n = len(self)
        if n < 1:
            raise Exception("sample on an empty replay memory")
        return self.gather((random if rng is None else rng).sample(range(n), batch_size))


class EmptyReplayMemory(Exception):
    """A prioritized sample found no transition to draw."""


class PrioritizedReplayMemory(DeviceReplayMemory):
    """``DeviceReplayMemory`` with prioritized replay (Schaul et al. 2016, proportional variant), on the device.

    Every transition carries a sampling mass, ``(|td_act| + |td_ptr| + eps) ** alpha`` from the TD errors of its last replay,
    or the largest mass set so far when it enters the memory, so that a new transition is likely drawn at least once.
    ``sample_prioritized`` draws a stratified minibatch in proportion to the masses with the importance weights that undo
    the bias, ``update_priorities`` writes the new errors back.  ``TrainerB200.replay(..., memory=this, beta=...)`` runs the
    whole sequence.

        memory = PrioritizedReplayMemory(bg, depth=16, alpha=0.6)
        ...                                           # push as for DeviceReplayMemory
        trainer.replay(trainer.batch_size, memory=memory, beta=0.4)

    The sampler's random stream is Philox keyed by ``seed`` and the number of samples drawn, so a run is reproducible.
    With ``n_step`` > 1 a transition enters with the largest mass at the push that makes it a candidate (n frames later)."""

    def __init__(self, bg, depth=16, track=None, ships=None, alpha=0.6, eps=1e-6, seed=0, n_step=1, gamma=0.9):
        alpha, eps = float(alpha), float(eps)
        if not (0.0 <= alpha < float("inf")) or not (0.0 <= eps < float("inf")):
            raise Exception("Invalid priorities : need finite alpha >= 0 and eps >= 0, got alpha={} eps={}.".format(alpha, eps))
        super().__init__(bg, depth=depth, track=track, ships=ships, n_step=n_step, gamma=gamma)
        cfg = _lib.OfbReplayPrioConfig(alpha=alpha, eps=eps, seed=int(seed) & (2 ** 64 - 1))
        with torch.cuda.device(self.device):
            _lib.check(self._lib.ofb_replay_enable_priorities(self._h, C.byref(cfg)))
        self.alpha, self.eps, self.seed = alpha, eps, int(seed)
        self._n_transitions = self.depth * self.track * len(self.ships)
        self._n_valid = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._sampled = None                             # (frames at the last sample, its ids)

    def sample_prioritized(self, batch_size, beta):
        """Draw ``batch_size`` transitions in proportion to their masses -> ``gather``'s namespace plus ``ids`` (int32 [B],
        for ``update_priorities``) and ``weight`` (float32 [B], the importance weights (mass / min mass) ** -beta <= 1).
        Reads the number of drawable transitions: one host synchronisation.  Raises ``EmptyReplayMemory`` when there is
        none."""
        B, beta = int(batch_size), float(beta)
        if B < 1:
            raise Exception("Invalid batch : {} samples.".format(B))
        if not (0.0 <= beta < float("inf")):
            raise Exception("Invalid beta {} : expected a finite value >= 0.".format(beta))
        ids = torch.empty((B,), dtype=torch.int32, device=self.device)
        weight = torch.empty((B,), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ofb_replay_sample_prioritized(self._h, B, beta, _ptr(ids), _ptr(weight), _ptr(self._n_valid),
                                                           self._stream()))
        self.launch_count += 3
        if int(self._n_valid.item()) < 1:
            raise EmptyReplayMemory("sample on an empty replay memory")
        out = self._gather_ids(ids)
        out.ids, out.weight = ids, weight
        self._sampled = (self.frames, ids)
        return out

    def update_priorities(self, ids, td_act, td_ptr):
        """Set the masses of the transitions ``ids`` (int32 [B] from ``sample_prioritized``) from their TD errors
        ``td_act`` / ``td_ptr`` (float32 [B], ``TrainerB200.td_errors``) and raise the largest mass.  The ids must come
        from a sample taken since the last push; ids other than that sample's own tensor are range-checked, which
        synchronises the host."""
        if self._sampled is None or self._sampled[0] != self.frames:
            raise Exception("Invalid ids : a push happened since the sample they come from.")
        B = ids.numel() if isinstance(ids, torch.Tensor) else 0
        for name, t, dt in (("ids", ids, torch.int32), ("td_act", td_act, torch.float32), ("td_ptr", td_ptr, torch.float32)):
            if not isinstance(t, torch.Tensor) or t.dtype != dt or t.device != self.device or tuple(t.shape) != (B,) or \
                    not t.is_contiguous():
                raise Exception("Invalid {} : expected a contiguous {} tensor of shape ({},) on {}.".format(name, dt, B, self.device))
        if B < 1:
            raise Exception("Invalid ids : no transition.")
        if ids is not self._sampled[1] and (int(ids.min()) < 0 or int(ids.max()) >= self._n_transitions):
            raise Exception("Invalid ids : outside [0, {}).".format(self._n_transitions))
        _lib.check(self._lib.ofb_replay_update_priorities(self._h, _ptr(ids), _ptr(td_act), _ptr(td_ptr), B, self._stream()))
        self.launch_count += 1

    def masses(self):
        """Device copy of the sampling masses, float32 [depth * track * P] indexed by transition id (slot, arena, ship)."""
        out = torch.empty((self._n_transitions,), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ofb_replay_read_priorities(self._h, _ptr(out), None, None, self._stream()))
        return out

    def max_mass(self):
        """Device copy of the largest mass set so far (float32 [1]); new transitions enter with it."""
        out = torch.empty((1,), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ofb_replay_read_priorities(self._h, None, _ptr(out), None, self._stream()))
        return out

    def sample_stats(self):
        """Device copy of (total mass, smallest non-zero mass) of the last ``sample_prioritized`` (float64 [2]), what the
        ranks of a data-parallel replay combine into Schaul's weights over all their memories.  No host synchronisation."""
        out = torch.empty((2,), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.ofb_replay_sample_stats(self._h, _ptr(out), self._stream()))
        self.launch_count += 1
        return out

    def rescale_weights(self, weight, beta, local_stats, global_ratio):
        """In place on ``weight`` (float32 [B] from ``sample_prioritized`` with the same ``beta``): the factor
        ((m_min / M) / g) ** -beta that turns this memory's importance weights into those over the union of the ranks'
        memories (include/ofb_replay.h).  ``local_stats``: ``sample_stats()``; ``global_ratio``: float64 [1], g = the
        minimum over the ranks of m_min / M.  Device only."""
        for name, t, dt, n in (("weight", weight, torch.float32, None), ("local_stats", local_stats, torch.float64, 2),
                               ("global_ratio", global_ratio, torch.float64, 1)):
            if not isinstance(t, torch.Tensor) or t.dtype != dt or t.device != self.device or not t.is_contiguous() or \
                    t.dim() != 1 or (n is not None and t.numel() != n):
                raise Exception("Invalid {} : expected a contiguous 1-d {} tensor on {}.".format(name, dt, self.device))
        _lib.check(self._lib.ofb_replay_rescale_weights(_ptr(weight), weight.numel(), float(beta), _ptr(local_stats),
                                                        _ptr(global_ratio), self._stream()))
        self.launch_count += 1

    def last_total(self):
        """Device copy of the fp64 total mass the last ``sample_prioritized`` drew from (float64 [1])."""
        out = torch.empty((1,), dtype=torch.float64, device=self.device)
        _lib.check(self._lib.ofb_replay_read_priorities(self._h, None, None, _ptr(out), self._stream()))
        return out
