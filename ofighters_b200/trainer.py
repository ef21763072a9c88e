"""B200 counterpart of the reference's ``Trainer`` update path (agents/qlearnIA_V2.py:47-299) and its epsilon
schedules (lib/epsilon.py:18-86) -- SURVEY.md 8(f) rank 1.

    reference                                             here
    ----------------------------------------------------  ---------------------------------------------------
    Trainer(learning_rate, epsilon, batch_size, memory)   TrainerB200(weights=None, learning_rate=..., ...)
    .remember(state, iaction, ipointer, reward, next, d)  .remember(...)   state = (maps_bits [2,5000], vec [8])
    .replay(batch_size) -> History (loss)                 .replay(batch_size) -> History-like (.history["loss"])
    .get_best_action(obs, rand=True)                      .get_best_action(maps_bits, vec, rand=True)
    .decay_epsilon()                                      .decay_epsilon()
    model.fit(x, y, epochs=1, batch_size=B)               .fit(maps_bits, vec, target_act, target_ptr)
    Epsilon_cos(period) / Epsilon_decay()                 epsilon.EpsilonSchedule (closed form in t, evaluated on the device)
    .save(id)  /  load_model(name)                        .save(id) -> .npz of Keras-layout arrays / TrainerB200.load(path)

``predict`` runs on the inference engine (PolicyB200: tcgen05 kernels, BN folded, moving statistics); ``fit`` runs
libofb's training kernels (fp32, BatchNormalization on batch statistics, Keras' Adam) through include/ofb_train.h and
then refreshes the inference engine's weights.  There is no torch / CPU fallback for either.
"""
import ctypes as C
import os
import random
import time
from collections import deque
from types import SimpleNamespace

import torch

from . import _lib
from .epsilon import Epsilon_cos, Epsilon_decay, EpsilonSchedule  # noqa: F401  (re-exported: Trainer(epsilon=Epsilon_cos(...)))
from .policy import WEIGHT_SPEC, PolicyB200, keras_default_weights
from .replay import DeviceReplayMemory, EmptyReplayMemory, PrioritizedReplayMemory


def flatten_weights(weights):
    """Keras-layout dict -> the flat fp32 array of include/ofb_train.h (WEIGHT_SPEC order)."""
    parts = []
    for name, shape in WEIGHT_SPEC:
        if name not in weights:
            raise Exception("missing weight " + name)
        t = torch.as_tensor(weights[name]).detach().to("cpu", torch.float32).contiguous()
        if tuple(t.shape) != tuple(shape):
            raise Exception("weight {} : expected shape {} but got shape {}.".format(name, shape, tuple(t.shape)))
        parts.append(t.reshape(-1))
    return torch.cat(parts).contiguous()


def unflatten_weights(flat):
    out, off = {}, 0
    for name, shape in WEIGHT_SPEC:
        n = 1
        for d in shape:
            n *= d
        out[name] = flat[off:off + n].reshape(shape).clone()
        off += n
    return out


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def blend_weights(weights, target, tau):
    """The target network's soft update theta- <- tau * theta + (1 - tau) * theta-, elementwise in fp32 over Keras-layout
    dicts: tau and 1 - tau are rounded to fp32 once and ``tau * w + (1 - tau) * wt`` is evaluated in that order without
    fma, so tau = 1 returns ``weights``' values exactly."""
    a = torch.tensor(float(tau), dtype=torch.float32)
    b = torch.tensor(1.0 - float(tau), dtype=torch.float32)
    return {k: a * weights[k].to(torch.float32) + b * target[k].to(torch.float32) for k in weights}


class TrainerB200:
    def __init__(self, weights=None, name=None, learning_rate=0.001, epsilon=None, batch_size=30, memory_size=400,
                 device=None, seed=0, max_ships=64, bn_unbiased_moving_var=False, target_update=None, target_tau=1.0,
                 double_dqn=False, reducer=None):
        """Defaults are the reference constructor's (qlearnIA_V2.py:48); the module-level TRAINER is built with
        ``learning_rate=0.0001, epsilon=Epsilon_cos(period=110*400), batch_size=8`` (:304-310).

        Target network (Mnih et al. 2015; the reference has none, so it is off by default): ``target_update=C`` keeps a second
        inference engine, ``target_model``, whose weights start as the initial ones and, after every optimiser step with
        ``steps % C == 0``, become ``tau * theta + (1 - tau) * theta-`` (``target_tau``, 0 < tau <= 1; BN moving statistics
        included).  ``replay`` then bootstraps from the target's predictions on the next observations.  ``double_dqn=True``
        (needs ``target_update``) lets the online network choose the action and the pointer and the target score them
        (``ofb_trainer_td_targets_double``).  With ``target_update=None`` every path launches what it launched before.

        Data-parallel learning (the reference has one trainer on one machine; opt-in): ``reducer`` is an object with
        ``rank``, ``world``, ``all_reduce(tensor, op="sum")`` (in place, in the current stream's order; ops "sum" and "min") and
        ``broadcast(tensor, src=0)`` -- ``sharding.DistReducer`` over ``torch.distributed``.  Every rank then builds its trainer
        with the same arguments; rank 0's initial weights are broadcast, ``fit`` is one Adam step on the union of the ranks'
        batches (``ofb_trainer_fit_shard``: BatchNormalization statistics, losses and gradients summed over the ranks, so the
        replicas stay identical) and ``replay`` with a ``DeviceReplayMemory`` draws ``batch_size`` transitions from each rank's
        own memory.  Both are collective: every rank must call them at the same point."""
        if target_update is not None:
            if isinstance(target_update, bool) or int(target_update) != target_update or int(target_update) < 1:
                raise Exception("Invalid target_update {} : expected an int >= 1 (optimiser steps between refreshes) or None."
                                .format(target_update))
            if not 0.0 < float(target_tau) <= 1.0:
                raise Exception("Invalid target_tau {} : expected 0 < tau <= 1.".format(target_tau))
        elif double_dqn:
            raise Exception("Invalid double_dqn : Double DQN scores the online choice with a target network; "
                            "give target_update too.")
        if not torch.cuda.is_available():
            raise _lib.OfbError("TrainerB200 needs a CUDA device: fit and predict are hand-written sm_100a kernels "
                                "and have no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self._lib = _lib.load()
        self.state_size = 320008
        self.action_size = 2
        self.gamma = 0.9                                 # :51
        self.epsilon = epsilon if epsilon is not None else Epsilon_decay()
        self.learning_rate = learning_rate
        self.memory = deque(maxlen=memory_size)
        self.batch_size = batch_size
        self.name = name
        self.ptr_values = None
        self.act_values = None
        self.launch_count = 0
        weights = weights if weights is not None else keras_default_weights(seed)
        flat = flatten_weights(weights)
        self.reducer = reducer
        self.rank = int(reducer.rank) if reducer is not None else 0
        self.world = int(reducer.world) if reducer is not None else 1
        if reducer is not None:                           # one set of initial weights: rank 0's
            flat_dev = flat.to(self.device)
            reducer.broadcast(flat_dev, src=0)
            flat = flat_dev.cpu()
            weights = unflatten_weights(flat)
        # per-rank stream of the uniform draws of a sharded replay (ranks drawing the same positions would draw the same
        # frame, arena and ship of their own memories)
        self._rng = random.Random("ofighters-dp-replay:%d:%d" % (int(seed), self.rank))
        cfg = _lib.OfbTrainConfig()
        self._lib.ofb_train_default_config(C.byref(cfg))
        cfg.lr = float(learning_rate)
        cfg.max_batch = max(int(batch_size), 1)
        cfg.bn_unbiased_moving_var = 1 if bn_unbiased_moving_var else 0
        h = C.c_void_p()
        _lib.check(self._lib.ofb_trainer_create(C.c_void_p(flat.data_ptr()), flat.numel(), C.byref(cfg),
                                                self.device.index or 0, C.byref(h)))
        self._h = h
        self.max_batch = cfg.max_batch
        self._reduce_error = None
        if reducer is not None:                           # caller-owned exchange buffers, summed by the reducer's callback
            self._xstats = torch.zeros(_lib.TRAIN_STATS_LEN, dtype=torch.float64, device=self.device)
            self._xgrads = torch.zeros(flat.numel(), dtype=torch.float32, device=self.device)
            _lib.check(self._lib.ofb_trainer_set_exchange(h, _ptr(self._xstats), _ptr(self._xgrads)))
            self._reduce_cb = _lib.REDUCE_FN(self._on_reduce)      # kept alive as long as the handle
            _lib.check(self._lib.ofb_trainer_set_reducer(h, self._reduce_cb, None))
        self.model = PolicyB200(weights, device=self.device, max_ships=max_ships)   # the predict() side
        self._loss = torch.zeros(3, dtype=torch.float32, device=self.device)
        self.target_update = None if target_update is None else int(target_update)
        self.target_tau = float(target_tau)
        self.double_dqn = bool(double_dqn)
        self.target_model = None
        self.target_updates = 0
        if self.target_update is not None:
            self._target_w = unflatten_weights(flat)      # fp32 host copy of theta-, Keras layouts
            self.target_model = PolicyB200(self._target_w, device=self.device, max_ships=max_ships)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                self._lib.ofb_trainer_destroy(h)
            except Exception:
                pass
            self._h = None

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _exchange_slice(self, stage):
        """The slice of the exchange buffers a reduce stage sums (include/ofb_train.h)."""
        if _lib.STAGE_FWD_BN <= stage < _lib.STAGE_FWD_BN + _lib.TRAIN_N_BN:
            o = _lib.TRAIN_STATS_FWD + 16 * (stage - _lib.STAGE_FWD_BN)
            return self._xstats[o:o + 16]
        if stage == _lib.STAGE_LOSS:
            return self._xstats[_lib.TRAIN_STATS_LOSS:_lib.TRAIN_STATS_LOSS + 2]
        if _lib.STAGE_BWD_BN <= stage < _lib.STAGE_BWD_BN + _lib.TRAIN_N_BN:
            o = _lib.TRAIN_STATS_BWD + 16 * (stage - _lib.STAGE_BWD_BN)
            return self._xstats[o:o + 16]
        if stage == _lib.STAGE_GRADS:
            return self._xgrads
        raise Exception("unknown reduce stage {}".format(stage))

    def _on_reduce(self, ctx, stage, stream):
        """The C hook of a sharded fit, called on the thread (and current stream) of ``fit``.  An exception must not
        unwind through C: it is kept for ``fit`` to raise and the fit is aborted with a non-zero return."""
        try:
            self.reducer.all_reduce(self._exchange_slice(int(stage)))
            return 0
        except BaseException as e:                       # noqa: B902 -- KeyboardInterrupt included: C cannot unwind it
            self._reduce_error = e
            return 1

    def _all_ranks(self, flag):
        """True when ``flag`` holds on every rank (an all-reduce MIN; one host synchronisation)."""
        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=self.device)
        self.reducer.all_reduce(t, op="min")
        return bool(int(t.item()))

    # ------------------------------------------------------------------ weights
    def get_weights(self):
        flat = torch.empty(len_flat(), dtype=torch.float32)
        _lib.check(self._lib.ofb_trainer_get_weights(self._h, C.c_void_p(flat.data_ptr()), self._stream()))
        return unflatten_weights(flat)

    def get_target_weights(self):
        """The target network's weights theta- (Keras-layout fp32 host copies); needs ``target_update``."""
        if self.target_model is None:
            raise Exception("no target network : the trainer was built with target_update=None")
        return {k: v.clone() for k, v in self._target_w.items()}

    def get_grads(self):
        flat = torch.empty(len_flat(), dtype=torch.float32)
        _lib.check(self._lib.ofb_trainer_get_grads(self._h, C.c_void_p(flat.data_ptr()), self._stream()))
        return unflatten_weights(flat)

    @property
    def steps(self):
        return int(self._lib.ofb_trainer_steps(self._h))

    def sync_model(self):
        """Hand the trained weights to the inference engine (BN folded from the moving statistics)."""
        self.model.load_weights(self.get_weights())

    def save(self, id=None, overwrite=False, folder="networks"):
        """``Trainer.save`` (:289-298): same naming -- ``keras-model[-<name> | -<timestamp>][-<id>]`` under ``folder`` -- but
        the file is an ``.npz`` of the Keras-layout arrays of WEIGHT_SPEC (what ``PolicyB200.load_weights`` / ``load`` take);
        Keras' HDF5 container is out of scope.  Returns the path."""
        import numpy as np
        name = "keras-model-" + (self.name if self.name else time.strftime("%Y-%m-%d_%H-%M-%S"))
        if id:
            name += "-" + str(id)
        os.makedirs(folder, exist_ok=True)
        path = os.path.join(folder, name + ".npz")
        if os.path.exists(path) and not overwrite:
            raise Exception("{} exists and overwrite is False.".format(path))
        np.savez(path, **{k.replace("/", "."): v.numpy() for k, v in self.get_weights().items()})
        return path

    @staticmethod
    def load_weights_file(path):
        """Inverse of ``save``: the Keras-layout dict (``load_model`` of :70 for this format)."""
        import numpy as np
        with np.load(path) as f:
            return {k.replace(".", "/"): torch.from_numpy(f[k]) for k in f.files}

    # ------------------------------------------------------------------ fit / predict
    def _check_batch(self, maps_bits, vec):
        B = maps_bits.shape[0]
        if maps_bits.dtype != torch.int32 or tuple(maps_bits.shape) != (B, 2, 5000) or not maps_bits.is_contiguous() \
                or maps_bits.device != self.device:
            raise Exception("Invalid maps : expected contiguous int32 [B, 2, 5000] bit maps on {}.".format(self.device))
        if B < 1 or B > self.max_batch:
            raise Exception("Invalid batch : {} samples but the trainer was sized for {}.".format(B, self.max_batch))
        vec = vec.to(device=self.device, dtype=torch.float32).contiguous().reshape(-1, 8)
        if vec.shape[0] != B:
            raise Exception("Invalid vector input : expected shape {} but got shape {}.".format((B, 8), tuple(vec.shape)))
        return B, vec

    def fit(self, maps_bits, vec, target_act, target_ptr, sync_model=True, sample_weight=None, batch_global=None):
        """``model.fit(x=[img, vec], y=[act, ptr], epochs=1, batch_size=B)`` (:286): one Adam step.  Returns the loss
        tensor (total, mse(output1), mse(output2)) of the batch before the update (device, float32 [3]).
        ``sample_weight``: float [B] of weights >= 0 -- ``model.fit(..., sample_weight=w)``: each head's loss becomes
        (1/B) sum_b w_b mse_b, and the returned losses are the weighted ones (include/ofb_train.h).
        With a ``reducer`` the step is on the union of every rank's batch, whose size an all-reduce of the local B gives
        (``batch_global`` overrides it), and the losses are the global batch's."""
        B, vec = self._check_batch(maps_bits, vec)
        target_act = target_act.to(device=self.device, dtype=torch.float32).contiguous()
        target_ptr = target_ptr.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(target_act.shape) != (B, 2) or target_ptr.numel() != B * 160000:
            raise Exception("Invalid targets : expected shapes {} and {}.".format((B, 2), (B, 400, 400, 1)))
        if sample_weight is not None:
            sample_weight = torch.as_tensor(sample_weight).to(device=self.device, dtype=torch.float32).contiguous()
            if tuple(sample_weight.shape) != (B,):
                raise Exception("Invalid sample_weight : expected shape {} but got shape {}.".format((B,), tuple(sample_weight.shape)))
        if self.reducer is not None or batch_global is not None:
            if batch_global is None:                      # ranks cannot disagree on the global batch: it is their sum
                n = torch.tensor([B], dtype=torch.int32, device=self.device)
                self.reducer.all_reduce(n)
                batch_global = int(n.item())
            self._reduce_error = None
            rc = self._lib.ofb_trainer_fit_shard(self._h, _ptr(maps_bits), _ptr(vec), _ptr(target_act), _ptr(target_ptr),
                                                 _ptr(sample_weight), B, int(batch_global), _ptr(self._loss), self._stream())
            if rc < 0 and self._reduce_error is not None:
                err, self._reduce_error = self._reduce_error, None
                raise _lib.OfbError("libofb error %d: %s" % (rc, self._lib.ofb_last_error().decode())) from err
            _lib.check(rc)
        elif sample_weight is None:
            _lib.check(self._lib.ofb_trainer_fit(self._h, _ptr(maps_bits), _ptr(vec), _ptr(target_act), _ptr(target_ptr), B,
                                                 _ptr(self._loss), self._stream()))
        else:
            _lib.check(self._lib.ofb_trainer_fit_weighted(self._h, _ptr(maps_bits), _ptr(vec), _ptr(target_act), _ptr(target_ptr),
                                                          _ptr(sample_weight), B, _ptr(self._loss), self._stream()))
        self.launch_count += self.KERNELS_PER_FIT
        loss = self._loss.clone()
        refresh = self.target_update is not None and self.steps % self.target_update == 0
        if sync_model or refresh:
            w = self.get_weights()
            if sync_model:
                self.model.load_weights(w)
            if refresh:                                   # the same host weights feed the target's blend
                self._target_w = blend_weights(w, self._target_w, self.target_tau)
                self.target_model.load_weights(self._target_w)
                self.target_updates += 1
        return loss

    KERNELS_PER_FIT = 96          # forward 33 + backward 62 + Adam (memsets not counted)

    def forward_train(self, maps_bits, vec):
        """Training-mode predictions (batch statistics) -- what ``fit`` differentiates.  -> act [B,2], ptr [B,400,400]."""
        B, vec = self._check_batch(maps_bits, vec)
        act = torch.empty((B, 2), dtype=torch.float32, device=self.device)
        ptr = torch.empty((B, 400, 400), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ofb_trainer_forward(self._h, _ptr(maps_bits), _ptr(vec), B, _ptr(act), _ptr(ptr), self._stream()))
        return act, ptr

    def predict(self, maps_bits, vec):
        """``model.predict`` on bit maps: (act [B,2], ptr [B,400,400]) from the inference engine."""
        r = self.model.forward(maps_bits, vec, 1, want_ptr=True)
        return r["act"], r["ptr"]

    # ------------------------------------------------------------------ reference surface
    def decay_epsilon(self):
        self.epsilon.next()

    def random_play(self):
        """qlearnIA_V2.py:317-321"""
        iaction = random.randint(0, self.action_size - 1)
        return [iaction, (random.randint(0, 400 - 1), random.randint(0, 400 - 1))]

    def get_best_action(self, maps_bits, vec, rand=True):
        """:199-235 for one observation: maps_bits [2,5000] (or [1,2,5000]), vec [8] -> [iaction, (x, y)]."""
        if rand and random.random() <= self.epsilon.get():
            return self.random_play()
        r = self.model.forward(maps_bits.reshape(1, 2, 5000).contiguous(), vec.reshape(1, 8), 1, want_ptr=True)
        self.act_values = r["act"][0]
        self.ptr_values = r["ptr"][0]
        xy = r["xy"][0].tolist()
        return [int(r["iaction"][0]), (int(xy[0]), int(xy[1]))]

    def remember(self, state, iaction, ipointer, reward, next_state, done):
        """:237-238.  ``state`` / ``next_state`` = (maps_bits int32 [2,5000], vec float32 [8]) device tensors."""
        self.memory.append([state, iaction, ipointer, reward, next_state, done])

    def td_errors(self, act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done, discount=None):
        """Signed TD errors target - prediction at the entries ``replay``'s targets overwrite, with the targets' own fp32
        arithmetic: (td_act, td_ptr) float32 [B] on the device.  Inputs as ``ofb_trainer_td_targets`` takes them;
        ``discount`` (float32 [B], an n-step memory's gamma^k) replaces ``gamma`` when it is given."""
        B = act_obs.shape[0]
        td_act = torch.empty((B,), dtype=torch.float32, device=self.device)
        td_ptr = torch.empty((B,), dtype=torch.float32, device=self.device)
        args = [_ptr(t) for t in (act_obs, ptr_obs, act_next, ptr_next, iaction, pointer, reward, done)]
        if discount is None:
            _lib.check(self._lib.ofb_trainer_td_errors(*args, float(self.gamma), B, _ptr(td_act), _ptr(td_ptr), self._stream()))
        else:
            _lib.check(self._lib.ofb_trainer_td_errors_discounted(*args, _ptr(discount), B, _ptr(td_act), _ptr(td_ptr),
                                                                  self._stream()))
        self.launch_count += 1
        return td_act, td_ptr

    def _td_targets(self, act_o, ptr_o, act_n, ptr_n, iaction, pointer, reward, done, discount, B):
        """``ofb_trainer_td_targets`` in place on (act_o, ptr_o); with a ``discount`` [B] its discounted form."""
        args = [_ptr(t) for t in (act_o, ptr_o, act_n, ptr_n, iaction, pointer, reward, done)]
        if discount is None:
            _lib.check(self._lib.ofb_trainer_td_targets(*args, float(self.gamma), B, _ptr(act_o), _ptr(ptr_o), self._stream()))
        else:
            _lib.check(self._lib.ofb_trainer_td_targets_discounted(*args, _ptr(discount), B, _ptr(act_o), _ptr(ptr_o),
                                                                   self._stream()))
        self.launch_count += 1

    def _predict_next(self, maps_n, vec_n):
        """Predictions on the next observations for the max-bootstrap: the target network's when there is one."""
        if self.target_model is None:
            return self.predict(maps_n, vec_n)
        r = self.target_model.forward(maps_n, vec_n, 1, want_ptr=True)
        return r["act"], r["ptr"]

    def _td_targets_double(self, act_o, ptr_o, maps_n, vec_n, iaction, pointer, reward, done, discount, B, want_td=False):
        """Double DQN targets in place on (act_o, ptr_o): the online network selects on the next observations, the target
        network evaluates.  -> (td_act, td_ptr) float32 [B] of the same pass when ``want_td``, else (None, None)."""
        act_n, ptr_n = self.predict(maps_n, vec_n)
        tg = self.target_model.forward(maps_n, vec_n, 1, want_ptr=True)
        td_act = td_ptr = None
        if want_td:
            td_act = torch.empty((B,), dtype=torch.float32, device=self.device)
            td_ptr = torch.empty((B,), dtype=torch.float32, device=self.device)
        _lib.check(self._lib.ofb_trainer_td_targets_double(
            *[_ptr(t) for t in (act_o, ptr_o, act_n, ptr_n, tg["act"], tg["ptr"], iaction, pointer, reward, done)],
            float(self.gamma), _ptr(discount), B, _ptr(act_o), _ptr(ptr_o), _ptr(td_act), _ptr(td_ptr), self._stream()))
        self.launch_count += 1
        return td_act, td_ptr

    def _check_memory(self, memory):
        if memory.device != self.device:
            raise Exception("Invalid memory : it lives on {} but the trainer on {}.".format(memory.device, self.device))
        if memory.n_step > 1 and float(memory.gamma) != float(self.gamma):
            raise Exception("Invalid memory : its {}-step returns are discounted by gamma = {} but the trainer's gamma is {}."
                            .format(memory.n_step, memory.gamma, self.gamma))

    def replay(self, batch_size, memory=None, beta=1.0):
        """:240-287.  Targets from predictions on obs and next_obs; like the reference, the fitted INPUTS are the
        next observations (``inputs1[i] = img_input`` is evaluated after img_input was rebuilt from next_obs, :281-282).
        ``memory``: a ``replay.DeviceReplayMemory`` to draw the minibatch from instead of ``self.memory`` (same
        ``random.sample`` draw over its transitions in age order).  With a ``replay.PrioritizedReplayMemory`` the minibatch
        is drawn in proportion to the priorities, the TD errors of the predictions set the drawn transitions' new
        priorities, and the fit weighs each sample by its importance weight, annealed by ``beta`` (ignored otherwise); the
        History then also reports ``td_error``, the batch mean of |td_act| + |td_ptr|.  With an n-step memory
        (``memory.n_step`` > 1, whose ``gamma`` must be the trainer's) the targets are R + gamma^k max Q(s_{t+k}) of each
        sample's window (``ofb_trainer_td_targets_discounted``).  With a target network (``target_update``) the max-bootstrap
        reads the target's predictions on the next observations; with ``double_dqn`` the online network selects and the
        target evaluates (``ofb_trainer_td_targets_double``, which on the prioritized path also gives the TD errors).
        With a ``reducer`` see ``_replay_shard``: a collective call that returns None when some rank had nothing to draw."""
        if self.reducer is not None:
            return self._replay_shard(batch_size, memory, beta)
        if isinstance(memory, PrioritizedReplayMemory):
            return self._replay_prioritized(batch_size, memory, beta)
        dev = self.device
        if memory is None:
            batch_size = min(batch_size, len(self.memory))
            if batch_size < 1:
                raise Exception("replay on an empty memory")
            minibatch = random.sample(self.memory, batch_size)
            maps_o = torch.stack([m[0][0] for m in minibatch]).to(dev).contiguous()
            vec_o = torch.stack([m[0][1] for m in minibatch]).to(dev).contiguous()
            maps_n = torch.stack([m[4][0] for m in minibatch]).to(dev).contiguous()
            vec_n = torch.stack([m[4][1] for m in minibatch]).to(dev).contiguous()
            iaction = torch.tensor([int(m[1]) for m in minibatch], dtype=torch.int32, device=dev)
            pointer = torch.tensor([[int(m[2][0]), int(m[2][1])] for m in minibatch], dtype=torch.int32, device=dev)
            reward = torch.tensor([float(m[3]) for m in minibatch], dtype=torch.float32, device=dev)
            done = torch.tensor([1 if m[5] else 0 for m in minibatch], dtype=torch.uint8, device=dev)
            discount = None
        else:
            self._check_memory(memory)
            batch_size = min(batch_size, len(memory))
            if batch_size < 1:
                raise Exception("replay on an empty memory")
            if batch_size > self.max_batch:
                raise Exception("Invalid batch : {} samples but the trainer was sized for {}.".format(batch_size, self.max_batch))
            mb = memory.sample(batch_size)
            maps_o, vec_o, maps_n, vec_n = mb.maps_obs, mb.vec_obs, mb.maps_next, mb.vec_next
            iaction, pointer, reward, done = mb.iaction, mb.pointer, mb.reward, mb.done
            discount = mb.discount if memory.n_step > 1 else None
        act_o, ptr_o = self.predict(maps_o, vec_o)
        if self.double_dqn:
            self._td_targets_double(act_o, ptr_o, maps_n, vec_n, iaction, pointer, reward, done, discount, batch_size)
        else:
            act_n, ptr_n = self._predict_next(maps_n, vec_n)
            self._td_targets(act_o, ptr_o, act_n, ptr_n, iaction, pointer, reward, done, discount, batch_size)
        loss = self.fit(maps_n, vec_n, act_o, ptr_o)
        host = loss.cpu().tolist()
        return SimpleNamespace(history={"loss": [host[0]], "output1_loss": [host[1]], "output2_loss": [host[2]]})

    def _replay_prioritized(self, batch_size, memory, beta):
        self._check_memory(memory)
        batch_size = int(batch_size)
        if batch_size < 1 or batch_size > self.max_batch:
            raise Exception("Invalid batch : {} samples but the trainer was sized for {}.".format(batch_size, self.max_batch))
        mb = memory.sample_prioritized(batch_size, beta)
        act_o, ptr_o = self.predict(mb.maps_obs, mb.vec_obs)
        discount = mb.discount if memory.n_step > 1 else None
        if self.double_dqn:
            td_act, td_ptr = self._td_targets_double(act_o, ptr_o, mb.maps_next, mb.vec_next, mb.iaction, mb.pointer, mb.reward,
                                                     mb.done, discount, batch_size, want_td=True)
            memory.update_priorities(mb.ids, td_act, td_ptr)
        else:
            act_n, ptr_n = self._predict_next(mb.maps_next, mb.vec_next)
            fields = (act_o, ptr_o, act_n, ptr_n, mb.iaction, mb.pointer, mb.reward, mb.done)
            td_act, td_ptr = self.td_errors(*fields, discount=discount)
            memory.update_priorities(mb.ids, td_act, td_ptr)
            self._td_targets(*fields, discount, batch_size)
        loss = self.fit(mb.maps_next, mb.vec_next, act_o, ptr_o, sample_weight=mb.weight)
        host = torch.cat([loss, (td_act.abs() + td_ptr.abs()).mean().reshape(1)]).cpu().tolist()
        return SimpleNamespace(history={"loss": [host[0]], "output1_loss": [host[1]], "output2_loss": [host[2]],
                                        "td_error": [host[3]]})


    def _replay_shard(self, batch_size, memory, beta):
        """``replay`` of a data-parallel trainer, collective over the ranks.  Each rank draws ``batch_size`` transitions
        (fewer if its memory holds fewer) from its own ``DeviceReplayMemory``, so the global batch is the sum over the ranks
        (the DDP convention); the targets come from the rank's replica and the fit is ``ofb_trainer_fit_shard``.
          * Whether to replay is decided together: an all-reduce MIN of "this rank can draw"; when some rank cannot, every
            rank skips (returns None), so all ranks make the same collective calls.
          * Uniform draws use the rank's own ``random.Random``, seeded from (seed, rank).
          * Prioritized draws are stratified by shard: rank r draws in proportion to its masses, P(i) = m_i / (W M_r), and
            the importance weights are rescaled to Schaul's weights over the union of the memories, with g = the minimum
            over ranks of m_min,r / M_r from one fp64 all-reduce MIN on the device (``ofb_replay_rescale_weights``).
            Priorities are updated locally.
        n-step returns, the target network and Double DQN are per-rank and need nothing more."""
        if not isinstance(memory, DeviceReplayMemory):
            raise Exception("Invalid memory : a data-parallel replay draws from a replay.DeviceReplayMemory on every rank.")
        self._check_memory(memory)
        B = int(batch_size)
        if B < 1 or B > self.max_batch:
            raise Exception("Invalid batch : {} samples but the trainer was sized for {}.".format(B, self.max_batch))
        prioritized = isinstance(memory, PrioritizedReplayMemory)
        if prioritized:
            try:
                mb = memory.sample_prioritized(B, beta)
            except EmptyReplayMemory:
                mb = None
            have = mb is not None
        else:
            n = len(memory)
            have = n > 0
        if not self._all_ranks(have):
            return None
        if prioritized:
            stats = memory.sample_stats()
            ratio = (stats[1:2] / stats[0:1]).contiguous()
            self.reducer.all_reduce(ratio, op="min")
            memory.rescale_weights(mb.weight, beta, stats, ratio)
            weight = mb.weight
        else:
            B = min(B, n)
            mb = memory.sample(B, rng=self._rng)
            weight = None
        discount = mb.discount if memory.n_step > 1 else None
        act_o, ptr_o = self.predict(mb.maps_obs, mb.vec_obs)
        td_act = td_ptr = None
        if self.double_dqn:
            td_act, td_ptr = self._td_targets_double(act_o, ptr_o, mb.maps_next, mb.vec_next, mb.iaction, mb.pointer, mb.reward,
                                                     mb.done, discount, B, want_td=prioritized)
        else:
            act_n, ptr_n = self._predict_next(mb.maps_next, mb.vec_next)
            fields = (act_o, ptr_o, act_n, ptr_n, mb.iaction, mb.pointer, mb.reward, mb.done)
            if prioritized:
                td_act, td_ptr = self.td_errors(*fields, discount=discount)
            self._td_targets(*fields, discount, B)
        if prioritized:
            memory.update_priorities(mb.ids, td_act, td_ptr)
        loss = self.fit(mb.maps_next, mb.vec_next, act_o, ptr_o, sample_weight=weight)
        parts = [loss] if not prioritized else [loss, (td_act.abs() + td_ptr.abs()).mean().reshape(1)]
        host = torch.cat(parts).cpu().tolist()
        hist = {"loss": [host[0]], "output1_loss": [host[1]], "output2_loss": [host[2]], "batch": [B]}
        if prioritized:
            hist["td_error"] = [host[3]]
        return SimpleNamespace(history=hist)


def len_flat():
    n = 0
    for _, shape in WEIGHT_SPEC:
        k = 1
        for d in shape:
            k *= d
        n += k
    return n


class QLearner:
    """Batched counterpart of ``QlearnIA.play``'s learning bookkeeping (agents/qlearnIA_V2.py:372-417) on top of one shared
    ``TrainerB200`` ("All bots share the same trainer", :362).  The policy ship of each of the first ``track`` arenas is a
    QlearnIA bot with ids 1..track (bot id 1 = arena 0): every frame it remembers (previous_obs, previous_action,
    previous_pointer, obs.reward, obs, obs.done) until it has seen its own death (:376-392); ANY bot replays when it dies
    (:378-385); bot id 1 alone advances epsilon -- once per decision it takes, i.e. not after its death and not during the
    collecting phase (:394-401) -- replays every ``replay_every`` total steps (:403-405) and snapshots the model every
    ``snapshot`` episodes (:416-417).  During the first ``collecting_steps`` total steps every policy ship plays
    ``random_play()`` (:394-396).  Observations stay on the device: obs = (maps_bits [2,5000], head [8]).

    ``actor``: the inference engine that drives the arenas (default: the trainer's own ``model``).  With a separate actor
    (multi-GPU: every rank's actor is refreshed from the broadcast weights at common points) the trainer's own small
    ``model`` keeps serving ``replay``'s predictions with the latest weights."""

    def __init__(self, trainer, track=8, replay_every=50, collecting_steps=20, snapshot=50, actor=None, snapshot_folder="networks"):
        self.trainer = trainer
        self.actor = actor if actor is not None else trainer.model
        self.track = int(track)
        self.replay_every = int(replay_every)
        self.collecting_steps = int(collecting_steps)
        self.snapshot = int(snapshot)
        self.snapshot_folder = snapshot_folder
        self.total_steps = 0          # Agent.total_steps of bot 1 (never reset, agents/agent.py:66-68)
        self.steps = 0                # Agent.steps: frames since the last reset
        self.episode = 0
        self.losses = []
        self.epsilons = []
        self.saved = []
        self.previous = [None] * self.track
        self.done = [False] * self.track

    @property
    def collecting(self):
        """True while the NEXT decision belongs to the random collecting phase (``total_steps < collecting_steps`` is
        evaluated after Agent.step incremented the counter)."""
        return self.total_steps + 1 < self.collecting_steps

    def reset(self):
        """``QlearnIA.reset`` (:359-369) + ``Agent.reset`` (agents/agent.py:59-64): log epsilon, forget the previous action."""
        self.episode += 1
        self.steps = 0
        self.epsilons.append(self.trainer.epsilon.get())
        self.previous = [None] * self.track
        self.done = [False] * self.track

    def act(self, bg, maps_bits):
        """One frame of every QlearnIA ship: choose (collecting phase / eps-greedy with the trainer's schedule on the
        device), write the action rows, then the bookkeeping of ``observe`` with the actions that are PLAYED.
        -> (iaction, xy, replayed)"""
        collecting = self.collecting
        iact, xy = self.actor.act(bg, maps_bits, epsilon=self.trainer.epsilon, collecting=collecting)
        return iact, xy, self.observe(bg, maps_bits, iact, xy)

    def observe(self, bg, maps_bits, iaction, xy, ship=None):
        """Call once per frame right after the policy ships' PLAYED actions (iaction [A*P], xy [A*P,2]) were written for
        the current observation.  Returns True when the trainer's weights changed (a replay ran)."""
        if ship is None:
            ship = int(bg._policy_ship_idx[0]) if getattr(bg, "_policy_ship_idx", None) is not None else 0
        K = min(self.track, bg.n_arenas)
        P = iaction.numel() // bg.n_arenas
        heads = bg.obs_vec[:K, ship, :]
        alive = bg.state(("ship_alive",))["ship_alive"][:K, ship].tolist()
        rewards = heads[:, 0].tolist()
        ia = iaction.reshape(bg.n_arenas, P)[:K, 0].tolist()
        pt = xy.reshape(bg.n_arenas, P, 2)[:K, 0].tolist()
        self.total_steps += 1
        self.steps += 1
        collecting = self.total_steps < self.collecting_steps
        replayed = False
        for k in range(K):
            if self.done[k]:                              # `if self.done: return None` (:375)
                continue
            obs = (maps_bits[k].clone(), heads[k].clone())
            done = not alive[k]
            if done:                                      # every bot replays on its own death (:376-385)
                replayed |= self._replay()
                self.done[k] = True
            if self.previous[k] is not None:
                po, pa, pp = self.previous[k]
                self.trainer.remember(po, pa, pp, rewards[k], obs, done)
            self.previous[k] = (obs, int(ia[k]), (int(pt[k][0]), int(pt[k][1])))
            if k == 0:                                    # "All bots share the same trainer so we only save it once"
                if not collecting:
                    self.trainer.decay_epsilon()          # (:398-401)
                if self.total_steps % self.replay_every == 0:
                    replayed |= self._replay()            # (:403-405)
                if self.snapshot > 0 and self.episode > 0 and self.episode % self.snapshot == 0 and self.steps < 2:
                    self.saved.append(self.trainer.save(id="iteration-%s" % self.episode, overwrite=True,
                                                        folder=self.snapshot_folder))     # (:416-417)
        return replayed

    def _replay(self):
        if len(self.trainer.memory) == 0:
            return False
        h = self.trainer.replay(self.trainer.batch_size)
        self.losses.append(h.history["loss"][0])
        return True


class BatchedQLearner:
    """``QLearner``'s loop for every arena a ``replay.DeviceReplayMemory`` tracks: the policy ships of the whole batch feed one
    shared ``TrainerB200``.  Each frame ``act`` chooses the actions (the collecting phase's ``random_play()`` for the first
    ``collecting_steps`` frames, then eps-greedy with the trainer's schedule, on the device), pushes the snapshot and the
    PLAYED actions into the memory, advances epsilon once outside the collecting phase, replays ``trainer.batch_size``
    transitions every ``replay_every`` frames once the memory holds one, and saves a snapshot of the model on the first frame
    of every ``snapshot``-th episode.  The caller steps the frame and calls ``reset`` at every restart, as with ``QLearner``.

    Departures from ``QlearnIA.play`` (agents/qlearnIA_V2.py:372-417), which ``QLearner`` follows for a few tracked arenas:
      * no replay at each death: at this scale that would be thousands of fits per frame; replays come every
        ``replay_every`` frames only;
      * the memory is bounded in frames (the last ``depth - 1``), not in transitions (``memory_size``);
      * epsilon advances once per frame, not once per decision of bot 1 (which stops at its death);
      * no host synchronisation on frames without a replay.

    ``actor``: the inference engine that drives the arenas (default: the trainer's own ``model``, which every fit refreshes).

    With a ``replay.PrioritizedReplayMemory`` each replay is prioritized, with the importance-sampling exponent annealed
    linearly from ``beta0`` to 1 over ``beta_frames`` frames: beta = min(1, beta0 + (1 - beta0) * total_steps / beta_frames)
    (``betas`` logs the value of every replay).  With a uniform memory ``beta0`` and ``beta_frames`` play no part.

    Data-parallel (a trainer built with a ``reducer``; every rank runs its own learner on its own shard of the arenas,
    ``sharding.make_sharded_battleground``): at a replay frame every rank calls the collective ``trainer.replay``, which
    skips on every rank when some rank holds no transition yet, and fits one global batch of ``world * batch_size``
    samples.  Snapshots are saved by rank 0 only."""

    def __init__(self, trainer, memory, replay_every=50, collecting_steps=20, snapshot=50, actor=None, snapshot_folder="networks",
                 beta0=0.4, beta_frames=100_000):
        if memory.device != trainer.device:
            raise Exception("Invalid memory : it lives on {} but the trainer on {}.".format(memory.device, trainer.device))
        self.trainer = trainer
        self.memory = memory
        self.actor = actor if actor is not None else trainer.model
        self.replay_every = int(replay_every)
        self.collecting_steps = int(collecting_steps)
        self.snapshot = int(snapshot)
        self.snapshot_folder = snapshot_folder
        self.total_steps = 0
        self.steps = 0
        self.episode = 0
        self.losses = []
        self.epsilons = []
        self.saved = []
        self.prioritized = isinstance(memory, PrioritizedReplayMemory)
        self.beta0, self.beta_frames = float(beta0), int(beta_frames)
        if self.prioritized and (not 0.0 <= self.beta0 <= 1.0 or self.beta_frames < 1):
            raise Exception("Invalid beta schedule : need 0 <= beta0 <= 1 and beta_frames >= 1.")
        self.betas = []

    @property
    def beta(self):
        """The importance-sampling exponent of a replay at this frame (prioritized memory)."""
        return min(1.0, self.beta0 + (1.0 - self.beta0) * self.total_steps / self.beta_frames)

    @property
    def collecting(self):
        """True while the NEXT frame belongs to the random collecting phase (as ``QLearner.collecting``)."""
        return self.total_steps + 1 < self.collecting_steps

    def reset(self):
        """Episode bookkeeping at a restart: log epsilon, count the episode."""
        self.episode += 1
        self.steps = 0
        self.epsilons.append(self.trainer.epsilon.get())

    def act(self, bg, maps_bits):
        """One frame of every policy ship: choose and write the action rows, remember, learn.  -> (iaction, xy, replayed)"""
        if bg is not self.memory.bg:
            raise Exception("Invalid battleground : the memory remembers another battleground's arenas.")
        collecting = self.collecting
        iact, xy = self.actor.act(bg, maps_bits, epsilon=self.trainer.epsilon, collecting=collecting)
        self.memory.push(iact, xy)
        self.total_steps += 1
        self.steps += 1
        if not collecting:
            self.trainer.decay_epsilon()
        replayed = False
        if self.total_steps % self.replay_every == 0 and self.trainer.reducer is not None:
            h = self.trainer.replay(self.trainer.batch_size, memory=self.memory, beta=self.beta)   # collective
            if h is not None:
                self.losses.append(h.history["loss"][0])
                if self.prioritized:
                    self.betas.append(self.beta)
                replayed = True
        elif self.total_steps % self.replay_every == 0 and self.prioritized:
            try:                                          # the sample reads whether there is a transition to draw
                h = self.trainer.replay(self.trainer.batch_size, memory=self.memory, beta=self.beta)
            except EmptyReplayMemory:
                h = None
            if h is not None:
                self.losses.append(h.history["loss"][0])
                self.betas.append(self.beta)
                replayed = True
        elif self.total_steps % self.replay_every == 0 and len(self.memory) > 0:
            h = self.trainer.replay(self.trainer.batch_size, memory=self.memory)
            self.losses.append(h.history["loss"][0])
            replayed = True
        if self.snapshot > 0 and self.episode > 0 and self.episode % self.snapshot == 0 and self.steps < 2 and self.trainer.rank == 0:
            self.saved.append(self.trainer.save(id="iteration-%s" % self.episode, overwrite=True, folder=self.snapshot_folder))
        return iact, xy, replayed
