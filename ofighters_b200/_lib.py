"""ctypes binding of libofb.so (include/ofb.h).  No torch types cross this boundary: tensors
are passed as raw device pointers, streams as ``cudaStream_t`` integers.

The library is built in-tree by ``ofighters_b200.build``; if it is missing the import of the
product path fails loudly -- there is no CPU fallback.
"""
import ctypes as C
import os

from . import build as _build

OFB_MAP_BITS, OFB_MAP_BF16, OFB_MAP_U8 = 0, 1, 2
BOT_KINDS = {"idle": 0, "random": 1, "turret": 2, "runner": 3, "thrust": 4, "shoot": 5, "stress": 6,
             "external": 255}


class OfbConfig(C.Structure):
    _fields_ = [("n_ships", C.c_int32), ("laser_cap", C.c_int32), ("width", C.c_int32), ("height", C.c_int32),
                ("max_time", C.c_int32), ("reward_kill", C.c_int32), ("reward_death", C.c_int32),
                ("reward_aim", C.c_int32), ("reward_trajectory", C.c_int32), ("reserved", C.c_int32 * 7)]


STATE_VIEW_FIELDS = ["time", "n_lasers", "kills", "deaths", "shots", "overflow", "episode", "near_ties",
                     "ship_x", "ship_y", "ship_px", "ship_py", "ship_hull", "ship_reward", "ship_score",
                     "ship_steps", "ship_alive", "laser_x", "laser_y", "laser_dx", "laser_dy",
                     "laser_owner", "laser_destroyed"]


class OfbStateView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in STATE_VIEW_FIELDS]


class OfbConvWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("kernel", "bias", "gamma", "beta", "mean", "var")]


class OfbDenseWeights(C.Structure):
    _fields_ = [("kernel", C.c_void_p), ("bias", C.c_void_p)]


class OfbPolicyWeights(C.Structure):
    _fields_ = [("conv", OfbConvWeights * 4), ("dense1", OfbDenseWeights), ("dense2", OfbDenseWeights),
                ("output1", OfbDenseWeights), ("updense1", OfbDenseWeights), ("upconv", OfbConvWeights * 4)]


class OfbTrainConfig(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float),
                ("bn_momentum", C.c_float), ("bn_eps", C.c_float), ("bn_unbiased_moving_var", C.c_int32),
                ("max_batch", C.c_int32), ("reserved", C.c_int32 * 8)]


class OfbReplayPrioConfig(C.Structure):
    _fields_ = [("alpha", C.c_float), ("eps", C.c_float), ("seed", C.c_uint64), ("reserved", C.c_int32 * 8)]


class OfbEpsSchedule(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("start", C.c_double), ("period", C.c_double),
                ("decay", C.c_double), ("floor", C.c_double)]


EPS_CONST, EPS_COSINE, EPS_DECAY = 0, 1, 2
ENGINE_TENSOR, ENGINE_CUDA_CORE = 0, 1
POLICY_BILINEAR_TF1, POLICY_UNFUSED_TAIL, POLICY_DENSE_TRUNK, POLICY_CC_SPARSE_TRUNK, POLICY_UNFUSED_TRUNK, POLICY_TAIL_PAIR = 1, 2, 4, 8, 16, 32


class OfbError(RuntimeError):
    pass


# include/ofb_train.h: the data-parallel fit's reduce hook and the layout of its fp64 exchange buffer
REDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p)
TRAIN_N_BN, TRAIN_STATS_FWD, TRAIN_STATS_LOSS, TRAIN_STATS_BWD, TRAIN_STATS_LEN = 7, 0, 112, 114, 226
STAGE_FWD_BN, STAGE_LOSS, STAGE_BWD_BN, STAGE_GRADS = 0, 7, 8, 15


_lib = None


def lib_path():
    return _build.LIB


def load():
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if not os.path.exists(path):
        raise OfbError("libofb.so not built (%s); run `python -m ofighters_b200.build` -- "
                       "there is no CPU fallback" % path)
    lib = C.CDLL(path)
    vp, i64, u64, u32, i32 = C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32, C.c_int
    lib.ofb_abi_version.restype = i32
    lib.ofb_last_error.restype = C.c_char_p
    lib.ofb_default_config.argtypes = [C.POINTER(OfbConfig)]
    lib.ofb_default_config.restype = None
    lib.ofb_create.argtypes = [C.POINTER(OfbConfig), i64, i32, vp, vp, C.POINTER(vp)]
    lib.ofb_destroy.argtypes = [vp]
    lib.ofb_laser_cap.argtypes = [vp]
    lib.ofb_state_stride.argtypes = [vp]
    lib.ofb_state_stride.restype = i64
    lib.ofb_step_host.argtypes = [vp, vp, vp, vp]
    lib.ofb_step_host_async.argtypes = [vp, vp, vp, vp]
    lib.ofb_host_wait.argtypes = [vp]
    lib.ofb_step_bots.argtypes = [vp, i32, vp, u64, i64, u32, vp, vp, vp]
    lib.ofb_step_bots.restype = i32
    lib.ofb_frame.argtypes = [vp, vp, vp, vp, vp]
    lib.ofb_frame_bots.argtypes = [vp, i32, vp, u64, i64, u32, vp, vp, vp, vp]
    lib.ofb_frame_host_async.argtypes = [vp, vp, vp, vp, vp]
    lib.ofb_frame_host_async_i16.argtypes = [vp, vp, vp, vp, vp]
    lib.ofb_frame_host_async_i16.restype = i32
    lib.ofb_obs_pack_i16.argtypes = [vp, vp, i64, vp]
    lib.ofb_obs_pack_i16.restype = i32
    lib.ofb_debug_frame_prof.argtypes = [vp]
    lib.ofb_debug_frame_prof.restype = i32
    lib.ofb_debug_last_frame_fused.argtypes = []
    lib.ofb_debug_last_frame_fused.restype = i32
    for name in ("ofb_frame", "ofb_frame_bots", "ofb_frame_host_async"):
        getattr(lib, name).restype = i32
    lib.ofb_reset.argtypes = [vp, vp, vp, vp, vp]
    lib.ofb_step.argtypes = [vp, vp, vp, vp]
    lib.ofb_obs_vec.argtypes = [vp, vp, vp]
    lib.ofb_stats.argtypes = [vp, vp, vp]
    lib.ofb_stats.restype = i32
    lib.ofb_raster.argtypes = [vp, vp, i32, vp]
    lib.ofb_bot_actions.argtypes = [vp, i32, vp, u64, i64, u32, vp, vp]
    lib.ofb_random_spawn.argtypes = [i64, i32, i32, i32, u64, i64, u32, vp, vp]
    lib.ofb_state_export.argtypes = [vp, C.POINTER(OfbStateView), vp]
    lib.ofb_state_import.argtypes = [vp, C.POINTER(OfbStateView), vp]
    lib.ofb_policy_create.argtypes = [C.POINTER(OfbPolicyWeights), i32, i32, C.POINTER(vp)]
    lib.ofb_policy_create_opts.argtypes = [C.POINTER(OfbPolicyWeights), i32, i32, i32, C.POINTER(vp)]
    lib.ofb_policy_create_opts.restype = i32
    lib.ofb_policy_set_taps.argtypes = [vp, i32]
    lib.ofb_policy_set_taps.restype = i32
    lib.ofb_policy_destroy.argtypes = [vp]
    lib.ofb_policy_set_weights.argtypes = [vp, C.POINTER(OfbPolicyWeights), vp]
    lib.ofb_policy_set_weights.restype = i32
    lib.ofb_policy_set_engine.argtypes = [vp, i32]
    lib.ofb_policy_forward.argtypes = [vp, vp, vp, i64, i32, vp, vp, vp, vp, vp]
    lib.ofb_policy_write_actions.argtypes = [vp, vp, i64, i32, vp, i32, C.c_float, u64, i64, u32, vp, vp]
    lib.ofb_policy_play_actions.argtypes = [vp, vp, i64, i32, vp, i32, C.POINTER(OfbEpsSchedule), C.c_double, i32, u64, i64, u32,
                                            vp, vp, vp]
    lib.ofb_policy_play_actions.restype = i32
    lib.ofb_eps_value.argtypes = [C.POINTER(OfbEpsSchedule), C.c_double]
    lib.ofb_eps_value.restype = C.c_float
    lib.ofb_policy_pack_image.argtypes = [vp, i32, i64, vp, vp]
    lib.ofb_policy_debug_tap.argtypes = [vp, i32, i64, vp, vp]
    lib.ofb_policy_profile.argtypes = [vp, i32, vp]
    lib.ofb_policy_profile.restype = i32
    lib.ofb_train_default_config.argtypes = [C.POINTER(OfbTrainConfig)]
    lib.ofb_train_default_config.restype = None
    lib.ofb_trainer_create.argtypes = [vp, i64, C.POINTER(OfbTrainConfig), i32, C.POINTER(vp)]
    lib.ofb_trainer_destroy.argtypes = [vp]
    lib.ofb_trainer_fit.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp]
    lib.ofb_trainer_forward.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    lib.ofb_trainer_td_targets.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, C.c_float, i32, vp, vp, vp]
    lib.ofb_trainer_fit_weighted.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, vp]
    lib.ofb_trainer_td_errors.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, C.c_float, i32, vp, vp, vp]
    lib.ofb_trainer_td_targets_discounted.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]
    lib.ofb_trainer_td_errors_discounted.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp]
    lib.ofb_trainer_td_targets_double.argtypes = [vp] * 10 + [C.c_float, vp, i32] + [vp] * 5
    lib.ofb_trainer_fit_shard.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, vp, vp]
    lib.ofb_trainer_set_exchange.argtypes = [vp, vp, vp]
    lib.ofb_trainer_set_reducer.argtypes = [vp, REDUCE_FN, vp]
    lib.ofb_trainer_get_weights.argtypes = [vp, vp, vp]
    lib.ofb_trainer_get_grads.argtypes = [vp, vp, vp]
    lib.ofb_trainer_steps.argtypes = [vp]
    lib.ofb_trainer_steps.restype = i64
    lib.ofb_replay_create.argtypes = [vp, i64, i64, vp, i32, i32, C.POINTER(vp)]
    lib.ofb_replay_destroy.argtypes = [vp]
    lib.ofb_replay_device_bytes.argtypes = [vp]
    lib.ofb_replay_device_bytes.restype = i64
    lib.ofb_replay_pushes.argtypes = [vp]
    lib.ofb_replay_pushes.restype = i64
    lib.ofb_replay_push.argtypes = [vp, vp, vp, vp, vp]
    lib.ofb_replay_index.argtypes = [vp, vp, vp, vp]
    lib.ofb_replay_gather.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.ofb_replay_set_n_step.argtypes = [vp, i32]
    lib.ofb_replay_gather_nstep.argtypes = [vp, vp, i32, C.c_float, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.ofb_replay_enable_priorities.argtypes = [vp, C.POINTER(OfbReplayPrioConfig)]
    lib.ofb_replay_sample_prioritized.argtypes = [vp, i32, C.c_float, vp, vp, vp, vp]
    lib.ofb_replay_update_priorities.argtypes = [vp, vp, vp, vp, i32, vp]
    lib.ofb_replay_read_priorities.argtypes = [vp, vp, vp, vp, vp]
    lib.ofb_replay_sample_stats.argtypes = [vp, vp, vp]
    lib.ofb_replay_rescale_weights.argtypes = [vp, i32, C.c_float, vp, vp, vp]
    for name in ("ofb_replay_create", "ofb_replay_destroy", "ofb_replay_push", "ofb_replay_index", "ofb_replay_gather",
                 "ofb_replay_enable_priorities", "ofb_replay_sample_prioritized", "ofb_replay_update_priorities",
                 "ofb_replay_read_priorities", "ofb_replay_set_n_step", "ofb_replay_gather_nstep", "ofb_replay_sample_stats",
                 "ofb_replay_rescale_weights"):
        getattr(lib, name).restype = i32
    for name in ("ofb_trainer_create", "ofb_trainer_destroy", "ofb_trainer_fit", "ofb_trainer_forward",
                 "ofb_trainer_td_targets", "ofb_trainer_fit_weighted", "ofb_trainer_td_errors", "ofb_trainer_get_weights", "ofb_trainer_get_grads",
                 "ofb_trainer_td_targets_discounted", "ofb_trainer_td_errors_discounted", "ofb_trainer_td_targets_double",
                 "ofb_trainer_fit_shard", "ofb_trainer_set_exchange", "ofb_trainer_set_reducer"):
        getattr(lib, name).restype = i32
    for name in ("ofb_policy_create", "ofb_policy_destroy", "ofb_policy_set_engine", "ofb_policy_forward",
                 "ofb_policy_write_actions", "ofb_policy_pack_image", "ofb_policy_debug_tap"):
        getattr(lib, name).restype = i32
    for name in ("ofb_create", "ofb_destroy", "ofb_laser_cap", "ofb_reset", "ofb_step", "ofb_step_host", "ofb_step_host_async", "ofb_host_wait", "ofb_obs_vec", "ofb_raster",
                 "ofb_bot_actions", "ofb_random_spawn", "ofb_state_export", "ofb_state_import"):
        getattr(lib, name).restype = i32
    _lib = lib
    return lib


def check(rc):
    if rc < 0:
        raise OfbError("libofb error %d: %s" % (rc, load().ofb_last_error().decode()))
    return rc
