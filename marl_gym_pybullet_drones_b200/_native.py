"""ctypes binding of `libbatchdrones.so` (the C-ABI in `include/batch_drones.h`).

There is no fallback: if the shared library has not been built, or the CUDA
runtime reports an error, the calls raise.  Build with
`python -m marl_gym_pybullet_drones_b200.build` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbatchdrones.so")

BD_TASK = {"hover": 0, "multihover": 1, "spiral": 2, "meetup": 3, "flock": 4, "leaderfollower": 5}
BD_ACT = {"rpm": 0, "one_d_rpm": 1, "pid": 2, "vel": 3, "one_d_pid": 4}
BD_MODEL = {"cf2x": 0, "cf2p": 1, "racer": 2}
BD_PRECISION = {"fp32": 0, "fp64": 1}
BD_INTEGRATOR = {"quat": 0, "euler": 1}
BD_RESET = {"fixed": 0, "jitter_philox": 1, "jitter_buffer": 2}
BD_SNAP_ANGV, BD_SNAP_CTRL, BD_SNAP_EPISODES = 1, 2, 4   # optional snapshot planes (bd_snapshot_layout)

EXPORTS = (
    "bd_create", "bd_destroy", "bd_set_init_poses", "bd_set_jitter", "bd_reset", "bd_step",
    "bd_step_host", "bd_step_host_compact", "bd_step_many", "bd_set_step_many_mode", "bd_stream_gate", "bd_get_rng_state", "bd_set_rng_state",
    "bd_debug_set_tile_epoch", "bd_l2_plan", "bd_l2_policy", "bd_get_state", "bd_set_state", "bd_get_targets", "bd_episode_stats",
    "bd_get_controller_state", "bd_set_controller_state", "bd_set_action_f32",
    "bd_snapshot_layout", "bd_snapshot_bytes", "bd_save_snapshot", "bd_load_snapshot", "bd_obs_dim", "bd_act_dim",
    "bd_action_buffer_size", "bd_substeps", "bd_launch_count", "bd_last_error", "bd_version",
    "bd_actor_create", "bd_actor_destroy", "bd_actor_set_weights", "bd_actor_forward", "bd_actor_set_trace", "bd_actor_launch_count",
    "bd_actor_last_error", "bd_actor_set_input_norm",
    "bd_rms_create", "bd_rms_destroy", "bd_rms_update", "bd_rms_batch_moments", "bd_rms_merge_moments", "bd_rms_normalize", "bd_rms_get", "bd_rms_set",
    "bd_rms_launch_count", "bd_rms_last_error",
    "bd_ppo_net_create", "bd_ppo_net_destroy", "bd_ppo_net_param_count", "bd_ppo_net_stats", "bd_ppo_net_pack", "bd_ppo_forward", "bd_ppo_sample", "bd_ppo_set_trace", "bd_ppo_set_train_mode", "bd_ppo_set_forward_mode",
    "bd_ppo_grad", "bd_ppo_adam_step", "bd_ppo_gae", "bd_ppo_adv_stats", "bd_ppo_launch_count", "bd_ppo_last_error",
    "bd_peer_create", "bd_peer_destroy", "bd_peer_handle_size", "bd_peer_get_handle", "bd_peer_open", "bd_peer_data", "bd_peer_allreduce",
    "bd_peer_unmap", "bd_peer_launch_count", "bd_peer_last_error",
)


class BdConfig(C.Structure):
    """Mirror of `struct bd_config` (include/batch_drones.h)."""

    _fields_ = [
        ("struct_size", C.c_int32), ("device", C.c_int32),
        ("n_envs", C.c_int32), ("n_drones", C.c_int32),
        ("task", C.c_int32), ("act_type", C.c_int32), ("drone_model", C.c_int32),
        ("precision", C.c_int32), ("aero_flags", C.c_int32), ("integrator", C.c_int32),
        ("pyb_freq", C.c_int32), ("ctrl_freq", C.c_int32),
        ("auto_reset", C.c_int32), ("reset_mode", C.c_int32),
        ("action_is_f32", C.c_int32), ("keep_ang_vel", C.c_int32),
        ("track_episodes", C.c_int32), ("ctrl_reset_on_reset", C.c_int32),
        ("seed", C.c_uint64),
        ("episode_len_sec", C.c_double),
        ("mass", C.c_double), ("arm", C.c_double), ("kf", C.c_double), ("km", C.c_double),
        ("ixx", C.c_double), ("iyy", C.c_double), ("izz", C.c_double), ("g", C.c_double),
        ("thrust2weight", C.c_double), ("gnd_eff_coeff", C.c_double), ("prop_radius", C.c_double),
        ("drag_coeff_xy", C.c_double), ("drag_coeff_z", C.c_double),
        ("dw_coeff_1", C.c_double), ("dw_coeff_2", C.c_double), ("dw_coeff_3", C.c_double),
        ("prop_xy", C.c_double * 8),
        ("spiral_radius", C.c_double), ("spiral_period", C.c_double), ("height_rate", C.c_double),
        ("target_center", C.c_double * 3),
        ("ctrl_mass", C.c_double), ("ctrl_kf", C.c_double), ("speed_limit", C.c_double),
    ]


class NativeError(RuntimeError):
    pass


_lib = None


def load():
    """Load the library once and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
            "`python -m marl_gym_pybullet_drones_b200.build` (needs nvcc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32p, u8p, f32p, dp = C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.POINTER(C.c_double)
    lib.bd_create.argtypes = [C.POINTER(BdConfig), C.POINTER(vp)]
    lib.bd_create.restype = C.c_int
    lib.bd_destroy.argtypes = [vp]
    lib.bd_destroy.restype = None
    lib.bd_set_init_poses.argtypes = [vp, dp, dp, C.c_int]
    lib.bd_set_init_poses.restype = C.c_int
    lib.bd_set_jitter.argtypes = [vp, vp, vp]
    lib.bd_set_jitter.restype = C.c_int
    lib.bd_reset.argtypes = [vp, u8p, f32p, vp]
    lib.bd_reset.restype = C.c_int
    lib.bd_step.argtypes = [vp, vp, f32p, vp, u8p, u8p, f32p, vp]
    lib.bd_step.restype = C.c_int
    lib.bd_step_host.argtypes = [vp, vp, f32p, vp, u8p, u8p, f32p, vp]
    lib.bd_step_host.restype = C.c_int
    lib.bd_step_host_compact.argtypes = [vp, vp, f32p, vp, u8p, u8p, C.POINTER(C.c_int32), C.POINTER(vp), C.POINTER(vp), vp]
    lib.bd_step_host_compact.restype = C.c_int
    lib.bd_step_many.argtypes = [vp, C.c_int, vp, f32p, vp, u8p, u8p, vp]
    lib.bd_step_many.restype = C.c_int
    lib.bd_set_step_many_mode.argtypes = [vp, C.c_int]
    lib.bd_set_step_many_mode.restype = C.c_int
    lib.bd_stream_gate.argtypes = [vp, vp]
    lib.bd_stream_gate.restype = C.c_int
    lib.bd_get_rng_state.argtypes = [vp, C.POINTER(C.c_uint64)]
    lib.bd_get_rng_state.restype = C.c_int
    lib.bd_set_rng_state.argtypes = [vp, C.POINTER(C.c_uint64)]
    lib.bd_set_rng_state.restype = C.c_int
    lib.bd_debug_set_tile_epoch.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.bd_debug_set_tile_epoch.restype = C.c_int
    lib.bd_get_state.argtypes = [vp, vp, vp, vp, vp]
    lib.bd_get_state.restype = C.c_int
    lib.bd_set_state.argtypes = [vp, vp, vp, vp, vp]
    lib.bd_set_state.restype = C.c_int
    lib.bd_get_targets.argtypes = [vp, vp, vp]
    lib.bd_get_targets.restype = C.c_int
    lib.bd_episode_stats.argtypes = [vp, vp, C.c_int, vp]
    lib.bd_episode_stats.restype = C.c_int
    lib.bd_get_controller_state.argtypes = [vp, vp, vp]
    lib.bd_get_controller_state.restype = C.c_int
    lib.bd_set_controller_state.argtypes = [vp, vp, vp]
    lib.bd_set_controller_state.restype = C.c_int
    lib.bd_set_action_f32.argtypes = [vp, C.c_int]
    lib.bd_set_action_f32.restype = C.c_int
    lib.bd_snapshot_layout.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64)]
    lib.bd_snapshot_layout.restype = C.c_int
    lib.bd_snapshot_bytes.argtypes = [vp]
    lib.bd_snapshot_bytes.restype = C.c_int64
    lib.bd_save_snapshot.argtypes = [vp, vp, vp]
    lib.bd_save_snapshot.restype = C.c_int
    lib.bd_load_snapshot.argtypes = [vp, vp, u8p, vp]
    lib.bd_load_snapshot.restype = C.c_int
    for name in ("bd_obs_dim", "bd_act_dim", "bd_action_buffer_size", "bd_substeps"):
        getattr(lib, name).argtypes = [vp]
        getattr(lib, name).restype = C.c_int
    ip = C.POINTER(C.c_int)
    lib.bd_l2_plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_char_p, ip, ip]
    lib.bd_l2_plan.restype = C.c_int
    lib.bd_l2_policy.argtypes = [vp, ip, ip]
    lib.bd_l2_policy.restype = C.c_int
    lib.bd_launch_count.argtypes = [vp]
    lib.bd_launch_count.restype = C.c_int64
    lib.bd_last_error.argtypes = []
    lib.bd_last_error.restype = C.c_char_p
    lib.bd_version.argtypes = []
    lib.bd_version.restype = C.c_int
    lib.bd_actor_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    lib.bd_actor_create.restype = C.c_int
    lib.bd_actor_destroy.argtypes = [vp]
    lib.bd_actor_destroy.restype = None
    lib.bd_actor_set_weights.argtypes = [vp] + [vp] * 7 + [vp]
    lib.bd_actor_set_weights.restype = C.c_int
    lib.bd_actor_forward.argtypes = [vp, vp, C.c_int64, vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp]
    lib.bd_actor_forward.restype = C.c_int
    lib.bd_actor_set_trace.argtypes = [vp, vp]
    lib.bd_actor_set_trace.restype = C.c_int
    lib.bd_actor_launch_count.argtypes = [vp]
    lib.bd_actor_launch_count.restype = C.c_int64
    lib.bd_actor_last_error.argtypes = []
    lib.bd_actor_last_error.restype = C.c_char_p
    lib.bd_actor_set_input_norm.argtypes = [vp, vp, vp, C.c_int, C.c_float]
    lib.bd_actor_set_input_norm.restype = C.c_int
    lib.bd_rms_create.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double, C.POINTER(vp)]
    lib.bd_rms_create.restype = C.c_int
    lib.bd_rms_destroy.argtypes = [vp]
    lib.bd_rms_destroy.restype = None
    lib.bd_rms_update.argtypes = [vp, vp, C.c_int64, vp]
    lib.bd_rms_update.restype = C.c_int
    lib.bd_rms_batch_moments.argtypes = [vp, vp, C.c_int64, vp, vp]
    lib.bd_rms_batch_moments.restype = C.c_int
    lib.bd_rms_merge_moments.argtypes = [vp, vp, C.c_int, vp]
    lib.bd_rms_merge_moments.restype = C.c_int
    lib.bd_rms_normalize.argtypes = [vp, vp, vp, C.c_int64, C.c_float, vp]
    lib.bd_rms_normalize.restype = C.c_int
    lib.bd_rms_get.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.bd_rms_get.restype = C.c_int
    lib.bd_rms_set.argtypes = [vp, vp, vp, vp, vp]
    lib.bd_rms_set.restype = C.c_int
    lib.bd_rms_launch_count.argtypes = [vp]
    lib.bd_rms_launch_count.restype = C.c_int64
    lib.bd_rms_last_error.argtypes = []
    lib.bd_rms_last_error.restype = C.c_char_p
    lib.bd_ppo_net_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.POINTER(vp)]
    lib.bd_ppo_net_create.restype = C.c_int
    lib.bd_ppo_net_destroy.argtypes = [vp]
    lib.bd_ppo_net_destroy.restype = None
    lib.bd_ppo_net_param_count.argtypes = [vp]
    lib.bd_ppo_net_param_count.restype = C.c_int64
    lib.bd_ppo_net_stats.argtypes = [vp]
    lib.bd_ppo_net_stats.restype = vp
    lib.bd_ppo_net_pack.argtypes = [vp, vp, vp]
    lib.bd_ppo_net_pack.restype = C.c_int
    lib.bd_ppo_forward.argtypes = [vp, vp, C.c_int, C.c_int, vp, C.c_int64, vp, vp, C.c_float, vp, vp]
    lib.bd_ppo_forward.restype = C.c_int
    lib.bd_ppo_sample.argtypes = [vp, vp, C.c_int, C.c_int, vp, vp, C.c_float, vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp]
    lib.bd_ppo_sample.restype = C.c_int
    lib.bd_ppo_set_trace.argtypes = [vp, vp]
    lib.bd_ppo_set_trace.restype = C.c_int
    lib.bd_ppo_set_train_mode.argtypes = [vp, C.c_int]
    lib.bd_ppo_set_train_mode.restype = C.c_int
    lib.bd_ppo_set_forward_mode.argtypes = [vp, C.c_int]
    lib.bd_ppo_set_forward_mode.restype = C.c_int
    lib.bd_ppo_grad.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int64, vp, vp, vp, vp, vp, vp, C.c_float, C.c_int,
                                C.c_float, vp, vp, C.c_float, C.c_int64, vp, vp, vp]
    lib.bd_ppo_grad.restype = C.c_int
    lib.bd_ppo_adam_step.argtypes = [vp, vp, vp, vp, vp, vp, C.c_float, C.c_float, C.c_float, C.c_float, vp, vp, C.c_float, vp, vp]
    lib.bd_ppo_adam_step.restype = C.c_int
    lib.bd_ppo_gae.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, vp, vp, vp, vp]
    lib.bd_ppo_gae.restype = C.c_int
    lib.bd_ppo_adv_stats.argtypes = [vp, vp, vp]
    lib.bd_ppo_adv_stats.restype = C.c_int
    lib.bd_ppo_launch_count.argtypes = [vp]
    lib.bd_ppo_launch_count.restype = C.c_int64
    lib.bd_ppo_last_error.argtypes = []
    lib.bd_ppo_last_error.restype = C.c_char_p
    lib.bd_peer_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(vp)]
    lib.bd_peer_create.restype = C.c_int
    lib.bd_peer_destroy.argtypes = [vp]
    lib.bd_peer_destroy.restype = None
    lib.bd_peer_handle_size.argtypes = []
    lib.bd_peer_handle_size.restype = C.c_int
    lib.bd_peer_get_handle.argtypes = [vp, vp]
    lib.bd_peer_get_handle.restype = C.c_int
    lib.bd_peer_open.argtypes = [vp, vp, C.c_int]
    lib.bd_peer_open.restype = C.c_int
    lib.bd_peer_data.argtypes = [vp]
    lib.bd_peer_data.restype = vp
    lib.bd_peer_allreduce.argtypes = [vp, C.c_int64, vp, C.c_int, vp]
    lib.bd_peer_allreduce.restype = C.c_int
    lib.bd_peer_launch_count.argtypes = [vp]
    lib.bd_peer_launch_count.restype = C.c_int64
    lib.bd_peer_unmap.argtypes = [vp]
    lib.bd_peer_unmap.restype = C.c_int
    lib.bd_peer_last_error.argtypes = []
    lib.bd_peer_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().bd_last_error().decode("utf-8", "replace")
        raise NativeError(f"{what} failed ({rc}): {msg}")
