"""`BatchAviary`: N environments x M drones stepped by one CUDA kernel per control step.

This is the device-resident replacement for "N copies of an aviary inside
SubprocVecEnv workers" (`safe_control_gym/envs/env_wrappers/vectorized_env/
subproc_vec_env.py:23-73` driving `gym_pybullet_drones/envs/BaseAviary.py:259-383`).
Observations, rewards and flags are torch tensors on the GPU, so a rollout loop
(`mappo/mappo.py:647-712`) consumes them with no host round trip.

Constructor arguments keep the reference's names and meaning
(`MultiHoverAviary.py:12-25`, `SpiralAviary.py:20-37`); attributes read by the
reference's callers (`NUM_DRONES`, `CTRL_FREQ`, `EPISODE_LEN_SEC`, `INIT_XYZS`,
`TARGET_POS`, `observation_space`, `action_space`, ...) are provided with the
same names.  Everything numeric is done by `libbatchdrones.so`; there is no CPU
path in this module.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple, Optional

import numpy as np
import torch

from . import _native
from .constants import DroneConstants, drone_constants
from .enums import ActionType, DroneModel, ObservationType, Physics, physics_aero_flags
from .spaces import Box

_TASKS = ("hover", "multihover", "spiral", "meetup", "flock", "leaderfollower")


class StepResult(NamedTuple):
    """Device tensors returned by `BatchAviary.step_device`."""

    obs: torch.Tensor          # (N, M, D) float32; reset obs for envs that just finished (auto_reset)
    reward: torch.Tensor       # (N,) float32 / float64
    terminated: torch.Tensor   # (N,) bool
    truncated: torch.Tensor    # (N,) bool
    terminal_obs: Optional[torch.Tensor]   # (N, M, D) float32, rows valid where done (or None)

    @property
    def done(self) -> torch.Tensor:
        return self.terminated | self.truncated


def _as_enum(cls, v):
    return v if isinstance(v, cls) else cls(v)


class BatchAviary:
    """Vectorised HoverAviary / MultiHoverAviary / SpiralFormationAviary on one GPU."""

    def __init__(self,
                 task: str = "multihover",
                 num_envs: int = 1,
                 drone_model: DroneModel = DroneModel.CF2X,
                 num_drones: int = 1,
                 neighbourhood_radius: float = np.inf,
                 initial_xyzs=None,
                 initial_rpys=None,
                 physics: Physics = Physics.DYN,
                 pyb_freq: int = 240,
                 ctrl_freq: int = 30,
                 gui: bool = False,
                 record: bool = False,
                 obs: ObservationType = ObservationType.KIN,
                 act: ActionType = ActionType.RPM,
                 *,
                 precision: str = "fp32",
                 device=None,
                 auto_reset: bool = True,
                 reset_mode: Optional[str] = None,
                 integrator: str = "quat",
                 keep_ang_vel: bool = False,
                 track_episode_stats: bool = False,
                 reset_controllers: bool = False,
                 action_dtype=None,
                 seed: int = 0,
                 spiral_radius: float = 0.4,
                 spiral_period: float = 10.0,
                 height_rate: float = 0.05,
                 target_center=(0.0, 0.0, 0.0)):
        if task not in _TASKS:
            raise ValueError(f"task must be one of {_TASKS}")
        drone_model = _as_enum(DroneModel, drone_model)
        physics = _as_enum(Physics, physics)
        obs = _as_enum(ObservationType, obs)
        act = _as_enum(ActionType, act)
        if gui or record:
            raise NotImplementedError("GUI / video recording need PyBullet's renderer (out of scope)")
        if obs != ObservationType.KIN:
            raise NotImplementedError("only ObservationType.KIN is produced by the GPU path")
        if act in (ActionType.PID, ActionType.VEL, ActionType.ONE_D_PID) and drone_model not in (
                DroneModel.CF2X, DroneModel.CF2P):   # BaseRLAviary.py:73-78
            raise ValueError("[ERROR] in BaseRLAviary.__init()__, no controller is available for the specified drone_model")
        if pyb_freq % ctrl_freq != 0:   # BaseAviary.py:79-80
            raise ValueError('[ERROR] in BaseAviary.__init__(), pyb_freq is not divisible by env_freq.')
        if precision not in _native.BD_PRECISION:
            raise ValueError("precision must be 'fp32' or 'fp64'")
        if not torch.cuda.is_available():
            raise RuntimeError("BatchAviary needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.type != "cuda":
            raise RuntimeError("BatchAviary needs a CUDA device; there is no CPU fallback")
        self._dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()

        self.task = task
        self.num_envs = int(num_envs)
        self.DRONE_MODEL = drone_model
        self.NUM_DRONES = 1 if task == "hover" else int(num_drones)
        self.NEIGHBOURHOOD_RADIUS = neighbourhood_radius
        self.PHYSICS = physics
        self.OBS_TYPE, self.ACT_TYPE = obs, act
        self.PYB_FREQ, self.CTRL_FREQ = int(pyb_freq), int(ctrl_freq)
        self.PYB_STEPS_PER_CTRL = int(self.PYB_FREQ / self.CTRL_FREQ)
        self.CTRL_TIMESTEP = 1. / self.CTRL_FREQ
        self.PYB_TIMESTEP = 1. / self.PYB_FREQ
        self.ACTION_BUFFER_SIZE = int(ctrl_freq // 2)
        self.EPISODE_LEN_SEC = 12 if task == "spiral" else 8
        self.precision = precision
        self.real_dtype = torch.float64 if precision == "fp64" else torch.float32
        if action_dtype is None:
            action_dtype = self.real_dtype
        if action_dtype not in (torch.float32, torch.float64) or (
                precision == "fp32" and action_dtype != torch.float32):
            raise ValueError("action_dtype must be float32 (or float64 in fp64 mode)")
        self.action_dtype = action_dtype
        self.auto_reset = bool(auto_reset)
        if reset_mode is None:
            reset_mode = "jitter_philox" if task == "multihover" else "fixed"
        if reset_mode not in _native.BD_RESET:
            raise ValueError(f"reset_mode must be one of {tuple(_native.BD_RESET)}")
        self.reset_mode = reset_mode

        k: DroneConstants = drone_constants(drone_model)
        self.K = k
        # reference attribute names (BaseAviary.py:97-128)
        self.M, self.L, self.KF, self.KM = k.M, k.L, k.KF, k.KM
        self.THRUST2WEIGHT_RATIO, self.J, self.J_INV = k.THRUST2WEIGHT_RATIO, k.J, k.J_INV
        self.G, self.GRAVITY = k.G, k.GRAVITY
        self.HOVER_RPM, self.MAX_RPM, self.MAX_THRUST = k.HOVER_RPM, k.MAX_RPM, k.MAX_THRUST
        self.MAX_XY_TORQUE, self.MAX_Z_TORQUE = k.MAX_XY_TORQUE, k.MAX_Z_TORQUE
        self.GND_EFF_COEFF, self.PROP_RADIUS, self.GND_EFF_H_CLIP = k.GND_EFF_COEFF, k.PROP_RADIUS, k.GND_EFF_H_CLIP
        self.DRAG_COEFF = k.DRAG_COEFF
        self.DW_COEFF_1, self.DW_COEFF_2, self.DW_COEFF_3 = k.DW_COEFF_1, k.DW_COEFF_2, k.DW_COEFF_3
        self.COLLISION_H, self.COLLISION_R, self.COLLISION_Z_OFFSET = k.COLLISION_H, k.COLLISION_R, k.COLLISION_Z_OFFSET
        self.MAX_SPEED_KMH = k.MAX_SPEED_KMH
        if task == "spiral":
            self.R, self.PERIOD = spiral_radius, spiral_period
            self.OMEGA = 2 * np.pi / self.PERIOD
            self.VZ = height_rate
            self.CENTER = np.array(target_center, dtype=np.float64)

        cfg = _native.BdConfig()
        cfg.struct_size = C.sizeof(_native.BdConfig)
        cfg.device = self._dev_index
        cfg.n_envs, cfg.n_drones = self.num_envs, self.NUM_DRONES
        cfg.task = _native.BD_TASK[task]
        cfg.act_type = _native.BD_ACT[act.value]
        cfg.drone_model = _native.BD_MODEL[drone_model.value]
        cfg.precision = _native.BD_PRECISION[precision]
        cfg.aero_flags = physics_aero_flags(physics)
        cfg.integrator = _native.BD_INTEGRATOR[integrator]
        cfg.pyb_freq, cfg.ctrl_freq = self.PYB_FREQ, self.CTRL_FREQ
        cfg.auto_reset = int(self.auto_reset)
        cfg.reset_mode = _native.BD_RESET[reset_mode]
        cfg.action_is_f32 = int(action_dtype == torch.float32)
        cfg.keep_ang_vel = int(keep_ang_vel)
        cfg.track_episodes = int(track_episode_stats)
        # DSL PID in the loop (ActionType.PID / VEL / ONE_D_PID): the reference always builds
        # DSLPIDControl(DroneModel.CF2X) (BaseRLAviary.py:76) and never resets it with the env
        cfg.ctrl_reset_on_reset = int(reset_controllers)
        kc: DroneConstants = drone_constants(DroneModel.CF2X)
        cfg.ctrl_mass, cfg.ctrl_kf = kc.M, kc.KF
        if act == ActionType.VEL:
            self.SPEED_LIMIT = 0.03 * k.MAX_SPEED_KMH * (1000 / 3600)             # BaseRLAviary.py:94-95
        cfg.speed_limit = float(getattr(self, "SPEED_LIMIT", 0.0))
        cfg.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        cfg.episode_len_sec = float(self.EPISODE_LEN_SEC)
        cfg.mass, cfg.arm, cfg.kf, cfg.km = k.M, k.L, k.KF, k.KM
        cfg.ixx, cfg.iyy, cfg.izz, cfg.g = k.IXX, k.IYY, k.IZZ, k.G
        cfg.thrust2weight, cfg.gnd_eff_coeff, cfg.prop_radius = k.THRUST2WEIGHT_RATIO, k.GND_EFF_COEFF, k.PROP_RADIUS
        cfg.drag_coeff_xy, cfg.drag_coeff_z = k.DRAG_COEFF_XY, k.DRAG_COEFF_Z
        cfg.dw_coeff_1, cfg.dw_coeff_2, cfg.dw_coeff_3 = k.DW_COEFF_1, k.DW_COEFF_2, k.DW_COEFF_3
        for i, (x, y, _z) in enumerate(k.PROP_OFFSETS):
            cfg.prop_xy[2 * i], cfg.prop_xy[2 * i + 1] = x, y
        cfg.spiral_radius, cfg.spiral_period, cfg.height_rate = spiral_radius, spiral_period, height_rate
        for i in range(3):
            cfg.target_center[i] = float(target_center[i])
        self._cfg = cfg
        self._lib = _native.load()
        self._h = C.c_void_p()
        _native.check(self._lib.bd_create(C.byref(cfg), C.byref(self._h)), "bd_create")

        self.ACTION_DIM = self._lib.bd_act_dim(self._h)
        self.OBS_DIM = self._lib.bd_obs_dim(self._h)
        M = self.NUM_DRONES
        # default initial poses (BaseAviary.py:194-203; SpiralAviary.py:47-53)
        if initial_xyzs is None:
            if task == "spiral":
                initial_xyzs = np.array([[spiral_radius * np.cos(2 * np.pi * i / M),
                                          spiral_radius * np.sin(2 * np.pi * i / M), 0.3] for i in range(M)])
            else:
                initial_xyzs = np.vstack([np.array([x * 4 * k.L for x in range(M)]),
                                          np.array([y * 4 * k.L for y in range(M)]),
                                          np.ones(M) * k.DEFAULT_SPAWN_Z]).transpose().reshape(M, 3)
        self.set_initial_poses(initial_xyzs, initial_rpys)

        # spaces of ONE env, as VecEnv exposes them (vec_env.py:23-30; BaseRLAviary.py:150-156,260-277)
        A, B = self.ACTION_DIM, self.ACTION_BUFFER_SIZE
        self.action_space = Box(low=-np.ones((M, A), dtype=np.float32), high=np.ones((M, A), dtype=np.float32),
                                dtype=np.float32)
        lo = np.full((M, self.OBS_DIM), -np.inf, dtype=np.float32)
        hi = np.full((M, self.OBS_DIM), np.inf, dtype=np.float32)
        if task != "spiral":   # SpiralAviary.py:103-116 uses +-inf everywhere
            lo[:, 2] = 0.0
            lo[:, 12:12 + A * B], hi[:, 12:12 + A * B] = -1.0, 1.0
        self.observation_space = Box(low=lo, high=hi, dtype=np.float32)
        self._terminal_obs = None
        self._out_cache = None
        self._bd_step = self._lib.bd_step
        self._closed = False

    # ------------------------------------------------------------------ utils
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_open(self):
        if self._closed or not self._h:
            raise RuntimeError("BatchAviary is closed")

    @property
    def launch_count(self) -> int:
        """Kernels launched by this aviary so far."""
        return int(self._lib.bd_launch_count(self._h))

    def set_initial_poses(self, initial_xyzs, initial_rpys=None):
        """Set INIT_XYZS / INIT_RPYS ((M,3) shared by all envs, or (N,M,3) per env) and, like the
        constructor (BaseAviary.py:212-214), put every env at exactly these poses (no jitter)."""
        M, N = self.NUM_DRONES, self.num_envs
        xyz = np.ascontiguousarray(np.asarray(initial_xyzs, dtype=np.float64))
        if xyz.shape == (M, 3):
            per_env = 0
        elif xyz.shape == (N, M, 3):
            per_env = 1
        else:   # BaseAviary.py:198-201
            raise ValueError("[ERROR] invalid initial_xyzs in BaseAviary.__init__(), "
                             "try initial_xyzs.reshape(NUM_DRONES,3)")
        rpy = None
        if initial_rpys is not None:
            rpy = np.ascontiguousarray(np.asarray(initial_rpys, dtype=np.float64))
            if rpy.shape != xyz.shape:
                raise ValueError("[ERROR] invalid initial_rpys in BaseAviary.__init__(), "
                                 "try initial_rpys.reshape(NUM_DRONES,3)")
        dp = C.POINTER(C.c_double)
        _native.check(self._lib.bd_set_init_poses(
            self._h, xyz.ctypes.data_as(dp), rpy.ctypes.data_as(dp) if rpy is not None else None, per_env),
            "bd_set_init_poses")
        self.INIT_XYZS = xyz
        self.INIT_RPYS = rpy if rpy is not None else np.zeros_like(xyz)

    # ------------------------------------------------------------- device API
    def reset_device(self, env_mask: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None):
        """Reset all envs (or those with `env_mask[e]` true); returns the obs tensor (N,M,D)."""
        self._check_open()
        if out is None:
            out = torch.zeros((self.num_envs, self.NUM_DRONES, self.OBS_DIM), dtype=torch.float32,
                              device=self.device)
        mask_ptr = None
        if env_mask is not None:
            env_mask = env_mask.to(device=self.device, dtype=torch.uint8).contiguous()
            mask_ptr = C.c_void_p(env_mask.data_ptr())
        _native.check(self._lib.bd_reset(self._h, mask_ptr, C.c_void_p(out.data_ptr()), self._stream()), "bd_reset")
        return out

    def step_device(self, actions: torch.Tensor, out: Optional[StepResult] = None,
                    want_terminal_obs: bool = False) -> StepResult:
        """One control step for all envs.  `actions`: (N,M,A) CUDA tensor of `action_dtype`."""
        self._check_open()
        N, M = self.num_envs, self.NUM_DRONES
        if self.precision == "fp64" and actions.dtype in (torch.float32, torch.float64):
            self._set_action_dtype(actions.dtype)
        if actions.device != self.device or actions.dtype != self.action_dtype or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=self.action_dtype).contiguous()
        if actions.numel() != N * M * self.ACTION_DIM:
            raise ValueError(f"actions must have shape ({N},{M},{self.ACTION_DIM})")
        if out is None:
            obs = torch.empty((N, M, self.OBS_DIM), dtype=torch.float32, device=self.device)
            reward = torch.empty((N,), dtype=self.real_dtype, device=self.device)
            term = torch.empty((N,), dtype=torch.uint8, device=self.device)
            trunc = torch.empty((N,), dtype=torch.uint8, device=self.device)
            ptrs = (obs.data_ptr(), reward.data_ptr(), term.data_ptr(), trunc.data_ptr())
            ret = None
        else:
            # a caller that steps into the same StepResult again and again (a rollout buffer slot, the bench) pays for
            # the pointer extraction once: at small batch sizes a step is bound by this call's host time
            cached = self._out_cache
            if cached is not None and cached[0] is out:
                ptrs = cached[1]
            else:
                ptrs = (out.obs.data_ptr(), out.reward.data_ptr(), out.terminated.data_ptr(), out.truncated.data_ptr())
                self._out_cache = (out, ptrs)
            ret = out
        tobs_ptr = None
        tobs = None
        if want_terminal_obs:
            if self._terminal_obs is None:
                self._terminal_obs = torch.zeros((N, M, self.OBS_DIM), dtype=torch.float32, device=self.device)
            tobs = self._terminal_obs
            tobs_ptr = tobs.data_ptr()
        rc = self._bd_step(self._h, actions.data_ptr(), ptrs[0], ptrs[1], ptrs[2], ptrs[3], tobs_ptr,
                           torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            _native.check(rc, "bd_step")
        if ret is None:
            return StepResult(obs, reward, term.view(torch.bool), trunc.view(torch.bool), tobs)
        return ret if tobs is None and ret.terminal_obs is None else ret._replace(terminal_obs=tobs)

    @staticmethod
    def pinned_array(shape, dtype=np.float32) -> np.ndarray:
        """Page-locked host array (for `step_host(..., actions_pinned=True)`)."""
        t = torch.empty(tuple(shape), dtype=getattr(torch, np.dtype(dtype).name), pin_memory=True)
        return t.numpy()

    def step_host(self, actions: np.ndarray, out: Optional[dict] = None, want_terminal_obs: bool = False,
                  actions_pinned: bool = False, compact_terminal_obs: bool = False, buffer_set: int = 0) -> dict:
        """Host-buffer step through `bd_step_host` (H2D + kernel + D2H + sync).

        `actions`: (N,M,A) numpy array.  Returns a dict of numpy arrays backed by
        pinned memory that is reused on a later call (copy what you keep): `buffer_set` (0 / 1) selects one
        of two sets of output buffers, so a caller that alternates them keeps the previous step's arrays
        intact for one more step.
        `actions_pinned=True`: `actions` already lives in page-locked memory (`pinned_array`) with the
        aviary's action dtype and is handed to the copy engine as it is; otherwise it is first copied
        into a pinned staging buffer (a 4 MB host memcpy at 65 536 x 4 drones, ~0.35 ms).
        `want_terminal_obs=True`: a full (N,M,D) `terminal_obs` array (rows valid where done).
        `compact_terminal_obs=True`: `bd_step_host_compact` instead — `done_idx` (ascending env indices of the
        envs that finished) and `terminal_rows` (len(done_idx), M, D); views of memory owned by the handle
        (two sets used alternately), valid until the next-but-one step.
        """
        self._check_open()
        N, M = self.num_envs, self.NUM_DRONES
        actions = np.asarray(actions)
        if self.precision == "fp64" and actions.dtype in (np.float32, np.float64):
            want = torch.float32 if actions.dtype == np.float32 else torch.float64
            if want != self.action_dtype:
                self._set_action_dtype(want)
                self._host_bufs = {}
        np_act = np.float32 if self.action_dtype == torch.float32 else np.float64
        if out is None:
            bufs = self.__dict__.setdefault("_host_bufs", {})
            out = bufs.get(buffer_set)
            if out is None:
                pin = dict(pin_memory=True)
                out = bufs[buffer_set] = dict(
                    actions=torch.empty((N, M, self.ACTION_DIM), dtype=self.action_dtype, **pin),
                    obs=torch.empty((N, M, self.OBS_DIM), dtype=torch.float32, **pin),
                    reward=torch.empty((N,), dtype=self.real_dtype, **pin),
                    terminated=torch.empty((N,), dtype=torch.uint8, **pin),
                    truncated=torch.empty((N,), dtype=torch.uint8, **pin),
                    terminal_obs=None)
        if want_terminal_obs and out.get("terminal_obs") is None:
            out["terminal_obs"] = torch.zeros((N, M, self.OBS_DIM), dtype=torch.float32, pin_memory=True)
        if actions_pinned:
            if actions.dtype != np_act or not actions.flags["C_CONTIGUOUS"] or actions.size != N * M * self.ACTION_DIM:
                raise ValueError("actions_pinned=True needs a C-contiguous (N,M,A) array of the aviary's action dtype")
            act_ptr = actions.ctypes.data
        else:
            out["actions"].numpy()[...] = np.asarray(actions, dtype=np_act).reshape(N, M, self.ACTION_DIM)
            act_ptr = out["actions"].data_ptr()
        res = dict(obs=out["obs"].numpy(), reward=out["reward"].numpy(),
                   terminated=out["terminated"].numpy().view(np.bool_),
                   truncated=out["truncated"].numpy().view(np.bool_), terminal_obs=None)
        if compact_terminal_obs:
            n_done, idx_p, rows_p = C.c_int32(0), C.c_void_p(), C.c_void_p()
            _native.check(self._lib.bd_step_host_compact(
                self._h, C.c_void_p(act_ptr), C.c_void_p(out["obs"].data_ptr()),
                C.c_void_p(out["reward"].data_ptr()), C.c_void_p(out["terminated"].data_ptr()),
                C.c_void_p(out["truncated"].data_ptr()), C.byref(n_done), C.byref(idx_p), C.byref(rows_p),
                self._stream()), "bd_step_host_compact")
            k = int(n_done.value)
            if k > 0:
                idx = np.ctypeslib.as_array(C.cast(idx_p, C.POINTER(C.c_int32)), shape=(k,))
                rows = np.ctypeslib.as_array(C.cast(rows_p, C.POINTER(C.c_float)), shape=(k, M, self.OBS_DIM))
            else:
                idx, rows = np.zeros((0,), dtype=np.int32), np.zeros((0, M, self.OBS_DIM), dtype=np.float32)
            res["done_idx"], res["terminal_rows"] = idx, rows
            return res
        tob = out.get("terminal_obs") if want_terminal_obs else None
        _native.check(self._lib.bd_step_host(
            self._h, C.c_void_p(act_ptr), C.c_void_p(out["obs"].data_ptr()),
            C.c_void_p(out["reward"].data_ptr()), C.c_void_p(out["terminated"].data_ptr()),
            C.c_void_p(out["truncated"].data_ptr()),
            C.c_void_p(tob.data_ptr()) if tob is not None else None, self._stream()), "bd_step_host")
        res["terminal_obs"] = tob.numpy() if tob is not None else None
        return res

    def step_many(self, actions: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor,
                  truncated: torch.Tensor, one_launch: bool = True) -> None:
        """K control steps with one host call (`bd_step_many`): `actions` (K,N,M,A), outputs (K,N,M,D) / (K,N);
        step i reads `actions[i]` and writes slot i.  For open-loop action tapes and latency-bound small batches: on the
        fast float kernel the K steps are ONE launch (states in registers, action history in shared memory across
        steps); `one_launch=False` forces K launches of the per-step kernel (what a closed-loop caller pays)."""
        self._check_open()
        mode = 0 if one_launch else 1
        if mode != getattr(self, "_many_mode", 0):
            _native.check(self._lib.bd_set_step_many_mode(self._h, mode), "bd_set_step_many_mode")
            self._many_mode = mode
        K = int(actions.shape[0])
        N, M = self.num_envs, self.NUM_DRONES
        if (actions.dtype != self.action_dtype or not actions.is_contiguous() or actions.device != self.device
                or actions.numel() != K * N * M * self.ACTION_DIM):
            raise ValueError(f"actions must be a contiguous ({K},{N},{M},{self.ACTION_DIM}) {self.action_dtype} CUDA tensor")
        for t, shape, dt in ((obs, (K, N, M, self.OBS_DIM), torch.float32), (reward, (K, N), self.real_dtype)):
            if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"output tensor must be contiguous {shape} {dt} on {self.device}")
        for t in (terminated, truncated):
            if tuple(t.shape) != (K, N) or t.element_size() != 1 or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"flag tensors must be contiguous ({K},{N}) bool / uint8 on {self.device}")
        rc = self._lib.bd_step_many(self._h, K, actions.data_ptr(), obs.data_ptr(), reward.data_ptr(),
                                    terminated.data_ptr(), truncated.data_ptr(),
                                    torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            _native.check(rc, "bd_step_many")

    def get_rng_state(self):
        """Philox key and counters of the on-device re-spawn draws (`bd_get_rng_state`): a 4-tuple of ints."""
        self._check_open()
        st = (C.c_uint64 * 4)()
        _native.check(self._lib.bd_get_rng_state(self._h, st), "bd_get_rng_state")
        return tuple(int(v) for v in st)

    def set_rng_state(self, state):
        """Restore what `get_rng_state` returned: a resumed run continues the random stream."""
        self._check_open()
        st = (C.c_uint64 * 4)(*[int(v) for v in state])
        _native.check(self._lib.bd_set_rng_state(self._h, st), "bd_set_rng_state")

    # --------------------------------------------------------------- snapshots
    @property
    def snapshot_nbytes(self) -> int:
        """Bytes of this aviary's snapshots (`bd_snapshot_bytes`)."""
        self._check_open()
        return int(self._lib.bd_snapshot_bytes(self._h))

    def snapshot(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The complete simulator state as an opaque uint8 tensor of `snapshot_nbytes` bytes on the aviary's device
        (`bd_save_snapshot`): drone states, targets, controller memory, action history, step counters, episode
        returns and accumulators, and the RNG state of the re-spawn draws.  Stream ordered, no host synchronisation.
        `out`: a contiguous, 256-byte aligned uint8 CUDA tensor of that size to write into."""
        self._check_open()
        n = self.snapshot_nbytes
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=self.device)
        elif (out.dtype != torch.uint8 or out.numel() != n or not out.is_contiguous() or out.device != self.device
              or out.data_ptr() % 256):
            raise ValueError(f"out must be a contiguous, 256-byte aligned uint8 tensor of {n} bytes on {self.device}")
        _native.check(self._lib.bd_save_snapshot(self._h, C.c_void_p(out.data_ptr()), self._stream()), "bd_save_snapshot")
        return out

    def restore(self, snap: torch.Tensor, env_mask: Optional[torch.Tensor] = None):
        """Put the state of `snapshot()` back (`bd_load_snapshot`); `snap` may live on the device or the CPU.

        `env_mask=None` restores everything, the RNG state of the re-spawn draws included: the aviary continues exactly
        as the one the snapshot was taken from.  With an (N,) bool mask only those envs are restored; the aviary's own
        RNG state and episode accumulators stay as they are.  The snapshot may come from an aviary with another seed,
        reset mode, `auto_reset` or device, and from one that keeps more planes (`keep_ang_vel`, `track_episode_stats`)
        than this one needs; shape, task, physics and constants must match.  Synchronises (the header is checked on
        the host).  Observations are not written: the observation of a saved state is the one the step returned when
        it was saved, and the caller keeps it with the snapshot."""
        self._check_open()
        snap = torch.as_tensor(snap)
        if snap.dtype != torch.uint8 or snap.dim() != 1:
            raise ValueError("[ERROR] in BatchAviary.restore(), snap must be a 1-D uint8 tensor from BatchAviary.snapshot()")
        if snap.numel() < 256:
            raise ValueError(f"[ERROR] in BatchAviary.restore(), a snapshot has at least 256 bytes, got {snap.numel()}")
        want = int(np.frombuffer(snap[:256].cpu().numpy().tobytes()[40:48], dtype=np.int64)[0])   # SnapHeader.bytes
        if snap.numel() < want:
            raise ValueError(f"[ERROR] in BatchAviary.restore(), the snapshot buffer holds {snap.numel()} bytes, "
                             f"its header says {want} (truncated)")
        temporary = False
        if snap.device != self.device or not snap.is_contiguous() or snap.data_ptr() % 256:
            buf = torch.empty(snap.numel(), dtype=torch.uint8, device=self.device)
            buf.copy_(snap)
            snap, temporary = buf, True
        mask_ptr = None
        if env_mask is not None:
            m = torch.as_tensor(env_mask)
            if m.numel() != self.num_envs:
                raise ValueError(f"[ERROR] in BatchAviary.restore(), env_mask must have {self.num_envs} entries")
            env_mask = m.to(device=self.device, dtype=torch.uint8).contiguous()
            temporary = temporary or env_mask.data_ptr() != m.data_ptr()
            mask_ptr = C.c_void_p(env_mask.data_ptr())
        rc = self._lib.bd_load_snapshot(self._h, C.c_void_p(snap.data_ptr()), mask_ptr, self._stream())
        if rc == -1:
            raise ValueError("[ERROR] in BatchAviary.restore(), " + self._lib.bd_last_error().decode("utf-8", "replace"))
        _native.check(rc, "bd_load_snapshot")
        if temporary:   # the unpack kernel reads them: keep them alive until it is done
            torch.cuda.current_stream(self.device).synchronize()

    def _set_action_dtype(self, dtype):
        """fp64 mode: follow the dtype of the actions handed in, like numpy does in the reference
        (float32 actions -> `1 + 0.05*a` is evaluated in float32, BaseRLAviary.py:192)."""
        if dtype == self.action_dtype:
            return
        torch.cuda.current_stream(self.device).synchronize()
        _native.check(self._lib.bd_set_action_f32(self._h, int(dtype == torch.float32)), "bd_set_action_f32")
        self.action_dtype = dtype

    # ------------------------------------------------------------ state access
    def get_state(self, with_rates: bool = False, with_step_counter: bool = False):
        """(N,M,20) `_getDroneStateVector` layout (BaseAviary.py:559-561) [+ rpy_rates, step_counter]."""
        self._check_open()
        N, M = self.num_envs, self.NUM_DRONES
        st = torch.empty((N, M, 20), dtype=self.real_dtype, device=self.device)
        rates = torch.empty((N, M, 3), dtype=self.real_dtype, device=self.device) if with_rates else None
        sc = torch.empty((N,), dtype=torch.int32, device=self.device) if with_step_counter else None
        _native.check(self._lib.bd_get_state(
            self._h, C.c_void_p(st.data_ptr()), C.c_void_p(rates.data_ptr()) if rates is not None else None,
            C.c_void_p(sc.data_ptr()) if sc is not None else None, self._stream()), "bd_get_state")
        res = (st,)
        if with_rates:
            res += (rates,)
        if with_step_counter:
            res += (sc,)
        return res[0] if len(res) == 1 else res

    def set_state(self, kin13: Optional[torch.Tensor] = None, targets: Optional[torch.Tensor] = None,
                  step_counter: Optional[torch.Tensor] = None):
        """Inject [pos3 quat4 vel3 body_rates3] (N,M,13), TARGET_POS (N,M,3), step counters (N,)."""
        N, M = self.num_envs, self.NUM_DRONES

        def prep(t, shape, dtype):
            if t is None:
                return None
            t = torch.as_tensor(t).to(device=self.device, dtype=dtype).contiguous()
            if tuple(t.shape) != shape:
                raise ValueError(f"expected shape {shape}, got {tuple(t.shape)}")
            return t
        kin13 = prep(kin13, (N, M, 13), self.real_dtype)
        targets = prep(targets, (N, M, 3), self.real_dtype)
        step_counter = prep(step_counter, (N,), torch.int32)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None  # noqa: E731
        _native.check(self._lib.bd_set_state(self._h, ptr(kin13), ptr(targets), ptr(step_counter), self._stream()),
                      "bd_set_state")
        # keep the tensors alive until the stream has consumed them
        torch.cuda.current_stream(self.device).synchronize()

    def get_targets(self) -> torch.Tensor:
        """TARGET_POS of every drone, (N,M,3)."""
        self._check_open()
        t = torch.empty((self.num_envs, self.NUM_DRONES, 3), dtype=self.real_dtype, device=self.device)
        _native.check(self._lib.bd_get_targets(self._h, C.c_void_p(t.data_ptr()), self._stream()), "bd_get_targets")
        return t

    def get_controller_state(self) -> torch.Tensor:
        """DSL PID memory of every drone, (N,M,9) = [integral_pos_e, integral_rpy_e, last_rpy]
        (DSLPIDControl.py:64-79); PID / VEL / ONE_D_PID action types only."""
        self._check_open()
        t = torch.empty((self.num_envs, self.NUM_DRONES, 9), dtype=self.real_dtype, device=self.device)
        _native.check(self._lib.bd_get_controller_state(self._h, C.c_void_p(t.data_ptr()), self._stream()),
                      "bd_get_controller_state")
        return t

    def set_controller_state(self, ctrl=None):
        """Overwrite the DSL PID memory ((N,M,9)); `None` zeroes it = `ctrl[k].reset()` on every drone."""
        self._check_open()
        ptr = None
        if ctrl is not None:
            c = torch.as_tensor(ctrl).to(device=self.device, dtype=self.real_dtype).contiguous()
            if tuple(c.shape) != (self.num_envs, self.NUM_DRONES, 9):
                raise ValueError("ctrl must have shape (N,M,9)")
            ptr = C.c_void_p(c.data_ptr())
        _native.check(self._lib.bd_set_controller_state(self._h, ptr, self._stream()), "bd_set_controller_state")
        if ctrl is not None:
            torch.cuda.current_stream(self.device).synchronize()   # `c` may be a temporary

    def episode_stats(self, reset: bool = True) -> torch.Tensor:
        """Device tensor [sum of returns, sum of lengths, count] of the episodes finished since the
        accumulators were last reset (`VecRecordEpisodeStatistics` on the device; no host sync).
        Needs `track_episode_stats=True` at construction."""
        self._check_open()
        out = torch.empty(3, dtype=torch.float64, device=self.device)
        _native.check(self._lib.bd_episode_stats(self._h, C.c_void_p(out.data_ptr()), int(reset), self._stream()),
                      "bd_episode_stats")
        return out

    def set_jitter(self, jitter: torch.Tensor):
        """Jitter draws in [-0.25,0.25) consumed by the next reset of each env (reset_mode='jitter_buffer')."""
        self._check_open()
        j = torch.as_tensor(jitter).to(device=self.device, dtype=self.real_dtype).contiguous()
        if tuple(j.shape) != (self.num_envs, self.NUM_DRONES, 3):
            raise ValueError("jitter must have shape (N,M,3)")
        _native.check(self._lib.bd_set_jitter(self._h, C.c_void_p(j.data_ptr()), self._stream()), "bd_set_jitter")
        torch.cuda.current_stream(self.device).synchronize()

    def close(self):
        if not self._closed and self._h:
            self._lib.bd_destroy(self._h)
            self._h = C.c_void_p()
        self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
