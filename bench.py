#!/usr/bin/env python
"""Throughput bench of the batched drone-step hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]

A "step" is one control step of every environment on this GPU = ONE launch of
`step_kernel` (S = pyb_freq/ctrl_freq physics substeps per drone).  The metric is
drone-substeps/s = N_envs * M * S * K / time, aggregated over all ranks.

* default workload: BASELINE.json configs[3] — MultiHoverAviary, M = 4 drones, RPM
  action, 240 Hz physics / 30 Hz control, fp32, auto-reset on, random actions;
  65,536 envs PER GPU (weak scaling: every rank steps its own env shard, no
  data-path collective; NCCL is used only for the barrier / max-time reduction).
* `value`  : inputs resident in HBM (pre-generated action pool, observations
  written into a rotating rollout buffer so the working set exceeds L2).
* `e2e`    : the same step through the host-buffer C-ABI call `bd_step_host`
  (pinned numpy in, pinned numpy out: H2D + kernel + D2H + sync each step).
* `roofline`: algorithmic bytes (SURVEY.md §8d) / measured kernel time vs the
  measured HBM copy peak in MEASURED_PEAKS.json.
* `e2e_vecenv`: the same step through the reference-protocol call `BatchVecEnv.step` (the 4-tuple with info dicts
  that `MAPPO.train_step` consumes): `bd_step_host_compact`, terminal observations only for finished envs.
* `small_batch`: BASELINE configs[3] as literally sharded (8192 envs per GPU), K steps per host call (`bd_step_many`).
* `mappo`: env-steps/s of `DeviceMAPPO.train_step` at configs[4]'s per-GPU shape (16 drones, downwash) with the time
  shares of rollout / returns / update and the measured cost of the NCCL gradient all-reduce (N > 1).
* `cpu_baseline` / `--impl reference`: the fp64 numpy oracle of the reference's
  Physics.DYN path (the reference itself needs PyBullet, which is not
  installable), run the way the reference runs it: one Python env object per env,
  SubprocVecEnv-style spawn workers + Pipes on all host cores, auto-reset.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "drone_substeps_per_sec"
UNIT = "drone-substeps/s"
GRID_1M = [[0.0, 0.0, 0.5], [1.0, 0.0, 0.5], [0.0, 1.0, 0.5], [1.0, 1.0, 0.5]]


def grid_xyzs(m: int):
    side = int(np.ceil(np.sqrt(m)))
    return np.array([[float(i % side), float(i // side), 0.5] for i in range(m)])


def algorithmic_bytes_per_drone_step(A: int, B: int, M: int, e: int = 4, extra_obs: int = 0) -> float:
    """SURVEY.md §8(d): read state 13 + action A + history (B-1)A + target 3;
    write state 13 + obs 12 + B*A (+extras); per env 14 B (reward, 2 flags, counter r/w)."""
    return e * (41 + 2 * B * A + extra_obs) + 14.0 / M


DUMP_BYTES = 64_000_000


def dump_rows(n: int, floats_per_row: int) -> np.ndarray:
    """Rows (envs) that --dump-outputs writes: all n if they fit DUMP_BYTES as float32 (with room for the .npy headers),
    else a fixed seeded sample, sorted, so that every run of the same shape writes the same envs."""
    keep = min(n, (DUMP_BYTES - 4096) // (4 * floats_per_row))
    if keep == n:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, keep, replace=False))


def write_outputs(out_dir: str, arrays: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# --------------------------------------------------------------------------- CPU arm
def _cpu_worker(remote, n_envs, m, seed):
    """SubprocVecEnv worker stand-in (subproc_vec_env.py:186-261) around the oracle."""
    sys.path.insert(0, ROOT)
    from oracle.aviary_oracle import OracleAviary, step_env_autoreset
    np.random.seed(seed)
    xyz = grid_xyzs(m)
    envs = [OracleAviary(task="multihover", num_drones=m, initial_xyzs=xyz, pyb_freq=240, ctrl_freq=30,
                         act="rpm") for _ in range(n_envs)]
    for e in envs:
        e.reset()
    remote.send("ready")
    while True:
        cmd, data = remote.recv()
        if cmd == "step":
            remote.send([step_env_autoreset(env, a) for env, a in zip(envs, data)])
        elif cmd == "close":
            remote.close()
            break


class CpuVecBaseline:
    """The oracle run like the reference's CPU path: spawn workers, Pipes, auto-reset."""

    def __init__(self, n_workers, envs_per_worker, m):
        ctx = mp.get_context("spawn")
        self.n_workers, self.envs_per_worker, self.m = n_workers, envs_per_worker, m
        self.remotes, self.procs = [], []
        for w in range(n_workers):
            parent, child = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(child, envs_per_worker, m, 1000 + w), daemon=True)
            p.start()
            child.close()
            self.remotes.append(parent)
            self.procs.append(p)
        for r in self.remotes:
            assert r.recv() == "ready"
        self.rng = np.random.default_rng(2)

    @property
    def num_envs(self):
        return self.n_workers * self.envs_per_worker

    def step(self):
        acts = self.rng.uniform(-1, 1, (self.num_envs, self.m, 4)).astype(np.float32)
        for r, a in zip(self.remotes, np.array_split(acts, self.n_workers)):
            r.send(("step", a))
        res = [x for r in self.remotes for x in r.recv()]
        obs, rews, dones, infos = zip(*res)
        return np.stack(obs), np.stack(rews), np.stack(dones)

    def close(self):
        for r in self.remotes:
            try:
                r.send(("close", None))
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=5)


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_cpu_baseline(steps: int, warmup: int, m: int, envs_per_worker: int = 4):
    cores = host_cores()
    vec = CpuVecBaseline(cores, envs_per_worker, m)
    try:
        for _ in range(warmup):
            vec.step()
        t0 = time.perf_counter()
        for _ in range(steps):
            vec.step()
        dt = time.perf_counter() - t0
    finally:
        vec.close()
    S = 8
    value = vec.num_envs * m * S * steps / dt
    sample = (f"{vec.num_envs} MultiHover envs x {m} drones ({cores} spawn workers x {envs_per_worker} envs, "
              f"Pipe IPC, auto-reset), {steps} control steps after {warmup} warm-up, fp64 numpy oracle")
    return dict(value=value, unit=UNIT, cores=cores, kind="port", sample=sample), dt / steps * 1e3


# ----------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region — in-process through NVML (nvidia_ml_py), every
    20 ms from a thread.  A child `nvidia-smi -lms 100` (round 1) costs the 20-step window 5 % (36.2 vs 34.5 us per step,
    `scripts/time_window.py`, profiles/README.md); the NVML thread costs nothing measurable.  Falls back to the child
    process when the module is missing."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.rows, self.proc, self.thread, self.nvml = [], None, None, None
        self._stop = threading.Event()
        self.smax = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _poll(self):
        nv = self.nvml
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)), int(get_reasons(self.handle))))
            except Exception:
                pass
            self._stop.wait(self.period)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            sm = [r[0] for r in self.rows]
            reasons = sorted({n for _, m in self.rows for n, bit in self.REASONS if m & bit})
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.smax, "reasons": reasons,
                    "samples": len(sm), "source": f"NVML in-process, every {self.period * 1e3:.0f} ms"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


# --------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from marl_gym_pybullet_drones_b200.batch_aviary import BatchAviary, StepResult

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1 (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from marl_gym_pybullet_drones_b200.dist import bind_host_thread_to_gpu
    # NUMA-local pinned buffers for the host-buffer legs when several ranks share the host (the 1-GPU run keeps every
    # core for the CPU baseline it also times)
    cpus = bind_host_thread_to_gpu(local_rank) if (world > 1 and not os.environ.get("BD_BENCH_NO_BIND")) else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    N, M, S, A, Bf = args.envs_per_gpu, args.drones, 8, 4, 15
    env = BatchAviary(task="multihover", num_envs=N, num_drones=M, initial_xyzs=grid_xyzs(M), pyb_freq=240,
                      ctrl_freq=30, act="rpm", precision="fp32", device=dev, auto_reset=True,
                      reset_mode="jitter_philox", seed=1234 + rank)
    D = env.OBS_DIM
    slots = args.rollout_slots
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    act_pool = (torch.rand((slots, N, M, A), generator=gen, device=dev) * 2 - 1).contiguous()
    obs_buf = torch.empty((slots, N, M, D), dtype=torch.float32, device=dev)
    rew_buf = torch.empty((slots, N), dtype=torch.float32, device=dev)
    term_buf = torch.empty((slots, N), dtype=torch.uint8, device=dev)
    trunc_buf = torch.empty((slots, N), dtype=torch.uint8, device=dev)
    obs_buf.zero_()     # first touch of every slot outside the timed window (the warm-up only reaches W of the slots)
    outs = [StepResult(obs_buf[i], rew_buf[i], term_buf[i].view(torch.bool), trunc_buf[i].view(torch.bool), None)
            for i in range(slots)]
    env.reset_device(out=obs_buf[0])

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def gpu_steps(n, start):
        """n control steps = n launches of the per-step kernel (the one a closed-loop rollout launches), issued with one
        host call per run of consecutive slots (`bd_step_many` in its k-launches mode; step k reads action set
        (start+k) % slots and writes observation slot (start+k) % slots).  The K-steps-in-one-launch kernel, which only
        open-loop action tapes can use, is reported separately (`small_batch`, `open_loop`)."""
        k = 0
        while k < n:
            i = (start + k) % slots
            run = min(n - k, slots - i)
            env.step_many(act_pool[i:i + run], obs_buf[i:i + run], rew_buf[i:i + run], term_buf[i:i + run],
                          trunc_buf[i:i + run], one_launch=False)
            k += run

    # the sampler starts BEFORE the warm-up: its start-up (NVML init) would otherwise leave the GPU idle for a few ms
    # right before the timed window, and a window that follows an idle gap runs ~1 us per step slower (clock ramp)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # pre-warm (untimed, before the W warm-up steps): the process has just initialised CUDA on an idle GPU, and W = 5
    # steps are 0.2 ms of work — not enough for the SM clock to leave its idle state, and too few for the episodes to
    # reach their stationary mix of running / re-spawning envs (nothing terminates in the first ~20 steps after a reset).
    # A step count, not a time: the timed steps then start from the same state in every run (--dump-outputs)
    for k in range(0, args.prewarm_steps, 64):
        gpu_steps(min(64, args.prewarm_steps - k), 0)
        torch.cuda.synchronize(dev)
    gpu_steps(args.warmup, 0)
    # (1) host in the loop: the K launches are issued while the GPU already runs the first ones.  In a 0.7 ms window
    # this adds the host's latency to an idle GPU (~15 us) and whatever jitters the launching thread — 34.9 us per step on
    # one GPU, 38-41 under torchrun with 2-8 ranks, for kernels that take 33.5 on every GPU.  Reported as
    # `host_in_loop_window`.
    sync_all()
    ev0.record()
    gpu_steps(args.steps, args.warmup)
    ev1.record()
    sync_all()
    ms_host = ev0.elapsed_time(ev1)
    # (2) THE TIMED REGION of `value`: the same K launches enqueued behind a gate kernel (bd_stream_gate: one thread
    # spinning on a page-locked flag) that the host opens once all K are queued — exactly K steps between two events on
    # the launching stream, synchronised on both sides, with no host-side gaps in the device timeline; what an
    # asynchronously enqueued rollout sees.
    import ctypes as C
    flag = torch.zeros(1, dtype=torch.int32, pin_memory=True)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    l0 = env.launch_count
    env._lib.bd_stream_gate(C.c_void_p(flag.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    g0.record()
    gpu_steps(args.steps, args.warmup)
    g1.record()
    flag[0] = 1
    sync_all()
    ms = g0.elapsed_time(g1)
    launches = env.launch_count - l0
    dump = None
    if args.dump_outputs and rank == 0:
        # what the last timed step returned, gathered on the device now: the steps below overwrite the rollout slots
        last = (args.warmup + args.steps - 1) % slots
        rows = torch.as_tensor(dump_rows(N, M * D + 3), device=dev)
        dump = {name: buf[last].index_select(0, rows).float() for name, buf in
                (("obs", obs_buf), ("reward", rew_buf), ("terminated", term_buf), ("truncated", trunc_buf))}
    if ms < 300:   # keep the GPU busy a little longer so nvidia-smi sees clocks under load
        t_end = time.time() + 0.4
        while time.time() < t_end:
            gpu_steps(50, 0)
            torch.cuda.synchronize(dev)
    clocks = sampler.stop()

    # ---- e2e: host buffers through bd_step_host (H2D + kernel + D2H + sync per step)
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    host_actions = env.pinned_array((min(slots, 4), N, M, A), np.float32)   # this step's inputs wait in pinned host memory
    host_actions[...] = act_pool[:min(slots, 4)].cpu().numpy()
    for k in range(3):
        env.step_host(host_actions[k % host_actions.shape[0]], actions_pinned=True)
    sync_all()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        res = env.step_host(host_actions[k % host_actions.shape[0]], actions_pinned=True)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    assert np.isfinite(res["reward"]).all()
    h2d = N * M * A * 4
    d2h = N * M * D * 4 + N * 4 + 2 * N

    # ---- what the host side can do at best: the same bytes per step as plain copies (H2D actions, D2H observations),
    # all ranks at the same time — the ceiling the e2e figure is a fraction of (PCIe link on 1 GPU, the host's memory /
    # root-complex bandwidth shared by the ranks on 8)
    pin_obs = torch.empty((N, M, D), dtype=torch.float32, pin_memory=True)
    pin_act = torch.from_numpy(host_actions[0])
    dev_act = torch.empty((N, M, A), dtype=torch.float32, device=dev)
    for _ in range(2):
        dev_act.copy_(pin_act, non_blocking=True)
        pin_obs.copy_(obs_buf[0], non_blocking=True)
    sync_all()
    t0 = time.perf_counter()
    n_copy = 10
    for _ in range(n_copy):
        dev_act.copy_(pin_act, non_blocking=True)
        pin_obs.copy_(obs_buf[0], non_blocking=True)
    torch.cuda.synchronize(dev)
    copy_ms = (time.perf_counter() - t0) * 1e3 / n_copy
    del pin_obs

    # ---- e2e through the reference's VecEnv protocol (what MAPPO.train_step calls): 4-tuple + info dicts
    vec_ms = None
    if args.vecenv_steps > 0:
        from marl_gym_pybullet_drones_b200.vec_env import BatchVecEnv
        venv = BatchVecEnv(env)
        abuf = venv.action_buffer()             # this step's actions wait in pinned host memory, like the e2e leg's
        abuf[...] = host_actions[0]
        for k in range(3):
            venv.step(abuf)
        sync_all()
        t0 = time.perf_counter()
        n_done = 0
        for k in range(args.vecenv_steps):
            o, r_, d_, info = venv.step(abuf)
            n_done += int(d_.sum())
        vec_ms = (time.perf_counter() - t0) * 1e3 / args.vecenv_steps
        first_done = int(np.flatnonzero(d_)[0]) if d_.any() else None
        if first_done is not None:
            assert info["n"][first_done]["terminal_observation"].shape == (M, D)

    # ---- configs[3] as literally sharded: 8192 envs per GPU, launch-bound without bd_step_many
    small = None
    if args.small_envs > 0 and args.small_envs != N:
        Ns = args.small_envs
        env_s = BatchAviary(task="multihover", num_envs=Ns, num_drones=M, initial_xyzs=grid_xyzs(M), pyb_freq=240,
                            ctrl_freq=30, act="rpm", precision="fp32", device=dev, auto_reset=True,
                            reset_mode="jitter_philox", seed=4321 + rank)
        Ks = 256                                # slots: 256 x 8192 x 4 x 72 x 4 B = 2.4 GB of observations (>> L2)
        a_s = (torch.rand((Ks, Ns, M, A), generator=gen, device=dev) * 2 - 1).contiguous()
        o_s = torch.empty((Ks, Ns, M, D), dtype=torch.float32, device=dev)
        r_s = torch.empty((Ks, Ns), dtype=torch.float32, device=dev)
        f_s = torch.empty((2, Ks, Ns), dtype=torch.uint8, device=dev)
        env_s.reset_device(out=o_s[0])
        env_s.step_many(a_s, o_s, r_s, f_s[0], f_s[1])
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 4
        for _ in range(reps):
            env_s.step_many(a_s, o_s, r_s, f_s[0], f_s[1])
        e1.record()
        torch.cuda.synchronize(dev)
        ms_many = e0.elapsed_time(e1) / (reps * Ks)
        out_s = StepResult(o_s[0], r_s[0], f_s[0, 0].view(torch.bool), f_s[1, 0].view(torch.bool), None)
        e0.record()
        for k in range(Ks):
            env_s.step_device(a_s[k], out=out_s)
        e1.record()
        torch.cuda.synchronize(dev)
        ms_single = e0.elapsed_time(e1) / Ks
        bpl = algorithmic_bytes_per_drone_step(A, Bf, M) * Ns * M
        small = {"envs_per_gpu": Ns, "ms_per_step_step_many": ms_many, "ms_per_step_one_call_per_step": ms_single,
                 "value": Ns * M * S / (ms_many * 1e-3), "unit": UNIT,
                 "roofline_frac": bpl / (ms_many * 1e-3) / 1e9 / 6553.0, "steps_per_host_call": Ks,
                 "note": "bd_step_many = ONE launch for the K steps (step_kernel_tile_many: states in registers, action "
                         "history in shared memory across steps); roofline_frac counts the ALGORITHMIC bytes of K single "
                         "steps (state + history re-read every step), of which the one-launch kernel moves only actions, "
                         "observations, rewards and flags"}
        env_s.close()

    # ---- open-loop tapes at the headline size: the K-steps-in-one-launch kernel (not usable by a closed-loop rollout)
    open_loop = None
    if args.open_loop_reps > 0:
        env.step_many(act_pool, obs_buf, rew_buf, term_buf, trunc_buf)          # warm-up (slots steps, one launch)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.open_loop_reps):
            env.step_many(act_pool, obs_buf, rew_buf, term_buf, trunc_buf)
        e1.record()
        torch.cuda.synchronize(dev)
        ms_ol = e0.elapsed_time(e1) / (args.open_loop_reps * slots)
        open_loop = {"ms_per_step": ms_ol, "value": world * N * M * S / (ms_ol * 1e-3), "unit": UNIT, "steps_per_launch": slots,
                     "hbm_bytes_per_step": N * M * (A * 4 + D * 4) + N * 6,
                     "hbm_gbs": (N * M * (A * 4 + D * 4) + N * 6) / (ms_ol * 1e-3) / 1e9,
                     "note": "bd_step_many, one launch per K steps: state and action history never leave the SM between "
                             "steps, so a step moves 304 B per drone (action in, observation row out) instead of 647.5"}

    t = torch.tensor([ms, e2e_s * 1e3, vec_ms if vec_ms is not None else 0.0, copy_ms, ms_host], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max, vec_ms_max, copy_ms_max, ms_host_max = float(t[0]), float(t[1]), float(t[2]), float(t[3]), float(t[4])
    units = world * N * M * S
    value = units * args.steps / (ms_max * 1e-3)
    e2e_value = units * e2e_steps / (e2e_ms_max * 1e-3)

    bytes_per_drone_step = algorithmic_bytes_per_drone_step(A, Bf, M)
    bytes_per_launch = bytes_per_drone_step * N * M
    kernel_ms = ms / max(launches, 1)
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"])
            peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        pass
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            with open(tpath) as f:
                tj = json.load(f)
            if tj.get("envs_per_gpu") == N and tj.get("drones") == M:
                traffic = tj.get("dram_bytes_per_launch")
        except Exception:
            pass

    line = None
    if rank == 0:
        cpu = None
        if world == 1:
            cpu, _ = run_cpu_baseline(args.cpu_steps, 2, M)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": (f"BASELINE configs[3]: MultiHoverAviary M={M} CF2X Physics.DYN 240Hz/30Hz KIN obs RPM "
                             f"action, {N} envs per GPU x {world} GPU(s), auto-reset, U(-1,1) actions"),
                "envs_per_gpu": N, "drones_per_env": M, "substeps_per_step": S, "obs_dim": D,
                "l2_policy": (f"inputs larger than L2: obs written to a {slots}-slot rotating rollout buffer "
                              f"({slots * N * M * D * 4 / 1e6:.0f} MB) + {slots}-slot action pool; state+history "
                              f"{(N * M * (64 + Bf * A * 4)) / 1e6:.0f} MB"),
                "parallelism": f"env-sharded x{world}, no data-path collective",
                "prewarm": f"{args.prewarm_steps} untimed steps before the {args.warmup} warm-up steps (SM clock out of idle, "
                           "episodes in their stationary running / re-spawning mix)",
                "timed_region": "K launches of the per-step kernel between two CUDA events on the launching stream, enqueued "
                                "behind a gate kernel the host opens when all K are queued (no host-side gaps), synchronised "
                                "(+ barrier) on both sides, max over ranks",
                "host_cpus_rank0": (f"{len(cpus)} CPUs near the GPU (NVML affinity)" if cpus else
                                    f"{host_cores()} (container cpuset; NVML affinity not applicable)")},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "traffic_source": "profiles/traffic.json: one isolated `ncu --set full` launch of this kernel "
                                           "(not measured in this run)" if traffic is not None else None,
                         "peak_source": peak_src,
                         "kernel": "bd::step_kernel_tile<MULTIHOVER,4,4,false>",
                         "algorithmic_bytes_per_launch": bytes_per_launch,
                         "algorithmic_bytes_per_drone_substep": bytes_per_drone_step / S,
                         "kernel_ms": kernel_ms},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "api": "BatchAviary.step_host -> bd_step_host (pinned numpy in/out)",
                    # the e2e path is bound by the host link, not by HBM: its own roofline
                    "roofline": {"bound": "host link (PCIe / host memory shared by the ranks)",
                                 "achieved": world * (h2d + d2h) / (e2e_ms_max / e2e_steps * 1e-3) / 1e9,
                                 "peak": world * (h2d + d2h) / (copy_ms_max * 1e-3) / 1e9, "unit": "GB/s",
                                 "frac": copy_ms_max / (e2e_ms_max / e2e_steps),
                                 "peak_source": "measured in this run: the same bytes per step as plain cudaMemcpyAsync "
                                                "copies from / to pinned memory, all ranks concurrently"}},
            "gpu_launches": int(launches),
            "host_in_loop_window": {"ms_per_step": ms_host_max / args.steps,
                                    "roofline_frac": bytes_per_launch / (ms_host_max / args.steps * 1e-3) / 1e9 / peak,
                                    "note": "the same K launches issued while the GPU runs (no gate): adds the host's latency "
                                            "to an idle GPU and launch-thread jitter to the device timeline"},
            "clocks": clocks,
        }
        if vec_ms is not None:
            line["e2e_vecenv"] = {"value": units / (vec_ms_max * 1e-3), "unit": UNIT, "ms_per_step": vec_ms_max,
                                  "ms_per_step_bd_step_host": e2e_ms_max / e2e_steps,
                                  "ratio_to_bd_step_host": vec_ms_max / (e2e_ms_max / e2e_steps),
                                  "steps": args.vecenv_steps,
                                  "api": "BatchVecEnv.step -> bd_step_host_compact (4-tuple, lazy info dicts, terminal "
                                         "observations of finished envs only)"}
        if small is not None:
            line["small_batch"] = small
        if open_loop is not None:
            line["open_loop"] = open_loop
    env.close()
    mappo = None
    if args.mappo_steps > 0:
        mappo = run_mappo_block(args, dev, rank, world)
    if line is not None and mappo is not None:
        line["mappo"] = mappo
    if dump is not None:
        write_outputs(args.dump_outputs, {name: t.cpu().numpy() for name, t in dump.items()})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)


def run_mappo_block(args, dev, rank, world):
    """`DeviceMAPPO.train_step` at BASELINE configs[4]'s per-GPU shape: 16-drone MultiHover with downwash, one epoch of
    large minibatches; every hot operation is one of this repo's kernels (step, fused actor, GAE scan, fused PPO
    update), the gradient all-reduce is NCCL.  Weak scaling: every rank owns `--mappo-envs` envs."""
    import torch
    import torch.distributed as dist
    from marl_gym_pybullet_drones_b200.batch_aviary import BatchAviary
    from marl_gym_pybullet_drones_b200.mappo import DeviceMAPPO
    N, M, T = args.mappo_envs, args.mappo_drones, args.mappo_rollout
    side = int(np.ceil(np.sqrt(M)))
    # 1 m grid centred on the origin (inside MultiHover's |x|, |y| <= 3 m box): the re-spawn rule redraws the +-0.25 m
    # jitter until all drones are 0.5 m apart (MultiHoverAviary.py:83-102) — a 0.6 m grid makes most draws fail and the
    # rollout spends more time in the retry loop than in the dynamics (92 ms vs 38 ms per 32-step rollout)
    xyz = np.array([[float(i % side) - 0.5 * (side - 1), float(i // side) - 0.5 * (side - 1), 0.5 + 0.05 * (i % 3)]
                    for i in range(M)])
    env = BatchAviary(task="multihover", num_envs=N, num_drones=M, initial_xyzs=xyz, physics="dyn_dw", precision="fp32",
                      device=dev, auto_reset=True, reset_mode="jitter_philox", seed=99 + rank, track_episode_stats=True)
    mb = max(1, (N * T) // args.mappo_minibatches)
    algo = DeviceMAPPO(env, seed=0, rollout_steps=T, hidden_dim=256, mini_batch_size=mb, opt_epochs=1,
                       update_impl="native", graph_update=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def step():
        ev[0].record()
        algo.collect_rollout()
        ev[1].record()
        algo.compute_returns()
        ev[2].record()
        res = algo.update()
        ev[3].record()
        torch.cuda.synchronize(dev)
        return res, [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
    step()                                  # warm-up: graph capture, allocator
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    tot = np.zeros(3)
    t0 = time.perf_counter()
    for _ in range(args.mappo_steps):
        res, parts = step()
        tot += parts
    wall_ms = (time.perf_counter() - t0) * 1e3 / args.mappo_steps
    parts_ms = tot / args.mappo_steps
    ar_us = nccl_us = None
    peer = getattr(algo, "_peer", None)
    if world > 1:                           # the collective that defines the multi-GPU design, timed on its own
        def timed(fn):
            for _ in range(5):
                fn()
            torch.cuda.synchronize(dev)
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(50):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / 50 * 1e3
        g = algo._joint_grad
        kl = algo.actor_net.stats[1:3]
        g2 = torch.zeros_like(g)            # NCCL on the same sizes (what the peer kernel replaces): gradients + KL pair
        nccl_us = timed(lambda: (dist.all_reduce(g2), dist.all_reduce(kl)))
        ar_us = timed(lambda: peer.all_reduce(extra=kl)) if peer is not None else nccl_us
    t = torch.tensor([wall_ms, parts_ms[0], parts_ms[1], parts_ms[2]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall_ms, r_ms, g_ms, u_ms = [float(x) for x in t]
    launches = env.launch_count + (algo.fused.launch_count if algo.fused is not None else 0) + \
        algo.actor_net.launch_count + algo.critic_net.launch_count
    n_mb = (N * T) // mb
    out = {"metric": "mappo_env_steps_per_sec", "value": world * N * T / (wall_ms * 1e-3), "unit": "env-steps/s",
           "drone_substeps_per_sec": world * N * M * 8 * T / (wall_ms * 1e-3),
           "train_step_ms": wall_ms, "rollout_ms": r_ms, "returns_ms": g_ms, "update_ms": u_ms,
           "shares": {"rollout": r_ms / wall_ms, "returns": g_ms / wall_ms, "update": u_ms / wall_ms},
           "config": {"workload": f"BASELINE configs[4] per-GPU shape: MultiHover M={M} + downwash, {N} envs per GPU x {world}, "
                                  f"rollout {T} steps, 1 epoch x {n_mb} minibatches of {mb} env-steps ({mb * M} actor rows)",
                      "update_impl": "native (bd_ppo.cu): tcgen05 fwd+bwd tile kernel, tcgen05 weight-gradient kernel, "
                                     "GAE scan, gated Adam; one CUDA graph per epoch" +
                                     ((", gradient + KL all-reduce as one NVLink peer-memory kernel per minibatch in the graph (bd_peer.cu)"
                                       if peer is not None else ", NCCL all-reduces in the graph") if world > 1 else "")},
           "collectives_per_train_step": {"gradient_allreduce": n_mb if world > 1 else 0,
                                          "kl_pair_allreduce": (0 if peer is not None else n_mb) if world > 1 else 0},
           "gradient_allreduce_impl": (("peer-memory kernel (bd_peer_allreduce), gradients + KL pair in one launch" if peer is not None
                                        else "NCCL, two calls") if world > 1 else None),
           "gradient_allreduce_us": ar_us,
           "nccl_same_sizes_us": nccl_us,
           "gradient_allreduce_share": (n_mb * ar_us * 1e-3 / wall_ms) if ar_us is not None else 0.0,
           "limiting_collective": ("joint actor+critic flat-gradient all-reduce (342 KB + 1.4 MB fp32 in one buffer), "
                                   "latency-bound" if world > 1 else None),
           "gpu_launches_total": int(launches), "policy_loss": res["policy_loss"], "approx_kl": res["approx_kl"]}
    algo.close()
    env.close()
    return out if rank == 0 else None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    M = args.drones
    cpu, ms_step = run_cpu_baseline(args.steps, args.warmup, M)
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT,
        "n_gpus": int(os.environ.get("WORLD_SIZE", str(args.gpus))), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": (f"BASELINE configs[3]: MultiHoverAviary M={M} CF2X Physics.DYN 240Hz/30Hz KIN obs RPM "
                                f"action; bounded sample on host cores: {cpu['sample']}")},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--drones", type=int, default=4)
    ap.add_argument("--rollout-slots", type=int, default=16)
    ap.add_argument("--open-loop-reps", type=int, default=8, help="timed bd_step_many launches of the open-loop leg (0 = skip)")
    ap.add_argument("--prewarm-steps", type=int, default=9216,
                    help="untimed steps before the W warm-up steps (the default is about 0.3 s on one B200)")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--cpu-steps", type=int, default=200)
    ap.add_argument("--vecenv-steps", type=int, default=20, help="steps of the VecEnv-protocol e2e leg (0 = skip)")
    ap.add_argument("--small-envs", type=int, default=8192, help="envs per GPU of the small-batch leg (0 = skip)")
    ap.add_argument("--mappo-steps", type=int, default=2, help="timed train steps of the MAPPO block (0 = skip)")
    ap.add_argument("--mappo-envs", type=int, default=131072)
    ap.add_argument("--mappo-drones", type=int, default=16)
    ap.add_argument("--mappo-rollout", type=int, default=32)
    ap.add_argument("--mappo-minibatches", type=int, default=128)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (obs, reward, terminated, truncated of rank 0) as "
                         "DIR/<name>.npy in float32; a fixed seeded sample of the envs when they exceed 64 MB. The inputs "
                         "are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the GPU path (--impl ours)")
    if args.impl == "reference":
        args.steps = 24 if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else args.warmup
        run_reference(args)
    else:
        args.steps = 1000 if args.steps is None else args.steps
        args.warmup = 100 if args.warmup is None else max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    # stdout carries exactly ONE line, the JSON result: anything libraries print on file descriptor 1 meanwhile
    # (e.g. NCCL's version banner) goes to stderr instead
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_real_stdout, "w", buffering=1)
    main()
