"""Time of a simulator snapshot save, full restore and masked restore (half the envs), DESIGN.md section 4.

For each shape: one aviary, two snapshot buffers used in rotation (together larger than the L2 at the default shapes),
warm-up, then --n calls of each kind.
  call time     CUDA events around --n back-to-back calls (a restore includes its header round trip: a 256-byte copy
                to the host and a stream synchronisation before the unpack launch)
  kernel time   device duration of the snapshot kernel, from a separate torch.profiler run of --n calls
  GB/s          bytes the kernel reads + writes (planes only, no padding) over kernel time, against --peak GB/s

    python scripts/time_snapshot.py [--n 100] [--out profiles/snapshot_times.txt]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from marl_gym_pybullet_drones_b200.batch_aviary import BatchAviary  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=100, help="calls per kind (rotating two snapshot buffers)")
ap.add_argument("--peak", type=float, default=6553.0, help="HBM bandwidth to compare with, GB/s (measured copy rate)")
ap.add_argument("--out", default=None, help="also write the report to this file")
args = ap.parse_args()

if not torch.cuda.is_available():
    raise SystemExit("time_snapshot.py needs a CUDA device")

SHAPES = [  # (label, BatchAviary keywords)
    ("65536 x 4 fp32", dict(num_envs=65536, num_drones=4, physics="dyn")),
    ("131072 x 16 fp32 downwash", dict(num_envs=131072, num_drones=16, physics="dyn_dw")),
]

lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def payload_bytes(env):
    """Bytes of state the snapshot carries (the planes without their 256-byte padding)."""
    n = env.num_envs * env.NUM_DRONES
    real = 8 if env.precision == "fp64" else 4
    b = n * 16 * real + n * env.ACTION_BUFFER_SIZE * env.ACTION_DIM * 4 + env.num_envs * 4
    if env._cfg.keep_ang_vel:
        b += n * 4 * real
    if env._cfg.act_type >= 2:
        b += n * 13 * real
    if env._cfg.track_episodes:
        b += env.num_envs * 4
    return b


def kernel_us(fn, n):
    """Mean device time of the snapshot kernel over n calls of fn (torch.profiler, CUDA activities)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
    ts = [e.time_range.elapsed_us() for e in prof.events()
          if e.device_type == DeviceType.CUDA and "snapshot_kernel" in e.name]
    if len(ts) != n:
        raise RuntimeError(f"expected {n} snapshot kernels in the trace, found {len(ts)}")
    return float(np.mean(ts))


def call_us(fn, n):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n


q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                    str(torch.cuda.current_device())], capture_output=True, text=True)
say(f"device: {torch.cuda.get_device_name()} | nvidia-smi: {q.stdout.strip() or 'n/a'}")
say(f"{args.n} calls per kind, two snapshot buffers in rotation; GB/s = (read + write bytes) / kernel time; "
    f"peak {args.peak:.0f} GB/s")
for label, kw in SHAPES:
    env = BatchAviary(task="multihover", act="rpm", seed=1, track_episode_stats=True, **kw)
    N = env.num_envs
    gen = torch.Generator(device="cuda").manual_seed(0)
    act = torch.rand((N, env.NUM_DRONES, env.ACTION_DIM), device="cuda", generator=gen) * 2 - 1
    for _ in range(20):
        env.step_device(act)
    bufs = [env.snapshot(), env.snapshot()]
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[torch.randperm(N, device="cuda", generator=gen)[:N // 2]] = 1
    nb, pb = env.snapshot_nbytes, payload_bytes(env)
    kinds = [
        ("save", lambda i: env.snapshot(out=bufs[i & 1]), 2 * pb),
        ("full restore", lambda i: env.restore(bufs[i & 1]), 2 * pb),
        ("masked restore (N/2)", lambda i: env.restore(bufs[i & 1], env_mask=mask), pb + N),
    ]
    say(f"\n{label}: snapshot {nb / 1e6:.1f} MB ({pb / 1e6:.1f} MB of planes)")
    for name, fn, moved in kinds:
        call_us(fn, 10)                      # warm-up
        c = call_us(fn, args.n)
        k = kernel_us(fn, args.n)
        gbs = moved / (k * 1e-6) / 1e9
        say(f"  {name:22s} call {c:8.1f} us   kernel {k:8.1f} us   {moved / 1e6:7.1f} MB moved   "
            f"{gbs:7.0f} GB/s = {100 * gbs / args.peak:5.1f} % of {args.peak:.0f}")
    env.close()
    del bufs, act, mask
    torch.cuda.empty_cache()

if args.out:
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
