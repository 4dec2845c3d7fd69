"""Step time of the fast kernel under each L2 residency policy (BD_L2_KEEP, DESIGN.md section 4).

For every size, rounds of: one handle per policy (the policy is read when the handle is created), warm-up, then
--n back-to-back launches between two CUDA events.  Actions and observation rows rotate through --slots buffers
(larger than the L2 at the sizes of interest, as in bench.py), so only the state and ring can be re-read from L2.
Policies alternate within a round; the median and range over the rounds are printed per (size, policy).

    python scripts/time_l2_policy.py --envs 65536 32768 --policies off state 1 2 4 7 14 default
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctypes as C  # noqa: E402

from marl_gym_pybullet_drones_b200.batch_aviary import BatchAviary, StepResult  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--envs", type=int, nargs="+", default=[65536])
ap.add_argument("--drones", type=int, default=4)
ap.add_argument("--policies", nargs="+", default=["off", "state", "1", "2", "4", "7", "14", "default"],
                help="BD_L2_KEEP values; 'default' = the budget rule")
ap.add_argument("--slots", type=int, default=16)
ap.add_argument("--n", type=int, default=1000)
ap.add_argument("--rounds", type=int, default=3)
args = ap.parse_args()

M = args.drones
side = int(np.ceil(np.sqrt(M)))
xyz = np.array([[float(i % side), float(i // side), 0.5] for i in range(M)])
print(torch.cuda.get_device_name(), flush=True)
for N in args.envs:
    times = {p: [] for p in args.policies}
    plan = {}
    S = args.slots
    gen = torch.Generator(device="cuda").manual_seed(0)
    acts = torch.rand((S, N, M, 4), device="cuda", generator=gen) * 2 - 1
    obs = torch.empty((S, N, M, 12 + 15 * 4), device="cuda")
    rew = torch.empty((S, N), device="cuda")
    te = torch.empty((S, N), dtype=torch.bool, device="cuda")
    tr = torch.empty((S, N), dtype=torch.bool, device="cuda")
    outs = [StepResult(obs[i], rew[i], te[i], tr[i], None) for i in range(S)]
    for _ in range(args.rounds):
        for p in args.policies:
            if p == "default":
                os.environ.pop("BD_L2_KEEP", None)
            else:
                os.environ["BD_L2_KEEP"] = p
            env = BatchAviary(task="multihover", num_envs=N, num_drones=M, initial_xyzs=xyz, auto_reset=True, seed=1,
                              track_episode_stats=True, action_dtype=torch.float32)
            ks, kk = C.c_int(), C.c_int()
            env._lib.bd_l2_policy(env._h, C.byref(ks), C.byref(kk))
            plan[p] = (ks.value, kk.value)
            env.reset_device(out=obs[0])
            for k in range(300):
                env.step_device(acts[k % S], out=outs[k % S])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(args.n):
                env.step_device(acts[k % S], out=outs[k % S])
            e1.record()
            torch.cuda.synchronize()
            times[p].append(e0.elapsed_time(e1) * 1e3 / args.n)
            env.close()
    os.environ.pop("BD_L2_KEEP", None)
    for p in args.policies:
        t = np.array(times[p])
        print(f"envs {N:7d} x {M}  BD_L2_KEEP={p:8s} plan (state {plan[p][0]}, slots {plan[p][1]:2d})  "
              f"median {np.median(t):6.2f} us/step  [{t.min():6.2f} .. {t.max():6.2f}]", flush=True)
    del acts, obs, rew, te, tr, outs
    torch.cuda.empty_cache()
