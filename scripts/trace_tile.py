"""Phase timeline of the training tile kernel (mlp_tile_kernel, actor minibatch of 32 768 x 4 rows): SM-clock stamps of
CTA 0's epilogue thread 0 per tile (bd_ppo_set_trace).      python scripts/trace_tile.py [--critic]"""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import test_gpu_ppo_kernels as t  # noqa: E402
from marl_gym_pybullet_drones_b200.ppo_native import PpoNet  # noqa: E402

critic = "--critic" in sys.argv
M, D, A, samples = 4, 72, 4, 32768
T, N = 32, 2048
obs, act, g = t._rollout(T, N, M, D, A, 7)
logp_old = torch.randn((T, N, M), device="cuda", generator=g) * 0.1 - 3
adv = torch.randn((T, N), device="cuda", generator=g)
ret = torch.randn((T, N), device="cuda", generator=g)
stats2 = torch.tensor([0.0, 1.0], device="cuda")
idx = torch.randperm(T * N, device="cuda", generator=g)[:samples].contiguous()
if critic:
    net = PpoNet(D, M, 1, False, samples)
    net.pack(t._flat(list(t._mlp(M * D, 1, 3).parameters())))
else:
    net = PpoNet(D, 1, A, True, samples * M)
    net.pack(t._flat([torch.full((A,), -0.5, device="cuda")] + list(t._mlp(D, A, 6).parameters())))
gr = torch.zeros(net.param_count, device="cuda")


def one():
    if critic:
        net.grad(gr, obs, N, M, idx, samples, critic=True, ret=ret)
    else:
        net.grad(gr, obs, N, M, idx, samples, critic=False, act=act, logp_old=logp_old, adv=adv, adv_stats=stats2, clip=0.2,
                 entropy_coef=0.005)


for _ in range(3):
    one()
torch.cuda.synchronize()
trace = torch.zeros((16, 16), dtype=torch.int64, device="cuda")
net._check(net._lib.bd_ppo_set_trace(net._h, C.c_void_p(trace.data_ptr())), "bd_ppo_set_trace")
one()
torch.cuda.synchronize()
net._lib.bd_ppo_set_trace(net._h, None)
tr = trace.cpu().numpy()
names = ["tile start", "inputs staged", "L1 complete", "H1 written", "L2 complete", "H2 written", "L3 complete", "loss done",
         "dH2 complete", "dZ2 written", "dH1 complete", "dZ1 written", "(loss inputs in)", "(dZ3 handed over)"]
rows = [j for j in range(16) if tr[j, 0] != 0]
for j in rows[:3] + rows[-1:]:
    print(f"tile {j} of CTA 0 (cycles since it started, delta)")
    prev = tr[j, 0]
    for k, nme in sorted(enumerate(names), key=lambda kn: tr[j, kn[0]]):
        if tr[j, k]:
            print(f"   {nme:14s} {tr[j, k] - tr[j, 0]:8d}  +{tr[j, k] - prev:6d}")
            prev = tr[j, k]
if len(rows) > 2:
    per = (tr[rows[-1], 0] - tr[rows[1], 0]) / (len(rows) - 2)
    print("cycles per tile (steady):", per)
