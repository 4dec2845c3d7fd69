"""Phase timeline of the two-tiles-in-flight forward kernel (mlp_fwd2_kernel): SM-clock stamps of CTA 0's epilogue
thread 0 and MMA thread per tile pair (bd_ppo_set_trace).

    python scripts/trace_fwd2.py [rows]
"""
import ctypes as C
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from marl_gym_pybullet_drones_b200.mappo import MLP  # noqa: E402
from marl_gym_pybullet_drones_b200.ppo_native import PpoNet  # noqa: E402

rows = int(sys.argv[1]) if len(sys.argv) > 1 and sys.argv[1].isdigit() else 262144
mlp = MLP(72, 4, [256, 256], "tanh").cuda()
logstd = torch.full((4,), -0.5, device="cuda")
obs = torch.randn(rows // 4, 4, 72, device="cuda")
net = PpoNet(72, 1, 4, True, 128)
net.pack(torch.cat([logstd] + [p.detach().reshape(-1) for p in mlp.parameters()]).contiguous())
act = torch.empty(rows, 4, device="cuda")
lp = torch.empty(rows, device="cuda")
for _ in range(3):
    net.sample(obs, act, lp, seed=1, offset=2)
torch.cuda.synchronize()
trace = torch.zeros((32, 64), dtype=torch.int64, device="cuda")
net._check(net._lib.bd_ppo_set_trace(net._h, C.c_void_p(trace.data_ptr())), "bd_ppo_set_trace")
net.sample(obs, act, lp, seed=1, offset=2)
torch.cuda.synchronize()
net._lib.bd_ppo_set_trace(net._h, None)
t = trace.cpu().numpy()
pairs = [j for j in range(32) if t[j, 0] != 0]
t0 = t[pairs[0], 0]
E = ["start", "L1A done", "H1A done", "XA' staged", "L1B done", "H1B done", "XB' staged", "L2A done", "H2A done", "-",
     "L2B done", "H2B done", "-", "L3A done", "outA done", "L3B done", "outB done"]
Mn = ["start", "OUT A ok", "OUT B ok", "L1A issued", "L1B issued", "H1A ready", "H1B ready", "L2A issued", "L2B issued", "H2A ready",
      "H2B ready", "L3A issued", "L3B issued"]
for j in pairs[:4] + pairs[-2:]:
    print(f"pair {j}: epilogue thread (cycles since kernel start, delta)")
    prev = t[j, 0]
    for k, name in enumerate(E):
        if t[j, k] and name != "-":
            print(f"   {name:12s} {t[j, k] - t0:8d}  +{t[j, k] - prev:6d}")
            prev = t[j, k]
    print(f"pair {j}: MMA thread")
    prev = t[j, 32]
    for k, name in enumerate(Mn):
        if t[j, 32 + k]:
            print(f"   {name:12s} {t[j, 32 + k] - t0:8d}  +{t[j, 32 + k] - prev:6d}")
            prev = t[j, 32 + k]
if len(pairs) > 2:
    print("cycles per pair (steady):", (t[pairs[-2], 0] - t[pairs[1], 0]) / (len(pairs) - 3))
