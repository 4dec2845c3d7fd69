"""Timing of the fused tcgen05 actor forward vs torch (fp32 and bf16 autocast) on the same rows."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from marl_gym_pybullet_drones_b200.actor import FusedActor  # noqa: E402
from marl_gym_pybullet_drones_b200.mappo import MLP  # noqa: E402

rows = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
mlp = MLP(72, 4, [256, 256], "tanh").cuda()
logstd = torch.full((4,), -0.5, device="cuda")
obs = torch.randn(rows, 72, device="cuda")
fa = FusedActor(72, 256, 4)
fa.set_weights(mlp, logstd)
act = torch.empty(rows, 4, device="cuda")
lp = torch.empty(rows, device="cuda")


def timeit(fn, n=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n


flops = rows * 2.0 * (72 * 256 + 256 * 256 + 256 * 4)
t = timeit(lambda: fa.forward(obs, out_act=act, out_logp=lp))
print(f"fused tcgen05 actor : {t:8.1f} us  {flops / t / 1e6:7.1f} TFLOP/s (useful flops)")
from marl_gym_pybullet_drones_b200.ppo_native import PpoNet  # noqa: E402
net = PpoNet(72, 1, 4, True, 128)
net.pack(torch.cat([logstd] + [p.detach().reshape(-1) for p in mlp.parameters()]).contiguous())
obs3 = obs.view(rows // 4, 4, 72)
t2 = timeit(lambda: net.sample(obs3, act, lp, seed=1, offset=2))
print(f"two-tile tcgen05 sample: {t2:8.1f} us  {flops / t2 / 1e6:7.1f} TFLOP/s (useful flops)  [bd_ppo_sample]")
out = torch.empty(rows, 4, device="cuda")
t3 = timeit(lambda: net.forward(obs3, rows // 4, 4, rows, out=out))
print(f"two-tile tcgen05 forward: {t3:8.1f} us  [bd_ppo_forward]")
cn = PpoNet(72, 4, 1, False, 128)
cm = MLP(4 * 72, 1, [256, 256], "tanh").cuda()
cn.pack(torch.cat([p.detach().reshape(-1) for p in cm.parameters()]).contiguous())
val = torch.empty(rows // 4, 1, device="cuda")
t4 = timeit(lambda: cn.forward(obs3, rows // 4, 4, rows // 4, out=val))
print(f"two-tile critic values ({rows // 4} rows x 4 chunks): {t4:8.1f} us")
if "--short" in sys.argv:
    sys.exit(0)
with torch.no_grad():
    def torch_fp32():
        m = mlp(obs)
        n = torch.randn_like(m)
        return m + logstd.exp() * n
    t32 = timeit(torch_fp32)
    print(f"torch fp32 MLP+sample: {t32:8.1f} us  {flops / t32 / 1e6:7.1f} TFLOP/s")
    torch.backends.cuda.matmul.allow_tf32 = True
    ttf = timeit(torch_fp32)
    print(f"torch tf32 MLP+sample: {ttf:8.1f} us  {flops / ttf / 1e6:7.1f} TFLOP/s")

    def torch_bf16():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            m = mlp(obs)
        n = torch.randn_like(m, dtype=torch.float32)
        return m.float() + logstd.exp() * n
    tb = timeit(torch_bf16)
    print(f"torch bf16 autocast  : {tb:8.1f} us  {flops / tb / 1e6:7.1f} TFLOP/s")
