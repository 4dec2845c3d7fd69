"""L2 residency plan of the fast step kernel (DESIGN.md section 4): the budget rule (host only) and, on the GPU,
bit-identical results under every eviction policy — the hints may only change where bytes come from."""
import ctypes as C
import os
import shutil

import numpy as np
import pytest

from marl_gym_pybullet_drones_b200 import _native
from marl_gym_pybullet_drones_b200 import build as bd_build

L2_B200 = 126 * 2**20     # cudaDevAttrL2CacheSize of a B200
BD_EINVAL = -1


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_native.LIB_PATH) or not bd_build.up_to_date():
        if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
            pytest.skip("nvcc not available and library not prebuilt")
        bd_build.build()
    return _native.load()


def plan(lib, n_envs, n_drones, force=None, act_dim=4, buf_slots=15, track=1, l2=L2_B200):
    s, k = C.c_int(-1), C.c_int(-1)
    rc = lib.bd_l2_plan(n_envs, n_drones, act_dim, buf_slots, track, l2, force.encode() if force is not None else None,
                        C.byref(s), C.byref(k))
    return rc, s.value, k.value


def test_budget_keeps_state_first_then_fewer_slots_as_n_grows(lib):
    prev = None
    for n_envs in (8192, 16384, 32768, 65536, 98304, 131072):
        rc, s, k = plan(lib, n_envs, 4)
        assert rc == 0
        assert s == 1, n_envs                    # the state comes first ...
        assert 0 <= k <= 14
        if prev is not None:
            assert k <= prev, (n_envs, k, prev)  # ... the slots shrink with the drone count
        prev = k
    assert plan(lib, 8192, 4)[2] == 14            # a small batch keeps the whole ring
    # the headline shape: state (16.8 MB) plus what fits of the ring (4.2 MB per slot)
    rc, s, k = plan(lib, 65536, 4)
    assert (s, k) == (1, 5)
    assert plan(lib, 131072, 4)[1:] == (1, 0)     # 34 MB of state: the state alone


def test_budget_switches_off_when_the_state_does_not_fit(lib):
    assert plan(lib, 131072, 16) == (0, 0, 0)     # the 16-drone swarm configuration: 134 MB of state
    assert plan(lib, 262144, 4) == (0, 0, 0)      # 1 M drones: 67 MB of state
    assert plan(lib, 65536, 4, l2=0) == (0, 0, 0)
    # A = 1 actions: a ring slot is 4 bytes per drone
    rc, s, k = plan(lib, 65536, 4, act_dim=1)
    assert rc == 0 and s == 1 and k > plan(lib, 65536, 4)[2]


def test_override(lib):
    assert plan(lib, 65536, 4, "off") == (0, 0, 0)
    assert plan(lib, 65536, 4, "state") == (0, 1, 0)
    assert plan(lib, 65536, 4, "7") == (0, 1, 7)
    assert plan(lib, 65536, 4, "0") == (0, 1, 0)
    assert plan(lib, 65536, 4, "99") == (0, 1, 14)          # at most B - 1 slots are ever read again
    assert plan(lib, 131072, 16, "state") == (0, 1, 0)      # the override ignores the budget (A/B runs)
    assert plan(lib, 65536, 4, "") == plan(lib, 65536, 4)   # empty: the budget rule
    for bad in ("all", "-1", "3x"):
        assert plan(lib, 65536, 4, bad)[0] == BD_EINVAL, bad


@pytest.mark.gpu
@pytest.mark.parametrize("N,T", [(65536, 400), (70001, 300)])
def test_every_l2_policy_gives_bit_identical_results(monkeypatch, N, T):
    """Several hundred pipelined steps with crashes and re-spawns, a foreign kernel producing some of the actions,
    at the headline shape and a ragged size: state, action ring (the history columns of the observation rows),
    observations, rewards, flags and episode statistics are bit-identical under every policy."""
    import torch
    from marl_gym_pybullet_drones_b200.batch_aviary import BatchAviary, StepResult
    M = 4
    xyz = np.array([[-0.5, -0.5, 0.5], [0.5, -0.5, 0.5], [-0.5, 0.5, 0.5], [0.5, 0.5, 0.5]])
    gen = torch.Generator(device="cuda").manual_seed(5)
    acts = torch.rand((8, N, M, 4), device="cuda", generator=gen) * 2 - 1.3      # descending: crashes and re-spawns
    results = []
    for policy, want in (("off", (0, 0)), ("state", (1, 0)), ("1", (1, 1)), ("7", (1, 7)), ("14", (1, 14))):
        monkeypatch.setenv("BD_L2_KEEP", policy)
        env = BatchAviary(task="multihover", num_envs=N, num_drones=M, initial_xyzs=xyz, seed=3, track_episode_stats=True,
                          precision="fp32", physics="dyn", action_dtype=torch.float32)
        s, k = C.c_int(-1), C.c_int(-1)
        assert env._lib.bd_l2_policy(env._h, C.byref(s), C.byref(k)) == 0
        assert (s.value, k.value) == want, policy
        out = StepResult(torch.empty((N, M, env.OBS_DIM), device="cuda"), torch.empty(N, device="cuda"),
                         torch.empty(N, dtype=torch.bool, device="cuda"), torch.empty(N, dtype=torch.bool, device="cuda"), None)
        env.reset_device()
        rsum = torch.zeros((), dtype=torch.float64, device="cuda")
        flags = torch.zeros(2, dtype=torch.int64, device="cuda")
        for t in range(T):
            if t % 10 == 9:    # actions written by a kernel enqueued right before the step
                env.step_device(torch.tanh(out.obs[:, :, 6:10] * 0.5) - 0.3, out=out)
            else:
                env.step_device(acts[t % 8], out=out)
            rsum += out.reward.double().sum()
            flags[0] += out.terminated.sum()
            flags[1] += out.truncated.sum()
        torch.cuda.synchronize()
        results.append((env.get_state(with_step_counter=True), out.obs.cpu(), out.reward.cpu(), out.terminated.cpu(),
                        out.truncated.cpu(), rsum.item(), flags.cpu(), env.episode_stats().cpu()))
        env.close()
    ref = results[0]
    assert ref[6][0] + ref[6][1] > N                         # many episodes ended and were re-spawned on the way
    for r in results[1:]:
        for x, y in zip(ref[0], r[0]):                     # drone state vectors, step counters
            assert torch.equal(x.cpu().nan_to_num(7.0), y.cpu().nan_to_num(7.0))
        assert torch.equal(ref[1], r[1]) and torch.equal(ref[2], r[2])
        assert torch.equal(ref[3], r[3]) and torch.equal(ref[4], r[4])
        assert ref[5] == r[5] and torch.equal(ref[6], r[6]) and torch.equal(ref[7], r[7])
