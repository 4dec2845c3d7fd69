"""Simulator snapshots (`bd_save_snapshot` / `bd_load_snapshot`, `BatchAviary.snapshot` / `restore`) and the
trainer checkpoints built on them (`DeviceMAPPO(save_env_state=True)`).

A restored handle must continue bit for bit like the one the snapshot was taken from, whatever its own seed and step
count were: the ring is stored by age, the Philox key and counter travel in the header."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GRID = np.array([[0.0, 0.0, 0.5], [1.0, 0.0, 0.5], [0.0, 1.0, 0.5], [1.0, 1.0, 0.5], [0.5, 0.5, 0.7]])


def _aviary(**kw):
    from marl_gym_pybullet_drones_b200 import BatchAviary
    M = kw.get("num_drones", 1)
    if "initial_xyzs" not in kw and kw.get("task") != "spiral":
        if M <= len(GRID):
            kw["initial_xyzs"] = GRID[:M]
        else:
            kw["initial_xyzs"] = np.array([[0.6 * (i % 4), 0.6 * (i // 4), 0.5] for i in range(M)])
    return BatchAviary(**kw)


def _bits(t):
    return t.contiguous().reshape(-1).view(torch.uint8)


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _tape(env, k, seed, scale=1.0, bias=0.0):
    """k random action sets; `bias` "climb" gives every env its own upward bias (hover: envs leave the box at z = 2 one
    after the other instead of never finishing)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    a = torch.rand((k, env.num_envs, env.NUM_DRONES, env.ACTION_DIM), generator=g) * 2 - 1
    if bias == "climb":
        a = 0.1 * a + torch.linspace(0.0, 1.0, env.num_envs).view(1, -1, 1, 1)
    else:
        a = a * scale + bias
    return a.to(device=env.device, dtype=env.action_dtype)


FLAVOURS = {
    "tile_multihover_philox": dict(task="multihover", num_envs=300, num_drones=4, act="rpm", reset_mode="jitter_philox",
                                   track_episode_stats=True),
    "hover_one_d_rpm": dict(task="hover", num_envs=257, act="one_d_rpm", track_episode_stats=True, bias="climb"),
    "generic_fp64_spiral_aero": dict(task="spiral", num_envs=61, num_drones=5, act="rpm", precision="fp64",
                                     physics="dyn_gnd_drag_dw", keep_ang_vel=True, track_episode_stats=True),
    "flock_fp32": dict(task="flock", num_envs=200, num_drones=4, act="rpm", track_episode_stats=True),
    # VEL moves at most 0.25 m/s: no env leaves the box within a few seconds, so half of the envs are reset at step 100
    # and the other half truncate (step 241) after the snapshot
    "vel": dict(task="multihover", num_envs=130, num_drones=2, act="vel", track_episode_stats=True, k1=228,
                reset_half_at=100),
    "pid": dict(task="multihover", num_envs=130, num_drones=2, act="pid", track_episode_stats=True),
    "m16_downwash": dict(task="multihover", num_envs=96, num_drones=16, act="rpm", physics="dyn_dw",
                         track_episode_stats=True),
    "euler": dict(task="multihover", num_envs=150, num_drones=2, act="rpm", integrator="euler", track_episode_stats=True),
}


def _compare_step(ra, rb, ea, eb, pid):
    assert _same(ra.obs, rb.obs)
    assert _same(ra.reward, rb.reward)
    assert torch.equal(ra.terminated, rb.terminated) and torch.equal(ra.truncated, rb.truncated)
    sa, qa, ca = ea.get_state(with_rates=True, with_step_counter=True)
    sb, qb, cb = eb.get_state(with_rates=True, with_step_counter=True)
    assert _same(sa, sb) and _same(qa, qb) and torch.equal(ca, cb)
    if pid:
        assert _same(ea.get_controller_state(), eb.get_controller_state())


@pytest.mark.parametrize("name", sorted(FLAVOURS))
def test_full_restore_continues_bit_identically(name):
    kw = dict(FLAVOURS[name])
    bias = kw.pop("bias", 0.0)
    k1 = kw.pop("k1", 63)
    reset_half_at = kw.pop("reset_half_at", None)
    pid = kw["act"] in ("vel", "pid")
    a = _aviary(seed=3, **kw)
    b = _aviary(seed=77, **kw)
    B = a.ACTION_BUFFER_SIZE
    k1b, k2 = 26, 40                    # total % B = 3 on the source, 11 on the target (B = 15)
    assert k1 % B == 3 and k1b % B == 11
    a.reset_device()
    b.reset_device()
    tape_a, tape_b = _tape(a, k1, 1, bias=bias), _tape(b, k1b, 2, bias=bias)
    for t in range(k1):
        if t == reset_half_at:
            a.reset_device(env_mask=torch.arange(a.num_envs, device=a.device) % 2 == 0)
        a.step_device(tape_a[t])
    for t in range(k1b):
        b.step_device(tape_b[t])
    _, sc = a.get_state(with_step_counter=True)
    finished_before = float(a.episode_stats(reset=False)[2])
    assert finished_before > 0 or int(sc.min()) != int(sc.max()), "every env is still in its first episode"
    rng_a = a.get_rng_state()
    snap = a.snapshot()
    assert snap.numel() == a.snapshot_nbytes and snap.dtype == torch.uint8 and snap.device == a.device
    b.restore(snap)
    assert b.get_rng_state()[:3] == rng_a[:3]
    tape = _tape(a, k2, 3, bias=bias)
    finished = 0
    for t in range(k2):
        ra = a.step_device(tape[t])
        rb = b.step_device(tape[t])
        _compare_step(ra, rb, a, b, pid)
        finished += int(ra.done.sum())
    assert finished > 0
    assert _same(a.episode_stats(), b.episode_stats())
    a.close()
    b.close()


def test_restore_from_cpu_copy_and_philox_respawns_match():
    """MultiHover re-spawns are drawn from Philox(seed; env, total steps, ...): after a full restore a handle with
    another seed and step count draws the source's positions.  The snapshot may travel through the CPU."""
    kw = FLAVOURS["tile_multihover_philox"]
    a, b = _aviary(seed=5, **kw), _aviary(seed=6, **kw)
    for x in _tape(a, 33, 4):
        a.step_device(x)
    for x in _tape(b, 9, 5):
        b.step_device(x)
    b.restore(a.snapshot().cpu())
    respawned = 0
    for x in _tape(a, 30, 6):
        ra, rb = a.step_device(x), b.step_device(x)
        assert _same(ra.obs, rb.obs)
        respawned += int(ra.done.sum())
        assert _same(a.get_targets(), b.get_targets())
    assert respawned > 0
    assert a.get_rng_state() == b.get_rng_state()


def test_masked_restore():
    kw = dict(task="multihover", num_envs=512, num_drones=2, act="rpm", reset_mode="fixed", track_episode_stats=True)
    src, dst = _aviary(seed=1, **kw), _aviary(seed=2, **kw)
    for x in _tape(src, 48, 7):
        src.step_device(x)
    for x in _tape(dst, 26, 8):
        dst.step_device(x)
    snap = src.snapshot()
    mask = torch.zeros(512, dtype=torch.bool, device=dst.device)
    mask[torch.randperm(512, generator=torch.Generator().manual_seed(0))[:256].to(dst.device)] = True
    before = dst.get_state(with_rates=True, with_step_counter=True)
    rng_before = dst.get_rng_state()
    stats_before = dst.episode_stats(reset=False)
    dst.restore(snap, env_mask=mask)
    after = dst.get_state(with_rates=True, with_step_counter=True)
    ref = src.get_state(with_rates=True, with_step_counter=True)
    keep = ~mask
    for x, y, r in zip(before, after, ref):
        assert _same(x[keep], y[keep])        # unmasked envs untouched
        assert _same(y[mask], r[mask])        # masked envs are the source's
    assert dst.get_rng_state() == rng_before
    assert _same(dst.episode_stats(reset=False), stats_before)
    for x in _tape(src, 40, 9):
        rs, rd = src.step_device(x), dst.step_device(x)
        assert _same(rs.obs[mask], rd.obs[mask]) and _same(rs.reward[mask], rd.reward[mask])
        assert torch.equal(rs.done[mask], rd.done[mask])
    assert _same(src.get_state()[mask], dst.get_state()[mask])


def test_restore_into_an_evaluation_aviary():
    """A training env's state restored into an aviary with auto_reset=False and no episode tracking (the snapshot's
    episode-return plane is ignored): outputs equal the source's up to each env's first done."""
    kw = dict(task="multihover", num_envs=256, num_drones=2, act="rpm", reset_mode="jitter_philox")
    src = _aviary(seed=1, auto_reset=True, track_episode_stats=True, **kw)
    ev = _aviary(seed=9, auto_reset=False, track_episode_stats=False, **kw)
    for x in _tape(src, 50, 11):
        src.step_device(x)
    ev.restore(src.snapshot())
    alive = torch.ones(256, dtype=torch.bool, device=src.device)
    for x in _tape(src, 60, 12):
        rs, re = src.step_device(x), ev.step_device(x)
        assert _same(rs.reward[alive], re.reward[alive])
        assert torch.equal(rs.terminated[alive], re.terminated[alive]) and torch.equal(rs.truncated[alive], re.truncated[alive])
        cont = alive & ~rs.done
        assert _same(rs.obs[cont], re.obs[cont])
        alive = cont
    assert int(alive.sum()) < 256


@pytest.mark.parametrize("pipeline", ["default", "0"])
def test_back_to_back_restore_then_step(pipeline, monkeypatch):
    """Restore immediately followed by a step (no synchronisation between them) at the headline shape: the step's
    early ring prefetch must not read planes the unpack kernel is writing.  Same results as with a synchronisation,
    and as bd_step_many (one launch) right after a restore."""
    if pipeline == "0":
        monkeypatch.setenv("BD_PIPELINE", "0")
    else:
        monkeypatch.delenv("BD_PIPELINE", raising=False)
    kw = dict(task="multihover", num_envs=65536, num_drones=4, act="rpm", reset_mode="jitter_philox",
              track_episode_stats=True)
    src, env = _aviary(seed=1, **kw), _aviary(seed=2, **kw)
    for x in _tape(src, 20, 1):
        src.step_device(x)
    for x in _tape(env, 7, 2):
        env.step_device(x)
    snap = src.snapshot()
    K = 6
    tape = _tape(env, K, 3).contiguous()

    def run(sync):
        env.restore(snap)            # device snapshot, no mask: nothing waits after the unpack launch
        if sync:
            torch.cuda.synchronize()
        outs = []
        for t in range(K):
            r = env.step_device(tape[t])
            outs.append((r.obs.clone(), r.reward.clone(), r.terminated.clone(), r.truncated.clone()))
        return outs, env.get_state()

    fast, st_fast = run(False)
    slow, st_slow = run(True)
    for x, y in zip(fast, slow):
        assert all(_same(p, q) for p, q in zip(x, y))
    assert _same(st_fast, st_slow)
    N, M, D = env.num_envs, env.NUM_DRONES, env.OBS_DIM
    obs = torch.empty((K, N, M, D), device=env.device)
    rew = torch.empty((K, N), device=env.device)
    term = torch.empty((K, N), dtype=torch.uint8, device=env.device)
    trunc = torch.empty((K, N), dtype=torch.uint8, device=env.device)
    env.restore(snap)
    env.step_many(tape, obs, rew, term, trunc)
    for t in range(K):
        assert _same(obs[t], slow[t][0]) and _same(rew[t], slow[t][1])
        assert torch.equal(term[t].bool(), slow[t][2]) and torch.equal(trunc[t].bool(), slow[t][3])
    src.close()
    env.close()


def test_graph_mode_save_and_masked_restore_full_refused():
    from marl_gym_pybullet_drones_b200.batch_aviary import StepResult
    import ctypes as C
    kw = dict(task="multihover", num_envs=256, num_drones=2, act="rpm", reset_mode="fixed")
    env = _aviary(seed=1, **kw)
    N, M, D = env.num_envs, env.NUM_DRONES, env.OBS_DIM
    act = torch.zeros((N, M, env.ACTION_DIM), device=env.device)
    out = StepResult(torch.empty((N, M, D), device=env.device), torch.empty(N, device=env.device),
                     torch.empty(N, dtype=torch.bool, device=env.device), torch.empty(N, dtype=torch.bool, device=env.device),
                     None)
    gen = torch.Generator(device="cpu").manual_seed(0)
    env.step_device(act, out=out)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        env.step_device(act, out=out)
    for _ in range(4):
        act.copy_(torch.rand(act.shape, generator=gen) * 2 - 1)
        g.replay()
    snap = env.snapshot()
    tape = torch.rand((5,) + tuple(act.shape), generator=gen) * 2 - 1
    first = []
    for t in range(5):
        act.copy_(tape[t])
        g.replay()
        first.append((out.obs.clone(), out.reward.clone()))
    env.restore(snap, env_mask=torch.ones(N, dtype=torch.bool))
    for t in range(5):
        act.copy_(tape[t])
        g.replay()
        assert _same(out.obs, first[t][0]) and _same(out.reward, first[t][1])
    with pytest.raises(ValueError, match="CUDA graph"):
        env.restore(snap)
    # neither call is capturable
    lib, h = env._lib, env._h
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        rc_save = lib.bd_save_snapshot(h, C.c_void_p(snap.data_ptr()), s)
        err_save = lib.bd_last_error()
        rc_load = lib.bd_load_snapshot(h, C.c_void_p(snap.data_ptr()), None, s)
        err_load = lib.bd_last_error()
    assert rc_save == -1 and b"capturing" in err_save
    assert rc_load == -1 and b"capturing" in err_load
    del g2
    env.close()


def test_refusals_carry_messages():
    base = dict(task="multihover", num_envs=64, num_drones=2, act="rpm")
    src = _aviary(seed=1, **base)
    snap = src.snapshot()
    cases = [
        (dict(base, num_drones=4), "drones"),
        (dict(base, task="flock"), "task"),
        (dict(base, precision="fp64"), "precision"),
        (dict(base, ctrl_freq=48), "ctrl_freq"),
        (dict(base, drone_model="cf2p"), "different configuration"),
        (dict(base, keep_ang_vel=True), "lacks"),
        (dict(base, track_episode_stats=True), "lacks"),
    ]
    for kw, what in cases:
        dst = _aviary(seed=2, **kw)
        with pytest.raises(ValueError, match=what):
            dst.restore(snap)
        dst.close()
    dst = _aviary(seed=2, **base)
    with pytest.raises(ValueError, match="truncated"):
        dst.restore(snap[:-256])
    bad = snap.clone()
    bad[0] ^= 1
    with pytest.raises(ValueError, match="magic"):
        dst.restore(bad)
    bad = snap.clone()
    bad[4] = 2                      # format version
    with pytest.raises(ValueError, match="version"):
        dst.restore(bad)
    dst.restore(snap)               # the good one still loads
    src.close()
    dst.close()


# ------------------------------------------------------------------------------------------------------- trainer
def _trainer_pair(tmp_path, **cfg):
    from marl_gym_pybullet_drones_b200 import DeviceMAPPO
    kw = dict(rollout_steps=16, hidden_dim=256, mini_batch_size=1024, opt_epochs=2, update_impl="native",
              save_env_state=True, **cfg)
    env_a = _aviary(task="multihover", num_envs=512, num_drones=2, seed=3, track_episode_stats=True)
    a = DeviceMAPPO(env_a, seed=1, **kw)
    assert a.native and a.fused is not None
    a.train_step()
    a.train_step()
    p = tmp_path / "ckpt.pt"
    a.save(p)
    env_b = _aviary(task="multihover", num_envs=512, num_drones=2, seed=3, track_episode_stats=True)
    b = DeviceMAPPO(env_b, seed=8, **kw)
    b.load(p)
    return a, b, p


def _rollout_tensors(x):
    return [x.obs, x.act, x.logp, x.rew, x.term, x.trunc, x.val]


def test_trainer_resume_continues_mid_episode(tmp_path):
    a, b, _ = _trainer_pair(tmp_path, norm_obs=False)
    a.collect_rollout()
    b.collect_rollout()
    for x, y in zip(_rollout_tensors(a), _rollout_tensors(b)):
        assert _same(x, y)
    _, sc = b.env.get_state(with_step_counter=True)
    assert int(sc.min()) != int(sc.max())          # no lock-step reset of every env
    for algo in (a, b):
        algo.compute_returns()
        algo.update()
    for oa, ob in zip((a.actor_opt, a.critic_opt), (b.actor_opt, b.critic_opt)):
        assert torch.allclose(oa.flat, ob.flat, rtol=1e-4, atol=1e-6)
    for algo in (a, b):
        algo.close()
        algo.env.close()


def test_trainer_resume_with_normalisers(tmp_path):
    a, b, _ = _trainer_pair(tmp_path, norm_obs=True, norm_reward=True)
    ra, rb = a.obs_normalizer.rms, b.obs_normalizer.rms
    assert _same(ra.mean, rb.mean) and _same(ra.var, rb.var) and ra.count == rb.count
    na, nb = a.reward_normalizer, b.reward_normalizer
    assert _same(na.mean, nb.mean) and _same(na.var, nb.var) and _same(na.count, nb.count) and _same(na.ret, nb.ret)
    a.collect_rollout()
    b.collect_rollout()
    for x, y in zip(_rollout_tensors(a), _rollout_tensors(b)):
        assert torch.allclose(x.float(), y.float(), rtol=1e-5, atol=1e-6)
    for algo in (a, b):
        algo.close()
        algo.env.close()


def test_trainer_default_checkpoint_and_foreign_shard(tmp_path):
    from marl_gym_pybullet_drones_b200 import DeviceMAPPO
    env = _aviary(task="multihover", num_envs=128, num_drones=2, seed=3, track_episode_stats=True)
    algo = DeviceMAPPO(env, seed=1, rollout_steps=8, mini_batch_size=512, opt_epochs=1)
    algo.train_step()
    sd = algo.state_dict()
    assert "resume" not in sd
    fresh = DeviceMAPPO(_aviary(task="multihover", num_envs=128, num_drones=2, seed=3, track_episode_stats=True),
                        seed=1, rollout_steps=8, mini_batch_size=512, opt_epochs=1)
    fresh.load_state_dict(sd)
    assert not fresh._reset_done and not fresh._resumed      # loads as before: the next rollout resets
    algo.cfg["save_env_state"] = True
    sd = algo.state_dict()
    assert {"env", "rank", "world", "env_offset", "env_count", "fused_seed", "reset_done"} <= set(sd["resume"])
    assert sd["resume"]["env"].device.type == "cpu"
    sd["resume"]["world"] = 2
    with pytest.raises(ValueError, match="rank 0 of 2"):
        fresh.load_state_dict(sd)
    for x in (algo, fresh):
        x.close()
        x.env.close()
