"""Hand-written PPO-update kernels (csrc/bd_ppo.cu) against plain PyTorch fp32 references of the same operations.

Reference formulas: `compute_policy_loss` / `compute_value_loss` / `update` (`mappo/agent.py:602-772`),
`_compute_single_agent_returns` + `normalize_advantages` (`mappo/buffer.py:561-614, 666-695`).

Stated tolerances (bf16 tensor-core operands, fp32 accumulation, tanh.approx):
  forward outputs            <= 2e-2 absolute on O(1) outputs
  losses / approx_kl         <= 2e-2 relative (|x| floor 1e-2)
  gradients                  relative L2 error per parameter tensor <= 8e-2, cosine similarity >= 0.996
                             (measured 1e-2 on biases, 4-6e-2 on weight matrices: bf16 rounding of dZ and of the activations)
  GAE / returns, Adam        fp32 arithmetic: <= 1e-5 / 1e-6
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _mlp(din, dout, seed):
    torch.manual_seed(seed)
    from marl_gym_pybullet_drones_b200.mappo import MLP
    return MLP(din, dout, [256, 256], "tanh").cuda()


def _flat(params):
    return torch.cat([p.detach().reshape(-1) for p in params]).contiguous()


def _rollout(T, N, M, D, A, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.randn((T + 1, N, M, D), device="cuda", generator=g)
    obs[..., :12] *= 0.5
    act = torch.randn((T, N, M, A), device="cuda", generator=g) * 0.6
    return obs, act, g


def _rel(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def _cos(a, b):
    return float(torch.dot(a.flatten(), b.flatten()) / (a.norm() * b.norm()).clamp_min(1e-20))


@pytest.mark.parametrize("T,N", [(7, 5), (32, 1000), (256, 176)])
def test_gae_kernel_matches_reference_scan(T, N):
    from marl_gym_pybullet_drones_b200 import ppo_native
    g = torch.Generator(device="cuda").manual_seed(T * 7 + N)
    rew = torch.randn((T, N), device="cuda", generator=g)
    term = (torch.rand((T, N), device="cuda", generator=g) < 0.05).to(torch.uint8)
    trunc = (torch.rand((T, N), device="cuda", generator=g) < 0.02).to(torch.uint8)
    for use_gae, vals in ((True, torch.randn((T + 1, N), device="cuda", generator=g)),
                          (True, torch.cat([torch.zeros((T, N), device="cuda"), torch.randn((1, N), device="cuda", generator=g)])),
                          (False, torch.randn((T + 1, N), device="cuda", generator=g))):
        ret, adv = torch.empty((T, N), device="cuda"), torch.empty((T, N), device="cuda")
        acc = torch.zeros(3, dtype=torch.float64, device="cuda")
        ppo_native.gae(rew, term, trunc, vals, 0.99, 0.95, use_gae, ret, adv, acc)
        # buffer.py:561-614 restated in float64 numpy, per env sequence
        r, v = rew.double().cpu().numpy(), vals.double().cpu().numpy()
        mask = 1.0 - (term | trunc).double().cpu().numpy()
        want_ret, want_adv = np.zeros((T, N)), np.zeros((T, N))
        rr, aa = v[T].copy(), np.zeros(N)
        for i in reversed(range(T)):
            rr = r[i] + 0.99 * mask[i] * rr
            if use_gae:
                td = r[i] + 0.99 * mask[i] * v[i + 1] - v[i]
                aa = aa * 0.95 * 0.99 * mask[i] + td
            else:
                aa = rr - v[i]
            want_ret[i], want_adv[i] = rr, aa
        assert np.abs(ret.cpu().numpy() - want_ret).max() <= 1e-4 * max(1.0, np.abs(want_ret).max())
        assert np.abs(adv.cpu().numpy() - want_adv).max() <= 1e-4 * max(1.0, np.abs(want_adv).max())
        st = torch.empty(2, device="cuda")
        ppo_native.adv_stats(acc, st)
        assert abs(float(st[0]) - want_adv.mean()) <= 1e-5 * max(1.0, abs(want_adv.mean()))
        assert abs(float(st[1]) - 1.0 / (want_adv.std() + 1e-8)) <= 1e-4 / (want_adv.std() + 1e-8)   # np.std: ddof = 0


@pytest.mark.parametrize("M,D,A,samples,critic", [(4, 72, 4, 300, False), (2, 72, 4, 1000, False), (4, 72, 4, 517, True),
                                                  (2, 27, 1, 260, False), (1, 72, 4, 129, True), (16, 72, 4, 200, True)])
def test_forward_matches_torch(M, D, A, samples, critic):
    from marl_gym_pybullet_drones_b200.ppo_native import PpoNet
    T, N = 6, 64
    obs, act, g = _rollout(T, N, M, D, A, 1)
    idx = torch.randint(0, T * N, (samples,), device="cuda", generator=g)
    if critic:
        mlp = _mlp(M * D, 1, 3)
        net = PpoNet(D, M, 1, False, samples)
        rows = samples
        x = obs[:T].reshape(T * N, M * D)[idx]
    else:
        mlp = _mlp(D, A, 4)
        net = PpoNet(D, 1, A, True, samples * M)
        rows = samples * M
        x = obs[:T].reshape(T * N, M, D)[idx].reshape(rows, D)
    params = ([torch.full((A,), -0.5, device="cuda")] if not critic else []) + list(mlp.parameters())
    net.pack(_flat(params))
    out = net.forward(obs, N, M, rows, idx=idx)
    want = mlp(x)
    assert float((out - want).abs().max()) <= 2e-2, float((out - want).abs().max())
    # with observation normalisation on load (per slot, per (agent, column))
    nmean = torch.randn((T + 1, M * D), device="cuda", generator=g) * 0.1
    nrstd = torch.rand((T + 1, M * D), device="cuda", generator=g) + 0.5
    out = net.forward(obs, N, M, rows, idx=idx, nmean=nmean, nrstd=nrstd, nclip=2.0)
    t = torch.div(idx, N, rounding_mode="floor")
    xn = ((obs[:T].reshape(T * N, M * D)[idx] - nmean[t]) * nrstd[t]).clamp(-2.0, 2.0)
    want = mlp(xn if critic else xn.reshape(rows, D))
    assert float((out - want).abs().max()) <= 2e-2
    net.close()


def test_forward_many_tiles_per_cta():
    """More tiles than 2 x SMs, odd count, ragged last tile: every CTA of the two-tiles-in-flight kernel runs several
    pairs plus a single; actor rows and critic rows (M input chunks)."""
    from marl_gym_pybullet_drones_b200.ppo_native import PpoNet
    T, N, M, D, A = 3, 30000, 4, 72, 4
    obs, act, g = _rollout(T, N, M, D, A, 11)
    samples = 128 * 148 * 5 // M + 77
    idx = torch.randint(0, T * N, (samples,), device="cuda", generator=g)
    mlp = _mlp(D, A, 4)
    net = PpoNet(D, 1, A, True, samples * M)
    net.pack(_flat([torch.full((A,), -0.5, device="cuda")] + list(mlp.parameters())))
    out = net.forward(obs, N, M, samples * M, idx=idx)
    with torch.no_grad():
        want = mlp(obs[:T].reshape(T * N, M, D)[idx].reshape(samples * M, D))
    assert float((out - want).abs().max()) <= 2e-2
    net.close()
    cm = _mlp(M * D, 1, 3)
    cnet = PpoNet(D, M, 1, False, T * N)
    cnet.pack(_flat(list(cm.parameters())))
    out = cnet.forward(obs, N, M, T * N)              # identity index: values of whole slots, 703 tiles
    with torch.no_grad():
        want = cm(obs[:T].reshape(T * N, M * D))
    assert float((out - want).abs().max()) <= 2e-2
    cnet.close()


@pytest.mark.parametrize("N,M,D,A", [(700, 4, 72, 4), (50, 2, 27, 1), (40000, 4, 72, 4), (3, 16, 72, 4)])
def test_sample_matches_torch(N, M, D, A):
    """`MAPPOActorCritic.step` (agent.py:389-415): act = mean + exp(logstd) eps, logp = summed Normal log-density;
    mean within the forward tolerance, act / logp exact given the mean and the noise (fp32, <= 1e-5)."""
    from marl_gym_pybullet_drones_b200.ppo_native import PpoNet
    g = torch.Generator(device="cuda").manual_seed(N + M)
    obs = torch.randn((N, M, D), device="cuda", generator=g)
    mlp = _mlp(D, A, 8)
    logstd = torch.linspace(-0.7, -0.2, A, device="cuda")
    net = PpoNet(D, 1, A, True, 128)
    net.pack(_flat([logstd] + list(mlp.parameters())))
    noise = torch.randn((N, M, A), device="cuda", generator=g)
    act, logp, mean = (torch.empty((N, M, A), device="cuda"), torch.empty((N, M, 1), device="cuda"),
                       torch.empty((N, M, A), device="cuda"))
    net.sample(obs, act, logp, noise=noise, out_mean=mean)
    with torch.no_grad():
        want_mean = mlp(obs.view(N * M, D)).view(N, M, A)
    assert float((mean - want_mean).abs().max()) <= 2e-2
    assert float((act - (mean + logstd.exp() * noise)).abs().max()) <= 1e-5
    want_lp = torch.distributions.Normal(mean, logstd.exp()).log_prob(act).sum(-1, keepdim=True)
    assert float((logp - want_lp).abs().max()) <= 2e-4
    # normalisation on load (one slot's statistics, per (agent, column))
    nmean = torch.randn((M * D,), device="cuda", generator=g) * 0.1
    nrstd = torch.rand((M * D,), device="cuda", generator=g) + 0.5
    net.sample(obs, act, logp, noise=noise, out_mean=mean, nmean=nmean, nrstd=nrstd, nclip=2.0)
    with torch.no_grad():
        xn = ((obs.view(N, M * D) - nmean) * nrstd).clamp(-2.0, 2.0)
        want_mean = mlp(xn.view(N * M, D)).view(N, M, A)
    assert float((mean - want_mean).abs().max()) <= 2e-2
    # Philox noise: deterministic in (seed, offset), different across offsets, standard normal moments
    a1, a2, a3 = torch.empty_like(act), torch.empty_like(act), torch.empty_like(act)
    net.sample(obs, a1, logp, seed=5, offset=9, out_mean=mean)
    net.sample(obs, a2, logp, seed=5, offset=9)
    net.sample(obs, a3, logp, seed=5, offset=10)
    assert torch.equal(a1, a2) and not torch.equal(a1, a3)
    eps = (a1 - mean) / logstd.exp()
    want_lp = (-0.5 * eps.pow(2) - logstd - 0.5 * math.log(2 * math.pi)).sum(-1, keepdim=True)
    net.sample(obs, a1, logp, seed=5, offset=9)
    assert float((logp - want_lp).abs().max()) <= 5e-3      # eps recovered through a division: looser
    if N * M * A >= 10000:
        assert abs(float(eps.mean())) <= 0.02 and abs(float(eps.var()) - 1.0) <= 0.03
        e3 = (a3 - mean) / logstd.exp()
        assert abs(float((eps * e3).mean())) <= 0.02        # streams of different offsets are uncorrelated
    net.close()


def _actor_reference(mlp, logstd, obs, act, logp_old, adv_n, idx, T, N, M, D, A, clip, ent_coef):
    mb = idx.numel()
    o = obs[:T].reshape(T * N, M, D)[idx].reshape(mb * M, D)
    a = act.reshape(T * N, M, A)[idx].reshape(mb * M, A)
    lpo = logp_old.reshape(T * N, M)[idx].reshape(mb * M, 1)
    ad = adv_n.reshape(T * N, 1)[idx].unsqueeze(1).expand(mb, M, 1).reshape(mb * M, 1)
    dist = torch.distributions.Normal(mlp(o), logstd.exp())
    lp = dist.log_prob(a).sum(-1, keepdim=True)
    ratio = torch.exp(lp - lpo)
    policy_loss = -torch.min(ratio * ad, torch.clamp(ratio, 1 - clip, 1 + clip) * ad).mean()
    entropy_loss = -dist.entropy().sum(-1).mean()
    kl = (lpo - lp).mean()
    return policy_loss, entropy_loss, kl


@pytest.mark.parametrize("M,samples", [(4, 1024), (2, 333), (1, 128), (4, 128 * 148 * 3 // 4 + 5)])
def test_actor_gradient_matches_autograd(M, samples):
    from marl_gym_pybullet_drones_b200 import ppo_native
    from marl_gym_pybullet_drones_b200.ppo_native import PpoNet
    T, N, D, A = 8, (200 if samples <= 1600 else 2000), 72, 4
    obs, act, g = _rollout(T, N, M, D, A, 5)
    mlp = _mlp(D, A, 6)
    logstd = torch.nn.Parameter(torch.tensor([-0.5, -0.3, -0.7, -0.5], device="cuda"))
    with torch.no_grad():      # "old" log-probs from a slightly different policy so that ratios spread around 1 and clip
        old = _mlp(D, A, 6)
        for p in old.parameters():
            p.add_(0.02 * torch.randn(p.shape, device="cuda", generator=g))
        d0 = torch.distributions.Normal(old(obs[:T].reshape(-1, D)), logstd.exp())
        logp_old = d0.log_prob(act.reshape(-1, A)).sum(-1).reshape(T, N, M).contiguous()
    adv = torch.randn((T, N), device="cuda", generator=g) * 3 + 1
    acc = torch.tensor([float(adv.sum()), float((adv.double() ** 2).sum()), float(adv.numel())], dtype=torch.float64, device="cuda")
    stats2 = torch.empty(2, device="cuda")
    ppo_native.adv_stats(acc, stats2)
    adv_n = (adv - adv.mean()) / (adv.std(unbiased=False) + 1e-8)
    idx = torch.randperm(T * N, device="cuda", generator=g)[:samples].contiguous()
    clip, ent = 0.2, 0.005
    pl, el, kl = _actor_reference(mlp, logstd, obs, act, logp_old, adv_n, idx, T, N, M, D, A, clip, ent)
    params = [logstd] + list(mlp.parameters())
    want = torch.autograd.grad(pl + ent * el, params)
    net = PpoNet(D, 1, A, True, samples * M)
    net.pack(_flat(params))
    grad = torch.zeros(net.param_count, device="cuda")
    net.grad(grad, obs, N, M, idx, samples, critic=False, act=act, logp_old=logp_old, adv=adv, adv_stats=stats2, clip=clip,
             entropy_coef=ent)
    torch.cuda.synchronize()
    st = net.stats.clone()
    rows = samples * M
    assert float(st[2]) == rows
    assert abs(float(st[0]) / rows - float(pl)) <= 2e-2 * max(abs(float(pl)), 1e-2), (float(st[0]) / rows, float(pl))
    assert abs(float(st[1]) / rows - float(kl)) <= 2e-2 * max(abs(float(kl)), 1e-2), (float(st[1]) / rows, float(kl))
    off = 0
    names = ["logstd", "W1", "b1", "W2", "b2", "W3", "b3"]
    for name, w in zip(names, want):
        got = grad[off:off + w.numel()].view_as(w)
        off += w.numel()
        assert _rel(got, w) <= 8e-2 and _cos(got, w) >= 0.996, (name, _rel(got, w), _cos(got, w))
    assert off == net.param_count
    net.close()


@pytest.mark.parametrize("M,samples,clipped", [(4, 700, False), (2, 256, True), (16, 150, False), (1, 130, False)])
def test_critic_gradient_matches_autograd(M, samples, clipped):
    from marl_gym_pybullet_drones_b200.ppo_native import PpoNet
    T, N, D = 8, 100, 72
    obs, _, g = _rollout(T, N, M, D, 4, 9)
    mlp = _mlp(M * D, 1, 10)
    ret = torch.randn((T, N), device="cuda", generator=g) * 2 + 3
    v_old = torch.randn((T, N), device="cuda", generator=g) * 0.3
    idx = torch.randperm(T * N, device="cuda", generator=g)[:samples].contiguous()
    x = obs[:T].reshape(T * N, M * D)[idx]
    v = mlp(x)
    r = ret.reshape(T * N, 1)[idx]
    if clipped:
        vo = v_old.reshape(T * N, 1)[idx]
        vc = vo + (v - vo).clamp(-0.2, 0.2)
        loss = 0.5 * torch.max((v - r).pow(2), (vc - r).pow(2)).mean()
    else:
        loss = 0.5 * (v - r).pow(2).mean()
    params = list(mlp.parameters())
    want = torch.autograd.grad(loss, params)
    net = PpoNet(D, M, 1, False, samples)
    net.pack(_flat(params))
    grad = torch.zeros(net.param_count, device="cuda")
    net.grad(grad, obs, N, M, idx, samples, critic=True, ret=ret, v_old=v_old, clip=0.2, use_clipped_value=clipped)
    torch.cuda.synchronize()
    assert abs(float(net.stats[0]) / samples - float(loss)) <= 2e-2 * max(abs(float(loss)), 1e-2)
    off = 0
    for name, w in zip(["W1", "b1", "W2", "b2", "W3", "b3"], want):
        got = grad[off:off + w.numel()].view_as(w)
        off += w.numel()
        assert _rel(got, w) <= 8e-2 and _cos(got, w) >= 0.996, (name, M, _rel(got, w), _cos(got, w))
    net.close()


def test_gated_adam_step_equals_torch_adam():
    """`bd_ppo_adam_step` == torch.optim.Adam step by step; a closed gate changes nothing (not even the step count)."""
    from marl_gym_pybullet_drones_b200.ppo_native import PpoNet
    D, A = 72, 4
    mlp = _mlp(D, A, 2)
    logstd = torch.nn.Parameter(torch.full((A,), -0.5, device="cuda"))
    params = [logstd] + list(mlp.parameters())
    opt = torch.optim.Adam(params, lr=3e-4)
    net = PpoNet(D, 1, A, True, 128)
    flat = _flat(params)
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    step = torch.zeros((), dtype=torch.float64, device="cuda")
    kl = torch.zeros(2, dtype=torch.float64, device="cuda")
    gates = torch.zeros((), dtype=torch.float64, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(0)
    for it in range(6):
        grad = torch.randn(flat.shape, device="cuda", generator=g) * 0.01
        open_gate = it != 3
        kl[0], kl[1] = (0.5 if open_gate else 2.0) * 0.015 * 100, 100.0      # approx_kl = 0.0075 / 0.03 vs 1.5 * 0.01
        before = flat.clone()
        net.adam_step(flat, m, v, grad, step, 3e-4, kl_sum=kl[0:1], kl_rows=kl[1:2], target_kl=0.01, gate_count=gates)
        if open_gate:
            off = 0
            for p in params:
                p.grad = grad[off:off + p.numel()].view_as(p).clone()
                off += p.numel()
            opt.step()
            assert float((flat - _flat(params)).abs().max()) <= 1e-7
        else:
            assert torch.equal(flat, before)
    torch.cuda.synchronize()
    assert float(step) == 5.0 and float(gates) == 5.0
    net.close()
