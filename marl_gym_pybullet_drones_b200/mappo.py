"""MAPPO with the whole rollout and update on the GPU (SURVEY.md §8f-1).

The reference trainer (`gym_pybullet_drones/mappo/mappo.py:619-1184`, `agent.py:339-423,602-772`,
`buffer.py:428-614`) crosses the host/device boundary twice per env step, runs GAE as a Python
triple loop in numpy and updates on 32-sample minibatches.  Here the envs live in a
`BatchAviary`; observations are written by the step kernel directly into the rollout buffer
slot they belong to, actions are sampled on the device and handed to the kernel without a copy,
GAE is a backwards scan over T device tensors, and the update uses large minibatches.

What is kept from the reference (and where it is switchable):
  * CTDE: one actor shared by all agents (`share_actor_weights`), tanh MLP obs_dim -> hidden ->
    hidden -> act_dim, state-independent `logstd = -0.5`, diagonal Gaussian whose log-prob is
    summed over action dims (`agent.py:87-130`, `distributions.py:9-21`); centralised critic on the
    concatenated local observations of the env's agents (`agent.py:164-223`, `mappo.py:583-617`);
  * the env's scalar reward is broadcast to every agent, mask = 1 - done (`mappo.py:758-772`);
  * `rollout_values="zeros"` reproduces the reference's rollout, which stores v = 0
    (`agent.py:413`), so GAE degenerates to lambda-returns; `"critic"` evaluates the critic
    during the rollout (textbook GAE);
  * advantages normalised over the whole buffer with (adv-mean)/(std+1e-8) (`buffer.py:666-695`);
  * clipped-ratio policy loss + entropy bonus, update skipped when the minibatch
    approx_kl > 1.5 target_kl (`agent.py:602-641,731`); critic loss 0.5 (V - mean_agents(ret))^2
    (`agent.py:643-700`); two Adam optimisers; no gradient clipping (`config.py:32` is unused);
  * truncation is not bootstrapped (the envs never emit 'TimeLimit.truncated', `mappo.py:827,845`).

The update itself is hand-written (`csrc/bd_ppo.cu`, `ppo_native.py`): per minibatch a fused tcgen05 kernel does
gather -> MLP forward -> loss -> backward through the hidden layers, a second tcgen05 kernel the weight gradients, and
small kernels the gradient reduction, the KL-gated Adam step and the bf16 repack; returns / advantages are one scan
kernel.  A whole epoch of minibatches is captured ONCE as a CUDA graph (also under multi-GPU: the NCCL all-reduces
are part of the graph).  `update_impl="torch"` keeps the round-1 torch-autograd update (library GEMMs) for shapes the
kernels do not cover (hidden != 256, obs_dim > 96) and for A/B measurements.

Multi-GPU: every rank owns its env shard; per optimiser step ONE NCCL all-reduce of the flat gradient buffer
(`GatedAdam.grad`), plus 2 doubles for the KL gate; advantage moments, normaliser moments and episode statistics are
small all-reduces per rollout.
"""
from __future__ import annotations

import math
import time
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn as nn

from .batch_aviary import BatchAviary, StepResult
from .dist import reduce_episode_stats
from .optim import GatedAdam

MAPPO_CONFIG = {   # reference mappo/config.py:3-48 with the learn_mappo.py:179-217 overrides
    "hidden_dim": 256,
    "activation": "tanh",
    "gamma": 0.99,
    "use_gae": True,
    "gae_lambda": 0.95,
    "clip_param": 0.2,
    "target_kl": 0.01,
    "entropy_coef": 0.005,
    "opt_epochs": 10,
    "mini_batch_size": 32,        # in ENV-steps (each sample carries all M agents), as in the reference
    "actor_lr": 3e-4,
    "critic_lr": 1e-3,
    "rollout_steps": 256,
    "rollout_values": "zeros",    # reference behaviour; "critic" = textbook GAE
    "use_clipped_value": False,
    "fused_actor": True,          # rollout-time actor forward + sampling as one tcgen05 kernel (actor.py)
    "graph_update": True,         # replay the update as a CUDA graph (native: one graph per epoch, collectives included)
    "peer_allreduce": True,       # several ranks on one node: gradient + KL all-reduce as ONE kernel over NVLink peer memory
                                  # (peer.py / csrc/bd_peer.cu) instead of two NCCL calls per minibatch; falls back to NCCL
    "update_impl": "auto",        # "native": hand-written kernels (bd_ppo.cu); "torch": autograd + library GEMMs;
                                  # "auto": native where the kernels cover the shape, else torch
    "matmul_precision": "tf32",   # PPO-update GEMMs: "tf32" (tensor cores, fp32 storage / accumulation), "fp32" (CUDA
                                  # cores), "bf16" (autocast: bf16 operands AND saved activations, fp32 master weights)
    "norm_obs": False,            # mappo/config.py:7-10; True in the Spiral config (env_select_learn_mappo.py:278)
    "norm_reward": False,
    "clip_obs": 10,
    "clip_reward": 10,
    "save_env_state": False,      # state_dict() also stores the simulator snapshot and the rollout loop's state under
                                  # "resume", so a resumed run continues mid-episode instead of resetting every env
}


class MLP(nn.Module):
    """`safe_control_gym/math_and_models/neural_networks.py:18-53` (default nn.Linear init)."""

    def __init__(self, input_dim, output_dim, hidden_dims, act="tanh"):
        super().__init__()
        dims = [input_dim] + list(hidden_dims) + [output_dim]
        self.fcs = nn.ModuleList([nn.Linear(dims[i], dims[i + 1]) for i in range(len(dims) - 1)])
        self.act = getattr(torch, act)

    def forward(self, x):
        for fc in self.fcs[:-1]:
            x = self.act(fc(x))
        return self.fcs[-1](x)


class ActorCritic(nn.Module):
    """Shared actor + centralised critic (`mappo/agent.py:225-337`)."""

    def __init__(self, obs_dim, act_dim, num_agents, hidden_dim=256, activation="tanh"):
        super().__init__()
        self.obs_dim, self.act_dim, self.num_agents = obs_dim, act_dim, num_agents
        self.actor = MLP(obs_dim, act_dim, [hidden_dim, hidden_dim], activation)
        self.logstd = nn.Parameter(-0.5 * torch.ones(act_dim))
        self.critic = MLP(num_agents * obs_dim, 1, [hidden_dim, hidden_dim], activation)

    def actor_parameters(self):
        """Order of `MLPActor.parameters()` in the reference (own parameter first, then `pi_net`), so
        that Adam states are interchangeable with `model_latest.pt` (`mappo/agent.py:87-110,588-594`)."""
        return [self.logstd] + list(self.actor.parameters())

    # reference parameter names (`MAPPOActorCritic.state_dict()`, mappo/agent.py:225-320)
    def reference_state_dict(self):
        sd = {"actor.logstd": self.logstd.detach().clone()}
        for k, v in self.actor.state_dict().items():
            sd["actor.pi_net." + k] = v.detach().clone()
        for k, v in self.critic.state_dict().items():
            sd["critic.v_net." + k] = v.detach().clone()
        return sd

    def load_reference_state_dict(self, sd):
        if "actor.logstd" not in sd:       # this repo's own key layout
            return self.load_state_dict(sd)
        own = {"logstd": sd["actor.logstd"]}
        for k, v in sd.items():
            if k.startswith("actor.pi_net."):
                own["actor." + k[len("actor.pi_net."):]] = v
            elif k.startswith("critic.v_net."):
                own["critic." + k[len("critic.v_net."):]] = v
        return self.load_state_dict(own)

    def dist(self, obs):
        return torch.distributions.Normal(self.actor(obs), self.logstd.exp())

    def logp(self, obs, act):
        return self.dist(obs).log_prob(act).sum(-1, keepdim=True)

    def value(self, global_obs):
        return self.critic(global_obs)


class DeviceMAPPO:
    """On-device MAPPO around a `BatchAviary` (`MAPPO.learn/train_step`, `mappo/mappo.py:289-1184`)."""

    def __init__(self, env: BatchAviary, seed: int = 0, **kwargs):
        self.cfg = dict(MAPPO_CONFIG)
        self.cfg.update(kwargs)
        self.env = env
        self.device = env.device
        if env.action_dtype != torch.float32:
            raise ValueError("DeviceMAPPO drives fp32 aviaries")
        if not env._cfg.track_episodes:
            raise ValueError("DeviceMAPPO needs BatchAviary(..., track_episode_stats=True)")
        self.N, self.M, self.D, self.A = env.num_envs, env.NUM_DRONES, env.OBS_DIM, env.ACTION_DIM
        self.T = int(self.cfg["rollout_steps"])
        torch.manual_seed(seed)   # same initial weights on every rank
        self.ac = ActorCritic(self.D, self.A, self.M, self.cfg["hidden_dim"], self.cfg["activation"]).to(self.device)
        # torch.optim.Adam's arithmetic and checkpoint format, with a device-side gate (optim.py)
        self.actor_opt = GatedAdam(self.ac.actor_parameters(), lr=self.cfg["actor_lr"])
        self.critic_opt = GatedAdam(self.ac.critic.parameters(), lr=self.cfg["critic_lr"])
        self._graph = None
        self._world = torch.distributed.get_world_size() if torch.distributed.is_initialized() else 1
        self._peer = None
        impl = str(self.cfg["update_impl"])
        if impl not in ("auto", "native", "torch"):
            raise ValueError("update_impl must be 'auto', 'native' or 'torch'")
        covered = (int(self.cfg["hidden_dim"]) == 256 and self.cfg["activation"] == "tanh" and self.D <= 96 and self.A <= 4
                   and self.M <= 16)
        if impl == "native" and not covered:
            raise ValueError("update_impl='native' needs hidden_dim 256, tanh, obs_dim <= 96, act_dim <= 4, <= 16 agents")
        self.native = impl != "torch" and covered
        if self.cfg["use_clipped_value"] and self.cfg["rollout_values"] != "critic":
            raise ValueError("use_clipped_value needs rollout_values='critic' (the reference clips around the stored "
                             "rollout value, which its own rollout leaves at zero: agent.py:413,683)")
        self.actor_net = self.critic_net = None
        self.gen = torch.Generator(device=self.device)
        rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
        self.gen.manual_seed(seed * 1000003 + rank)
        T, N, M, D, A = self.T, self.N, self.M, self.D, self.A
        dev = self.device
        # rollout storage; the step kernel writes obs[t+1] in place
        self.obs = torch.zeros((T + 1, N, M, D), device=dev)
        self.act = torch.zeros((T, N, M, A), device=dev)
        self.logp = torch.zeros((T, N, M, 1), device=dev)
        self.val = torch.zeros((T + 1, N, 1), device=dev)
        self.rew = torch.zeros((T, N), device=dev)
        self.term = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self.trunc = torch.zeros((T, N), dtype=torch.uint8, device=dev)
        self.ret = torch.zeros((T, N, 1), device=dev)
        self.adv = torch.zeros((T, N, 1), device=dev)
        self.adv_n = torch.zeros((T, N, 1), device=dev)
        self._adv_acc = torch.zeros(3, dtype=torch.float64, device=dev)     # sum adv, sum adv^2, count (all ranks)
        self._adv_stats = torch.zeros(2, device=dev)                        # mean, 1 / (std + 1e-8)
        self._run_actor = torch.zeros(4, dtype=torch.float64, device=dev)   # per-update sums of minibatch statistics
        self._run_critic = torch.zeros(4, dtype=torch.float64, device=dev)
        self._gates = torch.zeros((), dtype=torch.float64, device=dev)      # actor steps that passed the KL gate
        self._perm = torch.zeros(T * N, dtype=torch.int64, device=dev)
        if self.native:
            from .ppo_native import PpoNet
            self.critic_net = PpoNet(D, M, 1, False, max_rows=max(1, min(int(self.cfg["mini_batch_size"]), T * N)), device=dev)
            self.actor_net = PpoNet(D, 1, A, True, max_rows=max(1, min(int(self.cfg["mini_batch_size"]), T * N)) * M, device=dev)
            self._pack_native()
            if self._world > 1:
                # both networks' flat gradients live in ONE buffer: one NCCL all-reduce per minibatch instead of two (the
                # collectives are latency-bound: ~30 us each at 8 GPUs whatever their size up to a few MB)
                na, nc = self.actor_opt.grad.numel(), self.critic_opt.grad.numel()
                self._peer = None
                if self.cfg["peer_allreduce"]:
                    # ... and that buffer is this rank's block of peer-mapped memory: the gradient kernels write where the
                    # all-reduce kernel reads, and the collective (gradients + the KL pair of the gate) is one launch
                    from .peer import PeerAllReduce
                    self._peer = PeerAllReduce.create(na + nc, dev)
                self._joint_grad = self._peer.data if self._peer is not None else torch.zeros(na + nc, device=dev)
                self.actor_opt.grad = self._joint_grad[:na]
                self.critic_opt.grad = self._joint_grad[na:]
        # episode statistics (VecRecordEpisodeStatistics semantics, record_episode_statistics.py:144-171)
        # (the step kernel accumulates them: BatchAviary.episode_stats)
        self.total_env_steps = 0
        self._reset_done = False
        self._resumed = False     # obs[0] holds the observation a checkpoint's "resume" block restored
        self.fused = None
        if self.cfg["fused_actor"] and self.cfg["activation"] == "tanh":
            from ._native import NativeError
            from .actor import FusedActor
            try:
                self.fused = FusedActor(self.D, int(self.cfg["hidden_dim"]), self.A, device=self.device)
            except NativeError:
                self.fused = None   # shape outside the fused kernel's envelope: torch path
        self._fused_seed = seed * 7919 + rank
        self._fused_stale = True
        # running normalisers (mappo/mappo.py:130-135); statistics live on the device, the rollout buffer
        # keeps RAW observations plus the (mean, 1/std) that were current when each slot was produced
        from .normalization import BaseNormalizer, MeanStdNormalizer, RewardStdNormalizer
        self.obs_normalizer = BaseNormalizer()
        self.reward_normalizer = BaseNormalizer()
        self.norm_obs = bool(self.cfg["norm_obs"])
        if self.norm_obs:
            self.obs_normalizer = MeanStdNormalizer(shape=(M, D), clip=float(self.cfg["clip_obs"]), epsilon=1e-8, device=dev)
            self.nmean = torch.zeros((T + 1, M * D), device=dev)
            self.nrstd = torch.ones((T + 1, M * D), device=dev)
        if self.cfg["norm_reward"]:
            self.reward_normalizer = RewardStdNormalizer(gamma=self.cfg["gamma"], clip=float(self.cfg["clip_reward"]),
                                                         epsilon=1e-8, device=dev)

    # ------------------------------------------------------------------ rollout
    def reset(self):
        self.env.reset_device(out=self.obs[0])
        self.env.episode_stats(reset=True)
        self._observe(0)
        self._reset_done = True

    def _observe(self, t):
        """`self.obs = self.obs_normalizer(obs)` (mappo.py:165,804) without materialising it: update the
        running statistics with raw slot t and remember the (mean, 1/std) it is to be read with."""
        if self.norm_obs:
            self.obs_normalizer.update(self.obs[t])
            self.obs_normalizer.rms.stats(self.nmean[t], self.nrstd[t])

    def _normed(self, obs, t):
        """Normalised view of raw observations (..., M, D) of slot(s) t (torch path: critic, update)."""
        if not self.norm_obs:
            return obs
        shp = obs.shape
        o = obs.reshape(-1, self.M * self.D)
        c = float(self.cfg["clip_obs"])
        return ((o - self.nmean[t]) * self.nrstd[t]).clamp_(-c, c).view(shp)

    @torch.no_grad()
    def collect_rollout(self):
        """T env steps for all N envs; no host synchronisation inside the loop."""
        if not self._reset_done:
            self.reset()
        elif self._resumed:
            self._resumed = False                 # obs[0] and its statistics came from the checkpoint
        elif self.total_env_steps > 0:
            self.obs[0].copy_(self.obs[self.T])   # the rollout continues where the previous one stopped
            if self.norm_obs:
                self.nmean[0].copy_(self.nmean[self.T])
                self.nrstd[0].copy_(self.nrstd[self.T])
        T, N, M = self.T, self.N, self.M
        std = self.ac.logstd.exp()
        use_critic = self.cfg["rollout_values"] == "critic"
        if self.fused is not None and self._fused_stale:
            self.fused.set_weights(self.ac.actor, self.ac.logstd)     # bf16 tensor-core tiles of the current policy
            self._fused_stale = False
        for t in range(T):
            obs_t = self.obs[t]
            if self.fused is not None:
                if self.norm_obs:   # normalised on load inside the kernel
                    self.fused.set_input_norm(self.nmean[t], self.nrstd[t], period=M, clip=float(self.cfg["clip_obs"]))
                # one kernel: MLP on tcgen05, Gaussian sample (Philox), summed log-prob; writes act[t], logp[t]
                self.fused.forward(obs_t.view(N * M, self.D), seed=self._fused_seed,
                                   out_act=self.act[t].view(N * M, self.A), out_logp=self.logp[t].view(N * M))
            else:
                mean = self.ac.actor(self._normed(obs_t, t).view(N * M, self.D)).view(N, M, self.A)
                noise = torch.randn(mean.shape, device=self.device, generator=self.gen)
                self.act[t] = mean + std * noise                      # unclipped Gaussian (agent.py:399-400)
                self.logp[t] = (-0.5 * noise.pow(2) - self.ac.logstd - 0.5 * math.log(2 * math.pi)).sum(-1, keepdim=True)
            if use_critic:
                self._value_into(t)
            out = StepResult(self.obs[t + 1], self.rew[t], self.term[t].view(torch.bool),
                             self.trunc[t].view(torch.bool), None)
            self.env.step_device(self.act[t], out=out)   # episode statistics are kept by the step kernel
            self._observe(t + 1)
            if self.cfg["norm_reward"]:                  # mappo.py:805, raw rewards stay in the episode statistics
                self.rew[t] = self.reward_normalizer(self.rew[t], self.term[t] | self.trunc[t])
        # bootstrap value of the last observation (`last_val`, mappo.py:1049-1157)
        self._value_into(T)
        if not use_critic:
            self.val[:T].zero_()                                       # agent.py:413: v stored as zeros
        self.total_env_steps += T * N

    def _pack_native(self):
        """bf16 tensor-core copies of both networks from the fp32 master parameters (GatedAdam's flat buffers)."""
        if self.native:
            self.actor_net.pack(self.actor_opt.flat)
            self.critic_net.pack(self.critic_opt.flat)

    def _norm_args(self, t=None):
        """Per-slot observation statistics for the native kernels (slot t only, or all slots)."""
        if not self.norm_obs:
            return dict(nmean=None, nrstd=None, nclip=10.0)
        c = float(self.cfg["clip_obs"])
        if t is None:
            return dict(nmean=self.nmean, nrstd=self.nrstd, nclip=c)
        return dict(nmean=self.nmean[t:t + 1], nrstd=self.nrstd[t:t + 1], nclip=c)

    @torch.no_grad()
    def _value_into(self, t):
        """val[t] = V(global observation of slot t) (`MAPPOActorCritic.get_value`, agent.py:295-314)."""
        N, M = self.N, self.M
        if self.native:
            self.critic_net.forward(self.obs[t], N, M, N, out=self.val[t], **self._norm_args(t))
        else:
            self.val[t] = self.ac.value(self._normed(self.obs[t], t).view(N, M * self.D))

    @torch.no_grad()
    def compute_returns(self):
        """GAE / returns (`buffer.py:561-614`) as ONE scan kernel, per env (the reward is shared by the agents), and the
        buffer-wide advantage moments for `normalize_advantages` (`buffer.py:666-695`: population std over all ranks'
        advantages; the update kernels normalise on the fly, the torch path reads `adv_n`)."""
        from . import ppo_native
        T, N = self.T, self.N
        self._adv_acc.zero_()
        ppo_native.gae(self.rew, self.term, self.trunc, self.val.view(T + 1, N), self.cfg["gamma"], self.cfg["gae_lambda"],
                       self.cfg["use_gae"], self.ret.view(T, N), self.adv.view(T, N), self._adv_acc)
        if self._world > 1:
            torch.distributed.all_reduce(self._adv_acc)
        ppo_native.adv_stats(self._adv_acc, self._adv_stats)
        if not self.native:
            self.adv_n.copy_((self.adv - self._adv_stats[0]) * self._adv_stats[1])

    # ------------------------------------------------------------------- update
    def update(self) -> Dict[str, float]:
        """`MAPPOAgent.update` (agent.py:702-772) on device tensors."""
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = self.cfg["matmul_precision"] in ("tf32", "bf16")
        try:
            return self._update()
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev

    def _minibatch(self, idx):
        """One minibatch of `MAPPOAgent.update` (agent.py:702-772): actor step (KL-gated), critic step,
        statistics.  No host synchronisation; every tensor it touches has a fixed address, so it is
        capturable in a CUDA graph."""
        cfg = self.cfg
        T, N, M, D, A = self.T, self.N, self.M, self.D, self.A
        n = T * N
        mb = idx.numel()
        obs = self.obs[:T].view(n, M, D)
        ob = obs[idx]
        if self.norm_obs:
            ob = self._normed(ob, torch.div(idx, N, rounding_mode="floor"))
        o, a = ob.reshape(mb * M, D), self.act.view(n, M, A)[idx].reshape(mb * M, A)
        lp_old = self.logp.view(n, M, 1)[idx].reshape(mb * M, 1)
        ad = self.adv_n.view(n, 1, 1)[idx].expand(mb, M, 1).reshape(mb * M, 1)   # advantage tiled to every agent
        ret = self.ret.view(n, 1)[idx]                                            # = mean over agents of identical returns
        # torch.distributions.Normal's log_prob / entropy formulas written out: constructing the distribution
        # validates its arguments with a host read, which a CUDA-graph capture forbids
        bf16 = cfg["matmul_precision"] == "bf16"
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16, enabled=bf16):
            mean = self.ac.actor(o)
        mean, logstd = mean.float(), self.ac.logstd
        var = torch.exp(logstd) ** 2
        lp = (-((a - mean) ** 2) / (2 * var) - logstd - math.log(math.sqrt(2 * math.pi))).sum(-1, keepdim=True)
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + logstd).sum(-1)
        ratio = torch.exp(lp - lp_old)
        clip_adv = torch.clamp(ratio, 1 - cfg["clip_param"], 1 + cfg["clip_param"]) * ad
        policy_loss = -torch.min(ratio * ad, clip_adv).mean()
        entropy_loss = -ent.mean()
        approx_kl = (lp_old - lp).mean().detach()
        self.actor_opt.zero_grad()
        (policy_loss + cfg["entropy_coef"] * entropy_loss).backward()
        gate = None
        if self._world > 1:   # every rank must take the same gate decision or the replicas drift apart
            self.actor_opt.all_reduce_grad()
            torch.distributed.all_reduce(approx_kl)
            approx_kl = approx_kl / self._world
        if cfg["target_kl"] > 0:
            # KL gate (agent.py:731): the optimiser step (Adam moments and step count included) is skipped
            # entirely when the minibatch violates the constraint; decided on the device
            gate = approx_kl <= 1.5 * cfg["target_kl"]
        self.actor_opt.step(gate)
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16, enabled=bf16):
            v = self.ac.value(ob.reshape(mb, M * D))
        if cfg["use_clipped_value"]:                                              # agent.py:681-686
            v_old = self.val[:T].reshape(n, 1)[idx]
            v_clip = v_old + (v.float() - v_old).clamp(-cfg["clip_param"], cfg["clip_param"])
            value_loss = 0.5 * torch.max((v.float() - ret).pow(2), (v_clip - ret).pow(2)).mean()
        else:
            value_loss = 0.5 * (v.float() - ret).pow(2).mean()
        self.critic_opt.zero_grad()
        value_loss.backward()
        if self._world > 1:
            self.critic_opt.all_reduce_grad()
        self.critic_opt.step()
        self._stats += torch.stack([policy_loss.detach(), value_loss.detach(), entropy_loss.detach(), approx_kl,
                                    torch.ones((), device=self.device)])

    def _capture_minibatch(self, mb):
        """Capture `_minibatch` into a CUDA graph (one replay per minibatch instead of ~300 launches).
        The warm-up iterations torch requires before capture really train, so the trainable state is
        snapshotted and restored around them."""
        self._idx = torch.zeros(mb, dtype=torch.long, device=self.device)
        opts = (self.actor_opt, self.critic_opt)
        keep = [(o.flat.clone(), o.exp_avg.clone(), o.exp_avg_sq.clone(), o.step_t.clone()) for o in opts]
        stats = self._stats.clone()
        cur = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(3):
                self._minibatch(self._idx)
        cur.wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._minibatch(self._idx)
        for o, (f, m, v, st) in zip(opts, keep):
            o.flat.copy_(f); o.exp_avg.copy_(m); o.exp_avg_sq.copy_(v); o.step_t.copy_(st)
        self._stats.copy_(stats)
        return graph

    def _agree_minibatches(self, n_local):
        """Minibatch size and count every rank uses: each minibatch carries collectives (gradient all-reduce, KL pair),
        so ranks whose env shards differ in size (`dist.shard_envs` = np.array_split) must agree on the count —
        the smallest shard decides (ADVICE r1)."""
        n = n_local
        if self._world > 1:
            t = torch.tensor([n_local], dtype=torch.int64, device=self.device)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MIN)
            n = int(t.item())
        mb = max(1, min(int(self.cfg["mini_batch_size"]), n))
        return mb, n // mb

    def _native_minibatch(self, idx, mb):
        """One minibatch of `MAPPOAgent.update` (agent.py:702-772) on the hand-written kernels: actor gradient,
        [all-reduce], KL-gated Adam + repack; critic gradient, [all-reduce], Adam + repack.  No host synchronisation."""
        cfg, N, M, W = self.cfg, self.N, self.M, self._world
        a, c, ao, co = self.actor_net, self.critic_net, self.actor_opt, self.critic_opt
        norm = self._norm_args()
        a.grad(ao.grad, self.obs, N, M, idx, mb, critic=False, act=self.act, logp_old=self.logp, adv=self.adv,
               adv_stats=self._adv_stats, clip=cfg["clip_param"], entropy_coef=cfg["entropy_coef"],
               rows_global=mb * M * W, run_acc=self._run_actor, **norm)
        # (the critic's gradient does not depend on the actor's step: computed first so that ONE collective carries both)
        c.grad(co.grad, self.obs, N, M, idx, mb, critic=True, ret=self.ret, v_old=self.val, clip=cfg["clip_param"],
               use_clipped_value=bool(cfg["use_clipped_value"]), rows_global=mb * W, run_acc=self._run_critic, **norm)
        if W > 1:   # every rank must see the same gradients and take the same gate decision
            if self._peer is not None:
                self._peer.all_reduce(extra=a.stats[1:3])
            else:
                torch.distributed.all_reduce(self._joint_grad)
                torch.distributed.all_reduce(a.stats[1:3])
        a.adam_step(ao.flat, ao.exp_avg, ao.exp_avg_sq, ao.grad, ao.step_t, ao.lr, ao.betas, ao.eps,
                    kl_sum=a.stats[1:2], kl_rows=a.stats[2:3], target_kl=float(cfg["target_kl"]), gate_count=self._gates)
        c.adam_step(co.flat, co.exp_avg, co.exp_avg_sq, co.grad, co.step_t, co.lr, co.betas, co.eps)

    def _native_epoch(self, mb, num_mb):
        for i in range(num_mb):
            self._native_minibatch(self._perm[i * mb:(i + 1) * mb], mb)

    def _update_native(self) -> Dict[str, float]:
        cfg = self.cfg
        n = self.T * self.N
        mb, num_mb = self._agree_minibatches(n)
        if mb * self.M > self.actor_net.max_rows:
            raise RuntimeError("minibatch larger than the PpoNet scratch")
        self._run_actor.zero_()
        self._run_critic.zero_()
        use_graph = bool(cfg["graph_update"])
        if use_graph and (self._graph is None or self._graph_shape != (mb, num_mb)):
            if self._world > 1:      # the communicator must exist before a collective is captured
                torch.distributed.all_reduce(self._gates.clone())
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self._native_epoch(mb, num_mb)
            self._graph, self._graph_shape = graph, (mb, num_mb)
        for _ in range(int(cfg["opt_epochs"])):
            torch.randperm(n, device=self.device, generator=self.gen, out=self._perm)
            if use_graph:
                self._graph.replay()
            else:
                self._native_epoch(mb, num_mb)
        self._fused_stale = True
        ra, rc = self._run_actor.tolist(), self._run_critic.tolist()
        k = max(ra[2], 1.0)
        return {"policy_loss": ra[0] / k, "value_loss": rc[0] / max(rc[2], 1.0), "entropy_loss": ra[3] / k,
                "approx_kl": ra[1] / k}

    def _update(self) -> Dict[str, float]:
        if self.native:
            return self._update_native()
        cfg = self.cfg
        n = self.T * self.N
        mb, num_mb = self._agree_minibatches(n)
        if num_mb > 8192 and not getattr(self, "_warned_mb", False):
            import warnings
            warnings.warn(f"{num_mb} minibatches of {mb} samples per epoch: mini_batch_size is the reference's default "
                          f"(mappo/config.py:32) sized for a handful of envs; with {self.N} envs use e.g. {max(mb, n // 64)}")
            self._warned_mb = True
        if not hasattr(self, "_stats"):
            self._stats = torch.zeros(5, device=self.device)
        self._stats.zero_()
        use_graph = bool(cfg["graph_update"]) and self._world == 1
        if use_graph and (self._graph is None or self._idx.numel() != mb):
            self._graph = self._capture_minibatch(mb)
        for _ in range(int(cfg["opt_epochs"])):
            perm = torch.randperm(n, device=self.device, generator=self.gen)
            for i in range(num_mb):
                if use_graph:
                    self._idx.copy_(perm[i * mb:(i + 1) * mb])
                    self._graph.replay()
                else:
                    self._minibatch(perm[i * mb:(i + 1) * mb])
        self._fused_stale = True
        s = (self._stats[:4] / self._stats[4]).tolist()
        return {"policy_loss": s[0], "value_loss": s[1], "entropy_loss": s[2], "approx_kl": s[3]}

    # --------------------------------------------------------------------- loop
    def pop_episode_stats(self):
        """Mean return / length of the episodes finished since the last call (all ranks)."""
        s = self.env.episode_stats(reset=True)
        return reduce_episode_stats(s[0], s[1], s[2])

    def train_step(self) -> Dict[str, float]:
        t0 = time.time()
        self.collect_rollout()
        self.compute_returns()
        res = self.update()
        mean_r, mean_l, n_ep = self.pop_episode_stats()
        torch.cuda.synchronize(self.device)
        res.update(ep_return=mean_r, ep_length=mean_l, episodes=n_ep, total_env_steps=self.total_env_steps,
                   step_time=time.time() - t0)
        return res

    def learn(self, max_env_steps: int, log=None):
        history = []
        while self.total_env_steps < max_env_steps:
            res = self.train_step()
            history.append(res)
            if log is not None:
                log(res)
        return history

    @torch.no_grad()
    def select_action(self, obs: torch.Tensor, deterministic: bool = True) -> torch.Tensor:
        """`MAPPO.select_action` (mappo.py:272-287): mean action for evaluation."""
        if self.norm_obs:   # evaluation reads the frozen statistics (mappo.py:537,549)
            m, r = self.obs_normalizer.rms.stats()
            c = float(self.cfg["clip_obs"])
            obs = ((obs.reshape(-1, self.M * self.D) - m) * r).clamp(-c, c).view(obs.shape)
        if self.native and obs.dim() == 3 and obs.is_contiguous():
            n = obs.shape[0]         # obs is already normalised above: no per-slot statistics here
            mean = self.actor_net.forward(obs, n, self.M, n * self.M).view(n, self.M, self.A)
        else:
            mean = self.ac.actor(obs.reshape(-1, self.D)).view(*obs.shape[:-1], self.A)
        if deterministic:
            return mean
        return mean + self.ac.logstd.exp() * torch.randn(mean.shape, device=mean.device, generator=self.gen)

    @torch.no_grad()
    def run(self, env: Optional[BatchAviary] = None, n_episodes: int = 10, max_steps: Optional[int] = None):
        """`MAPPO.run` (mappo.py:534-581): evaluation with the current policy — deterministic actions, frozen
        observation statistics — returning `{'ep_returns', 'ep_lengths'}` of `n_episodes` episodes.  The reference
        plays them one after the other in a single env; here `env` (default: a fresh aviary configured like the
        training one with `n_episodes` envs, no auto-reset) plays one episode per env in parallel, each env counted
        up to its first `done`.  The per-step return is the env reward, = `mean(r)` over agents of the tiled reward
        (`record_episode_statistics.py:148`)."""
        own = env is None
        if own:
            t = self.env
            env = BatchAviary(task=t.task, num_envs=int(n_episodes), drone_model=t.DRONE_MODEL, num_drones=t.NUM_DRONES,
                              initial_xyzs=np.asarray(t.INIT_XYZS, dtype=np.float64).reshape(-1, 3)[:t.NUM_DRONES],
                              physics=t.PHYSICS, pyb_freq=t.PYB_FREQ, ctrl_freq=t.CTRL_FREQ, act=t.ACT_TYPE,
                              precision=t.precision, device=self.device, auto_reset=False, seed=12345)
        if env.auto_reset:
            raise ValueError("run() needs an aviary with auto_reset=False (episodes are counted up to their first done)")
        n = env.num_envs
        obs = env.reset_device()
        ret = torch.zeros(n, dtype=torch.float64, device=self.device)
        length = torch.zeros(n, dtype=torch.int64, device=self.device)
        alive = torch.ones(n, dtype=torch.bool, device=self.device)
        horizon = int(max_steps) if max_steps is not None else int(env.EPISODE_LEN_SEC * env.CTRL_FREQ) + 2
        for _ in range(horizon):
            res = env.step_device(self.select_action(obs, deterministic=True).to(env.action_dtype))
            ret += torch.where(alive, res.reward.double(), torch.zeros_like(ret))
            length += alive.long()
            alive &= ~res.done
            obs = res.obs
            if not bool(alive.any()):      # one scalar read-back per control step (evaluation is not the hot path)
                break
        out = {"ep_returns": ret.cpu().numpy(), "ep_lengths": length.cpu().numpy()}
        if own:
            env.close()
        return out

    def state_dict(self):
        """The reference's checkpoint layout (`MAPPO.save`, mappo/mappo.py:203-232): `agent` =
        {`ac` with the reference's parameter names, `actor_opt`, `critic_opt`}, `obs_normalizer`,
        `reward_normalizer`, `total_steps`, `obs` (the current, normalised observation).  With
        `save_env_state=True` one more key, `resume`, carries the simulator snapshot and the rollout loop's state
        (`_resume_state`); `load_state_dict` applies it whenever it is present."""
        sd = {"agent": {"ac": self.ac.reference_state_dict(), "actor_opt": self.actor_opt.state_dict(),
                        "critic_opt": self.critic_opt.state_dict()},
              "obs_normalizer": self.obs_normalizer.state_dict(),
              "reward_normalizer": self.reward_normalizer.state_dict(),
              "total_steps": self.total_env_steps,
              # mappo.py:203-229: the reference stores its RNG states so that a resumed run continues the stream
              "random_state": {"torch_generator": self.gen.get_state().cpu(),
                               "fused_calls": int(self.fused._calls) if self.fused is not None else 0},
              "env_random_state": [{"philox": self.env.get_rng_state()}]}
        t = self._current_slot()
        if self._reset_done:
            sd["obs"] = self._normed(self.obs[t], t).cpu().numpy()
        if self.cfg["save_env_state"]:
            sd["resume"] = self._resume_state(t)
        return sd

    def _current_slot(self):
        """Rollout slot holding the observation the next rollout starts from."""
        return self.T if self.total_env_steps > 0 and not self._resumed else 0

    def _shard(self):
        """(rank, world, env offset, env count) of this process's env shard; collective when world > 1."""
        rank = torch.distributed.get_rank() if torch.distributed.is_initialized() else 0
        offset = 0
        if self._world > 1:
            counts = torch.zeros(self._world, dtype=torch.int64, device=self.device)
            torch.distributed.all_gather_into_tensor(counts, torch.tensor([self.N], dtype=torch.int64, device=self.device))
            offset = int(counts[:rank].sum())
        return rank, self._world, offset, self.N

    def _resume_state(self, t):
        """What `load_state_dict` needs besides the reference-layout keys to continue mid-episode: the simulator
        snapshot, the raw observation slot the next rollout starts from (with its normaliser statistics), the
        normalisers' internals and the fused actor's noise seed.  With several ranks every rank saves its own shard."""
        rank, world, offset, count = self._shard()
        res = {"env": self.env.snapshot().cpu(), "rank": rank, "world": world, "env_offset": offset, "env_count": count,
               "reset_done": self._reset_done, "fused_seed": int(self._fused_seed)}
        if self._reset_done and self.norm_obs:   # without norm_obs, sd["obs"] already is the raw slot
            res["obs"] = self.obs[t].cpu()
            res["nmean"], res["nrstd"] = self.nmean[t].cpu(), self.nrstd[t].cpu()
        if self.norm_obs:
            res["obs_count"] = self.obs_normalizer.rms.count
        rn = self.reward_normalizer
        if isinstance(getattr(rn, "count", None), torch.Tensor):
            res["reward_count"] = rn.count.cpu()
            res["reward_ret"] = rn.ret.cpu() if rn.ret is not None else None
        return res

    def _load_resume(self, res, sd):
        rank, world, offset, count = self._shard()
        got = (res.get("rank"), res.get("world"), res.get("env_offset"), res.get("env_count"))
        if got != (rank, world, offset, count):
            raise ValueError(f"[ERROR] in DeviceMAPPO.load(), the checkpoint's env state belongs to rank {got[0]} of "
                             f"{got[1]} (envs {got[2]}..{got[2] + got[3] - 1 if got[3] else '?'}); this process is rank "
                             f"{rank} of {world} (envs {offset}..{offset + count - 1}). Re-sharding is not supported")
        if self.norm_obs and res.get("reset_done") and "nmean" not in res:
            raise ValueError("[ERROR] in DeviceMAPPO.load(), the checkpoint was saved without norm_obs")
        self.env.restore(res["env"])
        if res.get("reset_done"):
            raw = res["obs"] if "obs" in res else sd["obs"]
            self.obs[0].copy_(torch.as_tensor(raw).to(self.device))
            if self.norm_obs:
                self.nmean[0].copy_(res["nmean"].to(self.device))
                self.nrstd[0].copy_(res["nrstd"].to(self.device))
            self._reset_done = self._resumed = True
        else:
            self._reset_done = self._resumed = False
        if self.norm_obs and "obs_count" in res:
            self.obs_normalizer.rms.set(count=res["obs_count"])
        rn = self.reward_normalizer
        if "reward_count" in res and isinstance(getattr(rn, "count", None), torch.Tensor):
            rn.count = res["reward_count"].to(self.device)
            rn.ret = res["reward_ret"].to(self.device) if res["reward_ret"] is not None else None
        self._fused_seed = int(res["fused_seed"])

    def load_state_dict(self, sd):
        self.ac.load_reference_state_dict(sd["agent"]["ac"])
        self.actor_opt.load_state_dict(sd["agent"]["actor_opt"])
        self.critic_opt.load_state_dict(sd["agent"]["critic_opt"])
        if sd.get("obs_normalizer"):
            self.obs_normalizer.load_state_dict(sd["obs_normalizer"])
        if sd.get("reward_normalizer"):
            self.reward_normalizer.load_state_dict(sd["reward_normalizer"])
        self.total_env_steps = int(sd.get("total_steps", 0))
        rs = sd.get("random_state")
        if rs:
            self.gen.set_state(torch.as_tensor(rs["torch_generator"], dtype=torch.uint8).cpu())
            if self.fused is not None:
                self.fused._calls = int(rs.get("fused_calls", 0))
        ers = sd.get("env_random_state")
        if ers and isinstance(ers[0], dict) and "philox" in ers[0]:
            self.env.set_rng_state(ers[0]["philox"])
        if sd.get("resume") is not None:   # saved with save_env_state=True: continue mid-episode
            self._load_resume(sd["resume"], sd)
        self._fused_stale = True
        self._graph = None          # captured graphs have the old hyper-parameters (lr, betas) baked in
        self._pack_native()

    def close(self):
        """Release the captured update graph and the native networks.  With several ranks the graph holds NCCL collectives:
        it has to go BEFORE `torch.distributed.destroy_process_group()`, which otherwise waits forever for work the
        communicator still references."""
        self._graph = None
        torch.cuda.synchronize(self.device)
        for net in (self.actor_net, self.critic_net):
            if net is not None:
                net.close()
        self.actor_net = self.critic_net = None
        if getattr(self, "_peer", None) is not None:
            self.actor_opt.grad = self.critic_opt.grad = self._joint_grad = None
            self._peer.close()
            self._peer = None

    def save(self, path):
        torch.save(self.state_dict(), path)

    def load(self, path):
        self.load_state_dict(torch.load(path, map_location=self.device, weights_only=False))
