"""ctypes front end of the hand-written PPO-update kernels (`csrc/bd_ppo.cu`, C-ABI `bd_ppo_*`).

`PpoNet` holds one 3-layer tanh MLP (the MAPPO actor: in = obs_dim, rows = (sample, agent); or the centralised critic:
in = M chunks of obs_dim, rows = samples) in the form the tensor-core kernels read — bf16 K-step slabs repacked from the
fp32 master parameters, which stay where `optim.GatedAdam` keeps them (one flat fp32 buffer in torch's parameter order,
so checkpoints and the NCCL gradient all-reduce are unchanged).  Reference: `MAPPOAgent.update` /
`compute_policy_loss` / `compute_value_loss` (`mappo/agent.py:602-772`), `_compute_single_agent_returns`
(`mappo/buffer.py:561-614`).  There is no fallback: without the built library or a CUDA device the calls raise.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _native


def _p(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class PpoNet:
    HIDDEN = 256

    def __init__(self, in_dim: int, chunks: int, out_dim: int, has_logstd: bool, max_rows: int, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("PpoNet needs a CUDA device; there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.in_dim, self.chunks, self.out_dim, self.has_logstd = int(in_dim), int(chunks), int(out_dim), bool(has_logstd)
        self.max_rows = int(max_rows)
        self._lib = _native.load()
        self._h = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        rc = self._lib.bd_ppo_net_create(self.in_dim, self.chunks, self.out_dim, int(self.has_logstd), self.max_rows, idx,
                                         C.byref(self._h))
        self._check(rc, "bd_ppo_net_create")
        self.param_count = int(self._lib.bd_ppo_net_param_count(self._h))
        # statistics of the last bd_ppo_grad call, as a device tensor view: [0] sum loss, [1] sum (logp_old - logp),
        # [2] rows, [3:7] dlogstd sums, [7:11] db3 sums
        self.stats = self._wrap_stats()

    def _wrap_stats(self):
        ptr = self._lib.bd_ppo_net_stats(self._h)
        # a torch view of library-owned device memory (16 doubles), via the CUDA array interface
        class _Arr:
            pass
        a = _Arr()
        a.__cuda_array_interface__ = {"shape": (16,), "typestr": "<f8", "data": (int(ptr), False), "version": 2}
        with torch.cuda.device(self.device):
            return torch.as_tensor(a, device=self.device)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc, what):
        if rc != 0:
            raise _native.NativeError(f"{what} failed ({rc}): {self._lib.bd_ppo_last_error().decode()}")

    # ------------------------------------------------------------------------------------------------
    def pack(self, flat_params: torch.Tensor):
        """fp32 master parameters (flat, torch order: [logstd] W1 b1 W2 b2 W3 b3) -> bf16 tensor-core slabs."""
        if flat_params.dtype != torch.float32 or flat_params.numel() != self.param_count or not flat_params.is_contiguous():
            raise ValueError(f"flat_params must be a contiguous float32 tensor of {self.param_count} elements")
        self._check(self._lib.bd_ppo_net_pack(self._h, _p(flat_params), self._stream()), "bd_ppo_net_pack")

    def forward(self, obs: torch.Tensor, n_envs: int, n_agents: int, rows: int, idx: Optional[torch.Tensor] = None,
                nmean: Optional[torch.Tensor] = None, nrstd: Optional[torch.Tensor] = None, nclip: float = 10.0,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """out (rows, out_dim) = MLP(gathered rows of obs (slots, N, M, D)); critic nets read M chunks per row."""
        if out is None:
            out = torch.empty((rows, self.out_dim), device=self.device)
        self._check(self._lib.bd_ppo_forward(self._h, _p(obs), int(n_envs), int(n_agents), _p(idx), int(rows), _p(nmean),
                                             _p(nrstd), float(nclip), _p(out), self._stream()), "bd_ppo_forward")
        return out

    def sample(self, obs: torch.Tensor, out_act: torch.Tensor, out_logp: torch.Tensor, *, seed: int = 0, offset: int = 0,
               noise: Optional[torch.Tensor] = None, nmean=None, nrstd=None, nclip: float = 10.0,
               out_mean: Optional[torch.Tensor] = None):
        """Rollout-time policy step (`MAPPOActorCritic.step`, `mappo/agent.py:389-415`) in one launch: obs (N, M, D) of one
        slot -> out_act (N, M, A) = mean + exp(logstd) eps, out_logp (N, M[, 1]) = summed log-density.  eps = `noise`
        (N, M, A) standard normals, else Philox4x32-10 keyed by (seed; row, offset)."""
        N, M = int(obs.shape[0]), int(obs.shape[1])
        if out_act.numel() != N * M * self.out_dim or out_logp.numel() != N * M:
            raise ValueError("out_act / out_logp do not match obs (N, M, D)")
        self._check(self._lib.bd_ppo_sample(self._h, _p(obs), N, M, _p(nmean), _p(nrstd), float(nclip), _p(noise),
                                            int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), _p(out_act), _p(out_logp),
                                            _p(out_mean), self._stream()), "bd_ppo_sample")

    def grad(self, grad_out: torch.Tensor, obs: torch.Tensor, n_envs: int, n_agents: int, idx: Optional[torch.Tensor],
             samples: int, *, critic: bool, act=None, logp_old=None, adv=None, adv_stats=None, ret=None, v_old=None,
             clip: float = 0.2, use_clipped_value: bool = False, entropy_coef: float = 0.0, nmean=None, nrstd=None,
             nclip: float = 10.0, rows_global: int = 0, run_acc=None):
        """One minibatch: forward, loss, backward, weight gradients -> `grad_out` (flat, torch parameter order)."""
        self._check(self._lib.bd_ppo_grad(
            self._h, int(critic), _p(obs), int(n_envs), int(n_agents), _p(idx), int(samples), _p(act), _p(logp_old), _p(adv),
            _p(adv_stats), _p(ret), _p(v_old), float(clip), int(use_clipped_value), float(entropy_coef), _p(nmean), _p(nrstd),
            float(nclip), int(rows_global), _p(grad_out), _p(run_acc), self._stream()), "bd_ppo_grad")

    def adam_step(self, param, exp_avg, exp_avg_sq, grad, step, lr, betas=(0.9, 0.999), eps=1e-8, kl_sum=None, kl_rows=None,
                  target_kl: float = 0.0, gate_count=None):
        """torch.optim.Adam's step on the flat buffers, gated on the device by approx_kl <= 1.5 target_kl
        (`agent.py:731`), followed by the bf16 repack."""
        self._check(self._lib.bd_ppo_adam_step(
            self._h, _p(param), _p(exp_avg), _p(exp_avg_sq), _p(grad), _p(step), float(lr), float(betas[0]), float(betas[1]),
            float(eps), _p(kl_sum), _p(kl_rows), float(target_kl), _p(gate_count), self._stream()), "bd_ppo_adam_step")

    @property
    def launch_count(self):
        return int(self._lib.bd_ppo_launch_count(self._h))

    def close(self):
        if self._h:
            self._lib.bd_ppo_net_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def gae(rew, term, trunc, vals, gamma, lam, use_gae, ret, adv, acc3):
    """Returns / advantages of a whole rollout in ONE launch (`buffer.py:561-614`); acc3 += (sum adv, sum adv^2, count)."""
    lib = _native.load()
    T, N = rew.shape
    st = C.c_void_p(torch.cuda.current_stream(rew.device).cuda_stream)
    rc = lib.bd_ppo_gae(_p(rew), _p(term), _p(trunc), _p(vals), int(T), int(N), float(gamma), float(lam), int(bool(use_gae)),
                        _p(ret), _p(adv), _p(acc3), st)
    if rc != 0:
        raise _native.NativeError(f"bd_ppo_gae failed ({rc}): {lib.bd_ppo_last_error().decode()}")


def adv_stats(acc3, out2):
    """(sum, sum^2, count) -> (mean, 1/(std + 1e-8)) with `normalize_advantages`' rule (`buffer.py:666-695`)."""
    lib = _native.load()
    st = C.c_void_p(torch.cuda.current_stream(acc3.device).cuda_stream)
    rc = lib.bd_ppo_adv_stats(_p(acc3), _p(out2), st)
    if rc != 0:
        raise _native.NativeError(f"bd_ppo_adv_stats failed ({rc}): {lib.bd_ppo_last_error().decode()}")
