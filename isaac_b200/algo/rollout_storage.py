"""`RolloutStorage` with the reference's interface (algo/ppo/rollout_storage.py:35-182); GAE runs
in the CUDA scan kernel `hb_gae_returns` + `hb_gae_normalize` (C ABI, include/hector_b200.h).

Layout: time-major `[T, N, ·]` fp32 tensors in HBM like the reference.  The observation
buffers keep a padded leading dimension (640 / 1056 floats: whole 128-byte rows) so that every row starts on a
16-byte boundary — the alignment TMA tensor maps need for the MLP GEMMs — and expose
`[T, N, 615]` / `[T, N, 1050]` views under the reference's attribute names.
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import _lib
from .actor_critic import pitch


_FUSED_SCRATCH = {}


def gae_compute_returns(rewards, values, dones, last_values, returns, advantages, gamma, lam,
                        stats: Optional[torch.Tensor] = None, reduce_stats=None, fused: bool = True):
    """rollout_storage.py:122-136 on `[T,N,1]` (or `[T,N]`) CUDA tensors, in place into returns/advantages.
    Single GPU (no `reduce_stats`): ONE launch, `hb_gae_fused` (raw advantages stay in registers across a grid barrier on
    their statistics).  `reduce_stats(stats, count) -> count` lets a multi-GPU caller all-reduce (sum, sum sq) and the
    sample count across ranks between the two passes of the two-kernel form (SURVEY.md §8e)."""
    lib = _lib.load()
    T, N = rewards.shape[0], rewards.shape[1]
    for t in (rewards, values, dones, last_values, returns, advantages):
        if not (t.is_cuda and t.is_contiguous()):
            raise ValueError("gae_compute_returns needs contiguous CUDA tensors")
    if dones.dtype not in (torch.uint8, torch.bool):
        raise TypeError("dones must be uint8/bool")
    st = torch.cuda.current_stream(rewards.device).cuda_stream
    if fused and reduce_stats is None and stats is None and T * N > 1:
        scratch = _FUSED_SCRATCH.get(rewards.device)
        if scratch is None:          # HB_GAE_SCRATCH_DOUBLES {8 sums, 8 sums of squares, ticket}: zeroed once, re-armed by every launch
            scratch = _FUSED_SCRATCH[rewards.device] = torch.zeros(32, dtype=torch.float64, device=rewards.device)
        _lib.check(lib.hb_gae_fused(rewards.data_ptr(), values.data_ptr(), dones.data_ptr(), last_values.data_ptr(),
                                    returns.data_ptr(), advantages.data_ptr(), scratch.data_ptr(), T, N,
                                    float(gamma), float(lam), st), "hb_gae_fused")
        return returns, advantages
    if stats is None:
        stats = torch.empty(2, dtype=torch.float64, device=rewards.device)
    _lib.check(lib.hb_gae_returns(rewards.data_ptr(), values.data_ptr(), dones.data_ptr(), last_values.data_ptr(),
                                  returns.data_ptr(), advantages.data_ptr(), stats.data_ptr(), T, N,
                                  float(gamma), float(lam), st), "hb_gae_returns")
    count = T * N                       # samples behind `stats` (all ranks after reduce_stats)
    if reduce_stats is not None:
        count = reduce_stats(stats, count)
    if count > 1:
        _lib.check(lib.hb_gae_normalize_n(advantages.data_ptr(), stats.data_ptr(), int(count), T * N, st),
                   "hb_gae_normalize_n")
    return returns, advantages


class RolloutStorage:
    class Transition:
        def __init__(self):
            self.observations = None
            self.critic_observations = None
            self.actions = None
            self.rewards = None
            self.dones = None
            self.values = None
            self.actions_log_prob = None
            self.action_mean = None
            self.action_sigma = None
            self.hidden_states = None

        def clear(self):
            self.__init__()

    def observation_slot(self, k: int):
        """([N, num_obs], [N, num_privileged_obs]) views of slot k, 0 <= k <= T, at the storage's row pitch."""
        return (self._observations[k][:, :self.obs_shape[0]],
                self._privileged_observations[k][:, :self.privileged_obs_shape[0]])

    def __init__(self, num_envs, num_transitions_per_env, obs_shape, privileged_obs_shape, actions_shape,
                 device="cuda:0"):
        self.device = device
        self.obs_shape, self.privileged_obs_shape, self.actions_shape = obs_shape, privileged_obs_shape, actions_shape
        T, N = num_transitions_per_env, num_envs
        z = lambda *s, **kw: torch.zeros(*s, device=device, **kw)
        # rows at a 16-byte pitch (TMA operands), and one slot more than the reference's [T, N, *]: slot T receives the
        # observations that follow the last transition when the env writes straight into the storage
        # (PPO.attach_env; they become slot 0 of the next rollout)
        # (pitch = ceil32(width + 1): there is always room for the constant ones column the weight-gradient GEMM reads)
        self.obs_ld = pitch(obs_shape[0] + 1)
        self._observations = z(T + 1, N, self.obs_ld)
        self.observations = self._observations[:T, :, :obs_shape[0]]
        if privileged_obs_shape[0] is not None:
            self.priv_ld = pitch(privileged_obs_shape[0] + 1)
            self._privileged_observations = z(T + 1, N, self.priv_ld)
            self.privileged_observations = self._privileged_observations[:T, :, :privileged_obs_shape[0]]
        else:
            # no privileged observations: the critic reads the actor's (rollout_storage.py:157-160); the padded
            # buffer is shared so that the update's gathers work unchanged
            self.privileged_observations = None
            self.privileged_obs_shape = [obs_shape[0]]
            self.priv_ld, self._privileged_observations = self.obs_ld, self._observations
        self.rewards = z(T, N, 1)
        self.actions = z(T, N, *actions_shape)
        self.dones = z(T, N, 1, dtype=torch.uint8)
        self.actions_log_prob = z(T, N, 1)
        self.values = z(T, N, 1)
        self.returns = z(T, N, 1)
        self.advantages = z(T, N, 1)
        self.mu = z(T, N, *actions_shape)
        self.sigma = z(T, N, *actions_shape)
        self.num_transitions_per_env, self.num_envs = T, N
        self.saved_hidden_states_a = self.saved_hidden_states_c = None
        self.step = 0
        self.reduce_stats = None          # set by the multi-GPU wrapper

    def add_transitions(self, transition: "RolloutStorage.Transition"):
        if self.step >= self.num_transitions_per_env:
            raise AssertionError("Rollout buffer overflow")
        t = self.step
        self.observations[t].copy_(transition.observations)
        if self.privileged_observations is not None:
            self.privileged_observations[t].copy_(transition.critic_observations)
        self.actions[t].copy_(transition.actions)
        self.rewards[t].copy_(transition.rewards.view(-1, 1))
        self.dones[t].copy_(transition.dones.view(-1, 1))
        self.values[t].copy_(transition.values)
        self.actions_log_prob[t].copy_(transition.actions_log_prob.view(-1, 1))
        self.mu[t].copy_(transition.action_mean)
        self.sigma[t].copy_(transition.action_sigma)
        self.step += 1

    def clear(self):
        self.step = 0

    def compute_returns(self, last_values, gamma, lam):
        gae_compute_returns(self.rewards, self.values, self.dones, last_values.contiguous(), self.returns,
                            self.advantages, gamma, lam, reduce_stats=self.reduce_stats)

    def get_statistics(self):
        done = self.dones
        done[-1] = 1
        flat_dones = done.permute(1, 0, 2).reshape(-1, 1)
        done_indices = torch.cat((flat_dones.new_tensor([-1], dtype=torch.int64), flat_dones.nonzero(as_tuple=False)[:, 0]))
        trajectory_lengths = done_indices[1:] - done_indices[:-1]
        return trajectory_lengths.float().mean(), self.rewards.mean()

    def mini_batch_generator(self, num_mini_batches, num_epochs=8):
        """rollout_storage.py:146-182, for code that walks the storage itself (PPO.update() does not: it gathers the
        minibatches once per update with hb_ppo_gather_rows / hb_ppo_pack_samples and feeds the GEMMs from there).
        Same contract: ONE permutation of the first num_mini_batches * (T*N // num_mini_batches) samples, reused by
        every epoch; yields (obs, critic_obs, actions, target_values, advantages, returns, old_log_prob, old_mu,
        old_sigma, (None, None), None) per minibatch."""
        per_batch = self.num_envs * self.num_transitions_per_env // num_mini_batches
        order = torch.randperm(num_mini_batches * per_batch, device=self.device)
        critic_src = self.privileged_observations if self.privileged_observations is not None else self.observations
        fields = [t.flatten(0, 1) for t in (self.observations, critic_src, self.actions, self.values, self.advantages,
                                            self.returns, self.actions_log_prob, self.mu, self.sigma)]
        for _ in range(num_epochs):
            for chunk in order.split(per_batch):
                yield (*(f[chunk] for f in fields), (None, None), None)
