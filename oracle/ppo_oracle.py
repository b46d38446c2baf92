"""TEST INFRASTRUCTURE — CPU oracle for the RL stage (not a product path).

torch-on-CPU restatement of the rsl_rl fork under humanoid/algo/ppo of DRCL-USC/isaac:
rollout storage + GAE (rollout_storage.py:52-136), minibatch generator (:146-182),
ActorCritic MLPs with a diagonal Gaussian head (actor_critic.py:36-128) and the PPO
act / process_env_step / compute_returns / update cycle (ppo.py:91-184).

`torch` itself (nn.functional.linear/elu, autograd, optim.Adam, clip_grad_norm_) is
part of the oracle: the reference pins no torch version (setup.py:43-52).

Pinned against the unmodified reference by `tests/test_oracle_pinning.py` (live where the
reference is found, see `oracle/ref_harness.py`; via golden vectors everywhere).  Random draws are injected: `eps` for
the action sample (a = mu + sigma*eps) and the minibatch permutation.

Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference`
legs of `bench.py` may import this module.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

HALF_LOG_2PI = math.log(math.sqrt(2 * math.pi))


def init_actor_critic_params(num_obs=615, num_critic_obs=1050, num_actions=10,
                             actor_hidden=(512, 256, 128), critic_hidden=(768, 256, 128),
                             init_noise_std=1.0, seed=0) -> Dict[str, torch.Tensor]:
    """Parameters with the reference's state_dict keys and torch's default nn.Linear init
    (actor_critic.py:54-83: `actor.{0,2,4,6}`, `critic.{0,2,4,6}`, `std`)."""
    g = torch.Generator().manual_seed(seed)
    p: Dict[str, torch.Tensor] = {"std": init_noise_std * torch.ones(num_actions)}
    for net, dims in (("actor", (num_obs, *actor_hidden, num_actions)),
                      ("critic", (num_critic_obs, *critic_hidden, 1))):
        for i in range(len(dims) - 1):
            bound = 1.0 / math.sqrt(dims[i])
            p[f"{net}.{2 * i}.weight"] = (torch.rand(dims[i + 1], dims[i], generator=g) * 2 - 1) * bound
            p[f"{net}.{2 * i}.bias"] = (torch.rand(dims[i + 1], generator=g) * 2 - 1) * bound
    return p


PARAM_ORDER = (["std"] + [f"actor.{i}.{w}" for i in (0, 2, 4, 6) for w in ("weight", "bias")]
               + [f"critic.{i}.{w}" for i in (0, 2, 4, 6) for w in ("weight", "bias")])


def mlp(params, net: str, x: torch.Tensor) -> torch.Tensor:
    """Linear-ELU x3, Linear (actor_critic.py:54-77)."""
    for i in (0, 2, 4):
        x = F.elu(F.linear(x, params[f"{net}.{i}.weight"], params[f"{net}.{i}.bias"]))
    return F.linear(x, params[f"{net}.6.weight"], params[f"{net}.6.bias"])


def gaussian_log_prob(a, mu, sigma):
    """torch.distributions.Normal.log_prob summed over actions (actor_critic.py:119-120)."""
    var = sigma ** 2
    return (-((a - mu) ** 2) / (2 * var) - sigma.log() - HALF_LOG_2PI).sum(dim=-1)


def gaussian_entropy(sigma):
    """Normal.entropy summed over actions (actor_critic.py:107-109)."""
    return (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(sigma)).sum(dim=-1)


def gae_returns(rewards, values, dones, last_values, gamma, lam):
    """rollout_storage.py:122-136.  rewards/values [T,N,1], dones uint8 [T,N,1]."""
    T = rewards.shape[0]
    returns = torch.zeros_like(rewards)
    adv = 0
    for t in reversed(range(T)):
        nxt = last_values if t == T - 1 else values[t + 1]
        not_terminal = 1.0 - dones[t].float()
        delta = rewards[t] + not_terminal * gamma * nxt - values[t]
        adv = delta + not_terminal * gamma * lam * adv
        returns[t] = adv + values[t]
    advantages = returns - values
    advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
    return returns, advantages


class OraclePPO:
    def __init__(self, params: Dict[str, torch.Tensor], num_envs: int, num_steps: int,
                 num_learning_epochs=1, num_mini_batches=1, clip_param=0.2, gamma=0.998, lam=0.95,
                 value_loss_coef=1.0, entropy_coef=0.0, learning_rate=1e-3, max_grad_norm=1.0,
                 use_clipped_value_loss=True, schedule="fixed", desired_kl=0.01):
        self.params = {k: params[k].clone().requires_grad_(True) for k in PARAM_ORDER}
        self.optimizer = torch.optim.Adam([self.params[k] for k in PARAM_ORDER], lr=learning_rate)   # ppo.py:68
        self.learning_rate = learning_rate
        self.epochs, self.mini_batches = num_learning_epochs, num_mini_batches
        self.clip_param, self.gamma, self.lam = clip_param, gamma, lam
        self.value_loss_coef, self.entropy_coef = value_loss_coef, entropy_coef
        self.max_grad_norm, self.use_clipped_value_loss = max_grad_norm, use_clipped_value_loss
        self.schedule, self.desired_kl = schedule, desired_kl
        T, N = num_steps, num_envs
        nobs = self.params["actor.0.weight"].shape[1]
        npriv = self.params["critic.0.weight"].shape[1]
        nact = self.params["std"].shape[0]
        z = torch.zeros
        self.st = dict(observations=z(T, N, nobs), privileged_observations=z(T, N, npriv),
                       actions=z(T, N, nact), rewards=z(T, N, 1), dones=z(T, N, 1).byte(),
                       actions_log_prob=z(T, N, 1), values=z(T, N, 1), returns=z(T, N, 1),
                       advantages=z(T, N, 1), mu=z(T, N, nact), sigma=z(T, N, nact))
        self.T, self.N, self.step = T, N, 0
        self._tr = None

    # ppo.py:91-101
    @torch.no_grad()
    def act(self, obs, critic_obs, eps):
        mu = mlp(self.params, "actor", obs)
        sigma = mu * 0.0 + self.params["std"]
        actions = mu + sigma * eps
        values = mlp(self.params, "critic", critic_obs)
        self._tr = dict(observations=obs, privileged_observations=critic_obs, actions=actions, values=values,
                        actions_log_prob=gaussian_log_prob(actions, mu, sigma), mu=mu, sigma=sigma)
        return actions

    # ppo.py:103-113 + rollout_storage.py:87-100
    @torch.no_grad()
    def process_env_step(self, rewards, dones, infos):
        tr = self._tr
        r = rewards.clone()
        if "time_outs" in infos:
            r += self.gamma * torch.squeeze(tr["values"] * infos["time_outs"].unsqueeze(1), 1)
        if self.step >= self.T:
            raise AssertionError("Rollout buffer overflow")
        s, t = self.st, self.step
        for k in ("observations", "privileged_observations", "actions", "values", "mu", "sigma"):
            s[k][t].copy_(tr[k])
        s["rewards"][t].copy_(r.view(-1, 1))
        s["dones"][t].copy_(dones.view(-1, 1))
        s["actions_log_prob"][t].copy_(tr["actions_log_prob"].view(-1, 1))
        self.step += 1

    # ppo.py:115-117
    @torch.no_grad()
    def compute_returns(self, last_critic_obs):
        last_values = mlp(self.params, "critic", last_critic_obs)
        self.st["returns"], self.st["advantages"] = gae_returns(
            self.st["rewards"], self.st["values"], self.st["dones"], last_values, self.gamma, self.lam)

    # ppo.py:119-184 with rollout_storage.py:146-182 inlined
    def update(self, perm: torch.Tensor):
        """`perm` = the torch.randperm(num_mini_batches*mini_batch_size) draw (quirk 8: drawn once)."""
        B = self.N * self.T
        mb = B // self.mini_batches
        flat = {k: v.flatten(0, 1) for k, v in self.st.items()}
        mean_v = mean_s = 0.0
        plist = [self.params[k] for k in PARAM_ORDER]
        self.kl_trace: List[float] = []
        self.lr_trace: List[float] = []
        for _ in range(self.epochs):
            for i in range(self.mini_batches):
                idx = perm[i * mb:(i + 1) * mb]
                obs, cobs = flat["observations"][idx], flat["privileged_observations"][idx]
                a, v_old, adv, ret = flat["actions"][idx], flat["values"][idx], flat["advantages"][idx], flat["returns"][idx]
                lp_old, mu_old, sig_old = flat["actions_log_prob"][idx], flat["mu"][idx], flat["sigma"][idx]
                mu = mlp(self.params, "actor", obs)
                sigma = mu * 0.0 + self.params["std"]
                lp = gaussian_log_prob(a, mu, sigma)
                v = mlp(self.params, "critic", cobs)
                ent = gaussian_entropy(sigma)
                if self.desired_kl is not None and self.schedule == "adaptive":
                    with torch.inference_mode():
                        kl = torch.sum(torch.log(sigma / sig_old + 1.e-5)
                                       + (torch.square(sig_old) + torch.square(mu_old - mu)) / (2.0 * torch.square(sigma))
                                       - 0.5, axis=-1)
                        kl_mean = torch.mean(kl)
                        if kl_mean > self.desired_kl * 2.0:
                            self.learning_rate = max(1e-5, self.learning_rate / 1.5)
                        elif kl_mean < self.desired_kl / 2.0 and kl_mean > 0.0:
                            self.learning_rate = min(1e-2, self.learning_rate * 1.5)
                        for g in self.optimizer.param_groups:
                            g["lr"] = self.learning_rate
                        self.kl_trace.append(float(kl_mean))
                self.lr_trace.append(self.learning_rate)
                ratio = torch.exp(lp - torch.squeeze(lp_old))
                s1 = -torch.squeeze(adv) * ratio
                s2 = -torch.squeeze(adv) * torch.clamp(ratio, 1.0 - self.clip_param, 1.0 + self.clip_param)
                surrogate = torch.max(s1, s2).mean()
                if self.use_clipped_value_loss:
                    v_clip = v_old + (v - v_old).clamp(-self.clip_param, self.clip_param)
                    value_loss = torch.max((v - ret).pow(2), (v_clip - ret).pow(2)).mean()
                else:
                    value_loss = (ret - v).pow(2).mean()
                loss = surrogate + self.value_loss_coef * value_loss - self.entropy_coef * ent.mean()
                self.optimizer.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(plist, self.max_grad_norm)
                self.optimizer.step()
                mean_v += value_loss.item()
                mean_s += surrogate.item()
        n = self.epochs * self.mini_batches
        self.step = 0
        return mean_v / n, mean_s / n
