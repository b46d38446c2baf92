"""`PPO` with the reference's interface (algo/ppo/ppo.py:38-184) on the B200 kernels.

    act / process_env_step / compute_returns / update       same signatures and semantics
    actor_critic, optimizer.state_dict(), learning_rate, storage, transition   same attributes

Per minibatch step (hector's networks): 6 forward GEMMs (tcgen05, TF32 operands, fused bias + activation), one fused kernel for the two
output layers + the loss head (log-prob, clipped surrogate, clipped value loss, entropy, KL, their analytic
gradients, and the output layers' data / weight gradients), 4 data-gradient GEMMs (fused activation derivative), 6 split-K
weight-gradient GEMMs (bias gradients ride along as one more column), one gradient-norm reduction and one fused clip + Adam kernel that also applies the adaptive-KL learning-rate rule
on the device (no `.item()` sync per minibatch; the reference needs ~22, SURVEY.md §3.4).  The minibatch
permutation is drawn once per update and reused by every epoch (rollout_storage.py:149), so the index gathers
of `mini_batch_generator` are done once per update into minibatch-ordered buffers.
"""
from __future__ import annotations

import ctypes as C
from types import SimpleNamespace
from typing import Optional

import torch

from .. import _lib
from .._lib import (AdamParams, HB_OPT_TRACE_MAX, OPT_ERROR, OPT_LOSS_ACC, OPT_LR, OPT_STATS, OPT_STEP,
                    OPT_STEPS_IN_UPDATE, OPT_SUMSQ, OPT_TRACE, OPTIM_STATE_DOUBLES, PpoLossParams, ppo_rec)
from .actor_critic import ActorCritic, pad4, pitch
from .rollout_storage import RolloutStorage


class _AdamState:
    """torch.optim.Adam-compatible view of the fused optimizer state (on_policy_runner.py:281-282,291-293)."""

    def __init__(self, ppo: "PPO"):
        self._ppo = ppo
        self.param_groups = [{"lr": ppo._lr_host, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": 0,
                              "amsgrad": False, "params": list(range(len(self._views(ppo.actor_critic.flat))))}]

    def _views(self, buf):
        return [v for _, v in self._ppo.actor_critic.named_views(buf)]

    def state_dict(self):
        p = self._ppo
        state = {}
        if p._step > 0:
            exp_avg, exp_avg_sq = p._exp_avg, p._exp_avg_sq
            if p._peer is not None:          # sharded optimizer state: every rank owns a slice
                exp_avg, exp_avg_sq = p._peer.gather_sharded(exp_avg), p._peer.gather_sharded(exp_avg_sq)
            for i, (m, v) in enumerate(zip(self._views(exp_avg), self._views(exp_avg_sq))):
                state[i] = {"step": torch.tensor(float(p._step)), "exp_avg": m.clone().contiguous(),
                            "exp_avg_sq": v.clone().contiguous()}
        groups = [dict(self.param_groups[0], lr=p.learning_rate)]
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd):
        p = self._ppo
        for i, (m, v) in enumerate(zip(self._views(p._exp_avg), self._views(p._exp_avg_sq))):
            if i in sd["state"]:
                m.copy_(sd["state"][i]["exp_avg"].to(m.device))
                v.copy_(sd["state"][i]["exp_avg_sq"].to(v.device))
                p._set_step(int(sd["state"][i]["step"]))
        p.learning_rate = sd["param_groups"][0]["lr"]


class PPO:
    actor_critic: ActorCritic

    def __init__(self, actor_critic, num_learning_epochs=1, num_mini_batches=1, clip_param=0.2, gamma=0.998,
                 lam=0.95, value_loss_coef=1.0, entropy_coef=0.0, learning_rate=1e-3, max_grad_norm=1.0,
                 use_clipped_value_loss=True, schedule="fixed", desired_kl=0.01, device="cuda:0"):
        self._lib = _lib.load(check_device=True)
        self.device = torch.device(device)
        self.desired_kl, self.schedule = desired_kl, schedule
        self.actor_critic = actor_critic
        self.actor_critic.to(self.device)
        self.storage: Optional[RolloutStorage] = None
        self.transition = RolloutStorage.Transition()
        self.clip_param, self.num_learning_epochs, self.num_mini_batches = clip_param, num_learning_epochs, num_mini_batches
        self.value_loss_coef, self.entropy_coef = value_loss_coef, entropy_coef
        self.gamma, self.lam, self.max_grad_norm = gamma, lam, max_grad_norm
        self.use_clipped_value_loss = use_clipped_value_loss
        n = actor_critic.flat.numel()
        self._exp_avg = torch.zeros(n, device=self.device)
        self._exp_avg_sq = torch.zeros(n, device=self.device)
        # hb_optim_state (include/hector_b200.h): learning rate, Adam step count, gradient norm, loss sums and the
        # per-step {KL, learning rate} trace of the current update, all device-resident
        self._opt = torch.zeros(OPTIM_STATE_DOUBLES, dtype=torch.float64, device=self.device)
        self._opt_i64 = self._opt.view(torch.int64)
        self._lr_dev = self._opt[OPT_LR:OPT_LR + 1]
        self._stats = self._opt[OPT_STATS:OPT_STATS + 4]
        self._loss_acc = self._opt[OPT_LOSS_ACC:OPT_LOSS_ACC + 4]
        self._per_update = self._opt[OPT_SUMSQ:OPT_STEP]             # grad_sumsq, stats, loss_acc: zeroed per update()
        self._step = 0
        self._lr_host = float(learning_rate)
        self._lr_dev.fill_(float(learning_rate))
        self._lr_dirty = False
        self.optimizer = _AdamState(self)
        self.grad_allreduce = None          # multi-GPU hook: fn(flat_grad) sums gradients over ranks (NCCL path)
        self._peer = None                   # multi-GPU: isaac_b200.parallel.PeerOptimizer (fused reduce + Adam + broadcast)
        self.world_size = 1
        self.injected_eps = None            # parity: the Normal.sample() draw of the next act()
        self.injected_perm = None           # parity: the randperm of the next update()
        self._recorded_slot = None          # rollout slot already filled by the fast path of act()
        self._env = None                    # env that writes its observations straight into the rollout slots (attach_env)
        self._slots = None                  # (storage, {k: views and addresses of rollout slot k}), see _slot
        self._xa = self._xc = self._rec = None      # minibatch-ordered gathers of prepare_minibatches
        self.graph_rollout = True           # PPO.act: replay the hidden-layer GEMMs from a CUDA graph for small shards
        self.graph_rollout_max_envs = 16384
        self._act_graphs, self._act_stages = {}, {}
        # the action sample's N(0,1) draws come from the library's Philox generator (hb_ppo_draw_normal): call counter
        # AND key live on the device ({counter, ticket, key}), so the draw can sit inside the replayed act graph and
        # still follow seed()
        self._eps_state = torch.zeros(3, dtype=torch.int64, device=self.device)
        self.seed(0x9E3779B97F4A7C15)
        # update(): one CUDA graph per minibatch index (forward, loss head, backward, optimizer step), captured on the
        # second update and replayed for every epoch of every later update (single-GPU; data-parallel replicas launch
        # eagerly around their gradient all-reduce)
        self.graph_update = True
        self._update_graphs = {}
        self._updates_done = 0

    # ------------------------------------------------------------------ learning rate (device-resident)
    @property
    def learning_rate(self) -> float:
        if self._lr_dirty:
            self._lr_host = float(self._lr_dev.item())
            self._lr_dirty = False
        return self._lr_host

    @learning_rate.setter
    def learning_rate(self, v: float):
        self._lr_host = float(v)
        self._lr_dev.fill_(float(v))
        self._lr_dirty = False

    def init_storage(self, num_envs, num_transitions_per_env, actor_obs_shape, critic_obs_shape, action_shape):
        self.storage = RolloutStorage(num_envs, num_transitions_per_env, actor_obs_shape, critic_obs_shape,
                                      action_shape, self.device)
        self._act_graphs.clear()            # they address the previous storage's slots
        self._slots = None

    def test_mode(self):
        self.actor_critic.eval()

    def train_mode(self):
        self.actor_critic.train()

    # ------------------------------------------------------------------ rollout (ppo.py:91-117)
    def attach_env(self, env) -> None:
        """SURVEY.md §8(f) rank 1: from now on act() tells `env` (an isaac_b200 env) to write the observations of
        its next step() straight into the rollout slot act() will record them in, so the two observation copies of
        `add_transitions` (rollout_storage.py:90-92) disappear and the policy GEMMs read the slot in place.  Pass
        None to detach.  Nothing else changes for the caller: step() still returns the tensors it wrote."""
        if env is not None and not hasattr(env, "set_next_observation_buffers"):
            raise TypeError("attach_env needs an env with set_next_observation_buffers()")
        self._env = env
        s = self.storage
        if env is not None and s is not None and getattr(env, "_graphs", None) is not None and env.num_envs == s.num_envs:
            # act() returns the storage's action slots: their step graphs are captured now, not inside the first rollout
            env.prepare_action_buffers(*[s.actions[k] for k in range(s.num_transitions_per_env)])

    def seed(self, seed: int) -> None:
        """Seed of the action-sample generator (the reference seeds torch globally, helpers.py:95-106).  The key is
        device-resident: act graphs captured earlier draw from it on their next replay.  Data-parallel replicas need
        distinct seeds (isaac_b200.parallel.attach_data_parallel derives one per rank)."""
        self._eps_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        signed = self._eps_seed - (1 << 64) if self._eps_seed >= (1 << 63) else self._eps_seed
        self._eps_state.copy_(torch.tensor([0, 0, signed], dtype=torch.int64))

    def attach_peer_optimizer(self, peer) -> None:
        """Data-parallel replica: the optimizer step becomes hb_dp_optimizer_step over `peer`'s symmetric buffers (the
        ActorCritic has been re-bound to them); graphs that baked the old buffer addresses are dropped."""
        self._peer = peer
        self._act_graphs.clear(), self._update_graphs.clear()

    def _set_step(self, step: int) -> None:
        """Adam's step count (host mirror + hb_optim_state.step)."""
        self._step = int(step)
        self._opt_i64[OPT_STEP] = int(step)

    @property
    def _act_stage(self):
        """The eps staging buffer of the storage's shard width (tests read the draw of the last act())."""
        return self._act_stages.get(self.storage.num_envs if self.storage is not None else None)

    def _draw_eps(self, n, st):
        """[n, num_actions] N(0,1) draws into the staging buffer of this batch size (one per size, never freed: captured
        act graphs address it) - the eps of Normal.sample(), actor_critic.py:116."""
        stage = self._eps_stage(n)
        _lib.check(self._lib.hb_ppo_draw_normal(stage.data_ptr(), stage.numel(), self._eps_state.data_ptr(), st),
                   "hb_ppo_draw_normal")
        return stage

    def _eps_stage(self, n):
        stage = self._act_stages.get(n)
        if stage is None:
            stage = self._act_stages[n] = torch.zeros(n, self.actor_critic.num_actions, device=self.device)
        return stage

    def _slot(self, k):
        """Views and addresses of rollout slot k, built once per storage (tensor indexing costs microseconds)."""
        s = self.storage
        cache = self._slots
        if cache is None or cache[0] is not s:
            cache = self._slots = (s, {})
        e = cache[1].get(k)
        if e is None:
            e = cache[1][k] = SimpleNamespace(
                xa=s._observations[k], xc=s._privileged_observations[k], obs=s.observations[k],
                priv=s.privileged_observations[k], actions=s.actions[k], values=s.values[k],
                logp=s.actions_log_prob[k].view(-1), mu=s.mu[k], sigma=s.sigma[k], next=s.observation_slot(k + 1),
                rewards_ptr=s.rewards[k].data_ptr(), dones_ptr=s.dones[k].data_ptr())
            e.xa_ptr, e.xc_ptr, e.values_ptr = e.xa.data_ptr(), e.xc.data_ptr(), e.values.data_ptr()
            e.next_ptrs = (e.next[0].data_ptr(), e.next[1].data_ptr())
        return e

    def _act_fused(self, e, n, ws, st, eps):
        """The fast path's launches for slot e, eagerly or under graph capture: the three grouped hidden-layer GEMMs reading
        the slot's observations in place, then the fused output layers / sample / log-prob / value kernel writing into the
        slot.  Callers draw eps in the argument list, so the draw is issued before the first GEMM."""
        ac = self.actor_critic
        h3a, h3c = ac.forward_both(e.xa, e.xc, ws)
        La, Lc = ac.output_layers
        _lib.check(self._lib.hb_ppo_act_fused(h3a.data_ptr(), h3a.stride(0), h3c.data_ptr(), h3c.stride(0),
                                              ac._matrix(ac.flat, La).data_ptr(), ac._matrix(ac.flat, Lc).data_ptr(), La.ld,
                                              ac.std.data_ptr(), eps.data_ptr(), n, ac.num_actions, e.actions.data_ptr(),
                                              e.logp.data_ptr(), e.mu.data_ptr(), e.sigma.data_ptr(), e.values_ptr, st),
                   "hb_ppo_act_fused")

    def act(self, obs, critic_obs):
        """ppo.py:91-101.  Fast path (both last hidden layers 128 wide, rollout slot available): the observations
        are recorded in the slot first (16-byte row pitch: TMA cannot address 615- / 1050-float rows; no copy at all
        when the env wrote them there, see attach_env) and feed the GEMMs from the slot, three hidden-layer GEMMs per
        network, then ONE kernel for the two output layers, the sample, its log-prob, mu, sigma and the value, written
        straight into the storage slot (rollout_storage.py:87-100's copies of these tensors disappear).  Small shards
        replay all of it from one CUDA graph per slot."""
        ac, s = self.actor_critic, self.storage
        n = obs.shape[0]
        t = self.transition
        fast = (ac.fused_head and s is not None and s.step < s.num_transitions_per_env and n == s.num_envs
                and s.privileged_observations is not None and obs.is_cuda and critic_obs.is_cuda)
        if fast:
            k = s.step
            e = self._slot(k)
            if obs.data_ptr() != e.xa_ptr or obs.stride(0) != s.obs_ld:
                e.obs.copy_(obs)
            if critic_obs.data_ptr() != e.xc_ptr or critic_obs.stride(0) != s.priv_ld:
                e.priv.copy_(critic_obs)
            if self.graph_rollout and self.injected_eps is None and n <= self.graph_rollout_max_envs and ac.precision == "tf32":
                self._replay_act_graph(k, e, n)
            else:
                ws = ac.workspace(n)
                st = torch.cuda.current_stream(self.device).cuda_stream
                eps = self.injected_eps.contiguous() if self.injected_eps is not None else self._draw_eps(n, st)
                self._act_fused(e, n, ws, st, eps)
                self.injected_eps = None
            t.actions, t.values, t.actions_log_prob = e.actions, e.values, e.logp
            t.action_mean, t.action_sigma = e.mu, e.sigma
            t.observations, t.critic_observations = obs, critic_obs
            self._recorded_slot = k
            env = self._env
            if env is not None and env.num_envs == n:
                # slot T exists: it takes the observations after the last transition
                if e.next_ptrs[0] != obs.data_ptr() and e.next_ptrs[1] != critic_obs.data_ptr():
                    env.set_next_observation_buffers(*e.next)
            return t.actions
        st = torch.cuda.current_stream(self.device).cuda_stream
        ws = ac.workspace(n)
        eps = self.injected_eps if self.injected_eps is not None else self._draw_eps(n, st)
        self.injected_eps = None
        self._recorded_slot = None
        mu16 = ac._mlp_forward("actor", ac._as_operand(obs, ac.num_actor_obs), ws)
        v16 = ac._mlp_forward("critic", ac._as_operand(critic_obs, ac.num_critic_obs), ws)
        actions = torch.empty(n, ac.num_actions, device=self.device)
        logp = torch.empty(n, device=self.device)
        mu, sigma = torch.empty_like(actions), torch.empty_like(actions)
        _lib.check(self._lib.hb_ppo_act_head(mu16.data_ptr(), mu16.stride(0), ac.std.data_ptr(), eps.contiguous().data_ptr(), n,
                                             ac.num_actions, actions.data_ptr(), logp.data_ptr(), mu.data_ptr(), sigma.data_ptr(), st),
                   "hb_ppo_act_head")
        t.actions, t.values, t.actions_log_prob = actions, v16[:, :1].clone(), logp
        t.action_mean, t.action_sigma = mu, sigma
        t.observations, t.critic_observations = obs, critic_obs          # recorded before env.step() (ppo.py:98-100)
        return t.actions

    def _replay_act_graph(self, k, e, n):
        """Capture (once per rollout slot, hb_graph_*) and replay: the N(0,1) draw of the sample, the three grouped
        hidden-layer GEMMs reading the slot's observations in place, and the fused output layers / sample / log-prob /
        value kernel writing into the slot - library launches only."""
        entry = self._act_graphs.get(e.xa_ptr)
        if entry is None:
            ac, s, dev = self.actor_critic, self.storage, self.device
            ws = ac.workspace(n)
            if len(self._act_graphs) >= 4 * (s.num_transitions_per_env + 1):     # new storage: drop the stale graphs
                self._act_graphs.clear()
            self._eps_stage(n)          # allocated before capture (and without consuming a draw)
            g = _lib.LaunchGraph(dev).record(lambda st: self._act_fused(e, n, ws, st, self._draw_eps(n, st)))
            entry = self._act_graphs[e.xa_ptr] = (g, e, ws)       # keeps the slot views and the workspace alive
        entry[0].replay(torch.cuda.current_stream(self.device).cuda_stream)

    def process_env_step(self, rewards, dones, infos):
        """ppo.py:103-113.  After the fast path of act() only rewards (with the time-out bootstrap) and dones are
        left to record: one kernel."""
        t, s = self.transition, self.storage
        k = self._recorded_slot
        if k is not None and k == s.step and rewards.is_cuda and rewards.dtype == torch.float32:
            rewards, dones = rewards.contiguous(), dones.contiguous()
            if dones.dtype not in (torch.bool, torch.uint8):
                dones = dones != 0
            tos = infos.get("time_outs") if isinstance(infos, dict) else None
            if tos is not None:
                tos = tos.to(self.device).contiguous()
                if tos.dtype not in (torch.bool, torch.uint8):
                    tos = tos != 0
            st = torch.cuda.current_stream(self.device).cuda_stream
            e = self._slot(k)
            _lib.check(self._lib.hb_ppo_record_step(rewards.data_ptr(), dones.data_ptr(), e.values_ptr,
                                                    tos.data_ptr() if tos is not None else None, float(self.gamma),
                                                    rewards.numel(), e.rewards_ptr, e.dones_ptr, st),
                       "hb_ppo_record_step")
            s.step += 1
            self._recorded_slot = None
            t.clear()
            self.actor_critic.reset(dones)
            return
        t.rewards = rewards.clone()
        t.dones = dones
        if "time_outs" in infos:          # bootstrapping on time outs (ppo.py:106-108)
            t.rewards += self.gamma * torch.squeeze(t.values * infos["time_outs"].unsqueeze(1).to(self.device), 1)
        self.storage.add_transitions(t)
        t.clear()
        self.actor_critic.reset(dones)

    def compute_returns(self, last_critic_obs):
        last_values = self.actor_critic.evaluate(last_critic_obs)
        self.storage.compute_returns(last_values, self.gamma, self.lam)

    # ------------------------------------------------------------------ update (ppo.py:119-184)
    def minibatch_gradients(self, i: int):
        """Forward, loss head and backward of minibatch i of the gathered buffers (ppo.py:128-172): leaves the
        global-batch gradient in actor_critic.grad (all-reduced over ranks) and the loss sums in self._stats."""
        ac, lib, mb = self.actor_critic, self._lib, self._mb
        st = torch.cuda.current_stream(self.device).cuda_stream
        ws = ac.workspace(mb)
        xa, xc, rec = self._xa[i * mb:(i + 1) * mb], self._xc[i * mb:(i + 1) * mb], self._rec[i * mb:(i + 1) * mb]
        # self._stats is zero here: update() zeroes it once, the optimizer step's epilogue kernel re-arms it
        if ac.fused_head:
            h3a, h3c = ac.forward_both(xa, xc, ws)
            La, Lc = ac.output_layers
            dza, dzc = ws["actor"]["dz"][-1], ws["critic"]["dz"][-1]
            _lib.check(lib.hb_ppo_head_fused(
                h3a.data_ptr(), h3a.stride(0), h3c.data_ptr(), h3c.stride(0),
                ac._matrix(ac.flat, La).data_ptr(), ac._matrix(ac.flat, Lc).data_ptr(), La.ld, ac.std.data_ptr(),
                rec.data_ptr(), mb, mb * self.world_size, C.byref(self._lp), dza.data_ptr(), dzc.data_ptr(), dza.stride(0),
                ac._matrix(ac.grad, La).data_ptr(), ac._matrix(ac.grad, Lc).data_ptr(),
                ac.grad[ac._std_offset:].data_ptr(), self._stats.data_ptr(), st), "hb_ppo_head_fused")
            ac.backward_both(xa, xc, ws)
        else:
            mu16 = ac._mlp_forward("actor", xa, ws)
            v16 = ac._mlp_forward("critic", xc, ws)
            _lib.check(lib.hb_ppo_loss_head(mu16.data_ptr(), mu16.stride(0), v16.data_ptr(), v16.stride(0), ac.std.data_ptr(), rec.data_ptr(), mb,
                                            mb * self.world_size, C.byref(self._lp), ws["actor"]["d_out"].data_ptr(),
                                            ws["critic"]["d_out"].data_ptr(), ac.grad[ac._std_offset:].data_ptr(),
                                            self._stats.data_ptr(), st), "hb_ppo_loss_head")
            ac._mlp_backward("actor", xa, ws)
            ac._mlp_backward("critic", xc, ws)
        if self.grad_allreduce is not None:
            self.grad_allreduce(ac.grad, self._stats, ac._grad_wire)     # sums over ranks (grads already carry 1/global_mb)

    def optimizer_step(self, adaptive: int):
        """clip_grad_norm_ + Adam.step + zero_grad (ppo.py:171-174) with the adaptive-KL rule of :136-148 in one
        cooperative launch; learning rate, Adam's step count, the minibatch's loss sums and update()'s running sums
        all stay in hb_optim_state on the device, so nothing in the call changes from step to step."""
        ac, lib = self.actor_critic, self._lib
        st = torch.cuda.current_stream(self.device).cuda_stream
        ap = AdamParams(0.9, 0.999, 1e-8, float(self.max_grad_norm or 0.0), adaptive, float(self.desired_kl or 0.0),
                        self._mb * self.world_size)
        if self._peer is not None:          # all ranks: reduce + clip + Adam + broadcast over peer memory, one kernel
            _lib.check(lib.hb_dp_optimizer_step(self._peer.comm_ref, self._exp_avg.data_ptr(), self._exp_avg_sq.data_ptr(),
                                                ac.flat.numel(), C.byref(ap), self._opt.data_ptr(), st), "hb_dp_optimizer_step")
        else:
            _lib.check(lib.hb_optimizer_step(ac.flat.data_ptr(), ac.grad.data_ptr(), self._exp_avg.data_ptr(),
                                             self._exp_avg_sq.data_ptr(), ac.flat.numel(), C.byref(ap), self._opt.data_ptr(), st),
                       "hb_optimizer_step")
        self._step += 1

    def _update_graph(self, i: int, adaptive: int):
        """The launches of minibatch i's step as one CUDA graph (hb_graph_*): 3 grouped forward launches, the fused head,
        5 grouped backward launches, the optimizer step.  Every buffer address and every by-value argument is the same for
        all epochs and updates (the step's scalars live in hb_optim_state), so it is captured once."""
        key = (i, self._mb, self._xa.data_ptr(), self._xc.data_ptr(), self._rec.data_ptr(), adaptive, self.clip_param,
               self.value_loss_coef, self.entropy_coef, self.use_clipped_value_loss, self.max_grad_norm, self.desired_kl,
               self.actor_critic.precision)
        g = self._update_graphs.get(key)
        if g is None:
            if len(self._update_graphs) >= 4 * self.num_mini_batches:
                self._update_graphs.clear()
            self.actor_critic.workspace(self._mb)                   # allocated before capture
            step0 = self._step

            def launches(st):
                self.minibatch_gradients(i)
                self.optimizer_step(adaptive)

            g = self._update_graphs[key] = _lib.LaunchGraph(self.device).record(launches)
            self._step = step0                                       # capture executed nothing
        return g

    def prepare_minibatches(self, perm=None):
        """mini_batch_generator's gathers (rollout_storage.py:146-182), once per update (the permutation is
        reused by every epoch, :149)."""
        ac, lib, s = self.actor_critic, self._lib, self.storage
        dev = self.device
        st = torch.cuda.current_stream(dev).cuda_stream
        B = s.num_envs * s.num_transitions_per_env
        mb = B // self.num_mini_batches
        used = mb * self.num_mini_batches
        if perm is None:
            perm = torch.randperm(used, device=dev)
        perm = perm.to(dev, dtype=torch.int64).contiguous()
        ld_a, ld_c = pitch(ac.num_actor_obs + 1), pitch(ac.num_critic_obs + 1)      # 128-byte rows for the layer-1 GEMMs
        if self._xa is None or self._xa.shape[0] != used:
            self._xa = torch.zeros(used, ld_a, device=dev)
            self._xc = torch.zeros(used, ld_c, device=dev)
            self._rec = torch.zeros(used, ppo_rec(ac.num_actions), device=dev)
        _lib.check(lib.hb_ppo_gather_rows(s._observations.data_ptr(), s.obs_ld, self._xa.data_ptr(), ld_a,
                                          perm.data_ptr(), used, ac.num_actor_obs, ac.num_actor_obs, st), "gather obs")
        _lib.check(lib.hb_ppo_gather_rows(s._privileged_observations.data_ptr(), s.priv_ld, self._xc.data_ptr(), ld_c,
                                          perm.data_ptr(), used, ac.num_critic_obs, ac.num_critic_obs, st), "gather priv")
        _lib.check(lib.hb_ppo_pack_samples(perm.data_ptr(), used, s.actions.data_ptr(), s.mu.data_ptr(),
                                           s.sigma.data_ptr(), s.values.data_ptr(), s.advantages.data_ptr(),
                                           s.returns.data_ptr(), s.actions_log_prob.data_ptr(), ac.num_actions, self._rec.data_ptr(), st),
                   "hb_ppo_pack_samples")
        self._mb = mb
        self._lp = PpoLossParams(self.clip_param, self.value_loss_coef, self.entropy_coef, int(self.use_clipped_value_loss), ac.num_actions,
                                 ac.hb_activation)
        return mb

    def update(self):
        perm, self.injected_perm = self.injected_perm, None
        mb = self.prepare_minibatches(perm)
        adaptive = int(self.desired_kl is not None and self.schedule == "adaptive")
        self._per_update.zero_()                 # gradient norm scratch, minibatch loss sums, running sums
        self._opt_i64[OPT_STEPS_IN_UPDATE:OPT_STEPS_IN_UPDATE + 2].zero_()     # trace cursor, barrier ticket
        # the first update launches eagerly (lazy module load, cudaFuncSetAttribute); later ones replay graphs
        graphs = (self.graph_update and self.grad_allreduce is None and self._updates_done > 0
                  and self.actor_critic.fused_head and self.actor_critic.precision == "tf32")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        for _ in range(self.num_learning_epochs):
            for i in range(self.num_mini_batches):
                if graphs:
                    self._update_graph(i, adaptive).replay(stream)
                    self._step += 1
                else:
                    self.minibatch_gradients(i)
                    self.optimizer_step(adaptive)
        self._updates_done += 1
        self._lr_dirty = bool(adaptive)
        num_updates = self.num_learning_epochs * self.num_mini_batches
        host = self._opt.cpu()                   # the single host sync of the update (the reference's .item() calls)
        acc = host[OPT_LOSS_ACC:OPT_LOSS_ACC + 4]
        denom = num_updates * mb * self.world_size
        mean_surrogate_loss, mean_value_loss = float(acc[0]) / denom, float(acc[1]) / denom
        self.last_mean_kl = float(acc[2]) / denom
        err = int(host.view(torch.int64)[OPT_ERROR])
        if self._peer is not None and err != 0:
            raise _lib.HectorB200Error(f"hb_dp_optimizer_step: a peer rank did not arrive (phase {err})")
        k = min(num_updates, HB_OPT_TRACE_MAX)
        trace = host[OPT_TRACE:OPT_TRACE + 2 * k].view(k, 2)
        self.kl_trace, self.lr_trace = trace[:, 0].tolist(), trace[:, 1].tolist()     # per optimizer step of this update
        if adaptive:
            self._lr_host, self._lr_dirty = float(host[OPT_LR]), False
        self.storage.clear()
        return mean_value_loss, mean_surrogate_loss
