"""The library's device generator against its CPU reference (oracle/device_rng.py).

Every run without an injected tape (bench.py, OnPolicyRunner, anything that calls env.seed() / alg.seed()) takes its
randomness from Philox4x32-10 inside the kernels: the env step's reset, command, push, delay and noise draws and PPO.act's
action sample.  These tests compare those draws with the reference, directly and through the oracle.

Tolerances.  Uniform draws are exact (the top 24 bits of a word), so they enter the env exactly as a tape does and the
suite's env tolerances apply unchanged.  The normals use __logf / __sincosf in the kernels and float64 in the reference:
they agree to |dz| <= DZ_MAX (median <= DZ_MEDIAN).  A wrong word, slot, key or counter gives O(1) differences.
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from _util import ENV_ATOL, assert_close, assert_equal, to_np
from isaac_b200.synthetic import make_tape
from oracle import device_rng as R
from oracle import make_golden as mg
from test_env_parity import _View, compare_records, make_cuda_env

pytestmark = pytest.mark.gpu

DZ_MAX, DZ_MEDIAN = 1e-4, 1e-6
PPO_DEFAULT_KEY = 0x9E3779B97F4A7C15             # PPO's default seed: bit 63 set
KEYS = {"default": PPO_DEFAULT_KEY, "small": 7, "upper": 0x0001234500000005}
ENV_KEY = 0xF00DFACE0BADC0DE                      # bit 63 and upper bits set
SPECIAL_EP0 = [2399, 2400, 798, 799, 1599]        # time-outs at steps 1 / 2, command resampling at steps 1 / 2
STEP_COUNTER0 = 396                               # common_step_counter: step 4 of the window is a push step


def _signed(v):
    v &= 0xFFFFFFFFFFFFFFFF
    return v - (1 << 64) if v >= (1 << 63) else v


def _dz_stats(got, want):
    d = np.abs(np.asarray(got, np.float64) - np.asarray(want, np.float64))
    return float(d.max()), float(np.median(d))


# --------------------------------------------------------------------------- (a) hb_ppo_draw_normal
@pytest.mark.parametrize("call0", [0, 2 ** 32 - 1], ids=["call0", "call2^32-1"])
@pytest.mark.parametrize("key", list(KEYS.values()), ids=list(KEYS))
def test_ppo_draw_normal_matches_reference(lib, cuda_device, key, call0):
    """hb_ppo_draw_normal against ppo_normals: partial quads, one and several blocks, a hector_full shard (4096 x 18);
    the call counter advances by exactly one per launch, from 2^32 - 1 across the carry into its upper word.
    Measured on a B200 (1000 W power limit): max |dz| between 3.4e-6 and 7.5e-6 over these six cases."""
    dev = cuda_device
    state = torch.tensor([_signed(call0), 0, _signed(key)], dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    call, worst = call0, 0.0
    for count in (1, 3, 4, 40963, 4096 * 18):
        out = torch.full((count + 4,), 123.0, device=dev)
        assert lib.hb_ppo_draw_normal(out.data_ptr(), count, state.data_ptr(), st) == 0
        got = out.cpu().numpy()
        assert (got[count:] == 123.0).all(), "store past count"
        assert state.tolist() == [call + 1, 0, _signed(key)], f"count {count}: counter / ticket after the launch"
        dz_max, dz_med = _dz_stats(got[:count], R.ppo_normals(key, call, count))
        assert dz_max <= DZ_MAX, f"count {count}, call {call:#x}: max |dz| = {dz_max:.3e}"
        if count > 1000:
            assert dz_med <= DZ_MEDIAN, f"count {count}, call {call:#x}: median |dz| = {dz_med:.3e}"
        worst = max(worst, dz_max)
        call += 1
    print(f"hb_ppo_draw_normal key={key:#x} call0={call0:#x}: max |dz| = {worst:.3e}")


# --------------------------------------------------------------------------- (b) env step on the device generator
def _prologue_on_device(env, actions_in, dev):
    """What the step's action prologue (clip, delay, action noise) makes of `actions_in` at the env's current counter,
    computed by the library's own hb_env_action_prologue into a scratch copy of env.actions (the env is untouched)."""
    from isaac_b200 import _lib
    out = env.actions.clone()
    b = _lib.EnvBuffers.from_buffer_copy(env._b)
    b.actions = out.data_ptr()
    nz = _lib.EnvNoise()
    nz.rng_counter = env._rng_state.data_ptr()
    _lib.check(env._lib.hb_env_action_prologue(env._pp, C.byref(b), actions_in.data_ptr(), C.byref(nz),
                                               torch.cuda.current_stream(dev).cuda_stream), "hb_env_action_prologue")
    return out.cpu()


def _prologue_reference(cfg, a_in, prev, draws):
    """HectorFreeEnv.step's prologue (hector_env.py:158-169) on the reference draws, as the oracle spells it, and the
    extra absolute tolerance the Box-Muller deviation allows: |d(action_noise * z * a)| <= |action_noise| * DZ_MAX * |a|."""
    dr, clip = cfg.domain_rand, cfg.normalization.clip_actions
    a = torch.clip(a_in, -clip, clip)
    delay = draws.u_delay * dr.action_delay
    a = (1 - delay) * a + delay * prev
    margin = abs(dr.action_noise) * DZ_MAX * a.abs()
    return torch.clip(a + dr.action_noise * draws.z_action * a, -clip, clip), margin


def _run_env_case(dev, task, n, graph, counter0=None, steps=8):
    """The CUDA env on the device generator (cfg.seed = ENV_KEY, no tape at all, the constructor's reset included) against
    the oracle fed with env_draws at the counter the env reports.  The action prologue is checked on its own (it is the
    one place the env step multiplies by a normal draw); the oracle then steps from the prologue's output, so every
    other quantity is held to the suite's tolerances, the observation columns with noise excepted."""
    from oracle.hector_oracle import OracleHectorEnv
    from isaac_b200.envs import TASKS
    import isaac_b200.envs as envs
    cls_name, cfg_cls, _ = TASKS[task]
    cfg = cfg_cls()
    cfg.seed = ENV_KEY
    nd, nobs, npriv = cfg.env.num_actions, cfg.env.num_single_obs, cfg.env.single_num_privileged_obs
    tape = make_tape(n, steps, seed=3000 + n, fall_prob=0.03, randomize_gains=True, cfg=cfg_cls())
    tape.statics.episode_length0[:len(SPECIAL_EP0)] = torch.tensor(SPECIAL_EP0)
    env, phys = make_cuda_env(tape, dev, cfg=cfg, cls=getattr(envs, cls_name), device_rng=True)
    assert env._rng_state.tolist() == [1, _signed(ENV_KEY)], "the constructor's reset draws at counter 0 and advances it"
    ora = OracleHectorEnv(cfg_cls(), tape.statics, tape.physics[0], R.env_draws(ENV_KEY, 0, n, nd, nobs))
    counter = 1
    if counter0 is not None:
        env._rng_state[0] = counter0
        counter = counter0
    env.common_step_counter = ora.common_step_counter = STEP_COUNTER0
    if graph:
        env.enable_cuda_graph()
    got = {"obs_init": to_np(env.obs_buf), "priv_init": to_np(env.privileged_obs_buf)}
    want = {"obs_init": ora.obs_buf.numpy().copy(), "priv_init": ora.privileged_obs_buf.numpy().copy()}
    got_ids, want_ids, out = [], [], None
    actions = torch.zeros(n, nd, device=dev)         # one address: the graph path replays one captured prologue
    for t in range(1, steps):
        a_in = tape.noise[t].actions
        actions.copy_(a_in)
        draws = R.env_draws(ENV_KEY, counter, n, nd, nobs, actions=a_in)
        pro = _prologue_on_device(env, actions, dev)
        want_pro, margin = _prologue_reference(cfg, a_in, ora.actions, draws)
        assert_close(f"action prologue @{t}", pro.numpy(), want_pro.numpy(), atol=ENV_ATOL + margin.numpy())
        phys.load_frame(tape.physics[t].to(dev))
        out = env.step(actions)
        counter += 1
        assert int(env._rng_state[0].item()) == _signed(counter), f"step {t}: the step advances the counter by one"
        cpu_out = tuple(o.cpu() for o in out[:4]) + ({"time_outs": out[4]["time_outs"].cpu(),
                                                     "episode": {k: v.cpu() for k, v in out[4]["episode"].items()}},)
        mg.record_env_step(got, _View(env), cpu_out, env.root_states.cpu(), env.dof_state.cpu(), (nobs, npriv))
        got_ids.append(env.reset_env_ids[:int(env._reset_count.item())].cpu().numpy().copy())
        # the oracle steps from the kernel's prologue output (no delay, no action noise on top)
        zeros = lambda x: torch.zeros_like(x)
        o = ora.step(tape.physics[t], dataclasses.replace(draws, actions=pro, u_delay=zeros(draws.u_delay),
                                                          z_action=zeros(draws.z_action)))
        mg.record_env_step(want, ora, o, ora.root_states, ora.dof_state, (nobs, npriv))
        want_ids.append(ora.last_reset_ids.numpy().astype(np.int32))
    got = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in got.items()}
    want = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in want.items()}
    got["obs_final"], got["priv_final"] = to_np(out[0]), to_np(out[1])
    want["obs_final"], want["priv_final"] = to_np(o[0]), to_np(o[1])
    # observation noise: |d(z * noise_scale_vec * noise_level)| <= DZ_MAX * noise_scale_vec * noise_level, every frame
    col = ora.noise_scale_vec.numpy().astype(np.float64) * cfg.noise.noise_level * DZ_MAX
    stack = np.tile(col, cfg.env.frame_stack)
    compare_records(got, want, extra_atol={"obs_frame": col, "obs_init": stack, "obs_final": stack})
    for t, (a, b) in enumerate(zip(got_ids, want_ids)):
        assert_equal(f"reset_env_ids@{t}", a, b)
    # every kind of draw was taken: falls and time-outs (dof / root / command reset draws), resampling, a push step
    assert sum(len(i) for i in want_ids) > len(want_ids) and want["time_outs"].sum() >= 1
    assert phys.calls["set_root_state"] == 1
    return env


ENV_CASES = [("hector", 257), ("hector", 4096), ("hector_full", 1003), ("humanoid_ppo", 257)]


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
@pytest.mark.parametrize("task,n", ENV_CASES, ids=[f"{t}-{n}" for t, n in ENV_CASES])
def test_env_step_device_draws_match_oracle(lib, cuda_device, task, n, graph):
    """Reset (dof jitter, root xy, command), command resampling, push, action delay (humanoid_ppo: 0.5), action noise
    and observation noise of the device generator against the oracle on env_draws: a partial last 32-env tile
    (n = 257, 1003), 18 DOF (5 action-noise calls, 23 reset uniforms), eager launches and graph replay."""
    _run_env_case(cuda_device, task, n, graph)


def test_env_step_device_draws_cross_the_counter_carry(lib, cuda_device):
    """The step counter from 2^32 - 2: the third step draws with the upper counter word at 1."""
    env = _run_env_case(cuda_device, "hector", 257, False, counter0=2 ** 32 - 2, steps=5)
    assert int(env._rng_state[0].item()) == 2 ** 32 + 2


# --------------------------------------------------------------------------- (c) staged hooks vs the fused step
def test_staged_hooks_draw_like_the_fused_step(lib, cuda_device):
    """A subclass that overrides the four hooks (pass-through) runs the staged step; on the device generator it must take
    the same draws as the fused step - same results, same counter after every step, resets included - and a reset_idx()
    outside step() still advances the counter by one.  Of the other hooks called on their own, only compute_observations()
    advances it, and the next step() still advances it by exactly one."""
    from isaac_b200.envs.hector_config import HectorCfg
    from isaac_b200.envs.hector_env import HectorFreeEnvB200

    class Staged(HectorFreeEnvB200):
        def check_termination(self):
            super().check_termination()

        def compute_reward(self):
            super().compute_reward()

        def reset_idx(self, env_ids):
            super().reset_idx(env_ids)

        def compute_observations(self):
            super().compute_observations()

    dev, n, steps = cuda_device, 257, 7
    tape = make_tape(n, steps, seed=31, fall_prob=0.03, randomize_gains=True)
    tape.statics.episode_length0[:len(SPECIAL_EP0)] = torch.tensor(SPECIAL_EP0)
    runs = []
    for cls in (HectorFreeEnvB200, Staged):
        cfg = HectorCfg()
        cfg.seed = ENV_KEY
        env, phys = make_cuda_env(tape, dev, cfg=cfg, cls=cls, device_rng=True)
        env.common_step_counter = STEP_COUNTER0
        runs.append((env, phys, {}))
    assert runs[1][0]._hooks_overridden() and not runs[0][0]._hooks_overridden()
    for t in range(1, steps):
        for env, phys, rec in runs:
            phys.load_frame(tape.physics[t].to(dev))
            out = env.step(tape.noise[t].actions.to(dev))
            cpu_out = tuple(o.cpu() for o in out[:4]) + ({"time_outs": out[4]["time_outs"].cpu(),
                                                         "episode": {k: v.cpu() for k, v in out[4]["episode"].items()}},)
            mg.record_env_step(rec, _View(env), cpu_out, env.root_states.cpu(), env.dof_state.cpu())
        (fused, _, want), (staged, _, got) = runs
        assert int(fused._rng_state[0].item()) == t + 1
        assert int(staged._rng_state[0].item()) == t + 1, (f"step {t} ({int(want['reset'][-1].sum())} resets): staged counter "
                                                         f"{int(staged._rng_state[0].item())}, fused {t + 1}")
        compare_records({k: np.stack(v) for k, v in got.items()}, {k: np.stack(v) for k, v in want.items()})
    assert np.stack(want["reset"]).sum() > steps
    counter = lambda env: int(env._rng_state[0].item())
    for env, *_ in runs:
        before = int(env._rng_state[0].item())
        env.reset_idx(torch.tensor([0, 5, n - 1]))
        assert int(env._rng_state[0].item()) == before + 1, "reset_idx() outside step() advances the counter"
        before = counter(env)
        env.check_termination()
        env.compute_reward()
        assert counter(env) == before, "check_termination() / compute_reward() on their own leave the counter alone"
        env.compute_observations()
        assert counter(env) == before + 1, "compute_observations() on its own advances the counter by one"
        env.step(tape.noise[steps - 1].actions.to(dev))
        assert counter(env) == before + 2, "a step() after the hooks on their own advances the counter by one"


# --------------------------------------------------------------------------- (d) PPO.act on the library's draws
PPO_CASES = [("hector", True, 0), ("hector", False, 0), ("humanoid_ppo", True, 0), ("hector_full", True, 0),
             ("hector", True, 2 ** 32 - 1)]


@pytest.mark.parametrize("task,graph,call0", PPO_CASES,
                         ids=["hector-graph", "hector-eager", "humanoid_ppo", "hector_full-generic", "hector-call2^32-1"])
def test_ppo_act_draws_match_oracle(lib, cuda_device, task, graph, call0):
    """PPO.act with its own action sample (alg.seed, no injected_eps) against OraclePPO.act fed with ppo_normals: the
    draw of step k, recovered from the rollout slot as (actions - mu) / sigma, is call k of the stream; the rollout
    storage agrees with the oracle's at the TF32 tolerances of the other PPO parity tests.  hector and humanoid_ppo take
    the fused head (hector with and without graph replay), hector_full the generic path (output-layer GEMMs +
    hb_ppo_act_head)."""
    from isaac_b200.algo.actor_critic import ActorCritic
    from isaac_b200.algo.ppo import PPO
    from isaac_b200.envs import TASKS
    from oracle.ppo_oracle import OraclePPO, init_actor_critic_params
    dev = cuda_device
    _, cfg_cls, ppo_cls = TASKS[task]
    ec, pc = cfg_cls().env, ppo_cls().policy
    nobs, npriv, na = ec.num_observations, ec.num_privileged_obs, ec.num_actions
    n, T = 257, 5
    params = init_actor_critic_params(nobs, npriv, na, tuple(pc.actor_hidden_dims), tuple(pc.critic_hidden_dims), seed=4)
    ac = ActorCritic(nobs, npriv, na, actor_hidden_dims=pc.actor_hidden_dims, critic_hidden_dims=pc.critic_hidden_dims, device=dev)
    ac.load_state_dict(params)
    assert ac.fused_head == (task != "hector_full")
    cfg = dict(mg.PPO_ALG, schedule="fixed")
    alg = PPO(ac, device=dev, **cfg)
    alg.graph_rollout = graph
    alg.init_storage(n, T, [nobs], [npriv], [na])
    key = PPO_DEFAULT_KEY if call0 else 0x0BADF00D12345678
    alg.seed(key)
    alg._eps_state[0] = _signed(call0)
    ora = OraclePPO(params, n, T, **cfg)
    g = torch.Generator().manual_seed(8)
    eps_ref = []
    for k in range(T):
        obs, cobs = torch.randn(n, nobs, generator=g), torch.randn(n, npriv, generator=g)
        rew, dones, tos = torch.rand(n, generator=g), torch.rand(n, generator=g) < 0.1, torch.rand(n, generator=g) < 0.05
        alg.act(obs.to(dev), cobs.to(dev))
        eps = torch.from_numpy(R.ppo_normals(key, call0 + k, n * na)).view(n, na)
        ora.act(obs, cobs, eps)
        eps_ref.append(eps)
        alg.process_env_step(rew.to(dev), dones.to(dev), {"time_outs": tos.to(dev)})
        ora.process_env_step(rew, dones, {"time_outs": tos})
        assert int(alg._eps_state[0].item()) == _signed(call0 + k + 1), f"act {k}: one draw per call"
    s = alg.storage
    for k in range(T):
        a, mu, sigma = (x[k].double().cpu() for x in (s.actions, s.mu, s.sigma))
        dz = ((a - mu) / sigma - eps_ref[k].double()).abs().max().item()
        assert dz <= DZ_MAX, f"act {k}: the sample's draw differs from call {call0 + k:#x} of the stream by {dz:.3e}"
    rel = lambda x, y: float((x.double() - y.double()).norm() / y.double().norm().clamp_min(1e-30))
    for k in ("actions", "values", "mu", "actions_log_prob"):
        assert rel(getattr(s, k).cpu(), ora.st[k]) < 4e-3, (k, rel(getattr(s, k).cpu(), ora.st[k]))
    assert torch.equal(s.sigma.cpu(), ora.st["sigma"]) and torch.equal(s.dones.cpu(), ora.st["dones"])
