"""The runner level (algo/ppo/on_policy_runner.py): (1) the UNMODIFIED reference `OnPolicyRunner.learn` runs over the
drop-in classes - `isaac_b200.algo.PPO` / `ActorCritic` bound under the names its module resolves with `eval`, and
`HectorFreeEnvB200` as the VecEnv - as INTEGRATION.md claims; (2) this repo's runner, which keeps the per-step bookkeeping
on the device; (3) that bookkeeping against the reference's deque logic."""
import os
from collections import deque

import numpy as np
import pytest
import torch

from isaac_b200.envs.hector_config import HectorCfg
from isaac_b200.synthetic import make_tape
from oracle import ref_harness

pytestmark = pytest.mark.gpu

TRAIN_CFG = {
    "runner": dict(policy_class_name="ActorCritic", algorithm_class_name="PPO", num_steps_per_env=8, max_iterations=3,
                   save_interval=2, experiment_name="hector", run_name="", resume=False, load_run=-1, checkpoint=-1,
                   resume_path=None),
    "algorithm": dict(value_loss_coef=1.0, use_clipped_value_loss=True, clip_param=0.2, entropy_coef=0.001, num_learning_epochs=2,
                      num_mini_batches=4, learning_rate=1e-5, schedule="adaptive", gamma=0.994, lam=0.9, desired_kl=0.01,
                      max_grad_norm=1.0),
    "policy": dict(init_noise_std=1.0, actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128]),
}


def make_env(dev, n=256, graphs=False):
    from test_env_parity import make_cuda_env
    tape = make_tape(n, 2, seed=31, fall_prob=0.02)
    env, phys = make_cuda_env(tape, dev)
    env.seed(3)
    if graphs:
        env.enable_cuda_graph()
    return env


def test_reference_runner_learn_runs_over_dropin_classes(lib, cuda_device, tmp_path, monkeypatch):
    if ref_harness.reference_root() is None:
        pytest.skip("needs the upstream reference: set ISAAC_REFERENCE to a checkout of DRCL-USC/isaac")
    monkeypatch.setenv("WANDB_MODE", "disabled")
    ref_harness.install_isaacgym_stub()
    import importlib
    # (humanoid/algo/__init__.py rebinds `humanoid.algo.ppo` to the module ppo.py: attribute-style import would miss the file)
    ref_runner = importlib.import_module("humanoid.algo.ppo.on_policy_runner")          # the reference's file, unmodified
    from isaac_b200.algo import ActorCritic, PPO
    # the binding a maintainer adds: the two names the runner resolves with eval() (on_policy_runner.py:68,72)
    monkeypatch.setattr(ref_runner, "ActorCritic", ActorCritic)
    monkeypatch.setattr(ref_runner, "PPO", PPO)
    env = make_env(cuda_device)
    runner = ref_runner.OnPolicyRunner(env, TRAIN_CFG, log_dir=str(tmp_path), device=str(cuda_device))
    assert isinstance(runner.alg, PPO) and isinstance(runner.alg.actor_critic, ActorCritic)
    w0 = runner.alg.actor_critic.flat.clone()
    runner.learn(num_learning_iterations=3, init_at_random_ep_len=True)
    torch.cuda.synchronize()
    assert runner.current_learning_iteration == 3 and runner.tot_timesteps == 3 * 8 * env.num_envs
    assert not torch.equal(w0, runner.alg.actor_critic.flat) and torch.isfinite(runner.alg.actor_critic.flat).all()
    assert int(env.episode_length_buf.max()) > 8, "init_at_random_ep_len reached the kernels' buffer"
    saved = sorted(p for p in os.listdir(tmp_path) if p.endswith(".pt"))
    assert saved == ["model_0.pt", "model_2.pt", "model_3.pt"]
    # checkpoint round trip through the reference's own save / load
    ck = torch.load(tmp_path / "model_3.pt", map_location="cpu")
    assert set(ck) == {"model_state_dict", "optimizer_state_dict", "iter", "infos"} and ck["iter"] == 3
    assert list(ck["model_state_dict"])[0] == "std" and len(ck["optimizer_state_dict"]["state"]) == 17
    runner2 = ref_runner.OnPolicyRunner(make_env(cuda_device), TRAIN_CFG, log_dir=str(tmp_path / "b"), device=str(cuda_device))
    runner2.load(str(tmp_path / "model_3.pt"))
    assert torch.equal(runner2.alg.actor_critic.flat, runner.alg.actor_critic.flat) and runner2.alg._step == runner.alg._step
    policy = runner2.get_inference_policy(device=str(cuda_device))
    assert policy(env.get_observations()).shape == (env.num_envs, 10)


@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
def test_own_runner_learns_logs_and_checkpoints(lib, cuda_device, tmp_path, graphs):
    from isaac_b200.algo import OnPolicyRunner
    env = make_env(cuda_device, graphs=graphs)
    runner = OnPolicyRunner(env, TRAIN_CFG, log_dir=str(tmp_path), device=str(cuda_device))
    w0 = runner.alg.actor_critic.flat.clone()
    runner.learn(num_learning_iterations=3, init_at_random_ep_len=True)
    assert not torch.equal(w0, runner.alg.actor_critic.flat) and torch.isfinite(runner.alg.actor_critic.flat).all()
    keys = set(runner.last_log)
    assert {"Loss/value_function", "Loss/surrogate", "Loss/learning_rate", "Policy/mean_noise_std", "Perf/total_fps",
            "Perf/collection time", "Perf/learning_time", "Episode/rew_tracking_lin_vel"} <= keys
    assert sorted(p for p in os.listdir(tmp_path) if p.endswith(".pt")) == ["model_0.pt", "model_2.pt", "model_3.pt"]
    runner2 = OnPolicyRunner(make_env(cuda_device), TRAIN_CFG, log_dir=None, device=str(cuda_device))
    runner2.load(str(tmp_path / "model_3.pt"))
    assert torch.equal(runner2.alg.actor_critic.flat, runner.alg.actor_critic.flat)
    # the observations went straight into the rollout slots
    assert runner.alg.__dict__.get("_env") is env


def test_device_bookkeeping_matches_the_reference_deques(lib, cuda_device):
    """hb_runner_bookkeeping against on_policy_runner.py:140-154 executed literally (deque(maxlen=100), ascending env order)."""
    from isaac_b200.algo.on_policy_runner import EpisodeBuffers
    dev = cuda_device
    for n, p_done in ((37, 0.2), (4096, 0.01), (3000, 0.3)):
        g = torch.Generator().manual_seed(n)
        book = EpisodeBuffers(n, dev)
        rewbuffer, lenbuffer = deque(maxlen=100), deque(maxlen=100)
        cur_sum, cur_len = torch.zeros(n), torch.zeros(n)
        for step in range(12):
            rewards = torch.rand(n, generator=g)
            dones = torch.rand(n, generator=g) < p_done
            book.step(rewards.to(dev), dones.to(dev))
            cur_sum += rewards
            cur_len += 1
            new_ids = (dones > 0).nonzero(as_tuple=False)
            rewbuffer.extend(cur_sum[new_ids][:, 0].numpy().tolist())
            lenbuffer.extend(cur_len[new_ids][:, 0].numpy().tolist())
            cur_sum[new_ids] = 0
            cur_len[new_ids] = 0
        got_rew, got_len = book.deques()
        np.testing.assert_array_equal(np.float32(got_rew), np.float32(list(rewbuffer)))
        np.testing.assert_array_equal(np.float32(got_len), np.float32(list(lenbuffer)))
        assert torch.equal(book.cur_reward_sum.cpu(), cur_sum) and torch.equal(book.cur_episode_length.cpu(), cur_len)
        assert len(got_rew) == min(100, int(book.ring_state.item())) and len(got_rew) > 0
