"""TEST INFRASTRUCTURE — needs the reference (oracle/ref_harness.py): writes tests/golden/*.npz.

Runs the UNMODIFIED reference (through `oracle/ref_harness.py`) on seeded synthetic
tapes and records what it produced.  Without the reference, the oracle and the CUDA
path are checked against these files.

    python -m oracle.make_golden            # regenerate everything

Inputs are not stored: they are regenerated from the seed by
`isaac_b200.synthetic.make_tape` / `golden_ppo_inputs` (same torch build on both
machines); each file carries float64 checksums of the inputs so that a drift in the
generator is reported as such instead of as a parity failure.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from isaac_b200.synthetic import make_tape  # noqa: E402
from oracle.ppo_oracle import PARAM_ORDER, init_actor_critic_params  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

ENV_CASE = dict(n=32, steps=40, seed=20261018, fall_prob=0.01, step_counter0=393)
ENV_EP0 = [2395, 2399, 2400, 795, 798, 799, 1599, 0]       # forces time-outs and command resampling
# the action-delay branch of HectorFreeEnv.step (hector_env.py:166-167) is dead at the shipped action_delay = 0.0: a
# second, small case runs the reference with a non-zero delay
DELAY_CASE = dict(n=24, steps=8, seed=424242, fall_prob=0.05, action_delay=0.3)
# BASELINE configs[0]: 64 envs, num_steps_per_env = 24, 5 epochs x 4 minibatches.  Seed and learning rate are chosen
# so that every mean KL of the adaptive run stays >= 4.9e-3 away from the schedule's thresholds (0.005 / 0.02): the rule
# is a discontinuous function of that scalar, and the case exercises all of it - one x1.5 step, fourteen /1.5 steps and
# the 1e-5 floor (ppo.py:136-148).
PPO_CASE = dict(n=64, t=24, seed=11, param_seed=3)
PPO_ALG = dict(value_loss_coef=1.0, use_clipped_value_loss=True, clip_param=0.2, entropy_coef=0.001,
               num_learning_epochs=5, num_mini_batches=4, learning_rate=2e-3, schedule="adaptive",
               gamma=0.994, lam=0.9, desired_kl=0.01, max_grad_norm=1.0)
PPO_POLICY = dict(init_noise_std=1.0, actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128])


def env_golden_tape():
    c = ENV_CASE
    tape = make_tape(c["n"], c["steps"], seed=c["seed"], fall_prob=c["fall_prob"], randomize_gains=True)
    tape.statics.episode_length0[:len(ENV_EP0)] = torch.tensor(ENV_EP0)
    return tape


def tape_checksum(tape) -> np.ndarray:
    acc = [float(t.double().sum()) for fr in tape.physics
           for t in (fr.root_states, fr.dof_state, fr.contact_forces, fr.rigid_state)]
    acc += [float(t.double().sum()) for nz in tape.noise
            for t in (nz.actions, nz.u_delay, nz.z_action, nz.u_cmd, nz.u_push, nz.u_reset, nz.z_obs)]
    acc += [float(t.double().sum()) for t in (tape.statics.p_gains, tape.statics.d_gains, tape.statics.env_frictions,
                                              tape.statics.body_mass, tape.statics.env_origins,
                                              tape.statics.episode_length0)]
    return np.array(acc, dtype=np.float64)


ENV_STATE_KEYS = ("torques", "commands", "feet_air_time", "feet_height", "last_contacts", "episode_length_buf",
                  "last_root_vel", "last_dof_vel", "last_actions", "last_last_actions", "base_lin_vel",
                  "base_ang_vel", "base_euler_xyz", "projected_gravity", "rand_push_force", "rand_push_torque",
                  "actions")


def record_env_step(rec, env_like, out, root_states, dof_state, frames=(41, 70)):
    """Append one step's observable results (same recorder for reference, oracle and CUDA path); `frames` = the task's
    (num_single_obs, single_num_privileged_obs)."""
    obs, priv, rew, reset, extras = out
    rec.setdefault("obs_frame", []).append(obs[:, -frames[0]:].numpy().copy())
    rec.setdefault("priv_frame", []).append(priv[:, -frames[1]:].numpy().copy())
    rec.setdefault("rew", []).append(rew.numpy().copy())
    rec.setdefault("reset", []).append(reset.numpy().astype(np.uint8))
    rec.setdefault("time_outs", []).append(extras["time_outs"].numpy().astype(np.uint8))
    rec.setdefault("episode_extras", []).append(
        np.array([float(extras["episode"]["rew_" + k]) for k in sorted(env_like.episode_sums)], dtype=np.float32))
    rec.setdefault("episode_sums", []).append(
        np.stack([env_like.episode_sums[k].numpy() for k in sorted(env_like.episode_sums)]))
    rec.setdefault("root_states", []).append(root_states.numpy().copy())
    rec.setdefault("dof_state", []).append(dof_state.numpy().copy())
    for k in ENV_STATE_KEYS:
        v = getattr(env_like, k)
        rec.setdefault(k, []).append(v.numpy().astype(np.uint8 if v.dtype == torch.bool else v.numpy().dtype).copy())


def delay_golden_tape():
    c = DELAY_CASE
    return make_tape(c["n"], c["steps"], seed=c["seed"], fall_prob=c["fall_prob"], randomize_gains=True)


def delay_cfg(cfg):
    """The config edit of the action-delay case, for the reference's and for this repo's HectorCfg alike."""
    cfg.domain_rand.action_delay = DELAY_CASE["action_delay"]
    return cfg


def _run_reference_env(tape, steps, step_counter0, configure=None, task="hector"):
    from oracle.ref_harness import ReferenceEnv
    ref = ReferenceEnv(tape.statics, tape.physics[0], tape.noise[0], configure=configure, task=task)
    ref.env.common_step_counter = step_counter0
    frames = (ref.env.cfg.env.num_single_obs, ref.env.cfg.env.single_num_privileged_obs)
    rec = {"obs_init": ref.env.obs_buf.numpy().copy(), "priv_init": ref.env.privileged_obs_buf.numpy().copy()}
    for t in range(1, steps):
        out = ref.step(tape.physics[t], tape.noise[t])
        record_env_step(rec, ref.env, out, ref.root_states, ref.dof_state, frames)
    final = {"obs_final": out[0].numpy().copy(), "priv_final": out[1].numpy().copy()}
    arrays = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in rec.items()}
    arrays.update(final)
    arrays["input_checksum"] = tape_checksum(tape)
    arrays["reward_names"] = np.array(sorted(ref.env.episode_sums))
    return arrays


# the other two registered tasks (envs/__init__.py:46-48): short rollouts of the reference's own env classes
TASK_CASE = dict(n=24, steps=14, seed=777, fall_prob=0.03, step_counter0=394)
TASK_EP0 = [2399, 2400, 798, 799, 1599, 0]


def task_golden_tape(task):
    from isaac_b200.envs.tasks import TASKS
    c = TASK_CASE
    tape = make_tape(c["n"], c["steps"], seed=c["seed"], fall_prob=c["fall_prob"], randomize_gains=True, cfg=TASKS[task][1]())
    tape.statics.episode_length0[:len(TASK_EP0)] = torch.tensor(TASK_EP0)
    return tape


def make_task_goldens():
    for task in ("hector_full", "humanoid_ppo"):
        arrays = _run_reference_env(task_golden_tape(task), TASK_CASE["steps"], TASK_CASE["step_counter0"], task=task)
        path = os.path.join(GOLDEN_DIR, f"env_rollout_{task}_ref.npz")
        np.savez_compressed(path, **arrays)
        print(f"wrote {path}: {os.path.getsize(path) / 1e6:.2f} MB, resets={int(arrays['reset'].sum())}, "
              f"time_outs={int(arrays['time_outs'].sum())}, frames {arrays['obs_frame'].shape[-1]} / {arrays['priv_frame'].shape[-1]}")


def make_env_golden():
    arrays = _run_reference_env(env_golden_tape(), ENV_CASE["steps"], ENV_CASE["step_counter0"])
    path = os.path.join(GOLDEN_DIR, "env_rollout_ref.npz")
    np.savez_compressed(path, **arrays)
    n_reset = int(arrays["reset"].sum())
    print(f"wrote {path}: {os.path.getsize(path) / 1e6:.2f} MB, resets={n_reset}, "
          f"time_outs={int(arrays['time_outs'].sum())}")
    arrays = _run_reference_env(delay_golden_tape(), DELAY_CASE["steps"], 0, configure=delay_cfg)
    keep = ("actions", "torques", "obs_frame", "priv_frame", "rew", "reset", "last_actions", "last_last_actions",
            "input_checksum")
    path = os.path.join(GOLDEN_DIR, "env_action_delay_ref.npz")
    np.savez_compressed(path, **{k: arrays[k] for k in keep})
    print(f"wrote {path}: {os.path.getsize(path) / 1e6:.2f} MB (action_delay = {DELAY_CASE['action_delay']})")


HEIGHT_CASE = dict(n=48, seed=77, rows=420, cols=380, border_size=25.0, horizontal_scale=0.1, vertical_scale=0.005)
MEASURED_X = [-0.8, -0.7, -0.6, -0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8]     # legged_robot_config.py:55-56
MEASURED_Y = [-0.5, -0.4, -0.3, -0.2, -0.1, 0., 0.1, 0.2, 0.3, 0.4, 0.5]


def height_golden_inputs(n=None, seed=None):
    """Root states scattered over (and a little beyond) an int16 height field, arbitrary yaw and tilt."""
    c = HEIGHT_CASE
    n = n or c["n"]
    g = torch.Generator().manual_seed(seed or c["seed"])
    field = (torch.randn(c["rows"], c["cols"], generator=g) * 40).round().to(torch.int16)       # terrain.heightsamples
    root = torch.zeros(n, 13)
    extent_x, extent_y = c["rows"] * c["horizontal_scale"], c["cols"] * c["horizontal_scale"]
    root[:, 0] = torch.rand(n, generator=g) * (extent_x + 4.0) - c["border_size"] - 2.0            # some robots off the map: clipped
    root[:, 1] = torch.rand(n, generator=g) * (extent_y + 4.0) - c["border_size"] - 2.0
    root[:, 2] = 0.55
    q = torch.randn(n, 4, generator=g)
    q[: n // 4, :2] *= 0.05                                                                      # mostly upright, some tumbling
    root[:, 3:7] = q / q.norm(dim=-1, keepdim=True)
    return root, field


def make_height_golden():
    from oracle.ref_harness import reference_get_heights
    c = HEIGHT_CASE
    root, field = height_golden_inputs()
    h = reference_get_heights(root, field, MEASURED_X, MEASURED_Y, c["border_size"], c["horizontal_scale"], c["vertical_scale"])
    # (the reference's env_ids branch cannot run: it ends in .view(self.num_envs, -1), legged_robot.py:795 - every call
    # site passes no ids)
    path = os.path.join(GOLDEN_DIR, "heights_ref.npz")
    np.savez_compressed(path, heights=h.numpy(),
                        input_checksum=np.array([float(root.double().sum()), float(field.double().sum())]))
    print(f"wrote {path}: {os.path.getsize(path) / 1e6:.3f} MB, {tuple(h.shape)}")


def golden_ppo_inputs():
    """Seeded rollout inputs for the PPO golden case (regenerated on both sides)."""
    c = PPO_CASE
    g = torch.Generator().manual_seed(c["seed"])
    steps = []
    for _ in range(c["t"]):
        obs = torch.randn(c["n"], 615, generator=g)
        cobs = torch.randn(c["n"], 1050, generator=g)
        eps = torch.randn(c["n"], 10, generator=g)
        rew = torch.rand(c["n"], generator=g)
        dones = torch.rand(c["n"], generator=g) < 0.1
        time_outs = dones & (torch.rand(c["n"], generator=g) < 0.5)
        steps.append((obs, cobs, eps, rew, dones, time_outs))
    last = torch.randn(c["n"], 1050, generator=g)
    perm = torch.randperm(c["n"] * c["t"], generator=g)
    return steps, last, perm


def param_digest(params) -> dict:
    """Strided sample + float64 statistics of every tensor (keeps the fixture small)."""
    out = {}
    for k in PARAM_ORDER:
        v = params[k].detach().double().flatten()
        out[f"p/{k}/sample"] = v[::97].float().numpy()
        out[f"p/{k}/stats"] = np.array([float(v.sum()), float(v.abs().sum()), float((v * v).sum())])
    return out


def make_ppo_golden():
    from oracle.ref_harness import ReferencePPO
    c = PPO_CASE
    params = init_actor_critic_params(seed=c["param_seed"])
    ref = ReferencePPO(params, c["n"], c["t"], PPO_ALG, PPO_POLICY)
    steps, last, perm = golden_ppo_inputs()
    arrays = {"input_checksum": np.array([float(sum(float(x.double().sum()) for x in s)) for s in steps]
                                         + [float(last.double().sum()), float(perm.double().sum())]
                                         + [float(params[k].double().sum()) for k in PARAM_ORDER])}
    for obs, cobs, eps, rew, dones, tos in steps:
        ref.act(obs, cobs, eps)
        ref.process_env_step(rew, dones, {"time_outs": tos})
    ref.compute_returns(last)
    st = ref.alg.storage
    for k in ("actions", "values", "actions_log_prob", "mu", "sigma", "rewards", "dones", "returns", "advantages"):
        arrays["st/" + k] = getattr(st, k).numpy().copy()
    # one fixed-lr update (continuous in its inputs) and one adaptive-lr update (quirk 10)
    import copy
    for tag, sched in (("fixed", "fixed"), ("adaptive", "adaptive")):
        r = ReferencePPO(params, c["n"], c["t"], dict(PPO_ALG, schedule=sched), PPO_POLICY)
        for obs, cobs, eps, rew, dones, tos in steps:
            r.act(obs, cobs, eps)
            r.process_env_step(rew, dones, {"time_outs": tos})
        r.compute_returns(last)
        losses = r.update(perm)
        arrays[f"{tag}/losses"] = np.array(losses, dtype=np.float64)
        arrays[f"{tag}/lr"] = np.array([r.alg.learning_rate], dtype=np.float64)
        arrays[f"{tag}/lr_trace"] = np.array(r.lr_trace, dtype=np.float64)      # the rate each Adam step ran with
        for k, v in param_digest(dict(r.alg.actor_critic.state_dict())).items():
            arrays[f"{tag}/{k}"] = v
    path = os.path.join(GOLDEN_DIR, "ppo_update_ref.npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}: {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    make_env_golden()
    make_task_goldens()
    make_ppo_golden()
    make_height_golden()
