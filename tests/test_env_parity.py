"""Parity of the CUDA env stage (through the C ABI) with the reference's outputs.

- against the golden vectors the UNMODIFIED reference produced (tests/golden/env_rollout_ref.npz)
- against the CPU oracle on fresh seeded tapes (ragged N, both staging paths)
- size-independent properties at BASELINE sizes (frame-stack shift, ascending reset ids, ...)
Bit-exact: termination masks, reset env_ids, episode counters.  fp32 tensors: rtol 1e-5, atol 1e-6.
"""
import numpy as np
import pytest
import torch

from _util import ENV_ATOL, GOLDEN, assert_close, assert_equal, to_np
from isaac_b200.envs.hector_config import HectorCfg
from isaac_b200.synthetic import make_tape
from oracle import make_golden as mg

pytestmark = pytest.mark.gpu

EXACT = ("reset", "time_outs", "episode_length_buf", "last_contacts")


def make_cuda_env(tape, dev, cfg=None, cls=None, device_rng=False):
    """`device_rng`: the constructor's reset takes its draws from the device generator (cfg.seed) instead of the tape."""
    from isaac_b200.envs.hector_env import HectorFreeEnvB200
    from isaac_b200.physics import SyntheticPhysics
    from isaac_b200.synthetic import task_dims
    n = tape.statics.p_gains.shape[0]
    dims = task_dims(cfg or HectorCfg())
    phys = SyntheticPhysics(n, num_dof=dims.ndof, num_bodies=dims.nbody, device=dev)
    phys.load_frame(tape.physics[0].to(dev))
    env = (cls or HectorFreeEnvB200)(cfg or HectorCfg(), sim_device=str(dev), physics=phys, statics=tape.statics,
                                     initial_noise=None if device_rng else tape.noise[0].to(dev))
    env.episode_length_buf.copy_(tape.statics.episode_length0)
    return env, phys


def cuda_step(env, phys, frame, noise, dev):
    phys.load_frame(frame.to(dev))
    nz = noise.to(dev)
    env.inject_noise(nz)
    return env.step(nz.actions)


class _View:
    """Adapts the CUDA env to oracle.make_golden.record_env_step (CPU copies of its attributes)."""

    def __init__(self, env):
        self._env = env
        self.episode_sums = {k: v.cpu() for k, v in env.episode_sums.items()}

    def __getattr__(self, k):
        return getattr(self._env, k).cpu()


def run_cuda_case(tape, dev, step_counter0=0, cfg=None, cls=None):
    env, phys = make_cuda_env(tape, dev, cfg=cfg, cls=cls)
    env.common_step_counter = step_counter0
    frames = (env.cfg.env.num_single_obs, env.cfg.env.single_num_privileged_obs)
    rec = {"obs_init": to_np(env.obs_buf), "priv_init": to_np(env.privileged_obs_buf)}
    ids_per_step, out = [], None
    for t in range(1, len(tape.physics)):
        out = cuda_step(env, phys, tape.physics[t], tape.noise[t], dev)
        cpu_out = tuple(o.cpu() for o in out[:4]) + ({"time_outs": out[4]["time_outs"].cpu(),
                                                     "episode": {k: v.cpu() for k, v in out[4]["episode"].items()}},)
        mg.record_env_step(rec, _View(env), cpu_out, env.root_states.cpu(), env.dof_state.cpu(), frames)
        n = int(env._reset_count.item())
        ids_per_step.append(env.reset_env_ids[:n].cpu().numpy().copy())
    rec = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in rec.items()}
    rec["obs_final"], rec["priv_final"] = to_np(out[0]), to_np(out[1])
    return rec, ids_per_step, env, phys


def compare_records(got, want, extra_atol=None):
    """`extra_atol`: {record key: array broadcast against that record}, added to the suite's absolute tolerance."""
    extra_atol = extra_atol or {}
    for k in EXACT:
        assert_equal(k, got[k], want[k])
    for k in want:
        if k in EXACT or k in ("input_checksum", "reward_names"):
            continue
        w = want[k]
        if k.endswith("_init"):      # the constructor's compute_observations() is not clipped by the reference
            w = np.clip(w, -100.0, 100.0)   # (only step() clips, legged_robot.py:104-107); history frames are equal after the clip
        assert_close(k, got[k], w, atol=ENV_ATOL + extra_atol.get(k, 0.0))


@pytest.mark.parametrize("bulk", [1, 0])
def test_env_matches_reference_golden(lib, cuda_device, bulk):
    assert lib.hb_set_option(b"env_bulk_staging", bulk) == 0
    g = dict(np.load(f"{GOLDEN}/env_rollout_ref.npz"))
    tape = mg.env_golden_tape()
    np.testing.assert_array_equal(mg.tape_checksum(tape), g["input_checksum"])
    rec, ids, env, phys = run_cuda_case(tape, cuda_device, mg.ENV_CASE["step_counter0"])
    compare_records(rec, g)
    for t, got in enumerate(ids):
        assert_equal(f"reset_env_ids@{t}", got, np.nonzero(g["reset"][t])[0].astype(np.int32))
    assert phys.calls["set_root_state"] >= 1, "the golden case crosses a push step"
    lib.hb_set_option(b"env_bulk_staging", 1)


@pytest.mark.parametrize("n,bulk", [(257, 1), (257, 0), (31, 1), (1024, 1), (1, 1), (33, 0), (1003, 1)])
def test_env_matches_oracle_ragged(lib, cuda_device, n, bulk):
    from oracle.hector_oracle import OracleHectorEnv
    assert lib.hb_set_option(b"env_bulk_staging", bulk) == 0
    steps = 12
    tape = make_tape(n, steps, seed=1000 + n, fall_prob=0.03, randomize_gains=True)
    special = torch.tensor([2399, 2400, 798, 799, 1599])[:min(n, 5)]
    tape.statics.episode_length0[:special.numel()] = special
    ora = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    ora.common_step_counter = 395
    want = {"obs_init": ora.obs_buf.numpy().copy(), "priv_init": ora.privileged_obs_buf.numpy().copy()}
    want_ids, out = [], None
    for t in range(1, steps):
        out = ora.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(want, ora, out, ora.root_states, ora.dof_state)
        want_ids.append(ora.last_reset_ids.numpy().astype(np.int32))
    want = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in want.items()}
    want["obs_final"], want["priv_final"] = out[0].numpy(), out[1].numpy()
    rec, ids, _, _ = run_cuda_case(tape, cuda_device, 395)
    compare_records(rec, want)
    for t, (a, b) in enumerate(zip(ids, want_ids)):
        assert_equal(f"reset_env_ids@{t}", a, b)
    assert sum(len(i) for i in want_ids) > 0 or n < 8
    lib.hb_set_option(b"env_bulk_staging", 1)


@pytest.mark.parametrize("bulk", [1, 0])
@pytest.mark.parametrize("task", ["hector_full", "humanoid_ppo"])
def test_other_tasks_match_reference_golden(lib, cuda_device, task, bulk):
    """SURVEY.md §8f rank 4: the reference's other two registered tasks (envs/__init__.py:46-48) on the same kernels,
    instantiated for their layouts - hector_full (18 DOF, frames 65 / 94, the arm term of default_joint_pos, 21 active
    reward terms) and humanoid_ppo / XBot-L (12 DOF, frames 47 / 73, critic history of 3, action delay 0.5, the
    reference-trajectory error in the privileged frame, the joint_pos reward on last step's reference) - against rollouts
    of the reference's own env classes (resets, time-outs, command resampling, a push step)."""
    from isaac_b200.envs import TASKS
    import isaac_b200.envs as envs
    assert lib.hb_set_option(b"env_bulk_staging", bulk) == 0
    cls_name, cfg_cls, _ = TASKS[task]
    g = dict(np.load(f"{GOLDEN}/env_rollout_{task}_ref.npz"))
    tape = mg.task_golden_tape(task)
    np.testing.assert_array_equal(mg.tape_checksum(tape), g["input_checksum"])
    rec, ids, env, phys = run_cuda_case(tape, cuda_device, mg.TASK_CASE["step_counter0"], cfg=cfg_cls(), cls=getattr(envs, cls_name))
    compare_records(rec, g)
    for t, got in enumerate(ids):
        assert_equal(f"reset_env_ids@{t}", got, np.nonzero(g["reset"][t])[0].astype(np.int32))
    assert phys.calls["set_root_state"] >= 1 and env.obs_buf.shape[1] == cfg_cls().env.num_observations
    assert set(env.episode_sums) == set(str(k) for k in g["reward_names"])
    lib.hb_set_option(b"env_bulk_staging", 1)


@pytest.mark.parametrize("task,n", [("hector_full", 257), ("hector_full", 4096), ("humanoid_ppo", 1003), ("humanoid_ppo", 4096)])
def test_other_tasks_match_oracle(lib, cuda_device, task, n):
    """... and against the oracle (bit-equal to the reference on these tasks: tests/test_oracle_pinning.py) at ragged and
    BASELINE shard sizes, with the CUDA-graph replay of the step checked against the eager launches at the end."""
    from oracle.hector_oracle import OracleHectorEnv
    from isaac_b200.envs import TASKS
    import isaac_b200.envs as envs
    cls_name, cfg_cls, _ = TASKS[task]
    steps = 8
    tape = make_tape(n, steps, seed=2000 + n, fall_prob=0.02, randomize_gains=True, cfg=cfg_cls())
    tape.statics.episode_length0[:5] = torch.tensor([2399, 2400, 798, 799, 1599])
    ora = OracleHectorEnv(cfg_cls(), tape.statics, tape.physics[0], tape.noise[0])
    ora.common_step_counter = 396
    frames = (cfg_cls().env.num_single_obs, cfg_cls().env.single_num_privileged_obs)
    want = {"obs_init": ora.obs_buf.numpy().copy(), "priv_init": ora.privileged_obs_buf.numpy().copy()}
    want_ids, out = [], None
    for t in range(1, steps):
        out = ora.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(want, ora, out, ora.root_states, ora.dof_state, frames)
        want_ids.append(ora.last_reset_ids.numpy().astype(np.int32))
    want = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in want.items()}
    want["obs_final"], want["priv_final"] = out[0].numpy(), out[1].numpy()
    rec, ids, env, _ = run_cuda_case(tape, cuda_device, 396, cfg=cfg_cls(), cls=getattr(envs, cls_name))
    compare_records(rec, want)
    for t, (a, b) in enumerate(zip(ids, want_ids)):
        assert_equal(f"reset_env_ids@{t}", a, b)
    if task == "humanoid_ppo":          # (hector_full never reads its reference trajectory: joint_pos has scale 0, the kernel skips it)
        assert_close("ref_dof_pos", env.ref_dof_pos.cpu().numpy(), ora.ref_dof_pos.numpy())
    # graph replay == eager on this task's kernels (device generator, same seed)
    env_g, phys_g = make_cuda_env(tape, cuda_device, cfg=cfg_cls(), cls=getattr(envs, cls_name))
    env_e, phys_e = make_cuda_env(tape, cuda_device, cfg=cfg_cls(), cls=getattr(envs, cls_name))
    env_g.seed(4), env_e.seed(4)
    env_g.enable_cuda_graph()
    for t in range(1, 4):
        fr = tape.physics[t].to(cuda_device)
        phys_g.load_frame(fr), phys_e.load_frame(fr)
        a = tape.noise[t].actions.to(cuda_device)
        og, oe = env_g.step(a), env_e.step(a)
        for x, y, name in zip(og[:4], oe[:4], ("obs", "priv", "rew", "reset")):
            assert torch.equal(x, y), f"{task}: graph replay vs eager: {name} at step {t}"


def test_env_action_delay_matches_reference_golden(lib, cuda_device):
    """The action-delay branch of the step prologue (hector_env.py:166-167; action_delay = 0.3 instead of the shipped
    0.0) against what the unmodified reference produced."""
    g = dict(np.load(f"{GOLDEN}/env_action_delay_ref.npz"))
    tape = mg.delay_golden_tape()
    np.testing.assert_array_equal(mg.tape_checksum(tape), g["input_checksum"])
    rec, _, env, _ = run_cuda_case(tape, cuda_device, 0, cfg=mg.delay_cfg(HectorCfg()))
    assert abs(env._p.action_delay - 0.3) < 1e-7
    assert_equal("reset", rec["reset"], g["reset"])
    for k in ("actions", "torques", "obs_frame", "priv_frame", "rew", "last_actions", "last_last_actions"):
        assert_close(k, rec[k], g[k])


@pytest.mark.parametrize("n,steps,dr", [(4096, 4, False), (16384, 4, True), (65536, 3, False)],
                         ids=["configs1-4096", "configs2-16384-dr-noise", "configs3-65536"])
def test_env_matches_oracle_at_baseline_sizes(lib, cuda_device, n, steps, dr):
    """BASELINE.json's shard sizes against the CPU oracle itself, every recorded tensor (same comparison as the ragged
    cases): 4096 envs with the shipped constants (configs[1]); 16384 envs with per-env kp / kd, friction and mass
    domain randomisation and injected observation / action noise (configs[2]); 65536 envs (configs[3]'s total)."""
    from oracle.hector_oracle import OracleHectorEnv
    tape = make_tape(n, steps, seed=5000 + n, fall_prob=0.01, randomize_gains=dr)
    assert dr or tape.statics.p_gains.std(dim=0).max() == 0, "configs[1] / [3]: the shipped kp / kd constants"
    special = torch.tensor([2399, 2400, 798, 799, 1599])
    tape.statics.episode_length0[:5] = special
    ora = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    ora.common_step_counter = 398                      # the second step is a push step
    want = {"obs_init": ora.obs_buf.numpy().copy(), "priv_init": ora.privileged_obs_buf.numpy().copy()}
    want_ids, out = [], None
    for t in range(1, steps):
        out = ora.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(want, ora, out, ora.root_states, ora.dof_state)
        want_ids.append(ora.last_reset_ids.numpy().astype(np.int32))
    want = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in want.items()}
    want["obs_final"], want["priv_final"] = out[0].numpy(), out[1].numpy()
    rec, ids, _, phys = run_cuda_case(tape, cuda_device, 398)
    compare_records(rec, want)
    for t, (a, b) in enumerate(zip(ids, want_ids)):
        assert_equal(f"reset_env_ids@{t}", a, b)
    assert sum(len(i) for i in want_ids) > n // 200 and phys.calls["set_root_state"] >= 1
    if dr:
        assert tape.statics.p_gains.std() > 1 and tape.statics.env_frictions.unique().numel() > 100


def test_overridden_hooks_run_the_staged_step(lib, cuda_device):
    """SURVEY.md §8b: check_termination / compute_reward / reset_idx / compute_observations are overridable hooks with the
    reference's names.  A subclass that overrides them (here: pass-through overrides that count their calls) makes
    post_physics_step call them one by one in the reference's order (legged_robot.py:118-153), each a launch of the same
    kernel restricted to that span - and the golden rollout of the unmodified reference must come out all the same,
    resets, time-outs, push step and extras included.  A second subclass changes the reward through its hook."""
    from isaac_b200.envs.hector_env import HectorFreeEnvB200
    calls = {"check_termination": 0, "compute_reward": 0, "reset_idx": 0, "compute_observations": 0}
    seen_ids = []

    class Staged(HectorFreeEnvB200):
        def check_termination(self):
            calls["check_termination"] += 1
            super().check_termination()

        def compute_reward(self):
            calls["compute_reward"] += 1
            super().compute_reward()

        def reset_idx(self, env_ids):
            calls["reset_idx"] += 1
            if self.init_done and calls["check_termination"]:        # (the constructor resets every env first)
                seen_ids.append(torch.as_tensor(env_ids).cpu().numpy().astype(np.int32))
            super().reset_idx(env_ids)

        def compute_observations(self):
            calls["compute_observations"] += 1
            super().compute_observations()

    g = dict(np.load(f"{GOLDEN}/env_rollout_ref.npz"))
    tape = mg.env_golden_tape()
    rec, ids, env, phys = run_cuda_case(tape, cuda_device, mg.ENV_CASE["step_counter0"], cls=Staged)
    steps = mg.ENV_CASE["steps"] - 1
    assert calls["check_termination"] == calls["compute_reward"] == calls["compute_observations"] == steps
    assert calls["reset_idx"] == steps, "reset_idx is called every step (with an empty id list on most)"
    compare_records(rec, g)
    assert len(seen_ids) == steps
    for t, got in enumerate(seen_ids):       # env_ids = reset_buf.nonzero() as handed to the hook (legged_robot.py:142-143)
        assert_equal(f"reset_idx(env_ids)@{t}", got, np.nonzero(g["reset"][t])[0].astype(np.int32))

    class Bonus(HectorFreeEnvB200):
        def compute_reward(self):
            super().compute_reward()
            self.rew_buf += 1.0

    tape2 = make_tape(64, 3, seed=5)
    plain, p1 = make_cuda_env(tape2, cuda_device)
    bonus, p2 = make_cuda_env(tape2, cuda_device, cls=Bonus)
    for t in (1, 2):
        a = cuda_step(plain, p1, tape2.physics[t], tape2.noise[t], cuda_device)
        b = cuda_step(bonus, p2, tape2.physics[t], tape2.noise[t], cuda_device)
        assert torch.equal(b[2], a[2] + 1.0) and torch.equal(a[0], b[0]) and torch.equal(a[3], b[3])
    # the hooks also work on their own, on the current buffers (what play.py-style code does)
    before = plain.rew_buf.clone()
    plain.check_termination()
    f = tape2.physics[2].contact_forces.to(cuda_device)
    want_reset = (f[:, [0, 3, 8]].norm(dim=-1) > 1.0).any(dim=1) | (plain.episode_length_buf > 2400)
    assert torch.equal(plain.reset_buf, want_reset) and torch.equal(plain.rew_buf, before)


def test_get_heights_matches_reference_golden_and_oracle(lib, cuda_device):
    """LeggedRobot._get_heights (legged_robot.py:759-795) as a kernel: bit-exact against the reference's own output on the
    golden case and against the oracle at 4096 envs (every value is an int16 sample x vertical_scale: a cell index off by
    one would show), including an env_ids subset and the measure_heights refresh inside step()."""
    from oracle.hector_oracle import get_heights, height_points
    dev = cuda_device
    g = np.load(f"{GOLDEN}/heights_ref.npz")
    c = mg.HEIGHT_CASE
    for n, seed, golden in ((c["n"], None, g["heights"]), (4096, 9, None)):
        root, field = mg.height_golden_inputs(n=n, seed=seed)
        cfg = HectorCfg()
        cfg.terrain.measure_heights = True
        tape = make_tape(n, 2, seed=4)
        env, phys = make_cuda_env(tape, dev, cfg=cfg)
        env.set_height_field(field, mg.MEASURED_X, mg.MEASURED_Y)
        env.root_states.copy_(root)
        got = env._get_heights().cpu()
        want = get_heights(root, height_points(mg.MEASURED_X, mg.MEASURED_Y, n), field, c["border_size"],
                           c["horizontal_scale"], c["vertical_scale"])
        assert_equal("heights vs oracle", got.numpy(), want.numpy())
        if golden is not None:
            assert_equal("heights vs reference golden", got.numpy(), golden)
        ids = [3, n - 1, 7]
        assert_equal("env_ids subset", env._get_heights(ids).cpu().numpy(), want[ids].numpy())
        # step() refreshes measured_heights in the callback, i.e. from the state the physics produced, before any env is
        # reset (legged_robot.py:315-316)
        fr = tape.physics[1]
        fr.root_states[:, :2] = root[:, :2]
        cuda_step(env, phys, fr, tape.noise[1], dev)
        want2 = get_heights(fr.root_states, height_points(mg.MEASURED_X, mg.MEASURED_Y, n), field, c["border_size"],
                            c["horizontal_scale"], c["vertical_scale"])
        assert_equal("measured_heights after step", env.measured_heights.cpu().numpy(), want2.numpy())
        assert int(env.reset_buf.sum()) > 0 or n < 100


def test_pd_torque_law(lib, cuda_device):
    """legged_robot.py:339-355 alone, including clipping at the URDF effort limits."""
    from oracle.hector_oracle import OracleHectorEnv
    tape = make_tape(1000, 2, seed=5, randomize_gains=True)
    env, phys = make_cuda_env(tape, cuda_device)
    ora = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    a = 8.0 * torch.randn(1000, 10, generator=torch.Generator().manual_seed(1))
    fr = tape.physics[1]
    phys.load_frame(fr.to(cuda_device))
    ora.dof_state.copy_(fr.dof_state)
    env.actions.copy_(a)
    tau = env._compute_torques().cpu()
    want = ora.compute_torques(a)
    assert_close("torques", tau.numpy(), want.numpy())
    assert (want.abs() == ora.torque_limits).any(), "case must hit the torque limits"


@pytest.mark.parametrize("n", [4096, 16384, 65536])
def test_step_properties_at_baseline_sizes(lib, cuda_device, n):
    """Size-independent properties at BASELINE.json sizes (the oracle would take minutes here); the 16384-env case
    is BASELINE configs[2]: per-env kp / kd and friction / mass domain randomisation, injected noise."""
    dev = cuda_device
    tape = make_tape(n, 3, seed=7, fall_prob=0.01, randomize_gains=(n == 16384))
    env, phys = make_cuda_env(tape, dev)
    prev_obs, prev_priv = env.obs_buf.clone(), env.privileged_obs_buf.clone()
    for t in (1, 2):
        ep_before = env.episode_length_buf.clone()
        obs, priv, rew, reset, extras = cuda_step(env, phys, tape.physics[t], tape.noise[t], dev)
        torch.cuda.synchronize()
        keep = ~reset
        # frame stacking: slots 0..13 are last step's slots 1..14; reset envs restart from zeros
        assert torch.equal(obs[keep][:, :574], prev_obs[keep][:, 41:])
        assert torch.equal(priv[keep][:, :980], prev_priv[keep][:, 70:])
        assert (obs[reset][:, :574] == 0).all() and (priv[reset][:, :980] == 0).all()
        # termination mask = contact on base/thigh bodies or time-out (legged_robot.py:155-160)
        f = tape.physics[t].contact_forces.to(dev)
        want_reset = (f[:, [0, 3, 8]].norm(dim=-1) > 1.0).any(dim=1) | (ep_before + 1 > 2400)
        assert torch.equal(reset, want_reset)
        # reset ids: ascending, exactly nonzero(reset); counters restart
        cnt = int(env._reset_count.item())
        assert cnt == int(reset.sum()) and cnt > 0
        assert torch.equal(env.reset_env_ids[:cnt].long(), reset.nonzero().flatten())
        assert (env.episode_length_buf[reset] == 0).all()
        assert torch.equal(env.episode_length_buf[keep], ep_before[keep] + 1)
        assert (rew >= 0).all() and torch.isfinite(obs).all() and torch.isfinite(priv).all()
        assert obs.abs().max() <= 100 and priv.abs().max() <= 100
        # domain randomisation reaches the newest privileged frame: friction, mass / 30 (hector_env.py:210-211)
        assert torch.equal(priv[:, 980 + 64], tape.statics.env_frictions.to(dev).flatten())
        assert torch.equal(priv[:, 980 + 65].cpu(), (tape.statics.body_mass / 30.0).flatten())    # IEEE division, as on the CPU
        prev_obs, prev_priv = obs.clone(), priv.clone()
    env._apply_pending_resets()
    assert env.last_reset_count == cnt and phys.calls["set_dof_state_indexed"] >= 1


def test_returned_observations_survive_the_next_step(lib, cuda_device):
    """PPO.act keeps references to obs until process_env_step (ppo.py:99-100,111): ping-pong buffers."""
    tape = make_tape(64, 3, seed=3)
    env, phys = make_cuda_env(tape, cuda_device)
    o1 = cuda_step(env, phys, tape.physics[1], tape.noise[1], cuda_device)[0]
    snap = o1.clone()
    o2 = cuda_step(env, phys, tape.physics[2], tape.noise[2], cuda_device)[0]
    assert o1.data_ptr() != o2.data_ptr() and torch.equal(o1, snap)


def test_reset_then_step_matches_reference_reset(lib, cuda_device):
    """LeggedRobot.reset(): reset_idx(all) then step(zeros) (legged_robot.py:111-116)."""
    from oracle.hector_oracle import OracleHectorEnv
    tape = make_tape(96, 4, seed=11)
    env, phys = make_cuda_env(tape, cuda_device)
    ora = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    cuda_step(env, phys, tape.physics[1], tape.noise[1], cuda_device)
    ora.step(tape.physics[1], tape.noise[1])
    # reset_idx(all) with tape 2, then a zero-action step on frame 3
    nz2 = tape.noise[2].to(cuda_device)
    env.inject_noise(nz2)
    env.reset_idx(torch.arange(96))
    ora.reset_idx(torch.arange(96), tape.noise[2])
    import dataclasses
    nz3 = dataclasses.replace(tape.noise[3], actions=torch.zeros(96, 10))
    out = cuda_step(env, phys, tape.physics[3], nz3, cuda_device)
    want = ora.step(tape.physics[3], nz3)
    assert_close("obs", to_np(out[0]), want[0].numpy())
    assert_close("priv", to_np(out[1]), want[1].numpy())
    assert_close("rew", to_np(out[2]), want[2].numpy())
    assert_equal("reset", to_np(out[3]), to_np(want[3]))


def test_cuda_graph_replay_equals_eager(lib, cuda_device):
    """The captured step (2 graphs per ping-pong parity) must produce exactly what the eager launches
    produce from the same state and the same draws (both envs use the device generator: same seed, same
    step counter -> same draws)."""
    dev = cuda_device
    n = 512
    tape = make_tape(n, 6, seed=21, fall_prob=0.02)
    env_g, phys_g = make_cuda_env(tape, dev)
    env_e, phys_e = make_cuda_env(tape, dev)
    env_g.seed(9), env_e.seed(9)
    env_g.common_step_counter = env_e.common_step_counter = 397      # step 3 is a push step: the graph env takes the eager path there
    env_g.enable_cuda_graph()
    for t in range(1, 6):
        fr = tape.physics[t].to(dev)
        phys_g.load_frame(fr), phys_e.load_frame(fr)
        actions = tape.noise[t].actions.to(dev)
        out_g = env_g.step(actions)
        out_e = env_e.step(actions)
        torch.cuda.synchronize()
        for a, b, name in zip(out_g[:4], out_e[:4], ("obs", "priv", "rew", "reset")):
            assert torch.equal(a, b), f"{name} differs at step {t}"
        assert torch.equal(out_g[4]["time_outs"], out_e[4]["time_outs"])
        for k in out_e[4]["episode"]:
            assert torch.equal(out_g[4]["episode"][k], out_e[4]["episode"][k]), k
        assert torch.equal(env_g.episode_length_buf, env_e.episode_length_buf)
        assert torch.equal(env_g._episode_sums, env_e._episode_sums)
    env_g._apply_pending_resets()
    assert phys_g.calls["set_dof_state_indexed"] >= 1
    assert phys_g.calls["set_root_state"] == 1 and phys_e.calls["set_root_state"] == 1, "one push step in the window"


def test_device_generator_draws(lib, cuda_device):
    """The env's own draws (no injected tape): Philox in-kernel.  The observation noise must be N(0, 1) scaled by
    noise_scale_vec * noise_level on the noisy columns and absent elsewhere, independent across envs and steps,
    and a pure function of (seed, step): two envs with the same seed agree bit for bit, another seed does not."""
    n, dev = 4096, cuda_device
    tape = make_tape(n, 3, seed=77, fall_prob=0.0)
    tape.statics.episode_length0.fill_(10)           # no time-outs, no resampling: the newest frame is a pure function of the state
    cfg = HectorCfg()

    def run(seed, noise):
        c = HectorCfg()
        c.noise.add_noise = noise
        env, phys = make_cuda_env(tape, dev, cfg=c)
        env.seed(seed)
        frames = []
        for t in (1, 2):
            phys.load_frame(tape.physics[t].to(dev))
            obs = env.step(tape.noise[t].actions.to(dev))[0]
            frames.append(obs[:, -41:].clone())
        return torch.stack(frames)

    clean = run(1, False)
    a, b, c = run(1, True), run(1, True), run(2, True)
    assert torch.equal(a, b), "same seed, same step counter -> same draws"
    assert not torch.equal(a, c)
    scale = torch.tensor(list(make_cuda_env(tape, dev)[0]._p.noise_scale_vec[:41]), device=dev) * cfg.noise.noise_level
    noisy = scale > 0
    # action noise (domain_rand.action_noise) perturbs the action columns of both runs identically? no: the clean run has
    # add_noise off but the same action noise, so the action columns (scale 0) must agree exactly
    resid = a - clean
    assert torch.equal(resid[:, :, ~noisy], torch.zeros_like(resid[:, :, ~noisy]))
    z = resid[:, :, noisy] / scale[noisy]
    assert abs(z.mean().item()) < 0.01 and abs(z.std().item() - 1.0) < 0.01
    assert abs((z ** 4).mean().item() - 3.0) < 0.15                       # kurtosis of a normal
    z0, z1 = z[0].flatten(), z[1].flatten()
    assert abs(torch.corrcoef(torch.stack((z0, z1)))[0, 1].item()) < 0.01   # step to step
    cols = z[0]
    cc = torch.corrcoef(cols.T)
    assert (cc - torch.eye(cc.shape[0], device=dev)).abs().max().item() < 0.08   # column to column (n = 4096)
    assert abs(torch.corrcoef(torch.stack((cols[:-1, 0], cols[1:, 0])))[0, 1].item()) < 0.06   # env to env


@pytest.mark.parametrize("pitched", [False, True], ids=["dense", "pitched"])
@pytest.mark.parametrize("n", [1, 37, 1003, 4096])
def test_fused_shift_finalize_equals_separate_calls(lib, cuda_device, n, pitched):
    """hb_env_stack_finalize (what step() launches) against hb_env_stack_observations + hb_env_reset_finalize on the
    same inputs: identical frame stacks, id lists, counts, episode means and time-out latch (ragged sizes included:
    615 n is not a multiple of 4 for n = 1003, the last ballot word is partial for n = 37).  Both row layouts:
    dense [n,615] / [n,1050] and the 128-byte pitch the env and the rollout storage use (640 / 1056)."""
    from isaac_b200 import _lib
    dev = cuda_device
    tape = make_tape(n, 2, seed=3 + n, fall_prob=0.2)
    env, phys = make_cuda_env(tape, dev)
    ld_o, ld_p = (640, 1056) if pitched else (615, 1050)
    env._p.obs_ld, env._p.priv_ld = (ld_o, ld_p) if pitched else (0, 0)
    g = torch.Generator(device=dev).manual_seed(n)
    prev_o, prev_p = torch.randn(n, ld_o, device=dev, generator=g), torch.randn(n, ld_p, device=dev, generator=g)
    reset = torch.rand(n, device=dev, generator=g) < 0.3
    if n == 37:
        reset[36] = True           # the last, partial tile
    tiles = (n + 31) // 32
    pad = torch.zeros(tiles * 32, dtype=torch.bool, device=dev)
    pad[:n] = reset
    weights = (2 ** torch.arange(32, device=dev, dtype=torch.int64))
    ballots = (pad.view(tiles, 32).long() * weights).sum(1)
    ballots = torch.where(ballots >= 2 ** 31, ballots - 2 ** 32, ballots).to(torch.int32)
    sums = torch.rand(_lib.HB_NUM_REWARDS, dtype=torch.float64, device=dev, generator=g)
    st = torch.cuda.current_stream(dev).cuda_stream
    results = []
    for fused in (False, True):
        env.reset_buf.copy_(reset)
        env.time_out_buf.copy_(torch.rand(n, device=dev, generator=torch.Generator(device=dev).manual_seed(1)) < 0.5)
        env._time_outs_latched.zero_()
        env._scratch_ballots.copy_(ballots)
        env._scratch_sums.copy_(sums)
        env.reset_env_ids.fill_(-1)
        # the outputs live inside larger allocations with sentinel guards on both sides (compute-sanitizer is not
        # available on this pool: an out-of-bounds store of the ragged tail paths would show up here)
        GUARD = 1024
        raw_o = torch.full((n * ld_o + 2 * GUARD,), -3.0, device=dev)
        raw_p = torch.full((n * ld_p + 2 * GUARD,), -3.0, device=dev)
        new_o, new_p = raw_o[GUARD:GUARD + n * ld_o].view(n, ld_o), raw_p[GUARD:GUARD + n * ld_p].view(n, ld_p)
        new_o.fill_(7.0), new_p.fill_(7.0)
        assert new_o.data_ptr() % 16 == 0 and new_p.data_ptr() % 16 == 0
        means = torch.zeros(_lib.HB_NUM_REWARDS, device=dev)
        env._b.episode_means, env._b.episode_means_prev, env._b.episode_ring = means.data_ptr(), None, None
        P, B, hc = env._pp, env._pb, env._host_count.data_ptr()
        if fused:
            _lib.check(lib.hb_env_stack_finalize(P, B, prev_o.data_ptr(), prev_p.data_ptr(), new_o.data_ptr(), new_p.data_ptr(),
                                                 hc, None, st), "fused")
        else:
            _lib.check(lib.hb_env_stack_observations(P, B, prev_o.data_ptr(), prev_p.data_ptr(), new_o.data_ptr(),
                                                     new_p.data_ptr(), st), "stack")
            _lib.check(lib.hb_env_reset_finalize(P, B, new_o.data_ptr(), new_p.data_ptr(), hc, None, st), "finalize")
        torch.cuda.synchronize()
        for raw, size in ((raw_o, n * ld_o), (raw_p, n * ld_p)):
            assert (raw[:GUARD] == -3.0).all() and (raw[GUARD + size:] == -3.0).all(), "store outside the frame stack"
        cnt = int(env._reset_count.item())
        results.append((new_o.clone(), new_p.clone(), cnt, env.reset_env_ids[:cnt].clone(), means.clone(),
                        env._time_outs_latched.clone(), int(env._host_count[0]), env._scratch_sums.clone()))
    a, b = results
    for x, y in zip(a, b):
        assert (x == y) if isinstance(x, int) else torch.equal(x, y)
    new_o, new_p, cnt, ids, means, latch, host, sums_after = b
    keep = ~reset
    assert torch.equal(new_o[keep][:, :574], prev_o[keep][:, 41:615]) and (new_o[reset][:, :574] == 0).all()
    assert torch.equal(new_p[keep][:, :980], prev_p[keep][:, 70:1050]) and (new_p[reset][:, :980] == 0).all()
    assert (new_o[:, 574:] == 7.0).all() and (new_p[:, 980:] == 7.0).all(), "the newest-frame slot (and the row padding) belongs to post-physics"
    assert cnt == int(reset.sum()) == host and torch.equal(ids.long(), reset.nonzero().flatten())
    if cnt:
        np.testing.assert_allclose(means.cpu().numpy(), (sums / cnt).float().cpu().numpy() / 24.0, rtol=1e-6)
        assert torch.equal(latch, env.time_out_buf) and (sums_after == 0).all()


def test_soak_replayed_steps_and_learning_iterations(lib, cuda_device):
    """A few thousand replayed steps (CUDA graphs, device generator, PDL launches) and several full learning
    iterations: the invariants of a step must hold at every checkpoint and nothing may drift to NaN - guards the
    asynchronous machinery (graphs, programmatic dependent launches, ping-pong buffers, two-stream update)."""
    from isaac_b200.algo import ActorCritic, PPO
    dev = cuda_device
    n, frames = 2048, 4
    tape = make_tape(n, frames + 1, seed=99, fall_prob=0.01, randomize_gains=True)
    env, phys = make_cuda_env(tape, dev)
    env.seed(123)
    phys_frames = [f.to(dev) for f in tape.physics[1:]]
    env.enable_cuda_graph()
    actions = torch.zeros(n, 10, device=dev)
    prev_obs = env.obs_buf.clone()
    total_resets = 0
    for t in range(3000):
        phys.load_frame(phys_frames[t % frames])
        actions.normal_()
        check = t % 500 == 499
        if check:
            prev_obs = env.obs_buf.clone()
            ep_before = env.episode_length_buf.clone()
        obs, priv, rew, reset, extras = env.step(actions)
        if check:
            torch.cuda.synchronize()
            keep = ~reset
            assert torch.equal(obs[keep][:, :574], prev_obs[keep][:, 41:]), t
            assert (obs[reset][:, :574] == 0).all() and (priv[reset][:, :980] == 0).all()
            cnt = int(env._reset_count.item())
            assert cnt == int(reset.sum()) == int(env._host_count[0])
            assert torch.equal(env.reset_env_ids[:cnt].long(), reset.nonzero().flatten())
            assert torch.equal(env.episode_length_buf[keep], ep_before[keep] + 1)
            assert torch.isfinite(obs).all() and torch.isfinite(priv).all() and torch.isfinite(rew).all()
            assert (rew >= 0).all() and obs.abs().max() <= 100
            assert all(torch.isfinite(v) for v in extras["episode"].values())
            total_resets += cnt
    assert total_resets > 0 and int(env._rng_counter.item()) >= 3000
    # learning iterations driven like OnPolicyRunner.learn (on_policy_runner.py:124-170)
    torch.manual_seed(1)
    ac = ActorCritic(615, 1050, 10, actor_hidden_dims=[512, 256, 128], critic_hidden_dims=[768, 256, 128], device=dev)
    alg = PPO(ac, device=dev, num_learning_epochs=2, num_mini_batches=4, clip_param=0.2, gamma=0.994, lam=0.9,
              value_loss_coef=1.0, entropy_coef=0.001, learning_rate=1e-4, max_grad_norm=1.0, schedule="adaptive", desired_kl=0.01)
    T = 8
    alg.init_storage(n, T, [615], [1050], [10])
    obs, priv = env.get_observations(), env.get_privileged_observations()
    w0 = ac.flat.clone()
    for it in range(6):
        for t in range(T):
            a = alg.act(obs, priv)
            phys.load_frame(phys_frames[t % frames])
            obs, priv, rew, dones, infos = env.step(a)
            alg.process_env_step(rew, dones, infos)
        alg.compute_returns(priv)
        v_loss, s_loss = alg.update()
        assert np.isfinite(v_loss) and np.isfinite(s_loss) and np.isfinite(alg.last_mean_kl), (it, v_loss, s_loss)
        assert torch.isfinite(ac.flat).all() and 1e-5 <= alg.learning_rate <= 1e-2
    assert not torch.equal(w0, ac.flat) and (ac.grad == 0).all()


def test_caller_supplied_observation_buffers(lib, cuda_device):
    """set_next_observation_buffers: the step writes into the caller's pitched buffers (one step only) exactly what
    it would have written into its own pair; buffers of the wrong shape / pitch / aliasing the current ones are
    refused."""
    dev = cuda_device
    n = 257
    tape = make_tape(n, 4, seed=21, fall_prob=0.1)
    env_a, phys_a = make_cuda_env(tape, dev)
    env_b, phys_b = make_cuda_env(tape, dev)
    env_a.seed(5), env_b.seed(5)
    ext = [(torch.full((n, 640), 9.0, device=dev), torch.full((n, 1056), 9.0, device=dev)) for _ in range(2)]
    actions = torch.zeros(n, 10, device=dev)
    for k in range(3):
        frame = tape.physics[k + 1].to(dev)
        phys_a.load_frame(frame), phys_b.load_frame(frame)
        want_o, want_p = env_a.step(actions)[:2]
        if k < 2:
            o, p = ext[k][0][:, :615], ext[k][1][:, :1050]
            env_b.set_next_observation_buffers(o, p)
        got_o, got_p = env_b.step(actions)[:2]
        if k < 2:
            assert got_o.data_ptr() == o.data_ptr() and got_p.data_ptr() == p.data_ptr()
            assert (ext[k][0][:, 615:] == 9.0).all() and (ext[k][1][:, 1050:] == 9.0).all(), "row padding is never written"
        else:
            assert got_o.data_ptr() in (env_b._own[0][0].data_ptr(), env_b._own[1][0].data_ptr()), "one step only"
        assert torch.equal(got_o, want_o) and torch.equal(got_p, want_p), k
    with pytest.raises(ValueError):
        env_b.set_next_observation_buffers(torch.zeros(n, 615, device=dev), ext[0][1][:, :1050])     # dense rows
    with pytest.raises(ValueError):
        env_b.set_next_observation_buffers(ext[0][0][:-1, :615], ext[0][1][:-1, :1050])             # wrong num_envs
    with pytest.raises(ValueError):
        env_b.set_next_observation_buffers(env_b.obs_buf, ext[0][1][:, :1050])                      # aliases the current
