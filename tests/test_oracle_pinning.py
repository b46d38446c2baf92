"""Pins the CPU oracle (oracle/*.py) before anything is checked against it.

1. against golden vectors produced by the UNMODIFIED reference (tests/golden/*.npz,
   written by oracle/make_golden.py where the reference is installed);
2. where the reference is found (oracle/ref_harness.py): live, side by side, bit for bit;
3. the quaternion helpers (closed isaacgym.torch_utils, "parity unpinned" upstream)
   against scipy's rotations.
"""
import numpy as np
import pytest
import torch

from conftest import HAVE_REFERENCE
from _util import GOLDEN, assert_close, assert_equal, to_np
from isaac_b200.envs.hector_config import HectorCfg
from oracle import make_golden as mg
from oracle.hector_oracle import OracleHectorEnv, euler_xyz_wrapped, quat_apply, quat_rotate_inverse
from oracle.ppo_oracle import OraclePPO, PARAM_ORDER, init_actor_critic_params

needs_reference = pytest.mark.skipif(not HAVE_REFERENCE, reason="needs the upstream reference: set ISAAC_REFERENCE "
                                                                   "to a checkout of DRCL-USC/isaac")

# The oracle is torch-on-CPU like the reference: identical ops, so only the CPU's vector ISA
# (AVX2 vs AVX-512 libm paths) can move the last bit.
TIGHT = dict(rtol=2e-6, atol=2e-7)


def run_oracle_env_case():
    tape = mg.env_golden_tape()
    env = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    env.common_step_counter = mg.ENV_CASE["step_counter0"]
    rec = {"obs_init": env.obs_buf.numpy().copy(), "priv_init": env.privileged_obs_buf.numpy().copy()}
    out = None
    for t in range(1, mg.ENV_CASE["steps"]):
        out = env.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(rec, env, out, env.root_states, env.dof_state)
    rec = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in rec.items()}
    rec["obs_final"], rec["priv_final"] = out[0].numpy(), out[1].numpy()
    return tape, rec


def test_golden_inputs_regenerate():
    g = np.load(f"{GOLDEN}/env_rollout_ref.npz")
    np.testing.assert_allclose(mg.tape_checksum(mg.env_golden_tape()), g["input_checksum"], rtol=0, atol=0,
                               err_msg="synthetic tape generator drifted: regenerate goldens with oracle/make_golden.py")


def test_env_oracle_matches_reference_golden():
    g = np.load(f"{GOLDEN}/env_rollout_ref.npz")
    _, rec = run_oracle_env_case()
    assert list(g["reward_names"]) == sorted(rec_names()), "reward set / order differs"
    for k in ("reset", "time_outs", "episode_length_buf", "last_contacts"):
        assert_equal(k, rec[k], g[k])
    for k in rec:
        if k in ("reset", "time_outs", "episode_length_buf", "last_contacts"):
            continue
        assert_close(k, rec[k], g[k], **TIGHT)
    assert g["reset"].sum() > 20 and g["time_outs"].sum() > 0, "golden case must exercise resets and time-outs"


@pytest.mark.parametrize("task", ["hector_full", "humanoid_ppo"])
def test_env_oracle_other_tasks_match_reference_golden(task):
    """The other two registered tasks (hector_w_arm_env.py, humanoid_env.py) through the same oracle class, against the
    rollouts of the reference's own env classes stored by oracle/make_golden.py (resets, time-outs, command resampling,
    a push step)."""
    from isaac_b200.envs.tasks import TASKS
    cfg = TASKS[task][1]()
    g = np.load(f"{GOLDEN}/env_rollout_{task}_ref.npz")
    tape = mg.task_golden_tape(task)
    np.testing.assert_array_equal(mg.tape_checksum(tape), g["input_checksum"])
    env = OracleHectorEnv(cfg, tape.statics, tape.physics[0], tape.noise[0])
    env.common_step_counter = mg.TASK_CASE["step_counter0"]
    rec = {"obs_init": env.obs_buf.numpy().copy(), "priv_init": env.privileged_obs_buf.numpy().copy()}
    frames = (cfg.env.num_single_obs, cfg.env.single_num_privileged_obs)
    for t in range(1, mg.TASK_CASE["steps"]):
        out = env.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(rec, env, out, env.root_states, env.dof_state, frames)
    rec = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in rec.items()}
    rec["obs_final"], rec["priv_final"] = out[0].numpy(), out[1].numpy()
    assert list(g["reward_names"]) == sorted(env.episode_sums), "reward set / order differs"
    for k in rec:
        if k in ("reset", "time_outs", "episode_length_buf", "last_contacts"):
            assert_equal(k, rec[k], g[k])
        else:
            assert_close(k, rec[k], g[k], **TIGHT)
    assert g["reset"].sum() >= 5 and g["time_outs"].sum() > 0, "golden case must exercise resets and time-outs"


def test_env_oracle_action_delay_matches_reference_golden():
    """hector_env.py:166-167 with action_delay = 0.3 (dead code at the shipped 0.0): the reference's own outputs."""
    g = np.load(f"{GOLDEN}/env_action_delay_ref.npz")
    tape = mg.delay_golden_tape()
    np.testing.assert_array_equal(mg.tape_checksum(tape), g["input_checksum"])
    env = OracleHectorEnv(mg.delay_cfg(HectorCfg()), tape.statics, tape.physics[0], tape.noise[0])
    rec = {}
    for t in range(1, mg.DELAY_CASE["steps"]):
        out = env.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(rec, env, out, env.root_states, env.dof_state)
    assert_equal("reset", np.stack(rec["reset"]), g["reset"])
    for k in ("actions", "torques", "obs_frame", "priv_frame", "rew", "last_actions", "last_last_actions"):
        assert_close(k, np.stack(rec[k]), g[k], **TIGHT)
    # the delay really mixes in the previous action: without it the recorded actions differ
    plain = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    for t in range(1, 3):          # step 1 blends with the zero actions of the constructor's reset, step 2 with step 1's
        plain.step(tape.physics[t], tape.noise[t])
    assert np.abs(plain.actions.numpy() - g["actions"][1]).max() > 1e-3


def test_height_oracle_matches_reference_golden():
    """LeggedRobot._get_heights (legged_robot.py:759-795): the restatement against what the reference's own function
    returned for the golden case (robots on, at the edge of and off the height field; arbitrary orientation) - every
    height is an int16 sample times vertical_scale, so equality is exact."""
    from oracle.hector_oracle import get_heights, height_points
    g = np.load(f"{GOLDEN}/heights_ref.npz")
    root, field = mg.height_golden_inputs()
    np.testing.assert_array_equal(g["input_checksum"], [float(root.double().sum()), float(field.double().sum())])
    c = mg.HEIGHT_CASE
    pts = height_points(mg.MEASURED_X, mg.MEASURED_Y, c["n"])
    h = get_heights(root, pts, field, c["border_size"], c["horizontal_scale"], c["vertical_scale"])
    assert_equal("heights", h.numpy(), g["heights"])
    assert np.unique(g["heights"]).size > 100 and g["heights"].shape == (c["n"], 187)


@needs_reference
def test_height_oracle_equal_to_live_reference():
    from oracle.hector_oracle import get_heights, height_points
    from oracle.ref_harness import reference_get_heights
    c = mg.HEIGHT_CASE
    root, field = mg.height_golden_inputs(n=300, seed=5)
    want = reference_get_heights(root, field, mg.MEASURED_X, mg.MEASURED_Y, c["border_size"], c["horizontal_scale"], c["vertical_scale"])
    pts = height_points(mg.MEASURED_X, mg.MEASURED_Y, 300)
    got = get_heights(root, pts, field, c["border_size"], c["horizontal_scale"], c["vertical_scale"])
    assert torch.equal(got, want)


@needs_reference
def test_task_configs_equal_the_reference_configs():
    """isaac_b200.envs.tasks restates the three registered tasks' configs (envs/__init__.py:46-48) as deltas over
    HectorCfg: every hot-path field must equal the reference's own config object, env and PPO side."""
    import importlib
    from oracle import ref_harness
    from isaac_b200.envs import tasks
    from isaac_b200.envs.hector_config import HectorCfgPPO, class_to_dict
    ref_harness.install_isaacgym_stub()
    ours_only = {"body_names", "dof_names", "dof_effort", "num_envs", "horizontal_scale", "vertical_scale", "border_size",
                 "measured_points_x", "measured_points_y"}

    def diff(a, b, path=""):
        out = []
        for k, v in a.items():
            if k in ours_only:
                continue
            if k not in b:
                out.append(path + k + " (absent in the reference)")
            elif isinstance(v, dict):
                out += diff(v, b[k], path + k + ".")
            elif v != b[k]:
                out.append(f"{path}{k}: {v} != {b[k]}")
        return out

    for mod, name, mine in (("hector_config", "HectorCfg", HectorCfg), ("hector_config", "HectorCfgPPO", HectorCfgPPO),
                            ("hector_w_arm_config", "HectorFullCfg", tasks.HectorFullCfg),
                            ("hector_w_arm_config", "HectorFullCfgPPO", tasks.HectorFullCfgPPO),
                            ("humanoid_config", "XBotLCfg", tasks.XBotLCfg), ("humanoid_config", "XBotLCfgPPO", tasks.XBotLCfgPPO)):
        ref = getattr(importlib.import_module(f"humanoid.envs.custom.{mod}"), name)()
        assert diff(class_to_dict(mine()), class_to_dict(ref)) == [], name


@needs_reference
@pytest.mark.parametrize("task", ["hector_full", "humanoid_ppo"])
def test_env_oracle_bit_equal_to_live_reference_other_tasks(task):
    """The other two registered tasks (hector_w_arm_env.py, humanoid_env.py) through the same oracle class: side by side
    with the unmodified reference env on one tape - 30 steps with falls, time-outs, command resampling and a push step."""
    from oracle.ref_harness import ReferenceEnv
    from isaac_b200.envs.tasks import TASKS
    from isaac_b200.synthetic import make_tape
    cfg_cls = TASKS[task][1]
    tape = make_tape(48, 30, seed=123, fall_prob=0.02, cfg=cfg_cls(), randomize_gains=True)
    tape.statics.episode_length0[:6] = torch.tensor([2398, 2400, 797, 799, 1599, 0])
    ref = ReferenceEnv(tape.statics, tape.physics[0], tape.noise[0], task=task)
    ora = OracleHectorEnv(cfg_cls(), tape.statics, tape.physics[0], tape.noise[0])
    ref.env.common_step_counter = ora.common_step_counter = 390
    assert torch.equal(ref.env.obs_buf, ora.obs_buf) and torch.equal(ref.env.privileged_obs_buf, ora.privileged_obs_buf)
    assert torch.equal(ref.env.noise_scale_vec, ora.noise_scale_vec)
    resets = 0
    for t in range(1, 30):
        a = ref.step(tape.physics[t], tape.noise[t])
        b = ora.step(tape.physics[t], tape.noise[t])
        for x, y, name in zip(a[:4], b[:4], ("obs", "priv", "rew", "reset")):
            assert torch.equal(x, y), f"{task}: {name} differs at step {t}"
        assert torch.equal(ref.env.episode_length_buf, ora.episode_length_buf) and torch.equal(ref.env.torques, ora.torques)
        for k in ora.episode_sums:
            assert torch.equal(ref.env.episode_sums[k], ora.episode_sums[k]), (k, t)
        assert torch.equal(ref.env.ref_dof_pos, ora.ref_dof_pos) and torch.equal(ref.root_states, ora.root_states)
        resets += int(b[3].sum())
    assert resets > 10 and set(ora.episode_sums) == set(ref.env.episode_sums)
    assert a[0].shape[1] == cfg_cls().env.num_observations and a[1].shape[1] == cfg_cls().env.num_privileged_obs


def rec_names():
    env_scales = {k: v for k, v in vars(type(HectorCfg().rewards.scales)).items() if not k.startswith("_") and v != 0}
    return list(env_scales)


def test_ppo_oracle_matches_reference_golden():
    g = np.load(f"{GOLDEN}/ppo_update_ref.npz")
    c = mg.PPO_CASE
    params = init_actor_critic_params(seed=c["param_seed"])
    steps, last, perm = mg.golden_ppo_inputs()
    for sched in ("fixed", "adaptive"):
        alg = OraclePPO(params, c["n"], c["t"], **dict(mg.PPO_ALG, schedule=sched))
        for obs, cobs, eps, rew, dones, tos in steps:
            alg.act(obs, cobs, eps)
            alg.process_env_step(rew, dones, {"time_outs": tos})
        alg.compute_returns(last)
        for k in ("actions", "values", "actions_log_prob", "mu", "sigma", "rewards", "returns", "advantages"):
            assert_close(f"storage.{k}", alg.st[k].numpy(), g["st/" + k], rtol=1e-5, atol=1e-6)
        assert_equal("storage.dones", alg.st["dones"].numpy(), g["st/dones"])
        losses = alg.update(perm)
        assert_close(f"{sched}/losses", np.array(losses), g[f"{sched}/losses"], rtol=1e-5, atol=1e-7)
        assert_close(f"{sched}/lr", np.array([alg.learning_rate]), g[f"{sched}/lr"], rtol=1e-12, atol=0)
        digest = mg.param_digest({k: v.detach() for k, v in alg.params.items()})
        for k, v in digest.items():
            want = g[f"{sched}/{k}"]
            if k.endswith("/sample"):
                # Post-update weights after 20 Adam steps.  Adam divides every gradient element by its own running
                # magnitude, and where a gradient sum cancels down to near Adam's eps (1e-8) the last-bit differences between
                # two fp32 BLAS builds (another CPU's kernels) move the weight by a few 1e-6 (measured on two x86 hosts: at
                # most 6.4e-6, and 0.29 % of a tensor's samples): up to 0.5 % of the samples may leave the tight tolerance,
                # none by more than 1e-5.
                off = np.abs(v - want) > 1e-7 + 1e-5 * np.abs(want)
                assert int(off.sum()) <= want.size // 200, f"{sched}/{k}: {int(off.sum())} of {want.size} beyond rtol 1e-5 / atol 1e-7"
                assert_close(f"{sched}/{k}", v, want, rtol=1e-5, atol=1e-5)
            else:
                # float64 sum, |sum| and sum of squares over the whole tensor: the signed sum cancels, and the independent
                # last-bit deviations of its N elements add up as sqrt(N)
                numel = alg.params[k.split("/")[1]].numel()
                assert_close(f"{sched}/{k}", v, want, rtol=1e-5, atol=1e-7 * np.sqrt(numel))


def test_quaternion_helpers_against_scipy():
    from scipy.spatial.transform import Rotation as R
    g = torch.Generator().manual_seed(0)
    q = torch.randn(512, 4, generator=g, dtype=torch.float64)
    q = q / q.norm(dim=-1, keepdim=True)
    v = torch.randn(512, 3, generator=g, dtype=torch.float64)
    rot = R.from_quat(q.numpy())                       # scipy is xyzw too
    np.testing.assert_allclose(quat_apply(q, v).numpy(), rot.apply(v.numpy()), atol=1e-12)
    np.testing.assert_allclose(quat_rotate_inverse(q, v).numpy(), rot.inv().apply(v.numpy()), atol=1e-12)
    e = euler_xyz_wrapped(q.float()).double().numpy()
    ref = rot.as_euler("xyz")                          # extrinsic xyz == roll/pitch/yaw of the reference helper
    d = np.abs(e - ref)
    d = np.minimum(d, 2 * np.pi - d)
    assert d.max() < 5e-6


@needs_reference
def test_env_oracle_bit_equal_to_live_reference():
    from oracle.ref_harness import ReferenceEnv
    from isaac_b200.synthetic import make_tape
    tape = make_tape(48, 30, seed=99, fall_prob=0.02)
    tape.statics.episode_length0[:6] = torch.tensor([2398, 2400, 797, 799, 1599, 0])
    ref = ReferenceEnv(tape.statics, tape.physics[0], tape.noise[0])
    ora = OracleHectorEnv(HectorCfg(), tape.statics, tape.physics[0], tape.noise[0])
    ref.env.common_step_counter = ora.common_step_counter = 390
    assert torch.equal(ref.env.obs_buf, ora.obs_buf) and torch.equal(ref.env.privileged_obs_buf, ora.privileged_obs_buf)
    resets = 0
    for t in range(1, 30):
        a = ref.step(tape.physics[t], tape.noise[t])
        b = ora.step(tape.physics[t], tape.noise[t])
        for x, y in zip(a[:4], b[:4]):
            assert torch.equal(x, y), f"step {t}"
        assert torch.equal(a[4]["time_outs"], b[4]["time_outs"])
        for k in a[4]["episode"]:
            assert torch.equal(a[4]["episode"][k], b[4]["episode"][k]), k
        for k in ora.episode_sums:
            assert torch.equal(ref.env.episode_sums[k], ora.episode_sums[k]), k
        assert torch.equal(ref.root_states, ora.root_states) and torch.equal(ref.dof_state, ora.dof_state)
        assert torch.equal(ref.env.reset_buf.nonzero().flatten(), ora.last_reset_ids)
        resets += int(a[3].sum())
    assert resets > 10


@needs_reference
def test_ppo_oracle_bit_equal_to_live_reference():
    from oracle.ref_harness import ReferencePPO
    c = mg.PPO_CASE
    params = init_actor_critic_params(seed=5)
    steps, last, perm = mg.golden_ppo_inputs()
    ref = ReferencePPO(params, c["n"], c["t"], mg.PPO_ALG, mg.PPO_POLICY)
    ora = OraclePPO(params, c["n"], c["t"], **mg.PPO_ALG)
    for obs, cobs, eps, rew, dones, tos in steps:
        assert torch.equal(ref.act(obs, cobs, eps), ora.act(obs, cobs, eps))
        ref.process_env_step(rew, dones, {"time_outs": tos})
        ora.process_env_step(rew, dones, {"time_outs": tos})
    ref.compute_returns(last)
    ora.compute_returns(last)
    for k in ora.st:
        assert torch.equal(getattr(ref.alg.storage, k), ora.st[k]), k
    assert ref.update(perm) == ora.update(perm)
    sd = ref.alg.actor_critic.state_dict()
    for k in PARAM_ORDER:
        assert torch.equal(sd[k], ora.params[k].detach()), k
