"""Robots other than the three the reference ships: any joint count up to 23 described by a `TaskLayout` in the config
(isaac_b200.envs.tasks), run by the post-physics kernel that reads the layout at run time and by the runtime-shape
frame-stack launch.

- CPU: the layout's own checks (each error names its field), the config's agreement with it, `layout_for`.
- GPU: the runtime kernel is bit-equal to the compiled kernel of each built robot (hb_set_option("env_runtime_task", 1));
  new robots of both kinds, even and odd joint counts, with and without arms, against the oracle at the suite's
  tolerances; device draws; graph replay, staged hooks, other stack depths and the host mirror against the eager step;
  the runner end to end; out-of-range layouts refused before any launch.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from _util import GOLDEN, assert_close, assert_equal
from isaac_b200._lib import HB_TASK_HECTOR, HB_TASK_XBOT
from isaac_b200.envs.hector_config import HectorCfg
from isaac_b200.envs.tasks import HECTOR, HECTOR_FULL, MAX_DOF, XBOT, TaskLayout, XBotLCfg, layout_for
from isaac_b200.synthetic import make_tape

HB_ERR_BAD_ARG, HB_ERR_UNSUPPORTED = -1, -3


def robot_layout(kind, ndof, arms=False, name=None):
    """A made-up robot: two legs (the left one takes the odd joint) and, with `arms`, a 4-joint arm after each leg."""
    arm = 4 if arms else 0
    nl = (ndof + 1) // 2
    leg_l, leg_r = nl - arm, ndof - nl - arm
    assert leg_l >= 3 and leg_r >= 3
    yaw = (0, nl)
    arm_pair = (leg_l, nl + leg_r) if arms else (-1, -1)
    n = ndof
    return TaskLayout(name or f"robot{ndof}{'_arms' if arms else ''}_{'xbot' if kind == HB_TASK_XBOT else 'hector'}", kind, ndof,
                      yaw, arm_pair, (leg_l - 3, leg_l - 2, leg_l - 1), (nl + leg_r - 3, nl + leg_r - 2, nl + leg_r - 1),
                      ((5, 5 + n), (5 + n, 5 + 2 * n), (5 + 2 * n, 5 + 3 * n), (5 + 3 * n, 8 + 3 * n), (8 + 3 * n, 11 + 3 * n)))


def robot_cfg(lay, frame_stack=15, c_frame_stack=None):
    """A config class for `lay` on the env file of its kind (hector_env.py: HectorCfg, humanoid_env.py: XBotLCfg)."""
    base = XBotLCfg if lay.kind == HB_TASK_XBOT else HectorCfg
    fs, cfs = frame_stack, c_frame_stack or base.env.c_frame_stack
    nl = (lay.ndof + 1) // 2
    names = [f"{'L' if j < nl else 'R'}_j{j}_joint" for j in range(lay.ndof)]

    class Cfg(base):
        layout = lay

        class env(base.env):
            num_actions = lay.ndof
            frame_stack, c_frame_stack = fs, cfs
            num_single_obs, single_num_privileged_obs = lay.num_single_obs, lay.num_single_priv
            num_observations, num_privileged_obs = fs * lay.num_single_obs, cfs * lay.num_single_priv

        class asset(base.asset):
            foot_name, knee_name = "toe", "calf"
            terminate_after_contacts_on = ["base", "thigh"]
            penalize_contacts_on = ["base", "thigh"]
            body_names = ["base"] + [f"{s}_{b}" for s in "LR" for b in ("hip", "thigh", "calf", "toe")]
            dof_names = names
            dof_effort = [40.0 + 5 * (j % 4) for j in range(lay.ndof)]

        class init_state(base.init_state):
            default_joint_angles = {nm: 0.1 * ((j % 5) - 2) for j, nm in enumerate(names)}

        class control(base.control):
            stiffness = {"_j": 60.0}
            damping = {"_j": 4.0}

    return Cfg


# XBot kind: 6, 11, 20, 23 DOF; hector kind: 8, 14, 22 (with arms)
NEW = {f"xbot{n}": (HB_TASK_XBOT, n, False) for n in (6, 11, 20, 23)}
NEW.update({"hector8": (HB_TASK_HECTOR, 8, False), "hector14": (HB_TASK_HECTOR, 14, False),
            "hector22_arms": (HB_TASK_HECTOR, 22, True)})


def new_cfg(key, **kw):
    kind, n, arms = NEW[key]
    return robot_cfg(robot_layout(kind, n, arms), **kw)


# ============================================================================================== CPU
@pytest.mark.parametrize("field,kw", [
    ("kind", dict(kind=7)),
    ("ndof", dict(ndof=24)),
    ("ndof", dict(ndof=0)),
    ("yaw_roll", dict(yaw_roll=(0, 11))),
    ("yaw_roll", dict(yaw_roll=(-1, 6))),
    ("arm_pair", dict(arm_pair=(3, -1))),
    ("arm_pair", dict(arm_pair=(3, 11))),
    ("ref_left", dict(ref_left=(2, 3, 12))),
    ("ref_right", dict(ref_right=(8, 9))),
    ("noise_slices", dict(noise_slices=((5, 17), (17, 29), (29, 41), (41, 44)))),
    ("noise_slices", dict(noise_slices=((5, 17), (17, 29), (29, 41), (41, 44), (47, 50)))),
    ("noise_slices", dict(noise_slices=((5, 17), (17, 29), (29, 41), (44, 41), (44, 47)))),
])
def test_invalid_layout_names_the_field(field, kw):
    args = dict(name="bad", kind=HB_TASK_XBOT, ndof=12, yaw_roll=(0, 6), arm_pair=(-1, -1), ref_left=(2, 3, 4),
                ref_right=(8, 9, 10), noise_slices=XBOT.noise_slices)
    TaskLayout(**args)                                   # the base case is valid
    args.update(kw)
    with pytest.raises(ValueError, match=rf"TaskLayout 'bad': {field} = "):
        TaskLayout(**args)


def test_built_layouts_and_new_robots_are_valid():
    assert MAX_DOF == 23
    for lay in (HECTOR, HECTOR_FULL, XBOT):
        TaskLayout(*(getattr(lay, f) for f in lay.__dataclass_fields__))
    for key in NEW:
        cfg_cls = new_cfg(key)
        assert cfg_cls.layout.num_single_obs <= 80 and layout_for(cfg_cls()) is cfg_cls.layout


def test_layout_for_recognises_the_built_robots():
    from isaac_b200.envs import TASKS
    assert layout_for(TASKS["hector"][1]()) is HECTOR
    assert layout_for(TASKS["hector_full"][1]()) is HECTOR_FULL
    assert layout_for(TASKS["humanoid_ppo"][1]()) is XBOT


def test_unknown_robot_without_layout_says_how_to_describe_it():
    cfg = new_cfg("hector14")()
    del type(cfg).layout
    with pytest.raises(ValueError, match=r"num_actions=14, frames 53 / 82 is none of the built robots.*cfg\.layout = TaskLayout\("):
        layout_for(cfg)


@pytest.mark.parametrize("field", ["env.num_actions", "env.num_single_obs", "env.single_num_privileged_obs", "asset.dof_names"])
def test_config_disagreeing_with_its_layout_names_the_field(field):
    cfg = new_cfg("xbot11")()
    sec, name = field.split(".")
    v = getattr(getattr(cfg, sec), name)
    setattr(getattr(cfg, sec), name, v[:-1] if isinstance(v, list) else v + 1)
    with pytest.raises(ValueError, match=rf"config field {field} = "):
        layout_for(cfg)


# ============================================================================================== GPU
def _oracle_case(dev, cfg_cls, n, steps, seed):
    """The CUDA env and the oracle on one tape (injected noise, time-outs and resampling at steps 1 / 2, a push step at the
    window's fourth or second step);
    compared like test_env_parity.py: masks, ids and counters bit-exact, everything else at rtol 1e-5 / atol 1e-6."""
    from oracle import make_golden as mg
    from oracle.hector_oracle import OracleHectorEnv
    from test_env_parity import compare_records, run_cuda_case
    step_counter0 = 396 if steps > 4 else 398
    tape = make_tape(n, steps, seed=seed, fall_prob=0.03, randomize_gains=True, cfg=cfg_cls())
    tape.statics.episode_length0[:5] = torch.tensor([2399, 2400, 798, 799, 1599])[:n]
    ora = OracleHectorEnv(cfg_cls(), tape.statics, tape.physics[0], tape.noise[0])
    ora.common_step_counter = step_counter0
    frames = (cfg_cls.env.num_single_obs, cfg_cls.env.single_num_privileged_obs)
    want = {"obs_init": ora.obs_buf.numpy().copy(), "priv_init": ora.privileged_obs_buf.numpy().copy()}
    want_ids, out = [], None
    for t in range(1, steps):
        out = ora.step(tape.physics[t], tape.noise[t])
        mg.record_env_step(want, ora, out, ora.root_states, ora.dof_state, frames)
        want_ids.append(ora.last_reset_ids.numpy().astype(np.int32))
    want = {k: (np.stack(v) if isinstance(v, list) else v) for k, v in want.items()}
    want["obs_final"], want["priv_final"] = out[0].numpy(), out[1].numpy()
    rec, ids, env, phys = run_cuda_case(tape, dev, step_counter0, cfg=cfg_cls())
    compare_records(rec, want)
    for t, (a, b) in enumerate(zip(ids, want_ids)):
        assert_equal(f"reset_env_ids@{t}", a, b)
    if layout_for(cfg_cls()).kind == HB_TASK_XBOT:
        assert_close("ref_dof_pos", env.ref_dof_pos.cpu().numpy(), ora.ref_dof_pos.numpy())
    assert phys.calls["set_root_state"] >= 1
    return rec, want_ids, tape, env


@pytest.mark.gpu
@pytest.mark.parametrize("task", ["hector", "hector_full", "humanoid_ppo", "action_delay"])
def test_runtime_kernel_is_bit_equal_to_the_compiled_kernel(lib, cuda_device, task):
    """env_runtime_task = 1 sends the built robots through the runtime-layout kernel: the reference goldens still pass at
    the suite's tolerances, and every recorded tensor (observations, rewards, episode sums, masks, ids, counters, extras)
    is bit-equal to the compiled kernel's on the same tape."""
    from oracle import make_golden as mg
    from isaac_b200.envs import TASKS
    import isaac_b200.envs as envs
    from test_env_parity import compare_records, run_cuda_case
    if task == "hector":
        g, tape, kw, c0 = f"{GOLDEN}/env_rollout_ref.npz", mg.env_golden_tape(), {}, mg.ENV_CASE["step_counter0"]
    elif task == "action_delay":
        g, tape, kw, c0 = f"{GOLDEN}/env_action_delay_ref.npz", mg.delay_golden_tape(), dict(cfg=mg.delay_cfg(HectorCfg())), 0
    else:
        cls_name, cfg_cls, _ = TASKS[task]
        g, tape = f"{GOLDEN}/env_rollout_{task}_ref.npz", mg.task_golden_tape(task)
        kw, c0 = dict(cfg=cfg_cls(), cls=getattr(envs, cls_name)), mg.TASK_CASE["step_counter0"]
    g = dict(np.load(g))
    runs = {}
    try:
        for rt in (0, 1):
            assert lib.hb_set_option(b"env_runtime_task", rt) == 0
            rec, ids, env, _ = run_cuda_case(tape, cuda_device, c0, **kw)
            runs[rt] = (rec, ids, env.common_step_counter, {k: v.cpu() for k, v in env.episode_sums.items()})
    finally:
        lib.hb_set_option(b"env_runtime_task", 0)
    rec = runs[1][0]
    if task == "action_delay":
        assert_equal("reset", rec["reset"], g["reset"])
        for k in ("actions", "torques", "obs_frame", "priv_frame", "rew", "last_actions", "last_last_actions"):
            assert_close(k, rec[k], g[k])
    else:
        compare_records(rec, g)
    assert set(runs[0][0]) == set(rec)
    for k in rec:
        assert_equal(f"runtime vs compiled: {k}", rec[k], runs[0][0][k])
    for t, (a, b) in enumerate(zip(runs[1][1], runs[0][1])):
        assert_equal(f"reset_env_ids@{t}", a, b)
    assert runs[1][2] == runs[0][2]
    for k, v in runs[0][3].items():
        assert torch.equal(runs[1][3][k], v), f"episode_sums[{k}]"


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(NEW))
@pytest.mark.parametrize("n,steps", [(64, 7), (4096, 4)])
def test_new_robot_matches_oracle(lib, cuda_device, key, n, steps):
    rec, ids, _, _ = _oracle_case(cuda_device, new_cfg(key), n, steps, seed=7000 + n + NEW[key][1])
    assert sum(len(i) for i in ids) > 0 and rec["time_outs"].sum() >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["xbot23", "hector22_arms"])
def test_new_robot_matches_oracle_at_65536(lib, cuda_device, key):
    _oracle_case(cuda_device, new_cfg(key), 65536, 3, seed=8000 + NEW[key][1])


@pytest.mark.gpu
def test_new_robot_device_draws_match_reference(lib, cuda_device, monkeypatch):
    """No tape at all: every draw from the device generator, against the oracle on oracle/device_rng.py's draws."""
    from isaac_b200.envs import TASKS
    from test_device_rng import _run_env_case
    monkeypatch.setitem(TASKS, "robot_hector14", ("HectorFreeEnvB200", new_cfg("hector14"), None))
    _run_env_case(cuda_device, "robot_hector14", 257, False)
    monkeypatch.setitem(TASKS, "robot_xbot11", ("XBotLFreeEnvB200", new_cfg("xbot11"), None))
    _run_env_case(cuda_device, "robot_xbot11", 257, True)


def _steps(env, phys, tape, dev, steps):
    outs = []
    for t in range(1, steps):
        phys.load_frame(tape.physics[t].to(dev))
        nz = tape.noise[t].to(dev)
        env.inject_noise(nz)
        o = env.step(nz.actions)
        outs.append(tuple(x.clone() for x in o[:4]))
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["hector14", "xbot11"])
def test_new_robot_same_results_on_every_path(lib, cuda_device, key):
    """Graph replay, the staged hooks (an overridden compute_reward) and the host mirror give what the eager fused step
    gives, bit for bit."""
    from isaac_b200.envs.hector_env import HectorFreeEnvB200
    from isaac_b200.envs.host_mirror import HostObservationMirror
    from test_env_parity import make_cuda_env
    dev, cfg_cls = cuda_device, new_cfg(key)
    tape = make_tape(256, 6, seed=11, fall_prob=0.1, cfg=cfg_cls())

    class Staged(HectorFreeEnvB200):
        def compute_reward(self):
            super().compute_reward()

    eager, pe = make_cuda_env(tape, dev, cfg=cfg_cls())
    staged, ps = make_cuda_env(tape, dev, cfg=cfg_cls(), cls=Staged)
    want, got = _steps(eager, pe, tape, dev, 6), _steps(staged, ps, tape, dev, 6)
    for t, (a, b) in enumerate(zip(want, got)):
        for x, y, nm in zip(a, b, ("obs", "priv", "rew", "reset")):
            assert torch.equal(x, y), f"staged hooks vs fused: {nm} at step {t}"
    assert sum(int(w[3].sum()) for w in want) > 0
    # device generator: graph replay == eager, and the host mirror's views == the device tensors
    env_g, phys_g = make_cuda_env(tape, dev, cfg=cfg_cls())
    env_e, phys_e = make_cuda_env(tape, dev, cfg=cfg_cls())
    env_g.seed(4), env_e.seed(4)
    env_g.enable_cuda_graph()
    mirror = HostObservationMirror(env_e)
    resets = 0
    for t in range(1, 6):
        fr = tape.physics[t].to(dev)
        phys_g.load_frame(fr), phys_e.load_frame(fr)
        a = tape.noise[t].actions.to(dev)
        og, oe = env_g.step(a), env_e.step(a)
        for x, y, nm in zip(og[:4], oe[:4], ("obs", "priv", "rew", "reset")):
            assert torch.equal(x, y), f"graph replay vs eager: {nm} at step {t}"
        ho, hp = mirror.views(mirror.update(oe[0], oe[1]))
        assert torch.equal(ho, oe[0].cpu()) and torch.equal(hp, oe[1].cpu()), f"host mirror at step {t}"
        resets += int(oe[3].sum())
    assert resets > 0


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [1, 4, 15])
@pytest.mark.parametrize("robot", ["hector", "hector14", "xbot11"])
def test_stack_depths_through_the_runtime_shift(lib, cuda_device, robot, depth):
    """frame_stack = c_frame_stack = 1, 4, 15 (no compiled shape but the built robots' 15 / 15 and 15 / 3): against the
    oracle, and every step's carried frames are an exact copy of the previous stack shifted by one frame, zero for the
    envs just reset - what the scalar shift produced for these shapes."""
    dev = cuda_device
    if robot == "hector":
        class cfg_cls(HectorCfg):
            class env(HectorCfg.env):
                frame_stack = c_frame_stack = depth
                num_observations, num_privileged_obs = depth * 41, depth * 70
    else:
        cfg_cls = new_cfg(robot, frame_stack=depth, c_frame_stack=depth)
    _oracle_case(dev, cfg_cls, 257, 5, seed=900 + depth)
    from test_env_parity import make_cuda_env
    tape = make_tape(257, 5, seed=901 + depth, fall_prob=0.1, cfg=cfg_cls())
    env, phys = make_cuda_env(tape, dev, cfg=cfg_cls())
    fo, fp = cfg_cls.env.num_single_obs, cfg_cls.env.single_num_privileged_obs
    prev = (env.get_observations().clone(), env.get_privileged_observations().clone())
    for t in range(1, 5):
        phys.load_frame(tape.physics[t].to(dev))
        nz = tape.noise[t].to(dev)
        env.inject_noise(nz)
        obs, priv, _, reset, _ = env.step(nz.actions)
        for new, old, f in ((obs, prev[0], fo), (priv, prev[1], fp)):
            assert new.shape[1] == depth * f
            want = torch.where(reset[:, None], torch.zeros_like(old[:, f:]), old[:, f:])
            assert torch.equal(new[:, :new.shape[1] - f], want), f"carried frames at step {t}"
        prev = (obs.clone(), priv.clone())


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["xbot11", "hector22_arms"])
def test_runner_learns_on_a_new_robot(lib, cuda_device, tmp_path, key):
    """OnPolicyRunner over a new robot's env: 11 actions (the fused act and loss heads) and 22 (the generic heads)."""
    from isaac_b200.algo import OnPolicyRunner
    from test_env_parity import make_cuda_env
    from test_runner import TRAIN_CFG
    cfg_cls = new_cfg(key)

    def env_():
        env, _ = make_cuda_env(make_tape(256, 2, seed=31, fall_prob=0.02, cfg=cfg_cls()), cuda_device, cfg=cfg_cls())
        env.seed(3)
        return env

    env = env_()
    runner = OnPolicyRunner(env, TRAIN_CFG, log_dir=str(tmp_path), device=str(cuda_device))
    assert runner.alg.__dict__.get("_env") is env, "attach_env: the observations go straight into the rollout slots"
    w0 = runner.alg.actor_critic.flat.clone()
    runner.learn(num_learning_iterations=3, init_at_random_ep_len=True)
    assert not torch.equal(w0, runner.alg.actor_critic.flat) and torch.isfinite(runner.alg.actor_critic.flat).all()
    assert sorted(p for p in (tmp_path).iterdir() if p.suffix == ".pt")[-1].name == "model_3.pt"
    runner2 = OnPolicyRunner(env_(), TRAIN_CFG, log_dir=None, device=str(cuda_device))
    runner2.load(str(tmp_path / "model_3.pt"))
    assert torch.equal(runner2.alg.actor_critic.flat, runner.alg.actor_critic.flat)
    policy = runner2.get_inference_policy(device=str(cuda_device))
    assert policy(env.get_observations()).shape == (env.num_envs, NEW[key][1])


@pytest.mark.gpu
def test_out_of_range_layouts_are_refused(lib, cuda_device):
    """24 joints (frame 83) is HB_ERR_UNSUPPORTED, inconsistent frames or joint indices HB_ERR_BAD_ARG, each with the
    allowed range in hb_last_error(); nothing is launched."""
    from isaac_b200 import _lib
    from test_env_parity import make_cuda_env
    cfg_cls = new_cfg("xbot23")
    env, _ = make_cuda_env(make_tape(64, 2, seed=1, cfg=cfg_cls()), cuda_device, cfg=cfg_cls())
    nz = _lib.EnvNoise()
    nz.rng_counter = env._rng_state.data_ptr()
    o, p_ = env.get_observations(), env.get_privileged_observations()
    st = torch.cuda.current_stream(cuda_device).cuda_stream

    def call(**kw):
        p = _lib.EnvParams.from_buffer_copy(env._p)
        p.obs_ld = p.priv_ld = 0                     # dense rows: the row-pitch check passes for any frame size
        for k, v in kw.items():
            if isinstance(v, tuple):
                getattr(p, k)[:] = v
            else:
                setattr(p, k, v)
        n0 = lib.hb_launch_count()
        rc = lib.hb_env_post_physics(C.byref(p), env._pb, C.byref(nz), o.data_ptr(), p_.data_ptr(), _lib.HB_STAGE_STEP, st)
        assert lib.hb_launch_count() == n0
        return rc, lib.hb_last_error().decode()

    rc, msg = call(num_dof=24, num_single_obs=83, num_single_priv=121)
    assert rc == HB_ERR_UNSUPPORTED and "1 to 23 joints" in msg, msg
    rc, msg = call(num_single_obs=81)
    assert rc == HB_ERR_BAD_ARG and "3 num_dof + 11" in msg, msg
    rc, msg = call(yaw_roll=(0, 22))
    assert rc == HB_ERR_BAD_ARG and "yaw_roll" in msg and "j + 1 < num_dof=23" in msg, msg
    rc, msg = call(arm_pair=(4, -1))
    assert rc == HB_ERR_BAD_ARG and "arm_pair" in msg, msg
    rc, msg = call(ref_right=(20, 21, 23))
    assert rc == HB_ERR_BAD_ARG and "ref_left / ref_right" in msg, msg
    torch.cuda.synchronize()
