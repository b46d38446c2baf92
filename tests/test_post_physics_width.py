"""The eight-warp post-physics kernel (hb_set_option("post_warps", 8), chosen automatically for narrow shards) against the
four-warp kernel: the wide kernel splits each role's work by term, so every buffer a step writes must be bit-equal.

Each case runs the same steps twice from the same state on the device generator (no tape: reset, command, push and noise
draws all come from the kernels), once per width: time-outs and command resampling at steps 1 / 2, falls, a push step, a
full 32-env tile, a ragged last tile and a shard of 512 tiles."""
import pytest
import torch

from isaac_b200.synthetic import make_tape
from test_env_parity import make_cuda_env

KEY = 0x5EED0F00D
SPECIAL_EP0 = [2399, 2400, 798, 799, 1599]      # time-outs at steps 1 / 2, command resampling at steps 1 / 2
STEP_COUNTER0 = 396                             # common_step_counter: step 4 of the window is a push step
STEPS = 6

STATE = ["obs_buf", "privileged_obs_buf", "rew_buf", "reset_buf", "time_out_buf", "_episode_sums", "dof_state", "actions",
         "last_actions", "last_last_actions", "last_dof_vel", "last_root_vel", "root_states", "commands", "base_lin_vel",
         "base_ang_vel", "projected_gravity", "base_euler_xyz", "episode_length_buf", "feet_air_time", "feet_height",
         "last_feet_z", "last_contacts", "rand_push_force", "rand_push_torque", "ref_dof_pos", "_rng_state"]


def _task(name):
    """(config class, env class) of a built task, or of the runtime-layout robot xbot11 (11 joints, XBot-L kind)."""
    import isaac_b200.envs as envs
    from isaac_b200.envs import TASKS
    if name == "xbot11":
        from test_robot_layouts import new_cfg
        return new_cfg("xbot11"), envs.XBotLFreeEnvB200
    cls_name, cfg_cls, _ = TASKS[name]
    return cfg_cls, getattr(envs, cls_name)


def _snapshot(env, out):
    missing = [k for k in STATE if not isinstance(getattr(env, k, None), torch.Tensor)]
    assert not missing, f"env buffers not found: {missing}"
    snap = {k: getattr(env, k).clone() for k in STATE}
    snap["obs"], snap["priv"], snap["rew"], snap["reset"] = (x.clone() for x in out[:4])
    count = int(env._reset_count.item())
    snap["reset_count"] = count
    snap["reset_env_ids"] = env.reset_env_ids[:count].clone()
    if out[4].get("time_outs") is not None:
        snap["time_outs"] = out[4]["time_outs"].clone()
    for k, v in out[4]["episode"].items():
        snap[f"episode/{k}"] = v.clone()
    return snap


def _run(lib, dev, task, n, warps):
    assert lib.hb_set_option(b"post_warps", warps) == 0
    cfg_cls, cls = _task(task)
    cfg = cfg_cls()
    cfg.seed = KEY
    tape = make_tape(n, STEPS, seed=4000 + n, fall_prob=0.03, randomize_gains=True, cfg=cfg_cls())
    tape.statics.episode_length0[:len(SPECIAL_EP0)] = torch.tensor(SPECIAL_EP0)[:n]
    env, phys = make_cuda_env(tape, dev, cfg=cfg, cls=cls, device_rng=True)
    env.common_step_counter = STEP_COUNTER0
    snaps = [_snapshot(env, (env.obs_buf, env.privileged_obs_buf, env.rew_buf, env.reset_buf,
                             {"time_outs": env.time_out_buf, "episode": {}}))]
    for t in range(1, STEPS):
        phys.load_frame(tape.physics[t].to(dev))
        snaps.append(_snapshot(env, env.step(tape.noise[t].actions.to(dev))))
    torch.cuda.synchronize(dev)
    return snaps, phys.calls["set_root_state"]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [32, 4096 + 17, 16384])
@pytest.mark.parametrize("task", ["hector", "hector_full", "humanoid_ppo", "xbot11"])
def test_wide_kernel_is_bit_equal_to_four_warps(lib, cuda_device, task, n):
    try:
        four, pushes4 = _run(lib, cuda_device, task, n, 4)
        eight, pushes8 = _run(lib, cuda_device, task, n, 8)
    finally:
        lib.hb_set_option(b"post_warps", 0)
    assert pushes4 == pushes8 == 1, "the window has one push step"
    assert sum(s["reset_count"] for s in four[1:]) > 0, "the window has resets"
    for t, (a, b) in enumerate(zip(four, eight)):
        assert set(a) == set(b)
        for k in a:
            if isinstance(a[k], int):
                assert a[k] == b[k], f"step {t}: {k} {a[k]} != {b[k]}"
            else:
                assert torch.equal(a[k], b[k]), f"step {t}: {k} differs between 4 and 8 warps per tile"


def test_post_warps_accepts_0_4_8_only(lib):
    for v in (1, 2, 6, 16, -4):
        assert lib.hb_set_option(b"post_warps", v) == -1
    for v in (8, 4, 0):
        assert lib.hb_set_option(b"post_warps", v) == 0
