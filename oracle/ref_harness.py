"""TEST INFRASTRUCTURE.

Runs the UNMODIFIED reference (`humanoid/...`) on the CPU so that
(a) the oracle restatement in `oracle/hector_oracle.py` can be pinned against it,
(b) golden vectors can be generated for `tests/golden/` (see `oracle/make_golden.py`) and
(c) `bench.py --impl reference` can time the reference's own code on the host cores.

The reference is imported from a checkout of DRCL-USC/isaac: the one `$ISAAC_REFERENCE` names,
else `/root/reference` (its default location), else the copy that `baseline/install_ref.sh`
installed under `baseline/_ref` (git-ignored).  No reference source is part of this
repository's history.  `reference_root()` is None when none of them exists.

How (SURVEY.md §8c): the reference needs the closed third-party `isaacgym` package.
We register stub modules for it — `isaacgym.torch_utils` is a restatement of the
well-known public definitions of the 7 helpers the hot path calls — build
`HectorFreeEnv` with `__new__` (skipping `create_sim`, which needs the simulator),
seed the attributes `_create_envs` would have produced, and then call the reference's
own `_parse_cfg / _init_buffers / _prepare_reward_function / reset_idx / step`.

Random draws are injected: `torch.rand`, `torch.randn_like` and `torch_rand_float`
are patched to replay env-indexed tapes (`isaac_b200.synthetic.NoiseFrame`), which is
the contract the CUDA path implements ("noise injected as a supplied tensor").
"""
from __future__ import annotations

import contextlib
import math
import sys
import types
from unittest.mock import MagicMock

import numpy as np
import torch

import os

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _is_reference(root):
    return bool(root) and os.path.isfile(os.path.join(root, "humanoid", "envs", "custom", "hector_env.py"))


def reference_source():
    """The upstream checkout given by $ISAAC_REFERENCE, else the default location; None when neither holds it."""
    for root in (os.environ.get("ISAAC_REFERENCE"), "/root/reference"):
        if _is_reference(root):
            return root
    return None


def reference_root():
    """Where `humanoid` is imported from: the upstream checkout, else its copy under baseline/_ref."""
    for root in (reference_source(), os.path.join(_REPO, "baseline", "_ref")):
        if _is_reference(root):
            return root
    return None


REFERENCE_ROOT = reference_root()


# --------------------------------------------------------------------------------------
# isaacgym.torch_utils restatement (public definitions; SURVEY.md §8c "parity unpinned"
# for these helpers: Isaac Gym preview4 is not in the image, cross-checked against scipy
# in tests/test_oracle_pinning.py)
# --------------------------------------------------------------------------------------
def _quat_rotate_inverse(q, v):
    shape = q.shape
    q_w = q[:, -1]
    q_vec = q[:, :3]
    a = v * (2.0 * q_w ** 2 - 1.0).unsqueeze(-1)
    b = torch.cross(q_vec, v, dim=-1) * q_w.unsqueeze(-1) * 2.0
    c = q_vec * torch.bmm(q_vec.view(shape[0], 1, 3), v.view(shape[0], 3, 1)).squeeze(-1) * 2.0
    return a - b + c


def _quat_apply(a, b):
    shape = b.shape
    a = a.reshape(-1, 4)
    b = b.reshape(-1, 3)
    xyz = a[:, :3]
    t = xyz.cross(b, dim=-1) * 2
    return (b + a[:, 3:] * t + xyz.cross(t, dim=-1)).view(shape)


def _copysign(a, b):
    a = torch.tensor(a, device=b.device, dtype=torch.float).repeat(b.shape[0])
    return torch.abs(a) * torch.sign(b)


def _get_euler_xyz(q):
    qx, qy, qz, qw = 0, 1, 2, 3
    sinr_cosp = 2.0 * (q[:, qw] * q[:, qx] + q[:, qy] * q[:, qz])
    cosr_cosp = q[:, qw] * q[:, qw] - q[:, qx] * q[:, qx] - q[:, qy] * q[:, qy] + q[:, qz] * q[:, qz]
    roll = torch.atan2(sinr_cosp, cosr_cosp)
    sinp = 2.0 * (q[:, qw] * q[:, qy] - q[:, qz] * q[:, qx])
    pitch = torch.where(torch.abs(sinp) >= 1, _copysign(np.pi / 2.0, sinp), torch.asin(sinp))
    siny_cosp = 2.0 * (q[:, qw] * q[:, qz] + q[:, qx] * q[:, qy])
    cosy_cosp = q[:, qw] * q[:, qw] + q[:, qx] * q[:, qx] - q[:, qy] * q[:, qy] - q[:, qz] * q[:, qz]
    yaw = torch.atan2(siny_cosp, cosy_cosp)
    return roll % (2 * np.pi), pitch % (2 * np.pi), yaw % (2 * np.pi)


def _torch_rand_float(lower, upper, shape, device):
    return (upper - lower) * torch.rand(*shape, device=device) + lower


def _to_torch(x, dtype=torch.float, device="cpu", requires_grad=False):
    return torch.tensor(x, dtype=dtype, device=device, requires_grad=requires_grad)


def _get_axis_params(value, axis_idx, x_value=0.0, dtype=float, n_dims=3):
    zs = np.zeros((n_dims,))
    zs[axis_idx] = 1.0
    params = np.where(zs == 1.0, value, zs)
    params[0] = x_value
    return list(params.astype(dtype))


def _normalize(x, eps: float = 1e-9):
    return x / x.norm(p=2, dim=-1).clamp(min=eps, max=None).unsqueeze(-1)


def install_isaacgym_stub():
    if REFERENCE_ROOT is None:
        raise ImportError("the reference is not found: set ISAAC_REFERENCE to a checkout of DRCL-USC/isaac "
                          "or install one with baseline/install_ref.sh")
    if "isaacgym" in sys.modules:
        return
    tu = types.ModuleType("isaacgym.torch_utils")
    tu.quat_rotate_inverse = _quat_rotate_inverse
    tu.quat_apply = _quat_apply
    tu.get_euler_xyz = _get_euler_xyz
    tu.torch_rand_float = _torch_rand_float
    tu.to_torch = _to_torch
    tu.get_axis_params = _get_axis_params
    tu.normalize = _normalize
    tu.__all__ = ["quat_rotate_inverse", "quat_apply", "get_euler_xyz", "torch_rand_float",
                  "to_torch", "get_axis_params", "normalize"]
    gymtorch = types.ModuleType("isaacgym.gymtorch")
    gymtorch.wrap_tensor = lambda t: t
    gymtorch.unwrap_tensor = lambda t: t
    pkg = types.ModuleType("isaacgym")
    pkg.torch_utils, pkg.gymtorch = tu, gymtorch
    for name in ("gymapi", "gymutil", "terrain_utils"):
        m = MagicMock(name=f"isaacgym.{name}")
        setattr(pkg, name, m)
        sys.modules[f"isaacgym.{name}"] = m
    sys.modules["isaacgym"] = pkg
    sys.modules["isaacgym.torch_utils"] = tu
    sys.modules["isaacgym.gymtorch"] = gymtorch
    for name in ("matplotlib", "matplotlib.pyplot"):   # utils/logger.py:32 imports pyplot
        try:
            __import__(name)
        except ImportError:
            sys.modules[name] = MagicMock(name=name)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


# --------------------------------------------------------------------------------------
# Reference env built on synthetic gym tensors
# --------------------------------------------------------------------------------------
DOF_NAMES = ["L_hip_joint", "L_hip_roll_joint", "L_thigh_joint", "L_calf_joint", "L_toe_joint",
             "R_hip_joint", "R_hip_roll_joint", "R_thigh_joint", "R_calf_joint", "R_toe_joint"]
EFFORT = [33.5, 33.5, 33.5, 67.0, 33.5] * 2     # robot.urdf:124,166,217,291,320


class ReferenceEnv:
    """The reference HectorFreeEnv, stepping on supplied physics frames and noise tapes."""

    # task -> (env module, env class, config module, config class): what envs/__init__.py:46-48 registers
    TASKS = {"hector": ("hector_env", "HectorFreeEnv", "hector_config", "HectorCfg"),
             "hector_full": ("hector_w_arm_env", "HectorFullFreeEnv", "hector_w_arm_config", "HectorFullCfg"),
             "humanoid_ppo": ("humanoid_env", "XBotLFreeEnv", "humanoid_config", "XBotLCfg")}

    def __init__(self, statics, first_frame, first_noise, configure=None, task="hector"):
        """`configure(cfg)`: optional edits of the reference's config before the env parses it (e.g. a non-zero
        `domain_rand.action_delay`).  `task`: which of the reference's registered envs to build; the robot description
        (body / joint names, effort limits) that `_create_envs` would read from the URDF comes from this repo's config of
        the same task (isaac_b200.envs.tasks)."""
        install_isaacgym_stub()
        import importlib
        env_mod, env_cls, cfg_mod, cfg_cls = self.TASKS[task]
        he_mod = importlib.import_module(f"humanoid.envs.custom.{env_mod}")
        HectorFreeEnv = getattr(he_mod, env_cls)
        HectorCfg = getattr(importlib.import_module(f"humanoid.envs.custom.{cfg_mod}"), cfg_cls)
        import humanoid.envs.base.legged_robot as lr_mod
        self._mods = (lr_mod, he_mod)
        from isaac_b200.envs.tasks import TASKS as OUR_TASKS
        from isaac_b200.synthetic import task_dims
        asset = OUR_TASKS[task][1]().asset
        dims = task_dims(OUR_TASKS[task][1]())

        n = statics.p_gains.shape[0]
        e = HectorFreeEnv.__new__(HectorFreeEnv)
        cfg = HectorCfg()
        cfg.env.num_envs = n
        if configure is not None:
            configure(cfg)
        e.cfg = cfg
        e.sim_params = types.SimpleNamespace(dt=cfg.sim.dt)
        e.height_samples = None
        e.debug_viz = False
        e.init_done = False
        e._parse_cfg(cfg)
        # --- what BaseTask.__init__ allocates (base_task.py:43-92) ---
        e.gym = MagicMock(name="gym")
        e.sim = MagicMock(name="sim")
        e.device = "cpu"
        e.headless = True
        e.viewer = None
        e.num_envs = n
        e.num_obs = cfg.env.num_observations
        e.num_privileged_obs = cfg.env.num_privileged_obs
        e.num_actions = cfg.env.num_actions
        e.obs_buf = torch.zeros(n, e.num_obs)
        e.rew_buf = torch.zeros(n)
        e.reset_buf = torch.ones(n, dtype=torch.long)
        e.episode_length_buf = torch.zeros(n, dtype=torch.long)
        e.time_out_buf = torch.zeros(n, dtype=torch.bool)
        e.privileged_obs_buf = torch.zeros(n, e.num_privileged_obs)
        e.extras = {}
        # --- what create_sim/_create_envs produce (hector_env.py:114-132, legged_robot.py:587-681) ---
        e.up_axis_idx = 2
        e.num_dof = e.num_dofs = dims.ndof
        e.num_bodies = dims.nbody
        e.dof_names = list(asset.dof_names)
        find = lambda pats: [i for p in pats for i, nm in enumerate(asset.body_names) if p in nm]      # legged_robot.py:627-634
        e.feet_indices = torch.tensor(find([cfg.asset.foot_name]), dtype=torch.long)
        e.knee_indices = torch.tensor(find([cfg.asset.knee_name]), dtype=torch.long)
        e.penalised_contact_indices = torch.tensor(find(cfg.asset.penalize_contacts_on), dtype=torch.long)
        e.termination_contact_indices = torch.tensor(find(cfg.asset.terminate_after_contacts_on), dtype=torch.long)
        e.torque_limits = torch.tensor(asset.dof_effort) * cfg.safety.torque_limit
        e.env_frictions = statics.env_frictions.clone()
        e.body_mass = statics.body_mass.clone()
        e.custom_origins = cfg.terrain.mesh_type in ("heightfield", "trimesh")      # legged_robot.py:687-688
        e.env_origins = statics.env_origins.clone()
        e.terrain_levels = torch.zeros(n, dtype=torch.long)
        base_init = cfg.init_state.pos + cfg.init_state.rot + cfg.init_state.lin_vel + cfg.init_state.ang_vel
        e.base_init_state = torch.tensor(base_init, dtype=torch.float)
        # --- gym tensors ---
        self.root_states = first_frame.root_states.clone()
        self.dof_state = first_frame.dof_state.clone()
        self.contact_forces = first_frame.contact_forces.clone()
        self.rigid_state = first_frame.rigid_state.clone()
        e.gym.acquire_actor_root_state_tensor.return_value = self.root_states
        e.gym.acquire_dof_state_tensor.return_value = self.dof_state
        e.gym.acquire_net_contact_force_tensor.return_value = self.contact_forces.view(-1, 3)
        e.gym.acquire_rigid_body_state_tensor.return_value = self.rigid_state.view(-1, 13)
        e._init_buffers()
        e.p_gains[:] = statics.p_gains       # constants by default; randomised for BASELINE config 3
        e.d_gains[:] = statics.d_gains
        e._prepare_reward_function()
        e.init_done = True
        self.env = e
        self._noise = first_noise
        self._ctx = None
        self._install_rng_patches()
        # HectorFreeEnv.__init__ tail (hector_env.py:48-51)
        e.last_feet_z = 0.05
        e.feet_height = torch.zeros((n, 2))
        e.reset_idx(torch.tensor(range(n)))
        with self._patched_torch_rng(first_noise):
            e.compute_observations()
        e.episode_length_buf[:] = statics.episode_length0   # on_policy_runner.py:103-106

    # -- RNG injection -----------------------------------------------------------------
    def _install_rng_patches(self):
        e = self.env
        harness = self

        def tape_rand_float(lower, upper, shape, device):
            kind, ids, col = harness._ctx
            u = getattr(harness._noise, kind)[ids, col:col + shape[1]]
            assert u.shape == tuple(shape), (u.shape, shape, kind)
            harness._ctx = (kind, ids, col + shape[1])
            return (upper - lower) * u + lower

        for mod in self._mods:
            mod.torch_rand_float = tape_rand_float

        orig_resample = e._resample_commands
        orig_reset_dofs = e._reset_dofs
        orig_reset_root = e._reset_root_states
        orig_push = e._push_robots

        def resample(env_ids):
            if harness._ctx is None:            # called from _post_physics_step_callback
                harness._ctx = ("u_cmd", env_ids, 0)
                orig_resample(env_ids)
                harness._ctx = None
            else:                               # called from reset_idx: the command draws sit behind the dof and xy draws
                harness._ctx = ("u_reset", env_ids, e.num_dof + 2)      # (also when the xy jitter was not drawn: mesh 'plane')
                orig_resample(env_ids)

        def reset_dofs(env_ids):
            harness._ctx = ("u_reset", env_ids, 0)
            orig_reset_dofs(env_ids)

        def reset_root(env_ids):
            orig_reset_root(env_ids)

        def push():
            harness._ctx = ("u_push", torch.arange(e.num_envs), 0)
            orig_push()
            harness._ctx = None

        e._resample_commands = resample
        e._reset_dofs = reset_dofs
        e._reset_root_states = reset_root
        e._push_robots = push
        orig_reset_idx = type(e).reset_idx

        def reset_idx(env_ids):
            orig_reset_idx(e, env_ids)
            harness._ctx = None
        e.reset_idx = reset_idx

    def step(self, frame, noise):
        """One reference `step()` on the given physics frame with the given draws."""
        self._noise = noise
        self.root_states.copy_(frame.root_states)
        self.dof_state.copy_(frame.dof_state)
        self.contact_forces.copy_(frame.contact_forces)
        self.rigid_state.copy_(frame.rigid_state)
        with self._patched_torch_rng(noise):
            return self.env.step(noise.actions.clone())

    @staticmethod
    @contextlib.contextmanager
    def _patched_torch_rng(noise):
        """Replay `torch.rand` (action delay) and `torch.randn_like` (action / obs noise)."""
        real_rand, real_randn_like = torch.rand, torch.randn_like

        def fake_rand(*shape, **kw):
            assert tuple(shape[0]) == tuple(noise.u_delay.shape), shape
            return noise.u_delay.clone()

        def fake_randn_like(t, **kw):
            if t.shape == noise.z_action.shape:
                return noise.z_action.clone()
            assert t.shape == noise.z_obs.shape, t.shape
            return noise.z_obs.clone()

        torch.rand, torch.randn_like = fake_rand, fake_randn_like
        try:
            yield
        finally:
            torch.rand, torch.randn_like = real_rand, real_randn_like


# --------------------------------------------------------------------------------------
# Reference PPO (rsl_rl fork) with injected draws
# --------------------------------------------------------------------------------------
class ReferencePPO:
    """The reference `PPO` + `ActorCritic` + `RolloutStorage`, unmodified, on CPU.
    `torch.normal` (the Normal.sample() draw, actor_critic.py:115-117) and `torch.randperm`
    (rollout_storage.py:149) are replayed from supplied tensors."""

    def __init__(self, params, num_envs, num_steps, alg_cfg, policy_cfg):
        install_isaacgym_stub()
        from humanoid.algo import PPO, ActorCritic
        nobs = params["actor.0.weight"].shape[1]
        npriv = params["critic.0.weight"].shape[1]
        nact = params["std"].shape[0]
        ac = ActorCritic(nobs, npriv, nact, **policy_cfg)
        ac.load_state_dict({k: v.clone() for k, v in params.items()})
        self.alg = PPO(ac, device="cpu", **alg_cfg)
        self.alg.init_storage(num_envs, num_steps, [nobs], [npriv], [nact])
        self._eps = None
        self._perm = None

    @contextlib.contextmanager
    def _patched(self):
        real_normal, real_randperm = torch.normal, torch.randperm
        h = self

        def fake_normal(mean, std, **kw):
            eps = h._eps if (h._eps is not None and h._eps.shape == mean.shape) else torch.zeros_like(mean)
            return mean + std * eps

        def fake_randperm(n, **kw):
            assert h._perm is not None and h._perm.numel() == n
            return h._perm.clone()

        torch.normal, torch.randperm = fake_normal, fake_randperm
        try:
            yield
        finally:
            torch.normal, torch.randperm = real_normal, real_randperm

    def act(self, obs, critic_obs, eps):
        self._eps = eps
        with self._patched(), torch.inference_mode():
            return self.alg.act(obs, critic_obs)

    def process_env_step(self, rewards, dones, infos):
        with torch.inference_mode():
            self.alg.process_env_step(rewards, dones, infos)

    def compute_returns(self, last_critic_obs):
        with torch.inference_mode():
            self.alg.compute_returns(last_critic_obs)

    def update(self, perm):
        """Also records `lr_trace`: the learning rate of every optimizer step (read from the param group at the moment
        the reference calls `optimizer.step()`), which pins the adaptive-KL schedule step by step."""
        self._perm, self._eps = perm, None
        self.lr_trace = []
        opt = self.alg.optimizer
        real_step = opt.step

        def step(*a, **kw):
            self.lr_trace.append(float(opt.param_groups[0]["lr"]))
            return real_step(*a, **kw)

        opt.step = step
        try:
            with self._patched():
                return self.alg.update()
        finally:
            opt.step = real_step


# --------------------------------------------------------------------------------------
# Reference terrain height sampling (legged_robot.py:744-795), called unbound on a stub
# --------------------------------------------------------------------------------------
def reference_get_heights(root_states, height_samples, measured_points_x, measured_points_y, border_size, horizontal_scale,
                          vertical_scale, env_ids=None):
    """The reference's own `LeggedRobot._init_height_points` + `_get_heights` on the given state and int16 height field."""
    install_isaacgym_stub()
    from humanoid.envs.base.legged_robot import LeggedRobot
    tcfg = types.SimpleNamespace(mesh_type="trimesh", measured_points_x=measured_points_x, measured_points_y=measured_points_y,
                                 border_size=border_size, horizontal_scale=horizontal_scale, vertical_scale=vertical_scale)
    stub = types.SimpleNamespace(cfg=types.SimpleNamespace(terrain=tcfg), terrain=types.SimpleNamespace(cfg=tcfg), device="cpu",
                                 num_envs=root_states.shape[0], root_states=root_states, base_quat=root_states[:, 3:7],
                                 height_samples=height_samples)
    stub.height_points = LeggedRobot._init_height_points(stub)
    return LeggedRobot._get_heights(stub, env_ids)
