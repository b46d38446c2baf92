"""TEST INFRASTRUCTURE — CPU oracle for the hector env stage (not a product path).

A torch-on-CPU restatement of the reference's per-environment hot path:
PD torque law, action prologue, derived base quantities, heading command,
termination, the 18 active reward terms, reset bookkeeping, frame-stacked
observations and the `last_*` copies.  Each function cites the reference lines it
follows (paths relative to humanoid/ in DRCL-USC/isaac).

Pinning: `tests/test_oracle_pinning.py` checks this file against golden vectors that
`oracle/make_golden.py` produced by running the UNMODIFIED reference
(`oracle/ref_harness.py`); where the reference is found, the same test also steps it
live, side by side, and demands bit equality.  The quaternion helpers come
from the closed third-party `isaacgym.torch_utils` (setup.py:43, `isaacgym # preview4`,
absent from the reference checkout): they are restated from the public definitions and have
no reference-side test → *parity unpinned* for those three helpers; they are
cross-checked against scipy instead.

Only `tests/`, `__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference`
legs of `bench.py` may import this module.

All random draws are injected, indexed by env (see `isaac_b200.synthetic.NoiseFrame`).
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch

REWARD_FORMULAS = {}


def _reward(name):
    def deco(fn):
        REWARD_FORMULAS[name] = fn
        return fn
    return deco


# ----------------------------------------------------------------------------- helpers
def quat_rotate_inverse(q: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """isaacgym.torch_utils.quat_rotate_inverse (q = xyzw): a - b + c form (SURVEY.md §8c)."""
    w = q[:, 3]
    u = q[:, :3]
    a = v * (2.0 * w ** 2 - 1.0).unsqueeze(-1)
    b = torch.cross(u, v, dim=-1) * w.unsqueeze(-1) * 2.0
    c = u * torch.bmm(u.view(-1, 1, 3), v.view(-1, 3, 1)).squeeze(-1) * 2.0
    return a - b + c


def quat_apply(q: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """isaacgym.torch_utils.quat_apply: t = 2 (u x v); v + w t + u x t."""
    u = q[:, :3]
    t = u.cross(v, dim=-1) * 2
    return v + q[:, 3:] * t + u.cross(t, dim=-1)


def euler_xyz_wrapped(q: torch.Tensor) -> torch.Tensor:
    """get_euler_xyz_tensor, envs/base/legged_robot.py:50-55 on top of
    isaacgym.torch_utils.get_euler_xyz: angles mod 2pi, then (pi, 2pi) -> (-pi, 0)."""
    x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    roll = torch.atan2(2.0 * (w * x + y * z), w * w - x * x - y * y + z * z)
    sinp = 2.0 * (w * y - z * x)
    half_pi = torch.tensor(np.pi / 2.0, dtype=torch.float).repeat(q.shape[0])
    pitch = torch.where(torch.abs(sinp) >= 1, torch.abs(half_pi) * torch.sign(sinp), torch.asin(sinp))
    yaw = torch.atan2(2.0 * (w * z + x * y), w * w + x * x - y * y - z * z)
    e = torch.stack((roll % (2 * np.pi), pitch % (2 * np.pi), yaw % (2 * np.pi)), dim=1)
    e[e > np.pi] -= 2 * np.pi
    return e


def wrap_to_pi(a: torch.Tensor) -> torch.Tensor:
    """utils/math.py:46-49."""
    a = a % (2 * np.pi)
    return a - 2 * np.pi * (a > np.pi)


def height_points(measured_points_x, measured_points_y, num_envs: int) -> torch.Tensor:
    """LeggedRobot._init_height_points (legged_robot.py:744-757): the sampling grid in the base frame, [N, P, 3]."""
    y = torch.tensor(measured_points_y)
    x = torch.tensor(measured_points_x)
    grid_x, grid_y = torch.meshgrid(x, y, indexing="ij")
    points = torch.zeros(num_envs, grid_x.numel(), 3)
    points[:, :, 0] = grid_x.flatten()
    points[:, :, 1] = grid_y.flatten()
    return points


def get_heights(root_states, points, height_samples, border_size, horizontal_scale, vertical_scale, env_ids=None):
    """LeggedRobot._get_heights (legged_robot.py:759-795) with quat_apply_yaw (utils/math.py:39-43): terrain height under
    each point, min over the cell and its +x / +y neighbours of the int16 field."""
    if env_ids is not None:
        root_states, points = root_states[env_ids], points[env_ids]
    n, p = points.shape[:2]
    quat = root_states[:, 3:7].repeat(1, p).clone().view(-1, 4)
    quat[:, :2] = 0.0
    quat = quat / quat.norm(p=2, dim=-1).clamp(min=1e-9).unsqueeze(-1)          # isaacgym.torch_utils.normalize
    pts = quat_apply(quat, points.reshape(-1, 3)).view(n, p, 3) + root_states[:, :3].unsqueeze(1)
    pts = pts + border_size
    pts = (pts / horizontal_scale).long()
    px = torch.clip(pts[:, :, 0].reshape(-1), 0, height_samples.shape[0] - 2)
    py = torch.clip(pts[:, :, 1].reshape(-1), 0, height_samples.shape[1] - 2)
    h = torch.min(torch.min(height_samples[px, py], height_samples[px + 1, py]), height_samples[px, py + 1])
    return h.view(n, -1) * vertical_scale


def scaled_uniform(lo: float, hi: float, u: torch.Tensor) -> torch.Tensor:
    """isaacgym.torch_utils.torch_rand_float with the uniform draw supplied."""
    return (hi - lo) * u + lo


class OracleHectorEnv:
    """State + step of the env stage, on CPU, for N envs: `hector` (hector_env.py) and, through the task layout of the
    config (isaac_b200.envs.tasks), `hector_full` (hector_w_arm_env.py) and `humanoid_ppo` / XBot-L (humanoid_env.py) -
    the three env files differ in joint indices, the arm term of default_joint_pos and the privileged frame."""

    def __init__(self, cfg, statics, frame, noise):
        from isaac_b200.envs.tasks import layout_for
        self.cfg = cfg
        self.layout = layout_for(cfg)
        n = statics.p_gains.shape[0]
        self.num_envs = n
        self.num_dof = self.num_actions = cfg.env.num_actions
        self.feet = list(_find(cfg.asset.body_names, [cfg.asset.foot_name]))
        self.knees = list(_find(cfg.asset.body_names, [cfg.asset.knee_name]))
        self.term_bodies = list(_find(cfg.asset.body_names, cfg.asset.terminate_after_contacts_on))
        self.pen_bodies = list(_find(cfg.asset.body_names, cfg.asset.penalize_contacts_on))
        # _parse_cfg, legged_robot.py:711-722
        self.dt = cfg.control.decimation * cfg.sim.dt
        self.max_episode_length_s = cfg.env.episode_length_s
        self.max_episode_length = np.ceil(self.max_episode_length_s / self.dt)
        self.push_interval = np.ceil(cfg.domain_rand.push_interval_s / self.dt)
        self.resample_interval = int(cfg.commands.resampling_time / self.dt)
        # _prepare_reward_function, legged_robot.py:517-540 (alphabetical via class_to_dict)
        from isaac_b200.envs.hector_config import class_to_dict
        scales = class_to_dict(cfg.rewards.scales)
        self.reward_scales = {k: v * self.dt for k, v in scales.items() if v != 0}
        self.reward_names = [k for k in self.reward_scales if k != "termination"]
        self.episode_sums = {k: torch.zeros(n) for k in self.reward_scales}
        # gym tensors
        self.root_states = frame.root_states.clone()
        self.dof_state = frame.dof_state.clone()
        self.contact_forces = frame.contact_forces.clone()
        self.rigid_state = frame.rigid_state.clone()
        self.dof_pos = self.dof_state.view(n, self.num_dof, 2)[..., 0]
        self.dof_vel = self.dof_state.view(n, self.num_dof, 2)[..., 1]
        # _init_buffers, legged_robot.py:433-515
        os_ = cfg.normalization.obs_scales
        self.obs_scales = os_
        self.torque_limits = torch.tensor(cfg.asset.dof_effort) * cfg.safety.torque_limit   # :292
        self.p_gains = statics.p_gains.clone()
        self.d_gains = statics.d_gains.clone()
        self.default_dof_pos = torch.tensor(
            [cfg.init_state.default_joint_angles[k] for k in cfg.asset.dof_names]).unsqueeze(0)
        z = lambda *s: torch.zeros(*s)
        nd = self.num_dof
        self.torques, self.actions = z(n, nd), z(n, nd)
        self.last_actions, self.last_last_actions = z(n, nd), z(n, nd)
        self.last_dof_vel, self.last_root_vel = z(n, nd), z(n, 6)
        self.ref_dof_pos = z(n, nd)
        self.commands = z(n, cfg.commands.num_commands)
        self.commands_scale = torch.tensor([os_.lin_vel, os_.lin_vel, os_.ang_vel])
        self.feet_air_time = z(n, 2)
        self.last_contacts = torch.zeros(n, 2, dtype=torch.bool)
        self.gravity_vec = torch.tensor([0.0, 0.0, -1.0]).repeat(n, 1)
        self.forward_vec = torch.tensor([1.0, 0.0, 0.0]).repeat(n, 1)
        q = self.root_states[:, 3:7]
        self.base_lin_vel = quat_rotate_inverse(q, self.root_states[:, 7:10])
        self.base_ang_vel = quat_rotate_inverse(q, self.root_states[:, 10:13])
        self.projected_gravity = quat_rotate_inverse(q, self.gravity_vec)
        self.base_euler_xyz = euler_xyz_wrapped(q)
        self.rand_push_force, self.rand_push_torque = z(n, 3), z(n, 3)
        self.env_frictions = statics.env_frictions.clone()
        self.body_mass = statics.body_mass.clone()
        self.env_origins = statics.env_origins.clone()
        self.base_init_state = torch.tensor(cfg.init_state.pos + cfg.init_state.rot
                                            + cfg.init_state.lin_vel + cfg.init_state.ang_vel)
        self.obs_hist = z(n, cfg.env.frame_stack, cfg.env.num_single_obs)          # oldest .. newest
        self.priv_hist = z(n, cfg.env.c_frame_stack, cfg.env.single_num_privileged_obs)
        self.noise_scale_vec = self._noise_scale_vec()
        self.episode_length_buf = torch.zeros(n, dtype=torch.long)
        self.reset_buf = torch.ones(n, dtype=torch.long)         # base_task.py:82 (long until first step)
        self.time_out_buf = torch.zeros(n, dtype=torch.bool)
        self.rew_buf = z(n)
        self.extras: Dict = {}
        self.common_step_counter = 0
        self.last_reset_ids = torch.zeros(0, dtype=torch.long)
        # HectorFreeEnv.__init__ tail, hector_env.py:48-51
        self.last_feet_z = 0.05
        self.feet_height = z(n, 2)
        self.reset_idx(torch.arange(n), noise)
        self.compute_observations(noise)
        self.episode_length_buf[:] = statics.episode_length0

    # ------------------------------------------------------------------ hector_env.py:135-155
    def _noise_scale_vec(self):
        ns, os_ = self.cfg.noise.noise_scales, self.obs_scales
        v = torch.zeros(self.cfg.env.num_single_obs)
        sl = [slice(a, b) for a, b in self.layout.noise_slices]          # the literal slices of each env file
        v[sl[0]] = ns.dof_pos * os_.dof_pos
        v[sl[1]] = ns.dof_vel * os_.dof_vel
        v[sl[2]] = 0.0                         # previous actions
        v[sl[3]] = ns.ang_vel * os_.ang_vel
        v[sl[4]] = ns.quat * os_.quat          # hector: 38:42 silently clamps to 38:41 (quirk 6)
        return v

    # ------------------------------------------------------------------ legged_robot.py:339-355
    def compute_torques(self, actions):
        target = actions * self.cfg.control.action_scale
        tau = self.p_gains * (target + self.default_dof_pos - self.dof_pos) - self.d_gains * self.dof_vel
        return torch.clip(tau, -self.torque_limits, self.torque_limits)

    # ------------------------------------------------------------------ hector_env.py:158-169 + legged_robot.py:84-108
    def step(self, frame, noise):
        """`frame` plays the role of what PhysX refreshes; it is installed before the
        decimation loop because the stubbed `gym.simulate` does not evolve the state."""
        self.root_states.copy_(frame.root_states)
        self.dof_state.copy_(frame.dof_state)
        self.contact_forces.copy_(frame.contact_forces)
        self.rigid_state.copy_(frame.rigid_state)
        dr = self.cfg.domain_rand
        clip_a = self.cfg.normalization.clip_actions
        a = torch.clip(noise.actions, -clip_a, clip_a)
        delay = noise.u_delay * dr.action_delay
        a = (1 - delay) * a + delay * self.actions
        a = a + dr.action_noise * noise.z_action * a
        self.actions = torch.clip(a, -clip_a, clip_a)
        for _ in range(self.cfg.control.decimation):
            self.torques = self.compute_torques(self.actions)
        self.post_physics_step(noise)
        clip_o = self.cfg.normalization.clip_observations
        self.obs_buf = torch.clip(self.obs_buf, -clip_o, clip_o)
        self.privileged_obs_buf = torch.clip(self.privileged_obs_buf, -clip_o, clip_o)
        return self.obs_buf, self.privileged_obs_buf, self.rew_buf, self.reset_buf, self.extras

    # ------------------------------------------------------------------ legged_robot.py:118-153
    def post_physics_step(self, noise):
        self.episode_length_buf += 1
        self.common_step_counter += 1
        q = self.root_states[:, 3:7]
        self.base_lin_vel = quat_rotate_inverse(q, self.root_states[:, 7:10])
        self.base_ang_vel = quat_rotate_inverse(q, self.root_states[:, 10:13])
        self.projected_gravity = quat_rotate_inverse(q, self.gravity_vec)
        self.base_euler_xyz = euler_xyz_wrapped(q)
        self.post_physics_callback(noise)
        self.check_termination()
        self.compute_reward()
        ids = self.reset_buf.nonzero(as_tuple=False).flatten()
        self.last_reset_ids = ids
        self.reset_idx(ids, noise)
        self.compute_observations(noise)
        self.last_last_actions = self.last_actions.clone()
        self.last_actions = self.actions.clone()
        self.last_dof_vel = self.dof_vel.clone()
        self.last_root_vel = self.root_states[:, 7:13].clone()

    # ------------------------------------------------------------------ legged_robot.py:303-335, hector_env.py:53-68
    def post_physics_callback(self, noise):
        ids = (self.episode_length_buf % self.resample_interval == 0).nonzero(as_tuple=False).flatten()
        self.resample_commands(ids, noise.u_cmd[ids])
        if self.cfg.commands.heading_command:
            fwd = quat_apply(self.root_states[:, 3:7], self.forward_vec)
            heading = torch.atan2(fwd[:, 1], fwd[:, 0])
            self.commands[:, 2] = torch.clip(0.5 * wrap_to_pi(self.commands[:, 3] - heading), -1.0, 1.0)
        dr = self.cfg.domain_rand
        if dr.push_robots and (self.common_step_counter % self.push_interval == 0):
            self.rand_push_force[:, :2] = scaled_uniform(-dr.max_push_vel_xy, dr.max_push_vel_xy, noise.u_push[:, 0:2])
            self.root_states[:, 7:9] = self.rand_push_force[:, :2]
            self.rand_push_torque = scaled_uniform(-dr.max_push_ang_vel, dr.max_push_ang_vel, noise.u_push[:, 2:5])
            self.root_states[:, 10:13] = self.rand_push_torque

    def resample_commands(self, ids, u):
        r = self.cfg.commands.ranges
        self.commands[ids, 0] = scaled_uniform(r.lin_vel_x[0], r.lin_vel_x[1], u[:, 0:1]).squeeze(1)
        self.commands[ids, 1] = scaled_uniform(r.lin_vel_y[0], r.lin_vel_y[1], u[:, 1:2]).squeeze(1)
        self.commands[ids, 3] = scaled_uniform(r.heading[0], r.heading[1], u[:, 2:3]).squeeze(1)
        self.commands[ids, :2] *= (torch.norm(self.commands[ids, :2], dim=1) > 0.2).unsqueeze(1)

    # ------------------------------------------------------------------ legged_robot.py:155-160
    def check_termination(self):
        self.reset_buf = torch.any(torch.norm(self.contact_forces[:, self.term_bodies, :], dim=-1) > 1.0, dim=1)
        self.time_out_buf = self.episode_length_buf > self.max_episode_length
        self.reset_buf |= self.time_out_buf

    # ------------------------------------------------------------------ legged_robot.py:216-234
    def compute_reward(self):
        self.rew_buf = torch.zeros(self.num_envs)
        for name in self.reward_names:
            r = REWARD_FORMULAS[name](self) * self.reward_scales[name]
            self.rew_buf += r
            self.episode_sums[name] += r
        if self.cfg.rewards.only_positive_rewards:
            self.rew_buf = torch.clip(self.rew_buf, min=0.0)

    # ------------------------------------------------------------------ legged_robot.py:162-214,358-396; hector_env.py:256-261
    def reset_idx(self, ids, noise):
        if len(ids) == 0:
            return                                            # extras untouched (quirk 4)
        u = noise.u_reset[ids]
        nd = self.num_dof
        self.dof_pos[ids] = self.default_dof_pos + scaled_uniform(-0.15, 0.15, u[:, 0:nd])
        self.dof_vel[ids] = 0.0
        self.root_states[ids] = self.base_init_state
        self.root_states[ids, :3] += self.env_origins[ids]
        if self.cfg.terrain.mesh_type in ("heightfield", "trimesh"):      # custom_origins (legged_robot.py:381-384,687-688)
            self.root_states[ids, :2] += scaled_uniform(-1.0, 1.0, u[:, nd:nd + 2])
        self.resample_commands(ids, u[:, nd + 2:nd + 5])
        for buf in (self.last_last_actions, self.actions, self.last_actions, self.last_dof_vel, self.feet_air_time):
            buf[ids] = 0.0
        self.episode_length_buf[ids] = 0
        self.reset_buf[ids] = 1
        self.extras["episode"] = {}
        for k in self.episode_sums:
            self.extras["episode"]["rew_" + k] = torch.mean(self.episode_sums[k][ids]) / self.max_episode_length_s
            self.episode_sums[k][ids] = 0.0
        if self.cfg.terrain.mesh_type == "trimesh":
            self.extras["episode"]["terrain_level"] = torch.tensor(0.0)      # terrain_levels stay 0 without a curriculum
        if self.cfg.env.send_timeouts:
            self.extras["time_outs"] = self.time_out_buf
        q = self.root_states[:, 3:7]
        self.base_euler_xyz = euler_xyz_wrapped(q)
        self.projected_gravity[ids] = quat_rotate_inverse(q[ids], self.gravity_vec[ids])
        self.obs_hist[ids] = 0.0
        self.priv_hist[ids] = 0.0

    # ------------------------------------------------------------------ hector_env.py:70-88
    def phase(self):
        return self.episode_length_buf * self.dt / self.cfg.rewards.cycle_time

    def stance_mask(self):
        s = torch.sin(2 * torch.pi * self.phase())
        m = torch.zeros(self.num_envs, 2)
        m[:, 0] = s >= 0
        m[:, 1] = s < 0
        m[torch.abs(s) < 0.1] = 1
        return m

    def feet_contact(self):
        return self.contact_forces[:, self.feet, 2] > 5.0

    # ------------------------------------------------------------------ hector_env.py:90-111 / humanoid_env.py:120-142
    def compute_ref_state(self):
        s = torch.sin(2 * torch.pi * self.phase())
        sl, sr = s.clone(), s.clone()
        self.ref_dof_pos = torch.zeros_like(self.dof_pos)
        scale_1 = self.cfg.rewards.target_joint_pos_scale
        scale_2 = 2 * scale_1
        sl[sl > 0] = 0
        for j, sc in zip(self.layout.ref_left, (scale_1, scale_2, scale_1)):
            self.ref_dof_pos[:, j] = sl * sc
        sr[sr < 0] = 0
        for j, sc in zip(self.layout.ref_right, (scale_1, scale_2, scale_1)):
            self.ref_dof_pos[:, j] = sr * sc
        self.ref_dof_pos[torch.abs(s) < 0.1] = 0

    # ------------------------------------------------------------------ hector_env.py:172-254
    def compute_observations(self, noise):
        from isaac_b200._lib import HB_TASK_XBOT
        self.compute_ref_state()
        ph = self.phase()
        s = torch.sin(2 * torch.pi * ph).unsqueeze(1)
        c = torch.cos(2 * torch.pi * ph).unsqueeze(1)
        stance, contact = self.stance_mask(), self.feet_contact()
        os_ = self.obs_scales
        cmd_in = torch.cat((s, c, self.commands[:, :3] * self.commands_scale), dim=1)
        qd = (self.dof_pos - self.default_dof_pos) * os_.dof_pos
        dq = self.dof_vel * os_.dof_vel
        if self.layout.kind == HB_TASK_XBOT:        # humanoid_env.py:217-234
            priv = torch.cat((cmd_in, qd, dq, self.actions, self.dof_pos - self.ref_dof_pos,
                              self.base_lin_vel * os_.lin_vel, self.base_ang_vel * os_.ang_vel,
                              self.base_euler_xyz * os_.quat, self.rand_push_force[:, :2], self.rand_push_torque,
                              self.env_frictions, self.body_mass / 30.0, stance, contact), dim=-1)
        else:
            priv = torch.cat((cmd_in, qd, dq, self.actions,
                              self.base_lin_vel * os_.lin_vel, self.base_ang_vel * os_.ang_vel,
                              self.base_euler_xyz * os_.quat,
                              self.rigid_state[:, self.feet, :3].flatten(1), self.rigid_state[:, self.feet, 7:10].flatten(1),
                              self.root_states[:, :3], self.rand_push_force[:, :2], self.rand_push_torque,
                              self.env_frictions, self.body_mass / 30.0, stance, contact), dim=-1)
        frame = torch.cat((cmd_in, qd, dq, self.actions, self.base_ang_vel * os_.ang_vel,
                           self.base_euler_xyz * os_.quat), dim=-1)
        if self.cfg.noise.add_noise:
            frame = frame + noise.z_obs * self.noise_scale_vec * self.cfg.noise.noise_level
        self.obs_hist = torch.cat((self.obs_hist[:, 1:], frame.unsqueeze(1)), dim=1)
        self.priv_hist = torch.cat((self.priv_hist[:, 1:], priv.unsqueeze(1)), dim=1)
        self.obs_buf = self.obs_hist.reshape(self.num_envs, -1)
        self.privileged_obs_buf = self.priv_hist.reshape(self.num_envs, -1)


def _find(names, patterns):
    for p in patterns:
        for i, s in enumerate(names):
            if p in s:
                yield i


# ------------------------------------------------------------------------------------
# Reward terms (hector_env.py:264-539); each returns the unscaled term, shape [N]
# ------------------------------------------------------------------------------------
def _pair_distance_reward(xy, lo, hi):
    d = torch.norm(xy[:, 0, :] - xy[:, 1, :], dim=1)
    near = torch.clamp(d - lo, -0.5, 0.0)
    far = torch.clamp(d - hi, 0, 0.5)
    return (torch.exp(-torch.abs(near) * 100) + torch.exp(-torch.abs(far) * 100)) / 2


@_reward("feet_distance")          # :277-287
def _r_feet_distance(e):
    return _pair_distance_reward(e.rigid_state[:, e.feet, :2], e.cfg.rewards.min_dist, e.cfg.rewards.max_dist)


@_reward("knee_distance")          # :290-300
def _r_knee_distance(e):
    return _pair_distance_reward(e.rigid_state[:, e.knees, :2], e.cfg.rewards.min_dist, e.cfg.rewards.max_dist / 2)


@_reward("foot_slip")              # :303-313
def _r_foot_slip(e):
    speed = torch.sqrt(torch.norm(e.rigid_state[:, e.feet, 7:9], dim=2))
    speed *= e.feet_contact()
    return torch.sum(speed, dim=1)


@_reward("feet_air_time")          # :315-329  (stateful)
def _r_feet_air_time(e):
    contact = e.feet_contact()
    filt = torch.logical_or(torch.logical_or(contact, e.stance_mask()), e.last_contacts)
    e.last_contacts = contact
    first = (e.feet_air_time > 0.0) * filt
    e.feet_air_time += e.dt
    r = e.feet_air_time.clamp(0, 0.5) * first
    e.feet_air_time *= ~filt
    return r.sum(dim=1)


@_reward("feet_contact_number")    # :331-339
def _r_feet_contact_number(e):
    return torch.mean(torch.where(e.feet_contact() == e.stance_mask(), 1, -0.3), dim=1)


@_reward("orientation")            # :341-348
def _r_orientation(e):
    a = torch.exp(-torch.sum(torch.abs(e.base_euler_xyz[:, :2]), dim=1) * 10)
    b = torch.exp(-torch.norm(e.projected_gravity[:, :2], dim=1) * 20)
    return (a + b) / 2.0


@_reward("feet_contact_forces")    # :350-355
def _r_feet_contact_forces(e):
    f = torch.norm(e.contact_forces[:, e.feet, :], dim=-1)
    return torch.sum((f - e.cfg.rewards.max_contact_force).clip(0, 400), dim=1)


@_reward("default_joint_pos")      # :357-367; hector_w_arm_env.py:361-378 adds the arm term
def _r_default_joint_pos(e):
    d = e.dof_pos - e.default_dof_pos
    l, r = e.layout.yaw_roll
    yr = torch.norm(d[:, l:l + 2], dim=1) + torch.norm(d[:, r:r + 2], dim=1)
    yr = torch.clamp(yr - 0.1, 0, 50)
    out = torch.exp(-yr * 100)
    if e.layout.arm_pair[0] >= 0:
        la, ra = e.layout.arm_pair
        arm = torch.norm(d[:, la:la + 2], dim=1) + torch.norm(d[:, ra:ra + 2], dim=1)
        arm = torch.clamp(arm - 0.1, 0, 25)
        out = out + torch.exp(-arm * 2)
    return out - 0.01 * torch.norm(d, dim=1)


@_reward("joint_pos")              # :264-275 (ref_dof_pos is what the previous compute_observations left)
def _r_joint_pos(e):
    nrm = torch.norm(e.dof_pos - e.ref_dof_pos, dim=1)
    return torch.exp(-2 * nrm) - 0.2 * nrm.clamp(0, 0.5)


@_reward("vel_mismatch_exp")       # :395-405
def _r_vel_mismatch_exp(e):
    lin = torch.exp(-torch.square(e.base_lin_vel[:, 2]) * 10)
    ang = torch.exp(-torch.norm(e.base_ang_vel[:, :2], dim=1) * 5.0)
    return (lin + ang) / 2.0


@_reward("track_vel_hard")         # :407-424
def _r_track_vel_hard(e):
    lin_err = torch.norm(e.commands[:, :2] - e.base_lin_vel[:, :2], dim=1)
    ang_err = torch.abs(e.commands[:, 2] - e.base_ang_vel[:, 2])
    return (torch.exp(-lin_err * 10) + torch.exp(-ang_err * 10)) / 2.0 - 0.2 * (lin_err + ang_err)


@_reward("low_speed")              # :468-499
def _r_low_speed(e):
    speed, cmd = torch.abs(e.base_lin_vel[:, 0]), torch.abs(e.commands[:, 0])
    low, high = speed < 0.5 * cmd, speed > 1.2 * cmd
    r = torch.zeros_like(speed)
    r[low] = -1.0
    r[high] = 0.0
    r[~(low | high)] = 1.2
    r[torch.sign(e.base_lin_vel[:, 0]) != torch.sign(e.commands[:, 0])] = -2.0
    return r * (e.commands[:, 0].abs() > 0.1)


@_reward("base_height")            # :369-383
def _r_base_height(e):
    st = e.stance_mask()
    ground = torch.sum(e.rigid_state[:, e.feet, 2] * st, dim=1) / torch.sum(st, dim=1)
    h = e.root_states[:, 2] - (ground - 0.05)
    return torch.exp(-torch.abs(h - e.cfg.rewards.base_height_target) * 100)


@_reward("base_acc")               # :385-392
def _r_base_acc(e):
    return torch.exp(-torch.norm(e.last_root_vel - e.root_states[:, 7:13], dim=1) * 3)


@_reward("tracking_lin_vel")       # :426-433
def _r_tracking_lin_vel(e):
    err = torch.sum(torch.square(e.commands[:, :2] - e.base_lin_vel[:, :2]), dim=1)
    return torch.exp(-err * e.cfg.rewards.tracking_sigma)


@_reward("tracking_ang_vel")       # :435-443
def _r_tracking_ang_vel(e):
    err = torch.square(e.commands[:, 2] - e.base_ang_vel[:, 2])
    return torch.exp(-err * e.cfg.rewards.tracking_sigma)


@_reward("feet_clearance")         # :445-466  (stateful; last_feet_z starts as the float 0.05, :48)
def _r_feet_clearance(e):
    contact = e.feet_contact()
    z = e.rigid_state[:, e.feet, 2] - 0.05
    e.feet_height += z - e.last_feet_z
    e.last_feet_z = z
    swing = 1 - e.stance_mask()
    hit = torch.abs(e.feet_height - e.cfg.rewards.target_feet_height) < 0.01
    r = torch.sum(hit * swing, dim=1)
    e.feet_height *= ~contact
    return r


@_reward("torques")                # :501-506
def _r_torques(e):
    return torch.sum(torch.square(e.torques), dim=1)


@_reward("dof_vel")                # :508-513
def _r_dof_vel(e):
    return torch.sum(torch.square(e.dof_vel), dim=1)


@_reward("dof_acc")                # :515-520
def _r_dof_acc(e):
    return torch.sum(torch.square((e.last_dof_vel - e.dof_vel) / e.dt), dim=1)


@_reward("collision")              # :522-527
def _r_collision(e):
    return torch.sum(1.0 * (torch.norm(e.contact_forces[:, e.pen_bodies, :], dim=-1) > 0.1), dim=1)


@_reward("action_smoothness")      # :529-539
def _r_action_smoothness(e):
    t1 = torch.sum(torch.square(e.last_actions - e.actions), dim=1)
    t2 = torch.sum(torch.square(e.actions + e.last_last_actions - 2 * e.last_actions), dim=1)
    t3 = 0.05 * torch.sum(torch.abs(e.actions), dim=1)
    return t1 + t2 + t3
