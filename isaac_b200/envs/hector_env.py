"""`HectorFreeEnvB200` — drop-in for the reference's `HectorFreeEnv` / `LeggedRobot` hot path.

Same contract as the reference env (algo/vec_env.py:37-60; envs/base/legged_robot.py:84-153;
envs/custom/hector_env.py:158-261):

    step(actions[N,10]) -> obs[N,615], privileged_obs[N,1050], rew[N], reset[N] bool, extras
    reset() -> obs, privileged_obs;  get_observations();  get_privileged_observations()

and the same attribute names the runner and `play.py` read (dof_pos, dof_vel, torques,
commands, base_lin_vel, base_ang_vel, contact_forces, feet_indices, episode_sums, ...).
The per-step work is four kinds of kernel launch through the C ABI (include/hector_b200.h), 12 launches in all:

    hb_env_action_prologue      x1   hector_env.py:158-169
    hb_env_compute_torques      x decimation, around the opaque physics.simulate()
                                     (the CUDA-graph path fuses the prologue with the first sub-step:
                                     hb_env_prologue_torques)
    hb_env_post_physics         x1   legged_robot.py:118-234,303-396 + newest obs frames
    hb_env_stack_finalize       x1   hector_env.py:246-261 (frame stacking into the ping-pong buffers, history zeroing
                                     of the envs just reset) + legged_robot.py:142,198-209 (ascending reset ids,
                                     count, episode means, time_outs) - the fused form of
                                     hb_env_stack_observations + hb_env_reset_finalize

Observation tensors are `[N, 615]` / `[N, 1050]` views of rows at a 128-byte pitch (640 / 1056 floats); the caller may
supply the buffers of the next step (`set_next_observation_buffers`, what `PPO.attach_env` does with the rollout slots).
`enable_cuda_graph()` replays the step from two graphs of these launches (hb_graph_*), with no staging copy around them.

There is no torch/eager fallback: without libhectorb200.so construction fails.
`step()` never blocks on the GPU; the one host-visible value the reference needs (the reset
count for `gym.set_*_tensor_indexed`) is written to pinned memory by the kernel and consumed
right before the next `physics.simulate()`.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, NamedTuple, Optional

import numpy as np
import torch

from .. import _lib
from .._lib import (EnvBuffers, EnvNoise, EnvParams, HB_NUM_REWARDS, HB_STAGE_DERIVE, HB_STAGE_LAST, HB_STAGE_OBS,
                    HB_STAGE_PREPARE, HB_STAGE_PUSH, HB_STAGE_RESET_ALL, HB_STAGE_RESET_MASK, HB_STAGE_REWARD, HB_STAGE_STEP,
                    HB_STAGE_TERMINATION, REWARD_NAMES)
from .hector_config import class_to_dict
from .tasks import layout_for

_EXTRAS_RING = 256       # >= num_steps_per_env: episode-mean slots handed out through extras["episode"]


class _BufferPair(NamedTuple):
    """Observation and privileged-observation buffers of one step; `key` = their addresses, which key the step graphs."""
    obs: torch.Tensor
    priv: torch.Tensor
    key: tuple

    @classmethod
    def of(cls, obs, priv):
        return cls(obs, priv, (obs.data_ptr(), priv.data_ptr()))


def _find(names, patterns):
    return [i for p in patterns for i, s in enumerate(names) if p in s]


def _reset_pose_constants(quat_xyzw):
    """Euler angles and projected gravity of the reset pose, in fp32 and in the reference's operation
    order (get_euler_xyz_tensor, legged_robot.py:50-55; quat_rotate_inverse of (0,0,-1)): every reset
    env gets base_init_state's quaternion, so reset_idx's recomputation (:211-214) is a constant."""
    f = np.float32
    x, y, z, w = (f(v) for v in quat_xyzw)
    two_pi, pi = f(2 * np.pi), f(np.pi)
    roll = np.arctan2(f(2.0) * (w * x + y * z), ((w * w - x * x) - y * y) + z * z, dtype=f)
    sinp = f(2.0) * (w * y - z * x)
    pitch = f(np.pi / 2.0) * np.sign(sinp) if abs(sinp) >= 1 else np.arcsin(sinp, dtype=f)
    yaw = np.arctan2(f(2.0) * (w * z + x * y), ((w * w + x * x) - y * y) - z * z, dtype=f)
    eul = []
    for a in (roll, pitch, yaw):
        a = f(np.remainder(f(a), two_pi))
        eul.append(a - two_pi if a > pi else a)
    u, v = np.array([x, y, z], dtype=f), np.array([0.0, 0.0, -1.0], dtype=f)
    a = v * (f(2.0) * w * w - f(1.0))
    b = np.cross(u, v).astype(f) * w * f(2.0)
    c = u * f(np.dot(u, v)) * f(2.0)
    return eul, (a - b) + c


def build_env_params(cfg, num_envs: int, num_bodies: int, body_names, dof_names, dof_effort) -> EnvParams:
    """Resolve the config the way LeggedRobot._parse_cfg / _init_buffers / _prepare_reward_function /
    _get_noise_scale_vec do (legged_robot.py:433-540,711-722; hector_env.py:135-155); Python-double
    arithmetic first, fp32 at the end, exactly like scalars reach torch kernels in the reference."""
    p = EnvParams()
    p.abi_version = _lib.HB_ABI_VERSION
    lay = layout_for(cfg)
    p.num_envs, p.num_dof, p.num_bodies, p.task_kind = num_envs, cfg.env.num_actions, num_bodies, lay.kind
    p.yaw_roll[:], p.arm_pair[:], p.ref_left[:], p.ref_right[:] = lay.yaw_roll, lay.arm_pair, lay.ref_left, lay.ref_right
    scale_1 = cfg.rewards.target_joint_pos_scale          # compute_ref_state: scale_1, scale_2 = 2 * scale_1 (Python doubles)
    p.ref_scale[0], p.ref_scale[1] = scale_1, 2 * scale_1
    p.num_single_obs, p.frame_stack = cfg.env.num_single_obs, cfg.env.frame_stack
    p.num_single_priv, p.c_frame_stack = cfg.env.single_num_privileged_obs, cfg.env.c_frame_stack
    # rows at a 128-byte pitch: the observation buffers can then be rollout-storage slots and TMA operands
    p.obs_ld = (p.num_single_obs * p.frame_stack + 1 + 31) // 32 * 32       # ceil32(width + 1), like RolloutStorage
    p.priv_ld = (p.num_single_priv * p.c_frame_stack + 1 + 31) // 32 * 32
    feet = _find(body_names, [cfg.asset.foot_name])
    knees = _find(body_names, [cfg.asset.knee_name])
    term = _find(body_names, cfg.asset.terminate_after_contacts_on)
    pen = _find(body_names, cfg.asset.penalize_contacts_on)
    if len(feet) != 2 or len(knees) != 2:
        raise ValueError(f"the env step expects 2 feet and 2 knees, found {feet} / {knees}")
    if len(term) > _lib.HB_MAX_CONTACT_BODIES or len(pen) > _lib.HB_MAX_CONTACT_BODIES:
        raise ValueError("too many termination / penalised contact bodies")
    p.feet[:], p.knees[:] = feet, knees
    p.n_term, p.n_pen = len(term), len(pen)
    for i, b in enumerate(term):
        p.term_bodies[i] = b
    for i, b in enumerate(pen):
        p.pen_bodies[i] = b
    dt = cfg.control.decimation * cfg.sim.dt
    p.dt = dt
    p.max_episode_length = int(np.ceil(cfg.env.episode_length_s / dt))
    p.max_episode_length_s = cfg.env.episode_length_s
    p.resample_interval = int(cfg.commands.resampling_time / dt)
    p.heading_command = int(cfg.commands.heading_command)
    p.add_noise = int(cfg.noise.add_noise)
    p.only_positive_rewards = int(cfg.rewards.only_positive_rewards)
    p.custom_origins = int(cfg.terrain.mesh_type in ("heightfield", "trimesh"))
    p.action_scale = cfg.control.action_scale
    p.clip_actions = cfg.normalization.clip_actions
    p.clip_observations = cfg.normalization.clip_observations
    p.action_delay = cfg.domain_rand.action_delay
    p.action_noise = cfg.domain_rand.action_noise
    for j, name in enumerate(dof_names):
        p.default_dof_pos[j] = cfg.init_state.default_joint_angles[name]
        p.torque_limits[j] = dof_effort[j] * cfg.safety.torque_limit
    p.cycle_time = cfg.rewards.cycle_time
    r = cfg.commands.ranges
    for k, rng in enumerate((r.lin_vel_x, r.lin_vel_y, r.heading)):
        p.cmd_lo[k], p.cmd_span[k] = rng[0], rng[1] - rng[0]
    dr = cfg.domain_rand
    p.push_lin_lo, p.push_lin_span = -dr.max_push_vel_xy, dr.max_push_vel_xy - (-dr.max_push_vel_xy)
    p.push_ang_lo, p.push_ang_span = -dr.max_push_ang_vel, dr.max_push_ang_vel - (-dr.max_push_ang_vel)
    p.reset_dof_lo, p.reset_dof_span = -0.15, 0.15 - (-0.15)
    p.reset_xy_lo, p.reset_xy_span = -1.0, 1.0 - (-1.0)
    init = cfg.init_state.pos + cfg.init_state.rot + cfg.init_state.lin_vel + cfg.init_state.ang_vel
    for k in range(13):
        p.base_init_state[k] = init[k]
    eul, grav = _reset_pose_constants(init[3:7])
    for k in range(3):
        p.reset_euler[k], p.reset_gravity[k] = float(eul[k]), float(grav[k])
    os_ = cfg.normalization.obs_scales
    p.obs_lin_vel, p.obs_ang_vel, p.obs_dof_pos, p.obs_dof_vel, p.obs_quat = (
        os_.lin_vel, os_.ang_vel, os_.dof_pos, os_.dof_vel, os_.quat)
    p.noise_level = cfg.noise.noise_level
    ns = cfg.noise.noise_scales
    vec = np.zeros(p.num_single_obs, dtype=np.float32)          # _get_noise_scale_vec builds it in fp32, with the slices
    sl = [slice(a, b) for a, b in lay.noise_slices]             # each env file spells out (hector_env.py:145-155, ...)
    vec[sl[0]] = ns.dof_pos * os_.dof_pos
    vec[sl[1]] = ns.dof_vel * os_.dof_vel
    vec[sl[2]] = 0.0
    vec[sl[3]] = ns.ang_vel * os_.ang_vel
    vec[sl[4]] = ns.quat * os_.quat
    for k in range(p.num_single_obs):
        p.noise_scale_vec[k] = float(vec[k])
    scales = class_to_dict(cfg.rewards.scales)
    unknown = [k for k, v in scales.items() if v != 0 and k not in REWARD_NAMES]
    if unknown:
        raise ValueError(f"reward terms without a kernel implementation have non-zero scale: {unknown}")
    for k, name in enumerate(REWARD_NAMES):
        p.reward_scale[k] = scales.get(name, 0.0) * dt
    rw = cfg.rewards
    p.base_height_target, p.min_dist, p.max_dist = rw.base_height_target, rw.min_dist, rw.max_dist
    p.target_feet_height, p.tracking_sigma, p.max_contact_force = (
        rw.target_feet_height, rw.tracking_sigma, rw.max_contact_force)
    return p


class HectorFreeEnvB200:
    def __init__(self, cfg, sim_params=None, physics_engine=None, sim_device="cuda:0", headless=True, *,
                 physics, statics=None, body_names=None, dof_names=None, dof_effort=None,
                 initial_noise=None, dense_rows=False):
        """`physics`: the opaque stage (isaac_b200.physics).  `statics`: per-env constants that the
        reference collects while creating actors (legged_robot.py:256-301,683-709); defaults are the
        config constants.  body/dof names default to what Isaac Gym reports for the hector URDF."""
        self._lib = _lib.load(check_device=True)
        self.cfg = cfg
        self.sim_params = sim_params
        self.physics = physics
        self.device = torch.device(sim_device)
        self.headless = headless
        self.num_envs = N = physics.num_envs
        self.num_obs = cfg.env.num_observations
        self.num_privileged_obs = cfg.env.num_privileged_obs
        self.num_actions = cfg.env.num_actions
        self.num_dof = self.num_dofs = physics.num_dof
        self.num_bodies = physics.num_bodies
        body_names = body_names or cfg.asset.body_names
        self.dof_names = dof_names or cfg.asset.dof_names
        dof_effort = dof_effort or cfg.asset.dof_effort
        self._p = build_env_params(cfg, N, self.num_bodies, body_names, self.dof_names, dof_effort)
        if dense_rows:          # contiguous [N,615] / [N,1050] observation tensors like the reference's (no row padding)
            self._p.obs_ld, self._p.priv_ld = self._p.num_single_obs * self._p.frame_stack, self._p.num_single_priv * self._p.c_frame_stack
        # _parse_cfg (legged_robot.py:711-722)
        self.dt = cfg.control.decimation * cfg.sim.dt
        self.obs_scales = cfg.normalization.obs_scales
        self.max_episode_length_s = cfg.env.episode_length_s
        self.max_episode_length = np.ceil(self.max_episode_length_s / self.dt)
        self.push_interval = np.ceil(cfg.domain_rand.push_interval_s / self.dt)
        self.reward_scales = {k: v * self.dt for k, v in class_to_dict(cfg.rewards.scales).items() if v != 0}
        self.reward_names = [k for k in self.reward_scales if k != "termination"]
        dev, f32 = self.device, dict(dtype=torch.float32, device=self.device)
        z = lambda *s, **kw: torch.zeros(*s, **{**f32, **kw})
        # gym tensors (owned by the physics stage, used in place)
        self.root_states, self.dof_state = physics.root_states, physics.dof_state
        self.contact_forces, self.rigid_state = physics.contact_forces, physics.rigid_state
        self.dof_pos = self.dof_state.view(N, self.num_dof, 2)[..., 0]
        self.dof_vel = self.dof_state.view(N, self.num_dof, 2)[..., 1]
        self.base_quat = self.root_states[:, 3:7]
        as_idx = lambda v: torch.tensor(list(v), dtype=torch.long, device=dev)
        self.feet_indices, self.knee_indices = as_idx(self._p.feet), as_idx(self._p.knees)
        self.termination_contact_indices = as_idx(self._p.term_bodies[:self._p.n_term])
        self.penalised_contact_indices = as_idx(self._p.pen_bodies[:self._p.n_pen])
        self.torque_limits = torch.tensor(list(self._p.torque_limits[:self.num_dof]), **f32)
        self.default_dof_pos = torch.tensor(list(self._p.default_dof_pos[:self.num_dof]), **f32).unsqueeze(0)
        self.default_joint_pd_target = self.default_dof_pos.clone()
        # per-env constants
        self.p_gains, self.d_gains = z(N, self.num_dof), z(N, self.num_dof)
        for i, name in enumerate(self.dof_names):            # legged_robot.py:485-500
            for key in cfg.control.stiffness:
                if key in name:
                    self.p_gains[:, i] = cfg.control.stiffness[key]
                    self.d_gains[:, i] = cfg.control.damping[key]
        self.env_frictions, self.body_mass, self.env_origins = z(N, 1), z(N, 1), z(N, 3)
        self.custom_origins = bool(self._p.custom_origins)
        self.terrain_levels = torch.zeros(N, dtype=torch.long, device=dev)
        if statics is not None:
            self.p_gains.copy_(statics.p_gains), self.d_gains.copy_(statics.d_gains)
            self.env_frictions.copy_(statics.env_frictions), self.body_mass.copy_(statics.body_mass)
            self.env_origins.copy_(statics.env_origins)
        # env state (legged_robot.py:458-515, base_task.py:72-92)
        nd = self.num_dof
        self.actions, self.last_actions, self.last_last_actions = z(N, nd), z(N, nd), z(N, nd)
        self.last_dof_vel, self.last_root_vel, self.torques = z(N, nd), z(N, 6), z(N, nd)
        self.ref_dof_pos = z(N, nd)                                        # compute_ref_state (hector_env.py:90-111)
        self.commands = z(N, cfg.commands.num_commands)
        self.commands_scale = torch.tensor([self.obs_scales.lin_vel, self.obs_scales.lin_vel, self.obs_scales.ang_vel], **f32)
        self.base_lin_vel, self.base_ang_vel = z(N, 3), z(N, 3)
        self.projected_gravity, self.base_euler_xyz = z(N, 3), z(N, 3)
        self.feet_air_time, self.feet_height = z(N, 2), z(N, 2)
        self.last_feet_z = torch.full((N, 2), 0.05, **f32)                 # hector_env.py:48
        self.last_contacts = torch.zeros(N, 2, dtype=torch.bool, device=dev)
        self.rand_push_force, self.rand_push_torque = z(N, 3), z(N, 3)
        self._episode_sums = z(HB_NUM_REWARDS, N)
        self.episode_sums = {k: self._episode_sums[i] for i, k in enumerate(REWARD_NAMES) if k in self.reward_scales}
        self._episode_length_buf = torch.zeros(N, dtype=torch.long, device=dev)
        self.reset_buf = torch.ones(N, dtype=torch.bool, device=dev)
        self.time_out_buf = torch.zeros(N, dtype=torch.bool, device=dev)
        self.rew_buf = z(N)
        self.noise_scale_vec = torch.tensor(list(self._p.noise_scale_vec[:self._p.num_single_obs]), **f32)
        self.add_noise = bool(cfg.noise.add_noise)
        self.gravity_vec = torch.tensor([0.0, 0.0, -1.0], **f32).repeat(N, 1)
        self.forward_vec = torch.tensor([1.0, 0.0, 0.0], **f32).repeat(N, 1)
        # ping-pong observation buffers: the tensor returned by step() stays valid until the step
        # after next (PPO.act keeps references until process_env_step, ppo.py:99-100,111).  Rows sit at a
        # 128-byte pitch (640 / 1056 floats); a caller may hand the env the buffers of the NEXT step
        # (set_next_observation_buffers: the rollout storage's slots), else it alternates between its own two.
        self._own = [_BufferPair.of(z(N, self._p.obs_ld)[:, :self.num_obs],
                                    z(N, self._p.priv_ld)[:, :self.num_privileged_obs]) for _ in range(2)]
        self._cur_buf = self._own[0]
        self._next_out = None
        # reset compaction + extras
        self.reset_env_ids = torch.zeros(N, dtype=torch.int32, device=dev)
        self._reset_count = torch.zeros(1, dtype=torch.int32, device=dev)
        self._host_count = torch.zeros(1, dtype=torch.int32).pin_memory() if dev.type == "cuda" else torch.zeros(1, dtype=torch.int32)
        self._episode_means = z(_EXTRAS_RING, HB_NUM_REWARDS)
        # device-side cursor of that ring: the finalize kernel writes slot `cursor` and advances it, so a captured
        # launch sequence lands in a new slot on every replay; the host mirrors it with _step_index
        self._episode_ring = torch.tensor([0, _EXTRAS_RING], dtype=torch.int32, device=dev)
        self._time_outs_latched = torch.zeros(N, dtype=torch.bool, device=dev)
        tiles = (N + 31) // 32
        self._scratch_ballots = torch.zeros(tiles, dtype=torch.int32, device=dev)
        self._scratch_sums = torch.zeros(HB_NUM_REWARDS, dtype=torch.float64, device=dev)
        self._terrain_level_mean = torch.zeros((), **f32)
        # extras["episode"] dicts are prebuilt views into the ring (no per-step tensor indexing)
        self._extras_episode = []
        for slot in range(_EXTRAS_RING):
            d = {"rew_" + k: self._episode_means[slot, i] for i, k in enumerate(REWARD_NAMES) if k in self.reward_scales}
            if cfg.terrain.mesh_type == "trimesh":
                d["terrain_level"] = self._terrain_level_mean          # mean(terrain_levels): no curriculum -> constant
            self._extras_episode.append(d)
        self._events = [torch.cuda.Event(), torch.cuda.Event()] if dev.type == "cuda" else []
        self.extras: Dict = {}
        self.common_step_counter = 0
        self._step_index = 0
        self._pending_event: Optional[torch.cuda.Event] = None
        self._graphs = None
        self._injected = initial_noise      # draws consumed by the constructor's reset_idx(all)
        # device generator state {step counter, key}: both in device memory, so captured step graphs follow seed()
        self._rng_state = torch.zeros(2, dtype=torch.int64, device=dev)
        self._rng_counter = self._rng_state[:1]
        self.seed(int(getattr(cfg, "seed", 1)))
        self._b = EnvBuffers()
        self._nz = EnvNoise()
        self._draws_bound = False           # a launch sequence is open: _nz holds its draws (_in_sequence)
        self._bind_buffers()
        self.init_done = True
        # HectorFreeEnv.__init__ tail (hector_env.py:48-51): reset_idx(all) + compute_observations,
        # preceded by the derived quantities of _init_buffers (legged_robot.py:452,477-479)
        self._in_sequence(self._launch_post, HB_STAGE_DERIVE | HB_STAGE_RESET_ALL | HB_STAGE_OBS)
        self._apply_pending_resets()

    # ------------------------------------------------------------------ plumbing
    def _bind_buffers(self):
        b = self._b
        for name, t in dict(
                root_states=self.root_states, dof_state=self.dof_state, contact_forces=self.contact_forces,
                rigid_state=self.rigid_state, p_gains=self.p_gains, d_gains=self.d_gains,
                env_frictions=self.env_frictions, body_mass=self.body_mass, env_origins=self.env_origins,
                actions=self.actions, last_actions=self.last_actions, last_last_actions=self.last_last_actions,
                last_dof_vel=self.last_dof_vel, last_root_vel=self.last_root_vel, torques=self.torques,
                commands=self.commands, base_lin_vel=self.base_lin_vel, base_ang_vel=self.base_ang_vel,
                projected_gravity=self.projected_gravity, base_euler_xyz=self.base_euler_xyz,
                feet_air_time=self.feet_air_time, last_contacts=self.last_contacts, feet_height=self.feet_height,
                last_feet_z=self.last_feet_z, ref_dof_pos=self.ref_dof_pos, rand_push_force=self.rand_push_force,
                rand_push_torque=self.rand_push_torque, episode_sums=self._episode_sums,
                episode_length_buf=self.episode_length_buf, reset_buf=self.reset_buf, time_out_buf=self.time_out_buf,
                rew_buf=self.rew_buf, reset_env_ids=self.reset_env_ids, reset_count=self._reset_count,
                time_outs_latched=self._time_outs_latched, scratch_ballots=self._scratch_ballots,
                scratch_sums=self._scratch_sums, episode_means=self._episode_means,
                episode_ring=self._episode_ring).items():
            if not t.is_contiguous():
                raise ValueError(f"{name} must be contiguous")
            setattr(b, name, t.data_ptr())
        self._pp, self._pb, self._pn = C.byref(self._p), C.byref(self._b), C.byref(self._nz)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def set_next_observation_buffers(self, obs: torch.Tensor, privileged_obs: torch.Tensor) -> None:
        """The next step() writes its observations into these tensors instead of the env's own ping-pong pair
        (one step only).  They are what step() then returns; rows must sit at the env's pitch
        (`[N, num_obs]` views of `[N, 640]` / `[N, 1056]` fp32 buffers, 16-byte aligned) and must not be the
        buffers the current observations live in.  PPO.act points this at the rollout storage's next slot, so
        that `add_transitions`' observation copies (rollout_storage.py:90-92) never happen."""
        for t, width, ld in ((obs, self.num_obs, self._p.obs_ld), (privileged_obs, self.num_privileged_obs, self._p.priv_ld)):
            if (t.device != self.device or t.dtype != torch.float32 or tuple(t.shape) != (self.num_envs, width)
                    or t.stride() != (ld, 1) or t.data_ptr() % 16):
                raise ValueError(f"observation buffer must be a [{self.num_envs}, {width}] fp32 view with row pitch {ld} on {self.device}")
        pair = _BufferPair.of(obs, privileged_obs)
        if pair.key[0] == self._cur_buf.key[0] or pair.key[1] == self._cur_buf.key[1]:
            raise ValueError("the next observation buffers must not alias the current ones")
        self._next_out = pair

    def _take_output(self):
        """Where this step's observations go: the caller's buffers if it supplied any, else the own pair not in use."""
        out, cur = self._next_out, self._cur_buf
        if out is not None:
            self._next_out = None
            if out.key[0] != cur.key[0] and out.key[1] != cur.key[1]:
                return out
        return self._own[1] if cur is self._own[0] else self._own[0]

    def inject_noise(self, frame) -> None:
        """Use the supplied draws (isaac_b200.synthetic.NoiseFrame on this device) instead of the env's own generator for
        the next launch sequence - the next step(), or a hook or reset_idx() called on its own - "noise injected as a
        supplied tensor"."""
        self._injected = frame

    def _in_sequence(self, launch, *args):
        """Run launch(*args) inside a launch sequence: an eager step(), the constructor's reset, or a hook, reset_idx() or
        post_physics_step() called on its own.  The outermost call binds the sequence's draws once (_draw_noise) and
        releases them when it returns; the calls nested in it (the hooks of the staged step) use that binding.  Every
        draw of a sequence is taken at one counter value: the frame-stack finalize launch (HB_STAGE_STEP / OBS) advances
        the counter by one after them, and a reset-only finalize only when reset_idx() opened the sequence itself."""
        if self._draws_bound:
            return launch(*args)
        self._draw_noise(False)
        self._draws_bound = True
        try:
            return launch(*args)
        finally:
            self._draws_bound = False

    def _draw_noise(self, push: bool):
        """Fill `_nz` with draws and leave it so, without opening a launch sequence (_in_sequence): the injected tape if
        there is one (consumed here), otherwise the device generator (Philox; key and step counter in `self._rng_state`):
        the tensors the reference draws with torch.rand / randn_like (hector_env.py:166,168,241;
        legged_robot.py:327-332,366,384) are never materialised.  The constructor's reset draws at counter 0, step t of a
        freshly seeded env at counter t (oracle/device_rng.py mirrors the draws).  `push` is unused, kept for callers."""
        nz = self._nz
        if self._injected is not None:
            f, self._injected = self._injected, None
            self._noise_keepalive = f
            nz.u_delay, nz.z_action = f.u_delay.data_ptr(), f.z_action.data_ptr()
            nz.u_cmd, nz.u_push, nz.u_reset, nz.z_obs = (f.u_cmd.data_ptr(), f.u_push.data_ptr(),
                                                         f.u_reset.data_ptr(), f.z_obs.data_ptr())
            nz.rng_counter = None
            return
        self._bind_device_rng(nz)

    def _bind_device_rng(self, nz):
        nz.u_delay = nz.z_action = nz.u_cmd = nz.u_push = nz.u_reset = nz.z_obs = None
        nz.rng_counter = self._rng_state.data_ptr()

    def seed(self, seed: int) -> None:
        """Seed of the device generator (the reference seeds torch globally, helpers.py:95-106).  Key and counter are
        device-resident: step graphs captured earlier draw from the new key on their next replay.  Data-parallel
        shards must differ: seed each rank with `cfg.seed + rank` (isaac_b200.parallel.rank_seed)."""
        self._rng_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        signed = self._rng_seed - (1 << 64) if self._rng_seed >= (1 << 63) else self._rng_seed
        self._rng_state.copy_(torch.tensor([0, signed], dtype=torch.int64), non_blocking=False)

    # ------------------------------------------------------------------ the hot path
    def step(self, actions: torch.Tensor):
        """hector_env.py:158-169 + legged_robot.py:84-108."""
        self._st = self._stream()
        staged = actions.device != self.device or actions.dtype != torch.float32 or not actions.is_contiguous()
        if staged:
            actions = actions.to(self.device, dtype=torch.float32).contiguous()
        self.common_step_counter += 1
        push = bool(self.cfg.domain_rand.push_robots) and (self.common_step_counter % self.push_interval == 0)
        if self._graphs is not None and not push and self._injected is None and not self._hooks_overridden():
            return self._step_graph(actions, staged)
        return self._in_sequence(self._step_eager, actions, push)

    def _step_eager(self, actions, push):
        lib, st = self._lib, self._st
        _lib.check(lib.hb_env_action_prologue(self._pp, self._pb, actions.data_ptr(), self._pn, st),
                   "hb_env_action_prologue")
        phys, torques, pd, pp, pb = self.physics, self.torques, lib.hb_env_compute_torques, self._pp, self._pb
        for i in range(self.cfg.control.decimation):
            rc = pd(pp, pb, st)                   # _compute_torques, legged_robot.py:94
            if rc:
                _lib.check(rc, "hb_env_compute_torques")
            phys.set_dof_actuation_force(torques)
            if i == 0:
                self._apply_pending_resets()      # gym.set_*_indexed of the previous step's resets
            phys.simulate()
            phys.refresh_dof_state()
        self.post_physics_step(push)
        return self.obs_buf, self.privileged_obs_buf, self.rew_buf, self.reset_buf, self.extras

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def enable_cuda_graph(self):
        """Replay the step's launch sequence from CUDA graphs, for physics stages that need no host work between
        the decimation sub-steps (`physics.capturable`, e.g. the synthetic stage used by tests and bench.py).
        Two graphs per step: A = action prologue + first PD sub-step (one kernel); then the host hands the
        previous step's reset ids to the physics stage (legged_robot.py:370-372,394-396) while A runs; B = the
        remaining PD launches, post-physics, the frame-stack shift with the reset finalisation.  B is captured on
        first use for each (previous buffers, next buffers) pair - two for the env's own ping-pong pair, one per
        slot when the rollout storage supplies the buffers.  Push steps (every `push_interval`) and steps with
        injected noise take the eager path."""
        if not getattr(self.physics, "capturable", False):
            raise ValueError("this physics stage needs host calls between sub-steps; CUDA-graph replay is not possible")
        if self.device.type != "cuda":
            raise ValueError("CUDA graphs need a CUDA device")
        self._g_actions = torch.zeros(self.num_envs, self.num_actions, device=self.device)   # staging for odd inputs
        self._apply_pending_resets()
        torch.cuda.synchronize(self.device)
        self._g_nz = EnvNoise()
        self._bind_device_rng(self._g_nz)
        self._graphs_a, self._graphs = {}, {}
        self._graph_a(self._g_actions)
        self._graph_b(self._own[0], self._own[1]), self._graph_b(self._own[1], self._own[0])
        self.graph_launches_per_step = self.cfg.control.decimation + 2     # this library's kernels per replayed step (prologue+PD, PD x9, post, stack+finalize)

    def prepare_action_buffers(self, *tensors) -> None:
        """Capture the step's first graph for each of these action tensors now ([N, num_actions] fp32, contiguous, on
        the device) instead of at their first step() - e.g. the rollout storage's action slots."""
        if self._graphs is None:
            raise ValueError("enable_cuda_graph() first")
        for t in tensors:
            if (t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous()
                    or t.shape != self._g_actions.shape):
                raise ValueError(f"action buffers must be contiguous [{self.num_envs}, {self.num_actions}] fp32 tensors on {self.device}")
            self._graph_a(t)

    def _graph_a(self, actions):
        """Graph A reads the actions where the caller left them (one graph per address: the rollout storage's
        action slots, a policy's output buffer): no staging copy in front of the step."""
        key = actions.data_ptr()
        g = self._graphs_a.get(key)
        if g is None:
            if len(self._graphs_a) >= 256:
                self._graphs_a.clear()
            g = self._graphs_a[key] = _lib.LaunchGraph(self.device).record(lambda st: _lib.check(
                self._lib.hb_env_prologue_torques(self._pp, self._pb, key, C.byref(self._g_nz), st), "hb_env_prologue_torques"))
        return g

    def _graph_b(self, prev, out):
        key = (prev.key, out.key)
        entry = self._graphs.get(key)
        if entry is None:
            if len(self._graphs) >= 256:      # buffers keep changing (new storage): drop the stale graphs
                self._graphs.clear()
            def launches(st):
                for _ in range(self.cfg.control.decimation - 1):
                    _lib.check(self._lib.hb_env_compute_torques(self._pp, self._pb, st), "hb_env_compute_torques")
                self._launch_post_kernels(HB_STAGE_STEP, self._g_nz, prev, out, True, st)
            gb = _lib.LaunchGraph(self.device).record(launches)
            entry = self._graphs[key] = (gb, prev, out)      # the graph keeps its buffers alive
        return entry[0]

    def _step_graph(self, actions, staged=False):
        if actions.shape != self._g_actions.shape:
            raise ValueError(f"actions must be [{self.num_envs}, {self.num_actions}]")
        if staged:          # a converted temporary: its address is not worth a graph of its own
            self._g_actions.copy_(actions, non_blocking=True)
            actions = self._g_actions
        st = self._st
        self._graph_a(actions).replay(st)
        self._apply_pending_resets()          # gym.set_*_indexed of the previous step's resets
        out = self._take_output()
        self._graph_b(self._cur_buf, out).replay(st)
        self._cur_buf = out
        self._after_finalize()
        return out.obs, out.priv, self.rew_buf, self.reset_buf, self.extras

    def _compute_torques(self, actions=None):
        """legged_robot.py:339-355 on self.actions (one decimation sub-step)."""
        _lib.check(self._lib.hb_env_compute_torques(self._pp, self._pb, self._stream()), "hb_env_compute_torques")
        return self.torques

    def post_physics_step(self, push: bool = False):
        """legged_robot.py:118-153 (termination, rewards, resets, observations, last_* copies): ONE fused launch plus the
        frame-stack / finalisation launch.  If a subclass overrides one of the reference's hooks (check_termination,
        compute_reward, reset_idx, compute_observations), the step instead calls the hooks one after the other in the
        reference's order, each a launch of the same kernel restricted to that span - same results and the same draws,
        all taken in one launch sequence (_in_sequence): the reset inside it does not advance the counter, the frame-stack
        launch of compute_observations does."""
        self.physics.refresh_post_physics()
        if not self._hooks_overridden():
            self._in_sequence(self._launch_post, HB_STAGE_STEP | (HB_STAGE_PUSH if push else 0))
        else:
            self._in_sequence(self._post_physics_step_staged, push)
        if push:
            self.physics.set_root_state()

    # ------------------------------------------------------------------ the reference's hooks, one by one
    _HOOKS = ("check_termination", "compute_reward", "reset_idx", "compute_observations")

    def _hooks_overridden(self) -> bool:
        cls = type(self)
        flag = cls.__dict__.get("_hooks_overridden_cache")
        if flag is None:
            flag = any(getattr(cls, h) is not getattr(HectorFreeEnvB200, h) for h in self._HOOKS)
            cls._hooks_overridden_cache = flag
        return flag

    def _launch_stage(self, stages: int) -> None:
        """One launch of the post-physics kernel restricted to `stages` (PREPARE / TERMINATION / REWARD / LAST bits): it
        resets nothing, so no finalisation launch follows and the extras ring does not advance."""
        _lib.check(self._lib.hb_env_post_physics(self._pp, self._pb, self._pn, *self._cur_buf.key, stages, self._stream()),
                   "hb_env_post_physics")        # the current buffers are not written: no HB_STAGE_OBS bit

    def _post_physics_step_staged(self, push: bool) -> None:
        """post_physics_step as the reference spells it (legged_robot.py:118-153), through the overridable hooks."""
        self._measure_heights(self._stream())
        self._launch_stage(HB_STAGE_PREPARE | (HB_STAGE_PUSH if push else 0))      # :127-137
        self.check_termination()                                                   # :139
        self.compute_reward()                                                      # :140
        env_ids = self.reset_buf.nonzero(as_tuple=False).flatten()                 # :142
        self.reset_idx(env_ids)                                                    # :143
        self.compute_observations()                                                # :144
        self._launch_stage(HB_STAGE_LAST)                                          # :146-150

    def check_termination(self):
        """legged_robot.py:155-160: reset_buf = contact on a termination body | time-out; time_out_buf."""
        self._in_sequence(self._launch_stage, HB_STAGE_TERMINATION)

    def compute_reward(self):
        """legged_robot.py:216-234: rew_buf, episode_sums (alphabetical accumulation over the 18 active terms) and the
        stateful reward buffers (feet_air_time, last_contacts, feet_height, last_feet_z)."""
        self._in_sequence(self._launch_stage, HB_STAGE_REWARD)

    def compute_observations(self):
        """hector_env.py:172-254: the newest obs / privileged frames from the current state, pushed onto the 15-frame
        histories (the frame-stack launch)."""
        self._in_sequence(self._launch_post, HB_STAGE_OBS)

    def _launch_post(self, stages: int, advance: bool = True):
        """The post-physics launch restricted to `stages` and its finalize launch, on the bound draws (`_nz`)."""
        emit = bool(stages & (HB_STAGE_STEP | HB_STAGE_OBS))
        prev = self._cur_buf
        out = self._take_output() if emit else self._own[1 if prev is self._own[0] else 0]
        self._launch_post_kernels(stages, self._nz, prev, out, emit, self._stream(), advance)
        if emit:
            self._cur_buf = out
        self._after_finalize()

    def _launch_post_kernels(self, stages, nz, prev, out, emit, st, advance=True):
        """post-physics -> frame-stack shift + reset finalisation, on one stream, with the draws of the EnvNoise `nz`;
        prev / out = _BufferPair.  The finalize launch advances the generator counter unless `advance` is false."""
        lib = self._lib
        obs_new, priv_new = out.key
        if stages & HB_STAGE_STEP:
            self._measure_heights(st)        # _post_physics_step_callback, before anything is reset (legged_robot.py:315-316)
        _lib.check(lib.hb_env_post_physics(self._pp, self._pb, C.byref(nz), obs_new, priv_new, stages, st),
                   "hb_env_post_physics")
        counter = nz.rng_counter if advance else None
        if emit:        # shift + shard-wide reset results in one launch
            _lib.check(lib.hb_env_stack_finalize(self._pp, self._pb, *prev.key, obs_new, priv_new, self._host_count.data_ptr(),
                                                 counter, st), "hb_env_stack_finalize")
        else:
            _lib.check(lib.hb_env_reset_finalize(self._pp, self._pb, None, None, self._host_count.data_ptr(),
                                                 counter, st), "hb_env_reset_finalize")

    def _after_finalize(self):
        """Host side of a finalize launch: the extras slot it filled (the device ring cursor advances with _step_index),
        the event the reset count waits on, and time_outs."""
        if self._events:
            self._pending_event = self._events[self._step_index & 1]
            self._pending_event.record(torch.cuda.current_stream(self.device))
        self.extras["episode"] = self._extras_episode[self._step_index % _EXTRAS_RING]
        if self.cfg.env.send_timeouts:
            self.extras["time_outs"] = self._time_outs_latched
        self._step_index += 1

    def _apply_pending_resets(self):
        """The two opaque calls of _reset_dofs/_reset_root_states (legged_robot.py:370-372,394-396) need
        the reset count on the host; it is read from pinned memory once the producing kernel is done."""
        if self._pending_event is None:
            return
        self._pending_event.synchronize()
        self._pending_event = None
        n = int(self._host_count[0])
        self.last_reset_count = n
        if n > 0:
            self.physics.set_dof_state_indexed(self.reset_env_ids, n)
            self.physics.set_root_state_indexed(self.reset_env_ids, n)

    # ------------------------------------------------------------------ reference-named API
    @property
    def episode_length_buf(self):
        return self._episode_length_buf

    @episode_length_buf.setter
    def episode_length_buf(self, value):
        """The runner REBINDS this attribute (`env.episode_length_buf = torch.randint_like(...)`,
        on_policy_runner.py:103-106); the kernels address the original buffer, so the new values are copied into it."""
        self._episode_length_buf.copy_(torch.as_tensor(value).to(self._episode_length_buf.device, dtype=torch.long))

    @property
    def obs_buf(self):
        return self._cur_buf.obs

    @property
    def privileged_obs_buf(self):
        return self._cur_buf.priv

    def get_observations(self):
        return self.obs_buf

    def get_privileged_observations(self):
        return self.privileged_obs_buf

    def reset_idx(self, env_ids):
        """legged_robot.py:162-214 + hector_env.py:256-261 for an explicit id list.  Called on its own, it is a launch
        sequence: it takes its draws at the current counter and advances it; inside the staged step it draws at the
        step's counter and leaves the advance to compute_observations (_in_sequence)."""
        env_ids = torch.as_tensor(env_ids, device=self.device, dtype=torch.long)
        if env_ids.numel() == 0:
            return
        self.reset_buf.zero_()
        self.reset_buf[env_ids] = True
        self._in_sequence(self._launch_post, HB_STAGE_RESET_MASK, not self._draws_bound)
        for hist in (self._cur_buf.obs, self._cur_buf.priv):
            hist[env_ids] = 0.0
        self._apply_pending_resets()

    def reset(self):
        """legged_robot.py:111-116: reset all robots, then one step with zero actions."""
        self.reset_idx(torch.arange(self.num_envs, device=self.device))
        obs, priv, _, _, _ = self.step(torch.zeros(self.num_envs, self.num_actions, device=self.device))
        return obs, priv

    # ------------------------------------------------------------------ terrain heights (legged_robot.py:744-795)
    def set_height_field(self, height_samples, measured_points_x=None, measured_points_y=None) -> None:
        """Install the terrain's int16 height field (`Terrain.heightsamples` viewed [tot_rows, tot_cols],
        legged_robot.py:569,585) and the sampling grid of `_init_height_points` (:744-757; defaults:
        cfg.terrain.measured_points_x / _y).  From then on `_get_heights()` works and, when cfg.terrain.measure_heights is
        set, `measured_heights` is refreshed every step like `_post_physics_step_callback` does (:315-316)."""
        t = self.cfg.terrain
        xs = list(measured_points_x if measured_points_x is not None else t.measured_points_x)
        ys = list(measured_points_y if measured_points_y is not None else t.measured_points_y)
        self.height_samples = torch.as_tensor(height_samples).to(device=self.device, dtype=torch.int16).contiguous()
        if self.height_samples.dim() != 2:
            raise ValueError("height_samples must be [tot_rows, tot_cols]")
        gx, gy = torch.meshgrid(torch.tensor(xs, dtype=torch.float32), torch.tensor(ys, dtype=torch.float32), indexing="ij")
        self.num_height_points = gx.numel()
        self.height_points = torch.zeros(self.num_envs, self.num_height_points, 3, device=self.device)
        self.height_points[:, :, 0] = gx.flatten().to(self.device)
        self.height_points[:, :, 1] = gy.flatten().to(self.device)
        self._height_points_xy = self.height_points[0, :, :2].contiguous()        # the grid is the same for every env
        self.measured_heights = torch.zeros(self.num_envs, self.num_height_points, device=self.device)

    def _measure_heights(self, st) -> None:
        """measured_heights = _get_heights() of the callback (legged_robot.py:315-316), when the config asks for it; a
        plain launch on `st`, so it also sits in the captured step graph."""
        if getattr(self.cfg.terrain, "measure_heights", False) and getattr(self, "height_samples", None) is not None:
            self._launch_get_heights(None, self.measured_heights, st)

    def _launch_get_heights(self, ids, out, st) -> None:
        """Heights under the grid of points into `out`: of every env, or of the int32 env ids `ids`."""
        t = self.cfg.terrain
        _lib.check(self._lib.hb_env_get_heights(self.root_states.data_ptr(), self._height_points_xy.data_ptr(),
                                                self.num_height_points, self.height_samples.data_ptr(),
                                                self.height_samples.shape[0], self.height_samples.shape[1],
                                                float(t.border_size), float(t.horizontal_scale), float(t.vertical_scale),
                                                None if ids is None else ids.data_ptr(), out.shape[0], out.data_ptr(), st),
                   "hb_env_get_heights")

    def _get_heights(self, env_ids=None):
        """legged_robot.py:759-795: terrain height under the grid of points around each robot -> [N, P] (or [len(env_ids),
        P]; the reference's own env_ids branch cannot run, it ends in `.view(self.num_envs, -1)`)."""
        t = self.cfg.terrain
        if t.mesh_type == "plane":
            return torch.zeros(self.num_envs, getattr(self, "num_height_points", 0), device=self.device)
        if t.mesh_type == "none":
            raise NameError("Can't measure height with terrain mesh type 'none'")
        if getattr(self, "height_samples", None) is None:
            raise RuntimeError("no height field installed: call set_height_field(terrain.heightsamples ...) first")
        ids = None if env_ids is None else torch.as_tensor(env_ids, device=self.device, dtype=torch.int32).contiguous()
        out = self.measured_heights if ids is None else torch.empty(ids.numel(), self.num_height_points, device=self.device)
        self._launch_get_heights(ids, out, self._stream())
        return out

    @property
    def last_rigid_state(self):
        """Never read by the hector task (SURVEY.md §8 a9): materialised on demand only."""
        return self.rigid_state.clone()


class HectorFullFreeEnvB200(HectorFreeEnvB200):
    """`hector_full` (envs/custom/hector_w_arm_env.py): the 18-DOF robot with arms; same step, `HectorFullCfg`."""


class XBotLFreeEnvB200(HectorFreeEnvB200):
    """`humanoid_ppo` / XBot-L (envs/custom/humanoid_env.py): 12 DOF, reference-trajectory error in the privileged frame,
    critic history of 3 frames; same step, `XBotLCfg`."""
