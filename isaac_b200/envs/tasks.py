"""The reference's other two tasks on the same kernels (SURVEY.md §8f rank 4; reference registry: envs/__init__.py:46-48).

    hector        HectorFreeEnv      10 DOF, frames 41 / 70, stacks 15 / 15      envs/custom/hector_env.py, hector_config.py
    hector_full   HectorFullFreeEnv  18 DOF, frames 65 / 94, stacks 15 / 15      envs/custom/hector_w_arm_env.py, hector_w_arm_config.py
    humanoid_ppo  XBotLFreeEnv       12 DOF, frames 47 / 73, stacks 15 / 3       envs/custom/humanoid_env.py, humanoid_config.py

The env step is the same code for all three (the two hector tasks even share their env file but for joint indices, the
arm term of default_joint_pos and the reward table); what differs is collected in a `TaskLayout`: joint count, where the
privileged frame keeps its columns, and the joint-index constants the env files spell out literally.  Configs restate the
values of the reference's config files as overrides of `HectorCfg` (only what the hot path reads).

Any other robot whose env file is a copy of hector_env.py or humanoid_env.py runs on the same kernels: its config carries
`layout = TaskLayout(...)` with its joint count (up to MAX_DOF) and joint indices (INTEGRATION.md §1).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Tuple

from .._lib import HB_TASK_HECTOR, HB_TASK_XBOT
from .hector_config import HectorCfg, HectorCfgPPO, _Cfg

# the observation frame 3 ndof + 11 fits the kernels' 80 columns (HB_MAX_OBS); more joints would move the device draws
MAX_DOF = 23


@dataclass(frozen=True)
class TaskLayout:
    name: str
    kind: int                               # HB_TASK_HECTOR / HB_TASK_XBOT: layout of the privileged frame
    ndof: int
    yaw_roll: Tuple[int, int]               # default_joint_pos: first joint of each leg's (yaw, roll) pair
    arm_pair: Tuple[int, int]               # hector_full: first joint of each arm's pair; (-1, -1) otherwise
    ref_left: Tuple[int, int, int]          # compute_ref_state: joints following the negative / positive half of the gait sine
    ref_right: Tuple[int, int, int]
    # _get_noise_scale_vec, literally: (start, stop) of the dof_pos, dof_vel, zeroed-actions, ang_vel and quat assignments
    noise_slices: Tuple[Tuple[int, int], ...]

    def __post_init__(self):
        def bad(field, why):
            raise ValueError(f"TaskLayout {self.name!r}: {field} = {getattr(self, field)!r}: {why}")

        if self.kind not in (HB_TASK_HECTOR, HB_TASK_XBOT):
            bad("kind", "HB_TASK_HECTOR (hector_env.py frames) or HB_TASK_XBOT (humanoid_env.py frames)")
        if not isinstance(self.ndof, int) or not 1 <= self.ndof <= MAX_DOF:
            bad("ndof", f"1 to {MAX_DOF} joints (the observation frame 3 ndof + 11 must fit 80 columns)")
        pair = lambda j: isinstance(j, int) and 0 <= j and j + 1 < self.ndof
        if len(self.yaw_roll) != 2 or not all(pair(j) for j in self.yaw_roll):
            bad("yaw_roll", f"two first joints j of a (yaw, roll) pair, 0 <= j and j + 1 < ndof = {self.ndof}")
        if tuple(self.arm_pair) != (-1, -1) and (len(self.arm_pair) != 2 or not all(pair(j) for j in self.arm_pair)):
            bad("arm_pair", f"(-1, -1) without arms, else two first joints j with 0 <= j and j + 1 < ndof = {self.ndof}")
        for field in ("ref_left", "ref_right"):
            v = getattr(self, field)
            if len(v) != 3 or not all(isinstance(j, int) and 0 <= j < self.ndof for j in v):
                bad(field, f"three joint indices in [0, ndof = {self.ndof})")
        # (a stop past the frame is clipped, as numpy / torch slicing does: hector_env.py:155 assigns [38:42] of 41 columns)
        if len(self.noise_slices) != 5 or not all(len(s) == 2 and 0 <= s[0] < self.num_single_obs and s[0] <= s[1]
                                                  for s in self.noise_slices):
            bad("noise_slices", f"five (start, stop) pairs, 0 <= start < num_single_obs = {self.num_single_obs}, start <= stop "
                "(dof_pos, dof_vel, actions, ang_vel, quat)")

    def check_config(self, cfg) -> None:
        """ValueError naming the first config field that disagrees with this layout."""
        want = {"env.num_actions": self.ndof, "env.num_single_obs": self.num_single_obs,
                "env.single_num_privileged_obs": self.num_single_priv}
        got = {"env.num_actions": cfg.env.num_actions, "env.num_single_obs": cfg.env.num_single_obs,
               "env.single_num_privileged_obs": cfg.env.single_num_privileged_obs}
        names = getattr(getattr(cfg, "asset", None), "dof_names", None)
        if names is not None:
            want["asset.dof_names"], got["asset.dof_names"] = f"{self.ndof} names", f"{len(names)} names"
        for k in want:
            if got[k] != want[k]:
                raise ValueError(f"config field {k} = {got[k]} does not match TaskLayout {self.name!r} (ndof = {self.ndof}, "
                                 f"kind = {self.kind}): expected {want[k]}")

    @property
    def num_single_obs(self) -> int:
        return 5 + 3 * self.ndof + 6

    @property
    def num_single_priv(self) -> int:
        return 3 * self.ndof + 40 if self.kind == HB_TASK_HECTOR else 4 * self.ndof + 25


# hector_env.py:100-107,145-155,363-364
HECTOR = TaskLayout("hector", HB_TASK_HECTOR, 10, (0, 5), (-1, -1), (2, 3, 4), (7, 8, 9),
                    ((5, 15), (15, 25), (25, 35), (35, 38), (38, 42)))
# hector_w_arm_env.py:107-114 (the right-leg indices are the 10-DOF file's: they land on arm joints, the term has scale 0),
# :157-161 (the ang_vel slice starts one column early, inside the action block), :370-373
HECTOR_FULL = TaskLayout("hector_full", HB_TASK_HECTOR, 18, (0, 9), (5, 14), (2, 3, 4), (7, 8, 9),
                         ((5, 23), (23, 41), (41, 59), (58, 61), (61, 65)))
# humanoid_env.py:131-138,181-185,368-369
XBOT = TaskLayout("humanoid_ppo", HB_TASK_XBOT, 12, (0, 6), (-1, -1), (2, 3, 4), (8, 9, 10),
                  ((5, 17), (17, 29), (29, 41), (41, 44), (44, 47)))


def layout_for(cfg) -> TaskLayout:
    """The layout of a config: `cfg.layout` when it has one (checked against the config), else one of the three robots,
    recognised by its dimensions (this module's configs or the reference's own config objects)."""
    explicit = getattr(cfg, "layout", None)
    if isinstance(explicit, TaskLayout):
        explicit.check_config(cfg)
        return explicit
    for lay in (HECTOR, HECTOR_FULL, XBOT):
        if (cfg.env.num_actions == lay.ndof and cfg.env.num_single_obs == lay.num_single_obs
                and cfg.env.single_num_privileged_obs == lay.num_single_priv):
            return lay
    raise ValueError(
        f"num_actions={cfg.env.num_actions}, frames {cfg.env.num_single_obs} / {cfg.env.single_num_privileged_obs} is none of "
        "the built robots (hector 10/41/70, hector_full 18/65/94, XBot-L 12/47/73): describe the robot in its config, e.g. "
        "cfg.layout = TaskLayout(name='my_robot', kind=HB_TASK_HECTOR, ndof=12, yaw_roll=(0, 6), arm_pair=(-1, -1), "
        "ref_left=(2, 3, 4), ref_right=(8, 9, 10), noise_slices=((5, 17), (17, 29), (29, 41), (41, 44), (44, 47))) "
        f"(isaac_b200.envs.tasks; up to {MAX_DOF} joints; INTEGRATION.md §1)")


_LEG = ["hip_joint", "hip_roll_joint", "thigh_joint", "calf_joint", "toe_joint"]
_ARM = ["shoulder_yaw_joint", "shoulder_pitch_joint", "shoulder_roll_joint", "elbow_joint"]


class HectorFullCfg(HectorCfg):
    """hector_w_arm_config.py:4-200 as a delta over HectorCfg."""

    class env(HectorCfg.env):
        num_single_obs = 65
        num_observations = 15 * 65
        single_num_privileged_obs = 94
        num_privileged_obs = 15 * 94
        num_actions = 18

    class asset(HectorCfg.asset):
        terminate_after_contacts_on = ["base", "thigh", "shoulder", "twist", "roll"]
        # What Isaac Gym reports for resources/robots/hector_v2/xacro/robot_w_arm.urdf after collapse_fixed_joints: children in
        # alphabetical link order, depth first (legs before the arm of the same side: L_hip.. < L_twist.. < R_hip.. < R_twist..),
        # which is the joint order the env file indexes (hector_w_arm_env.py:370-373: arms at 5:7 / 14:16, right leg at 9:11)
        body_names = (["base"] + ["L_hip", "L_hip2", "L_thigh", "L_calf", "L_toe", "L_twist", "L_shoulder", "L_roll", "L_elbow"]
                      + ["R_hip", "R_hip2", "R_thigh", "R_calf", "R_toe", "R_twist", "R_shoulder", "R_roll", "R_elbow"])
        dof_names = [f"{side}_{j}" for side in ("L", "R") for j in _LEG + _ARM]
        dof_effort = [33.5, 33.5, 33.5, 67.0, 33.5, 17.0, 17.0, 17.0, 17.0, 33.5, 33.5, 33.5, 67.0, 33.5, 17.0, 17.0, 17.0, 24.0]

    class terrain(HectorCfg.terrain):
        mesh_type = "plane"

    class init_state(HectorCfg.init_state):
        default_joint_angles = dict(HectorCfg.init_state.default_joint_angles, **{
            f"{side}_{j}": (-0.785 if j == "elbow_joint" else 0.0) for side in ("L", "R") for j in _ARM})

    class control(HectorCfg.control):
        stiffness = {"hip_joint": 80.0, "hip_roll": 80.0, "thigh": 80.0, "calf": 80.0, "toe": 60.0,
                     "shoulder_yaw": 30.0, "shoulder_pitch": 30.0, "shoulder_roll": 30.0, "elbow": 30.0}
        damping = {"hip_joint": 5.0, "hip_roll": 5.0, "thigh": 5.0, "calf": 5.0, "toe": 3.0,
                   "shoulder_yaw": 3.0, "shoulder_pitch": 3.0, "shoulder_roll": 3.0, "elbow": 3.0}

    class domain_rand(HectorCfg.domain_rand):
        friction_range = [0.1, 2.0]
        added_mass_range = [-1.0, 4.0]
        max_push_vel_xy = 0.5

    class commands(HectorCfg.commands):
        class ranges(HectorCfg.commands.ranges):
            lin_vel_x = [-0.6, 0.8]

    class rewards(HectorCfg.rewards):
        min_dist = 0.2
        max_contact_force = 200

        class scales(HectorCfg.rewards.scales):
            feet_clearance = 1.2
            feet_contact_number = 1.5
            feet_air_time = 1.5
            feet_contact_forces = -0.02
            tracking_lin_vel = 1.2
            tracking_ang_vel = 1.1
            vel_mismatch_exp = 0.5
            low_speed = 0.2
            track_vel_hard = 0.5
            default_joint_pos = 1.2
            orientation = 1.0
            base_height = 0.8
            base_acc = 0.22
            action_smoothness = -0.002
            dof_vel = -1e-3
            collision = -1.0


class HectorFullCfgPPO(HectorCfgPPO):
    """hector_w_arm_config.py:207-244."""

    class policy(HectorCfgPPO.policy):
        actor_hidden_dims = [768, 512, 128]
        critic_hidden_dims = [768, 768, 768]

    class algorithm(HectorCfgPPO.algorithm):
        entropy_coef = 0.01
        num_learning_epochs = 5
        learning_rate = 1e-3
        gamma = 0.99
        lam = 0.95

    class runner(HectorCfgPPO.runner):
        experiment_name = "hector_arm"


_XLEG = ["leg_roll_joint", "leg_yaw_joint", "leg_pitch_joint", "knee_joint", "ankle_pitch_joint", "ankle_roll_joint"]


class XBotLCfg(HectorCfg):
    """humanoid_config.py:34-214 as a delta over HectorCfg."""

    class env(HectorCfg.env):
        c_frame_stack = 3
        num_single_obs = 47
        num_observations = 15 * 47
        single_num_privileged_obs = 73
        num_privileged_obs = 3 * 73
        num_actions = 12

    class safety(HectorCfg.safety):
        pos_limit = 1.0
        vel_limit = 1.0

    class asset(HectorCfg.asset):
        name = "XBot-L"
        foot_name = "ankle_roll"
        knee_name = "knee"
        terminate_after_contacts_on = ["base_link"]
        penalize_contacts_on = ["base_link"]
        # resources/robots/XBot/urdf/XBot-L.urdf after collapse_fixed_joints: only the two legs keep their joints
        body_names = ["base_link"] + [f"{side}_{j.replace('_joint', '_link')}" for side in ("left", "right") for j in _XLEG]
        dof_names = [f"{side}_{j}" for side in ("left", "right") for j in _XLEG]
        dof_effort = [100.0, 100.0, 250.0, 250.0, 100.0, 100.0] * 2

    class init_state(HectorCfg.init_state):
        pos = [0.0, 0.0, 0.95]
        default_joint_angles = {f"{side}_{j}": 0.0 for side in ("left", "right") for j in _XLEG}

    class control(HectorCfg.control):
        stiffness = {"leg_roll": 200.0, "leg_pitch": 350.0, "leg_yaw": 200.0, "knee": 350.0, "ankle": 15}
        damping = {"leg_roll": 10, "leg_pitch": 10, "leg_yaw": 10, "knee": 10, "ankle": 10}

    class domain_rand(HectorCfg.domain_rand):
        friction_range = [0.1, 2.0]
        added_mass_range = [-5.0, 5.0]
        max_push_vel_xy = 0.2
        action_delay = 0.5

    class commands(HectorCfg.commands):
        class ranges(HectorCfg.commands.ranges):
            lin_vel_x = [-0.3, 0.6]

    class rewards(HectorCfg.rewards):
        base_height_target = 0.89
        min_dist = 0.2
        max_contact_force = 700

        class scales(HectorCfg.rewards.scales):
            joint_pos = 1.6
            feet_clearance = 1.0
            feet_contact_number = 1.2
            feet_air_time = 1.0
            feet_contact_forces = -0.01
            tracking_lin_vel = 1.2
            tracking_ang_vel = 1.1
            vel_mismatch_exp = 0.5
            low_speed = 0.2
            track_vel_hard = 0.5
            default_joint_pos = 0.5
            orientation = 1.0
            base_height = 0.2
            base_acc = 0.2
            action_smoothness = -0.002
            dof_vel = -5e-4
            dof_acc = -1e-7
            collision = -1.0

    class normalization(HectorCfg.normalization):
        clip_observations = 18.0
        clip_actions = 18.0


class XBotLCfgPPO(HectorCfgPPO):
    """humanoid_config.py:217-261."""

    class runner(HectorCfgPPO.runner):
        max_iterations = 3001
        experiment_name = "XBot_ppo"


# envs/__init__.py:46-48: task name -> (env class name here, env config, train config)
TASKS = {
    "hector": ("HectorFreeEnvB200", HectorCfg, HectorCfgPPO),
    "hector_full": ("HectorFullFreeEnvB200", HectorFullCfg, HectorFullCfgPPO),
    "humanoid_ppo": ("XBotLFreeEnvB200", XBotLCfg, XBotLCfgPPO),
}
__all__ = ["TaskLayout", "MAX_DOF", "HECTOR", "HECTOR_FULL", "XBOT", "layout_for", "HectorFullCfg", "HectorFullCfgPPO", "XBotLCfg",
           "XBotLCfgPPO", "TASKS", "_Cfg"]
