"""ctypes binding of libhectorb200.so (the C ABI declared in include/hector_b200.h).

There is no CPU fallback: if the library is missing or the device is not sm_100,
`load()` raises.  Structures mirror the header field by field; `load()` checks
`sizeof` against the library so a drift between header and mirror fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HB_ABI_VERSION = 6
HB_MAX_DOF = 24
HB_MAX_OBS = 80
HB_NUM_REWARDS = 22
HB_MAX_CONTACT_BODIES = 16
HB_TASK_HECTOR, HB_TASK_XBOT = 0, 1

HB_STAGE_STEP = 0x1
HB_STAGE_RESET_ALL = 0x2
HB_STAGE_PUSH = 0x4
HB_STAGE_OBS = 0x8
HB_STAGE_DERIVE = 0x10
HB_STAGE_RESET_MASK = 0x20
HB_STAGE_PREPARE, HB_STAGE_TERMINATION, HB_STAGE_REWARD, HB_STAGE_LAST = 0x40, 0x80, 0x100, 0x200

# alphabetical = the reference's accumulation order (utils/helpers.py:47)
REWARD_NAMES = ("action_smoothness", "base_acc", "base_height", "collision", "default_joint_pos", "dof_acc",
                "dof_vel", "feet_air_time", "feet_clearance", "feet_contact_forces", "feet_contact_number",
                "feet_distance", "foot_slip", "joint_pos", "knee_distance", "low_speed", "orientation", "torques",
                "track_vel_hard", "tracking_ang_vel", "tracking_lin_vel", "vel_mismatch_exp")
assert len(REWARD_NAMES) == HB_NUM_REWARDS and list(REWARD_NAMES) == sorted(REWARD_NAMES)

_f, _i = C.c_float, C.c_int32
_fp = C.c_void_p   # device pointers travel as integers


class EnvParams(C.Structure):
    _fields_ = [
        ("abi_version", _i), ("num_envs", _i), ("task_kind", _i), ("num_dof", _i), ("num_bodies", _i),
        ("num_single_obs", _i), ("frame_stack", _i), ("num_single_priv", _i), ("c_frame_stack", _i),
        ("obs_ld", _i), ("priv_ld", _i),
        ("feet", _i * 2), ("knees", _i * 2),
        ("n_term", _i), ("term_bodies", _i * HB_MAX_CONTACT_BODIES),
        ("n_pen", _i), ("pen_bodies", _i * HB_MAX_CONTACT_BODIES),
        ("max_episode_length", _i), ("resample_interval", _i), ("heading_command", _i), ("add_noise", _i),
        ("only_positive_rewards", _i), ("custom_origins", _i),
        ("yaw_roll", _i * 2), ("arm_pair", _i * 2), ("ref_left", _i * 3), ("ref_right", _i * 3),
        ("action_scale", _f), ("clip_actions", _f), ("clip_observations", _f), ("action_delay", _f),
        ("action_noise", _f),
        ("default_dof_pos", _f * HB_MAX_DOF), ("torque_limits", _f * HB_MAX_DOF),
        ("ref_scale", _f * 2), ("dt", _f), ("cycle_time", _f), ("max_episode_length_s", _f),
        ("cmd_lo", _f * 3), ("cmd_span", _f * 3),
        ("push_lin_lo", _f), ("push_lin_span", _f), ("push_ang_lo", _f), ("push_ang_span", _f),
        ("reset_dof_lo", _f), ("reset_dof_span", _f), ("reset_xy_lo", _f), ("reset_xy_span", _f),
        ("base_init_state", _f * 13),
        ("obs_lin_vel", _f), ("obs_ang_vel", _f), ("obs_dof_pos", _f), ("obs_dof_vel", _f), ("obs_quat", _f),
        ("noise_level", _f), ("noise_scale_vec", _f * HB_MAX_OBS),
        ("reward_scale", _f * HB_NUM_REWARDS),
        ("base_height_target", _f), ("min_dist", _f), ("max_dist", _f), ("target_feet_height", _f),
        ("tracking_sigma", _f), ("max_contact_force", _f),
        ("reset_euler", _f * 3), ("reset_gravity", _f * 3),
    ]


_BUFFER_FIELDS = (
    "root_states", "dof_state", "contact_forces", "rigid_state", "p_gains", "d_gains", "env_frictions",
    "body_mass", "env_origins", "actions", "last_actions", "last_last_actions", "last_dof_vel", "last_root_vel",
    "torques", "commands", "base_lin_vel", "base_ang_vel", "projected_gravity", "base_euler_xyz", "feet_air_time",
    "last_contacts", "feet_height", "last_feet_z", "ref_dof_pos", "rand_push_force", "rand_push_torque", "episode_sums",
    "episode_length_buf", "reset_buf", "time_out_buf", "rew_buf", "reset_env_ids", "reset_count", "episode_means",
    "episode_means_prev", "episode_ring", "time_outs_latched", "scratch_ballots", "scratch_sums")


class EnvBuffers(C.Structure):
    _fields_ = [(name, _fp) for name in _BUFFER_FIELDS]


_NOISE_FIELDS = ("u_delay", "z_action", "u_cmd", "u_push", "u_reset", "z_obs")


class EnvNoise(C.Structure):
    _fields_ = [(name, _fp) for name in _NOISE_FIELDS] + [("rng_counter", _fp)]


HB_EPI_STORE, HB_EPI_BIAS, HB_EPI_BIAS_ACT, HB_EPI_ACT_BWD, HB_EPI_ATOMIC_ADD = range(5)
HB_EPI_BIAS_ELU, HB_EPI_ELU_BWD = HB_EPI_BIAS_ACT, HB_EPI_ACT_BWD
HB_ACT_ELU, HB_ACT_SELU, HB_ACT_RELU, HB_ACT_LRELU, HB_ACT_TANH, HB_ACT_SIGMOID = range(6)      # hb_activation
PPO_MAX_ACTIONS = 64                    # hb_ppo_pack_samples / _loss_head / _act_head take 1 to 64 actions
PPO_MAX_FUSED_ACTIONS = 15              # hb_ppo_head_fused / _act_fused take 1 to 15 (one lane pair per output)


def ppo_rec(num_actions: int) -> int:
    """HB_PPO_REC(num_actions): floats of one packed sample record."""
    return 3 * num_actions + 6


HB_PPO_ACT, HB_PPO_REC = 10, ppo_rec(10)          # the hector task's values


class GemmDesc(C.Structure):
    _fields_ = [("A", _fp), ("B", _fp), ("D", _fp), ("M", _i), ("N", _i), ("K", _i), ("lda", _i), ("ldb", _i),
                ("ldd", _i), ("a_mn_major", _i), ("b_mn_major", _i), ("epilogue", _i), ("bias", _fp),
                ("bias_stride", _i), ("H", _fp), ("ldh", _i), ("split_k", _i), ("tile_n", _i), ("precision", _i),
                ("workspace", _fp), ("workspace_floats", C.c_int64), ("activation", _i)]


HB_GEMM_TF32, HB_GEMM_3XTF32 = 0, 1


class PpoLossParams(C.Structure):
    _fields_ = [("clip_param", _f), ("value_loss_coef", _f), ("entropy_coef", _f), ("use_clipped_value_loss", _i),
                ("num_actions", _i), ("activation", _i)]


class AdamParams(C.Structure):
    _fields_ = [("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double), ("max_grad_norm", _f), ("adaptive", _i),
                ("desired_kl", C.c_double), ("kl_count", C.c_int64)]


HB_OPT_TRACE_MAX = 64


class OptimState(C.Structure):
    """Layout of hb_optim_state; on the Python side it is a float64 device tensor of OPTIM_STATE_DOUBLES elements whose
    integer fields are read through an int64 view (indices below are in 8-byte words)."""
    _fields_ = [("lr", C.c_double), ("grad_sumsq", C.c_double), ("stats", C.c_double * 4), ("loss_acc", C.c_double * 4),
                ("step", C.c_int64), ("steps_in_update", C.c_int64), ("ticket", C.c_uint64), ("reserved", C.c_uint64),
                ("go", C.c_uint64), ("bcast", _f * 4), ("trace", C.c_double * (2 * HB_OPT_TRACE_MAX))]


OPTIM_STATE_DOUBLES = C.sizeof(OptimState) // 8
OPT_LR, OPT_SUMSQ, OPT_STATS, OPT_LOSS_ACC, OPT_STEP, OPT_STEPS_IN_UPDATE, OPT_TICKET, OPT_ERROR, OPT_TRACE = 0, 1, 2, 6, 10, 11, 12, 13, 17
assert OptimState.trace.offset == 8 * OPT_TRACE and OptimState.reserved.offset == 8 * OPT_ERROR

HB_DP_MAX_RANKS = 8


class DpComm(C.Structure):
    _fields_ = [("world", _i), ("rank", _i), ("grad", _fp * HB_DP_MAX_RANKS), ("param", _fp * HB_DP_MAX_RANKS),
                ("mail", _fp * HB_DP_MAX_RANKS), ("flag", _fp * HB_DP_MAX_RANKS), ("grad_mc", _fp), ("param_mc", _fp)]


class HectorB200Error(RuntimeError):
    pass


_LIB: Optional[C.CDLL] = None
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libhectorb200.so")

_SIGNATURES = {
    "hb_last_error": (C.c_char_p, []),
    "hb_abi_version": (C.c_int, []),
    "hb_launch_count": (C.c_int64, []),
    "hb_launch_count_reset": (None, []),
    "hb_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "hb_sizeof_env_params": (C.c_int, []),
    "hb_sizeof_env_buffers": (C.c_int, []),
    "hb_sizeof_env_noise": (C.c_int, []),
    "hb_sizeof_gemm_desc": (C.c_int, []),
    "hb_sizeof_adam_params": (C.c_int, []),
    "hb_sizeof_optim_state": (C.c_int, []),
    "hb_check_device": (C.c_int, []),
    "hb_graph_begin": (C.c_int, [_fp]),
    "hb_graph_end": (C.c_int, [_fp, C.POINTER(C.c_void_p)]),
    "hb_graph_launch": (C.c_int, [_fp, _fp]),
    "hb_graph_destroy": (C.c_int, [_fp]),
    "hb_env_action_prologue": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), _fp, C.POINTER(EnvNoise), _fp]),
    "hb_env_prologue_torques": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), _fp, C.POINTER(EnvNoise), _fp]),
    "hb_env_compute_torques": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), _fp]),
    "hb_env_post_physics": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), C.POINTER(EnvNoise), _fp, _fp,
                                      C.c_int32, _fp]),
    "hb_env_stack_observations": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), _fp, _fp, _fp, _fp, _fp]),
    "hb_env_reset_finalize": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), _fp, _fp, _fp, _fp, _fp]),
    "hb_env_stack_finalize": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvBuffers), _fp, _fp, _fp, _fp, _fp, _fp, _fp]),
    "hb_env_get_heights": (C.c_int, [_fp, _fp, C.c_int32, _fp, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float, _fp,
                                     C.c_int64, _fp, _fp]),
    "hb_stack_shift": (C.c_int, [_fp, _fp, _fp, C.c_int32, C.c_int32, C.c_int32, _fp]),
    "hb_copy_rows": (C.c_int, [_fp, C.c_int64, _fp, C.c_int64, C.c_int64, C.c_int64, _fp]),
    "hb_env_mirror_frames": (C.c_int, [_fp, C.c_int32, C.c_int32, C.c_int32, _fp, C.c_int32, C.c_int32, C.c_int32, _fp, C.c_int32, _fp,
                                       C.c_int32, C.c_int32, _fp, C.c_int32, C.c_int32, C.c_int32, _fp]),
    "hb_gemm_tf32": (C.c_int, [C.POINTER(GemmDesc), _fp]),
    "hb_gemm_workspace_floats": (C.c_int64, [C.POINTER(GemmDesc)]),
    "hb_gemm_tf32_grouped": (C.c_int, [C.POINTER(GemmDesc), C.POINTER(GemmDesc), _fp]),
    "hb_gemm_set_pair_mode": (C.c_int, [C.c_int]),
    "hb_ppo_gather_rows": (C.c_int, [_fp, C.c_int32, _fp, C.c_int32, _fp, C.c_int64, C.c_int32, C.c_int32, _fp]),
    "hb_ppo_pack_samples": (C.c_int, [_fp, C.c_int64, _fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, _fp, _fp]),
    "hb_ppo_loss_head": (C.c_int, [_fp, C.c_int32, _fp, C.c_int32, _fp, _fp, C.c_int64, C.c_int64,
                                   C.POINTER(PpoLossParams), _fp, _fp, _fp, _fp, _fp]),
    "hb_ppo_head_fused": (C.c_int, [_fp, C.c_int32, _fp, C.c_int32, _fp, _fp, C.c_int32, _fp, _fp, C.c_int64, C.c_int64,
                                    C.POINTER(PpoLossParams), _fp, _fp, C.c_int32, _fp, _fp, _fp, _fp, _fp]),
    "hb_ppo_act_fused": (C.c_int, [_fp, C.c_int32, _fp, C.c_int32, _fp, _fp, C.c_int32, _fp, _fp, C.c_int64, C.c_int32, _fp, _fp,
                                   _fp, _fp, _fp, _fp]),
    "hb_ppo_record_step": (C.c_int, [_fp, _fp, _fp, _fp, C.c_float, C.c_int64, _fp, _fp, _fp]),
    "hb_ppo_draw_normal": (C.c_int, [_fp, C.c_int64, _fp, _fp]),
    "hb_ppo_act_head": (C.c_int, [_fp, C.c_int32, _fp, _fp, C.c_int64, C.c_int32, _fp, _fp, _fp, _fp, _fp]),
    "hb_optimizer_step": (C.c_int, [_fp, _fp, _fp, _fp, C.c_int64, C.POINTER(AdamParams), _fp, _fp]),
    "hb_runner_bookkeeping": (C.c_int, [_fp, _fp, C.c_int64, _fp, _fp, _fp, _fp, C.c_int32, _fp, _fp]),
    "hb_dp_optimizer_step": (C.c_int, [C.POINTER(DpComm), _fp, _fp, C.c_int64, C.POINTER(AdamParams), _fp, _fp]),
    "hb_sizeof_dp_comm": (C.c_int, []),
    "hb_gae_returns": (C.c_int, [_fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, C.c_int32, C.c_float, C.c_float, _fp]),
    "hb_gae_fused": (C.c_int, [_fp, _fp, _fp, _fp, _fp, _fp, _fp, C.c_int32, C.c_int32, C.c_float, C.c_float, _fp]),
    "hb_gae_normalize": (C.c_int, [_fp, _fp, C.c_int64, _fp]),
    "hb_gae_normalize_n": (C.c_int, [_fp, _fp, C.c_int64, C.c_int64, _fp]),
}


def load(check_device: bool = False) -> C.CDLL:
    """Load the shared library (raises if it has not been built: no fallback exists)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise HectorB200Error(
                f"{LIB_PATH} is missing: build it with `python -m isaac_b200.build` "
                "(the env/GAE/PPO hot path has no CPU or eager-torch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError = symbol missing = broken build
            fn.restype, fn.argtypes = res, args
        if lib.hb_abi_version() != HB_ABI_VERSION:
            raise HectorB200Error("ABI version mismatch between libhectorb200.so and isaac_b200/_lib.py")
        for fn, cls in ((lib.hb_sizeof_env_params, EnvParams), (lib.hb_sizeof_env_buffers, EnvBuffers),
                        (lib.hb_sizeof_env_noise, EnvNoise), (lib.hb_sizeof_adam_params, AdamParams),
                        (lib.hb_sizeof_gemm_desc, GemmDesc), (lib.hb_sizeof_dp_comm, DpComm),
                        (lib.hb_sizeof_optim_state, OptimState)):
            if fn() != C.sizeof(cls):
                raise HectorB200Error(f"struct {cls.__name__}: header says {fn()} bytes, ctypes mirror {C.sizeof(cls)}")
        _LIB = lib
    if check_device:
        check(_LIB.hb_check_device(), "hb_check_device")
    return _LIB


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = _LIB.hb_last_error().decode() if _LIB is not None else ""
        raise HectorB200Error(f"{what} failed (status {rc}): {msg}")


class LaunchGraph:
    """A replayable sequence of hb_* launches (hb_graph_begin / end / launch): what `torch.cuda.CUDAGraph` does for
    this library's kernels, without its allocator / generator bookkeeping around capture and replay.  `record(fn)` runs
    `fn(stream_handle)` under capture on a private stream; only hb_* calls (no torch ops) may be issued inside."""

    _capture_stream = {}

    def __init__(self, device):
        import torch
        self._lib = load()
        self._device = torch.device(device)
        self._exec = C.c_void_p()
        s = LaunchGraph._capture_stream.get(self._device)
        if s is None:
            s = LaunchGraph._capture_stream[self._device] = torch.cuda.Stream(self._device)
        self._stream = s

    def record(self, fn) -> "LaunchGraph":
        import gc
        import torch
        torch.cuda.synchronize(self._device)
        handle = self._stream.cuda_stream
        # No cyclic garbage collection while the stream is capturing: a collection that happens to run inside the capture
        # destroys whatever unreachable CUDA objects earlier code left behind (graphs, streams, pinned buffers) from this
        # thread, and a call that is not capturable invalidates the capture ("previous error during capture").
        gc_was_on = gc.isenabled()
        gc.disable()
        try:
            with torch.cuda.stream(self._stream):       # code that asks torch for the current stream lands on the capture stream
                check(self._lib.hb_graph_begin(handle), "hb_graph_begin")
                try:
                    fn(handle)
                finally:
                    rc = self._lib.hb_graph_end(handle, C.byref(self._exec))
        finally:
            if gc_was_on:
                gc.enable()
        check(rc, "hb_graph_end")
        return self

    def replay(self, stream_handle) -> None:
        rc = self._lib.hb_graph_launch(self._exec, stream_handle)
        if rc:
            check(rc, "hb_graph_launch")

    def __del__(self):
        try:
            if self._exec:
                self._lib.hb_graph_destroy(self._exec)
        except Exception:
            pass


def exported_symbols():
    return tuple(_SIGNATURES)
