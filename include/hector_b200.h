/*
 * hector_b200.h — C ABI of libhectorb200.so
 *
 * B200 (sm_100a) implementation of the data-parallel per-environment hot path of the
 * DRCL-USC/isaac `hector` task (humanoid-gym / legged_gym / rsl_rl fork).  The reference is
 * pure Python/PyTorch and has no FFI of its own; every entry point below replaces a span of
 * the reference's Python (cited as file:line relative to /root/reference/humanoid) and is what
 * a ctypes binding on the reference side would call (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *   - plain C: raw device pointers, sizes, POD structs, a CUDA stream passed as void*
 *     (cudaStream_t; NULL = legacy default stream).  No torch types.
 *   - every function returns HB_OK (0) or a negative hb_status; nothing throws or aborts.
 *     hb_last_error() gives a static, thread-local message for the last failure.
 *   - all floating tensors are fp32, row-major, and live in device memory owned by the
 *     caller.  The gym tensors (root_states, dof_state, contact_forces, rigid_state) are
 *     owned by PhysX and are read / written in place (envs/base/legged_robot.py:437-456).
 *   - calls are asynchronous on `stream`; the only host-visible result is `host_count` of
 *     hb_env_reset_finalize (a pinned int the kernel writes; wait on the stream before reading).
 */
#ifndef HECTOR_B200_H
#define HECTOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_ABI_VERSION 6

typedef enum hb_status {
    HB_OK = 0,
    HB_ERR_BAD_ARG = -1,     /* null pointer, misaligned pointer, unsupported dimension */
    HB_ERR_CUDA = -2,        /* cudaGetLastError() after a launch, or a failed runtime call */
    HB_ERR_UNSUPPORTED = -3  /* device is not sm_100 / feature not built */
} hb_status;

#define HB_MAX_DOF 24
#define HB_MAX_OBS 80
#define HB_NUM_REWARDS 22
#define HB_MAX_CONTACT_BODIES 16

/* The tasks the reference registers (envs/__init__.py:46-48) share the env step; they differ in the number of joints,
 * the frame sizes and the layout of the privileged frame:
 *   HB_TASK_HECTOR  hector (10 DOF, frames 41 / 70, stacks 15 / 15; envs/custom/hector_env.py) and hector_full (18 DOF,
 *                   frames 65 / 94; envs/custom/hector_w_arm_env.py): feet positions / velocities and the root position
 *                   in the privileged frame
 *   HB_TASK_XBOT    humanoid_ppo / XBot-L (12 DOF, frames 47 / 73, stacks 15 / 3; envs/custom/humanoid_env.py): the
 *                   reference-trajectory error q - ref_dof_pos instead */
#define HB_TASK_HECTOR 0
#define HB_TASK_XBOT 1

/* Reward terms in the reference's accumulation order: alphabetical, because
 * utils/helpers.py:47 walks dir() (envs/base/legged_robot.py:517-540). */
enum hb_reward_id {
    HB_R_ACTION_SMOOTHNESS = 0, HB_R_BASE_ACC, HB_R_BASE_HEIGHT, HB_R_COLLISION,
    HB_R_DEFAULT_JOINT_POS, HB_R_DOF_ACC, HB_R_DOF_VEL, HB_R_FEET_AIR_TIME,
    HB_R_FEET_CLEARANCE, HB_R_FEET_CONTACT_FORCES, HB_R_FEET_CONTACT_NUMBER,
    HB_R_FEET_DISTANCE, HB_R_FOOT_SLIP, HB_R_JOINT_POS, HB_R_KNEE_DISTANCE, HB_R_LOW_SPEED, HB_R_ORIENTATION,
    HB_R_TORQUES, HB_R_TRACK_VEL_HARD, HB_R_TRACKING_ANG_VEL, HB_R_TRACKING_LIN_VEL, HB_R_VEL_MISMATCH_EXP
};

/* Task constants (envs/custom/hector_config.py:4-200, resolved the way
 * LeggedRobot._parse_cfg / _init_buffers / _prepare_reward_function do). */
typedef struct hb_env_params {
    int32_t abi_version;            /* = HB_ABI_VERSION */
    int32_t num_envs;
    int32_t task_kind;              /* HB_TASK_HECTOR / HB_TASK_XBOT */
    int32_t num_dof;                /* 10 (hector), 18 (hector_full), 12 (XBot-L) */
    int32_t num_bodies;             /* 11 / 19 / 13 after collapse_fixed_joints */
    int32_t num_single_obs;         /* 41 / 65 / 47 */
    int32_t frame_stack;            /* 15 */
    int32_t num_single_priv;        /* 70 / 94 / 73 */
    int32_t c_frame_stack;          /* 15 / 15 / 3 */
    int32_t obs_ld, priv_ld;        /* row pitch, in floats, of every obs / privileged-obs buffer handed to the calls
                                       below; 0 = dense (frame_stack * num_single_obs).  A pitch that is a multiple of
                                       4 makes the rows TMA-addressable: the buffers can be the rollout storage's own
                                       slots (rollout_storage.py:60-61), SURVEY.md §8(f) rank 1.  The host classes use
                                       whole 128-byte rows (640 / 1056 floats for hector): a TMA box row then covers 4
                                       sectors instead of 5 (layer-1 GEMM 15 % faster) */
    int32_t feet[2];                /* rigid-body rows of the feet   (legged_robot.py:668-671) */
    int32_t knees[2];               /* rigid-body rows of the knees  (:672-674) */
    int32_t n_term;                 /* termination_contact_indices   (:680-682) */
    int32_t term_bodies[HB_MAX_CONTACT_BODIES];
    int32_t n_pen;                  /* penalised_contact_indices     (:676-678) */
    int32_t pen_bodies[HB_MAX_CONTACT_BODIES];
    int32_t max_episode_length;     /* ceil(episode_length_s / dt)   (:717-718) */
    int32_t resample_interval;      /* int(resampling_time / dt)     (:308) */
    int32_t heading_command;        /* commands.heading_command */
    int32_t add_noise;              /* noise.add_noise */
    int32_t only_positive_rewards;
    int32_t custom_origins;         /* root xy jitter at reset (:381-384) */
    /* joint index constants of the reward terms, as the task's env file spells them */
    int32_t yaw_roll[2];            /* first joint of the (yaw, roll) pair of the left / right leg: default_joint_pos
                                       (hector_env.py:363-364 -> 0, 5; hector_w_arm_env.py:370-373 -> 0, 9; humanoid_env.py -> 0, 6) */
    int32_t arm_pair[2];            /* hector_full: first joint of the left / right arm pair (5, 14; :371-378); else -1.
                                       Both pairs are joint-order constants of the three robots (0, num_dof/2 and 5, num_dof/2 + 5)
                                       and are compiled into the kernels: other values are refused (HB_ERR_BAD_ARG) */
    int32_t ref_left[3], ref_right[3];   /* compute_ref_state: joints driven by the left / right half of the gait sine
                                       (hector_env.py:100-107 -> 2,3,4 / 7,8,9; humanoid_env.py:131-138 -> 2,3,4 / 8,9,10) */
    /* control (legged_robot.py:339-355) */
    float action_scale;
    float clip_actions;
    float clip_observations;
    float action_delay;             /* domain_rand.action_delay  (hector_env.py:166) */
    float action_noise;             /* domain_rand.action_noise  (hector_env.py:168) */
    float default_dof_pos[HB_MAX_DOF];
    float torque_limits[HB_MAX_DOF];
    /* time */
    float ref_scale[2];             /* target_joint_pos_scale and twice it (compute_ref_state) */
    float dt;                       /* decimation * sim.dt */
    float cycle_time;
    float max_episode_length_s;
    /* uniform draws: value = span * u + lo, u in [0,1)  (isaacgym torch_rand_float) */
    float cmd_lo[3], cmd_span[3];   /* lin_vel_x, lin_vel_y, heading */
    float push_lin_lo, push_lin_span, push_ang_lo, push_ang_span;
    float reset_dof_lo, reset_dof_span;   /* -0.15 .. 0.15 (legged_robot.py:366) */
    float reset_xy_lo, reset_xy_span;     /* -1 .. 1       (:384) */
    float base_init_state[13];
    /* observation scaling (hector_env.py:172-254) */
    float obs_lin_vel, obs_ang_vel, obs_dof_pos, obs_dof_vel, obs_quat;
    float noise_level;
    float noise_scale_vec[HB_MAX_OBS];
    /* rewards: scale already multiplied by dt; 0 = term disabled */
    float reward_scale[HB_NUM_REWARDS];
    float base_height_target, min_dist, max_dist, target_feet_height, tracking_sigma, max_contact_force;
    /* get_euler_xyz_tensor / quat_rotate_inverse(gravity) of base_init_state's quaternion: what
     * reset_idx recomputes for a freshly reset env (legged_robot.py:211-214); same for every env */
    float reset_euler[3], reset_gravity[3];
} hb_env_params;

/* Device buffers of one env shard.  Pointers marked (gym) are PhysX-owned. */
typedef struct hb_env_buffers {
    /* (gym) */
    float *root_states;             /* [N,13]  pos quat(xyzw) linvel angvel */
    float *dof_state;               /* [N*ndof,2] (pos,vel) interleaved */
    const float *contact_forces;    /* [N,nbody,3] */
    const float *rigid_state;       /* [N,nbody,13] */
    /* per-env constants */
    const float *p_gains, *d_gains; /* [N,ndof] */
    const float *env_frictions;     /* [N,1] */
    const float *body_mass;         /* [N,1] */
    const float *env_origins;       /* [N,3] */
    /* env state */
    float *actions, *last_actions, *last_last_actions;   /* [N,ndof] */
    float *last_dof_vel;            /* [N,ndof] */
    float *last_root_vel;           /* [N,6] */
    float *torques;                 /* [N,ndof] */
    float *commands;                /* [N,4] */
    float *base_lin_vel, *base_ang_vel, *projected_gravity, *base_euler_xyz;   /* [N,3] */
    float *feet_air_time;           /* [N,2] */
    uint8_t *last_contacts;         /* [N,2] bool */
    float *feet_height, *last_feet_z;   /* [N,2] */
    float *ref_dof_pos;             /* [N,ndof] reference trajectory left by the last compute_observations (compute_ref_state);
                                       needed for the joint_pos reward and the XBot-L privileged frame, else may be NULL */
    float *rand_push_force, *rand_push_torque;   /* [N,3] */
    float *episode_sums;            /* [HB_NUM_REWARDS, N] */
    int64_t *episode_length_buf;    /* [N] */
    uint8_t *reset_buf;             /* [N] bool */
    uint8_t *time_out_buf;          /* [N] bool */
    float *rew_buf;                 /* [N] */
    /* reset compaction results */
    int32_t *reset_env_ids;         /* [N] ascending ids of the envs reset this step */
    int32_t *reset_count;           /* [1] device */
    float *episode_means;           /* [HB_NUM_REWARDS] mean(episode_sums[k][ids]) / max_episode_length_s; on a step
                                       without resets the values of episode_means_prev are carried over */
    const float *episode_means_prev;/* [HB_NUM_REWARDS] or NULL */
    int32_t *episode_ring;          /* NULL, or device int32[2] = {cursor, size}: episode_means is then the base of a ring
                                       [size][HB_NUM_REWARDS]; hb_env_reset_finalize / hb_env_stack_finalize write slot
                                       `cursor`, carry over from slot cursor-1 (episode_means_prev is ignored) and
                                       advance the cursor - the launch sequence of a step can then be replayed from one
                                       CUDA graph while every step's extras["episode"] keeps its own storage until the
                                       runner logs it (on_policy_runner.py:140-154 reads them an iteration later) */
    uint8_t *time_outs_latched;     /* [N] copy of time_out_buf taken only on steps with >=1 reset (extras["time_outs"]) */
    /* scratch: ceil(N/32) ballot words (one per 32-env tile) and HB_NUM_REWARDS fp64 accumulators (zeroed
     * once by the caller; hb_env_reset_finalize re-arms them) */
    uint32_t *scratch_ballots;
    double *scratch_sums;
} hb_env_buffers;

/* Per-step random draws, indexed by env.  A NULL pointer means: drawn on the device where it is consumed, if
 * rng_counter is set (Philox4x32-10, key = rng_counter[1], counter = (env, slot, rng_counter[0]); the tensors the
 * reference would have drawn with torch.rand / randn are never materialised); otherwise treated as 0 /
 * "no such draw".  hb_env_reset_finalize advances rng_counter[0] once per call sequence.  Counter AND key live in
 * device memory, so launches captured in a CUDA graph follow a re-seed (write rng_counter[1], zero rng_counter[0]). */
typedef struct hb_env_noise {
    const float *u_delay;           /* [N]    torch.rand((N,1))            hector_env.py:166 */
    const float *z_action;          /* [N,ndof] torch.randn_like(actions)  hector_env.py:168 */
    const float *u_cmd;             /* [N,3]  command resampling           legged_robot.py:327-330 */
    const float *u_push;            /* [N,5]  push lin xy + ang xyz        hector_env.py:58-63 */
    const float *u_reset;           /* [N,ndof+5] dof(ndof) root xy(2) cmd(3)  legged_robot.py:366,384,327-330 */
    const float *z_obs;             /* [N,num_single_obs] torch.randn_like(obs_buf)    hector_env.py:241 */
    const uint64_t *rng_counter;    /* [2] device: {step counter, key} of the device generator, or NULL */
} hb_env_noise;

/* stage mask for hb_env_post_physics */
#define HB_STAGE_STEP      0x1   /* the whole of post_physics_step (legged_robot.py:118-153) */
#define HB_STAGE_RESET_ALL 0x2   /* reset_idx(all envs) + compute_observations (hector_env.py:50-51) */
#define HB_STAGE_PUSH      0x4   /* this is a push step (common_step_counter % push_interval == 0) */
#define HB_STAGE_OBS       0x8   /* emit the newest frames even without HB_STAGE_STEP */
#define HB_STAGE_RESET_MASK 0x20 /* reset_idx(env_ids): reset the envs whose reset_buf was set by the caller */
#define HB_STAGE_DERIVE    0x10  /* _init_buffers: base_lin_vel / base_ang_vel / gravity of the initial state (:477-479) */
/* The reference's overridable hooks one by one (SURVEY.md §8b): each bit runs that span of post_physics_step on the
 * current buffers, exactly as HB_STAGE_STEP does inside the fused launch.  The reference's order is PREPARE,
 * TERMINATION, REWARD, [reset_idx(reset_buf.nonzero()) = HB_STAGE_RESET_MASK + hb_env_reset_finalize], OBS
 * (+ hb_env_stack_finalize), LAST.  Launches with only PREPARE / TERMINATION / REWARD / LAST bits reset nothing and
 * need no hb_env_reset_finalize behind them. */
#define HB_STAGE_PREPARE     0x40  /* legged_robot.py:127-137: episode_length_buf += 1, base quantities, _post_physics_step_callback */
#define HB_STAGE_TERMINATION 0x80  /* check_termination (:155-160): reset_buf, time_out_buf */
#define HB_STAGE_REWARD      0x100 /* compute_reward (:216-234): rew_buf, episode_sums, feet_air_time / last_contacts / feet_height / last_feet_z */
#define HB_STAGE_LAST        0x200 /* legged_robot.py:146-150: last_last_actions, last_actions, last_dof_vel, last_root_vel */

const char *hb_last_error(void);
int hb_abi_version(void);
/* Number of kernels this library has launched since load / since the last reset (bench bookkeeping). */
int64_t hb_launch_count(void);
void hb_launch_count_reset(void);
/* Tuning switches: "env_bulk_staging" 1 = 1-D bulk async copies (default), 0 = vector loads;
 * "pdl" = programmatic stream serialization of the step's launches (each kernel's launch and prologue overlap the
 * tail of its predecessor; griddepcontrol.wait guards the dependent data): 1 = all kernels, 0 = none, 2 or -1
 * (default) = only the PD-torque launches (measured on one box, 4096 envs: 52.0 us per step with the default, 52.7
 * with none, 60.4 with all; PD launches only: +5.6 % at 16384 envs, +2 % at 65536; all kernels: -13 % at 65536);
 * "gae_serial_min_envs" (default 8192): shards at least this wide run GAE one thread per env;
 * "env_runtime_task" 0 (default) / 1: the built robots too run post-physics on the kernel that reads the layout at run
 * time (for tests and A/B measurements). */
/* "coop_launch" 0 (default) / 1: the two kernels that contain a grid barrier (hb_optimizer_step, hb_gae_fused) size their
 * grid to what the device holds at once; with 1 they are also launched with the cooperative attribute (the driver then
 * guarantees co-residency but serialises the launch against everything else on the device: measured 24.8 us against
 * the plain launch for GAE at 4096 x 24).  Plain launches are safe as long as nothing that occupies the SMs waits for
 * these kernels - true for stream-ordered use in one process per GPU. */
/* "gemm_pdl" 1 (default) / 0: hb_gemm_tf32 launches with programmatic stream serialization (a GEMM's set-up - tensor-map
 * prefetch, barriers, TMEM allocation, cluster rendezvous - overlaps the previous kernel's last tiles). */
/* "gemm_tile_snake" 1 (default) / 0: the rounds of a GEMM launch's tile list are dealt to the persistent CTAs in alternating
 * direction, so the extra tiles of a partial last round land on the CTAs that hold the shortest earlier tiles (results do
 * not depend on it; the order of split-K float atomics does). */
int hb_set_option(const char *name, int value);
/* dst[r, 0:width] = src[r, 0:width] for `rows` rows at the given byte pitches: ONE 2-D DMA transfer (device or pinned host
 * memory on either side).  How a host consumer reads step()'s observation tensors ([N, width] views of pitched rows)
 * without moving the padding. */
int hb_copy_rows(void *dst, int64_t dst_pitch_bytes, const void *src, int64_t src_pitch_bytes, int64_t width_bytes, int64_t rows,
                 void *stream);

/* CUDA graphs of hb_* launch sequences (one env step, one PPO.act) without the framework's graph object:
 * begin capture on `stream` (not the legacy default stream), issue hb_* calls on it, end -> an executable graph;
 * launch it on any stream.  Only hb_* calls may be captured (nothing that allocates). */
int hb_graph_begin(void *stream);
int hb_graph_end(void *stream, void **graph_exec);
int hb_graph_launch(void *graph_exec, void *stream);
int hb_graph_destroy(void *graph_exec);

/* HectorFreeEnv.step prologue: clip, action delay, action noise, clip
 * (envs/custom/hector_env.py:158-169 + envs/base/legged_robot.py:90-91).
 * actions_in [N,ndof] -> buf->actions (which also supplies the previous actions). */
int hb_env_action_prologue(const hb_env_params *p, const hb_env_buffers *buf, const float *actions_in,
                           const hb_env_noise *noise, void *stream);

/* LeggedRobot._compute_torques (envs/base/legged_robot.py:339-355): one decimation sub-step.
 * Reads buf->actions, dof_state, p_gains, d_gains; writes buf->torques. */
int hb_env_compute_torques(const hb_env_params *p, const hb_env_buffers *buf, void *stream);

/* hb_env_action_prologue + the first hb_env_compute_torques of a step in one launch (what step() uses when no host
 * work is needed between the two: same results as the two calls). */
int hb_env_prologue_torques(const hb_env_params *p, const hb_env_buffers *buf, const float *actions_in,
                            const hb_env_noise *noise, void *stream);

/* LeggedRobot.post_physics_step without the observation stacking
 * (envs/base/legged_robot.py:118-153,155-234,303-335,358-396; hector_env.py:53-88,256-539):
 * derived base quantities, command resampling + heading command, push, termination, the 18
 * reward terms, per-env reset bookkeeping, the newest observation / privileged frames and the
 * last_* copies.  The newest frames are written (noise added, clipped) into the last frame slot of
 * obs_new / priv_new; hb_env_stack_observations fills the other slots.  Shard-wide results of
 * reset_idx (id list, count, episode means) are produced by hb_env_reset_finalize, which must
 * follow every call of this function.
 * The three built robots (hector 10 DOF 41/70, hector_full 18 DOF 65/94, XBot-L 12 DOF 47/73 with their joint pairs) run
 * kernels compiled for their layout; any other layout of either task_kind runs the kernel that reads num_dof, yaw_roll,
 * arm_pair, ref_left / ref_right from p: 1 to 23 joints (HB_ERR_UNSUPPORTED above), frames 3 num_dof + 11 and
 * 3 num_dof + 40 (XBot: 4 num_dof + 25), every joint index inside the robot (HB_ERR_BAD_ARG otherwise). */
int hb_env_post_physics(const hb_env_params *p, const hb_env_buffers *buf, const hb_env_noise *noise,
                        float *obs_new, float *priv_new, int32_t stages, void *stream);

/* Frame stacking of HectorFreeEnv.compute_observations (envs/custom/hector_env.py:246-254):
 * slots 0..S-2 of obs_new/priv_new <- slots 1..S-1 of obs_prev/priv_prev, for every env.  The shift
 * does not depend on this step's physics: it may be launched any time after the previous step, before
 * hb_env_reset_finalize. */
int hb_env_stack_observations(const hb_env_params *p, const hb_env_buffers *buf,
                              const float *obs_prev, const float *priv_prev,
                              float *obs_new, float *priv_new, void *stream);

/* The shard-wide half of reset_idx (envs/base/legged_robot.py:142,162-214; hector_env.py:256-261), after
 * hb_env_post_physics and hb_env_stack_observations of the same step:
 *   reset_env_ids / reset_count = reset_buf.nonzero() in ascending order (+ *host_count, an optional
 *   pinned host int: gym.set_*_tensor_indexed need the count on the host, legged_robot.py:370-372,394-396);
 *   episode_means (extras["episode"], :198-201) and time_outs_latched (extras["time_outs"], :208-209),
 *   both only refreshed on steps with >= 1 reset like the reference;
 *   slots 0..S-2 of obs_new/priv_new zeroed for the reset envs (pass NULL for both to skip: reset_idx
 *   called outside step());
 *   *rng_counter += 1 if the device generator is in use (the same pointer as hb_env_noise.rng_counter), else NULL. */
int hb_env_reset_finalize(const hb_env_params *p, const hb_env_buffers *buf, float *obs_new, float *priv_new,
                          int32_t *host_count, uint64_t *rng_counter, void *stream);

/* hb_env_stack_observations + hb_env_reset_finalize in ONE launch (what step() uses): the shift blocks zero the
 * carried frames of the envs whose reset_buf byte hb_env_post_physics just set, extra blocks at the end of the grid
 * produce the id list / count / episode means / time-out latch.  Same results as the two separate calls. */
int hb_env_stack_finalize(const hb_env_params *p, const hb_env_buffers *buf, const float *obs_prev, const float *priv_prev,
                          float *obs_new, float *priv_new, int32_t *host_count, uint64_t *rng_counter, void *stream);

/* LeggedRobot._get_heights (envs/base/legged_robot.py:759-795) for terrains with a height field (mesh_type 'heightfield'
 * / 'trimesh', measure_heights = True): heights[slot, j] = vertical_scale * min over the cell under point j (base frame
 * points_xy[j] = (x, y), rotated by the base yaw, utils/math.py:39-43, plus base position and border_size, divided by
 * horizontal_scale, truncated) and its +x and +y neighbours of the int16 field height_samples[rows, cols].
 * env_ids: `count` env indices (the reference's env_ids argument), or NULL for envs 0..count-1.  heights [count, num_points]. */
int hb_env_get_heights(const float *root_states, const float *points_xy, int32_t num_points, const int16_t *height_samples,
                       int32_t rows, int32_t cols, float border_size, float horizontal_scale, float vertical_scale,
                       const int32_t *env_ids, int64_t count, float *heights, void *stream);

/* Host mirror of the stacked observations for a consumer on the CPU (rl_device = cpu; on_policy_runner.py:136 moves obs
 * and critic_obs to the learner's device every step).  Only the newest frame of a step's [N, S*F] stack is new, so the
 * GPU sends just that: host_*_ring are PINNED HOST buffers [N, slots + S - 1, frame] (device-accessible: cudaHostAlloc /
 * torch pin_memory under unified addressing); the kernel stores the newest frame of every env - the last `frame` columns
 * of its row - at ring slot `slot` and, when slot < S - 1, also at `slot + slots`, so that the last S frames of an env
 * are one contiguous run and its stacked observation is a strided view of the ring (row pitch (slots + S - 1) * frame
 * floats; the caller advances slot = k mod slots and needs slots >= S + 1; the window of the last S frames starts at slot
 * a - (S - 1) if a >= S - 1, else a + slots - (S - 1), a = the slot just written).  Envs whose reset_buf byte is set get
 * the rest of their rings zeroed first (reset_idx clears the history, hector_env.py:256-261); reset_buf may be NULL.
 * obs or priv may be NULL: that history is left to another call (e.g. one by the copy engine, one by a kernel on a second
 * stream).  use_dma != 0: the frames travel as 2-D copies of the copy engine (one or two per history) and the kernel only zeroes
 * the rings of reset envs; 0: the kernel stores the frames itself.  1.8 - 3.6 MB per step over PCIe instead of 27 MB at
 * 4096 hector envs.  The views of a step are valid until the next call. */
int hb_env_mirror_frames(const float *obs, int32_t obs_ld, int32_t obs_row, int32_t obs_frame, const float *priv, int32_t priv_ld,
                         int32_t priv_row, int32_t priv_frame, const uint8_t *reset_buf, int32_t num_envs, float *host_obs_ring,
                         int32_t obs_slots, int32_t obs_slot, float *host_priv_ring, int32_t priv_slots, int32_t priv_slot, int32_t use_dma,
                         void *stream);

/* One frame-stack shift on its own, dense rows: next[:, 0:row-frame] = prev[:, frame:row] (zeros for envs whose
 * reset_buf byte is set, if reset_buf is not NULL); next[:, row-frame:row] is left alone. */
int hb_stack_shift(const float *prev, float *next, const uint8_t *reset_buf, int32_t num_envs, int32_t row,
                   int32_t frame, void *stream);

/* RolloutStorage.compute_returns (algo/ppo/rollout_storage.py:122-136).
 * rewards, values, returns, advantages: [T,N] fp32; dones [T,N] uint8; last_values [N].
 * Pass 1 writes returns and the raw advantages (returns - values) and accumulates
 * (sum, sum of squares) in fp64 into stats[0..1]; pass 2 normalises
 * with the unbiased std.  Multi-GPU callers all-reduce `stats` between the two passes. */
int hb_gae_returns(const float *rewards, const float *values, const uint8_t *dones, const float *last_values,
                   float *returns, float *advantages, double *stats, int32_t T, int32_t N,
                   float gamma, float lam, void *stream);
int hb_gae_normalize(float *advantages, const double *stats, int64_t count, void *stream);
/* Same, when `stats` were summed over `stat_count` samples (all ranks) and this rank holds `count`. */
int hb_gae_normalize_n(float *advantages, const double *stats, int64_t stat_count, int64_t count, void *stream);
/* Single-GPU form of the whole of compute_returns in ONE launch: one thread per env, the raw advantages stay in
 * shared memory across a grid barrier on (sum, sum sq) and are written once, normalised - 17 instead of 25 bytes per sample
 * and one launch instead of memset + two kernels.  scratch: HB_GAE_SCRATCH_DOUBLES doubles of device memory (8 slots of
 * sums, 8 of sums of squares, a ticket), zero before the first call (the launch re-arms them).  Falls back to
 * hb_gae_returns + hb_gae_normalize for longer rollouts or shards too wide for one co-resident grid.  Multi-GPU callers
 * use the two-call form (the statistics are all-reduced between the passes).
 * Option "gae_threads": block width, 0 (default: 64 up to 8192 envs, else 256) / 32 / 64 / 128 / 256. */
#define HB_GAE_SCRATCH_DOUBLES 32
int hb_gae_fused(const float *rewards, const float *values, const uint8_t *dones, const float *last_values, float *returns,
                 float *advantages, double *scratch, int32_t T, int32_t N, float gamma, float lam, void *stream);

/* ------------------------------------------------------------------------------------------------
 * PPO update (algo/ppo/ppo.py:119-184, actor_critic.py:36-128, rollout_storage.py:146-182)
 * ---------------------------------------------------------------------------------------------- */

/* One GEMM of the ActorCritic MLPs on the tcgen05 tensor cores (TF32 operands read from fp32
 * storage through TMA, fp32 accumulation in TMEM):   D[M,N] (+)= A[M,K] * B[N,K]^T.
 * K-major operand: memory is [rows(M or N), K] row-major.  MN-major operand (a_mn_major /
 * b_mn_major = 1): memory is [K, rows] row-major, i.e. the same row-major activations / weights
 * seen from the backward pass; no transposed copies are made.  Leading dimensions are in floats
 * and must be multiples of 4; base pointers 16-byte aligned. */
enum hb_gemm_epilogue {
    HB_EPI_STORE = 0,      /* D = acc */
    HB_EPI_BIAS = 1,       /* D = acc + bias[n]                       nn.Linear (actor_critic.py:62,74) */
    HB_EPI_BIAS_ACT = 2,   /* D = f(acc + bias[n])                    nn.Linear + activation f (:56-60) */
    HB_EPI_ACT_BWD = 3,    /* D = acc * f'(z) with H = f(z)           autograd of the above */
    HB_EPI_ATOMIC_ADD = 4, /* D += acc (split-K weight gradients; D must be zeroed by the caller) */
    HB_EPI_BIAS_ELU = HB_EPI_BIAS_ACT,     /* the names from before the activation became a descriptor field */
    HB_EPI_ELU_BWD = HB_EPI_ACT_BWD
};
/* The activation f of HB_EPI_BIAS_ACT / HB_EPI_ACT_BWD: the set of get_activation in algo/ppo/actor_critic.py, with
 * torch's definitions.  Every f' is written in the forward output h = f(z), which is what the data-gradient epilogue reads:
 *   HB_ACT_ELU      z > 0 ? z : exp(z) - 1                       h > 0 ? 1 : h + 1
 *   HB_ACT_SELU     s * (z > 0 ? z : a * (exp(z) - 1))           h > 0 ? s : h + s * a     (a = 1.6732632, s = 1.0507010)
 *   HB_ACT_RELU     max(z, 0)                                    h > 0 ? 1 : 0              ("crelu" maps here too)
 *   HB_ACT_LRELU    z > 0 ? z : 0.01 z                           h > 0 ? 1 : 0.01
 *   HB_ACT_TANH     tanh(z)                                      1 - h * h
 *   HB_ACT_SIGMOID  1 / (1 + exp(-z))                            (1 - h) * h
 * In HB_GEMM_TF32 mode the non-ELU activations are built for the layouts these epilogues have in an MLP: HB_EPI_BIAS_ACT
 * with A and B K-major, HB_EPI_ACT_BWD with A K-major and B MN-major (HB_ERR_UNSUPPORTED otherwise); ELU takes every
 * layout.  An unknown value is HB_ERR_BAD_ARG. */
enum hb_activation {
    HB_ACT_ELU = 0,
    HB_ACT_SELU = 1,
    HB_ACT_RELU = 2,
    HB_ACT_LRELU = 3,
    HB_ACT_TANH = 4,
    HB_ACT_SIGMOID = 5,
    HB_ACT_COUNT = 6
};
/* A, B (and, for every epilogue but HB_EPI_ATOMIC_ADD, D and H) are moved by TMA: 16-byte aligned bases, leading dimensions
 * that are multiples of 4 floats (HB_ERR_BAD_ARG otherwise).  Ragged M / N are clipped by the tensor maps. */
typedef struct hb_gemm_desc {
    const float *A, *B;
    float *D;
    int32_t M, N, K;
    int32_t lda, ldb, ldd;
    int32_t a_mn_major, b_mn_major;
    int32_t epilogue;            /* hb_gemm_epilogue */
    const float *bias;           /* bias[n * bias_stride] */
    int32_t bias_stride;
    const float *H;              /* HB_EPI_ELU_BWD: forward activations [M, ldh] */
    int32_t ldh;
    int32_t split_k;             /* HB_EPI_ATOMIC_ADD only: >1 = number of splits of the contraction; 0 = automatic
                                    (about two rounds of tiles over the SMs) */
    int32_t tile_n;              /* 0 = automatic; 128 forces 128-wide tiles */
    int32_t precision;           /* hb_gemm_precision */
    float *workspace;            /* HB_GEMM_3XTF32: scratch for the split operands, 16-byte aligned, */
    int64_t workspace_floats;    /*   at least hb_gemm_workspace_floats(desc) floats */
    int32_t activation;          /* hb_activation of HB_EPI_BIAS_ACT / HB_EPI_ACT_BWD; 0 = ELU */
} hb_gemm_desc;
/* Arithmetic of the products.  HB_GEMM_TF32: operands truncated to TF32 by the tensor core (10-bit mantissa), fp32
 * accumulation - the fast path.  HB_GEMM_3XTF32: every operand is split x = hi + lo (hi = x rounded to TF32, lo = x - hi)
 * and the tensor core sums a_hi*b_hi + a_lo*b_hi + a_hi*b_lo in the same fp32 accumulator (one contraction of 3 K): the
 * dropped a_lo*b_lo term is 2^-22 relative, i.e. the result is fp32-grade like the reference's nn.Linear
 * (algo/ppo/actor_critic.py:54-83) at about a third of the TF32 throughput. */
enum hb_gemm_precision { HB_GEMM_TF32 = 0, HB_GEMM_3XTF32 = 1 };
int hb_gemm_tf32(const hb_gemm_desc *desc, void *stream);
int64_t hb_gemm_workspace_floats(const hb_gemm_desc *desc);
/* Two GEMMs of the same kind (same epilogue and operand layouts: the actor's and the critic's GEMM of one layer,
 * actor_critic.py:54-77) in ONE launch: the persistent CTAs walk the concatenated tile list, so both networks share every
 * wave of tiles and a launch's pipeline set-up / drain is paid once per layer.  Results are those of two hb_gemm_tf32
 * calls; problems whose tile shapes cannot share a kernel (or HB_GEMM_3XTF32) fall back to exactly that. */
int hb_gemm_tf32_grouped(const hb_gemm_desc *desc0, const hb_gemm_desc *desc1, void *stream);
/* 256-wide tiles are computed by pairs of CTAs (tcgen05.mma.cta_group::2, 2-CTA clusters: each SM stages half of the
 * B tile) unless switched off (on = 0: one CTA per tile everywhere; for A/B measurements). */
int hb_gemm_set_pair_mode(int on);

/* mini_batch_generator's index gathers (rollout_storage.py:165-180), done once per update because the
 * permutation is drawn once and reused by every epoch (:149): dst[i, 0:cols] = src[perm[i], 0:cols];
 * if ones_col >= 0, dst[i, ones_col] = 1 (the constant column that turns bias gradients into one more
 * column of the weight-gradient GEMM). */
int hb_ppo_gather_rows(const float *src, int32_t ld_src, float *dst, int32_t ld_dst, const int64_t *perm,
                       int64_t rows, int32_t cols, int32_t ones_col, void *stream);

/* Per-sample record, gathered in minibatch order: actions[A] old_mu[A] old_sigma[A] old_value advantage
 * return old_log_prob 0 0 = HB_PPO_REC(A) floats; A = num_actions, 1 to 64 (hb_ppo_pack_samples, hb_ppo_loss_head
 * and hb_ppo_act_head) or 1 to 15 (hb_ppo_head_fused, hb_ppo_act_fused).  A count below 1 is HB_ERR_BAD_ARG, one above
 * the entry point's limit HB_ERR_UNSUPPORTED; either is refused before any launch. */
#define HB_PPO_REC(num_actions) (3 * (num_actions) + 6)
int hb_ppo_pack_samples(const int64_t *perm, int64_t rows, const float *actions, const float *mu, const float *sigma,
                        const float *values, const float *advantages, const float *returns, const float *log_prob,
                        int32_t num_actions, float *records, void *stream);

typedef struct hb_ppo_loss_params {
    float clip_param, value_loss_coef, entropy_coef;
    int32_t use_clipped_value_loss;
    int32_t num_actions;          /* 1 to 64 (hb_ppo_loss_head), 1 to 15 (hb_ppo_head_fused) */
    int32_t activation;           /* hb_activation of the hidden layers (hb_ppo_head_fused's f'); 0 = ELU */
} hb_ppo_loss_params;
/* Loss head and its analytic backward for one minibatch (ppo.py:130-168): Gaussian log-prob, ratio,
 * clipped surrogate, clipped value loss, entropy bonus, KL to the behaviour policy.
 * mu [mb, ld_mu] (first A = num_actions columns), value [mb, ld_v] (first column), std[A], records [mb, HB_PPO_REC(A)].
 * Writes d_mu [mb, ld_mu] and d_value [mb, ld_v] (padding columns zeroed), accumulates d_std[A] and
 * stats[4] = {sum surrogate, sum value loss, sum kl, sum entropy} (fp64; caller zeroes both). */
int hb_ppo_loss_head(const float *mu, int32_t ld_mu, const float *value, int32_t ld_v, const float *std,
                     const float *records, int64_t mb, int64_t mb_global, const hb_ppo_loss_params *lp, float *d_mu,
                     float *d_value, float *d_std, double *stats, void *stream);

/* Update path, output layers fused with the loss head: for hidden width 128 (hector_config.py:207-210) the last
 * nn.Linear of both MLPs (actor_critic.py:62,74) is evaluated with fp32 FMAs inside the loss kernel, together with
 * its data gradient (into dz3 = d loss / d pre-activation of the last hidden layer, f' of lp->activation applied) and its weight /
 * bias gradients (accumulated into g4_actor [>=A rows, ld_w] and g4_critic [>=1 row, ld_w], packed [W | b]).
 * h3_* [mb, ld_h]: last hidden activations; w4_* packed [W | b] with leading dimension ld_w; records, std, lp,
 * d_std, stats as in hb_ppo_loss_head.  A = lp->num_actions, 1 to 15: one lane pair per action and one for the value
 * (wider heads: hb_gemm_tf32 + hb_ppo_loss_head). */
int hb_ppo_head_fused(const float *h3_actor, int32_t ld_ha, const float *h3_critic, int32_t ld_hc, const float *w4_actor,
                      const float *w4_critic, int32_t ld_w, const float *std, const float *records, int64_t mb,
                      int64_t mb_global, const hb_ppo_loss_params *lp, float *dz3_actor, float *dz3_critic, int32_t ld_dz,
                      float *g4_actor, float *g4_critic, float *d_std, double *stats, void *stream);

/* N(0,1) draws for the action sample (algo/ppo/ppo.py:93 -> actor_critic.py:116 `distribution.sample()`): count floats
 * from the library's Philox4x32-10 generator; state = device uint64[3] {call counter, 0, key}: the counter is advanced by
 * the launch itself, so the call can sit in a replayed CUDA graph, draw fresh numbers every replay and follow a re-seed
 * (write the key, zero the counter). */
int hb_ppo_draw_normal(float *out, int64_t count, uint64_t *state, void *stream);

/* PPO.act head (ppo.py:91-101, actor_critic.py:111-120): a = mu + sigma*eps, log-prob, copies of mu/sigma; 1 to 64
 * actions. */
int hb_ppo_act_head(const float *mu, int32_t ld_mu, const float *std, const float *eps, int64_t n, int32_t num_actions,
                    float *actions, float *log_prob, float *mu_out, float *sigma_out, void *stream);

/* Rollout side.  hb_ppo_act_fused: the output layers of both MLPs (hidden width 128) + PPO.act's sampling head
 * (ppo.py:91-101, actor_critic.py:111-120): a = mu + sigma * eps, log-prob, mu, sigma and the value, written to
 * caller-chosen destinations - normally the rollout-storage slot of the step (rollout_storage.py:87-100), so
 * add_transitions' copies of these tensors disappear.  actions/mu_out/sigma_out [n, num_actions] with 1 to 15 actions,
 * log_prob/values [n].
 * hb_ppo_record_step: PPO.process_env_step's record (ppo.py:103-113): rewards_out = rewards + gamma * values *
 * time_outs (time_outs may be NULL), dones_out = dones as uint8. */
int hb_ppo_act_fused(const float *h3_actor, int32_t ld_ha, const float *h3_critic, int32_t ld_hc, const float *w4_actor,
                     const float *w4_critic, int32_t ld_w, const float *std, const float *eps, int64_t n, int32_t num_actions,
                     float *actions, float *log_prob, float *mu_out, float *sigma_out, float *values, void *stream);
int hb_ppo_record_step(const float *rewards, const uint8_t *dones, const float *values, const uint8_t *time_outs, float gamma,
                       int64_t n, float *rewards_out, uint8_t *dones_out, void *stream);

typedef struct hb_adam_params {
    double beta1, beta2, eps;     /* torch.optim.Adam defaults 0.9, 0.999, 1e-8 (ppo.py:68); doubles like the Python floats */
    float max_grad_norm;          /* clip_grad_norm_ (ppo.py:173); <= 0 disables clipping */
    int32_t adaptive;             /* 1: schedule == 'adaptive' and desired_kl is set (ppo.py:136-148) */
    double desired_kl;
    int64_t kl_count;             /* samples behind state->stats[2] (the global minibatch) */
} hb_adam_params;

/* Optimizer scalars, resident in device memory (8-byte aligned): nothing about a step travels by value, so the launch
 * sequence of one minibatch step can be captured once and replayed for every step of every update. */
#define HB_OPT_TRACE_MAX 64
typedef struct hb_optim_state {
    double lr;                    /* learning rate; the adaptive-KL rule updates it in place */
    double grad_sumsq;            /* scratch, zero between steps */
    double stats[4];              /* this minibatch's loss sums {surrogate, value loss, kl, entropy}: accumulated by
                                     hb_ppo_head_fused / hb_ppo_loss_head (all-reduced over ranks), zero between steps */
    double loss_acc[4];           /* running sums over the update (ppo.py:176-178); the host zeroes them per update() */
    int64_t step;                 /* Adam's step count t (bias corrections 1 - beta^t) */
    int64_t steps_in_update;      /* optimizer steps since the host last zeroed it: index into trace */
    uint64_t ticket;              /* grid barrier of hb_optimizer_step; zero between steps */
    uint64_t reserved;            /* hb_dp_optimizer_step: 0, or the phase in which a peer failed to arrive (time-out) */
    uint64_t go;                  /* hb_dp_optimizer_step: local gate, monotonic */
    float bcast[4];               /* hb_dp_optimizer_step: clip scale, step size, sqrt(bias_correction2) of the step */
    double trace[2 * HB_OPT_TRACE_MAX];   /* {mean KL, learning rate after the rule} of step i < HB_OPT_TRACE_MAX of the update */
} hb_optim_state;

/* clip_grad_norm_ + torch.optim.Adam.step (defaults, no weight decay) + optimizer.zero_grad over one flat parameter
 * buffer, with the adaptive learning-rate rule evaluated on the device from state->stats[2] - ONE cooperative launch
 * (gradient norm, grid barrier, update; ppo.py:136-148,171-174).  On return (stream order): gradients zeroed,
 * state->stats folded into state->loss_acc and zeroed, state->step and state->steps_in_update advanced. */
int hb_optimizer_step(float *params, float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, const hb_adam_params *ap,
                      hb_optim_state *state, void *stream);

/* OnPolicyRunner.learn's per-step bookkeeping (algo/ppo/on_policy_runner.py:140-154) without its two nonzero() + .cpu()
 * round trips per step: cur_reward_sum += rewards, cur_episode_length += 1, and for every env with dones != 0, in
 * ascending env order, (sum, length) is pushed into two rings of `capacity` entries (the reference's deque(maxlen=100)
 * buffers) and the running values restart at 0.  ring_state[0] counts the entries ever pushed (device int64, zero at
 * start): entry j of the deque view is ring[(ring_state[0] - count + j) % capacity], count = min(ring_state[0], capacity). */
int hb_runner_bookkeeping(const float *rewards, const uint8_t *dones, int64_t n, float *cur_reward_sum, float *cur_episode_length,
                          float *ring_rewards, float *ring_lengths, int32_t capacity, int64_t *ring_state, void *stream);

/* Data-parallel replicas (SURVEY.md §8e; the reference is single-device).  Every rank's flat gradient / parameter
 * buffers, a mailbox and a flag array are mapped into every rank's address space (symmetric memory over NVLink /
 * NVSwitch; the host passes the peer pointers).  hb_dp_optimizer_step is ONE kernel per rank that replaces the gradient
 * all-reduce, clip_grad_norm_, Adam, zero_grad and the parameter broadcast: each rank sums ITS 1/world slice of the
 * gradient over all ranks (peer loads, or multimem.ld_reduce through the switch when grad_mc is set), exchanges slice
 * norms and loss sums through the mailboxes, applies clip + Adam to its slice (optimizer state is sharded: a rank only
 * touches its slice of exp_avg / exp_avg_sq) and stores the new parameters into all ranks' buffers (peer stores or
 * multimem.st).  state as in hb_optimizer_step; state->reserved != 0 afterwards means a peer did not arrive in time.
 * All ranks must call it the same number of times with the same state->step. */
#define HB_DP_MAX_RANKS 8
typedef struct hb_dp_comm {
    int32_t world, rank;
    float *grad[HB_DP_MAX_RANKS];      /* flat gradient buffers (n floats), [rank] = this rank's own */
    float *param[HB_DP_MAX_RANKS];     /* flat parameter buffers (n floats) */
    double *mail[HB_DP_MAX_RANKS];     /* mailboxes: HB_DP_MAX_RANKS x 8 doubles each */
    uint32_t *flag[HB_DP_MAX_RANKS];   /* flag arrays: 3 x HB_DP_MAX_RANKS words each, zero before the first step */
    float *grad_mc, *param_mc;         /* multicast (NVLS) addresses of the gradient / parameter buffers, or NULL */
} hb_dp_comm;
int hb_dp_optimizer_step(const hb_dp_comm *comm, float *exp_avg, float *exp_avg_sq, int64_t n, const hb_adam_params *ap,
                         hb_optim_state *state, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HECTOR_B200_H */
