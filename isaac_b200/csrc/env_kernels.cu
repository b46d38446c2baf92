// Env-stage kernels of the hector hot path (SURVEY.md §8 rows a1-a9), sm_100a.
//
// Compiled with --fmad=false: the reference evaluates every expression as separate fp32 torch
// ops, so no multiply-add may be contracted here; operation order follows the reference lines
// cited at each block (paths relative to /root/reference/humanoid).
//
// Data layout: the gym tensors are read in place.  Work is tiled as ONE WARP PER 32-ENV TILE:
// every [N, row] tensor of a tile is a contiguous slab in HBM, which the warp stages into
// shared memory either with 1-D bulk async copies (TMA engine, one mbarrier) or with coalesced
// vector loads, and then each lane owns one env and reads its row from shared memory.
#include <math.h>
#include <string.h>

#include "hb_common.cuh"

namespace {

// The three tasks the reference registers (envs/__init__.py:46-48) share one env step; they differ in the number of
// joints and in the privileged frame:
//   KIND_HECTOR  hector (10 DOF, hector_env.py:195-226) and hector_full (18 DOF, hector_w_arm_env.py:202-233):
//                [cmd 5 | q-q0 N | dq N | a N | lin 3 | ang 3 | euler 3 | feet pos 6 | feet vel 6 | root pos 3 | push 2+3 |
//                 friction | mass/30 | stance 2 | contact 2]                                        = 3 N + 40
//   KIND_XBOT    humanoid_ppo / XBot-L (12 DOF, humanoid_env.py:217-234): the reference-trajectory error instead of the
//                feet / root entries: [cmd 5 | q-q0 N | dq N | a N | q-ref N | lin 3 | ang 3 | euler 3 | push 2+3 |
//                 friction | mass/30 | stance 2 | contact 2]                                        = 4 N + 25
// The observation frame is [cmd 5 | q-q0 N | dq N | a N | ang 3 | euler 3] = 3 N + 11 for all of them.
constexpr int KIND_HECTOR = 0, KIND_XBOT = 1;
// Any other robot with the same env file runs the same kernel with its joint count and joint pairs read at run time
// (RuntimeTask), up to MAX_TASK_DOF joints: an observation frame 3 N + 11 <= HB_MAX_OBS, so that its draws stay inside the
// Philox slots below.
constexpr int MAX_TASK_DOF = (HB_MAX_OBS - 11) / 3;

// Column offsets of the frames and the joint pairs of default_joint_pos of a task with `ndof` joints
struct TaskDims {
    int NDOF, OBS, B0, B1, P_DIFF, P_LIN, P_ANG, P_EUL, P_FEET_POS, P_FEET_VEL, P_ROOT, P_PUSH_F, P_PUSH_T, P_FRICTION, P_MASS,
        P_STANCE, P_CONTACT, PRIV, U_RESET, YAW_L, YAW_R, ARM_L, ARM_R;
    bool HAS_ARMS;
};
__host__ __device__ constexpr TaskDims task_dims(int ndof, int kind, int yaw_l, int yaw_r, int arm_l, int arm_r) {
    TaskDims d{};
    d.NDOF = ndof;
    d.OBS = 5 + 3 * ndof + 6;
    d.B0 = 5 + 3 * ndof;                                 // end of the joint columns
    d.B1 = kind == KIND_XBOT ? d.B0 + ndof : d.B0;       // start of the base-velocity columns
    d.P_DIFF = d.B0;                                     // KIND_XBOT only
    d.P_LIN = d.B1, d.P_ANG = d.B1 + 3, d.P_EUL = d.B1 + 6;
    d.P_FEET_POS = d.B1 + 9, d.P_FEET_VEL = d.B1 + 15, d.P_ROOT = d.B1 + 21;      // KIND_HECTOR only
    d.P_PUSH_F = kind == KIND_XBOT ? d.B1 + 9 : d.B1 + 24;
    d.P_PUSH_T = d.P_PUSH_F + 2, d.P_FRICTION = d.P_PUSH_F + 5, d.P_MASS = d.P_PUSH_F + 6, d.P_STANCE = d.P_PUSH_F + 7;
    d.P_CONTACT = d.P_PUSH_F + 9;
    d.PRIV = d.P_CONTACT + 2;
    d.U_RESET = ndof + 5;                                // dof offsets, root xy, command draws (legged_robot.py:366,384,327-330)
    d.YAW_L = yaw_l, d.YAW_R = yaw_r, d.ARM_L = arm_l, d.ARM_R = arm_r;
    d.HAS_ARMS = arm_l >= 0;
    return d;
}

// OPT_: the optional reward terms (joint_pos with the reference trajectory, vel_mismatch_exp, track_vel_hard, low_speed:
// zero-scale in hector_config.py) are compiled in.  A config that scales none of them runs the kernel without their code:
// the four-role kernel is bound by instruction latency and its footprint (6.5 k SASS instructions with them, 5.5 k without).
// The kernel reads a task's dimensions from `T::dims(p)`: this empty object, whose members are compile-time constants, or
// RuntimeTask's TaskDims.  CAP sizes the per-lane joint arrays.
template <int NDOF_, int KIND_, bool OPT_ = true>
struct Task {
    static constexpr int NDOF = NDOF_, KIND = KIND_, CAP = NDOF_;
    static constexpr bool OPT = OPT_ || KIND_ == 1;                 // XBot-L always maintains the reference trajectory
    static constexpr bool RUNTIME = false;
    // default_joint_pos (hector_env.py:357-367, hector_w_arm_env.py:371-378, humanoid_env.py:368-369): first joint of each
    // leg's (yaw, roll) pair and, with arms, of each arm's pair - joint-order constants of the three robots
    static constexpr bool HAS_ARMS = NDOF_ == 18;
    static constexpr TaskDims d() {
        return task_dims(NDOF_, KIND_, 0, NDOF_ / 2, HAS_ARMS ? 5 : -1, HAS_ARMS ? NDOF_ / 2 + 5 : -1);
    }
    static constexpr int YAW_L = d().YAW_L, YAW_R = d().YAW_R, ARM_L = d().ARM_L, ARM_R = d().ARM_R;
    static constexpr int OBS = d().OBS, B0 = d().B0, B1 = d().B1, P_DIFF = d().P_DIFF, P_LIN = d().P_LIN, P_ANG = d().P_ANG,
                         P_EUL = d().P_EUL, P_FEET_POS = d().P_FEET_POS, P_FEET_VEL = d().P_FEET_VEL, P_ROOT = d().P_ROOT,
                         P_PUSH_F = d().P_PUSH_F, P_PUSH_T = d().P_PUSH_T, P_FRICTION = d().P_FRICTION, P_MASS = d().P_MASS,
                         P_STANCE = d().P_STANCE, P_CONTACT = d().P_CONTACT, PRIV = d().PRIV, U_RESET = d().U_RESET;
    __device__ static Task dims(const hb_env_params &) { return Task{}; }
};
// Any other robot of a kind: joint count and pairs read from hb_env_params (validated by the launcher), every optional
// term compiled in
template <int KIND_>
struct RuntimeTask {
    static constexpr int KIND = KIND_, CAP = MAX_TASK_DOF;
    static constexpr bool OPT = true, RUNTIME = true;
    __device__ static TaskDims dims(const hb_env_params &p) {
        return task_dims(p.num_dof, KIND_, p.yaw_roll[0], p.yaw_roll[1], p.arm_pair[0], p.arm_pair[1]);
    }
};
static_assert(Task<10, KIND_HECTOR>::OBS == 41 && Task<10, KIND_HECTOR>::PRIV == 70, "hector (hector_config.py:12-14)");
static_assert(Task<18, KIND_HECTOR>::OBS == 65 && Task<18, KIND_HECTOR>::PRIV == 94, "hector_full (hector_w_arm_config.py:12-14)");
static_assert(Task<12, KIND_XBOT>::OBS == 47 && Task<12, KIND_XBOT>::PRIV == 73, "XBot-L (humanoid_config.py:46-48)");
constexpr int TILE = 32;

constexpr float TWO_PI_F = 6.283185307179586f;    // float32(2*np.pi)
constexpr float PI_F = 3.141592653589793f;        // float32(np.pi)
constexpr float HALF_PI_F = 1.5707963267948966f;

struct Vec3 {
    float x, y, z;
};

__device__ __forceinline__ Vec3 cross3(const Vec3 &a, const Vec3 &b) {
    return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}

// isaacgym.torch_utils.quat_rotate_inverse, q = (x,y,z,w): a - b + c (SURVEY.md §8c)
__device__ __forceinline__ Vec3 quat_rotate_inverse(const float q[4], const Vec3 &v) {
    const float w = q[3];
    const Vec3 u = {q[0], q[1], q[2]};
    const float s = 2.0f * (w * w) - 1.0f;
    const Vec3 cr = cross3(u, v);
    const float dot = u.x * v.x + u.y * v.y + u.z * v.z;
    Vec3 o;
    o.x = (v.x * s - (cr.x * w) * 2.0f) + (u.x * dot) * 2.0f;
    o.y = (v.y * s - (cr.y * w) * 2.0f) + (u.y * dot) * 2.0f;
    o.z = (v.z * s - (cr.z * w) * 2.0f) + (u.z * dot) * 2.0f;
    return o;
}

// isaacgym.torch_utils.quat_apply: t = 2 (u x v); v + w t + u x t
__device__ __forceinline__ Vec3 quat_apply(const float q[4], const Vec3 &v) {
    const Vec3 u = {q[0], q[1], q[2]};
    Vec3 t = cross3(u, v);
    t.x *= 2.0f, t.y *= 2.0f, t.z *= 2.0f;
    const Vec3 ut = cross3(u, t);
    return {(v.x + q[3] * t.x) + ut.x, (v.y + q[3] * t.y) + ut.y, (v.z + q[3] * t.z) + ut.z};
}

// torch.remainder(a, m) for floats
__device__ __forceinline__ float py_mod(float a, float m) {
    float r = fmodf(a, m);
    if (r != 0.0f && ((r < 0.0f) != (m < 0.0f))) r += m;
    return r;
}

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }

// ------------------------------------------------------------------------------------------
// Device-side draws (SURVEY.md §8f rank 3).  When the caller supplies no tape for a draw, it is generated
// where it is consumed with Philox4x32-10 (the generator behind torch.rand / curand): key = the env's seed (device memory),
// counter = (env, slot, step), so a draw is a pure function of (seed, step, env, slot) - no state besides
// the step counter, no tape written to or read from HBM, and rare draws (resets, command resampling,
// pushes) cost nothing on the steps that do not need them.  Slots of one env and step:
//   0-5 z_action[<=24] | 6-25 z_obs[<=80] | 26-33 u_reset[<=29] | 34 u_cmd[3] | 35-36 u_push[5] | 37 u_delay
// ------------------------------------------------------------------------------------------
struct Rng {
    uint32_t k0, k1, s0, s1;
    bool on;
};
__device__ __forceinline__ Rng make_rng(const hb_env_noise &nz) {
    Rng r;
    r.on = nz.rng_counter != nullptr;
    // {step counter, key} both live in device memory: a captured launch picks up a re-seed on its next replay
    const unsigned long long step = r.on ? nz.rng_counter[0] : 0ull, key = r.on ? nz.rng_counter[1] : 0ull;
    r.k0 = (uint32_t)key, r.k1 = (uint32_t)(key >> 32);
    r.s0 = (uint32_t)step, r.s1 = (uint32_t)(step >> 32);
    return r;
}
constexpr int SLOT_Z_ACTION = 0, SLOT_Z_OBS = 6, SLOT_U_RESET = 26, SLOT_U_CMD = 34, SLOT_U_PUSH = 35, SLOT_U_DELAY = 37;

using hb::philox4x32_10;
__device__ __forceinline__ void rng_uniform4(const Rng &g, int env, int slot, float u[4]) {      // [0, 1)
    const uint4 x = philox4x32_10((uint32_t)env, (uint32_t)slot, g.s0, g.s1, g.k0, g.k1);
    u[0] = (float)(x.x >> 8) * 5.9604644775390625e-8f, u[1] = (float)(x.y >> 8) * 5.9604644775390625e-8f;
    u[2] = (float)(x.z >> 8) * 5.9604644775390625e-8f, u[3] = (float)(x.w >> 8) * 5.9604644775390625e-8f;
}
__device__ __forceinline__ void rng_normal4(const Rng &g, int env, int slot, float z[4]) {       // Box-Muller
    const uint4 x = philox4x32_10((uint32_t)env, (uint32_t)slot, g.s0, g.s1, g.k0, g.k1);
    const float u0 = (float)((x.x >> 8) + 1u) * 5.9604644775390625e-8f, u1 = (float)((x.z >> 8) + 1u) * 5.9604644775390625e-8f;
    const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u1));
    float s0, c0, s1, c1;
    __sincosf(TWO_PI_F * ((float)(x.y >> 8) * 5.9604644775390625e-8f), &s0, &c0);
    __sincosf(TWO_PI_F * ((float)(x.w >> 8) * 5.9604644775390625e-8f), &s1, &c1);
    z[0] = r0 * c0, z[1] = r0 * s0, z[2] = r1 * c1, z[3] = r1 * s1;
}
// element `idx` of a per-env vector of uniforms that starts at `slot`
__device__ __forceinline__ void rng_uniforms(const Rng &g, int env, int slot, int first, int count, float *out) {
    for (int c = first / 4; c <= (first + count - 1) / 4; ++c) {
        float u[4];
        rng_uniform4(g, env, slot + c, u);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int idx = c * 4 + k - first;
            if (idx >= 0 && idx < count) out[idx] = u[k];
        }
    }
}

// ------------------------------------------------------------------------------------------
// a2: HectorFreeEnv.step prologue (hector_env.py:158-169, legged_robot.py:90-91)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float action_prologue(const float *__restrict__ a_in, const float *__restrict__ actions,
                                                 const hb_env_noise &nz, const Rng &rng, int i, int ndof, float clip,
                                                 float action_delay, float action_noise) {
    const int env = i / ndof, j = i - env * ndof;
    float a = clampf(a_in[i], -clip, clip);
    float ud = 0.0f;
    if (action_delay != 0.0f) {
        if (nz.u_delay) ud = nz.u_delay[env];
        else if (rng.on) rng_uniforms(rng, env, SLOT_U_DELAY, 0, 1, &ud);
    }
    const float delay = ud * action_delay;
    a = (1.0f - delay) * a + delay * actions[i];
    float z = 0.0f;
    if (nz.z_action) {
        z = nz.z_action[i];
    } else if (rng.on && action_noise != 0.0f) {
        float z4[4];
        rng_normal4(rng, env, SLOT_Z_ACTION + (j >> 2), z4);
        z = z4[j & 3];
    }
    a = a + (action_noise * z) * a;
    return clampf(a, -clip, clip);
}

__global__ void __launch_bounds__(256)
action_prologue_kernel(const float *__restrict__ a_in, float *__restrict__ actions, const __grid_constant__ hb_env_noise nz,
                       int total, int ndof, float clip, float action_delay, float action_noise) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const Rng rng = make_rng(nz);
    actions[i] = action_prologue(a_in, actions, nz, rng, i, ndof, clip, action_delay, action_noise);
}

// ------------------------------------------------------------------------------------------
// a1: LeggedRobot._compute_torques (legged_robot.py:339-355).  Two DOFs per thread so that the
// interleaved (pos,vel) pairs are one 16-byte load and everything else an 8-byte access.
// ------------------------------------------------------------------------------------------
struct PdConsts {
    float q0[HB_MAX_DOF];
    float lim[HB_MAX_DOF];
};

__global__ void __launch_bounds__(256)
pd_torque_kernel(const float4 *__restrict__ dof_state2, const float2 *__restrict__ actions2,
                 const float2 *__restrict__ kp2, const float2 *__restrict__ kd2, float2 *__restrict__ torques2,
                 int pairs, int ndof, float action_scale, const __grid_constant__ PdConsts c) {
    hb::pdl_trigger();                       // the next launch of the step may be scheduled behind this one
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    hb::pdl_wait();                          // predecessor (prologue / previous sub-step / physics) complete
    if (i >= pairs) return;
    const float4 s = dof_state2[i];          // q0 qd0 q1 qd1
    const float2 a = actions2[i], kp = kp2[i], kd = kd2[i];
    const int j = (2 * i) % ndof;            // ndof even: a pair never straddles two envs
    float2 t;
    t.x = kp.x * ((a.x * action_scale + c.q0[j]) - s.x) - kd.x * s.y;
    t.y = kp.y * ((a.y * action_scale + c.q0[j + 1]) - s.z) - kd.y * s.w;
    t.x = clampf(t.x, -c.lim[j], c.lim[j]);
    t.y = clampf(t.y, -c.lim[j + 1], c.lim[j + 1]);
    torques2[i] = t;
}

// step()'s first launch: the action prologue (hector_env.py:158-169) and the first decimation sub-step's torques
// (legged_robot.py:93-94) in one kernel - a thread owns a DOF pair of one env, so it can run the prologue of its two
// actions and go straight on to the PD law.
__global__ void __launch_bounds__(256)
prologue_pd_kernel(const float *__restrict__ a_in, float *__restrict__ actions, const __grid_constant__ hb_env_noise nz,
                   float clip, float action_delay, float action_noise, const float4 *__restrict__ dof_state2,
                   const float2 *__restrict__ kp2, const float2 *__restrict__ kd2, float2 *__restrict__ torques2, int pairs,
                   int ndof, float action_scale, const __grid_constant__ PdConsts c) {
    hb::pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pairs) return;
    const Rng rng = make_rng(nz);
    float2 a;
    a.x = action_prologue(a_in, actions, nz, rng, 2 * i, ndof, clip, action_delay, action_noise);
    a.y = action_prologue(a_in, actions, nz, rng, 2 * i + 1, ndof, clip, action_delay, action_noise);
    reinterpret_cast<float2 *>(actions)[i] = a;
    const float4 s = dof_state2[i];
    const float2 kp = kp2[i], kd = kd2[i];
    const int j = (2 * i) % ndof;
    float2 t;
    t.x = kp.x * ((a.x * action_scale + c.q0[j]) - s.x) - kd.x * s.y;
    t.y = kp.y * ((a.y * action_scale + c.q0[j + 1]) - s.z) - kd.y * s.w;
    t.x = clampf(t.x, -c.lim[j], c.lim[j]);
    t.y = clampf(t.y, -c.lim[j + 1], c.lim[j + 1]);
    torques2[i] = t;
}

__global__ void __launch_bounds__(256)
pd_torque_scalar_kernel(const float *__restrict__ dof_state, const float *__restrict__ actions,
                        const float *__restrict__ kp, const float *__restrict__ kd, float *__restrict__ torques,
                        int total, int ndof, float action_scale, const __grid_constant__ PdConsts c) {
    hb::pdl_trigger();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    hb::pdl_wait();
    if (i >= total) return;
    const int j = i % ndof;
    const float t = kp[i] * ((actions[i] * action_scale + c.q0[j]) - dof_state[2 * i]) - kd[i] * dof_state[2 * i + 1];
    torques[i] = clampf(t, -c.lim[j], c.lim[j]);
}

// ------------------------------------------------------------------------------------------
// a3-a9: post_physics_step.  One CTA = one 32-env tile, four specialised warps, lane = env.
//
//   warp 0 "base"    root quaternion work: base_lin_vel / base_ang_vel / projected_gravity / euler,
//                    command resampling + heading command, push; rewards base_acc, orientation,
//                    tracking_ang_vel, tracking_lin_vel
//   warp 1 "joints"  dof / action terms: action_smoothness, default_joint_pos, dof_acc, dof_vel, torques
//   warp 2 "feet"    gait phase, contacts, termination + time-out -> reset flag; base_height, collision,
//                    feet_air_time, feet_clearance, feet_contact_forces, feet_contact_number,
//                    feet_distance, foot_slip, knee_distance
//   warp 3 "ledger"  episode sums; after the barrier: alphabetical reward accumulation
//                    (legged_robot.py:216-234), reset compaction and episode means
//
// Every warp stays convergent (all lanes run the same code on different envs), the serial chain
// per env is a quarter of the fused version, and each warp only fetches its own slice of code.
// Phase A (rewards, reset flag) | barrier | phase B (reset_idx effects, newest frames, write-back)
// | barrier | coalesced store of the frames.
//
// post_physics_wide_kernel: eight warps, each role a pair of halves (warps 0-2 the first halves of base / joints / feet, 3-5 their second
// halves, 6-7 the ledger pair).  At one or two tiles per SM nothing hides a warp's dependent chain, so the pair splits
// it.  The split is by term: every reward term, frame column, write-back and draw is computed by one half with exactly
// the four-warp kernel's operations (values both halves need are computed by both, the same way), so the two widths
// write bit-identical results.
//   base    first: base_lin/ang_vel, projected_gravity, euler, orientation, vel_mismatch_exp and their columns
//           second: command resampling + heading, push, base_acc, tracking_*, track_vel_hard, low_speed, the root and
//           command write-back and columns
//   joints  first: action_smoothness, default_joint_pos, joint_pos; after barrier 1 the reset of the dofs, the
//           reference trajectory and the privileged columns
//           second: dof_acc, dof_vel, torques, the last_* roll-forward; after barrier 1 the noisy observation columns
//   feet    first: termination, gait, feet_air_time, feet_contact_forces, feet_contact_number, foot_slip, the reset
//           flag and the episode / contact state
//           second: collision, base_height, feet_clearance (and its state), feet_distance, knee_distance, the columns
//   ledger  first: the alphabetical reward sum; second: the episode sums and their reset-env means; both: the noise
// ------------------------------------------------------------------------------------------
struct TileLayout {          // float offsets into the CTA's shared-memory tile
    int root, dof, contact, actions, last_actions, last_last_actions, last_dof_vel, torques, last_root_vel,
        commands, z_obs, terms, gait_s, gait_c, flags, rsums, so, sp, total;
};

// The staged inputs are dead once every role has passed barrier 1 (each lane keeps its env's values in
// registers), so the newest-frame staging tiles so/sp reuse the same bytes: ~19 KB per CTA instead of
// ~38 KB, which is what bounds the number of resident tiles per SM.
// The wide kernel's ledger pair keeps the reset envs' episode sums apart from the terms (rsums), which the other half
// is still reading.
__host__ __device__ constexpr TileLayout make_layout(int nbody, bool with_noise, int NDOF, int OBS, int PRIV, bool wide = false) {
    TileLayout L{};
    int o = 0;
    L.root = o, o += TILE * 13;
    L.dof = o, o += TILE * NDOF * 2;
    L.contact = o, o += TILE * nbody * 3;
    L.actions = o, o += TILE * NDOF;
    L.last_actions = o, o += TILE * NDOF;
    L.last_last_actions = o, o += TILE * NDOF;
    L.last_dof_vel = o, o += TILE * NDOF;
    L.torques = o, o += TILE * NDOF;
    L.last_root_vel = o, o += TILE * 6;
    L.commands = o, o += TILE * 4;
    L.so = 0;
    L.sp = TILE * OBS;
    const int out_end = TILE * (OBS + PRIV);
    o = o > out_end ? o : out_end;
    L.z_obs = o, o += with_noise ? TILE * OBS : 0;      // read by the store loop: must outlive the inputs
    L.terms = o, o += HB_NUM_REWARDS * TILE;
    L.gait_s = o, o += TILE;
    L.gait_c = o, o += TILE;
    L.flags = o, o += TILE;
    L.rsums = o, o += wide ? HB_NUM_REWARDS * TILE : 0;
    L.total = o;
    return L;
}
// dynamic shared memory the launcher allows post_physics_kernel: enough for the largest task (MAX_TASK_DOF joints, the longer
// XBot-L privileged frame, 32 bodies, observation noise)
constexpr int POST_SMEM_MAX = 96 * 1024;
static_assert(make_layout(32, true, MAX_TASK_DOF, task_dims(MAX_TASK_DOF, KIND_XBOT, 0, 0, 0, 0).OBS,
                          task_dims(MAX_TASK_DOF, KIND_XBOT, 0, 0, 0, 0).PRIV, true).total * 4 <= POST_SMEM_MAX,
              "the largest task's tile fits the dynamic shared memory of post_physics_kernel");

// a compile-time flag passed as an argument (which halves of its role a post_physics_kernel warp computes)
template <bool V>
struct On {
    __device__ constexpr operator bool() const { return V; }
};

// all warps of the tile (named barrier 1: the roles meet at different program points)
template <bool kWide = false>
__device__ __forceinline__ void tile_barrier() {
    if constexpr (kWide) asm volatile("bar.sync 1, 256;" ::: "memory");
    else asm volatile("bar.sync 1, 128;" ::: "memory");
}

__device__ __forceinline__ float norm3(const float *f) { return sqrtf((f[0] * f[0] + f[1] * f[1]) + f[2] * f[2]); }

// torch.remainder(a, 2*pi) for |a| < 2*pi (every angle here), general fmodf path kept out of line
__device__ __noinline__ float py_mod_slow(float a, float m) { return py_mod(a, m); }
__device__ __forceinline__ float mod_two_pi(float a) {
    if (fabsf(a) < TWO_PI_F) return (a < 0.0f) ? a + TWO_PI_F : a;
    return py_mod_slow(a, TWO_PI_F);
}
// get_euler_xyz_tensor (envs/base/legged_robot.py:50-55) over isaacgym get_euler_xyz
__device__ __noinline__ Vec3 euler_xyz_wrapped_nl(float x, float y, float z, float w) {
    float roll = atan2f(2.0f * (w * x + y * z), ((w * w - x * x) - y * y) + z * z);
    const float sinp = 2.0f * (w * y - z * x);
    float pitch;
    if (fabsf(sinp) >= 1.0f) {
        const float sg = (sinp > 0.0f) ? 1.0f : ((sinp < 0.0f) ? -1.0f : 0.0f);
        pitch = HALF_PI_F * sg;
    } else {
        pitch = asinf(sinp);
    }
    float yaw = atan2f(2.0f * (w * z + x * y), ((w * w + x * x) - y * y) - z * z);
    roll = mod_two_pi(roll), pitch = mod_two_pi(pitch), yaw = mod_two_pi(yaw);
    if (roll > PI_F) roll -= TWO_PI_F;
    if (pitch > PI_F) pitch -= TWO_PI_F;
    if (yaw > PI_F) yaw -= TWO_PI_F;
    return {roll, pitch, yaw};
}

#ifdef HB_POST_TIMING
// debug build: per-(tile, warp) SM-clock stamps at the phase boundaries of post_physics_kernel (8 warp rows per tile:
// the four-warp kernel fills the first four)
__device__ long long g_post_stamps[4096 * 8 * 8];
__device__ unsigned long long g_post_gt[4096 * 3];          // globaltimer ns: CTA start, stores done, tail done
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define HB_GT(slot)                                                                        \
    do {                                                                                   \
        if (threadIdx.x == 0 && blockIdx.x < 4096) g_post_gt[blockIdx.x * 3 + (slot)] = gtime(); \
    } while (0)
#define HB_STAMP(slot)                                                                                   \
    do {                                                                                                 \
        if (lane == 0 && blockIdx.x < 4096) g_post_stamps[(blockIdx.x * 8 + warp) * 8 + (slot)] = clock64(); \
    } while (0)
#else
#define HB_STAMP(slot) do { } while (0)
#define HB_GT(slot) do { } while (0)
#endif

template <bool kBulk, typename T>
__global__ void __launch_bounds__(4 * TILE, T::RUNTIME ? 4 : (T::CAP <= 12 ? 8 : 5))
post_physics_kernel(const __grid_constant__ hb_env_params p, const __grid_constant__ hb_env_buffers b,
                    const __grid_constant__ hb_env_noise nz, float *__restrict__ obs_new,
                    float *__restrict__ priv_new, int stages) {
    constexpr int KIND = T::KIND, CAP = T::CAP;
    const auto D = T::dims(p);      // (the three robots: every D.X below is a constant expression)
    const int NDOF = D.NDOF, OBS = D.OBS, PRIV = D.PRIV, PRIV_PAD = D.PRIV, U_RESET = D.U_RESET;
    extern __shared__ __align__(128) float sm[];
    __shared__ __align__(8) uint64_t bar;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int N = p.num_envs;
    const int env0 = blockIdx.x * TILE;
    const int nv = min(TILE, N - env0);
    const int env = env0 + lane;
    const bool valid = lane < nv;
    const int ln = valid ? lane : 0;
    // HB_STAGE_STEP is the whole of post_physics_step in one launch; the finer bits run one of the reference's hooks on
    // its own (check_termination, compute_reward, compute_observations, and the head / tail of post_physics_step), so that
    // a host that calls - or overrides - them one by one gets the same buffers as the fused launch
    const bool do_step = stages & HB_STAGE_STEP;
    const bool do_prepare = do_step || (stages & HB_STAGE_PREPARE);
    const bool do_term = do_step || (stages & HB_STAGE_TERMINATION);
    const bool do_rew = do_step || (stages & HB_STAGE_REWARD);
    const bool do_last = do_step || (stages & HB_STAGE_LAST);
    const bool derive = do_prepare || (stages & HB_STAGE_DERIVE);
    const bool emit_obs = do_step || (stages & HB_STAGE_OBS);
    const bool any_reset = do_step || (stages & (HB_STAGE_RESET_ALL | HB_STAGE_RESET_MASK));
    const Rng rng = make_rng(nz);
    const bool with_noise = p.add_noise && (nz.z_obs != nullptr || rng.on);
    const bool tape_noise = p.add_noise && nz.z_obs != nullptr;
    HB_STAMP(0);
    HB_GT(0);
    const TileLayout L = make_layout(p.num_bodies, with_noise, NDOF, OBS, PRIV);
    const int crow = p.num_bodies * 3;
    const float dt = p.dt;
    const float clip = p.clip_observations;
    float *terms = sm + L.terms;
    float *so = sm + L.so, *sp = sm + L.sp;
    // obs_now = frame + (randn * noise_scale_vec) * noise_level, then the +-clip of step() (hector_env.py:241-243,
    // legged_robot.py:104-105); k is a compile-time column after unrolling
    auto noisy_clip = [&](float v, int k) {
        if (with_noise) v = v + (sm[L.z_obs + ln * OBS + k] * p.noise_scale_vec[k]) * p.noise_level;
        return clampf(v, -clip, clip);
    };
    int *flags = reinterpret_cast<int *>(sm + L.flags);

    // ---------------- stage the tile's input slabs into shared memory ----------------
    hb::pdl_trigger();
    hb::pdl_wait();              // everything above overlapped the tail of the last PD sub-step
    const size_t e0 = env0;
    const bool full = (nv == TILE);
    const bool bulk = kBulk && full;
    if (bulk && threadIdx.x == 0) {
        hb::mbar_init(&bar, 1);
        hb::fence_mbar_init();
        hb::mbar_expect_tx(&bar, TILE * 4u * (13 + 2 * NDOF + crow + 5 * NDOF + 6 + 4 + (tape_noise ? OBS : 0)));
    }
    auto stage = [&](const float *src, int dst, int row) {
        if (bulk) {
            if (threadIdx.x == 0) hb::bulk_g2s(sm + dst, src, TILE * 4u * row, &bar);
        } else {
            const int count = nv * row;
            for (int k = threadIdx.x; k < count; k += blockDim.x) sm[dst + k] = __ldg(src + k);
        }
    };
    stage(b.root_states + e0 * 13, L.root, 13);
    stage(b.dof_state + e0 * NDOF * 2, L.dof, NDOF * 2);
    stage(b.contact_forces + e0 * crow, L.contact, crow);
    stage(b.actions + e0 * NDOF, L.actions, NDOF);
    stage(b.last_actions + e0 * NDOF, L.last_actions, NDOF);
    stage(b.last_last_actions + e0 * NDOF, L.last_last_actions, NDOF);
    stage(b.last_dof_vel + e0 * NDOF, L.last_dof_vel, NDOF);
    stage(b.torques + e0 * NDOF, L.torques, NDOF);
    stage(b.last_root_vel + e0 * 6, L.last_root_vel, 6);
    stage(b.commands + e0 * 4, L.commands, 4);
    if (tape_noise) stage(nz.z_obs + e0 * OBS, L.z_obs, OBS);

    __syncthreads();                             // mbarrier init / plain staging visible to every warp
    // Each role first issues its own global loads (they overlap the bulk copies), then waits for the tile.

    // =========================================================================================
    if (warp == 0) {
        long long ep_len = 0;
        float push_f[2] = {0.f, 0.f}, push_t[3] = {0.f, 0.f, 0.f};
        if (valid) {
            ep_len = b.episode_length_buf[env];
            push_f[0] = b.rand_push_force[env * 3], push_f[1] = b.rand_push_force[env * 3 + 1];
#pragma unroll
            for (int k = 0; k < 3; ++k) push_t[k] = b.rand_push_torque[env * 3 + k];
        }
        if (bulk) hb::mbar_wait(&bar, 0);
        HB_STAMP(1);
        float root[13], cmd[4];
#pragma unroll
        for (int k = 0; k < 13; ++k) root[k] = sm[L.root + ln * 13 + k];
#pragma unroll
        for (int k = 0; k < 4; ++k) cmd[k] = sm[L.commands + ln * 4 + k];
        Vec3 lin = {0.f, 0.f, 0.f}, ang = {0.f, 0.f, 0.f}, grav = {0.f, 0.f, 0.f}, eul = {0.f, 0.f, 0.f};
        const float *quat = root + 3;
        if (derive) {        // legged_robot.py:127-135 (and _init_buffers :452,477-479)
            lin = quat_rotate_inverse(quat, {root[7], root[8], root[9]});
            ang = quat_rotate_inverse(quat, {root[10], root[11], root[12]});
            grav = quat_rotate_inverse(quat, {0.0f, 0.0f, -1.0f});
        } else if (valid) {  // reset / observation-only pass: keep the stored values
            lin = {b.base_lin_vel[env * 3], b.base_lin_vel[env * 3 + 1], b.base_lin_vel[env * 3 + 2]};
            ang = {b.base_ang_vel[env * 3], b.base_ang_vel[env * 3 + 1], b.base_ang_vel[env * 3 + 2]};
            grav = {b.projected_gravity[env * 3], b.projected_gravity[env * 3 + 1], b.projected_gravity[env * 3 + 2]};
        }
        eul = euler_xyz_wrapped_nl(quat[0], quat[1], quat[2], quat[3]);
        if (do_prepare) {
            ep_len += 1;
            // -------- _post_physics_step_callback, legged_robot.py:303-335 --------
            if (valid && (ep_len % p.resample_interval) == 0 && (nz.u_cmd || rng.on)) {
                float u[3];
                if (nz.u_cmd) u[0] = nz.u_cmd[(size_t)env * 3], u[1] = nz.u_cmd[(size_t)env * 3 + 1], u[2] = nz.u_cmd[(size_t)env * 3 + 2];
                else rng_uniforms(rng, env, SLOT_U_CMD, 0, 3, u);
                cmd[0] = p.cmd_span[0] * u[0] + p.cmd_lo[0];
                cmd[1] = p.cmd_span[1] * u[1] + p.cmd_lo[1];
                cmd[3] = p.cmd_span[2] * u[2] + p.cmd_lo[2];
                const float keep = (sqrtf(cmd[0] * cmd[0] + cmd[1] * cmd[1]) > 0.2f) ? 1.0f : 0.0f;
                cmd[0] *= keep, cmd[1] *= keep;
            }
            if (p.heading_command) {
                const Vec3 fwd = quat_apply(quat, {1.0f, 0.0f, 0.0f});
                const float heading = atan2f(fwd.y, fwd.x);
                float e = mod_two_pi(cmd[3] - heading);                 // wrap_to_pi, utils/math.py:46-49
                e = e - TWO_PI_F * ((e > PI_F) ? 1.0f : 0.0f);
                cmd[2] = clampf(0.5f * e, -1.0f, 1.0f);
            }
            if ((stages & HB_STAGE_PUSH) && valid && (nz.u_push || rng.on)) {       // _push_robots, hector_env.py:53-68
                float u[5];
                if (nz.u_push) {
#pragma unroll
                    for (int k = 0; k < 5; ++k) u[k] = nz.u_push[(size_t)env * 5 + k];
                } else {
                    rng_uniforms(rng, env, SLOT_U_PUSH, 0, 5, u);
                }
                push_f[0] = p.push_lin_span * u[0] + p.push_lin_lo;
                push_f[1] = p.push_lin_span * u[1] + p.push_lin_lo;
                root[7] = push_f[0], root[8] = push_f[1];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    push_t[k] = p.push_ang_span * u[2 + k] + p.push_ang_lo;
                    root[10 + k] = push_t[k];
                }
                b.rand_push_force[env * 3] = push_f[0], b.rand_push_force[env * 3 + 1] = push_f[1];
#pragma unroll
                for (int k = 0; k < 3; ++k) b.rand_push_torque[env * 3 + k] = push_t[k];
            }
        }
        if (do_rew) {
            {   // base_acc, hector_env.py:385-392 (root velocity after the push)
                float ss = 0.f;
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const float d = sm[L.last_root_vel + ln * 6 + k] - root[7 + k];
                    ss += d * d;
                }
                terms[HB_R_BASE_ACC * TILE + lane] = expf(-sqrtf(ss) * 3.0f);
            }
            {   // orientation, :341-348
                const float a = expf(-(fabsf(eul.x) + fabsf(eul.y)) * 10.0f);
                const float g = expf(-sqrtf(grav.x * grav.x + grav.y * grav.y) * 20.0f);
                terms[HB_R_ORIENTATION * TILE + lane] = (a + g) / 2.0f;
            }
            {   // tracking_ang_vel :435-443, tracking_lin_vel :426-433
                const float ea = (cmd[2] - ang.z) * (cmd[2] - ang.z);
                terms[HB_R_TRACKING_ANG_VEL * TILE + lane] = expf(-ea * p.tracking_sigma);
                const float ex = cmd[0] - lin.x, ey = cmd[1] - lin.y;
                terms[HB_R_TRACKING_LIN_VEL * TILE + lane] = expf(-(ex * ex + ey * ey) * p.tracking_sigma);
            }
            if (T::OPT && p.reward_scale[HB_R_VEL_MISMATCH_EXP] != 0.0f) {      // hector_env.py:395-405
                const float lm = expf(-(lin.z * lin.z) * 10.0f);
                const float am = expf(-sqrtf(ang.x * ang.x + ang.y * ang.y) * 5.0f);
                terms[HB_R_VEL_MISMATCH_EXP * TILE + lane] = (lm + am) / 2.0f;
            }
            if (T::OPT && p.reward_scale[HB_R_TRACK_VEL_HARD] != 0.0f) {        // :407-424
                const float ex = cmd[0] - lin.x, ey = cmd[1] - lin.y;
                const float le = sqrtf(ex * ex + ey * ey), ae = fabsf(cmd[2] - ang.z);
                terms[HB_R_TRACK_VEL_HARD * TILE + lane] = (expf(-le * 10.0f) + expf(-ae * 10.0f)) / 2.0f - 0.2f * (le + ae);
            }
            if (T::OPT && p.reward_scale[HB_R_LOW_SPEED] != 0.0f) {             // :468-499
                const float sp_abs = fabsf(lin.x), cm_abs = fabsf(cmd[0]);
                const bool too_low = sp_abs < 0.5f * cm_abs, too_high = sp_abs > 1.2f * cm_abs;
                const float sgn_v = (lin.x > 0.0f) ? 1.0f : ((lin.x < 0.0f) ? -1.0f : 0.0f);
                const float sgn_c = (cmd[0] > 0.0f) ? 1.0f : ((cmd[0] < 0.0f) ? -1.0f : 0.0f);
                float r = 0.0f;
                if (too_low) r = -1.0f;
                if (too_high) r = 0.0f;
                if (!(too_low || too_high)) r = 1.2f;
                if (sgn_v != sgn_c) r = -2.0f;
                r = r * ((cm_abs > 0.1f) ? 1.0f : 0.0f);
                terms[HB_R_LOW_SPEED * TILE + lane] = r;
            }
        }
        HB_STAMP(2);
        tile_barrier();                                           // ---- barrier 1 ----
        HB_STAMP(3);
        const bool reset = valid && (flags[lane] & 1);
        const float gs = reset ? 0.0f : sm[L.gait_s + lane], gc = reset ? 1.0f : sm[L.gait_c + lane];
        if (reset) {         // _reset_root_states + _resample_commands + the gravity/euler fix-up (:373-396,321-335,211-214)
            float u5[5];        // root xy jitter (2) and the command draws (3): columns NDOF .. NDOF+4 of the reset draws
            if (nz.u_reset) {
#pragma unroll
                for (int k = 0; k < 5; ++k) u5[k] = nz.u_reset[(size_t)env * U_RESET + NDOF + k];
            } else {
                rng_uniforms(rng, env, SLOT_U_RESET, NDOF, 5, u5);
            }
#pragma unroll
            for (int k = 0; k < 13; ++k) root[k] = p.base_init_state[k];
#pragma unroll
            for (int k = 0; k < 3; ++k) root[k] += b.env_origins[env * 3 + k];
            if (p.custom_origins) {
                root[0] += p.reset_xy_span * u5[0] + p.reset_xy_lo;
                root[1] += p.reset_xy_span * u5[1] + p.reset_xy_lo;
            }
            cmd[0] = p.cmd_span[0] * u5[2] + p.cmd_lo[0];
            cmd[1] = p.cmd_span[1] * u5[3] + p.cmd_lo[1];
            cmd[3] = p.cmd_span[2] * u5[4] + p.cmd_lo[2];
            const float keep = (sqrtf(cmd[0] * cmd[0] + cmd[1] * cmd[1]) > 0.2f) ? 1.0f : 0.0f;
            cmd[0] *= keep, cmd[1] *= keep;
            grav = {p.reset_gravity[0], p.reset_gravity[1], p.reset_gravity[2]};
            eul = {p.reset_euler[0], p.reset_euler[1], p.reset_euler[2]};
        }
        if (valid) {
            if (reset) {
#pragma unroll
                for (int k = 0; k < 13; ++k) b.root_states[(size_t)env * 13 + k] = root[k];
            } else if (stages & HB_STAGE_PUSH) {
                b.root_states[(size_t)env * 13 + 7] = root[7], b.root_states[(size_t)env * 13 + 8] = root[8];
#pragma unroll
                for (int k = 0; k < 3; ++k) b.root_states[(size_t)env * 13 + 10 + k] = root[10 + k];
            }
            if (derive) {
                b.base_lin_vel[env * 3] = lin.x, b.base_lin_vel[env * 3 + 1] = lin.y, b.base_lin_vel[env * 3 + 2] = lin.z;
                b.base_ang_vel[env * 3] = ang.x, b.base_ang_vel[env * 3 + 1] = ang.y, b.base_ang_vel[env * 3 + 2] = ang.z;
            }
            if (do_last) {
#pragma unroll
                for (int k = 0; k < 6; ++k) b.last_root_vel[(size_t)env * 6 + k] = root[7 + k];
            }
            b.projected_gravity[env * 3] = grav.x, b.projected_gravity[env * 3 + 1] = grav.y, b.projected_gravity[env * 3 + 2] = grav.z;
            b.base_euler_xyz[env * 3] = eul.x, b.base_euler_xyz[env * 3 + 1] = eul.y, b.base_euler_xyz[env * 3 + 2] = eul.z;
#pragma unroll
            for (int k = 0; k < 4; ++k) b.commands[(size_t)env * 4 + k] = cmd[k];
        }
        if (emit_obs) {      // command input, base velocities, euler, root position, push (hector_env.py:186-226)
            const int B0 = D.B0;
            float o[11];
            o[0] = gs, o[1] = gc;
            o[2] = cmd[0] * p.obs_lin_vel, o[3] = cmd[1] * p.obs_lin_vel, o[4] = cmd[2] * p.obs_ang_vel;
            o[5] = ang.x * p.obs_ang_vel, o[6] = ang.y * p.obs_ang_vel, o[7] = ang.z * p.obs_ang_vel;
            o[8] = eul.x * p.obs_quat, o[9] = eul.y * p.obs_quat, o[10] = eul.z * p.obs_quat;
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                so[lane * OBS + k] = noisy_clip(o[k], k);
                sp[lane * PRIV_PAD + k] = clampf(o[k], -clip, clip);
            }
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                sp[lane * PRIV_PAD + D.P_ANG + k] = clampf(o[5 + k], -clip, clip);
                so[lane * OBS + B0 + k] = noisy_clip(o[5 + k], B0 + k);
            }
            sp[lane * PRIV_PAD + D.P_LIN] = clampf(lin.x * p.obs_lin_vel, -clip, clip);
            sp[lane * PRIV_PAD + D.P_LIN + 1] = clampf(lin.y * p.obs_lin_vel, -clip, clip);
            sp[lane * PRIV_PAD + D.P_LIN + 2] = clampf(lin.z * p.obs_lin_vel, -clip, clip);
            if (KIND == KIND_HECTOR) {
#pragma unroll
                for (int k = 0; k < 3; ++k) sp[lane * PRIV_PAD + D.P_ROOT + k] = clampf(root[k], -clip, clip);
            }
            sp[lane * PRIV_PAD + D.P_PUSH_F] = clampf(push_f[0], -clip, clip);
            sp[lane * PRIV_PAD + D.P_PUSH_F + 1] = clampf(push_f[1], -clip, clip);
#pragma unroll
            for (int k = 0; k < 3; ++k) sp[lane * PRIV_PAD + D.P_PUSH_T + k] = clampf(push_t[k], -clip, clip);
        }
    } else if (warp == 1) {
        // ================================ joints ================================
        if (bulk) hb::mbar_wait(&bar, 0);
        HB_STAMP(1);
        // Only q, qd and the actions stay live across the barrier; the previous-step buffers are consumed
        // (and, on a step, rolled forward: legged_robot.py:146-148) joint by joint before it.
        // The reference trajectory (compute_ref_state, hector_env.py:90-111 / humanoid_env.py:120-142) is STATE: it is
        // refreshed inside compute_observations, so the joint_pos reward of a step sees the one the previous step left.
        const bool joint_pos_on = T::OPT && p.reward_scale[HB_R_JOINT_POS] != 0.0f;
        const bool use_ref = T::OPT && (KIND == KIND_XBOT || joint_pos_on) && b.ref_dof_pos != nullptr;
        long long ep_len = 0;
        if (use_ref && valid) ep_len = b.episode_length_buf[env] + (do_prepare ? 1 : 0);
        float q[CAP], qd[CAP], act[CAP];
#pragma unroll
        for (int j = 0; j < CAP; ++j) {
            if (T::RUNTIME && j == NDOF) break;
            q[j] = sm[L.dof + ln * NDOF * 2 + 2 * j];
            qd[j] = sm[L.dof + ln * NDOF * 2 + 2 * j + 1];
            act[j] = sm[L.actions + ln * NDOF + j];
        }
        if (do_rew || do_last) {
            float t1 = 0.f, t2 = 0.f, t3 = 0.f, ss = 0.f, acc = 0.f, vel = 0.f, tq = 0.f, rr = 0.f;
            float dy0 = 0.f, dy1 = 0.f, dy2 = 0.f, dy3 = 0.f, da0 = 0.f, da1 = 0.f, da2 = 0.f, da3 = 0.f;
            const int yl = D.YAW_L, yr_ = D.YAW_R, al = D.ARM_L, ar_ = D.ARM_R;      // (checked against p by the launcher)
#pragma unroll
            for (int j = 0; j < CAP; ++j) {
                if (T::RUNTIME && j == NDOF) break;
                const float lact = sm[L.last_actions + ln * NDOF + j];
                const float llact = sm[L.last_last_actions + ln * NDOF + j];
                const float ldv = sm[L.last_dof_vel + ln * NDOF + j];
                const float d1 = lact - act[j];                        // action_smoothness, hector_env.py:529-539
                t1 += d1 * d1;
                const float d2 = (act[j] + llact) - 2.0f * lact;
                t2 += d2 * d2;
                t3 += fabsf(act[j]);
                const float d = q[j] - p.default_dof_pos[j];           // default_joint_pos, :357-367
                ss += d * d;
                // hip yaw / roll of both legs (and, hector_full, the first two arm joints of both arms:
                // hector_w_arm_env.py:371-378); the index pairs are task constants
                // (j is a compile-time value in the unrolled loop: these are plain register copies)
                dy0 = (j == yl) ? d : dy0, dy1 = (j == yl + 1) ? d : dy1;
                dy2 = (j == yr_) ? d : dy2, dy3 = (j == yr_ + 1) ? d : dy3;
                if (D.HAS_ARMS) {
                    da0 = (j == al) ? d : da0, da1 = (j == al + 1) ? d : da1;
                    da2 = (j == ar_) ? d : da2, da3 = (j == ar_ + 1) ? d : da3;
                }
                if (joint_pos_on && use_ref && do_rew) {               // joint_pos, hector_env.py:264-275
                    const float e = q[j] - (valid ? b.ref_dof_pos[(size_t)env * NDOF + j] : 0.0f);
                    rr += e * e;
                }
                const float a = (ldv - qd[j]) / dt;                    // dof_acc :515-520
                acc += a * a;
                vel += qd[j] * qd[j];                                  // dof_vel :508-513
                const float tau = sm[L.torques + ln * NDOF + j];       // torques :501-506
                tq += tau * tau;
                if (valid && do_last) {                                // legged_robot.py:146-148 (reset envs: zeroed below)
                    b.last_last_actions[(size_t)env * NDOF + j] = lact;
                    b.last_actions[(size_t)env * NDOF + j] = act[j];
                    b.last_dof_vel[(size_t)env * NDOF + j] = qd[j];
                }
            }
            if (do_rew) {
                terms[HB_R_ACTION_SMOOTHNESS * TILE + lane] = (t1 + t2) + 0.05f * t3;
                float yr = sqrtf(dy0 * dy0 + dy1 * dy1) + sqrtf(dy2 * dy2 + dy3 * dy3);
                yr = clampf(yr - 0.1f, 0.0f, 50.0f);
                float djp = expf(-yr * 100.0f);
                if (D.HAS_ARMS) {
                    float ar = sqrtf(da0 * da0 + da1 * da1) + sqrtf(da2 * da2 + da3 * da3);
                    ar = clampf(ar - 0.1f, 0.0f, 25.0f);
                    djp = djp + expf(-ar * 2.0f);
                }
                terms[HB_R_DEFAULT_JOINT_POS * TILE + lane] = djp - 0.01f * sqrtf(ss);
                if (joint_pos_on) {
                    const float nrm = sqrtf(rr);
                    terms[HB_R_JOINT_POS * TILE + lane] = expf(-2.0f * nrm) - 0.2f * clampf(nrm, 0.0f, 0.5f);
                }
                terms[HB_R_DOF_ACC * TILE + lane] = acc;
                terms[HB_R_DOF_VEL * TILE + lane] = vel;
                terms[HB_R_TORQUES * TILE + lane] = tq;
            }
        }
        HB_STAMP(2);
        tile_barrier();                                           // ---- barrier 1 ----
        HB_STAMP(3);
        const bool reset = valid && (flags[lane] & 1);
        if (reset) {         // _reset_dofs (legged_robot.py:358-372) + buffer zeroing (:186-191)
            float u[CAP];
            if (nz.u_reset) {
#pragma unroll
                for (int j = 0; j < CAP; ++j) {
                    if (T::RUNTIME && j == NDOF) break;
                    u[j] = nz.u_reset[(size_t)env * U_RESET + j];
                }
            } else {
                rng_uniforms(rng, env, SLOT_U_RESET, 0, NDOF, u);
            }
#pragma unroll
            for (int j = 0; j < CAP; ++j) {
                if (T::RUNTIME && j == NDOF) break;
                q[j] = p.default_dof_pos[j] + (p.reset_dof_span * u[j] + p.reset_dof_lo);
                qd[j] = 0.0f;
                act[j] = 0.0f;
                b.dof_state[((size_t)env * NDOF + j) * 2] = q[j];
                b.dof_state[((size_t)env * NDOF + j) * 2 + 1] = 0.0f;
                b.actions[(size_t)env * NDOF + j] = 0.0f;
                b.last_actions[(size_t)env * NDOF + j] = 0.0f;
                b.last_last_actions[(size_t)env * NDOF + j] = 0.0f;
                b.last_dof_vel[(size_t)env * NDOF + j] = 0.0f;
            }
        }
        if (emit_obs) {
            float sl = 0.0f, sr = 0.0f;
            if (use_ref) {       // compute_ref_state of this compute_observations call
                if (reset) ep_len = 0;
                const float sn = sinf(TWO_PI_F * (((float)ep_len * dt) / p.cycle_time));
                sl = fminf(sn, 0.0f), sr = fmaxf(sn, 0.0f);
                if (fabsf(sn) < 0.1f) sl = sr = 0.0f;               // double support
            }
#pragma unroll
            for (int j = 0; j < CAP; ++j) {
                if (T::RUNTIME && j == NDOF) break;
                if (use_ref) {
                    float ref = 0.0f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const float sc = (k == 1) ? p.ref_scale[1] : p.ref_scale[0];
                        if (j == p.ref_left[k]) ref = sl * sc;
                        if (j == p.ref_right[k]) ref = sr * sc;
                    }
                    if (valid) b.ref_dof_pos[(size_t)env * NDOF + j] = ref;
                    if (KIND == KIND_XBOT) sp[lane * PRIV_PAD + D.P_DIFF + j] = clampf(q[j] - ref, -clip, clip);
                }
                float v0 = (q[j] - p.default_dof_pos[j]) * p.obs_dof_pos, v1 = qd[j] * p.obs_dof_vel;
                sp[lane * PRIV_PAD + 5 + j] = clampf(v0, -clip, clip);
                sp[lane * PRIV_PAD + 5 + NDOF + j] = clampf(v1, -clip, clip);
                sp[lane * PRIV_PAD + 5 + 2 * NDOF + j] = clampf(act[j], -clip, clip);
                so[lane * OBS + 5 + j] = noisy_clip(v0, 5 + j);
                so[lane * OBS + 5 + NDOF + j] = noisy_clip(v1, 5 + NDOF + j);
                so[lane * OBS + 5 + 2 * NDOF + j] = noisy_clip(act[j], 5 + 2 * NDOF + j);
            }
        }
    } else if (warp == 2) {
        // ================================ feet / contacts / gait ================================
        long long ep_len = 0;
        float foot_pos[2][3], foot_vel[2][3], knee_xy[2][2], air[2], fh[2], lz[2];
        bool last_ct[2];
        float friction, mass;
        {
            const int ev = valid ? env : env0;         // invalid lanes of a ragged tile mirror the tile's first env
            ep_len = b.episode_length_buf[ev];
            friction = b.env_frictions[ev], mass = b.body_mass[ev];
            const float *rs = b.rigid_state + (size_t)ev * p.num_bodies * 13;
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                const float *r = rs + p.feet[f] * 13;
#pragma unroll
                for (int k = 0; k < 3; ++k) foot_pos[f][k] = __ldg(r + k), foot_vel[f][k] = __ldg(r + 7 + k);
                const float *kr = rs + p.knees[f] * 13;
                knee_xy[f][0] = __ldg(kr), knee_xy[f][1] = __ldg(kr + 1);
                air[f] = b.feet_air_time[ev * 2 + f];
                fh[f] = b.feet_height[ev * 2 + f];
                lz[f] = b.last_feet_z[ev * 2 + f];
                last_ct[f] = b.last_contacts[ev * 2 + f] != 0;
            }
        }
        if (bulk) hb::mbar_wait(&bar, 0);
        HB_STAMP(1);
        const float *cf = sm + L.contact + ln * crow;
        float foot_f[2][3];
#pragma unroll
        for (int f = 0; f < 2; ++f)
#pragma unroll
            for (int k = 0; k < 3; ++k) foot_f[f][k] = cf[p.feet[f] * 3 + k];
        const float root_z = sm[L.root + ln * 13 + 2];
        bool term = false, time_out = false;
        float gs = 0.0f, gc = 1.0f, st[2] = {1.0f, 1.0f};
        const bool ct[2] = {foot_f[0][2] > 5.0f, foot_f[1][2] > 5.0f};
        if (do_prepare) ep_len += 1;
        if (do_term) {   // -------- check_termination, legged_robot.py:155-160 --------
#pragma unroll 1
            for (int i = 0; i < p.n_term; ++i) term |= norm3(cf + p.term_bodies[i] * 3) > 1.0f;
            time_out = ep_len > (long long)p.max_episode_length;
            term |= time_out;
        }
        if (do_rew) {    // collision, hector_env.py:522-527
            float coll = 0.f;
#pragma unroll 1
            for (int i = 0; i < p.n_pen; ++i) coll += (norm3(cf + p.pen_bodies[i] * 3) > 0.1f) ? 1.0f : 0.0f;
            terms[HB_R_COLLISION * TILE + lane] = coll;
        }
        bool reset = do_step && term;        // the fused step resets what it has just found terminated
        {   // -------- gait phase, hector_env.py:70-88 --------
            const float arg = TWO_PI_F * (((float)ep_len * dt) / p.cycle_time);
            sincosf(arg, &gs, &gc);
            st[0] = (gs >= 0.0f) ? 1.0f : 0.0f, st[1] = (gs < 0.0f) ? 1.0f : 0.0f;
            if (fabsf(gs) < 0.1f) st[0] = st[1] = 1.0f;
        }
        if (do_rew) {
            {   // base_height, :369-383
                const float ground = (foot_pos[0][2] * st[0] + foot_pos[1][2] * st[1]) / (st[0] + st[1]);
                const float h = root_z - (ground - 0.05f);
                terms[HB_R_BASE_HEIGHT * TILE + lane] = expf(-fabsf(h - p.base_height_target) * 100.0f);
            }
            float r_air = 0.f, r_clr = 0.f, cfz = 0.f, num = 0.f, slip = 0.f;
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                {   // feet_air_time, :315-329 (stateful)
                    const bool filt = ct[f] || (st[f] != 0.0f) || last_ct[f];
                    last_ct[f] = ct[f];
                    const bool first = (air[f] > 0.0f) && filt;
                    air[f] += dt;
                    r_air += clampf(air[f], 0.0f, 0.5f) * (first ? 1.0f : 0.0f);
                    air[f] *= filt ? 0.0f : 1.0f;
                }
                {   // feet_clearance, :445-466 (stateful)
                    const float z = foot_pos[f][2] - 0.05f;
                    fh[f] += z - lz[f];
                    lz[f] = z;
                    const float hit = (fabsf(fh[f] - p.target_feet_height) < 0.01f) ? 1.0f : 0.0f;
                    r_clr += hit * (1.0f - st[f]);
                    fh[f] *= ct[f] ? 0.0f : 1.0f;
                }
                // feet_contact_forces :350-355, feet_contact_number :331-339, foot_slip :303-313
                cfz += clampf(norm3(foot_f[f]) - p.max_contact_force, 0.0f, 400.0f);
                num += (ct[f] == (st[f] != 0.0f)) ? 1.0f : -0.3f;
                const float spd = sqrtf(sqrtf(foot_vel[f][0] * foot_vel[f][0] + foot_vel[f][1] * foot_vel[f][1]));
                slip += spd * (ct[f] ? 1.0f : 0.0f);
            }
            terms[HB_R_FEET_AIR_TIME * TILE + lane] = r_air;
            terms[HB_R_FEET_CLEARANCE * TILE + lane] = r_clr;
            terms[HB_R_FEET_CONTACT_FORCES * TILE + lane] = cfz;
            terms[HB_R_FEET_CONTACT_NUMBER * TILE + lane] = num / 2.0f;
            terms[HB_R_FOOT_SLIP * TILE + lane] = slip;
            {   // feet_distance :277-287, knee_distance :290-300
                float dx = foot_pos[0][0] - foot_pos[1][0], dy = foot_pos[0][1] - foot_pos[1][1];
                float d = sqrtf(dx * dx + dy * dy);
                float dmin = clampf(d - p.min_dist, -0.5f, 0.0f), dmax = clampf(d - p.max_dist, 0.0f, 0.5f);
                terms[HB_R_FEET_DISTANCE * TILE + lane] = (expf(-fabsf(dmin) * 100.0f) + expf(-fabsf(dmax) * 100.0f)) / 2.0f;
                dx = knee_xy[0][0] - knee_xy[1][0], dy = knee_xy[0][1] - knee_xy[1][1];
                d = sqrtf(dx * dx + dy * dy);
                dmin = clampf(d - p.min_dist, -0.5f, 0.0f), dmax = clampf(d - p.max_dist / 2.0f, 0.0f, 0.5f);
                terms[HB_R_KNEE_DISTANCE * TILE + lane] = (expf(-fabsf(dmin) * 100.0f) + expf(-fabsf(dmax) * 100.0f)) / 2.0f;
            }
        }
        if (stages & HB_STAGE_RESET_ALL) reset = true;
        if ((stages & HB_STAGE_RESET_MASK) && valid) reset = reset || (b.reset_buf[env] != 0);   // reset_idx(env_ids)
        reset = reset && valid;
        flags[lane] = (reset ? 1 : 0) | (time_out ? 2 : 0);
        sm[L.gait_s + lane] = gs, sm[L.gait_c + lane] = gc;
        HB_STAMP(2);
        tile_barrier();                                           // ---- barrier 1 ----
        HB_STAMP(3);
        if (reset) {
            ep_len = 0, air[0] = air[1] = 0.0f;
            st[0] = st[1] = 1.0f;                                   // phase 0: sin = 0 -> double support
        }
        if (valid) {
            b.feet_air_time[env * 2] = air[0], b.feet_air_time[env * 2 + 1] = air[1];
            b.episode_length_buf[env] = ep_len;
            if (any_reset) b.reset_buf[env] = reset ? 1 : 0;
            else if (do_term) b.reset_buf[env] = term ? 1 : 0;           // check_termination on its own: the mask only
            if (do_term) b.time_out_buf[env] = time_out ? 1 : 0;
            if (do_rew) {
#pragma unroll
                for (int f = 0; f < 2; ++f) {
                    b.last_contacts[env * 2 + f] = last_ct[f] ? 1 : 0;
                    b.feet_height[env * 2 + f] = fh[f];
                    b.last_feet_z[env * 2 + f] = lz[f];
                }
            }
        }
        if (emit_obs) {
            if (KIND == KIND_HECTOR) {
#pragma unroll
                for (int f = 0; f < 2; ++f)
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        sp[lane * PRIV_PAD + D.P_FEET_POS + f * 3 + k] = clampf(foot_pos[f][k], -clip, clip);
                        sp[lane * PRIV_PAD + D.P_FEET_VEL + f * 3 + k] = clampf(foot_vel[f][k], -clip, clip);
                    }
            }
            sp[lane * PRIV_PAD + D.P_FRICTION] = clampf(friction, -clip, clip);
            sp[lane * PRIV_PAD + D.P_MASS] = clampf(mass / 30.0f, -clip, clip);
            sp[lane * PRIV_PAD + D.P_STANCE] = st[0], sp[lane * PRIV_PAD + D.P_STANCE + 1] = st[1];
            sp[lane * PRIV_PAD + D.P_CONTACT] = ct[0] ? 1.0f : 0.0f, sp[lane * PRIV_PAD + D.P_CONTACT + 1] = ct[1] ? 1.0f : 0.0f;
        }
    } else {
        // ================================ ledger ================================
        // (terms with scale 0 are not part of the task: the reference has no episode sum for them - their rows stay zero
        // and are neither read nor written)
        float sums[HB_NUM_REWARDS];
#pragma unroll
        for (int k = 0; k < HB_NUM_REWARDS; ++k)
            sums[k] = (valid && p.reward_scale[k] != 0.0f) ? b.episode_sums[(size_t)k * N + env] : 0.0f;
        if (with_noise && !tape_noise && emit_obs) {
            // the tile's observation noise, drawn by this otherwise idle warp while the other roles are in phase A:
            // 11 Philox calls of 4 normals per env; calls whose four columns all have zero noise scale are skipped
            const int CALLS = (OBS + 3) / 4;
            float *z = sm + L.z_obs;
            for (int c = lane; c < nv * CALLS; c += 32) {
                const int e = c / CALLS, q = c - e * CALLS;
                bool any = false;
#pragma unroll
                for (int k = 0; k < 4; ++k) any = any || (q * 4 + k < OBS && p.noise_scale_vec[q * 4 + k] != 0.0f);
                float z4[4] = {0.f, 0.f, 0.f, 0.f};
                if (any) rng_normal4(rng, env0 + e, SLOT_Z_OBS + q, z4);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (q * 4 + k < OBS) z[e * OBS + q * 4 + k] = z4[k];
            }
        }
        HB_STAMP(2);
        tile_barrier();                                           // ---- barrier 1 ----
        HB_STAMP(3);
        const bool reset = valid && (flags[lane] & 1);
        if (do_rew) {        // compute_reward, legged_robot.py:216-234: alphabetical accumulation
            float rew = 0.0f;
#pragma unroll
            for (int k = 0; k < HB_NUM_REWARDS; ++k) {
                if (p.reward_scale[k] != 0.0f) {
                    const float r = terms[k * TILE + lane] * p.reward_scale[k];
                    rew += r;
                    sums[k] += r;
                }
            }
            if (p.only_positive_rewards) rew = fmaxf(rew, 0.0f);
            if (valid) b.rew_buf[env] = rew;
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, reset);
        __syncwarp();
#pragma unroll
        for (int k = 0; k < HB_NUM_REWARDS; ++k) {
            if (p.reward_scale[k] != 0.0f) {
                terms[k * TILE + lane] = reset ? sums[k] : 0.0f;    // episode sums of the envs being reset (:198-201)
                if (reset) sums[k] = 0.0f;
                if (valid) b.episode_sums[(size_t)k * N + env] = sums[k];
            }
        }
        __syncwarp();
        // ---------------- reset ids + episode means ----------------
        // Each tile publishes its ballot; reset_finalize_kernel turns the ballots into the ascending id
        // list (like reset_buf.nonzero()) and the count.  The per-term sums of the reset envs
        // (legged_robot.py:198-201) go straight into 18 fp64 accumulators: fp64 addition of these
        // fp32 values is order-independent far below fp32 resolution.
        if (ballot && lane < HB_NUM_REWARDS && p.reward_scale[lane] != 0.0f) {
            float v = 0.0f;
#pragma unroll 8
            for (int e = 0; e < TILE; ++e) v += terms[lane * TILE + ((e + lane) & 31)];
            atomicAdd(b.scratch_sums + lane, (double)v);
        }
        if (lane == 0) b.scratch_ballots[blockIdx.x] = ballot;     // consumed by reset_finalize_kernel
    }

    // ---------------- coalesced store of the newest frames into the last slot of the stacked buffers ----------------
    // by the three roles that wrote them (named barrier 2, 96 threads); the ledger warp is busy with its ticket
    HB_STAMP(4);
    if (warp < 3) {
        asm volatile("bar.sync 2, 96;" ::: "memory");             // ---- barrier 2 ----
        HB_STAMP(5);
        if (emit_obs) {
            // 96 threads walk the tile's frames with (row, column) advanced incrementally: no per-element division.
            // Privileged frames leave as 8-byte pairs (row starts are 8-byte aligned: 4200 r + 3920 bytes).
            constexpr int NT = 3 * TILE;
            const int P2 = PRIV / 2;
            const int orow = p.frame_stack * OBS, prow = p.c_frame_stack * PRIV;
            const int ostride = p.obs_ld ? p.obs_ld : orow, pstride = p.priv_ld ? p.priv_ld : prow;   // row pitch
            const int t = threadIdx.x;
            if ((PRIV & 1) == 0 && ((pstride | prow) & 1) == 0 && (reinterpret_cast<uintptr_t>(priv_new) & 7u) == 0) {
                int r = t / P2, c2 = t - r * P2;
                float2 *dst = reinterpret_cast<float2 *>(priv_new + (size_t)env0 * pstride + (prow - PRIV));
                const float2 *src = reinterpret_cast<const float2 *>(sp);
                const int half = pstride / 2;
                while (r < nv) {
                    dst[(size_t)r * half + c2] = src[r * P2 + c2];
                    r += NT / P2, c2 += NT % P2;
                    if (c2 >= P2) c2 -= P2, r += 1;
                }
            } else {
                int r = t / PRIV, c = t - r * PRIV;
                while (r < nv) {
                    priv_new[(size_t)(env0 + r) * pstride + (prow - PRIV) + c] = sp[r * PRIV + c];
                    r += NT / PRIV, c += NT % PRIV;
                    if (c >= PRIV) c -= PRIV, r += 1;
                }
            }
            int r = t / OBS, c = t - r * OBS;
            float *dst = obs_new + (size_t)env0 * ostride + (orow - OBS);
            while (r < nv) {
                dst[(size_t)r * ostride + c] = so[r * OBS + c];
                r += NT / OBS, c += NT % OBS;
                if (c >= OBS) c -= OBS, r += 1;
            }
        }
    }
    HB_STAMP(6);
    HB_GT(1);
}

// The eight-warp kernel (described above): the roles' code of post_physics_kernel with each term under the flag of the half
// that computes it.  It runs where at most a few tiles share an SM: its register budget is that of two resident tiles.
template <bool kBulk, typename T>
__global__ void __launch_bounds__(8 * TILE, 2)
post_physics_wide_kernel(const __grid_constant__ hb_env_params p, const __grid_constant__ hb_env_buffers b,
                    const __grid_constant__ hb_env_noise nz, float *__restrict__ obs_new,
                    float *__restrict__ priv_new, int stages) {
    constexpr int KIND = T::KIND, CAP = T::CAP;
    const auto D = T::dims(p);      // (the three robots: every D.X below is a constant expression)
    const int NDOF = D.NDOF, OBS = D.OBS, PRIV = D.PRIV, PRIV_PAD = D.PRIV, U_RESET = D.U_RESET;
    extern __shared__ __align__(128) float sm[];
    __shared__ __align__(8) uint64_t bar;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int role = warp < 6 ? warp % 3 : 3;      // 0 base, 1 joints, 2 feet, 3 ledger
    const bool second = warp < 6 ? warp >= 3 : warp == 7;      // the warp runs its role's second half
    // A role body takes (h0, h1): whether it computes its role's first / second half of the terms, as compile-time
    // constants so that each half's code is compiled on its own
    auto run = [&](auto &&body) {
        if (!second) body(On<true>{}, On<false>{});
        else body(On<false>{}, On<true>{});
    };
    const int N = p.num_envs;
    const int env0 = blockIdx.x * TILE;
    const int nv = min(TILE, N - env0);
    const int env = env0 + lane;
    const bool valid = lane < nv;
    const int ln = valid ? lane : 0;
    // HB_STAGE_STEP is the whole of post_physics_step in one launch; the finer bits run one of the reference's hooks on
    // its own (check_termination, compute_reward, compute_observations, and the head / tail of post_physics_step), so that
    // a host that calls - or overrides - them one by one gets the same buffers as the fused launch
    const bool do_step = stages & HB_STAGE_STEP;
    const bool do_prepare = do_step || (stages & HB_STAGE_PREPARE);
    const bool do_term = do_step || (stages & HB_STAGE_TERMINATION);
    const bool do_rew = do_step || (stages & HB_STAGE_REWARD);
    const bool do_last = do_step || (stages & HB_STAGE_LAST);
    const bool derive = do_prepare || (stages & HB_STAGE_DERIVE);
    const bool emit_obs = do_step || (stages & HB_STAGE_OBS);
    const bool any_reset = do_step || (stages & (HB_STAGE_RESET_ALL | HB_STAGE_RESET_MASK));
    const Rng rng = make_rng(nz);
    const bool with_noise = p.add_noise && (nz.z_obs != nullptr || rng.on);
    const bool tape_noise = p.add_noise && nz.z_obs != nullptr;
    HB_STAMP(0);
    HB_GT(0);
    const TileLayout L = make_layout(p.num_bodies, with_noise, NDOF, OBS, PRIV, true);
    const int crow = p.num_bodies * 3;
    const float dt = p.dt;
    const float clip = p.clip_observations;
    float *terms = sm + L.terms;
    float *so = sm + L.so, *sp = sm + L.sp;
    // obs_now = frame + (randn * noise_scale_vec) * noise_level, then the +-clip of step() (hector_env.py:241-243,
    // legged_robot.py:104-105); k is a compile-time column after unrolling
    auto noisy_clip = [&](float v, int k) {
        if (with_noise) v = v + (sm[L.z_obs + ln * OBS + k] * p.noise_scale_vec[k]) * p.noise_level;
        return clampf(v, -clip, clip);
    };
    int *flags = reinterpret_cast<int *>(sm + L.flags);

    // ---------------- stage the tile's input slabs into shared memory ----------------
    hb::pdl_trigger();
    hb::pdl_wait();              // everything above overlapped the tail of the last PD sub-step
    const size_t e0 = env0;
    const bool full = (nv == TILE);
    const bool bulk = kBulk && full;
    if (bulk && threadIdx.x == 0) {
        hb::mbar_init(&bar, 1);
        hb::fence_mbar_init();
        hb::mbar_expect_tx(&bar, TILE * 4u * (13 + 2 * NDOF + crow + 5 * NDOF + 6 + 4 + (tape_noise ? OBS : 0)));
    }
    auto stage = [&](const float *src, int dst, int row) {
        if (bulk) {
            if (threadIdx.x == 0) hb::bulk_g2s(sm + dst, src, TILE * 4u * row, &bar);
        } else {
            const int count = nv * row;
            for (int k = threadIdx.x; k < count; k += blockDim.x) sm[dst + k] = __ldg(src + k);
        }
    };
    stage(b.root_states + e0 * 13, L.root, 13);
    stage(b.dof_state + e0 * NDOF * 2, L.dof, NDOF * 2);
    stage(b.contact_forces + e0 * crow, L.contact, crow);
    stage(b.actions + e0 * NDOF, L.actions, NDOF);
    stage(b.last_actions + e0 * NDOF, L.last_actions, NDOF);
    stage(b.last_last_actions + e0 * NDOF, L.last_last_actions, NDOF);
    stage(b.last_dof_vel + e0 * NDOF, L.last_dof_vel, NDOF);
    stage(b.torques + e0 * NDOF, L.torques, NDOF);
    stage(b.last_root_vel + e0 * 6, L.last_root_vel, 6);
    stage(b.commands + e0 * 4, L.commands, 4);
    if (tape_noise) stage(nz.z_obs + e0 * OBS, L.z_obs, OBS);

    __syncthreads();                             // mbarrier init / plain staging visible to every warp
    // Each role first issues its own global loads (they overlap the bulk copies), then waits for the tile.

    // =========================================================================================
    auto base = [&](auto h0, auto h1) {
        long long ep_len = 0;
        float push_f[2] = {0.f, 0.f}, push_t[3] = {0.f, 0.f, 0.f};
        if (h1 && valid) {
            ep_len = b.episode_length_buf[env];
            push_f[0] = b.rand_push_force[env * 3], push_f[1] = b.rand_push_force[env * 3 + 1];
#pragma unroll
            for (int k = 0; k < 3; ++k) push_t[k] = b.rand_push_torque[env * 3 + k];
        }
        if (bulk) hb::mbar_wait(&bar, 0);
        HB_STAMP(1);
        float root[13], cmd[4];
#pragma unroll
        for (int k = 0; k < 13; ++k) root[k] = sm[L.root + ln * 13 + k];
#pragma unroll
        for (int k = 0; k < 4; ++k) cmd[k] = sm[L.commands + ln * 4 + k];
        Vec3 lin = {0.f, 0.f, 0.f}, ang = {0.f, 0.f, 0.f}, grav = {0.f, 0.f, 0.f}, eul = {0.f, 0.f, 0.f};
        const float *quat = root + 3;
        if (derive) {        // legged_robot.py:127-135 (and _init_buffers :452,477-479)
            lin = quat_rotate_inverse(quat, {root[7], root[8], root[9]});
            ang = quat_rotate_inverse(quat, {root[10], root[11], root[12]});
            grav = quat_rotate_inverse(quat, {0.0f, 0.0f, -1.0f});
        } else if (valid) {  // reset / observation-only pass: keep the stored values
            lin = {b.base_lin_vel[env * 3], b.base_lin_vel[env * 3 + 1], b.base_lin_vel[env * 3 + 2]};
            ang = {b.base_ang_vel[env * 3], b.base_ang_vel[env * 3 + 1], b.base_ang_vel[env * 3 + 2]};
            grav = {b.projected_gravity[env * 3], b.projected_gravity[env * 3 + 1], b.projected_gravity[env * 3 + 2]};
        }
        if (h0) eul = euler_xyz_wrapped_nl(quat[0], quat[1], quat[2], quat[3]);
        if (h1 && do_prepare) {
            ep_len += 1;
            // -------- _post_physics_step_callback, legged_robot.py:303-335 --------
            if (valid && (ep_len % p.resample_interval) == 0 && (nz.u_cmd || rng.on)) {
                float u[3];
                if (nz.u_cmd) u[0] = nz.u_cmd[(size_t)env * 3], u[1] = nz.u_cmd[(size_t)env * 3 + 1], u[2] = nz.u_cmd[(size_t)env * 3 + 2];
                else rng_uniforms(rng, env, SLOT_U_CMD, 0, 3, u);
                cmd[0] = p.cmd_span[0] * u[0] + p.cmd_lo[0];
                cmd[1] = p.cmd_span[1] * u[1] + p.cmd_lo[1];
                cmd[3] = p.cmd_span[2] * u[2] + p.cmd_lo[2];
                const float keep = (sqrtf(cmd[0] * cmd[0] + cmd[1] * cmd[1]) > 0.2f) ? 1.0f : 0.0f;
                cmd[0] *= keep, cmd[1] *= keep;
            }
            if (p.heading_command) {
                const Vec3 fwd = quat_apply(quat, {1.0f, 0.0f, 0.0f});
                const float heading = atan2f(fwd.y, fwd.x);
                float e = mod_two_pi(cmd[3] - heading);                 // wrap_to_pi, utils/math.py:46-49
                e = e - TWO_PI_F * ((e > PI_F) ? 1.0f : 0.0f);
                cmd[2] = clampf(0.5f * e, -1.0f, 1.0f);
            }
            if ((stages & HB_STAGE_PUSH) && valid && (nz.u_push || rng.on)) {       // _push_robots, hector_env.py:53-68
                float u[5];
                if (nz.u_push) {
#pragma unroll
                    for (int k = 0; k < 5; ++k) u[k] = nz.u_push[(size_t)env * 5 + k];
                } else {
                    rng_uniforms(rng, env, SLOT_U_PUSH, 0, 5, u);
                }
                push_f[0] = p.push_lin_span * u[0] + p.push_lin_lo;
                push_f[1] = p.push_lin_span * u[1] + p.push_lin_lo;
                root[7] = push_f[0], root[8] = push_f[1];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    push_t[k] = p.push_ang_span * u[2 + k] + p.push_ang_lo;
                    root[10 + k] = push_t[k];
                }
                b.rand_push_force[env * 3] = push_f[0], b.rand_push_force[env * 3 + 1] = push_f[1];
#pragma unroll
                for (int k = 0; k < 3; ++k) b.rand_push_torque[env * 3 + k] = push_t[k];
            }
        }
        if (do_rew) {
            if (h1) {   // base_acc, hector_env.py:385-392 (root velocity after the push)
                float ss = 0.f;
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    const float d = sm[L.last_root_vel + ln * 6 + k] - root[7 + k];
                    ss += d * d;
                }
                terms[HB_R_BASE_ACC * TILE + lane] = expf(-sqrtf(ss) * 3.0f);
            }
            if (h0) {   // orientation, :341-348
                const float a = expf(-(fabsf(eul.x) + fabsf(eul.y)) * 10.0f);
                const float g = expf(-sqrtf(grav.x * grav.x + grav.y * grav.y) * 20.0f);
                terms[HB_R_ORIENTATION * TILE + lane] = (a + g) / 2.0f;
            }
            if (h1) {   // tracking_ang_vel :435-443, tracking_lin_vel :426-433
                const float ea = (cmd[2] - ang.z) * (cmd[2] - ang.z);
                terms[HB_R_TRACKING_ANG_VEL * TILE + lane] = expf(-ea * p.tracking_sigma);
                const float ex = cmd[0] - lin.x, ey = cmd[1] - lin.y;
                terms[HB_R_TRACKING_LIN_VEL * TILE + lane] = expf(-(ex * ex + ey * ey) * p.tracking_sigma);
            }
            if (h0 && T::OPT && p.reward_scale[HB_R_VEL_MISMATCH_EXP] != 0.0f) {      // hector_env.py:395-405
                const float lm = expf(-(lin.z * lin.z) * 10.0f);
                const float am = expf(-sqrtf(ang.x * ang.x + ang.y * ang.y) * 5.0f);
                terms[HB_R_VEL_MISMATCH_EXP * TILE + lane] = (lm + am) / 2.0f;
            }
            if (h1 && T::OPT && p.reward_scale[HB_R_TRACK_VEL_HARD] != 0.0f) {        // :407-424
                const float ex = cmd[0] - lin.x, ey = cmd[1] - lin.y;
                const float le = sqrtf(ex * ex + ey * ey), ae = fabsf(cmd[2] - ang.z);
                terms[HB_R_TRACK_VEL_HARD * TILE + lane] = (expf(-le * 10.0f) + expf(-ae * 10.0f)) / 2.0f - 0.2f * (le + ae);
            }
            if (h1 && T::OPT && p.reward_scale[HB_R_LOW_SPEED] != 0.0f) {             // :468-499
                const float sp_abs = fabsf(lin.x), cm_abs = fabsf(cmd[0]);
                const bool too_low = sp_abs < 0.5f * cm_abs, too_high = sp_abs > 1.2f * cm_abs;
                const float sgn_v = (lin.x > 0.0f) ? 1.0f : ((lin.x < 0.0f) ? -1.0f : 0.0f);
                const float sgn_c = (cmd[0] > 0.0f) ? 1.0f : ((cmd[0] < 0.0f) ? -1.0f : 0.0f);
                float r = 0.0f;
                if (too_low) r = -1.0f;
                if (too_high) r = 0.0f;
                if (!(too_low || too_high)) r = 1.2f;
                if (sgn_v != sgn_c) r = -2.0f;
                r = r * ((cm_abs > 0.1f) ? 1.0f : 0.0f);
                terms[HB_R_LOW_SPEED * TILE + lane] = r;
            }
        }
        HB_STAMP(2);
        tile_barrier<true>();                                     // ---- barrier 1 ----
        HB_STAMP(3);
        const bool reset = valid && (flags[lane] & 1);
        const float gs = reset ? 0.0f : sm[L.gait_s + lane], gc = reset ? 1.0f : sm[L.gait_c + lane];
        if (reset) {         // _reset_root_states + _resample_commands + the gravity/euler fix-up (:373-396,321-335,211-214)
            if (h1) {
                float u5[5];        // root xy jitter (2) and the command draws (3): columns NDOF .. NDOF+4 of the reset draws
                if (nz.u_reset) {
#pragma unroll
                    for (int k = 0; k < 5; ++k) u5[k] = nz.u_reset[(size_t)env * U_RESET + NDOF + k];
                } else {
                    rng_uniforms(rng, env, SLOT_U_RESET, NDOF, 5, u5);
                }
#pragma unroll
                for (int k = 0; k < 13; ++k) root[k] = p.base_init_state[k];
#pragma unroll
                for (int k = 0; k < 3; ++k) root[k] += b.env_origins[env * 3 + k];
                if (p.custom_origins) {
                    root[0] += p.reset_xy_span * u5[0] + p.reset_xy_lo;
                    root[1] += p.reset_xy_span * u5[1] + p.reset_xy_lo;
                }
                cmd[0] = p.cmd_span[0] * u5[2] + p.cmd_lo[0];
                cmd[1] = p.cmd_span[1] * u5[3] + p.cmd_lo[1];
                cmd[3] = p.cmd_span[2] * u5[4] + p.cmd_lo[2];
                const float keep = (sqrtf(cmd[0] * cmd[0] + cmd[1] * cmd[1]) > 0.2f) ? 1.0f : 0.0f;
                cmd[0] *= keep, cmd[1] *= keep;
            }
            grav = {p.reset_gravity[0], p.reset_gravity[1], p.reset_gravity[2]};
            eul = {p.reset_euler[0], p.reset_euler[1], p.reset_euler[2]};
        }
        if (valid) {
            if (h1 && reset) {
#pragma unroll
                for (int k = 0; k < 13; ++k) b.root_states[(size_t)env * 13 + k] = root[k];
            } else if (h1 && (stages & HB_STAGE_PUSH)) {
                b.root_states[(size_t)env * 13 + 7] = root[7], b.root_states[(size_t)env * 13 + 8] = root[8];
#pragma unroll
                for (int k = 0; k < 3; ++k) b.root_states[(size_t)env * 13 + 10 + k] = root[10 + k];
            }
            if (h0 && derive) {
                b.base_lin_vel[env * 3] = lin.x, b.base_lin_vel[env * 3 + 1] = lin.y, b.base_lin_vel[env * 3 + 2] = lin.z;
                b.base_ang_vel[env * 3] = ang.x, b.base_ang_vel[env * 3 + 1] = ang.y, b.base_ang_vel[env * 3 + 2] = ang.z;
            }
            if (h1 && do_last) {
#pragma unroll
                for (int k = 0; k < 6; ++k) b.last_root_vel[(size_t)env * 6 + k] = root[7 + k];
            }
            if (h0) {
                b.projected_gravity[env * 3] = grav.x, b.projected_gravity[env * 3 + 1] = grav.y, b.projected_gravity[env * 3 + 2] = grav.z;
                b.base_euler_xyz[env * 3] = eul.x, b.base_euler_xyz[env * 3 + 1] = eul.y, b.base_euler_xyz[env * 3 + 2] = eul.z;
            }
            if (h1) {
#pragma unroll
                for (int k = 0; k < 4; ++k) b.commands[(size_t)env * 4 + k] = cmd[k];
            }
        }
        if (emit_obs) {      // command input, base velocities, euler, root position, push (hector_env.py:186-226)
            const int B0 = D.B0;
            float o[11];
            o[0] = gs, o[1] = gc;
            o[2] = cmd[0] * p.obs_lin_vel, o[3] = cmd[1] * p.obs_lin_vel, o[4] = cmd[2] * p.obs_ang_vel;
            o[5] = ang.x * p.obs_ang_vel, o[6] = ang.y * p.obs_ang_vel, o[7] = ang.z * p.obs_ang_vel;
            o[8] = eul.x * p.obs_quat, o[9] = eul.y * p.obs_quat, o[10] = eul.z * p.obs_quat;
            if (h1) {
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    so[lane * OBS + k] = noisy_clip(o[k], k);
                    sp[lane * PRIV_PAD + k] = clampf(o[k], -clip, clip);
                }
            }
            if (h0) {
#pragma unroll
                for (int k = 0; k < 6; ++k) {
                    sp[lane * PRIV_PAD + D.P_ANG + k] = clampf(o[5 + k], -clip, clip);
                    so[lane * OBS + B0 + k] = noisy_clip(o[5 + k], B0 + k);
                }
                sp[lane * PRIV_PAD + D.P_LIN] = clampf(lin.x * p.obs_lin_vel, -clip, clip);
                sp[lane * PRIV_PAD + D.P_LIN + 1] = clampf(lin.y * p.obs_lin_vel, -clip, clip);
                sp[lane * PRIV_PAD + D.P_LIN + 2] = clampf(lin.z * p.obs_lin_vel, -clip, clip);
            }
            if (h1) {
                if (KIND == KIND_HECTOR) {
#pragma unroll
                    for (int k = 0; k < 3; ++k) sp[lane * PRIV_PAD + D.P_ROOT + k] = clampf(root[k], -clip, clip);
                }
                sp[lane * PRIV_PAD + D.P_PUSH_F] = clampf(push_f[0], -clip, clip);
                sp[lane * PRIV_PAD + D.P_PUSH_F + 1] = clampf(push_f[1], -clip, clip);
#pragma unroll
                for (int k = 0; k < 3; ++k) sp[lane * PRIV_PAD + D.P_PUSH_T + k] = clampf(push_t[k], -clip, clip);
            }
        }
    };
    auto joints = [&](auto h0, auto h1) {
        // ================================ joints ================================
        if (bulk) hb::mbar_wait(&bar, 0);
        HB_STAMP(1);
        // Only q, qd and the actions stay live across the barrier; the previous-step buffers are consumed
        // (and, on a step, rolled forward: legged_robot.py:146-148) joint by joint before it.
        // The reference trajectory (compute_ref_state, hector_env.py:90-111 / humanoid_env.py:120-142) is STATE: it is
        // refreshed inside compute_observations, so the joint_pos reward of a step sees the one the previous step left.
        const bool joint_pos_on = T::OPT && p.reward_scale[HB_R_JOINT_POS] != 0.0f;
        const bool use_ref = T::OPT && (KIND == KIND_XBOT || joint_pos_on) && b.ref_dof_pos != nullptr;
        long long ep_len = 0;
        if (use_ref && valid) ep_len = b.episode_length_buf[env] + (do_prepare ? 1 : 0);
        float q[CAP], qd[CAP], act[CAP];
#pragma unroll
        for (int j = 0; j < CAP; ++j) {
            if (T::RUNTIME && j == NDOF) break;
            q[j] = sm[L.dof + ln * NDOF * 2 + 2 * j];
            qd[j] = sm[L.dof + ln * NDOF * 2 + 2 * j + 1];
            act[j] = sm[L.actions + ln * NDOF + j];
        }
        if (do_rew || do_last) {
            float t1 = 0.f, t2 = 0.f, t3 = 0.f, ss = 0.f, acc = 0.f, vel = 0.f, tq = 0.f, rr = 0.f;
            float dy0 = 0.f, dy1 = 0.f, dy2 = 0.f, dy3 = 0.f, da0 = 0.f, da1 = 0.f, da2 = 0.f, da3 = 0.f;
            const int yl = D.YAW_L, yr_ = D.YAW_R, al = D.ARM_L, ar_ = D.ARM_R;      // (checked against p by the launcher)
#pragma unroll
            for (int j = 0; j < CAP; ++j) {
                if (T::RUNTIME && j == NDOF) break;
                const float lact = sm[L.last_actions + ln * NDOF + j];
                const float llact = sm[L.last_last_actions + ln * NDOF + j];
                const float ldv = sm[L.last_dof_vel + ln * NDOF + j];
                if (h0) {
                    const float d1 = lact - act[j];                    // action_smoothness, hector_env.py:529-539
                    t1 += d1 * d1;
                    const float d2 = (act[j] + llact) - 2.0f * lact;
                    t2 += d2 * d2;
                    t3 += fabsf(act[j]);
                    const float d = q[j] - p.default_dof_pos[j];       // default_joint_pos, :357-367
                    ss += d * d;
                    // hip yaw / roll of both legs (and, hector_full, the first two arm joints of both arms:
                    // hector_w_arm_env.py:371-378); the index pairs are task constants
                    // (j is a compile-time value in the unrolled loop: these are plain register copies)
                    dy0 = (j == yl) ? d : dy0, dy1 = (j == yl + 1) ? d : dy1;
                    dy2 = (j == yr_) ? d : dy2, dy3 = (j == yr_ + 1) ? d : dy3;
                    if (D.HAS_ARMS) {
                        da0 = (j == al) ? d : da0, da1 = (j == al + 1) ? d : da1;
                        da2 = (j == ar_) ? d : da2, da3 = (j == ar_ + 1) ? d : da3;
                    }
                    if (joint_pos_on && use_ref && do_rew) {           // joint_pos, hector_env.py:264-275
                        const float e = q[j] - (valid ? b.ref_dof_pos[(size_t)env * NDOF + j] : 0.0f);
                        rr += e * e;
                    }
                }
                if (h1) {
                    const float a = (ldv - qd[j]) / dt;                // dof_acc :515-520
                    acc += a * a;
                    vel += qd[j] * qd[j];                              // dof_vel :508-513
                    const float tau = sm[L.torques + ln * NDOF + j];   // torques :501-506
                    tq += tau * tau;
                    if (valid && do_last) {                            // legged_robot.py:146-148 (reset envs: zeroed below)
                        b.last_last_actions[(size_t)env * NDOF + j] = lact;
                        b.last_actions[(size_t)env * NDOF + j] = act[j];
                        b.last_dof_vel[(size_t)env * NDOF + j] = qd[j];
                    }
                }
            }
            if (do_rew && h0) {
                terms[HB_R_ACTION_SMOOTHNESS * TILE + lane] = (t1 + t2) + 0.05f * t3;
                float yr = sqrtf(dy0 * dy0 + dy1 * dy1) + sqrtf(dy2 * dy2 + dy3 * dy3);
                yr = clampf(yr - 0.1f, 0.0f, 50.0f);
                float djp = expf(-yr * 100.0f);
                if (D.HAS_ARMS) {
                    float ar = sqrtf(da0 * da0 + da1 * da1) + sqrtf(da2 * da2 + da3 * da3);
                    ar = clampf(ar - 0.1f, 0.0f, 25.0f);
                    djp = djp + expf(-ar * 2.0f);
                }
                terms[HB_R_DEFAULT_JOINT_POS * TILE + lane] = djp - 0.01f * sqrtf(ss);
                if (joint_pos_on) {
                    const float nrm = sqrtf(rr);
                    terms[HB_R_JOINT_POS * TILE + lane] = expf(-2.0f * nrm) - 0.2f * clampf(nrm, 0.0f, 0.5f);
                }
            }
            if (do_rew && h1) {
                terms[HB_R_DOF_ACC * TILE + lane] = acc;
                terms[HB_R_DOF_VEL * TILE + lane] = vel;
                terms[HB_R_TORQUES * TILE + lane] = tq;
            }
        }
        HB_STAMP(2);
        tile_barrier<true>();                                     // ---- barrier 1 ----
        HB_STAMP(3);
        const bool reset = valid && (flags[lane] & 1);
        if (reset) {         // _reset_dofs (legged_robot.py:358-372) + buffer zeroing (:186-191)
            float u[CAP];
            if (nz.u_reset) {
#pragma unroll
                for (int j = 0; j < CAP; ++j) {
                    if (T::RUNTIME && j == NDOF) break;
                    u[j] = nz.u_reset[(size_t)env * U_RESET + j];
                }
            } else {
                rng_uniforms(rng, env, SLOT_U_RESET, 0, NDOF, u);
            }
#pragma unroll
            for (int j = 0; j < CAP; ++j) {
                if (T::RUNTIME && j == NDOF) break;
                q[j] = p.default_dof_pos[j] + (p.reset_dof_span * u[j] + p.reset_dof_lo);
                qd[j] = 0.0f;
                act[j] = 0.0f;
                if (h0) {
                    b.dof_state[((size_t)env * NDOF + j) * 2] = q[j];
                    b.dof_state[((size_t)env * NDOF + j) * 2 + 1] = 0.0f;
                    b.actions[(size_t)env * NDOF + j] = 0.0f;
                    b.last_actions[(size_t)env * NDOF + j] = 0.0f;
                    b.last_last_actions[(size_t)env * NDOF + j] = 0.0f;
                    b.last_dof_vel[(size_t)env * NDOF + j] = 0.0f;
                }
            }
        }
        if (emit_obs) {
            float sl = 0.0f, sr = 0.0f;
            if (h0 && use_ref) {       // compute_ref_state of this compute_observations call
                if (reset) ep_len = 0;
                const float sn = sinf(TWO_PI_F * (((float)ep_len * dt) / p.cycle_time));
                sl = fminf(sn, 0.0f), sr = fmaxf(sn, 0.0f);
                if (fabsf(sn) < 0.1f) sl = sr = 0.0f;               // double support
            }
#pragma unroll
            for (int j = 0; j < CAP; ++j) {
                if (T::RUNTIME && j == NDOF) break;
                if (h0 && use_ref) {
                    float ref = 0.0f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const float sc = (k == 1) ? p.ref_scale[1] : p.ref_scale[0];
                        if (j == p.ref_left[k]) ref = sl * sc;
                        if (j == p.ref_right[k]) ref = sr * sc;
                    }
                    if (valid) b.ref_dof_pos[(size_t)env * NDOF + j] = ref;
                    if (KIND == KIND_XBOT) sp[lane * PRIV_PAD + D.P_DIFF + j] = clampf(q[j] - ref, -clip, clip);
                }
                float v0 = (q[j] - p.default_dof_pos[j]) * p.obs_dof_pos, v1 = qd[j] * p.obs_dof_vel;
                if (h0) {
                    sp[lane * PRIV_PAD + 5 + j] = clampf(v0, -clip, clip);
                    sp[lane * PRIV_PAD + 5 + NDOF + j] = clampf(v1, -clip, clip);
                    sp[lane * PRIV_PAD + 5 + 2 * NDOF + j] = clampf(act[j], -clip, clip);
                }
                if (h1) {
                    so[lane * OBS + 5 + j] = noisy_clip(v0, 5 + j);
                    so[lane * OBS + 5 + NDOF + j] = noisy_clip(v1, 5 + NDOF + j);
                    so[lane * OBS + 5 + 2 * NDOF + j] = noisy_clip(act[j], 5 + 2 * NDOF + j);
                }
            }
        }
    };
    auto feet = [&](auto h0, auto h1) {
        // ================================ feet / contacts / gait ================================
        long long ep_len = 0;
        float foot_pos[2][3], foot_vel[2][3], knee_xy[2][2], air[2], fh[2], lz[2];
        bool last_ct[2];
        float friction, mass;
        {
            const int ev = valid ? env : env0;         // invalid lanes of a ragged tile mirror the tile's first env
            ep_len = b.episode_length_buf[ev];
            friction = b.env_frictions[ev], mass = b.body_mass[ev];
            const float *rs = b.rigid_state + (size_t)ev * p.num_bodies * 13;
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                const float *r = rs + p.feet[f] * 13;
#pragma unroll
                for (int k = 0; k < 3; ++k) foot_pos[f][k] = __ldg(r + k), foot_vel[f][k] = __ldg(r + 7 + k);
                const float *kr = rs + p.knees[f] * 13;
                knee_xy[f][0] = __ldg(kr), knee_xy[f][1] = __ldg(kr + 1);
                air[f] = b.feet_air_time[ev * 2 + f];
                fh[f] = b.feet_height[ev * 2 + f];
                lz[f] = b.last_feet_z[ev * 2 + f];
                last_ct[f] = b.last_contacts[ev * 2 + f] != 0;
            }
        }
        if (bulk) hb::mbar_wait(&bar, 0);
        HB_STAMP(1);
        const float *cf = sm + L.contact + ln * crow;
        float foot_f[2][3];
#pragma unroll
        for (int f = 0; f < 2; ++f)
#pragma unroll
            for (int k = 0; k < 3; ++k) foot_f[f][k] = cf[p.feet[f] * 3 + k];
        const float root_z = sm[L.root + ln * 13 + 2];
        bool term = false, time_out = false;
        float gs = 0.0f, gc = 1.0f, st[2] = {1.0f, 1.0f};
        const bool ct[2] = {foot_f[0][2] > 5.0f, foot_f[1][2] > 5.0f};
        if (do_prepare) ep_len += 1;
        if (h0 && do_term) {   // -------- check_termination, legged_robot.py:155-160 --------
#pragma unroll 1
            for (int i = 0; i < p.n_term; ++i) term |= norm3(cf + p.term_bodies[i] * 3) > 1.0f;
            time_out = ep_len > (long long)p.max_episode_length;
            term |= time_out;
        }
        if (h1 && do_rew) {    // collision, hector_env.py:522-527
            float coll = 0.f;
#pragma unroll 1
            for (int i = 0; i < p.n_pen; ++i) coll += (norm3(cf + p.pen_bodies[i] * 3) > 0.1f) ? 1.0f : 0.0f;
            terms[HB_R_COLLISION * TILE + lane] = coll;
        }
        bool reset = do_step && term;        // the fused step resets what it has just found terminated
        {   // -------- gait phase, hector_env.py:70-88 --------
            const float arg = TWO_PI_F * (((float)ep_len * dt) / p.cycle_time);
            sincosf(arg, &gs, &gc);
            st[0] = (gs >= 0.0f) ? 1.0f : 0.0f, st[1] = (gs < 0.0f) ? 1.0f : 0.0f;
            if (fabsf(gs) < 0.1f) st[0] = st[1] = 1.0f;
        }
        if (do_rew) {
            if (h1) {   // base_height, :369-383
                const float ground = (foot_pos[0][2] * st[0] + foot_pos[1][2] * st[1]) / (st[0] + st[1]);
                const float h = root_z - (ground - 0.05f);
                terms[HB_R_BASE_HEIGHT * TILE + lane] = expf(-fabsf(h - p.base_height_target) * 100.0f);
            }
            float r_air = 0.f, r_clr = 0.f, cfz = 0.f, num = 0.f, slip = 0.f;
#pragma unroll
            for (int f = 0; f < 2; ++f) {
                if (h0) {   // feet_air_time, :315-329 (stateful)
                    const bool filt = ct[f] || (st[f] != 0.0f) || last_ct[f];
                    last_ct[f] = ct[f];
                    const bool first = (air[f] > 0.0f) && filt;
                    air[f] += dt;
                    r_air += clampf(air[f], 0.0f, 0.5f) * (first ? 1.0f : 0.0f);
                    air[f] *= filt ? 0.0f : 1.0f;
                }
                if (h1) {   // feet_clearance, :445-466 (stateful)
                    const float z = foot_pos[f][2] - 0.05f;
                    fh[f] += z - lz[f];
                    lz[f] = z;
                    const float hit = (fabsf(fh[f] - p.target_feet_height) < 0.01f) ? 1.0f : 0.0f;
                    r_clr += hit * (1.0f - st[f]);
                    fh[f] *= ct[f] ? 0.0f : 1.0f;
                }
                if (h0) {   // feet_contact_forces :350-355, feet_contact_number :331-339, foot_slip :303-313
                    cfz += clampf(norm3(foot_f[f]) - p.max_contact_force, 0.0f, 400.0f);
                    num += (ct[f] == (st[f] != 0.0f)) ? 1.0f : -0.3f;
                    const float spd = sqrtf(sqrtf(foot_vel[f][0] * foot_vel[f][0] + foot_vel[f][1] * foot_vel[f][1]));
                    slip += spd * (ct[f] ? 1.0f : 0.0f);
                }
            }
            if (h0) terms[HB_R_FEET_AIR_TIME * TILE + lane] = r_air;
            if (h1) terms[HB_R_FEET_CLEARANCE * TILE + lane] = r_clr;
            if (h0) {
                terms[HB_R_FEET_CONTACT_FORCES * TILE + lane] = cfz;
                terms[HB_R_FEET_CONTACT_NUMBER * TILE + lane] = num / 2.0f;
                terms[HB_R_FOOT_SLIP * TILE + lane] = slip;
            }
            if (h1) {   // feet_distance :277-287, knee_distance :290-300
                float dx = foot_pos[0][0] - foot_pos[1][0], dy = foot_pos[0][1] - foot_pos[1][1];
                float d = sqrtf(dx * dx + dy * dy);
                float dmin = clampf(d - p.min_dist, -0.5f, 0.0f), dmax = clampf(d - p.max_dist, 0.0f, 0.5f);
                terms[HB_R_FEET_DISTANCE * TILE + lane] = (expf(-fabsf(dmin) * 100.0f) + expf(-fabsf(dmax) * 100.0f)) / 2.0f;
                dx = knee_xy[0][0] - knee_xy[1][0], dy = knee_xy[0][1] - knee_xy[1][1];
                d = sqrtf(dx * dx + dy * dy);
                dmin = clampf(d - p.min_dist, -0.5f, 0.0f), dmax = clampf(d - p.max_dist / 2.0f, 0.0f, 0.5f);
                terms[HB_R_KNEE_DISTANCE * TILE + lane] = (expf(-fabsf(dmin) * 100.0f) + expf(-fabsf(dmax) * 100.0f)) / 2.0f;
            }
        }
        if (h0) {
            if (stages & HB_STAGE_RESET_ALL) reset = true;
            if ((stages & HB_STAGE_RESET_MASK) && valid) reset = reset || (b.reset_buf[env] != 0);   // reset_idx(env_ids)
            reset = reset && valid;
            flags[lane] = (reset ? 1 : 0) | (time_out ? 2 : 0);
            sm[L.gait_s + lane] = gs, sm[L.gait_c + lane] = gc;
        }
        HB_STAMP(2);
        tile_barrier<true>();                                     // ---- barrier 1 ----
        HB_STAMP(3);
        if (!h0) reset = (flags[lane] & 1) != 0;                 // (the first half's flag)
        if (reset) {
            ep_len = 0, air[0] = air[1] = 0.0f;
            st[0] = st[1] = 1.0f;                                   // phase 0: sin = 0 -> double support
        }
        if (valid) {
            if (h0) {
                b.feet_air_time[env * 2] = air[0], b.feet_air_time[env * 2 + 1] = air[1];
                b.episode_length_buf[env] = ep_len;
                if (any_reset) b.reset_buf[env] = reset ? 1 : 0;
                else if (do_term) b.reset_buf[env] = term ? 1 : 0;           // check_termination on its own: the mask only
                if (do_term) b.time_out_buf[env] = time_out ? 1 : 0;
            }
            if (do_rew) {
#pragma unroll
                for (int f = 0; f < 2; ++f) {
                    if (h0) b.last_contacts[env * 2 + f] = last_ct[f] ? 1 : 0;
                    if (h1) b.feet_height[env * 2 + f] = fh[f], b.last_feet_z[env * 2 + f] = lz[f];
                }
            }
        }
        if (h1 && emit_obs) {
            if (KIND == KIND_HECTOR) {
#pragma unroll
                for (int f = 0; f < 2; ++f)
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        sp[lane * PRIV_PAD + D.P_FEET_POS + f * 3 + k] = clampf(foot_pos[f][k], -clip, clip);
                        sp[lane * PRIV_PAD + D.P_FEET_VEL + f * 3 + k] = clampf(foot_vel[f][k], -clip, clip);
                    }
            }
            sp[lane * PRIV_PAD + D.P_FRICTION] = clampf(friction, -clip, clip);
            sp[lane * PRIV_PAD + D.P_MASS] = clampf(mass / 30.0f, -clip, clip);
            sp[lane * PRIV_PAD + D.P_STANCE] = st[0], sp[lane * PRIV_PAD + D.P_STANCE + 1] = st[1];
            sp[lane * PRIV_PAD + D.P_CONTACT] = ct[0] ? 1.0f : 0.0f, sp[lane * PRIV_PAD + D.P_CONTACT + 1] = ct[1] ? 1.0f : 0.0f;
        }
    };
    auto ledger = [&](auto h0, auto h1) {
        // ================================ ledger ================================
        // (terms with scale 0 are not part of the task: the reference has no episode sum for them - their rows stay zero
        // and are neither read nor written)
        float sums[HB_NUM_REWARDS];
#pragma unroll
        for (int k = 0; k < HB_NUM_REWARDS; ++k)
            sums[k] = (valid && p.reward_scale[k] != 0.0f) ? b.episode_sums[(size_t)k * N + env] : 0.0f;
        if (with_noise && !tape_noise && emit_obs) {
            // the tile's observation noise, drawn by this otherwise idle warp while the other roles are in phase A:
            // 11 Philox calls of 4 normals per env; calls whose four columns all have zero noise scale are skipped
            const int CALLS = (OBS + 3) / 4;
            float *z = sm + L.z_obs;
            for (int c = h0 ? lane : lane + 32; c < nv * CALLS; c += 64) {      // (the pair interleaves)
                const int e = c / CALLS, q = c - e * CALLS;
                bool any = false;
#pragma unroll
                for (int k = 0; k < 4; ++k) any = any || (q * 4 + k < OBS && p.noise_scale_vec[q * 4 + k] != 0.0f);
                float z4[4] = {0.f, 0.f, 0.f, 0.f};
                if (any) rng_normal4(rng, env0 + e, SLOT_Z_OBS + q, z4);
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (q * 4 + k < OBS) z[e * OBS + q * 4 + k] = z4[k];
            }
        }
        HB_STAMP(2);
        tile_barrier<true>();                                     // ---- barrier 1 ----
        HB_STAMP(3);
        const bool reset = valid && (flags[lane] & 1);
        float *rsums = sm + L.rsums;                           // the reset envs' sums (the first half still reads terms)
        if (do_rew) {        // compute_reward, legged_robot.py:216-234: alphabetical accumulation
            float rew = 0.0f;
#pragma unroll
            for (int k = 0; k < HB_NUM_REWARDS; ++k) {
                if (p.reward_scale[k] != 0.0f) {
                    const float r = terms[k * TILE + lane] * p.reward_scale[k];
                    rew += r;
                    sums[k] += r;
                }
            }
            if (h0) {
                if (p.only_positive_rewards) rew = fmaxf(rew, 0.0f);
                if (valid) b.rew_buf[env] = rew;
            }
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, reset);
        __syncwarp();
#pragma unroll
        for (int k = 0; k < HB_NUM_REWARDS; ++k) {
            if (h1 && p.reward_scale[k] != 0.0f) {
                rsums[k * TILE + lane] = reset ? sums[k] : 0.0f;    // episode sums of the envs being reset (:198-201)
                if (reset) sums[k] = 0.0f;
                if (valid) b.episode_sums[(size_t)k * N + env] = sums[k];
            }
        }
        __syncwarp();
        // ---------------- reset ids + episode means ----------------
        // Each tile publishes its ballot; reset_finalize_kernel turns the ballots into the ascending id
        // list (like reset_buf.nonzero()) and the count.  The per-term sums of the reset envs
        // (legged_robot.py:198-201) go straight into 18 fp64 accumulators: fp64 addition of these
        // fp32 values is order-independent far below fp32 resolution.
        if (h1 && ballot && lane < HB_NUM_REWARDS && p.reward_scale[lane] != 0.0f) {
            float v = 0.0f;
#pragma unroll 8
            for (int e = 0; e < TILE; ++e) v += rsums[lane * TILE + ((e + lane) & 31)];
            atomicAdd(b.scratch_sums + lane, (double)v);
        }
        if (h0 && lane == 0) b.scratch_ballots[blockIdx.x] = ballot;     // consumed by reset_finalize_kernel
    };
    if (role == 0) run(base);
    else if (role == 1) run(joints);
    else if (role == 2) run(feet);
    else run(ledger);

    // ---------------- coalesced store of the newest frames into the last slot of the stacked buffers ----------------
    // by the three roles that wrote them (named barrier 2, 96 threads; wide: their six warps, 192 threads); the ledger is
    // busy with its ticket
    HB_STAMP(4);
    constexpr int NT = 6 * TILE;
    if (warp < NT / 32) {
        asm volatile("bar.sync 2, 192;" ::: "memory");            // ---- barrier 2 ----
        HB_STAMP(5);
        if (emit_obs) {
            // NT threads walk the tile's frames with (row, column) advanced incrementally: no per-element division.
            // Privileged frames leave as 8-byte pairs (row starts are 8-byte aligned: 4200 r + 3920 bytes).
            const int P2 = PRIV / 2;
            const int orow = p.frame_stack * OBS, prow = p.c_frame_stack * PRIV;
            const int ostride = p.obs_ld ? p.obs_ld : orow, pstride = p.priv_ld ? p.priv_ld : prow;   // row pitch
            const int t = threadIdx.x;
            if ((PRIV & 1) == 0 && ((pstride | prow) & 1) == 0 && (reinterpret_cast<uintptr_t>(priv_new) & 7u) == 0) {
                int r = t / P2, c2 = t - r * P2;
                float2 *dst = reinterpret_cast<float2 *>(priv_new + (size_t)env0 * pstride + (prow - PRIV));
                const float2 *src = reinterpret_cast<const float2 *>(sp);
                const int half = pstride / 2;
                while (r < nv) {
                    dst[(size_t)r * half + c2] = src[r * P2 + c2];
                    r += NT / P2, c2 += NT % P2;
                    if (c2 >= P2) c2 -= P2, r += 1;
                }
            } else {
                int r = t / PRIV, c = t - r * PRIV;
                while (r < nv) {
                    priv_new[(size_t)(env0 + r) * pstride + (prow - PRIV) + c] = sp[r * PRIV + c];
                    r += NT / PRIV, c += NT % PRIV;
                    if (c >= PRIV) c -= PRIV, r += 1;
                }
            }
            int r = t / OBS, c = t - r * OBS;
            float *dst = obs_new + (size_t)env0 * ostride + (orow - OBS);
            while (r < nv) {
                dst[(size_t)r * ostride + c] = so[r * OBS + c];
                r += NT / OBS, c += NT % OBS;
                if (c >= OBS) c -= OBS, r += 1;
            }
        }
    }
    HB_STAMP(6);
    HB_GT(1);
}

// ------------------------------------------------------------------------------------------
// a8 (stacking): new[:, 0:(S-1)*F] = prev[:, F:S*F]  — a flat copy shifted by one frame with a
// hole of F floats per row (the newest frame, written by post_physics_kernel).  With kZero the
// carried frames of the envs post-physics just reset are written as zeros (reset_idx,
// hector_env.py:256-261); without it that is left to reset_finalize_kernel.
// Destination vectors are 16-byte aligned; the source is 4*F bytes further on, which is only
// 4-byte aligned for F = 41, so each thread loads the aligned vector below its source window
// and takes the missing floats from its neighbour lane (shuffle); F % 4 picks the rotation.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld_vec_guarded(const float *__restrict__ prev, uint32_t s, uint32_t total) {
    const uint32_t e = s * 4u;                         // ragged last vector of the buffer (N*row % 4 != 0)
    float4 v;
    v.x = (e < total) ? __ldg(prev + e) : 0.0f;
    v.y = (e + 1 < total) ? __ldg(prev + e + 1) : 0.0f;
    v.z = (e + 2 < total) ? __ldg(prev + e + 2) : 0.0f;
    v.w = (e + 3 < total) ? __ldg(prev + e + 3) : 0.0f;
    return v;
}

// The shape of one history's stack: rows of `row` floats, the last `frame` of them the newest frame, at a pitch of `ld`
// floats.  A built robot's shape is all constants (FixedShift): the row split of a vector index is then a multiply-shift
// and the rotation is resolved at compile time.
template <int ROW, int LD, int FRAME>
struct FixedShift {
    static constexpr bool kFixed = true;
    static constexpr uint32_t row = ROW, ld = LD, frame = FRAME;
    __device__ __forceinline__ static uint32_t div(uint32_t e) { return e / (uint32_t)LD; }
};

// Any other shape: any robot's frames, any stack depth.  inv_ld = ceil(2^64 / ld): for e < 2^32, e / ld =
// umul64hi(e, inv_ld) exactly (the error term e (inv_ld ld - 2^64) / 2^64 stays below 1), two wide multiplies instead of
// a division per vector.
struct ShiftShape {
    static constexpr bool kFixed = false;
    uint32_t row, ld, frame;
    unsigned long long inv_ld;
    __device__ __forceinline__ uint32_t div(uint32_t e) const { return (uint32_t)__umul64hi(e, inv_ld); }
};

// Block `blk` of the shift of one history (`total` floats): 256 threads, UNROLL vectors each.  kZero: the carried frames
// of the envs flagged in reset_buf are written as zeros.  A compiled shape shuffles only the floats its rotation needs,
// and kZero alone decides the zeroing.  The runtime shape shuffles all three floats, with no branch on the rotation, and
// serves the plain shift too in the same kernel, so there a null reset_buf means no zeroing.
template <typename Shape, int UNROLL, bool kZero>
__device__ __forceinline__ void stack_shift(const float *__restrict__ prev, float *__restrict__ next, const uint32_t total,
                                            const uint32_t blk, const Shape sh, const uint8_t *__restrict__ reset_buf) {
    const uint32_t LD = sh.ld, KEEP = sh.row - sh.frame;     // floats of a row that are carried over
    const uint32_t ROT = sh.frame & 3u;                      // source misalignment in floats
    const uint32_t FVEC = sh.frame >> 2;                     // whole vectors of shift
    const bool vec_rows = (LD & 3u) == 0;                    // the buffer is whole vectors: predicated loads
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t total_vec = total >> 2;              // whole vectors
    const uint32_t tail_vec = (total + 3u) >> 2;
    const uint32_t warp_base = (blk * blockDim.x + (threadIdx.x - lane)) * UNROLL;
    const float4 *p4 = reinterpret_cast<const float4 *>(prev);
    float4 *n4 = reinterpret_cast<float4 *>(next);
    float4 v[UNROLL], w[UNROLL];
    uint8_t rz[UNROLL];
    // all loads first (UNROLL independent 16-byte requests in flight per thread, plus the row's reset flag)
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const uint32_t s = warp_base + u * 32u + lane + FVEC;          // aligned source vector below the window
        const uint32_t e = (warp_base + u * 32u + lane) * 4u;
        const uint32_t r = sh.div(e);
        rz[u] = (kZero && (Shape::kFixed || reset_buf) && e < total) ? __ldg(reset_buf + r) : 0;
        if (!Shape::kFixed) w[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        // vector-aligned rows: a destination vector that lies, like the one before it, wholly in the newest-frame
        // hole or the padding needs no source (neither for itself nor for its left neighbour's spill-over)
        if (vec_rows) {
            const bool need = e - r * LD < KEEP + 4u;
            v[u] = hb::ld_stream4_if(p4 + s, need && s < total_vec);
            if (ROT != 0) w[u] = hb::ld_stream4_if(p4 + s + 1u, need && lane == 31u && s + 1u < total_vec);
        } else {
            v[u] = (s < total_vec) ? hb::ld_stream4(p4 + s) : ld_vec_guarded(prev, s, total);
            if (ROT != 0 && lane == 31u)                                // no neighbour lane: fetch the spill-over
                w[u] = (s + 1u < total_vec) ? hb::ld_stream4(p4 + s + 1u) : ld_vec_guarded(prev, s + 1u, total);
        }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        const uint32_t i = warp_base + u * 32u + lane;                  // destination vector index
        float4 o = v[u];
        if (ROT != 0 || !Shape::kFixed) {
            float nx0 = __shfl_down_sync(0xffffffffu, v[u].x, 1);       // first floats of vector s+1
            float nx1 = ROT > 1 || !Shape::kFixed ? __shfl_down_sync(0xffffffffu, v[u].y, 1) : 0.0f;
            float nx2 = ROT > 2 || !Shape::kFixed ? __shfl_down_sync(0xffffffffu, v[u].z, 1) : 0.0f;
            if (lane == 31u) nx0 = w[u].x, nx1 = w[u].y, nx2 = w[u].z;
            if (ROT == 1) o = make_float4(v[u].y, v[u].z, v[u].w, nx0);
            else if (ROT == 2) o = make_float4(v[u].z, v[u].w, nx0, nx1);
            else if (ROT == 3) o = make_float4(v[u].w, nx0, nx1, nx2);
        }
        if (i >= tail_vec) continue;
        const uint32_t e0 = i * 4u;                      // first destination float
        const uint32_t r0 = sh.div(e0);
        const uint32_t c0 = e0 - r0 * LD;
        if (vec_rows && c0 >= KEEP) continue;            // vector-aligned rows: newest-frame hole / padding
        if (c0 + 3u < KEEP && i < total_vec) {           // whole vector inside the carried part of one row
            if (rz[u]) o = make_float4(0.f, 0.f, 0.f, 0.f);
            hb::st_stream4(n4 + i, o);
        } else {                                         // touches the newest-frame hole or a row boundary
            const float ov[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
            for (uint32_t k = 0; k < 4u; ++k) {
                uint32_t c = c0 + k, r = r0;
                if (c >= LD) c -= LD, r += 1u;
                if (c < KEEP && e0 + k < total) {               // (past the buffer's end r is num_envs: no flag to read)
                    const bool zero = kZero && (Shape::kFixed || reset_buf) &&
                                      (vec_rows ? rz[u] != 0 : reset_buf[r] != 0);   // (a vector of a pitched row stays in its row)
                    next[e0 + k] = zero ? 0.0f : ov[k];
                }
            }
        }
    }
}

// generic shapes / unaligned buffers / optional per-env zeroing (reset_buf may be null)
__global__ void __launch_bounds__(256)
stack_shift_scalar_kernel(const float *__restrict__ prev, float *__restrict__ next,
                          const uint8_t *__restrict__ reset_buf, long long total, int row, int ld, int frame) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int r = (int)(i / ld), c = (int)(i - (long long)r * ld);
    if (c < row - frame) next[i] = (reset_buf && reset_buf[r]) ? 0.0f : prev[i + frame];
}

// What reset_idx needs from the whole shard, after post_physics_kernel published one ballot per 32-env
// tile and the shift wrote the carried frames:
//   * env_ids = reset_buf.nonzero() (legged_robot.py:142): ascending ids + count (device and pinned host copy);
//   * extras["episode"] means (:198-201) from the fp64 accumulators, only refreshed when >= 1 env was reset
//     (quirk 4; otherwise the previous step's values are carried into this step's slot);
//   * extras["time_outs"] (:208-209), also only then;
//   * obs_history / critic_history zeroing of the reset envs (hector_env.py:256-261).
// Every CTA owns a contiguous segment of tiles; it sums the popcounts before its segment (8 KB of ballots at
// 65536 envs: cheaper to recount per CTA than to chain CTAs), scans its own, writes its ids in order and zeroes
// the carried frames of its reset envs, one warp per (env, buffer).
constexpr int FIN_THREADS = 256;

__device__ __forceinline__ int block_sum(int v, int *scratch) {        // all threads get the total
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int w = 0; w < FIN_THREADS / 32; ++w) t += scratch[w];
    return t;
}

__device__ __forceinline__ void
reset_finalize_body(const hb_env_params &p, const hb_env_buffers &b, float *__restrict__ obs_new, float *__restrict__ priv_new,
                    int tiles, int seg, int32_t *host_count, unsigned long long *rng_counter, const int blk, const int nblk) {
    __shared__ int scratch[FIN_THREADS / 32];
    __shared__ int wbase[FIN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t_lo = blk * seg, t_hi = min(t_lo + seg, tiles);
    int before = 0, rest = 0;
#pragma unroll 4
    for (int t = threadIdx.x; t < tiles; t += FIN_THREADS) {
        const int c = (t < t_lo || t >= t_hi) ? __popc(__ldg(b.scratch_ballots + t)) : 0;
        before += (t < t_lo) ? c : 0;
        rest += (t >= t_hi) ? c : 0;
    }
    const int prefix = block_sum(before, scratch);
    const int after = block_sum(rest, scratch);
    // this CTA's tiles: consecutive threads own consecutive tiles (segments longer than the CTA go in rounds)
    int seg_count = 0;
    for (int t0 = t_lo; t0 < t_hi; t0 += FIN_THREADS) {
        const int t = t0 + threadIdx.x;
        unsigned m = (t < t_hi) ? __ldg(b.scratch_ballots + t) : 0u;
        const int cnt = __popc(m);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        __syncthreads();
        if (lane == 31) wbase[warp] = incl;
        __syncthreads();
        int off = prefix + seg_count + incl - cnt, round_total = 0;
#pragma unroll
        for (int w = 0; w < FIN_THREADS / 32; ++w) {
            off += (w < warp) ? wbase[w] : 0;
            round_total += wbase[w];
        }
        while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            b.reset_env_ids[off++] = t * TILE + bit;
        }
        seg_count += round_total;
    }
    const int total = prefix + seg_count + after;
    if (blk == 0) {
        float *means = b.episode_means;
        const float *means_prev = b.episode_means_prev;
        int cursor = 0, ring = 0;
        if (b.episode_ring) {                        // this step's slot of the extras ring, the previous step's behind it
            cursor = b.episode_ring[0], ring = b.episode_ring[1];
            means = b.episode_means + (size_t)cursor * HB_NUM_REWARDS;
            means_prev = b.episode_means + (size_t)((cursor + ring - 1) % ring) * HB_NUM_REWARDS;
        }
        __syncthreads();                             // every thread has read the cursor before thread 0 advances it
        if (threadIdx.x == 0) {
            *b.reset_count = total;
            if (host_count) *host_count = total;
            if (rng_counter) *rng_counter += 1ull;       // the next call draws from a fresh counter
            if (b.episode_ring) b.episode_ring[0] = (cursor + 1) % ring;
        }
        if (threadIdx.x < HB_NUM_REWARDS) {
            const int k = threadIdx.x;
            if (total > 0) {
                means[k] = (float)(b.scratch_sums[k] / (double)total) / p.max_episode_length_s;
                b.scratch_sums[k] = 0.0;             // re-armed for the next step
            } else if (means_prev && means_prev != means) {
                means[k] = means_prev[k];
            }
        }
    }
    if (total == 0) return;
    if (b.time_outs_latched) {
        for (int i = blk * FIN_THREADS + threadIdx.x; i < p.num_envs; i += nblk * FIN_THREADS)
            b.time_outs_latched[i] = b.time_out_buf[i];
    }
    if (!obs_new || seg_count == 0) return;
    __syncthreads();                                 // this CTA's ids are visible to all of its warps
    const int row_a = p.frame_stack * p.num_single_obs, row_b = p.c_frame_stack * p.num_single_priv;
    const int keep_a = row_a - p.num_single_obs, keep_b = row_b - p.num_single_priv;
    for (int j = warp; j < 2 * seg_count; j += FIN_THREADS / 32) {
        const int env = b.reset_env_ids[prefix + (j >> 1)];
        float *dst = (j & 1) ? priv_new + (size_t)env * (p.priv_ld ? p.priv_ld : row_b)
                             : obs_new + (size_t)env * (p.obs_ld ? p.obs_ld : row_a);
        const int keep = (j & 1) ? keep_b : keep_a;
        for (int c = lane; c < keep; c += 32) dst[c] = 0.0f;
    }
}

__global__ void __launch_bounds__(FIN_THREADS)
reset_finalize_kernel(const __grid_constant__ hb_env_params p, const __grid_constant__ hb_env_buffers b,
                      float *__restrict__ obs_new, float *__restrict__ priv_new, int tiles, int seg,
                      int32_t *host_count, unsigned long long *rng_counter) {
    hb::pdl_trigger();
    hb::pdl_wait();              // post-physics (ballots, sums) and the shift are complete
    reset_finalize_body(p, b, obs_new, priv_new, tiles, seg, host_count, rng_counter, blockIdx.x, gridDim.x);
}

// Arguments of the reset finalisation for a frame-stack launch that runs it (reset_finalize_body without the zeroing),
// or none (NoFinalize: the plain shift)
struct FinalizeArgs {
    static constexpr bool kOn = true;
    hb_env_params p;
    hb_env_buffers b;
    int tiles, seg;
    int32_t *host_count;
    unsigned long long *rng_counter;
};
struct NoFinalize { static constexpr bool kOn = false; };

// The frame-stack shift of both histories: blocks [0, blocks_a) shift history a, the next blocks_b history b.  With
// FinalizeArgs, the step's last launch: the carried frames of the envs post-physics just reset are zeroed (reset flags
// fin.b.reset_buf, hector_env.py:256-261) and the shard-wide half of reset_idx (ids, count, episode means, time-out latch)
// runs in a few extra blocks of the same grid - one launch less on the step's dependency chain than shift +
// reset_finalize_kernel.  Blocks per SM with finalisation: 6 for a compiled shape (40 registers), 4 for the runtime shape
// (56 registers).
template <typename SA, typename SB, typename Fin>
__global__ void __launch_bounds__(256, !Fin::kOn ? 0 : (SA::kFixed ? 6 : 4))
stack_shift_kernel(const float *__restrict__ prev_a, float *__restrict__ next_a, uint32_t total_a, uint32_t blocks_a,
                   const float *__restrict__ prev_b, float *__restrict__ next_b, uint32_t total_b, uint32_t blocks_b,
                   const __grid_constant__ Fin fin, const SA sa, const SB sb) {
    static_assert(FIN_THREADS == 256, "shift and finalize blocks share one launch");
    // Only the launch overlaps the predecessor (post-physics): the plain shift reads nothing that kernel writes, but
    // running this bandwidth-bound copy beside the latency-bound post-physics kernel was measured to cost more than
    // it hides (+13 % step time at 65 536 envs), so the data movement starts after it.
    hb::pdl_trigger();
    hb::pdl_wait();              // post-physics complete: reset flags, ballots, sums
    if constexpr (Fin::kOn) {
        // the finalize blocks come FIRST in the grid: their short latency chain (ballot scan, ids, means) then runs
        // under the shift instead of behind its last block
        const uint32_t fin_blocks = gridDim.x - blocks_a - blocks_b;
        if (blockIdx.x < fin_blocks) {
            reset_finalize_body(fin.p, fin.b, nullptr, nullptr, fin.tiles, fin.seg, fin.host_count, fin.rng_counter, blockIdx.x,
                                fin_blocks);
        } else {
            const uint32_t blk = blockIdx.x - fin_blocks;
            if (blk < blocks_a) stack_shift<SA, 4, true>(prev_a, next_a, total_a, blk, sa, fin.b.reset_buf);
            else stack_shift<SB, 4, true>(prev_b, next_b, total_b, blk - blocks_a, sb, fin.b.reset_buf);
        }
    } else {
        if (blockIdx.x < blocks_a) stack_shift<SA, 4, false>(prev_a, next_a, total_a, blockIdx.x, sa, nullptr);
        else stack_shift<SB, 4, false>(prev_b, next_b, total_b, blockIdx.x - blocks_a, sb, nullptr);
    }
}

// ------------------------------------------------------------------------------------------
// LeggedRobot._get_heights (legged_robot.py:759-795; SURVEY.md §8f rank 3): terrain height under a grid of points around
// each robot.  The points (base frame, z = 0) are rotated by the base's yaw - quat_apply_yaw (utils/math.py:39-43):
// x, y of the quaternion zeroed, normalised, quat_apply - shifted by the base position and the terrain border, divided by
// the horizontal scale and truncated to a cell; the height is the minimum of the cell and its +x / +y neighbours in the
// int16 height field, times the vertical scale.  One thread per (env, point); the field (a few MB) lives in L2, the
// [N, P] output is written coalesced.  Same fp32 operation order as the reference (this unit is built without FMA
// contraction), so the cell indices - and with them the heights - are bit-exact.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
get_heights_kernel(const float *__restrict__ root_states, const float *__restrict__ points_xy, const int16_t *__restrict__ field,
                   int rows, int cols, float border, float hscale, float vscale, long long total, int npoints,
                   const int32_t *__restrict__ env_ids, float *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long slot = i / npoints;
    const int j = (int)(i - slot * npoints);
    const long long env = env_ids ? env_ids[slot] : slot;
    const float *root = root_states + env * 13;
    // quat_apply_yaw: q = normalize((0, 0, qz, qw)); the norm sums the four squares in order (two exact zeros first)
    const float z0 = root[5], w0 = root[6];
    float nrm = sqrtf(((0.0f + 0.0f) + z0 * z0) + w0 * w0);
    nrm = fmaxf(nrm, 1e-9f);
    const float qz = z0 / nrm, qw = w0 / nrm;
    const float px = points_xy[2 * j], py = points_xy[2 * j + 1];
    // t = 2 * cross((0,0,qz), (px,py,0)) = 2 * (-(qz*py), qz*px, 0);  v + w*t + cross((0,0,qz), t)
    const float tx = (0.0f - qz * py) * 2.0f, ty = (qz * px - 0.0f) * 2.0f;
    const float rx = (px + qw * tx) + (0.0f - qz * ty);
    const float ry = (py + qw * ty) + (qz * tx - 0.0f);
    const float wx = ((rx + root[0]) + border) / hscale, wy = ((ry + root[1]) + border) / hscale;
    long long cx = (long long)wx, cy = (long long)wy;              // .long(): truncation toward zero
    cx = cx < 0 ? 0 : (cx > rows - 2 ? rows - 2 : cx);
    cy = cy < 0 ? 0 : (cy > cols - 2 ? cols - 2 : cy);
    const int16_t h1 = __ldg(field + cx * cols + cy), h2 = __ldg(field + (cx + 1) * cols + cy), h3 = __ldg(field + cx * cols + cy + 1);
    int16_t h = h1 < h2 ? h1 : h2;
    h = h < h3 ? h : h3;
    out[i] = (float)h * vscale;
}

// ------------------------------------------------------------------------------------------
// Host mirror of the stacked observations (a consumer on the CPU, rl_device = cpu: on_policy_runner.py:136 moves obs and
// critic_obs to the learner's device every step).  Of a step's [N, S*F] stack only the newest frame is new - the rest is
// the previous stack shifted by one frame - so instead of 27 MB per step (4096 hector envs) the GPU sends the newest
// frames: per env a ring of C + S - 1 frame slots in PINNED HOST memory (C >= S + 1); frame k goes to slot k mod C and,
// when that slot is one of the first S - 1, also to slot k mod C + C, so that the last S frames are always one contiguous
// run of S*F floats: the stacked observation of env n is a strided VIEW of the ring (row pitch (C + S - 1) * F floats),
// with nothing to move on the host.  The kernel stores straight into the mapped host rings over PCIe (one warp per env);
// for an env that the step reset, the other slots of its rings are zeroed first (reset_idx clears the history:
// hector_env.py:256-261).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
mirror_frames_kernel(const float *__restrict__ obs, int obs_ld, int row_a, int fa, const float *__restrict__ priv, int priv_ld, int row_b,
                     int fb, const uint8_t *__restrict__ reset_buf, int n, float *__restrict__ ring_a, int ca, int slot_a,
                     float *__restrict__ ring_b, int cb, int slot_b, int zero_only) {
    const int lane = threadIdx.x & 31, env = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= n) return;
    const int sa = row_a / fa, sb = row_b / fb;                      // frames per stack
    const int na = ca + sa - 1, nb = cb + sb - 1;                    // slots per ring
    const int dup_a = slot_a < sa - 1 ? slot_a + ca : -1, dup_b = slot_b < sb - 1 ? slot_b + cb : -1;
    float *ra = ring_a + (size_t)env * na * fa, *rb = ring_b + (size_t)env * nb * fb;
    if (reset_buf && reset_buf[env]) {          // every slot but those that receive the new frame (disjoint addresses: no ordering needed)
        for (int i = lane; obs && i < na * fa; i += 32) {
            const int sl = i / fa;
            if (sl != slot_a && sl != dup_a) ra[i] = 0.0f;
        }
        for (int i = lane; priv && i < nb * fb; i += 32) {
            const int sl = i / fb;
            if (sl != slot_b && sl != dup_b) rb[i] = 0.0f;
        }
    }
    if (zero_only) return;                      // the frames travel by DMA (hb_copy_rows) in this mode
    if (obs) {                                  // (either history may be left to another call)
        const float *oa = obs + (size_t)env * obs_ld + (row_a - fa);
        for (int i = lane; i < fa; i += 32) {
            const float v = oa[i];
            ra[slot_a * fa + i] = v;
            if (dup_a >= 0) ra[dup_a * fa + i] = v;
        }
    }
    if (priv) {
        const float *ob = priv + (size_t)env * priv_ld + (row_b - fb);
        for (int i = lane; i < fb; i += 32) {
            const float v = ob[i];
            rb[slot_b * fb + i] = v;
            if (dup_b >= 0) rb[dup_b * fb + i] = v;
        }
    }
}

int g_use_bulk = 1;
int g_runtime_task = 0;      // 1: the three built robots too run post_physics_kernel with the layout read at run time
int g_post_warps = 0;        // warps per post_physics_kernel tile, 4 or 8 (0: by shard width)
// Shards of at most this many 32-env tiles per SM run the eight-warp post-physics kernel: there the tiles of an SM are too
// few to hide one another's dependent chains (DESIGN.md §3, scripts/ab_post_physics.py: faster at 2.4 and 2.6 tiles per
// SM, slower from 3.0)
constexpr float POST_WIDE_MAX_TILES_PER_SM = 2.5f;

// Frame stacks of the three tasks (hector_config.py:8-20, hector_w_arm_config.py:8-20, humanoid_config.py:42-52): rows
// either dense or at the 128-byte pitch ceil32(row + 1) (TMA-addressable: the rollout storage's slots)
constexpr int pitchc(int v) { return (v + 31) / 32 * 32; }      // whole 128-byte lines: TMA box rows then touch 4 sectors, not 5
template <int OBS_, int S_, int PRIV_, int CS_>
struct StackShape {
    static constexpr int FRAME_A = OBS_, ROW_A = S_ * OBS_, LD_A = pitchc(ROW_A + 1);
    static constexpr int FRAME_B = PRIV_, ROW_B = CS_ * PRIV_, LD_B = pitchc(ROW_B + 1);
};
using ShapeHector = StackShape<41, 15, 70, 15>;
using ShapeHectorFull = StackShape<65, 15, 94, 15>;
using ShapeXBot = StackShape<47, 15, 73, 3>;

template <typename S>
struct DenseRows : S { static constexpr int LD_A = S::ROW_A, LD_B = S::ROW_B; };     // a built shape with dense rows

// blocks of stack_shift (256 threads, 4 float4 each) over `total` floats
uint32_t shift_blocks(uint32_t total) { return ((total + 3u) / 4u + 4 * 256 - 1) / (4 * 256); }

bool fits_u32(int n, int row) { return (long long)n * row + 64 * 1024 < (1ll << 32); }

template <typename T, bool kBulk, bool kWide>
int launch_post_physics(const hb_env_params *p, const hb_env_buffers *buf, const hb_env_noise *noise, float *obs_new,
                        float *priv_new, int32_t stages, cudaStream_t st) {
    const bool with_noise = p->add_noise && (noise->z_obs || noise->rng_counter);
    const TileLayout L = make_layout(p->num_bodies, with_noise, p->num_dof, p->num_single_obs, p->num_single_priv, kWide);
    const auto kernel = kWide ? post_physics_wide_kernel<kBulk, T> : post_physics_kernel<kBulk, T>;
    const size_t smem = (size_t)L.total * sizeof(float);
    const int tiles = (p->num_envs + TILE - 1) / TILE;
    static bool attr_set = false;
    if (!attr_set) {
        HB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, POST_SMEM_MAX));
        attr_set = true;
    }
    HB_CUDA(hb::launch_pdl(hb::use_pdl_post(p->num_envs), kernel, dim3(tiles), dim3((kWide ? 8 : 4) * TILE),
                           smem, st, *p, *buf,
                           *noise, obs_new, priv_new, (int)stages));
    HB_CHECK_LAUNCH("post_physics_kernel");
    return HB_OK;
}

// The frame-stack shift of both histories (a: actor, b: critic): shapes and grid, which built shape they are (0 hector,
// 1 hector_full, 2 XBot-L) and in which layout (0 = not a built shape, 1 = dense rows, 2 = 128-byte pitch), and whether
// the compiled kernel of that shape applies (fast) or else the runtime-shape kernel (vec: 16-byte aligned buffers).
// reset_buf: the envs whose carried frames a shift without finalisation zeroes (null: none).
struct StackPlan {
    ShiftShape a, b;
    int num_envs, shape, layout;
    bool fast, vec;
    uint32_t total_a, total_b, blocks_a, blocks_b;
    const uint8_t *reset_buf;
};

// (ld 0: a stack of no frames in the caller's params, which shifts nothing - no reciprocal, no division by zero)
ShiftShape shift_shape(int row, int ld, int frame) {
    return {(uint32_t)row, (uint32_t)ld, (uint32_t)frame, ld > 0 ? ~0ull / (unsigned long long)ld + 1ull : 0ull};
}

template <typename S>
int shape_layout(const StackPlan &s) {
    if (s.a.row != S::ROW_A || s.a.frame != S::FRAME_A || s.b.row != S::ROW_B || s.b.frame != S::FRAME_B) return 0;
    return s.a.ld == S::ROW_A && s.b.ld == S::ROW_B ? 1 : (s.a.ld == S::LD_A && s.b.ld == S::LD_B ? 2 : 0);
}

StackPlan stack_plan(int num_envs, ShiftShape a, ShiftShape b, bool aligned) {
    StackPlan s;
    s.a = a, s.b = b, s.num_envs = num_envs, s.reset_buf = nullptr;
    const int layouts[3] = {shape_layout<ShapeHector>(s), shape_layout<ShapeHectorFull>(s), shape_layout<ShapeXBot>(s)};
    s.shape = layouts[0] ? 0 : (layouts[1] ? 1 : 2);
    s.layout = layouts[s.shape];
    s.vec = aligned && fits_u32(num_envs, a.ld > b.ld ? a.ld : b.ld);
    s.fast = s.vec && s.layout != 0;
    s.total_a = (uint32_t)num_envs * a.ld, s.total_b = (uint32_t)num_envs * b.ld;
    // a stack of one frame carries nothing over: no shift blocks
    s.blocks_a = a.row > a.frame ? shift_blocks(s.total_a) : 0;
    s.blocks_b = b.row > b.frame ? shift_blocks(s.total_b) : 0;
    return s;
}

// The env's two histories
StackPlan stack_plan(const hb_env_params *p, const float *obs_prev, const float *priv_prev, const float *obs_new,
                     const float *priv_new) {
    const int row_a = p->frame_stack * p->num_single_obs, row_b = p->c_frame_stack * p->num_single_priv;
    return stack_plan(p->num_envs, shift_shape(row_a, p->obs_ld ? p->obs_ld : row_a, p->num_single_obs),
                      shift_shape(row_b, p->priv_ld ? p->priv_ld : row_b, p->num_single_priv),
                      hb::aligned16(obs_prev) && hb::aligned16(obs_new) && hb::aligned16(priv_prev) && hb::aligned16(priv_new));
}

// One dense history (hb_stack_shift), in slot b if it has the shape of hector's critic history, else in slot a; the other
// slot is empty.  Hector's two dense histories, without reset flags, run the compiled kernel of hector's dense stack.
StackPlan stack_plan(int num_envs, int row, int frame, bool aligned, const uint8_t *reset_buf) {
    using H = DenseRows<ShapeHector>;
    const bool in_b = row == H::ROW_B && frame == H::FRAME_B;
    StackPlan s = {};
    (in_b ? s.b : s.a) = shift_shape(row, row, frame);
    const uint32_t total = (uint32_t)num_envs * row;
    (in_b ? s.total_b : s.total_a) = total;
    (in_b ? s.blocks_b : s.blocks_a) = shift_blocks(total);
    s.num_envs = num_envs, s.reset_buf = reset_buf;
    s.shape = 0, s.layout = in_b || (row == H::ROW_A && frame == H::FRAME_A) ? 1 : 0;
    s.vec = aligned && fits_u32(num_envs, row);
    s.fast = s.vec && s.layout != 0 && !reset_buf;
    return s;
}

// Grid of the shard-wide reset finalisation: each CTA owns a contiguous segment of at least 8 32-env tiles
struct FinalizeGrid { int tiles, seg, blocks; };

FinalizeGrid finalize_grid(int num_envs) {
    const int tiles = (num_envs + TILE - 1) / TILE;
    int seg = (tiles + hb::sm_count() - 1) / hb::sm_count();
    if (seg < 8) seg = 8;
    return {tiles, seg, (tiles + seg - 1) / seg};
}

// The frame-stack launch of plan s: the compiled kernel of a built shape (fast), else the runtime-shape kernel (vec),
// else the scalar shift of each history.  With `finalize` the reset finalisation of p / buf runs too: in the same grid,
// its blocks first, or behind the scalar shift as reset_finalize_kernel.  p null: a lone shift (hb_stack_shift), launched
// without PDL.
int launch_stack(const hb_env_params *p, const hb_env_buffers *buf, const StackPlan &s, const float *prev_a, const float *prev_b,
                 float *next_a, float *next_b, bool finalize, int32_t *host_count, uint64_t *rng_counter, cudaStream_t st) {
    if (!s.vec) {           // unaligned or oversized buffers
        const ShiftShape *sh[2] = {&s.a, &s.b};
        const float *prev[2] = {prev_a, prev_b};
        float *next[2] = {next_a, next_b};
        for (int h = 0; h < 2; ++h) {
            if (sh[h]->row <= sh[h]->frame) continue;       // carries nothing over (the block counts may have wrapped here)
            const long long total = (long long)s.num_envs * sh[h]->ld;
            stack_shift_scalar_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(prev[h], next[h], s.reset_buf, total,
                                                                                       sh[h]->row, sh[h]->ld, sh[h]->frame);
            HB_CHECK_LAUNCH("stack_shift_scalar_kernel");
        }
        return finalize ? hb_env_reset_finalize(p, buf, next_a, next_b, host_count, rng_counter, st) : HB_OK;
    }
    FinalizeArgs fin = {};
    uint32_t fin_blocks = 0;
    if (finalize) {
        const FinalizeGrid g = finalize_grid(s.num_envs);
        fin = {*p, *buf, g.tiles, g.seg, host_count, reinterpret_cast<unsigned long long *>(rng_counter)};
        fin_blocks = (uint32_t)g.blocks;
    } else {
        fin.b.reset_buf = const_cast<uint8_t *>(s.reset_buf);      // the runtime-shape kernel's zeroing (only read)
    }
    if (s.blocks_a + s.blocks_b + fin_blocks == 0) return HB_OK;
    const bool pdl_stack = p && hb::use_pdl_stack(s.num_envs);
    auto launch = [&](auto kernel, bool pdl, auto fin_, auto sa, auto sb) {
        return hb::launch_pdl(pdl, kernel, dim3(fin_blocks + s.blocks_a + s.blocks_b), dim3(256), 0, st, prev_a, next_a, s.total_a,
                              s.blocks_a, prev_b, next_b, s.total_b, s.blocks_b, fin_, sa, sb);
    };
    // a built shape: the kernel whose FixedShift constants are its StackShape (pitched rows) or DenseRows
    auto built = [&](auto shape) {
        using R = decltype(shape);
        using A = FixedShift<R::ROW_A, R::LD_A, R::FRAME_A>;
        using B = FixedShift<R::ROW_B, R::LD_B, R::FRAME_B>;
        return finalize ? launch(stack_shift_kernel<A, B, FinalizeArgs>, pdl_stack, fin, A{}, B{})
                        : launch(stack_shift_kernel<A, B, NoFinalize>, p && hb::use_pdl(s.num_envs), NoFinalize{}, A{}, B{});
    };
    auto rows = [&](auto shape) {
        using S = decltype(shape);
        return s.layout == 2 ? built(S{}) : built(DenseRows<S>{});
    };
    HB_CUDA(!s.fast ? launch(stack_shift_kernel<ShiftShape, ShiftShape, FinalizeArgs>, pdl_stack, fin, s.a, s.b)
                    : (s.shape == 0 ? rows(ShapeHector{}) : (s.shape == 1 ? rows(ShapeHectorFull{}) : rows(ShapeXBot{}))));
    HB_CHECK_LAUNCH("stack_shift_kernel");
    return HB_OK;
}

PdConsts pd_consts(const hb_env_params *p) {
    PdConsts c;
    for (int j = 0; j < HB_MAX_DOF; ++j) c.q0[j] = p->default_dof_pos[j], c.lim[j] = p->torque_limits[j];
    return c;
}

// two DOFs per thread: an even joint count, 16-byte (pos, vel) pairs and 8-byte aligned per-DOF buffers
bool pd_vectorizable(const hb_env_params *p, const hb_env_buffers *buf) {
    return (p->num_dof % 2 == 0) && hb::aligned16(buf->dof_state) &&
           ((reinterpret_cast<uintptr_t>(buf->actions) | reinterpret_cast<uintptr_t>(buf->p_gains) |
             reinterpret_cast<uintptr_t>(buf->d_gains) | reinterpret_cast<uintptr_t>(buf->torques)) & 7u) == 0;
}

}  // namespace

// ==============================================================================================
// C ABI
// ==============================================================================================
extern "C" {

#ifdef HB_POST_TIMING
int hb_debug_post_stamps(long long *dst_host, int count) {
    HB_CUDA(cudaMemcpyFromSymbol(dst_host, g_post_stamps, sizeof(long long) * count));
    return HB_OK;
}
int hb_debug_post_globaltimes(unsigned long long *dst_host, int count) {
    HB_CUDA(cudaMemcpyFromSymbol(dst_host, g_post_gt, sizeof(unsigned long long) * count));
    return HB_OK;
}
#endif

int hb_set_option(const char *name, int value) {
    if (name && !strcmp(name, "env_bulk_staging")) {
        g_use_bulk = value;
        return HB_OK;
    }
    if (name && !strcmp(name, "env_runtime_task")) {
        g_runtime_task = value != 0;
        return HB_OK;
    }
    if (name && !strcmp(name, "post_warps")) {
        HB_REQUIRE(value == 0 || value == 4 || value == 8, "hb_set_option: post_warps must be 0, 4 or 8");
        g_post_warps = value;
        return HB_OK;
    }
    if (name && !strcmp(name, "gemm_pdl")) {
        hb::g_gemm_pdl = value != 0;
        return HB_OK;
    }
    if (name && !strcmp(name, "gemm_tile_snake")) {
        hb::g_gemm_snake = value != 0;
        return HB_OK;
    }
    if (name && !strcmp(name, "gae_serial_min_envs")) {
        hb::g_gae_serial_min_envs = value;
        return HB_OK;
    }
    if (name && !strcmp(name, "gae_threads")) {
        HB_REQUIRE(value == 0 || value == 32 || value == 64 || value == 128 || value == 256, "hb_set_option: gae_threads must be 0, 32, 64, 128 or 256");
        hb::g_gae_threads = value;
        return HB_OK;
    }
    if (name && !strcmp(name, "pdl")) {
        hb::g_use_pdl = value;
        return HB_OK;
    }
    if (name && !strcmp(name, "coop_launch")) {
        hb::g_coop_launch = value != 0;
        return HB_OK;
    }
    hb::set_error("hb_set_option: unknown option '%s'", name ? name : "(null)");
    return HB_ERR_BAD_ARG;
}

// The layout of a robot that post_physics_kernel reads at run time (RuntimeTask)
static int check_runtime_task(const hb_env_params *p) {
    const int n = p->num_dof;
    if (n > MAX_TASK_DOF) {
        hb::set_error("hb_env_post_physics: num_dof=%d is not supported (1 to %d joints: the observation frame 3 num_dof + 11 "
                      "must fit %d columns)", n, MAX_TASK_DOF, HB_MAX_OBS);
        return HB_ERR_UNSUPPORTED;
    }
    HB_REQUIRE(p->task_kind == HB_TASK_HECTOR || p->task_kind == HB_TASK_XBOT, "hb_env_post_physics: task_kind=%d (0 hector, 1 XBot-L)",
               p->task_kind);
    const TaskDims d = task_dims(n, p->task_kind == HB_TASK_XBOT ? KIND_XBOT : KIND_HECTOR, 0, 0, 0, 0);
    HB_REQUIRE(p->num_single_obs == d.OBS && p->num_single_priv == d.PRIV,
               "hb_env_post_physics: frames %d / %d do not match num_dof=%d task_kind=%d (%d / %d: 3 num_dof + 11 and %s)",
               p->num_single_obs, p->num_single_priv, n, p->task_kind, d.OBS, d.PRIV,
               p->task_kind == HB_TASK_XBOT ? "4 num_dof + 25" : "3 num_dof + 40");
    auto pair_ok = [&](int j) { return j >= 0 && j + 1 < n; };
    HB_REQUIRE(pair_ok(p->yaw_roll[0]) && pair_ok(p->yaw_roll[1]),
               "hb_env_post_physics: yaw_roll (%d, %d): each pair's first joint j needs 0 <= j and j + 1 < num_dof=%d", p->yaw_roll[0],
               p->yaw_roll[1], n);
    HB_REQUIRE((p->arm_pair[0] == -1 && p->arm_pair[1] == -1) || (pair_ok(p->arm_pair[0]) && pair_ok(p->arm_pair[1])),
               "hb_env_post_physics: arm_pair (%d, %d): -1, -1 (no arms) or first joints j with 0 <= j and j + 1 < num_dof=%d",
               p->arm_pair[0], p->arm_pair[1], n);
    for (int k = 0; k < 3; ++k)
        HB_REQUIRE(p->ref_left[k] >= 0 && p->ref_left[k] < n && p->ref_right[k] >= 0 && p->ref_right[k] < n,
                   "hb_env_post_physics: ref_left / ref_right [%d] = %d / %d outside [0, num_dof=%d)", k, p->ref_left[k], p->ref_right[k], n);
    return HB_OK;
}

static int check_params(const hb_env_params *p, const hb_env_buffers *buf, const char *who) {
    HB_REQUIRE(p && buf, "%s: null params/buffers", who);
    HB_REQUIRE(p->abi_version == HB_ABI_VERSION, "%s: ABI version %d != %d", who, p->abi_version, HB_ABI_VERSION);
    HB_REQUIRE(p->num_envs > 0, "%s: num_envs must be positive", who);
    HB_REQUIRE(p->resample_interval > 0, "%s: resample_interval must be positive", who);
    HB_REQUIRE(p->num_dof > 0 && p->num_dof <= HB_MAX_DOF, "%s: num_dof=%d out of range", who, p->num_dof);
    HB_REQUIRE((p->obs_ld == 0 || p->obs_ld >= p->frame_stack * p->num_single_obs) &&
                   (p->priv_ld == 0 || p->priv_ld >= p->c_frame_stack * p->num_single_priv),
               "%s: obs_ld / priv_ld (%d / %d) shorter than a row", who, p->obs_ld, p->priv_ld);
    return HB_OK;
}

int hb_env_action_prologue(const hb_env_params *p, const hb_env_buffers *buf, const float *actions_in,
                           const hb_env_noise *noise, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_action_prologue")) return rc;
    HB_REQUIRE(actions_in && buf->actions, "hb_env_action_prologue: null actions");
    const int total = p->num_envs * p->num_dof;
    hb_env_noise none = {};
    action_prologue_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        actions_in, buf->actions, noise ? *noise : none, total, p->num_dof, p->clip_actions, p->action_delay, p->action_noise);
    HB_CHECK_LAUNCH("action_prologue_kernel");
    return HB_OK;
}

int hb_env_prologue_torques(const hb_env_params *p, const hb_env_buffers *buf, const float *actions_in,
                            const hb_env_noise *noise, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_prologue_torques")) return rc;
    HB_REQUIRE(actions_in && buf->actions && buf->dof_state && buf->p_gains && buf->d_gains && buf->torques,
               "hb_env_prologue_torques: null buffer");
    if (!pd_vectorizable(p, buf)) {        // unaligned buffers / odd joint count: the two separate launches
        if (int rc = hb_env_action_prologue(p, buf, actions_in, noise, stream)) return rc;
        return hb_env_compute_torques(p, buf, stream);
    }
    const int pairs = p->num_envs * p->num_dof / 2;
    hb_env_noise none = {};
    prologue_pd_kernel<<<(pairs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        actions_in, buf->actions, noise ? *noise : none, p->clip_actions, p->action_delay, p->action_noise,
        reinterpret_cast<const float4 *>(buf->dof_state), reinterpret_cast<const float2 *>(buf->p_gains),
        reinterpret_cast<const float2 *>(buf->d_gains), reinterpret_cast<float2 *>(buf->torques), pairs, p->num_dof,
        p->action_scale, pd_consts(p));
    HB_CHECK_LAUNCH("prologue_pd_kernel");
    return HB_OK;
}

int hb_env_compute_torques(const hb_env_params *p, const hb_env_buffers *buf, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_compute_torques")) return rc;
    HB_REQUIRE(buf->dof_state && buf->actions && buf->p_gains && buf->d_gains && buf->torques,
               "hb_env_compute_torques: null buffer");
    const PdConsts c = pd_consts(p);
    const int total = p->num_envs * p->num_dof;
    if (pd_vectorizable(p, buf)) {
        const int pairs = total / 2;
        HB_CUDA(hb::launch_pdl(hb::use_pdl_small_kernel(p->num_envs), pd_torque_kernel, dim3((pairs + 255) / 256), dim3(256), 0, (cudaStream_t)stream,
                               reinterpret_cast<const float4 *>(buf->dof_state), reinterpret_cast<const float2 *>(buf->actions),
                               reinterpret_cast<const float2 *>(buf->p_gains), reinterpret_cast<const float2 *>(buf->d_gains),
                               reinterpret_cast<float2 *>(buf->torques), pairs, p->num_dof, p->action_scale, c));
    } else {
        HB_CUDA(hb::launch_pdl(hb::use_pdl_small_kernel(p->num_envs), pd_torque_scalar_kernel, dim3((total + 255) / 256), dim3(256), 0, (cudaStream_t)stream,
                               (const float *)buf->dof_state, (const float *)buf->actions, buf->p_gains, buf->d_gains,
                               buf->torques, total, p->num_dof, p->action_scale, c));
    }
    HB_CHECK_LAUNCH("pd_torque_kernel");
    return HB_OK;
}

int hb_env_post_physics(const hb_env_params *p, const hb_env_buffers *buf, const hb_env_noise *noise,
                        float *obs_new, float *priv_new, int32_t stages, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_post_physics")) return rc;
    HB_REQUIRE(noise && obs_new && priv_new, "hb_env_post_physics: null noise/obs pointers");
    HB_REQUIRE(p->num_bodies > 0 && p->num_bodies <= 32, "hb_env_post_physics: num_bodies out of range");
    HB_REQUIRE(p->n_term >= 0 && p->n_term <= HB_MAX_CONTACT_BODIES && p->n_pen >= 0 &&
                   p->n_pen <= HB_MAX_CONTACT_BODIES, "hb_env_post_physics: too many contact bodies");
    HB_REQUIRE(noise->u_reset || noise->rng_counter, "hb_env_post_physics: u_reset or the device generator is required (any env may reset)");
    HB_REQUIRE(buf->scratch_ballots && buf->scratch_sums, "hb_env_post_physics: null scratch buffers");
    HB_REQUIRE((p->reward_scale[HB_R_JOINT_POS] == 0.0f && p->task_kind != HB_TASK_XBOT) || buf->ref_dof_pos,
               "hb_env_post_physics: ref_dof_pos is required (joint_pos reward / XBot-L privileged frame)");
    // bulk staging needs 16-byte aligned slabs: base pointers aligned and 32-env tiles (128-byte multiples)
    bool bulk = g_use_bulk != 0;
    const void *slabs[] = {buf->root_states, buf->dof_state, buf->contact_forces, buf->actions, buf->last_actions,
                           buf->last_last_actions, buf->last_dof_vel, buf->torques, buf->last_root_vel,
                           buf->commands};
    bool all_aligned = true;
    for (const void *s : slabs) all_aligned = all_aligned && hb::aligned16(s);
    HB_REQUIRE(all_aligned, "hb_env_post_physics: state tensors must be 16-byte aligned");
    if (p->add_noise && noise->z_obs && !hb::aligned16(noise->z_obs)) bulk = false;      // caller-supplied draws at an odd offset: plain loads
    cudaStream_t st = (cudaStream_t)stream;
    // the three registered tasks (envs/__init__.py:46-48)
    using Hector = Task<10, KIND_HECTOR, true>;
    using HectorSlim = Task<10, KIND_HECTOR, false>;
    using HectorFull = Task<18, KIND_HECTOR, true>;
    using HectorFullSlim = Task<18, KIND_HECTOR, false>;
    using XBot = Task<12, KIND_XBOT, true>;
    // the joint pairs of default_joint_pos are constants of the three robots, compiled into their kernels
    auto matches = [&](int ndof, int kind, int obs, int priv) {
        const bool arms = ndof == 18;
        return !g_runtime_task && p->num_dof == ndof && p->task_kind == kind && p->num_single_obs == obs &&
               p->num_single_priv == priv && p->yaw_roll[0] == 0 && p->yaw_roll[1] == ndof / 2 &&
               p->arm_pair[0] == (arms ? 5 : -1) && p->arm_pair[1] == (arms ? ndof / 2 + 5 : -1);
    };
    // a config that scales none of the optional terms runs the kernel compiled without them
    const bool opt = p->reward_scale[HB_R_JOINT_POS] != 0.0f || p->reward_scale[HB_R_VEL_MISMATCH_EXP] != 0.0f ||
                     p->reward_scale[HB_R_TRACK_VEL_HARD] != 0.0f || p->reward_scale[HB_R_LOW_SPEED] != 0.0f;
    const int tiles = (p->num_envs + TILE - 1) / TILE;
    const bool wide = g_post_warps ? g_post_warps == 8 : tiles <= POST_WIDE_MAX_TILES_PER_SM * hb::sm_count();
    auto launch = [&](auto task) {
        using T = decltype(task);
        if (wide)
            return bulk ? launch_post_physics<T, true, true>(p, buf, noise, obs_new, priv_new, stages, st)
                        : launch_post_physics<T, false, true>(p, buf, noise, obs_new, priv_new, stages, st);
        return bulk ? launch_post_physics<T, true, false>(p, buf, noise, obs_new, priv_new, stages, st)
                    : launch_post_physics<T, false, false>(p, buf, noise, obs_new, priv_new, stages, st);
    };
    if (matches(10, HB_TASK_HECTOR, Hector::OBS, Hector::PRIV)) return opt ? launch(Hector{}) : launch(HectorSlim{});
    if (matches(18, HB_TASK_HECTOR, HectorFull::OBS, HectorFull::PRIV)) return opt ? launch(HectorFull{}) : launch(HectorFullSlim{});
    if (matches(12, HB_TASK_XBOT, XBot::OBS, XBot::PRIV)) return launch(XBot{});
    // any other robot: the kernel with the layout read from p
    if (int rc = check_runtime_task(p)) return rc;
    return p->task_kind == HB_TASK_XBOT ? launch(RuntimeTask<KIND_XBOT>{}) : launch(RuntimeTask<KIND_HECTOR>{});
}

int hb_env_get_heights(const float *root_states, const float *points_xy, int32_t num_points, const int16_t *height_samples,
                       int32_t rows, int32_t cols, float border_size, float horizontal_scale, float vertical_scale,
                       const int32_t *env_ids, int64_t count, float *heights, void *stream) {
    HB_REQUIRE(root_states && points_xy && height_samples && heights, "hb_env_get_heights: null buffer");
    HB_REQUIRE(num_points > 0 && rows >= 2 && cols >= 2 && count > 0 && horizontal_scale > 0.0f, "hb_env_get_heights: bad sizes");
    const long long total = (long long)count * num_points;
    get_heights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        root_states, points_xy, height_samples, rows, cols, border_size, horizontal_scale, vertical_scale, total, num_points,
        env_ids, heights);
    HB_CHECK_LAUNCH("get_heights_kernel");
    return HB_OK;
}

int hb_stack_shift(const float *prev, float *next, const uint8_t *reset_buf, int32_t num_envs, int32_t row,
                   int32_t frame, void *stream) {
    HB_REQUIRE(prev && next && prev != next, "hb_stack_shift: null or aliasing buffers");
    HB_REQUIRE(num_envs > 0 && frame > 0 && row > frame, "hb_stack_shift: bad shape");
    const StackPlan s = stack_plan(num_envs, row, frame, hb::aligned16(prev) && hb::aligned16(next), reset_buf);
    const bool in_b = s.b.row != 0;                     // the history went to slot b
    return launch_stack(nullptr, nullptr, s, in_b ? nullptr : prev, in_b ? prev : nullptr, in_b ? nullptr : next,
                        in_b ? next : nullptr, false, nullptr, nullptr, (cudaStream_t)stream);
}

int hb_env_stack_observations(const hb_env_params *p, const hb_env_buffers *buf, const float *obs_prev,
                              const float *priv_prev, float *obs_new, float *priv_new, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_stack_observations")) return rc;
    HB_REQUIRE(obs_prev && priv_prev && obs_new && priv_new, "hb_env_stack_observations: null buffer");
    HB_REQUIRE(obs_prev != obs_new && priv_prev != priv_new, "hb_env_stack_observations: prev and new must not alias");
    return launch_stack(p, buf, stack_plan(p, obs_prev, priv_prev, obs_new, priv_new), obs_prev, priv_prev, obs_new, priv_new,
                        false, nullptr, nullptr, (cudaStream_t)stream);
}

int hb_env_stack_finalize(const hb_env_params *p, const hb_env_buffers *buf, const float *obs_prev, const float *priv_prev,
                          float *obs_new, float *priv_new, int32_t *host_count, uint64_t *rng_counter, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_stack_finalize")) return rc;
    HB_REQUIRE(obs_prev && priv_prev && obs_new && priv_new && buf->reset_buf, "hb_env_stack_finalize: null buffer");
    HB_REQUIRE(obs_prev != obs_new && priv_prev != priv_new, "hb_env_stack_finalize: prev and new must not alias");
    HB_REQUIRE(buf->scratch_ballots && buf->scratch_sums && buf->reset_env_ids && buf->reset_count && buf->episode_means,
               "hb_env_stack_finalize: null scratch/result buffers");
    return launch_stack(p, buf, stack_plan(p, obs_prev, priv_prev, obs_new, priv_new), obs_prev, priv_prev, obs_new, priv_new,
                        true, host_count, rng_counter, (cudaStream_t)stream);
}

int hb_env_mirror_frames(const float *obs, int32_t obs_ld, int32_t obs_row, int32_t obs_frame, const float *priv, int32_t priv_ld,
                         int32_t priv_row, int32_t priv_frame, const uint8_t *reset_buf, int32_t num_envs, float *host_obs_ring,
                         int32_t obs_slots, int32_t obs_slot, float *host_priv_ring, int32_t priv_slots, int32_t priv_slot, int32_t use_dma,
                         void *stream) {
    HB_REQUIRE((obs || priv) && host_obs_ring && host_priv_ring && num_envs > 0, "hb_env_mirror_frames: null buffer");
    HB_REQUIRE(obs_frame > 0 && obs_row >= obs_frame && obs_ld >= obs_row && priv_frame > 0 && priv_row >= priv_frame && priv_ld >= priv_row,
               "hb_env_mirror_frames: bad row shapes");
    HB_REQUIRE(obs_row % obs_frame == 0 && priv_row % priv_frame == 0, "hb_env_mirror_frames: a row is a whole number of frames");
    HB_REQUIRE(obs_slots * obs_frame > obs_row && priv_slots * priv_frame > priv_row && obs_slot >= 0 && obs_slot < obs_slots &&
                   priv_slot >= 0 && priv_slot < priv_slots,
               "hb_env_mirror_frames: a ring needs more slots than the stack has frames (C >= S + 1), slot index inside [0, C)");
    const int warps = 8;
    cudaStream_t st = (cudaStream_t)stream;
    if (use_dma) {          // frames by the copy engine (2-D copies with frame-wide rows), the kernel only zeroes the rings of reset envs
        if (reset_buf) {
            mirror_frames_kernel<<<(num_envs + warps - 1) / warps, warps * 32, 0, st>>>(
                obs, obs_ld, obs_row, obs_frame, priv, priv_ld, priv_row, priv_frame, reset_buf, num_envs, host_obs_ring, obs_slots, obs_slot,
                host_priv_ring, priv_slots, priv_slot, 1);
        }
        const int sa = obs_row / obs_frame, sb = priv_row / priv_frame;
        const size_t pitch_a = (size_t)(obs_slots + sa - 1) * obs_frame * 4, pitch_b = (size_t)(priv_slots + sb - 1) * priv_frame * 4;
        auto dma = [&](float *ring, size_t pitch, int slot, int frame, const float *src, int ld, int row) {
            return cudaMemcpy2DAsync(ring + (size_t)slot * frame, pitch, src + (row - frame), (size_t)ld * 4, (size_t)frame * 4, (size_t)num_envs,
                                     cudaMemcpyDeviceToHost, st);
        };
        if (obs) {
            HB_CUDA(dma(host_obs_ring, pitch_a, obs_slot, obs_frame, obs, obs_ld, obs_row));
            if (obs_slot < sa - 1) HB_CUDA(dma(host_obs_ring, pitch_a, obs_slot + obs_slots, obs_frame, obs, obs_ld, obs_row));
        }
        if (priv) {
            HB_CUDA(dma(host_priv_ring, pitch_b, priv_slot, priv_frame, priv, priv_ld, priv_row));
            if (priv_slot < sb - 1) HB_CUDA(dma(host_priv_ring, pitch_b, priv_slot + priv_slots, priv_frame, priv, priv_ld, priv_row));
        }
        return HB_OK;
    }
    mirror_frames_kernel<<<(num_envs + warps - 1) / warps, warps * 32, 0, st>>>(
        obs, obs_ld, obs_row, obs_frame, priv, priv_ld, priv_row, priv_frame, reset_buf, num_envs, host_obs_ring, obs_slots, obs_slot,
        host_priv_ring, priv_slots, priv_slot, 0);
    HB_CHECK_LAUNCH("mirror_frames_kernel");
    return HB_OK;
}

int hb_env_reset_finalize(const hb_env_params *p, const hb_env_buffers *buf, float *obs_new, float *priv_new,
                          int32_t *host_count, uint64_t *rng_counter, void *stream) {
    if (int rc = check_params(p, buf, "hb_env_reset_finalize")) return rc;
    HB_REQUIRE(buf->scratch_ballots && buf->scratch_sums && buf->reset_env_ids && buf->reset_count && buf->episode_means,
               "hb_env_reset_finalize: null scratch/result buffers");
    HB_REQUIRE((obs_new == nullptr) == (priv_new == nullptr), "hb_env_reset_finalize: pass both frame stacks or neither");
    HB_REQUIRE(!buf->time_outs_latched || buf->time_out_buf, "hb_env_reset_finalize: latch without time_out_buf");
    const FinalizeGrid g = finalize_grid(p->num_envs);
    HB_CUDA(hb::launch_pdl(hb::use_pdl(p->num_envs), reset_finalize_kernel, dim3(g.blocks), dim3(FIN_THREADS), 0, (cudaStream_t)stream, *p, *buf,
                           obs_new, priv_new, g.tiles, g.seg, host_count, reinterpret_cast<unsigned long long *>(rng_counter)));
    HB_CHECK_LAUNCH("reset_finalize_kernel");
    return HB_OK;
}

}  // extern "C"
