// PPO update kernels around the tcgen05 GEMMs (SURVEY.md §8 rows a12, a14, a15), sm_100a.
//   - minibatch gathers (rollout_storage.py:146-182), done once per update
//   - loss head + analytic backward (ppo.py:130-168) and the PPO.act sampling head (ppo.py:91-101)
//   - clip_grad_norm_ + Adam with the adaptive-KL learning rate evaluated on the device (ppo.py:136-148,171-174)
#include <math.h>

#include "hb_common.cuh"

namespace {

// The PPO head kernels are templated on the number of actions NA.  10 (hector), 12 (XBot-L) and 18 (hector_full) are
// compiled for their count; every other count runs the NA_RUNTIME instantiation, which takes it as a kernel argument
// (loss_head_kernel: LossCoefs::num_actions).  A sample's record is 3 NA + 6 floats.  HB_PPO_DISPATCH picks the
// instantiation, HB_PPO_FUSED_DISPATCH that of the fused heads.  Each entry point first checks 1 <= na <= max with
// HB_PPO_CHECK_ACTIONS: below 1 is HB_ERR_BAD_ARG, above the limit HB_ERR_UNSUPPORTED, and `msg` (printf format, one %d
// for the count) names the range.
constexpr int NA_RUNTIME = 0;
constexpr int MAX_ACTIONS = 64;
constexpr int MAX_FUSED_ACTIONS = 15;       // one lane pair per action and one for the value in a 16-value butterfly
#define HB_PPO_CHECK_ACTIONS(na, max, msg)                                                \
    if ((na) < 1 || (na) > (max)) {                                                       \
        hb::set_error(msg, (int)(na));                                                    \
        return (na) < 1 ? HB_ERR_BAD_ARG : HB_ERR_UNSUPPORTED;                            \
    }
#define HB_PPO_DISPATCH(na, CALL)                                                         \
    switch (na) {                                                                         \
        case 10: { constexpr int NA = 10; CALL; break; }                                  \
        case 12: { constexpr int NA = 12; CALL; break; }                                  \
        case 18: { constexpr int NA = 18; CALL; break; }                                  \
        default: { constexpr int NA = NA_RUNTIME; CALL; break; }                          \
    }
#define HB_PPO_FUSED_DISPATCH(na, CALL)                                                   \
    switch (na) {                                                                         \
        case 10: { constexpr int NA = 10; CALL; break; }                                  \
        case 12: { constexpr int NA = 12; CALL; break; }                                  \
        default: { constexpr int NA = NA_RUNTIME; CALL; break; }                          \
    }
constexpr float HALF_LOG_2PI = 0.91893853320467274178f;     // log(sqrt(2*pi))

__global__ void __launch_bounds__(256)
gather_rows_kernel(const float *__restrict__ src, int ld_src, float *__restrict__ dst, int ld_dst,
                   const int64_t *__restrict__ perm, long long rows, int cols, int ones_col) {
    const int lane = threadIdx.x & 31;
    const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;      // one warp per row
    if (row >= rows) return;
    const float *s = src + (size_t)perm[row] * ld_src;
    float *d = dst + (size_t)row * ld_dst;
    const int vec = cols >> 2;
    const float4 *s4 = reinterpret_cast<const float4 *>(s);
    float4 *d4 = reinterpret_cast<float4 *>(d);
    // a row is a few KB at a random place: all of a lane's 16-byte loads are issued before the first store
    constexpr int INFLIGHT = 9;          // 9 x 32 lanes x 4 floats = rows of up to 1152 floats in one round
    for (int base = 0; base < vec; base += INFLIGHT * 32) {
        float4 v[INFLIGHT];
#pragma unroll
        for (int u = 0; u < INFLIGHT; ++u) {
            const int i = base + u * 32 + lane;
            if (i < vec) v[u] = hb::ld_stream4(s4 + i);
        }
#pragma unroll
        for (int u = 0; u < INFLIGHT; ++u) {
            const int i = base + u * 32 + lane;
            if (i < vec) hb::st_stream4(d4 + i, v[u]);
        }
    }
    for (int i = (vec << 2) + lane; i < cols; i += 32) d[i] = s[i];
    if (ones_col >= 0 && lane == 0) d[ones_col] = 1.0f;
}

template <int NA>
__global__ void __launch_bounds__(256)
pack_samples_kernel(const int64_t *__restrict__ perm, long long rows, const float *__restrict__ actions,
                    const float *__restrict__ mu, const float *__restrict__ sigma, const float *__restrict__ values,
                    const float *__restrict__ adv, const float *__restrict__ ret, const float *__restrict__ logp,
                    float *__restrict__ rec, int num_actions) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    const int na = NA != NA_RUNTIME ? NA : num_actions;
    const int REC = 3 * na + 6;
    const long long j = perm[i];
    float *r = rec + i * REC;
#pragma unroll
    for (int k = 0; k < na; ++k) {
        r[k] = actions[j * na + k];
        r[na + k] = mu[j * na + k];
        r[2 * na + k] = sigma[j * na + k];
    }
    r[3 * na] = values[j], r[3 * na + 1] = adv[j], r[3 * na + 2] = ret[j], r[3 * na + 3] = logp[j];
    r[3 * na + 4] = 0.0f, r[3 * na + 5] = 0.0f;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// The loss coefficients as the kernels take them by value: hb_ppo_loss_params without its activation field, which picks
// the instantiation of head_fused_kernel instead; a field added to the header struct does not move the kernels' parameters.
struct LossCoefs {
    float clip_param, value_loss_coef, entropy_coef;
    int32_t use_clipped_value_loss, num_actions;
};
inline LossCoefs loss_coefs(const hb_ppo_loss_params &p) {
    return {p.clip_param, p.value_loss_coef, p.entropy_coef, p.use_clipped_value_loss, p.num_actions};
}

// ppo.py:130-168 and its gradient w.r.t. mu, value and std.  One thread per sample.
template <int NA>
__global__ void __launch_bounds__(256)
loss_head_kernel(const float *__restrict__ mu, int ld_mu, const float *__restrict__ value, int ld_v,
                 const float *__restrict__ stdp, const float *__restrict__ rec, long long mb, double inv_b,
                 float ent_scale, LossCoefs lp, float *__restrict__ d_mu, float *__restrict__ d_value,
                 float *__restrict__ d_std, double *__restrict__ stats) {
    __shared__ float s_dstd[8][NA];
    __shared__ double s_stat[8][4];
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float sig[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) sig[j] = stdp[j];
    float g_std[NA];
#pragma unroll
    for (int j = 0; j < NA; ++j) g_std[j] = 0.0f;
    double st_s = 0.0, st_v = 0.0, st_k = 0.0, st_e = 0.0;
    if (i < mb) {
        const float *r = rec + i * (3 * NA + 6);
        const float *m = mu + i * ld_mu;
        float lp_new = 0.0f, kl = 0.0f, ent = 0.0f, diff[NA];
#pragma unroll
        for (int j = 0; j < NA; ++j) {
            const float var = sig[j] * sig[j];
            diff[j] = r[j] - m[j];
            lp_new += (-(diff[j] * diff[j]) / (2.0f * var) - logf(sig[j])) - HALF_LOG_2PI;      // Normal.log_prob
            const float so = r[2 * NA + j], dm = r[NA + j] - m[j];
            kl += (logf(sig[j] / so + 1.e-5f) + (so * so + dm * dm) / (2.0f * var)) - 0.5f;      // ppo.py:138-139
            ent += (0.5f + HALF_LOG_2PI) + logf(sig[j]);                                          // Normal.entropy
        }
        const float v_old = r[3 * NA], adv = r[3 * NA + 1], ret = r[3 * NA + 2], lp_old = r[3 * NA + 3];
        // clipped surrogate (ppo.py:152-156); torch.max splits the gradient evenly on ties
        const float ratio = expf(lp_new - lp_old);
        const float lo = 1.0f - lp.clip_param, hi = 1.0f + lp.clip_param;
        const float s1 = -adv * ratio, s2 = -adv * fminf(fmaxf(ratio, lo), hi);
        const float inr = (ratio >= lo && ratio <= hi) ? 1.0f : 0.0f;
        const float w1 = s1 > s2 ? 1.0f : (s1 == s2 ? 0.5f : 0.0f);
        const float g_ratio = -adv * (w1 + (1.0f - w1) * inr);
        const float g_lp = (float)((double)(g_ratio * ratio) * inv_b);
        st_s = (double)fmaxf(s1, s2);
        // value loss (ppo.py:158-166)
        const float v = value[i * ld_v];
        float g_v;
        if (lp.use_clipped_value_loss) {
            const float dv = v - v_old;
            const float vc = v_old + fminf(fmaxf(dv, -lp.clip_param), lp.clip_param);
            const float l1 = (v - ret) * (v - ret), l2 = (vc - ret) * (vc - ret);
            const float inv = (dv >= -lp.clip_param && dv <= lp.clip_param) ? 1.0f : 0.0f;
            const float u1 = l1 > l2 ? 1.0f : (l1 == l2 ? 0.5f : 0.0f);
            g_v = 2.0f * (v - ret) * u1 + 2.0f * (vc - ret) * inv * (1.0f - u1);
            st_v = (double)fmaxf(l1, l2);
        } else {
            g_v = -2.0f * (ret - v);
            st_v = (double)((ret - v) * (ret - v));
        }
        st_k = (double)kl, st_e = (double)ent;
        float *dm_out = d_mu + i * ld_mu;
#pragma unroll
        for (int j = 0; j < NA; ++j) {
            const float var = sig[j] * sig[j];
            dm_out[j] = g_lp * (diff[j] / var);
            g_std[j] = g_lp * ((diff[j] * diff[j]) / (var * sig[j]) - 1.0f / sig[j]);
        }
        for (int j = NA; j < ld_mu; ++j) dm_out[j] = 0.0f;
        float *dv_out = d_value + i * ld_v;
        dv_out[0] = (float)((double)(lp.value_loss_coef * g_v) * inv_b);
        for (int j = 1; j < ld_v; ++j) dv_out[j] = 0.0f;
    }
#pragma unroll
    for (int j = 0; j < NA; ++j) {
        const float s = warp_sum(g_std[j]);
        if (lane == 0) s_dstd[warp][j] = s;
    }
    st_s = warp_sum(st_s), st_v = warp_sum(st_v), st_k = warp_sum(st_k), st_e = warp_sum(st_e);
    if (lane == 0) s_stat[warp][0] = st_s, s_stat[warp][1] = st_v, s_stat[warp][2] = st_k, s_stat[warp][3] = st_e;
    __syncthreads();
    if (threadIdx.x < NA) {
        float s = 0.0f;
        for (int w = 0; w < 8; ++w) s += s_dstd[w][threadIdx.x];
        // entropy bonus: -entropy_coef * mean(entropy) -> d/dsigma_j = -coef / sigma_j (added once, by block 0)
        // (ent_scale = local / global minibatch size, so that the sum over ranks counts it once)
        if (blockIdx.x == 0) s += ent_scale * (-lp.entropy_coef / sig[threadIdx.x]);
        atomicAdd(d_std + threadIdx.x, s);
    } else if (threadIdx.x >= 32 && threadIdx.x < 36) {
        const int k = threadIdx.x - 32;
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += s_stat[w][k];
        atomicAdd(stats + k, s);
    }
}

// The same loss head for any count up to MAX_ACTIONS (lp.num_actions).  The three per-action arrays of the template
// above would take 3 x 64 registers a thread at 64 actions, so nothing is kept per action here: sigma sits in shared
// memory, the second pass re-reads the record and mu for (action - mu), and each action's std gradient is summed over
// the warp as soon as it is formed.  Same arithmetic, summed over the actions in the same order.
template <>
__global__ void __launch_bounds__(256)
loss_head_kernel<NA_RUNTIME>(const float *__restrict__ mu, int ld_mu, const float *__restrict__ value, int ld_v,
                             const float *__restrict__ stdp, const float *__restrict__ rec, long long mb, double inv_b,
                             float ent_scale, LossCoefs lp, float *__restrict__ d_mu, float *__restrict__ d_value,
                             float *__restrict__ d_std, double *__restrict__ stats) {
    __shared__ float s_sig[MAX_ACTIONS];
    __shared__ float s_dstd[8][MAX_ACTIONS];
    __shared__ double s_stat[8][4];
    const int na = lp.num_actions;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < na) s_sig[threadIdx.x] = stdp[threadIdx.x];
    __syncthreads();
    const bool live = i < mb;
    const float *r = rec + i * (3 * na + 6);
    const float *m = mu + i * ld_mu;
    float g_lp = 0.0f;
    double st_s = 0.0, st_v = 0.0, st_k = 0.0, st_e = 0.0;
    if (live) {
        float lp_new = 0.0f, kl = 0.0f, ent = 0.0f;
        for (int j = 0; j < na; ++j) {
            const float sg = s_sig[j], var = sg * sg;
            const float diff = r[j] - m[j];
            lp_new += (-(diff * diff) / (2.0f * var) - logf(sg)) - HALF_LOG_2PI;                    // Normal.log_prob
            const float so = r[2 * na + j], dm = r[na + j] - m[j];
            kl += (logf(sg / so + 1.e-5f) + (so * so + dm * dm) / (2.0f * var)) - 0.5f;            // ppo.py:138-139
            ent += (0.5f + HALF_LOG_2PI) + logf(sg);                                                // Normal.entropy
        }
        const float v_old = r[3 * na], adv = r[3 * na + 1], ret = r[3 * na + 2], lp_old = r[3 * na + 3];
        // clipped surrogate (ppo.py:152-156); torch.max splits the gradient evenly on ties
        const float ratio = expf(lp_new - lp_old);
        const float lo = 1.0f - lp.clip_param, hi = 1.0f + lp.clip_param;
        const float s1 = -adv * ratio, s2 = -adv * fminf(fmaxf(ratio, lo), hi);
        const float inr = (ratio >= lo && ratio <= hi) ? 1.0f : 0.0f;
        const float w1 = s1 > s2 ? 1.0f : (s1 == s2 ? 0.5f : 0.0f);
        const float g_ratio = -adv * (w1 + (1.0f - w1) * inr);
        g_lp = (float)((double)(g_ratio * ratio) * inv_b);
        st_s = (double)fmaxf(s1, s2);
        // value loss (ppo.py:158-166)
        const float v = value[i * ld_v];
        float g_v;
        if (lp.use_clipped_value_loss) {
            const float dv = v - v_old;
            const float vc = v_old + fminf(fmaxf(dv, -lp.clip_param), lp.clip_param);
            const float l1 = (v - ret) * (v - ret), l2 = (vc - ret) * (vc - ret);
            const float inv = (dv >= -lp.clip_param && dv <= lp.clip_param) ? 1.0f : 0.0f;
            const float u1 = l1 > l2 ? 1.0f : (l1 == l2 ? 0.5f : 0.0f);
            g_v = 2.0f * (v - ret) * u1 + 2.0f * (vc - ret) * inv * (1.0f - u1);
            st_v = (double)fmaxf(l1, l2);
        } else {
            g_v = -2.0f * (ret - v);
            st_v = (double)((ret - v) * (ret - v));
        }
        st_k = (double)kl, st_e = (double)ent;
        float *dv_out = d_value + i * ld_v;
        dv_out[0] = (float)((double)(lp.value_loss_coef * g_v) * inv_b);
        for (int j = 1; j < ld_v; ++j) dv_out[j] = 0.0f;
    }
    float *dm_out = d_mu + i * ld_mu;
    for (int j = 0; j < na; ++j) {                  // every lane takes part in the warp sums, rows past mb with 0
        float g_std = 0.0f;
        if (live) {
            const float sg = s_sig[j], var = sg * sg;
            const float diff = r[j] - m[j];
            dm_out[j] = g_lp * (diff / var);
            g_std = g_lp * ((diff * diff) / (var * sg) - 1.0f / sg);
        }
        g_std = warp_sum(g_std);
        if (lane == 0) s_dstd[warp][j] = g_std;
    }
    if (live)
        for (int j = na; j < ld_mu; ++j) dm_out[j] = 0.0f;
    st_s = warp_sum(st_s), st_v = warp_sum(st_v), st_k = warp_sum(st_k), st_e = warp_sum(st_e);
    if (lane == 0) s_stat[warp][0] = st_s, s_stat[warp][1] = st_v, s_stat[warp][2] = st_k, s_stat[warp][3] = st_e;
    __syncthreads();
    if (threadIdx.x < na) {
        float s = 0.0f;
        for (int w = 0; w < 8; ++w) s += s_dstd[w][threadIdx.x];
        // entropy bonus, added once by block 0 (see loss_head_kernel)
        if (blockIdx.x == 0) s += ent_scale * (-lp.entropy_coef / s_sig[threadIdx.x]);
        atomicAdd(d_std + threadIdx.x, s);
    } else if (threadIdx.x >= MAX_ACTIONS && threadIdx.x < MAX_ACTIONS + 4) {
        const int k = threadIdx.x - MAX_ACTIONS;
        double s = 0.0;
        for (int w = 0; w < 8; ++w) s += s_stat[w][k];
        atomicAdd(stats + k, s);
    }
}

// ------------------------------------------------------------------------------------------------------------
// Fused output layers + loss head (update path).  The last nn.Linear of both MLPs is 128 -> 10 / 128 -> 1:
// 1 290 + 129 MACs per sample, far too thin for a 128-row tensor-core tile, and it sits between the last hidden
// activations and the loss.  One pass over the minibatch does, per sample (one warp per row, lane = 4 features):
//   mu = H3a W4a^T + b, v = H3c W4c^T + b          actor_critic.py:62,74 (fp32 FMAs, not TF32)
//   loss head and its gradient (ppo.py:130-168)     same arithmetic as loss_head_kernel
//   dz3 = (d_out W4) * f'(H3)                       data gradient into the last hidden layer (f: ACT, hb_activation)
//   G4 += d_out^T [H3 | 1]                          weight + bias gradients, reduced per CTA, then atomics
// so H3 is read once and mu / value / d_out never touch HBM.
// ------------------------------------------------------------------------------------------------------------
constexpr int HID = 128;                 // last hidden width of both networks (hector_config.py:207-210)
constexpr int HEAD_THREADS = 384;       // 12 warps x 168 registers = one CTA per SM: a third of the per-CTA gradient atomics of 3 x 128

// Sum 16 per-lane values over the warp with 16 shuffles instead of 80: every exchange halves the number of
// values a lane carries (butterfly over lane bits 4..1), the last one adds lane bit 0.  Value i ends up, fully
// summed, on lanes 2i and 2i + 1.
__device__ __forceinline__ float warp_reduce16(float (&v)[16], int lane) {
#pragma unroll
    for (int step = 0; step < 4; ++step) {
        const int off = 16 >> step, half = 8 >> step;           // lane distance, values kept
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (k < half) {
                const float send = upper ? v[k] : v[k + half];   // the half this lane gives away
                const float recv = __shfl_xor_sync(0xffffffffu, send, off);
                v[k] = (upper ? v[k + half] : v[k]) + recv;
            }
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

template <int NA, int ACT>
__global__ void __launch_bounds__(HEAD_THREADS, 1)
head_fused_kernel(const float *__restrict__ h3a, int ld_ha, const float *__restrict__ h3c, int ld_hc,
                  const float *__restrict__ w4a, const float *__restrict__ w4c, int ld_w, const float *__restrict__ stdp,
                  const float *__restrict__ rec, long long mb, double inv_b, float ent_scale, LossCoefs lp,
                  float *__restrict__ dz3a, float *__restrict__ dz3c, int ld_dz, float *__restrict__ g4a,
                  float *__restrict__ g4c, float *__restrict__ d_std, double *__restrict__ stats) {
    constexpr int NB = NA != NA_RUNTIME ? NA : MAX_FUSED_ACTIONS;     // bound of the per-action arrays and loops
    static_assert(NB + 1 <= 16, "the 16-value butterfly holds at most 15 actions and the value");
    const int na = NA != NA_RUNTIME ? NA : lp.num_actions;         // na action means + 1 value: one lane pair each
    __shared__ __align__(16) float s_w[(NB + 1) * HID];    // output-layer weights, row j = action j, row na = value
    __shared__ float s_g[(NB + 1) * (HID + 1)];            // CTA-level weight/bias gradient accumulators
    __shared__ float s_dstd[NB];
    __shared__ double s_stat[4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < (na + 1) * HID; i += HEAD_THREADS) {
        const int j = i / HID, k = i - j * HID;
        s_w[i] = (j < na) ? w4a[(size_t)j * ld_w + k] : w4c[k];
    }
    for (int i = threadIdx.x; i < (na + 1) * (HID + 1); i += HEAD_THREADS) s_g[i] = 0.0f;
    if (threadIdx.x < na) s_dstd[threadIdx.x] = 0.0f;
    if (threadIdx.x < 4) s_stat[threadIdx.x] = 0.0;
    // After the butterfly, output `o` of a row lives on lanes 2o, 2o+1: lane pair o < na owns action o, pair na the value,
    // and the pairs past it idle.
    const int o = lane >> 1;
    const bool own_action = o < na, even = (lane & 1) == 0;
    const float bias = (o < na) ? w4a[(size_t)o * ld_w + HID] : (o == na ? w4c[HID] : 0.0f);
    // row-invariant pieces of the loss for this lane's action (ppo.py:130-168)
    const float sg = own_action ? stdp[o] : 1.0f;
    const float var = sg * sg, log_sg = logf(sg);
    const float inv_2var = 1.0f / (2.0f * var), inv_var = 1.0f / var, inv_var_sg = 1.0f / (var * sg), inv_sg = 1.0f / sg;
    const float inv_bf = (float)inv_b;
    float ga[NB][4], gc[4], gb = 0.0f, gstd = 0.0f;        // weight grads of this lane's 4 columns; bias / std grad of output o
#pragma unroll
    for (int j = 0; j < NB; ++j) ga[j][0] = ga[j][1] = ga[j][2] = ga[j][3] = 0.0f;
    gc[0] = gc[1] = gc[2] = gc[3] = 0.0f;
    float stf[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    __syncthreads();
    const float4 *w4 = reinterpret_cast<const float4 *>(s_w);

    const long long warps = (long long)gridDim.x * (HEAD_THREADS / 32);
    long long row = (long long)blockIdx.x * (HEAD_THREADS / 32) + warp;
    // software pipeline: the activations and the record of the NEXT row are in flight while this one is processed
    struct RowIn {
        float4 ha, hc;
        float act, mu, sig, v_old, adv, ret, lp_old;
    };
    auto load_row = [&](long long rw) {
        RowIn in;
        in.ha = hb::ld_stream4(reinterpret_cast<const float4 *>(h3a + (size_t)rw * ld_ha) + lane);
        in.hc = hb::ld_stream4(reinterpret_cast<const float4 *>(h3c + (size_t)rw * ld_hc) + lane);
        const float *r = rec + rw * (3 * na + 6);
        in.act = own_action ? __ldg(r + o) : 0.0f, in.mu = own_action ? __ldg(r + na + o) : 0.0f;
        in.sig = own_action ? __ldg(r + 2 * na + o) : 1.0f;
        in.v_old = __ldg(r + 3 * na), in.adv = __ldg(r + 3 * na + 1), in.ret = __ldg(r + 3 * na + 2), in.lp_old = __ldg(r + 3 * na + 3);
        return in;
    };
    RowIn nxt_in = {};
    if (row < mb) nxt_in = load_row(row);
    for (; row < mb; row += warps) {
        const RowIn in = nxt_in;
        if (row + warps < mb) nxt_in = load_row(row + warps);
        const float ha[4] = {in.ha.x, in.ha.y, in.ha.z, in.ha.w}, hc[4] = {in.hc.x, in.hc.y, in.hc.z, in.hc.w};
        const float r_act = in.act, r_mu = in.mu, r_sig = in.sig;
        const float v_old = in.v_old, adv = in.adv, ret = in.ret, lp_old = in.lp_old;
        // ---- output layers: partial dot products over this lane's 4 features, then the 16-shuffle reduction ----
        float part[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (j < na) {
                const float4 w = w4[j * (HID / 4) + lane];
                part[j] = ((ha[0] * w.x + ha[1] * w.y) + ha[2] * w.z) + ha[3] * w.w;
            } else if (j == na) {
                const float4 w = w4[j * (HID / 4) + lane];
                part[j] = ((hc[0] * w.x + hc[1] * w.y) + hc[2] * w.z) + hc[3] * w.w;
            } else {
                part[j] = 0.0f;
            }
        }
        const float out = warp_reduce16(part, lane) + bias;               // mu_o on pair o < na, value on pair na
        const float v = __shfl_sync(0xffffffffu, out, 2 * na);
        // ---- loss head (same arithmetic as loss_head_kernel), the per-action part on the lane pair of the action ----
        const float diff = r_act - out, dm = r_mu - out;
        float lp_j = 0.0f, kl_j = 0.0f, ent_j = 0.0f;
        if (own_action && even) {
            // divisions by the (row-invariant) variance are multiplications by its reciprocal here
            lp_j = (-(diff * diff) * inv_2var - log_sg) - HALF_LOG_2PI;                                      // Normal.log_prob
            kl_j = (logf(sg / r_sig + 1.e-5f) + (r_sig * r_sig + dm * dm) * inv_2var) - 0.5f;               // ppo.py:138-139
            ent_j = (0.5f + HALF_LOG_2PI) + log_sg;                                                           // Normal.entropy
        }
        // sum over the actions in the reference's order (j = 0..na-1) so that the result matches loss_head_kernel; the
        // idle pairs past na (NB > na) add exact zeros
        float lp_new = 0.0f, kl = 0.0f, ent = 0.0f;
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            lp_new += __shfl_sync(0xffffffffu, lp_j, 2 * j);
            kl += __shfl_sync(0xffffffffu, kl_j, 2 * j);
            ent += __shfl_sync(0xffffffffu, ent_j, 2 * j);
        }
        const float ratio = expf(lp_new - lp_old);                 // clipped surrogate (ppo.py:152-156)
        const float lo = 1.0f - lp.clip_param, hi = 1.0f + lp.clip_param;
        const float s1 = -adv * ratio, s2 = -adv * fminf(fmaxf(ratio, lo), hi);
        const float inr = (ratio >= lo && ratio <= hi) ? 1.0f : 0.0f;
        const float w1 = s1 > s2 ? 1.0f : (s1 == s2 ? 0.5f : 0.0f);       // torch.max splits the gradient evenly on ties
        const float g_ratio = -adv * (w1 + (1.0f - w1) * inr);
        const float g_lp = (g_ratio * ratio) * inv_bf;
        float g_v, st_v;
        if (lp.use_clipped_value_loss) {                           // value loss (ppo.py:158-166)
            const float dv = v - v_old;
            const float vc = v_old + fminf(fmaxf(dv, -lp.clip_param), lp.clip_param);
            const float l1 = (v - ret) * (v - ret), l2 = (vc - ret) * (vc - ret);
            const float inv = (dv >= -lp.clip_param && dv <= lp.clip_param) ? 1.0f : 0.0f;
            const float u1 = l1 > l2 ? 1.0f : (l1 == l2 ? 0.5f : 0.0f);
            g_v = 2.0f * (v - ret) * u1 + 2.0f * (vc - ret) * inv * (1.0f - u1);
            st_v = fmaxf(l1, l2);
        } else {
            g_v = -2.0f * (ret - v);
            st_v = (ret - v) * (ret - v);
        }
        g_v = (lp.value_loss_coef * g_v) * inv_bf;
        // gradient w.r.t. this lane's output: d_mu_o on the action pairs, d_value on pair na
        const float g_out = own_action ? g_lp * (diff * inv_var) : (o == na ? g_v : 0.0f);
        if (own_action && even) gstd += g_lp * ((diff * diff) * inv_var_sg - inv_sg);
        if (even) gb += g_out;
        stf[0] += fmaxf(s1, s2), stf[1] += st_v, stf[2] += kl, stf[3] += ent;       // a warp sees a few dozen rows: fp32 is enough here
        // ---- data gradient through the last activation (f'(z) from h = f(z)) and weight gradients ----
        float da[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            if (j < na) {
                const float gm = __shfl_sync(0xffffffffu, g_out, 2 * j);
                const float4 w = w4[j * (HID / 4) + lane];
                da[0] += gm * w.x, da[1] += gm * w.y, da[2] += gm * w.z, da[3] += gm * w.w;
#pragma unroll
                for (int i = 0; i < 4; ++i) ga[j][i] += gm * ha[i];
            }
        }
        const float4 wc = w4[na * (HID / 4) + lane];
        const float wcv[4] = {wc.x, wc.y, wc.z, wc.w};
        float dc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            da[i] *= hb::act_grad<ACT>(ha[i]);
            dc[i] = (g_v * wcv[i]) * hb::act_grad<ACT>(hc[i]);
            gc[i] += g_v * hc[i];
        }
        hb::st_stream4(reinterpret_cast<float4 *>(dz3a + (size_t)row * ld_dz) + lane, make_float4(da[0], da[1], da[2], da[3]));
        hb::st_stream4(reinterpret_cast<float4 *>(dz3c + (size_t)row * ld_dz) + lane, make_float4(dc[0], dc[1], dc[2], dc[3]));
    }
    // CTA reduction in shared memory, then one atomic per parameter and CTA
#pragma unroll
    for (int j = 0; j < NB; ++j)
        if (j < na)
#pragma unroll
            for (int i = 0; i < 4; ++i) atomicAdd(&s_g[j * (HID + 1) + lane * 4 + i], ga[j][i]);
#pragma unroll
    for (int i = 0; i < 4; ++i) atomicAdd(&s_g[na * (HID + 1) + lane * 4 + i], gc[i]);
    if (even && o <= na) atomicAdd(&s_g[o * (HID + 1) + HID], gb);
    if (even && own_action) atomicAdd(&s_dstd[o], gstd);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) atomicAdd(&s_stat[k], (double)stf[k]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (na + 1) * (HID + 1); i += HEAD_THREADS) {
        const int j = i / (HID + 1), k = i - j * (HID + 1);
        float *dst = (j < na) ? g4a + (size_t)j * ld_w + k : g4c + k;
        atomicAdd(dst, s_g[i]);
    }
    if (threadIdx.x < na) {
        float sacc = s_dstd[threadIdx.x];
        // entropy bonus: -entropy_coef * mean(entropy) -> d/dsigma_j = -coef / sigma_j (added once, by block 0)
        if (blockIdx.x == 0) sacc += ent_scale * (-lp.entropy_coef / stdp[threadIdx.x]);
        atomicAdd(d_std + threadIdx.x, sacc);
    } else if (threadIdx.x >= 32 && threadIdx.x < 36) {
        atomicAdd(stats + (threadIdx.x - 32), s_stat[threadIdx.x - 32]);
    }
}

// ------------------------------------------------------------------------------------------------------------
// Rollout side (SURVEY.md §8f rank 1): PPO.act's output layers + sampling head in one launch, writing straight into
// the rollout-storage slot of this step (ppo.py:91-101, actor_critic.py:111-120, rollout_storage.py:87-100), and
// PPO.process_env_step's reward bootstrap + record (ppo.py:103-113).  One warp per env, same lane mapping as
// head_fused_kernel (lane = 4 hidden features; output o lands on lanes 2o, 2o+1).
// ------------------------------------------------------------------------------------------------------------
template <int NA>
__global__ void __launch_bounds__(256)
act_fused_kernel(const float *__restrict__ h3a, int ld_ha, const float *__restrict__ h3c, int ld_hc,
                 const float *__restrict__ w4a, const float *__restrict__ w4c, int ld_w, const float *__restrict__ stdp,
                 const float *__restrict__ eps, long long n, float *__restrict__ actions, float *__restrict__ logp,
                 float *__restrict__ mu_out, float *__restrict__ sigma_out, float *__restrict__ values, int num_actions) {
    constexpr int NB = NA != NA_RUNTIME ? NA : MAX_FUSED_ACTIONS;
    static_assert(NB + 1 <= 16, "the 16-value butterfly holds at most 15 actions and the value");
    const int na = NA != NA_RUNTIME ? NA : num_actions;
    __shared__ __align__(16) float s_w[(NB + 1) * HID];
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < (na + 1) * HID; i += blockDim.x) {
        const int j = i / HID, k = i - j * HID;
        s_w[i] = (j < na) ? w4a[(size_t)j * ld_w + k] : w4c[k];
    }
    const int o = lane >> 1;
    const bool own_action = o < na;
    const float bias = (o < na) ? w4a[(size_t)o * ld_w + HID] : (o == na ? w4c[HID] : 0.0f);
    const float sg = own_action ? stdp[o] : 1.0f;
    __syncthreads();
    const float4 *w4 = reinterpret_cast<const float4 *>(s_w);
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n; row += warps) {
        const float4 ha = hb::ld_stream4(reinterpret_cast<const float4 *>(h3a + (size_t)row * ld_ha) + lane);
        const float4 hc = hb::ld_stream4(reinterpret_cast<const float4 *>(h3c + (size_t)row * ld_hc) + lane);
        const float e = own_action ? __ldg(eps + row * na + o) : 0.0f;
        float part[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (j < na) {
                const float4 w = w4[j * (HID / 4) + lane];
                part[j] = ((ha.x * w.x + ha.y * w.y) + ha.z * w.z) + ha.w * w.w;
            } else if (j == na) {
                const float4 w = w4[j * (HID / 4) + lane];
                part[j] = ((hc.x * w.x + hc.y * w.y) + hc.z * w.z) + hc.w * w.w;
            } else {
                part[j] = 0.0f;
            }
        }
        const float out = warp_reduce16(part, lane) + bias;
        const float sgm = out * 0.0f + sg;                              // actor_critic.py:113
        const float act = out + sgm * e;                                // Normal.sample with the draw supplied
        const float d = act - out;
        const float lp_j = own_action ? (-(d * d) / (2.0f * (sgm * sgm)) - logf(sgm)) - HALF_LOG_2PI : 0.0f;
        float lp = 0.0f;
#pragma unroll
        for (int j = 0; j < NB; ++j) lp += __shfl_sync(0xffffffffu, lp_j, 2 * j);      // pairs past na add exact zeros
        if ((lane & 1) == 0) {
            if (own_action) {
                actions[row * na + o] = act, mu_out[row * na + o] = out, sigma_out[row * na + o] = sgm;
            } else if (o == na) {
                values[row] = out;
            }
        }
        if (lane == 0) logp[row] = lp;
    }
}

// rewards_out = rewards + gamma * (values * time_outs)  (ppo.py:106-108; plain copy without time_outs); dones -> uint8
__global__ void __launch_bounds__(256)
record_step_kernel(const float *__restrict__ rewards, const uint8_t *__restrict__ dones, const float *__restrict__ values,
                   const uint8_t *__restrict__ time_outs, float gamma, long long n, float *__restrict__ rewards_out,
                   uint8_t *__restrict__ dones_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float r = rewards[i];
    // separate roundings, like the reference's three torch ops (this unit is compiled with FMA contraction on)
    if (time_outs) r = __fadd_rn(r, __fmul_rn(gamma, __fmul_rn(values[i], time_outs[i] ? 1.0f : 0.0f)));
    rewards_out[i] = r;
    dones_out[i] = dones[i] ? 1 : 0;
}

template <int NA>
__global__ void __launch_bounds__(256)
act_head_kernel(const float *__restrict__ mu, int ld_mu, const float *__restrict__ stdp, const float *__restrict__ eps,
                long long n, float *__restrict__ actions, float *__restrict__ logp, float *__restrict__ mu_out,
                float *__restrict__ sigma_out, int num_actions) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int na = NA != NA_RUNTIME ? NA : num_actions;
    float lp = 0.0f;
#pragma unroll
    for (int j = 0; j < na; ++j) {
        const float m = mu[i * ld_mu + j];
        const float s = m * 0.0f + stdp[j];                         // actor_critic.py:113
        const float a = m + s * eps[i * na + j];                    // Normal.sample with the draw supplied
        const float d = a - m;
        lp += (-(d * d) / (2.0f * (s * s)) - logf(s)) - HALF_LOG_2PI;
        actions[i * na + j] = a, mu_out[i * na + j] = m, sigma_out[i * na + j] = s;
    }
    logp[i] = lp;
}

// ------------------------------------------------------------------------------------------------------------
// clip_grad_norm_ + torch.optim.Adam.step (single-tensor semantics, no amsgrad / weight decay) + optimizer.zero_grad +
// the adaptive-KL learning-rate rule (ppo.py:136-148,171-174) + update()'s running loss sums (:176-178) in ONE launch.
// Every scalar of the optimizer (learning rate, Adam's step count, gradient norm, the minibatch's loss sums) lives in
// hb_optim_state in device memory, so the launch takes no per-step host values and a captured minibatch step can be
// replayed for every step of every update.
//   phase 1  each thread loads its gradient vectors ONCE (kept in registers) and the grid reduces their sum of squares;
//   barrier  ticket in hb_optim_state (cooperative launch: all blocks are co-resident);
//   phase 2  every block derives clip coefficient / bias corrections / new learning rate from the same device values,
//            checks in a second time, and applies Adam; the LAST block to check in (everyone has read the old values by
//            then) publishes the new learning rate, folds the loss sums, bumps the step count and re-arms the state.
// ------------------------------------------------------------------------------------------------------------
constexpr int OPT_THREADS = 256;
constexpr int OPT_REGV = 8;          // float4 gradient vectors a thread carries from phase 1 to phase 2

__global__ void __launch_bounds__(OPT_THREADS)
optimizer_step_kernel(float *__restrict__ p, float *__restrict__ g, float *__restrict__ m, float *__restrict__ v, long long n,
                      const hb_adam_params ap, hb_optim_state *__restrict__ st) {
    __shared__ double s_red[OPT_THREADS / 32];
    __shared__ float s_scal[3];                                    // clip scale, step size, sqrt(bias_correction2)
    const long long nvec = n >> 2;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    const float4 *g4 = reinterpret_cast<const float4 *>(g);
    float4 gv[OPT_REGV];
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < OPT_REGV; ++k) {
        const long long i = tid + k * stride;
        gv[k] = (i < nvec) ? g4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        acc += ((double)gv[k].x * gv[k].x + (double)gv[k].y * gv[k].y) + ((double)gv[k].z * gv[k].z + (double)gv[k].w * gv[k].w);
    }
    for (long long i = tid + OPT_REGV * stride; i < nvec; i += stride) {           // larger buffers: re-read in phase 2
        const float4 x = g4[i];
        acc += ((double)x.x * x.x + (double)x.y * x.y) + ((double)x.z * x.z + (double)x.w * x.w);
    }
    if (tid == 0)
        for (long long i = nvec << 2; i < n; ++i) acc += (double)g[i] * g[i];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
    __syncthreads();
    unsigned long long *ticket = reinterpret_cast<unsigned long long *>(&st->ticket);
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < OPT_THREADS / 32; ++w) t += s_red[w];
        atomicAdd(&st->grad_sumsq, t);
        __threadfence();
        atomicAdd(ticket, 1ull);
        while (hb::ld_acquire_u64(ticket) < (unsigned long long)gridDim.x) { }  // ---- grid barrier ----
        const volatile hb_optim_state *sv = st;
        double lr = sv->lr;
        const double kl = sv->stats[2] / (double)ap.kl_count;
        if (ap.adaptive) {                                          // ppo.py:140-148
            if (kl > ap.desired_kl * 2.0) lr = fmax(1e-5, lr / 1.5);
            else if (kl < ap.desired_kl / 2.0 && kl > 0.0) lr = fmin(1e-2, lr * 1.5);
        }
        float scale = 1.0f;
        if (ap.max_grad_norm > 0.0f) {          // clip_grad_norm_: coef = max_norm / (total_norm + 1e-6), clamped to 1
            const float total = (float)sqrt(sv->grad_sumsq);
            const float coef = ap.max_grad_norm / (total + 1e-6f);
            scale = coef < 1.0f ? coef : 1.0f;
        }
        const long long t_adam = sv->step + 1;
        const double bc1 = 1.0 - pow(ap.beta1, (double)t_adam), bc2 = 1.0 - pow(ap.beta2, (double)t_adam);
        s_scal[0] = scale, s_scal[1] = (float)(lr / bc1), s_scal[2] = (float)sqrt(bc2);
        __threadfence();
        const unsigned long long arrived = atomicAdd(ticket, 1ull);
        if (arrived == 2ull * gridDim.x - 1ull) {                   // every block has read the old state: publish the new one
            const long long idx = st->steps_in_update;
            if (idx >= 0 && idx < HB_OPT_TRACE_MAX) st->trace[2 * idx] = kl, st->trace[2 * idx + 1] = lr;
            st->steps_in_update = idx + 1;
            st->lr = lr;
#pragma unroll
            for (int k = 0; k < 4; ++k) st->loss_acc[k] += st->stats[k], st->stats[k] = 0.0;
            st->grad_sumsq = 0.0;
            st->step = t_adam;
            __threadfence();
            *ticket = 0ull;
        }
    }
    __syncthreads();
    const float scale = s_scal[0], step_size = s_scal[1], bc2_sqrt = s_scal[2];
    const float w1 = (float)(1.0 - ap.beta1), b2 = (float)ap.beta2, w2 = (float)(1.0 - ap.beta2), eps = (float)ap.eps;
    auto update = [&](float &pi, float gi, float &mi, float &vi) {
        gi = gi * scale;
        mi = mi + (gi - mi) * w1;                                   // exp_avg.lerp_(grad, 1 - beta1)
        vi = vi * b2 + w2 * (gi * gi);                              // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        pi = pi - step_size * (mi / denom);                         // param.addcdiv_(exp_avg, denom, value=-step_size)
    };
    auto update4 = [&](long long i, const float4 &gq) {
        float4 p4 = *reinterpret_cast<float4 *>(p + 4 * i), m4 = *reinterpret_cast<float4 *>(m + 4 * i);
        float4 v4 = *reinterpret_cast<float4 *>(v + 4 * i);
        update(p4.x, gq.x, m4.x, v4.x), update(p4.y, gq.y, m4.y, v4.y);
        update(p4.z, gq.z, m4.z, v4.z), update(p4.w, gq.w, m4.w, v4.w);
        *reinterpret_cast<float4 *>(p + 4 * i) = p4, *reinterpret_cast<float4 *>(m + 4 * i) = m4;
        *reinterpret_cast<float4 *>(v + 4 * i) = v4;
        *reinterpret_cast<float4 *>(g + 4 * i) = make_float4(0.f, 0.f, 0.f, 0.f);      // optimizer.zero_grad()
    };
#pragma unroll
    for (int k = 0; k < OPT_REGV; ++k) {
        const long long i = tid + k * stride;
        if (i < nvec) update4(i, gv[k]);
    }
    for (long long i = tid + OPT_REGV * stride; i < nvec; i += stride) update4(i, g4[i]);
    if (tid == 0)
        for (long long i = nvec << 2; i < n; ++i) {
            update(p[i], g[i], m[i], v[i]);
            g[i] = 0.0f;
        }
}

// ------------------------------------------------------------------------------------------------------------
// Data-parallel optimizer step over peer memory (SURVEY.md §8e): ONE kernel per rank replaces the gradient all-reduce
// (NCCL), clip_grad_norm_, Adam and the parameter broadcast.  Every rank's flat gradient and parameter buffers are
// mapped into every other rank's address space (NVLink / NVSwitch peer access; the host passes the pointers):
//   start barrier (flags)    every rank's backward has finished
//   phase A                  rank r reads ITS 1/G slice of the flat gradient from all G ranks (peer loads, or one
//                            multimem.ld_reduce per vector when the NVSwitch multicast address is given), sums them in
//                            registers and reduces the slice's sum of squares over the grid
//   mailbox exchange         slice norms and the minibatch's loss sums go to every peer (5 doubles), flag barrier: every
//                            rank now derives the same clip coefficient, KL mean and learning rate
//   phase B                  Adam on the slice (optimizer state is sharded: a rank only ever touches its slice of m, v),
//                            the new parameters are stored into ALL ranks' parameter buffers (peer stores / multimem.st);
//                            the rank's own gradient buffer is zeroed
//   end barrier              all slices have landed in this rank's parameters before the next forward pass reads them
// NVLink traffic per rank and step: (G-1)/G of the gradient in, (G-1)/G of the parameters out (2 x 5.3 MB at G = 8)
// instead of NCCL's ring / tree passes over the whole buffer, and no SM hand-over between NCCL and the GEMMs.
// Spin loops give up after ~2 s and set state->reserved (a rank that never arrives must not hang the GPU).
// ------------------------------------------------------------------------------------------------------------
constexpr int DP_THREADS = 256;
constexpr int DP_REGV = 8;
constexpr int DP_MAIL = 8;           // doubles per sender in a mailbox

__device__ __forceinline__ void st_release_sys_u32(uint32_t *p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 multimem_ld_reduce4(const float *mc) {
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(mc)
                 : "memory");
    return v;
}
__device__ __forceinline__ void multimem_st4(float *mc, const float4 &v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// bounded spin: false on time-out
template <typename Pred>
__device__ __forceinline__ bool spin_until(Pred done) {
    const long long t0 = clock64();
    while (!done()) {
        if (clock64() - t0 > 4000000000ll) return false;       // ~2 s at 2 GHz
    }
    return true;
}

// cross-rank barrier by the first `world` threads of one block: tell every peer, wait for every peer
__device__ __forceinline__ bool rank_barrier(const hb_dp_comm &c, int phase, uint32_t epoch) {
    bool ok = true;
    if ((int)threadIdx.x < c.world) {
        const int peer = threadIdx.x;
        st_release_sys_u32(c.flag[peer] + phase * HB_DP_MAX_RANKS + c.rank, epoch);
        const uint32_t *mine = c.flag[c.rank] + phase * HB_DP_MAX_RANKS + peer;
        ok = spin_until([&] { return ld_acquire_sys_u32(mine) >= epoch; });
    }
    return __syncthreads_and(ok);
}

__global__ void __launch_bounds__(DP_THREADS)
dp_optimizer_step_kernel(const __grid_constant__ hb_dp_comm c, float *__restrict__ m, float *__restrict__ v, long long n,
                         const hb_adam_params ap, hb_optim_state *__restrict__ st) {
    __shared__ double s_red[DP_THREADS / 32];
    __shared__ float s_scal[3];
    __shared__ int s_flag;
    const int W = c.world, R = c.rank;
    const long long nvec = n >> 2;
    const long long per = (nvec + W - 1) / W, lo = (long long)R * per, hi = lo + per < nvec ? lo + per : nvec;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    unsigned long long *ticket = reinterpret_cast<unsigned long long *>(&st->ticket);
    unsigned long long *go = reinterpret_cast<unsigned long long *>(&st->go);
    const uint32_t epoch = (uint32_t)(st->step + 1);                // identical on every rank, advances every step
    float *g_own = c.grad[R], *p_own = c.param[R];

    // ---- start barrier: block 0 meets the peers, then opens the local gate ----
    if (blockIdx.x == 0) {
        const bool ok = rank_barrier(c, 0, epoch);
        if (threadIdx.x == 0) {
            if (!ok) st->reserved = 1;
            __threadfence();
            atomicExch(go, 3ull * epoch + 1ull);
        }
    }
    if (threadIdx.x == 0) {
        const bool ok = spin_until([&] { return hb::ld_acquire_u64(go) >= 3ull * epoch + 1ull; });
        if (!ok) st->reserved = 2;
    }
    __syncthreads();

    // ---- phase A: reduce this rank's slice of the gradient over all ranks ----
    float4 gv[DP_REGV];
    double acc = 0.0;
    auto reduce_vec = [&](long long i) {
        if (c.grad_mc) return multimem_ld_reduce4(c.grad_mc + 4 * i);
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int p = 0; p < W; ++p) {
            const float4 x = *reinterpret_cast<const float4 *>(c.grad[p] + 4 * i);
            s.x += x.x, s.y += x.y, s.z += x.z, s.w += x.w;
        }
        return s;
    };
#pragma unroll
    for (int k = 0; k < DP_REGV; ++k) {
        const long long i = lo + tid + k * stride;
        gv[k] = (i < hi) ? reduce_vec(i) : make_float4(0.f, 0.f, 0.f, 0.f);
        acc += ((double)gv[k].x * gv[k].x + (double)gv[k].y * gv[k].y) + ((double)gv[k].z * gv[k].z + (double)gv[k].w * gv[k].w);
    }
    // longer slices: the sums are parked in this rank's OWN gradient buffer - no other rank reads that range (every rank
    // reads only its own slice of everybody's buffer), and each element is read before it is overwritten by the same thread
    for (long long i = lo + tid + DP_REGV * stride; i < hi; i += stride) {
        const float4 x = reduce_vec(i);
        acc += ((double)x.x * x.x + (double)x.y * x.y) + ((double)x.z * x.z + (double)x.w * x.w);
        *reinterpret_cast<float4 *>(g_own + 4 * i) = x;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < DP_THREADS / 32; ++w) t += s_red[w];
        atomicAdd(&st->grad_sumsq, t);
        __threadfence();
        s_flag = (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull);
    }
    __syncthreads();
    // ---- mailbox exchange by the last block of this rank ----
    if (s_flag) {
        if ((int)threadIdx.x < W) {
            double *box = c.mail[threadIdx.x] + (size_t)R * DP_MAIL;           // my row in the peer's mailbox
            const volatile hb_optim_state *sv = st;
            box[0] = sv->grad_sumsq;
#pragma unroll
            for (int k = 0; k < 4; ++k) box[1 + k] = sv->stats[k];
            __threadfence_system();
        }
        __syncthreads();
        const bool ok = rank_barrier(c, 1, epoch);
        if (threadIdx.x == 0) {
            if (!ok) st->reserved = 3;
            double sumsq = 0.0, tot[4] = {0.0, 0.0, 0.0, 0.0};
            const volatile double *mine = c.mail[R];
            for (int p = 0; p < W; ++p) {
                sumsq += mine[p * DP_MAIL];
#pragma unroll
                for (int k = 0; k < 4; ++k) tot[k] += mine[p * DP_MAIL + 1 + k];
            }
            double lr = st->lr;
            const double kl = tot[2] / (double)ap.kl_count;
            if (ap.adaptive) {
                if (kl > ap.desired_kl * 2.0) lr = fmax(1e-5, lr / 1.5);
                else if (kl < ap.desired_kl / 2.0 && kl > 0.0) lr = fmin(1e-2, lr * 1.5);
            }
            float scale = 1.0f;
            if (ap.max_grad_norm > 0.0f) {
                const float total = (float)sqrt(sumsq);
                const float coef = ap.max_grad_norm / (total + 1e-6f);
                scale = coef < 1.0f ? coef : 1.0f;
            }
            const long long t_adam = st->step + 1;
            const double bc1 = 1.0 - pow(ap.beta1, (double)t_adam), bc2 = 1.0 - pow(ap.beta2, (double)t_adam);
            st->bcast[0] = scale, st->bcast[1] = (float)(lr / bc1), st->bcast[2] = (float)sqrt(bc2);
            // the step's bookkeeping (same totals on every rank)
            const long long idx = st->steps_in_update;
            if (idx >= 0 && idx < HB_OPT_TRACE_MAX) st->trace[2 * idx] = kl, st->trace[2 * idx + 1] = lr;
            st->steps_in_update = idx + 1;
            st->lr = lr;
#pragma unroll
            for (int k = 0; k < 4; ++k) st->loss_acc[k] += tot[k], st->stats[k] = 0.0;
            st->grad_sumsq = 0.0;
            *ticket = 0ull;
            __threadfence();
            atomicExch(go, 3ull * epoch + 2ull);
        }
    }
    if (threadIdx.x == 0) {
        const bool ok = spin_until([&] { return hb::ld_acquire_u64(go) >= 3ull * epoch + 2ull; });
        if (!ok) st->reserved = 4;
        const volatile float *bc = st->bcast;
        s_scal[0] = bc[0], s_scal[1] = bc[1], s_scal[2] = bc[2];
    }
    __syncthreads();

    // ---- phase B: Adam on the slice, parameters out to every rank, own gradients zeroed ----
    const float scale = s_scal[0], step_size = s_scal[1], bc2_sqrt = s_scal[2];
    const float w1 = (float)(1.0 - ap.beta1), b2 = (float)ap.beta2, w2 = (float)(1.0 - ap.beta2), eps = (float)ap.eps;
    auto update = [&](float &pi, float gi, float &mi, float &vi) {
        gi = gi * scale;
        mi = mi + (gi - mi) * w1;
        vi = vi * b2 + w2 * (gi * gi);
        const float denom = sqrtf(vi) / bc2_sqrt + eps;
        pi = pi - step_size * (mi / denom);
    };
    auto update4 = [&](long long i, const float4 &gq) {
        float4 p4 = *reinterpret_cast<float4 *>(p_own + 4 * i), m4 = *reinterpret_cast<float4 *>(m + 4 * i);
        float4 v4 = *reinterpret_cast<float4 *>(v + 4 * i);
        update(p4.x, gq.x, m4.x, v4.x), update(p4.y, gq.y, m4.y, v4.y);
        update(p4.z, gq.z, m4.z, v4.z), update(p4.w, gq.w, m4.w, v4.w);
        *reinterpret_cast<float4 *>(m + 4 * i) = m4, *reinterpret_cast<float4 *>(v + 4 * i) = v4;
        if (c.param_mc) {
            multimem_st4(c.param_mc + 4 * i, p4);
        } else {
#pragma unroll 4
            for (int p = 0; p < W; ++p) *reinterpret_cast<float4 *>(c.param[p] + 4 * i) = p4;
        }
    };
#pragma unroll
    for (int k = 0; k < DP_REGV; ++k) {
        const long long i = lo + tid + k * stride;
        if (i < hi) update4(i, gv[k]);
    }
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long long i = lo + tid + DP_REGV * stride; i < hi; i += stride) {
        update4(i, *reinterpret_cast<const float4 *>(g_own + 4 * i));
        *reinterpret_cast<float4 *>(g_own + 4 * i) = zero4;
    }
#pragma unroll
    for (int k = 0; k < DP_REGV; ++k) {
        const long long i = lo + tid + k * stride;
        if (i < hi) *reinterpret_cast<float4 *>(g_own + 4 * i) = zero4;
    }
    // every peer has finished reading this rank's gradients (it passed the mailbox barrier): zero the rest of the buffer
    // for the next backward pass (optimizer.zero_grad)
    for (long long i = tid; i < nvec - (hi - lo); i += stride) {
        const long long j = i < lo ? i : i + (hi - lo);
        *reinterpret_cast<float4 *>(g_own + 4 * j) = zero4;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) s_flag = (atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x - 1ull);
    __syncthreads();
    // ---- end barrier: all ranks' slices have landed here before anything reads the parameters ----
    if (s_flag) {
        const bool ok = rank_barrier(c, 2, epoch);
        if (threadIdx.x == 0) {
            if (!ok) st->reserved = 5;
            st->step = st->step + 1;
            __threadfence();
            *ticket = 0ull;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// Runner bookkeeping (on_policy_runner.py:140-154): cur_reward_sum += rewards; cur_episode_length += 1; for the envs that
// finished an episode, IN ASCENDING ENV ORDER, push (sum, length) into the two deque(maxlen=100) buffers and restart the
// running values.  The reference does this with nonzero() + .cpu() twice per step; here it is one small launch and the
// deques are rings in device memory (ring_state[0] = entries ever pushed), read once per iteration by log().
// One block walks the envs in chunks of its size, so that the ring order equals the reference's extend() order.
// ------------------------------------------------------------------------------------------------------------
constexpr int BOOK_THREADS = 1024;

__global__ void __launch_bounds__(BOOK_THREADS)
runner_bookkeeping_kernel(const float *__restrict__ rewards, const uint8_t *__restrict__ dones, long long n,
                          float *__restrict__ cur_reward_sum, float *__restrict__ cur_episode_length, float *__restrict__ ring_rew,
                          float *__restrict__ ring_len, int capacity, long long *__restrict__ ring_state) {
    __shared__ int warp_tot[BOOK_THREADS / 32];
    __shared__ long long base, step_total;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // pass 1: how many episodes end in this step (a deque keeps only the last `capacity` of them: earlier ones must not
    // be written at all, or they would race with the later entry that lands in the same ring slot)
    int mine = 0;
    for (long long e = threadIdx.x; e < n; e += BOOK_THREADS) mine += dones[e] != 0;
    mine = __reduce_add_sync(0xffffffffu, mine);
    if (lane == 0) warp_tot[warp] = mine;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
        for (int w = 0; w < BOOK_THREADS / 32; ++w) t += warp_tot[w];
        step_total = t;
        base = ring_state[0];
    }
    __syncthreads();
    const long long keep_from = base + step_total - capacity;       // global index of the oldest entry that survives
    for (long long e0 = 0; e0 < n; e0 += BOOK_THREADS) {
        const long long e = e0 + threadIdx.x;
        bool done = false;
        float sum = 0.f, len = 0.f;
        if (e < n) {
            sum = cur_reward_sum[e] + rewards[e];
            len = cur_episode_length[e] + 1.0f;
            done = dones[e] != 0;
        }
        const unsigned ballot = __ballot_sync(0xffffffffu, done);
        __syncthreads();
        if (lane == 0) warp_tot[warp] = __popc(ballot);
        __syncthreads();
        int before = __popc(ballot & ((1u << lane) - 1u)), total = 0;
        for (int w = 0; w < BOOK_THREADS / 32; ++w) {
            before += (w < warp) ? warp_tot[w] : 0;
            total += warp_tot[w];
        }
        if (done) {
            const long long idx = base + before;
            if (idx >= keep_from) ring_rew[idx % capacity] = sum, ring_len[idx % capacity] = len;
            sum = 0.f, len = 0.f;
        }
        if (e < n) cur_reward_sum[e] = sum, cur_episode_length[e] = len;
        __syncthreads();
        if (threadIdx.x == 0) base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) ring_state[0] = base;
}

// N(0,1) draws for the action sample of PPO.act (ppo.py:93, Normal.sample()): Philox4x32-10 keyed by state[2], counter =
// (quad index, a domain tag, the call counter), Box-Muller on the four words.  state[0] = call counter, state[1] = ticket,
// state[2] = key - all in device memory: every block reads counter and key first, the last block to finish advances the
// counter, so the launch can sit in a replayed graph, draw fresh numbers every replay and follow a re-seed.
__global__ void __launch_bounds__(256)
draw_normal_kernel(float *__restrict__ out, long long count, unsigned long long *__restrict__ state) {
    const unsigned long long call = *reinterpret_cast<volatile unsigned long long *>(state);
    const unsigned long long key = *reinterpret_cast<volatile unsigned long long *>(state + 2);
    const uint32_t k0 = (uint32_t)key, k1 = (uint32_t)(key >> 32);
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q * 4 < count) {
        const uint4 x = hb::philox4x32_10((uint32_t)q, 0x50504F00u ^ (uint32_t)(q >> 32), (uint32_t)call, (uint32_t)(call >> 32), k0, k1);
        const float scale = 5.9604644775390625e-8f;                 // 2^-24
        const float u0 = (float)((x.x >> 8) + 1u) * scale, u1 = (float)((x.z >> 8) + 1u) * scale;      // (0, 1]
        const float r0 = sqrtf(-2.0f * __logf(u0)), r1 = sqrtf(-2.0f * __logf(u1));
        float s0, c0, s1, c1;
        __sincosf(6.283185307179586f * ((float)(x.y >> 8) * scale), &s0, &c0);
        __sincosf(6.283185307179586f * ((float)(x.w >> 8) * scale), &s1, &c1);
        const float z[4] = {r0 * c0, r0 * s0, r1 * c1, r1 * s1};
        if (q * 4 + 3 < count && (reinterpret_cast<uintptr_t>(out) & 15u) == 0) {
            reinterpret_cast<float4 *>(out)[q] = make_float4(z[0], z[1], z[2], z[3]);
        } else {
            for (int k = 0; k < 4 && q * 4 + k < count; ++k) out[q * 4 + k] = z[k];
        }
    }
    __syncthreads();                                                // the whole block has read the counter
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned long long ticket = atomicAdd(state + 1, 1ull);
        if (ticket == (unsigned long long)gridDim.x - 1ull) {
            state[1] = 0ull;
            *reinterpret_cast<volatile unsigned long long *>(state) = call + 1ull;
        }
    }
}

}  // namespace

extern "C" {

int hb_ppo_gather_rows(const float *src, int32_t ld_src, float *dst, int32_t ld_dst, const int64_t *perm, int64_t rows,
                       int32_t cols, int32_t ones_col, void *stream) {
    HB_REQUIRE(src && dst && perm && rows > 0 && cols > 0, "hb_ppo_gather_rows: bad arguments");
    HB_REQUIRE(hb::aligned16(src) && hb::aligned16(dst) && ld_src % 4 == 0 && ld_dst % 4 == 0,
               "hb_ppo_gather_rows: rows must start on 16-byte boundaries");
    HB_REQUIRE(ones_col < ld_dst, "hb_ppo_gather_rows: ones_col outside the destination row");
    const long long threads = rows * 32;
    gather_rows_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, ld_src, dst, ld_dst, perm,
                                                                                          rows, cols, ones_col);
    HB_CHECK_LAUNCH("gather_rows_kernel");
    return HB_OK;
}

int hb_ppo_pack_samples(const int64_t *perm, int64_t rows, const float *actions, const float *mu, const float *sigma,
                        const float *values, const float *advantages, const float *returns, const float *log_prob,
                        int32_t num_actions, float *records, void *stream) {
    HB_REQUIRE(perm && actions && mu && sigma && values && advantages && returns && log_prob && records && rows > 0,
               "hb_ppo_pack_samples: bad arguments");
    HB_PPO_CHECK_ACTIONS(num_actions, MAX_ACTIONS, "hb_ppo_pack_samples: num_actions = %d (1 to 64)");
    HB_PPO_DISPATCH(num_actions, (pack_samples_kernel<NA><<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        perm, rows, actions, mu, sigma, values, advantages, returns, log_prob, records, num_actions)));
    HB_CHECK_LAUNCH("pack_samples_kernel");
    return HB_OK;
}

int hb_ppo_loss_head(const float *mu, int32_t ld_mu, const float *value, int32_t ld_v, const float *std,
                     const float *records, int64_t mb, int64_t mb_global, const hb_ppo_loss_params *lp, float *d_mu,
                     float *d_value, float *d_std, double *stats, void *stream) {
    HB_REQUIRE(mu && value && std && records && lp && d_mu && d_value && d_std && stats, "hb_ppo_loss_head: null buffer");
    HB_PPO_CHECK_ACTIONS(lp->num_actions, MAX_ACTIONS, "hb_ppo_loss_head: num_actions = %d (1 to 64)");
    HB_REQUIRE(mb > 0 && mb_global >= mb && ld_mu >= lp->num_actions && ld_v >= 1, "hb_ppo_loss_head: bad sizes");
    HB_PPO_DISPATCH(lp->num_actions, (loss_head_kernel<NA><<<(unsigned)((mb + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        mu, ld_mu, value, ld_v, std, records, mb, 1.0 / (double)mb_global, (float)((double)mb / (double)mb_global), loss_coefs(*lp), d_mu,
        d_value, d_std, stats)));
    HB_CHECK_LAUNCH("loss_head_kernel");
    return HB_OK;
}

int hb_ppo_head_fused(const float *h3_actor, int32_t ld_ha, const float *h3_critic, int32_t ld_hc, const float *w4_actor,
                      const float *w4_critic, int32_t ld_w, const float *std, const float *records, int64_t mb,
                      int64_t mb_global, const hb_ppo_loss_params *lp, float *dz3_actor, float *dz3_critic, int32_t ld_dz,
                      float *g4_actor, float *g4_critic, float *d_std, double *stats, void *stream) {
    HB_REQUIRE(h3_actor && h3_critic && w4_actor && w4_critic && std && records && lp && dz3_actor && dz3_critic &&
                   g4_actor && g4_critic && d_std && stats, "hb_ppo_head_fused: null buffer");
    HB_PPO_CHECK_ACTIONS(lp->num_actions, MAX_FUSED_ACTIONS,
                         "hb_ppo_head_fused: num_actions = %d (1 to 15; wider heads use hb_gemm_tf32 + hb_ppo_loss_head)");
    HB_REQUIRE(mb > 0 && mb_global >= mb, "hb_ppo_head_fused: bad sizes");
    HB_REQUIRE(ld_ha >= HID + 1 && ld_hc >= HID + 1 && ld_w >= HID + 1 && ld_dz >= HID && ld_ha % 4 == 0 && ld_hc % 4 == 0 &&
                   ld_w % 4 == 0 && ld_dz % 4 == 0,
               "hb_ppo_head_fused: rows of %d features (+ ones column), leading dimensions multiples of 4", HID);
    HB_REQUIRE(hb::aligned16(h3_actor) && hb::aligned16(h3_critic) && hb::aligned16(w4_actor) && hb::aligned16(w4_critic) &&
                   hb::aligned16(dz3_actor) && hb::aligned16(dz3_critic), "hb_ppo_head_fused: 16-byte aligned buffers");
    long long blocks = (mb + HEAD_THREADS / 32 - 1) / (HEAD_THREADS / 32);
    const long long cap = hb::sm_count();                // one resident CTA per SM (__launch_bounds__)
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    const double inv_b = 1.0 / (double)mb_global;
    const float ent_scale = (float)((double)mb / (double)mb_global);
    const LossCoefs coefs = loss_coefs(*lp);
    HB_PPO_FUSED_DISPATCH(lp->num_actions, HB_ACT_DISPATCH(lp->activation, (head_fused_kernel<NA, ACT><<<grid, HEAD_THREADS, 0,
        (cudaStream_t)stream>>>(h3_actor, ld_ha, h3_critic, ld_hc, w4_actor, w4_critic, ld_w, std, records, mb, inv_b, ent_scale,
        coefs, dz3_actor, dz3_critic, ld_dz, g4_actor, g4_critic, d_std, stats))));
    HB_CHECK_LAUNCH("head_fused_kernel");
    return HB_OK;
}

int hb_ppo_draw_normal(float *out, int64_t count, uint64_t *state, void *stream) {
    HB_REQUIRE(out && state && count > 0, "hb_ppo_draw_normal: bad arguments");
    const long long quads = (count + 3) / 4;
    draw_normal_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        out, (long long)count, reinterpret_cast<unsigned long long *>(state));
    HB_CHECK_LAUNCH("draw_normal_kernel");
    return HB_OK;
}

int hb_ppo_act_head(const float *mu, int32_t ld_mu, const float *std, const float *eps, int64_t n, int32_t num_actions,
                    float *actions, float *log_prob, float *mu_out, float *sigma_out, void *stream) {
    HB_PPO_CHECK_ACTIONS(num_actions, MAX_ACTIONS, "hb_ppo_act_head: num_actions = %d (1 to 64)");
    HB_REQUIRE(mu && std && eps && actions && log_prob && mu_out && sigma_out && n > 0 && ld_mu >= num_actions,
               "hb_ppo_act_head: bad arguments");
    HB_PPO_DISPATCH(num_actions, (act_head_kernel<NA><<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        mu, ld_mu, std, eps, n, actions, log_prob, mu_out, sigma_out, num_actions)));
    HB_CHECK_LAUNCH("act_head_kernel");
    return HB_OK;
}

int hb_ppo_act_fused(const float *h3_actor, int32_t ld_ha, const float *h3_critic, int32_t ld_hc, const float *w4_actor,
                     const float *w4_critic, int32_t ld_w, const float *std, const float *eps, int64_t n, int32_t num_actions,
                     float *actions, float *log_prob, float *mu_out, float *sigma_out, float *values, void *stream) {
    HB_REQUIRE(h3_actor && h3_critic && w4_actor && w4_critic && std && eps && actions && log_prob && mu_out && sigma_out &&
                   values && n > 0, "hb_ppo_act_fused: bad arguments");
    HB_PPO_CHECK_ACTIONS(num_actions, MAX_FUSED_ACTIONS,
                         "hb_ppo_act_fused: num_actions = %d (1 to 15; wider heads use hb_gemm_tf32 + hb_ppo_act_head)");
    HB_REQUIRE(ld_ha >= HID && ld_hc >= HID && ld_w >= HID + 1 && ld_ha % 4 == 0 && ld_hc % 4 == 0 && ld_w % 4 == 0,
               "hb_ppo_act_fused: rows of %d features, leading dimensions multiples of 4", HID);
    HB_REQUIRE(hb::aligned16(h3_actor) && hb::aligned16(h3_critic) && hb::aligned16(w4_actor) && hb::aligned16(w4_critic),
               "hb_ppo_act_fused: 16-byte aligned buffers");
    long long blocks = (n + 7) / 8;
    const long long cap = 8ll * hb::sm_count();
    const unsigned grid = (unsigned)(blocks < cap ? blocks : cap);
    HB_PPO_FUSED_DISPATCH(num_actions, (act_fused_kernel<NA><<<grid, 256, 0, (cudaStream_t)stream>>>(
        h3_actor, ld_ha, h3_critic, ld_hc, w4_actor, w4_critic, ld_w, std, eps, n, actions, log_prob, mu_out, sigma_out, values,
        num_actions)));
    HB_CHECK_LAUNCH("act_fused_kernel");
    return HB_OK;
}

int hb_ppo_record_step(const float *rewards, const uint8_t *dones, const float *values, const uint8_t *time_outs, float gamma,
                       int64_t n, float *rewards_out, uint8_t *dones_out, void *stream) {
    HB_REQUIRE(rewards && dones && rewards_out && dones_out && n > 0 && (!time_outs || values), "hb_ppo_record_step: bad arguments");
    record_step_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rewards, dones, values, time_outs, gamma, n,
                                                                                      rewards_out, dones_out);
    HB_CHECK_LAUNCH("record_step_kernel");
    return HB_OK;
}

int hb_optimizer_step(float *params, float *grads, float *exp_avg, float *exp_avg_sq, int64_t n, const hb_adam_params *ap,
                      hb_optim_state *state, void *stream) {
    HB_REQUIRE(params && grads && exp_avg && exp_avg_sq && ap && state && n > 0, "hb_optimizer_step: bad arguments");
    HB_REQUIRE(!ap->adaptive || ap->kl_count > 0, "hb_optimizer_step: adaptive schedule needs kl_count");
    HB_REQUIRE(hb::aligned16(params) && hb::aligned16(grads) && hb::aligned16(exp_avg) && hb::aligned16(exp_avg_sq) &&
                   (reinterpret_cast<uintptr_t>(state) & 7u) == 0, "hb_optimizer_step: 16-byte aligned buffers");
    // all blocks wait on one another: the grid must be co-resident (cooperative launch), two blocks per SM at most
    const long long want = ((n >> 2) + OPT_THREADS - 1) / OPT_THREADS;
    const long long cap = 2ll * hb::sm_count();
    const unsigned grid = (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
    HB_CUDA(hb::launch_coop(optimizer_step_kernel, dim3(grid), dim3(OPT_THREADS), 0, (cudaStream_t)stream, params, grads, exp_avg,
                            exp_avg_sq, (long long)n, *ap, state));
    HB_CHECK_LAUNCH("optimizer_step_kernel");
    return HB_OK;
}

int hb_runner_bookkeeping(const float *rewards, const uint8_t *dones, int64_t n, float *cur_reward_sum, float *cur_episode_length,
                          float *ring_rewards, float *ring_lengths, int32_t capacity, int64_t *ring_state, void *stream) {
    HB_REQUIRE(rewards && dones && cur_reward_sum && cur_episode_length && ring_rewards && ring_lengths && ring_state && n > 0 &&
                   capacity > 0, "hb_runner_bookkeeping: bad arguments");
    runner_bookkeeping_kernel<<<1, BOOK_THREADS, 0, (cudaStream_t)stream>>>(rewards, dones, (long long)n, cur_reward_sum, cur_episode_length,
                                                                           ring_rewards, ring_lengths, capacity,
                                                                           reinterpret_cast<long long *>(ring_state));
    HB_CHECK_LAUNCH("runner_bookkeeping_kernel");
    return HB_OK;
}

int hb_dp_optimizer_step(const hb_dp_comm *comm, float *exp_avg, float *exp_avg_sq, int64_t n, const hb_adam_params *ap,
                         hb_optim_state *state, void *stream) {
    HB_REQUIRE(comm && exp_avg && exp_avg_sq && ap && state && n > 0 && n % 4 == 0, "hb_dp_optimizer_step: bad arguments (n must be a multiple of 4)");
    HB_REQUIRE(comm->world >= 1 && comm->world <= HB_DP_MAX_RANKS && comm->rank >= 0 && comm->rank < comm->world,
               "hb_dp_optimizer_step: world %d / rank %d out of range", comm->world, comm->rank);
    for (int p = 0; p < comm->world; ++p)
        HB_REQUIRE(comm->grad[p] && comm->param[p] && comm->mail[p] && comm->flag[p] && hb::aligned16(comm->grad[p]) &&
                       hb::aligned16(comm->param[p]), "hb_dp_optimizer_step: peer %d buffers missing or misaligned", p);
    HB_REQUIRE(!ap->adaptive || ap->kl_count > 0, "hb_dp_optimizer_step: adaptive schedule needs kl_count");
    HB_REQUIRE(hb::aligned16(exp_avg) && hb::aligned16(exp_avg_sq), "hb_dp_optimizer_step: 16-byte aligned optimizer state");
    const long long per = ((n >> 2) + comm->world - 1) / comm->world;
    const long long want = (per + DP_THREADS - 1) / DP_THREADS;
    const long long cap = hb::sm_count();                  // blocks wait on one another and on the peers: one per SM, all resident
    const unsigned grid = (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
    HB_CUDA(hb::launch_coop(dp_optimizer_step_kernel, dim3(grid), dim3(DP_THREADS), 0, (cudaStream_t)stream, *comm, exp_avg,
                            exp_avg_sq, (long long)n, *ap, state));
    HB_CHECK_LAUNCH("dp_optimizer_step_kernel");
    return HB_OK;
}

}  // extern "C"
