// GAE (SURVEY.md §8 row a10): RolloutStorage.compute_returns, algo/ppo/rollout_storage.py:122-136.
//
//   delta_t = r_t + (nnt_t*gamma) * V_{t+1} - V_t,  A_t = delta_t + ((nnt_t*gamma)*lam) * A_{t+1},
//   returns_t = A_t + V_t, advantages = (returns - V) normalised by mean / unbiased std over T*N.
//
// Layout [T, N]: time-major, so a (t, 32 envs) row is one 128-byte line.  The recurrence
// A_t = d_t + c_t*A_{t+1} is a first-order linear scan over t: composing the affine maps
// (c, d) is associative, so one warp scans 32 time steps of one env with 5 shuffle rounds.
// A CTA takes a tile of 32 envs: the [T x 32] slab is loaded row by row (coalesced) into
// shared memory, every warp scans envs of the tile (lane = time step, chunks of 32 steps with a
// carry for T > 32), results go back through shared memory and are written row by row.
// Compiled with --fmad=false (same op sequence as the reference within one step).
#include "hb_common.cuh"

namespace {

constexpr int ENVS = 32;       // envs per CTA tile
constexpr int WARPS = 8;

__global__ void __launch_bounds__(WARPS * 32)
gae_scan_kernel(const float *__restrict__ rewards, const float *__restrict__ values,
                const uint8_t *__restrict__ dones, const float *__restrict__ last_values,
                float *__restrict__ returns, float *__restrict__ advantages, double *__restrict__ stats, int T, int N,
                float gamma, float lam) {
    extern __shared__ float sm[];
    // per (t, e): c = nnt*gamma*lam (scan multiplier), d = delta; then overwritten with A_t
    float *sc = sm;                       // [T][ENVS+1]
    float *sd = sm + (size_t)T * (ENVS + 1);
    float *sv = sd + (size_t)T * (ENVS + 1);
    __shared__ double red[2][WARPS];
    hb::pdl_trigger();              // the normalise kernel may be scheduled behind this grid's tail (it waits before reading)
    const int env0 = blockIdx.x * ENVS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int e = env0 + lane;
    const bool ok = e < N;

    // phase 1: coalesced loads; lane = env, warps stride over t.  All of a warp's loads are issued before the first
    // shared-memory store (up to ITERS time steps per warp), so a tile pays one memory latency, not one per time step.
    constexpr int ITERS = 4;
    for (int tb = warp; tb < T; tb += WARPS * ITERS) {
        float r[ITERS], v[ITERS], vn[ITERS], nnt[ITERS];
#pragma unroll
        for (int u = 0; u < ITERS; ++u) {
            const int t = tb + u * WARPS;
            r[u] = v[u] = vn[u] = nnt[u] = 0.f;
            if (ok && t < T) {
                const size_t i = (size_t)t * N + e;
                r[u] = rewards[i];
                v[u] = values[i];
                vn[u] = (t == T - 1) ? last_values[e] : values[i + N];
                nnt[u] = 1.0f - (float)dones[i];
            }
        }
#pragma unroll
        for (int u = 0; u < ITERS; ++u) {
            const int t = tb + u * WARPS;
            if (t < T) {
                const float g = nnt[u] * gamma;
                sd[t * (ENVS + 1) + lane] = (r[u] + g * vn[u]) - v[u];
                sc[t * (ENVS + 1) + lane] = g * lam;
                sv[t * (ENVS + 1) + lane] = v[u];
            }
        }
    }
    __syncthreads();

    // phase 2: lane = time step (reversed so that the scan runs from T-1 down to 0)
    for (int el = warp; el < ENVS; el += WARPS) {
        float carry = 0.0f;                                   // A_{t+1} entering the chunk
        for (int base = 0; base < T; base += 32) {
            const int k = base + lane;                        // k-th step counted from the end
            const int t = T - 1 - k;
            float c = 0.f, d = 0.f;
            if (k < T) c = sc[t * (ENVS + 1) + el], d = sd[t * (ENVS + 1) + el];
            // inclusive scan of affine maps f_k(x) = d + c*x composed as f_k o f_{k-1} ... : result (C, D)
            float C = c, D = d;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const float Cp = __shfl_up_sync(0xffffffffu, C, o);
                const float Dp = __shfl_up_sync(0xffffffffu, D, o);
                if (lane >= o) {
                    D = D + C * Dp;
                    C = C * Cp;
                }
            }
            const float A = D + C * carry;
            if (k < T) sd[t * (ENVS + 1) + el] = A;
            carry = __shfl_sync(0xffffffffu, A, 31);
        }
    }
    __syncthreads();

    // phase 3: coalesced stores + statistics of the raw advantages
    double s1 = 0.0, s2 = 0.0;
    for (int t = warp; t < T; t += WARPS) {
        if (ok) {
            const size_t i = (size_t)t * N + e;
            const float v = sv[t * (ENVS + 1) + lane];
            const float ret = sd[t * (ENVS + 1) + lane] + v;
            const float adv = ret - v;
            returns[i] = ret;
            advantages[i] = adv;
            s1 += (double)adv;
            s2 += (double)adv * (double)adv;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) red[0][warp] = s1, red[1][warp] = s2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, q = 0.0;
        for (int w = 0; w < WARPS; ++w) a += red[0][w], q += red[1][w];
        atomicAdd(stats, a);
        atomicAdd(stats + 1, q);
    }
}

// ------------------------------------------------------------------------------------------
// Wide shards: one THREAD per env walks the time dimension serially (the reference's own loop and operation order,
// rollout_storage.py:127-134), lane = env so every load and store is one coalesced 128-byte row.  The warp scan
// above spends ~220 instructions per sample on shuffles and shared-memory transposes (ncu at 65 536 x 24: 71 % issue
// active, 10 % DRAM) - it is the right shape when N is small and T long, this one when N alone fills the GPU.
// Time steps go in chunks of CHUNK: the loads of the next chunk are in flight while the current one is consumed.
// ------------------------------------------------------------------------------------------
constexpr int SERIAL_THREADS = 128;

template <int CHUNK>
__global__ void __launch_bounds__(SERIAL_THREADS)
gae_serial_kernel(const float *__restrict__ rewards, const float *__restrict__ values,
                  const uint8_t *__restrict__ dones, const float *__restrict__ last_values,
                  float *__restrict__ returns, float *__restrict__ advantages, double *__restrict__ stats, int T, int N,
                  float gamma, float lam) {
    hb::pdl_trigger();
    __shared__ double red[2][SERIAL_THREADS / 32];
    const int e = blockIdx.x * SERIAL_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double s1 = 0.0, s2 = 0.0;
    if (e < N) {
        float r[CHUNK], v[CHUNK], nr[CHUNK], nv[CHUNK];
        uint8_t d[CHUNK], nd[CHUNK];
        auto load = [&](int t_hi, float *rr, float *vv, uint8_t *dd) {          // steps t_hi, t_hi - 1, ...
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) {
                const int t = t_hi - u;
                rr[u] = vv[u] = 0.f, dd[u] = 0;
                if (t >= 0) {
                    const size_t i = (size_t)t * N + e;
                    rr[u] = rewards[i], vv[u] = values[i], dd[u] = dones[i];
                }
            }
        };
        float next_v = last_values[e], adv = 0.0f;
        load(T - 1, r, v, d);
        for (int t_hi = T - 1; t_hi >= 0; t_hi -= CHUNK) {
            load(t_hi - CHUNK, nr, nv, nd);                                       // prefetch (predicated off below t = 0)
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) {
                const int t = t_hi - u;
                if (t >= 0) {
                    const float g = (1.0f - (float)d[u]) * gamma;
                    const float delta = (r[u] + g * next_v) - v[u];
                    adv = delta + (g * lam) * adv;
                    const float ret = adv + v[u];
                    const float raw = ret - v[u];                                 // advantages = returns - values (:135)
                    const size_t i = (size_t)t * N + e;
                    returns[i] = ret;
                    advantages[i] = raw;
                    s1 += (double)raw;
                    s2 += (double)raw * (double)raw;
                    next_v = v[u];
                }
            }
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) r[u] = nr[u], v[u] = nv[u], d[u] = nd[u];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) red[0][warp] = s1, red[1][warp] = s2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, q = 0.0;
        for (int w = 0; w < SERIAL_THREADS / 32; ++w) a += red[0][w], q += red[1][w];
        atomicAdd(stats, a);
        atomicAdd(stats + 1, q);
    }
}

// ------------------------------------------------------------------------------------------
// Single-GPU form: the whole of compute_returns in ONE launch.  One thread per env as above, but the T raw advantages
// of the env stay on chip (shared memory) while the grid agrees on (sum, sum of squares): block reduction -> fp64 atomics -> ticket
// barrier (cooperative launch: every block is resident) -> mean / unbiased std -> the normalised advantages are written
// once.  Against memset + scan + normalise this drops two launches and the write + re-read of the raw advantages
// (17 instead of 25 bytes per sample).  scratch = {sum, sum sq, ticket, -}: zero on entry, re-armed by the last block.
// ------------------------------------------------------------------------------------------

// The grid agrees on (sum, sum of squares): every block adds its pair to one of GAE_SLOTS slot pairs (blocks spread over the
// slots, so that hundreds of fp64 atomics do not queue on one address), takes a ticket, spins until all blocks have (every
// block is resident: the launch is sized to one wave), reads the slots and derives mean / unbiased std
// (rollout_storage.py:136).  The last reader re-arms the scratch for the next launch.
// scratch (HB_GAE_SCRATCH_DOUBLES = 32): [0..7] sums, [8..15] sums of squares, [16] ticket.  Called by one thread per block.
constexpr int GAE_SLOTS = 8;
__device__ __forceinline__ void grid_statistics(double *__restrict__ scratch, double a, double q, double n, float *s_norm) {
    unsigned long long *ticket = reinterpret_cast<unsigned long long *>(scratch + 2 * GAE_SLOTS);
    const int slot = blockIdx.x & (GAE_SLOTS - 1);
    atomicAdd(scratch + slot, a);
    atomicAdd(scratch + GAE_SLOTS + slot, q);
    __threadfence();
    atomicAdd(ticket, 1ull);
    while (hb::ld_acquire_u64(ticket) < (unsigned long long)gridDim.x) { }       // ---- grid barrier ----
    const volatile double *sv = scratch;
    double s1 = 0.0, s2 = 0.0;
#pragma unroll
    for (int k = 0; k < GAE_SLOTS; ++k) s1 += sv[k], s2 += sv[GAE_SLOTS + k];
    const double mean = s1 / n;
    double var = (s2 - n * mean * mean) / (n - 1.0);                             // unbiased (rollout_storage.py:136)
    if (var < 0.0) var = 0.0;
    s_norm[0] = (float)mean, s_norm[1] = (float)sqrt(var) + 1e-8f;
    __threadfence();
    if (atomicAdd(ticket, 1ull) == 2ull * gridDim.x - 1ull) {                    // every block has read: re-arm
#pragma unroll
        for (int k = 0; k < 2 * GAE_SLOTS; ++k) scratch[k] = 0.0;
        __threadfence();
        *ticket = 0ull;
    }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
gae_fused_kernel(const float *__restrict__ rewards, const float *__restrict__ values, const uint8_t *__restrict__ dones,
                 const float *__restrict__ last_values, float *__restrict__ returns, float *__restrict__ advantages,
                 double *__restrict__ scratch, int T, int N, float gamma, float lam) {
    constexpr int CHUNK = 8;
    extern __shared__ float s_raw[];          // [T][THREADS]: this block's raw advantages, parked across the grid barrier
    __shared__ double red[2][THREADS / 32];
    __shared__ float s_norm[2];
    const int e = blockIdx.x * THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool ok = e < N;
    double s1 = 0.0, s2 = 0.0;
    if (ok) {
        float r[CHUNK], v[CHUNK], nr[CHUNK], nv[CHUNK];
        uint8_t d[CHUNK], nd[CHUNK];
        auto load = [&](int t_hi, float *rr, float *vv, uint8_t *dd) {          // steps t_hi, t_hi - 1, ...
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) {
                const int t = t_hi - u;
                rr[u] = vv[u] = 0.f, dd[u] = 0;
                if (t >= 0) {
                    const size_t i = (size_t)t * N + e;
                    rr[u] = rewards[i], vv[u] = values[i], dd[u] = dones[i];
                }
            }
        };
        float next_v = last_values[e], adv = 0.0f;
        load(T - 1, r, v, d);
#pragma unroll 1
        for (int t_hi = T - 1; t_hi >= 0; t_hi -= CHUNK) {
            load(t_hi - CHUNK, nr, nv, nd);                                       // next chunk in flight
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) {
                const int t = t_hi - u;
                if (t >= 0) {
                    const float g = (1.0f - (float)d[u]) * gamma;
                    const float delta = (r[u] + g * next_v) - v[u];
                    adv = delta + (g * lam) * adv;
                    const float ret = adv + v[u];
                    const float raw = ret - v[u];                                 // advantages = returns - values (:135)
                    returns[(size_t)t * N + e] = ret;
                    s_raw[t * THREADS + threadIdx.x] = raw;
                    s1 += (double)raw;
                    s2 += (double)raw * (double)raw;
                    next_v = v[u];
                }
            }
#pragma unroll
            for (int u = 0; u < CHUNK; ++u) r[u] = nr[u], v[u] = nv[u], d[u] = nd[u];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane == 0) red[0][warp] = s1, red[1][warp] = s2;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, q = 0.0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) a += red[0][w], q += red[1][w];
        grid_statistics(scratch, a, q, (double)T * (double)N, s_norm);
    }
    __syncthreads();
    const float m = s_norm[0], denom = s_norm[1];
    if (ok) {
#pragma unroll 4
        for (int t = 0; t < T; ++t) advantages[(size_t)t * N + e] = (s_raw[t * THREADS + threadIdx.x] - m) / denom;
    }
}

__global__ void __launch_bounds__(256)
gae_normalize_kernel(float *__restrict__ adv, const double *__restrict__ stats, long long stat_count,
                     long long count) {
    hb::pdl_wait();                 // the scan (or the all-reduce of its statistics) is complete
    // mean and unbiased std from (sum, sum of squares), rollout_storage.py:136
    const double n = (double)stat_count;
    const double mean = stats[0] / n;
    double var = (stats[1] - n * mean * mean) / (n - 1.0);
    if (var < 0.0) var = 0.0;
    const float m = (float)mean;
    const float denom = (float)sqrt(var) + 1e-8f;
    // four advantages per thread where the buffer allows it (the fp64 preamble above is per thread)
    const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 + 3 < count && (reinterpret_cast<uintptr_t>(adv) & 15u) == 0) {
        float4 a = *reinterpret_cast<float4 *>(adv + i4);
        a.x = (a.x - m) / denom, a.y = (a.y - m) / denom, a.z = (a.z - m) / denom, a.w = (a.w - m) / denom;
        *reinterpret_cast<float4 *>(adv + i4) = a;
    } else {
        for (long long i = i4; i < count && i < i4 + 4; ++i) adv[i] = (adv[i] - m) / denom;
    }
}

template <int THREADS>
int launch_gae_fused(const float *rewards, const float *values, const uint8_t *dones, const float *last_values,
                     float *returns, float *advantages, double *scratch, int T, int N, float gamma, float lam,
                     cudaStream_t st, bool *fits) {
    auto kern = gae_fused_kernel<THREADS>;
    const size_t smem = (size_t)T * THREADS * sizeof(float);
    *fits = false;
    if (smem > 64 * 1024) return HB_OK;
    static bool attr = false;
    if (!attr) {
        HB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        attr = true;
    }
    int per_sm = 0;
    HB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem));
    const int grid = (N + THREADS - 1) / THREADS;
    *fits = grid <= per_sm * hb::sm_count();                 // the blocks wait for one another: all must be resident
    if (!*fits) return HB_OK;
    HB_CUDA(hb::launch_coop(kern, dim3(grid), dim3(THREADS), smem, st, rewards, values, dones, last_values, returns, advantages,
                            scratch, T, N, gamma, lam));
    HB_CHECK_LAUNCH("gae_fused_kernel");
    return HB_OK;
}

}  // namespace

extern "C" {

int hb_gae_returns(const float *rewards, const float *values, const uint8_t *dones, const float *last_values,
                   float *returns, float *advantages, double *stats, int32_t T, int32_t N, float gamma, float lam,
                   void *stream) {
    HB_REQUIRE(rewards && values && dones && last_values && returns && advantages && stats, "hb_gae_returns: null buffer");
    HB_REQUIRE(T > 0 && N > 0, "hb_gae_returns: T and N must be positive");
    const size_t smem = (size_t)3 * T * (ENVS + 1) * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    HB_CUDA(cudaMemsetAsync(stats, 0, 2 * sizeof(double), st));
    if (N >= hb::g_gae_serial_min_envs) {
        gae_serial_kernel<8><<<(N + SERIAL_THREADS - 1) / SERIAL_THREADS, SERIAL_THREADS, 0, st>>>(
            rewards, values, dones, last_values, returns, advantages, stats, T, N, gamma, lam);
        HB_CHECK_LAUNCH("gae_serial_kernel");
        return HB_OK;
    }
    HB_REQUIRE(smem <= 200 * 1024, "hb_gae_returns: T=%d too long for one tile", T);
    if (smem > 48 * 1024) {
        HB_CUDA(cudaFuncSetAttribute(gae_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    gae_scan_kernel<<<(N + ENVS - 1) / ENVS, WARPS * 32, smem, st>>>(rewards, values, dones, last_values, returns,
                                                                     advantages, stats, T, N, gamma, lam);
    HB_CHECK_LAUNCH("gae_scan_kernel");
    return HB_OK;
}

int hb_gae_fused(const float *rewards, const float *values, const uint8_t *dones, const float *last_values, float *returns,
                 float *advantages, double *scratch, int32_t T, int32_t N, float gamma, float lam, void *stream) {
    HB_REQUIRE(rewards && values && dones && last_values && returns && advantages && scratch, "hb_gae_fused: null buffer");
    HB_REQUIRE(T > 0 && N > 0 && (long long)T * N > 1, "hb_gae_fused: T and N must be positive, T * N > 1");
    HB_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 7u) == 0, "hb_gae_fused: scratch must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    bool fits = false;
    int rc = HB_OK;
    // Block width: the launch's fixed cost is the grid barrier (two fp64 atomics, a ticket and a spin per block), so wide
    // shards take wide blocks (65 536 envs: 13.6 us with 256 threads, 15.1 with 128, 19.8 with 64; 16 384 envs: 10.0 / 10.1 /
    // 10.9), narrow ones enough blocks to spread the loads over the SMs (4096 envs: 9.1 us with 64 or 128, 9.6 with 32)
    const int threads = hb::g_gae_threads ? hb::g_gae_threads : (N <= 8192 ? 64 : 256);
#define HB_GAE(TH) launch_gae_fused<TH>(rewards, values, dones, last_values, returns, advantages, scratch, T, N, gamma, lam, st, &fits)
    if (threads == 32) rc = HB_GAE(32);
    else if (threads == 64) rc = HB_GAE(64);
    else if (threads == 256) rc = HB_GAE(256);
    else rc = HB_GAE(128);
    if (!rc && !fits && threads == 256) rc = HB_GAE(128);      // long rollouts: 256 threads x T floats may not fit in shared memory
#undef HB_GAE
    if (rc) return rc;
    if (fits) return HB_OK;
    // long rollouts / shards too wide for one co-resident grid: the two-kernel form (scratch doubles as the statistics)
    if (int rc2 = hb_gae_returns(rewards, values, dones, last_values, returns, advantages, scratch, T, N, gamma, lam, stream)) return rc2;
    if (int rc2 = hb_gae_normalize_n(advantages, scratch, (int64_t)T * N, (int64_t)T * N, stream)) return rc2;
    HB_CUDA(cudaMemsetAsync(scratch, 0, HB_GAE_SCRATCH_DOUBLES * sizeof(double), st));
    return HB_OK;
}

int hb_gae_normalize_n(float *advantages, const double *stats, int64_t stat_count, int64_t count, void *stream) {
    HB_REQUIRE(advantages && stats && stat_count > 1 && count > 0, "hb_gae_normalize: bad arguments");
    HB_CUDA(hb::launch_pdl(true, gae_normalize_kernel, dim3((unsigned)((count + 1023) / 1024)), dim3(256), 0,
                           (cudaStream_t)stream, advantages, stats, (long long)stat_count, (long long)count));
    HB_CHECK_LAUNCH("gae_normalize_kernel");
    return HB_OK;
}

int hb_gae_normalize(float *advantages, const double *stats, int64_t count, void *stream) {
    return hb_gae_normalize_n(advantages, stats, count, count, stream);
}

}  // extern "C"
