// Shared host/device helpers for libhectorb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "hector_b200.h"

namespace hb {

// ---- error plumbing (C ABI: never throw, return hb_status) -------------------------------
void set_error(const char *fmt, ...);
extern thread_local char g_error[512];
void count_launch(int n = 1);

#define HB_REQUIRE(cond, ...)                          \
    do {                                               \
        if (!(cond)) {                                 \
            hb::set_error(__VA_ARGS__);                \
            return HB_ERR_BAD_ARG;                     \
        }                                              \
    } while (0)

#define HB_CHECK_LAUNCH(what)                                                         \
    do {                                                                              \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess) {                                                     \
            hb::set_error("%s: %s", what, cudaGetErrorString(e__));                   \
            return HB_ERR_CUDA;                                                       \
        }                                                                             \
        hb::count_launch();                                                           \
    } while (0)

#define HB_CUDA(call)                                                                 \
    do {                                                                              \
        cudaError_t e__ = (call);                                                     \
        if (e__ != cudaSuccess) {                                                     \
            hb::set_error("%s: %s", #call, cudaGetErrorString(e__));                  \
            return HB_ERR_CUDA;                                                       \
        }                                                                             \
    } while (0)

// Runs CALL with `constexpr int ACT` = the hb_activation value `act` (the kernels take the activation as a template
// parameter); an unknown value is HB_ERR_BAD_ARG.
#define HB_ACT_CASE(A, CALL) case A: { constexpr int ACT = A; CALL; break; }
#define HB_ACT_DISPATCH(act, CALL)                                                        \
    switch (act) {                                                                        \
        HB_ACT_CASE(HB_ACT_ELU, CALL)                                                     \
        HB_ACT_CASE(HB_ACT_SELU, CALL)                                                    \
        HB_ACT_CASE(HB_ACT_RELU, CALL)                                                    \
        HB_ACT_CASE(HB_ACT_LRELU, CALL)                                                   \
        HB_ACT_CASE(HB_ACT_TANH, CALL)                                                    \
        HB_ACT_CASE(HB_ACT_SIGMOID, CALL)                                                 \
        default:                                                                          \
            hb::set_error("unknown activation %d (hb_activation)", (int)(act));          \
            return HB_ERR_BAD_ARG;                                                        \
    }

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int sm_count();   // cached cudaDevAttrMultiProcessorCount of the current device
extern int g_use_pdl;   // "pdl" option: programmatic stream serialization of the step's kernels: 1 = all, 0 = none,
                        // 2 or -1 (default) = only the PD-torque launches.  On the large kernels (post-physics, frame
                        // stack) the early-resident dependents and the completion flush behind griddepcontrol.wait
                        // cost more than the overlap gains at every shard size measured (52.0 vs 60.4 us per step at
                        // 4096 envs, -13 % at 65 536).  3 = PD launches + post-physics, 4 = PD launches + frame stack:
                        // round 2, 4096 envs: 43.1 (default) / 49.2 (3) / 43.4 (4) / 49.4 (1) us per step; 16 384 envs:
                        // 73.0 / 77.5 / 78.7 / 79.4
extern int g_gae_serial_min_envs;   // "gae_serial_min_envs" option: shards at least this wide run GAE one thread per env (default 8192)
extern int g_gae_threads;   // "gae_threads" option: block width of the single-launch GAE (0 = by shard width; 32 / 64 / 128 / 256)
extern int g_coop_launch;   // "coop_launch" option: 1 = kernels with a grid barrier (optimizer step, single-launch GAE) are launched with the
                            // cooperative attribute; 0 (default) = plain launches of a grid that fits the device (see hector_b200.h)
extern int g_gemm_snake;  // "gemm_tile_snake" option: 1 (default) = rounds of the GEMM tile list are dealt to the CTAs in alternating direction
extern int g_gemm_pdl;  // "gemm_pdl" option: 1 (default) = GEMM launches overlap their set-up with the previous kernel's tail
inline bool use_pdl(int num_envs) { (void)num_envs; return g_use_pdl == 1; }
inline bool use_pdl_post(int num_envs) { return g_use_pdl == 3 || use_pdl(num_envs); }      // 3: PD launches + post-physics
inline bool use_pdl_stack(int num_envs) { return g_use_pdl == 4 || use_pdl(num_envs); }     // 4: PD launches + frame stack / finalize
inline bool use_pdl_small_kernel(int num_envs) { return g_use_pdl >= 2 || g_use_pdl < 0 || use_pdl(num_envs); }

#ifdef __CUDACC__
// <<<grid, block, smem, stream>>> with the programmatic-dependent-launch attribute (kernels call hb::pdl_wait()).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cfg.attrs = at, cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// <<<grid, block, smem, stream>>> of a kernel whose blocks wait on one another at a grid barrier: the caller sizes the grid
// to be co-resident, and the "coop_launch" option adds the cooperative attribute (g_coop_launch).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_coop(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = g_coop_launch ? 1 : 0;
    cfg.attrs = at, cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// ---- device helpers -------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP) --------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared, `bytes` multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global
__device__ __forceinline__ void bulk_s2g(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// Programmatic dependent launch: a kernel launched with hb::launch_pdl may start while its predecessor in the stream
// (or graph) is still running; it must not touch what the predecessor produces before pdl_wait() returns (= the
// predecessor grid has completed and its writes are visible).  pdl_trigger() lets the NEXT kernel start early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// acquire load of a grid-barrier ticket or flag written by other blocks
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// streaming loads / stores (data touched once per step: keep it out of L1)
__device__ __forceinline__ float4 ld_stream4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
// predicated form: zeros, and no memory access, when `pred` is false (branch-free)
__device__ __forceinline__ float4 ld_stream4_if(const float4 *p, bool pred) {
    float4 v;
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.u32 q, %5, 0;\n"
        "mov.f32 %0, 0f00000000;\n"
        "mov.f32 %1, 0f00000000;\n"
        "mov.f32 %2, 0f00000000;\n"
        "mov.f32 %3, 0f00000000;\n"
        "@q ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];\n"
        "}\n"
        : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
        : "l"(p), "r"((uint32_t)pred));
    return v;
}
__device__ __forceinline__ void st_stream4(float4 *p, const float4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// Hidden-layer activations of the MLPs (hb_activation, torch's definitions: include/hector_b200.h).  act_fwd with
// ACCURATE = true uses libm's expm1f / expf (fp32-grade, the 3xTF32 epilogue pass); otherwise the exponentials are __expf,
// whose error is far below the TF32 operand rounding of the GEMM in front of it.  act_grad(h) is f'(z) written in the
// forward output h = f(z).
constexpr float SELU_ALPHA = 1.6732632423543772848170429916717f, SELU_SCALE = 1.0507009873554804934193349852946f;
template <int ACT, bool ACCURATE>
__device__ __forceinline__ float act_fwd(float z) {
    if constexpr (ACT == HB_ACT_ELU) return z > 0.0f ? z : (ACCURATE ? expm1f(z) : __expf(z) - 1.0f);
    else if constexpr (ACT == HB_ACT_SELU) return z > 0.0f ? SELU_SCALE * z : (SELU_SCALE * SELU_ALPHA) * (ACCURATE ? expm1f(z) : __expf(z) - 1.0f);
    else if constexpr (ACT == HB_ACT_RELU) return z > 0.0f ? z : 0.0f;
    else if constexpr (ACT == HB_ACT_LRELU) return z > 0.0f ? z : 0.01f * z;
    else if constexpr (ACT == HB_ACT_TANH) return tanhf(z);
    else return 1.0f / (1.0f + (ACCURATE ? expf(-z) : __expf(-z)));
}
template <int ACT>
__device__ __forceinline__ float act_grad(float h) {
    if constexpr (ACT == HB_ACT_ELU) return h > 0.0f ? 1.0f : h + 1.0f;
    else if constexpr (ACT == HB_ACT_SELU) return h > 0.0f ? SELU_SCALE : h + SELU_SCALE * SELU_ALPHA;
    else if constexpr (ACT == HB_ACT_RELU) return h > 0.0f ? 1.0f : 0.0f;
    else if constexpr (ACT == HB_ACT_LRELU) return h > 0.0f ? 1.0f : 0.01f;
    else if constexpr (ACT == HB_ACT_TANH) return 1.0f - h * h;
    else return (1.0f - h) * h;
}

// Philox4x32-10 (counter c0..c3, key k0 k1): the library's device generator (env noise, PPO action sample)
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0, c1 = l1, c2 = h0 ^ c3 ^ k1, c3 = l0;
        k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

#endif  // __CUDACC__
}  // namespace hb
