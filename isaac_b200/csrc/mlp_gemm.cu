// tcgen05 / TMEM / TMA GEMM for the ActorCritic MLPs (SURVEY.md §8 rows a13-a15), sm_100a only.
//
//   D[M,N] (+)= A[M,K] * B[N,K]^T          fp32 storage, TF32 tensor-core math, fp32 accumulation in TMEM
//
// One CTA computes a sequence of 128 x BN output tiles (optionally K-splits of them):
//   warp 8      TMA producer: 2-D tiled tensor maps, 128-byte swizzle, NSTAGE-deep mbarrier ring
//   warp 9      allocates TMEM (two accumulators) and issues tcgen05.mma.cta_group::1.kind::tf32 (one elected
//               lane); tcgen05.commit releases smem stages and hands finished accumulators to the epilogue
//   warps 0-7   epilogue: tcgen05.ld the accumulator quarter / column half that belongs to the warp
//               (lane = row), apply the fused tail in registers - bias + activation f (forward), f' (dgrad: the
//               forward activations arrive by TMA, one 32 x 32 block ahead) - write the block into a 128-byte-swizzled
//               shared-memory tile and hand it to a TMA store; split-K wgrad tiles leave as vector red.add instead
// The kernel is persistent: one CTA per SM walks a static tile list, so barrier / TMEM setup is paid once and
// the epilogue of one tile overlaps the main loop of the next.
//
// Operand layouts.  "K-major" = the contraction index is contiguous in memory (activations
// [rows, features] as A, nn.Linear weights [out, in] as B: the forward pass).  "MN-major" = the
// M/N index is contiguous (weights as B of dgrad, activations / gradients as A and B of wgrad), so
// backward needs no transposed copies: the same row-major tensors are read through a different
// tensor map + UMMA descriptor (LayoutType SWIZZLE_128B, a_major/b_major bits of the instruction
// descriptor).
#include <cuda.h>

#include "hb_common.cuh"

namespace {

constexpr int BM = 128;           // UMMA M (cta_group::1)
constexpr int BK = 32;            // floats per k-block = one 128-byte swizzle row
constexpr int UMMA_K = 8;         // tf32: 32 bytes of K per instruction
constexpr int EPI_WARPS = 8;          // two warps per TMEM lane quarter, each takes half of the tile's columns
constexpr int PRODUCER_WARP = EPI_WARPS, MMA_WARP = EPI_WARPS + 1;
constexpr int GEMM_THREADS = (EPI_WARPS + 2) * 32;

enum Epilogue { EPI_STORE = 0, EPI_BIAS = 1, EPI_BIAS_ACT = 2, EPI_ACT_BWD = 3, EPI_ATOMIC = 4 };

struct GemmArgs {
    int M, N, K;                  // logical sizes (K = contraction length)
    int kb_per_split;             // k-blocks of one k split
    int tiles_m, tiles_n, splits, total_tiles;   // tile list: (k split, m tile, n tile), n fastest
    float *D;                     // [M, ldd]
    int ldd;
    const float *bias;            // bias[n * bias_stride] (weights and bias share one packed matrix)
    int bias_stride;
    const float *H;               // EPI_ACT_BWD: forward activations [M, ldh]
    int ldh;
    int snake;                    // rounds of the tile list dealt in alternating direction (problem 0's value counts)
};

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(void *smem, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(hb::smem_u32(smem)), "l"(map), "r"(c0), "r"(c1), "r"(hb::smem_u32(bar))
        : "memory");
}
// pair mode (cta_group::2): both CTAs of a 2-CTA cluster load, the transaction bytes land on the leader's barrier
__device__ __forceinline__ void tma_load_2d_pair(void *smem, const CUtensorMap *map, int c0, int c1, uint32_t leader_bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(hb::smem_u32(smem)), "l"(map), "r"(c0), "r"(c1), "r"(leader_bar)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {      // same variable in CTA `rank` of the cluster
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t *dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(hb::smem_u32(dst_smem)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t *bar) {      // arrives on the same barrier of both CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     hb::smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap *map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(hb::smem_u32(dst_smem)),
                 "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(hb::smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float *v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float *v) {      // 32 consecutive columns of this warp's 32 lanes
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]),
          "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]),
          "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// TMA store of a shared-memory box (written by this warp with ordinary stores, then fenced into the async proxy)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *map, int c0, int c1, const void *smem) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(map), "r"(c0), "r"(c1),
                 "r"(hb::smem_u32(smem))
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// UMMA shared-memory descriptor (cute::UMMA::SmemDescriptor): start address, leading / stride byte
// offsets in 16-byte units, version 1 (Blackwell), layout type in bits [61,64).
//   K-major operands : LayoutType SWIZZLE_128B (2): rows of 32 tf32 = 128 bytes, 16-byte chunks XOR-ed with
//                      (row % 8); SBO = 1024 bytes between 8-row groups.
//   MN-major operands: 32-bit types only exist as SWIZZLE_128B_BASE32B (1) (CUTLASS: "for mn-major tf32
//                      operands, SW128_32B is the only available smem layout"): rows of 32 MN-elements,
//                      32-byte chunks XOR-ed with (row % 4); LBO = stride between 32-element MN blocks,
//                      SBO = 512 bytes between 4-row K groups.
constexpr uint32_t LAYOUT_SW128 = 2, LAYOUT_SW128_BASE32B = 1;
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}

// Instruction descriptor (cute::UMMA::InstrDescriptor): F32 accumulate, TF32 x TF32.
__host__ __device__ constexpr uint32_t make_idesc(int n, bool a_mn, bool b_mn, int m = BM) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// PAIR = two CTAs of a cluster (two SMs) compute one 256 x BN tile with tcgen05.mma.cta_group::2: each CTA stages
// its own 128 rows of A but only HALF of the B tile (the tensor core reads the other half from the peer's shared
// memory).  These TF32 GEMMs are bound by operand delivery (L2 -> SMEM, ~12 TB/s chip-wide), not by the tensor
// pipe: per CTA and k-block a pair moves 32 KB instead of 48 KB for the same 128 x 256 x 32 MACs.
constexpr int H_TILE_BYTES = 4096;                // f' epilogue: per warp, one TMA-loaded 32 x 32 block of forward activations
template <int BN, bool PAIR, int EPI = 0>
__host__ __device__ constexpr int stages_for() {
    // the f' kernels give one stage to the epilogue warps' activation tiles (their K is a layer width: few k-blocks)
    return (PAIR ? 6 : (BN >= 256 ? 4 : (BN >= 128 ? 6 : 8))) - (EPI != 3 ? 0 : (BN >= 128 ? 1 : (BN >= 64 ? 2 : 0)));
}

constexpr int EPI_TILE_FLOATS = 32 * 33;          // per epilogue warp: one padded 32 x 32 transpose tile
template <int BN, bool PAIR, int EPI = 0>
__host__ __device__ constexpr size_t smem_bytes_for() {
    return (size_t)stages_for<BN, PAIR, EPI>() * (BM * BK * 4 + (PAIR ? BN / 2 : BN) * BK * 4) + EPI_WARPS * EPI_TILE_FLOATS * 4 +
           (EPI == 3 ? EPI_WARPS * H_TILE_BYTES : 0) + 1024;
}
static_assert(smem_bytes_for<256, true, 3>() <= 227 * 1024 && smem_bytes_for<256, false, 3>() <= 227 * 1024 &&
                  smem_bytes_for<128, false, 3>() <= 227 * 1024 && smem_bytes_for<64, false, 3>() <= 227 * 1024,
              "f' kernels: stages + output tiles + activation tiles must fit in shared memory");
static_assert((EPI_WARPS * EPI_TILE_FLOATS * 4) % 1024 == 0, "the activation tiles behind the output tiles stay 1024-byte aligned");

// Persistent, warp-specialised: one CTA per SM walks a static list of output tiles
//   tile t = blockIdx.x + i * gridDim.x  ->  (k split, m tile, n tile), n fastest so that the CTAs running at the
//   same time share the rows of A in L2 (the weights are small and always L2-resident).
// Three pipelines: shared-memory stages (TMA <-> MMA), two TMEM accumulators (MMA <-> epilogue: the epilogue of tile
// i overlaps the main loop of tile i + 1), and the tile list.
// GROUPED: one launch may carry TWO problems of the same kind (the actor's and the critic's GEMM of one layer): the tile
// list is problem 0's tiles followed by problem 1's, dealt round-robin to the persistent CTAs, so both networks share
// every wave of tiles and the pipeline set-up / drain of a launch is paid once per layer instead of once per network.
// ACT: the hb_activation of EPI_BIAS_ACT / EPI_ACT_BWD (HB_ACT_ELU for the other epilogues).
template <int BN, bool A_MN, bool B_MN, int EPI, bool PAIR, int ACT>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tf32_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_b0,
                 const __grid_constant__ GemmArgs g0, const __grid_constant__ CUtensorMap map_a1,
                 const __grid_constant__ CUtensorMap map_b1, const __grid_constant__ GemmArgs g1,
                 const __grid_constant__ CUtensorMap map_d0, const __grid_constant__ CUtensorMap map_d1,
                 const __grid_constant__ CUtensorMap map_h0, const __grid_constant__ CUtensorMap map_h1) {
    constexpr int NSTAGE = stages_for<BN, PAIR, EPI>();
    constexpr int BN_CTA = PAIR ? BN / 2 : BN;               // B rows staged by this CTA
    constexpr int A_BYTES = BM * BK * 4, B_BYTES = BN_CTA * BK * 4;
    constexpr uint32_t ACC_COLS = BN < 32 ? 32 : BN;          // TMEM columns of one accumulator
    constexpr uint32_t TMEM_COLS = 2 * ACC_COLS;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t *sa = smem, *sb = smem + NSTAGE * A_BYTES;
    float *epi_smem = reinterpret_cast<float *>(smem + NSTAGE * (A_BYTES + B_BYTES));
    __shared__ __align__(8) uint64_t full_bar[NSTAGE], empty_bar[NSTAGE], acc_full[2], acc_empty[2], h_bar[EPI_WARPS];
    __shared__ uint32_t tmem_base_smem;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int all_tiles = g0.total_tiles + g1.total_tiles;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;     // 0 = leader (issues the MMAs, owns full / acc_empty barriers)
    const int first_tile = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int tile_step = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    // Round r of the tile list goes to the CTAs in alternating direction (boustrophedon): the CTAs that take the extra
    // tiles of a partial last round are then the ones whose earlier tiles came from the END of the previous round - in a
    // grouped launch the second, smaller problem - instead of the ones already holding the longest tiles.
    auto tile_at = [&](int round) { return round * tile_step + (((round & 1) && g0.snake) ? tile_step - 1 - first_tile : first_tile); };

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) hb::mbar_init(&full_bar[s], 1), hb::mbar_init(&empty_bar[s], 1);
#pragma unroll
        for (int a = 0; a < 2; ++a) hb::mbar_init(&acc_full[a], 1), hb::mbar_init(&acc_empty[a], PAIR ? 2 * EPI_WARPS : EPI_WARPS);
#pragma unroll
        for (int w = 0; w < EPI_WARPS; ++w) hb::mbar_init(&h_bar[w], 1);
        hb::fence_mbar_init();
    }
    if (warp == PRODUCER_WARP && lane == 0) {
        prefetch_tmap(&map_a0), prefetch_tmap(&map_b0);
        if (EPI != EPI_ATOMIC) prefetch_tmap(&map_d0);
        if (EPI == EPI_ACT_BWD) prefetch_tmap(&map_h0);
        if (g1.total_tiles > 0) {
            prefetch_tmap(&map_a1), prefetch_tmap(&map_b1);
            if (EPI != EPI_ATOMIC) prefetch_tmap(&map_d1);
            if (EPI == EPI_ACT_BWD) prefetch_tmap(&map_h1);
        }
    }
    if (warp == MMA_WARP) {
        if (PAIR) tmem_alloc_pair(&tmem_base_smem, TMEM_COLS);
        else tmem_alloc(&tmem_base_smem, TMEM_COLS);
    }
    tc_fence_before();
    if (PAIR) cluster_sync();        // the peer's barriers are initialised before anything arrives on them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_smem;
    // Programmatic dependent launch: everything above (tensor-map prefetch, barriers, TMEM, cluster rendezvous) ran
    // while the previous kernel of the stream was still draining its last tiles; its results are touched only from here.
    hb::pdl_trigger();
    hb::pdl_wait();

    auto tile_coords = [&](int t, const GemmArgs &g, int &m0, int &n0, int &kb_begin, int &nkb) {
        // n fastest, then m, then the k split: the tiles in flight at any time share their k slices of A and B, so
        // with split-K (weight gradients: both operands are minibatch-sized) every byte is fetched from HBM once
        const int kb_total = (g.K + BK - 1) / BK;
        const int nt = t % g.tiles_n;
        const int rest = t / g.tiles_n;
        const int mt = rest % g.tiles_m;
        const int z = rest / g.tiles_m;
        m0 = PAIR ? (mt * 2 + (int)rank) * BM : mt * BM, n0 = nt * BN;
        kb_begin = z * g.kb_per_split;
        nkb = min(kb_begin + g.kb_per_split, kb_total) - kb_begin;
    };

    if (warp == PRODUCER_WARP) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            uint32_t it = 0;
            for (int round = 0; round * tile_step < all_tiles; ++round) {
                const int t = tile_at(round);
                if (t >= all_tiles) break;           // (only in the last round)
                const bool second = t >= g0.total_tiles;
                const GemmArgs &g = second ? g1 : g0;
                const CUtensorMap *pmap_a = second ? &map_a1 : &map_a0, *pmap_b = second ? &map_b1 : &map_b0;
                int m0, n0, kb_begin, nkb;
                tile_coords(second ? t - g0.total_tiles : t, g, m0, n0, kb_begin, nkb);
                const int nb0 = n0 + (PAIR ? (int)rank * BN_CTA : 0);      // this CTA's rows of the B tile
                for (int i = 0; i < nkb; ++i, ++it) {
                    const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1;
                    hb::mbar_wait(&empty_bar[s], ph ^ 1);
                    const int k0 = (kb_begin + i) * BK;
                    if (PAIR) {
                        // both CTAs' bytes are counted on the leader's barrier
                        if (rank == 0) hb::mbar_expect_tx(&full_bar[s], 2 * (A_BYTES + B_BYTES));
                        const uint32_t bar = mapa_shared(hb::smem_u32(&full_bar[s]), 0);
                        if (A_MN) {
#pragma unroll
                            for (int j = 0; j < BM / 32; ++j) tma_load_2d_pair(sa + s * A_BYTES + j * 4096, pmap_a, m0 + 32 * j, k0, bar);
                        } else {
                            tma_load_2d_pair(sa + s * A_BYTES, pmap_a, k0, m0, bar);
                        }
                        if (B_MN) {
#pragma unroll
                            for (int j = 0; j < BN_CTA / 32; ++j) tma_load_2d_pair(sb + s * B_BYTES + j * 4096, pmap_b, nb0 + 32 * j, k0, bar);
                        } else {
                            tma_load_2d_pair(sb + s * B_BYTES, pmap_b, k0, nb0, bar);
                        }
                    } else {
                        hb::mbar_expect_tx(&full_bar[s], A_BYTES + B_BYTES);
                        if (A_MN) {      // tensor map dims (M, K): boxes of 32 m x 32 k, one 4 KB swizzle block each
#pragma unroll
                            for (int j = 0; j < BM / 32; ++j) tma_load_2d(sa + s * A_BYTES + j * 4096, pmap_a, m0 + 32 * j, k0, &full_bar[s]);
                        } else {         // tensor map dims (K, M): one box of 32 k x 128 rows
                            tma_load_2d(sa + s * A_BYTES, pmap_a, k0, m0, &full_bar[s]);
                        }
                        if (B_MN) {
#pragma unroll
                            for (int j = 0; j < BN / 32; ++j) tma_load_2d(sb + s * B_BYTES + j * 4096, pmap_b, n0 + 32 * j, k0, &full_bar[s]);
                        } else {
                            tma_load_2d(sb + s * B_BYTES, pmap_b, k0, n0, &full_bar[s]);
                        }
                    }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        // ===================== MMA issuer =====================
        constexpr uint32_t idesc = make_idesc(BN < 16 ? 16 : BN, A_MN, B_MN, PAIR ? 2 * BM : BM);
        uint32_t it = 0, acc_it = 0;
        for (int round = 0; round * tile_step < all_tiles && rank == 0; ++round, ++acc_it) {
            const int t = tile_at(round);
            if (t >= all_tiles) break;
            const bool second = t >= g0.total_tiles;
            int m0, n0, kb_begin, nkb;
            tile_coords(second ? t - g0.total_tiles : t, second ? g1 : g0, m0, n0, kb_begin, nkb);
            const uint32_t a = acc_it & 1, aph = (acc_it >> 1) & 1;
            hb::mbar_wait(&acc_empty[a], aph ^ 1);           // the epilogue has drained this accumulator
            tc_fence_after();
            const uint32_t tmem_acc = tmem_base + a * ACC_COLS;
            for (int i = 0; i < nkb; ++i, ++it) {
                const uint32_t s = it % NSTAGE, ph = (it / NSTAGE) & 1;
                hb::mbar_wait(&full_bar[s], ph);
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t a_addr = hb::smem_u32(sa + s * A_BYTES), b_addr = hb::smem_u32(sb + s * B_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        // K-major: 8 tf32 = 32 bytes further along the swizzled 128-byte row;
                        // MN-major: 8 k-rows = one 1024-byte swizzle atom further
                        const uint64_t ad = A_MN ? make_desc(a_addr + k * 1024, 4096, 512, LAYOUT_SW128_BASE32B)
                                                 : make_desc(a_addr + k * 32, 16, 1024, LAYOUT_SW128);
                        const uint64_t bd = B_MN ? make_desc(b_addr + k * 1024, 4096, 512, LAYOUT_SW128_BASE32B)
                                                 : make_desc(b_addr + k * 32, 16, 1024, LAYOUT_SW128);
                        if (PAIR) umma_tf32_pair(tmem_acc, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
                        else umma_tf32(tmem_acc, ad, bd, idesc, (i > 0 || k > 0) ? 1u : 0u);
                    }
                    if (PAIR) {        // both CTAs' stages / epilogues are released
                        umma_commit_pair(&empty_bar[s]);
                        if (i == nkb - 1) umma_commit_pair(&acc_full[a]);
                    } else {
                        umma_commit(&empty_bar[s]);                  // frees the smem stage once the MMAs have read it
                        if (i == nkb - 1) umma_commit(&acc_full[a]); // accumulator complete -> epilogue
                    }
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== epilogue (warps 0-7) =====================
        // Warp w reads TMEM lanes 32*(w%4) .. +31 (the hardware's lane-quarter rule) and the column half w/4.
        // The accumulator arrives with lane = row.  Global traffic wants lane = column (128-byte rows), so
        // every 32 x 32 block goes through a padded shared-memory tile private to the warp: activations for
        // f' come in coalesced, results leave coalesced.
        const int quarter = warp & 3, half = warp >> 2;
        constexpr int HALF_COLS = BN >= 64 ? BN / 2 : BN;          // narrow tiles: the second warp of a quarter idles
        const int c_begin = BN >= 64 ? half * HALF_COLS : 0;
        const int c_end = (BN >= 64 || half == 0) ? c_begin + HALF_COLS : 0;
        float *tile = epi_smem + warp * EPI_TILE_FLOATS;
        uint32_t acc_it = 0, h_phase = 0;
        for (int round = 0; round * tile_step < all_tiles; ++round, ++acc_it) {
            const int t = tile_at(round);
            if (t >= all_tiles) break;
            const bool second = t >= g0.total_tiles;
            const GemmArgs &g = second ? g1 : g0;
            int m0, n0, kb_begin, nkb;
            tile_coords(second ? t - g0.total_tiles : t, g, m0, n0, kb_begin, nkb);
            const uint32_t a = acc_it & 1, aph = (acc_it >> 1) & 1;
            const int mw = m0 + quarter * 32;                  // first row of this warp
            // f': the warp's 32 x 32 blocks of the forward activations arrive by TMA in its second tile, one block ahead
            // of their use (the first while the accumulator is still being computed), with the same 128-byte swizzle
            uint8_t *htile = reinterpret_cast<uint8_t *>(epi_smem) + EPI_WARPS * EPI_TILE_FLOATS * 4 + warp * H_TILE_BYTES;
            const CUtensorMap *pmap_h = second ? &map_h1 : &map_h0;
            auto fetch_h = [&](int c) {                        // block at tile column c (one lane issues)
                if (lane == 0) {
                    hb::mbar_expect_tx(&h_bar[warp], H_TILE_BYTES);
                    tma_load_2d(htile, pmap_h, n0 + c, mw, &h_bar[warp]);
                }
            };
            if (EPI == EPI_ACT_BWD && c_begin < c_end && n0 + c_begin < g.N && mw < g.M) {
                if (g.N - (n0 + c_begin) > 32 && c_begin + 32 < c_end) {       // pull the blocks after the first towards L2 meanwhile
                    const int row = mw + lane, n_lo = n0 + c_begin + 32;
                    if (row < g.M) {
                        const float *hrow = g.H + (size_t)row * g.ldh + n_lo;
                        const int bytes = min(c_end - c_begin - 32, g.N - n_lo) * 4;
                        for (int o = 0; o < bytes; o += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char *>(hrow) + o));
                    }
                }
                fetch_h(c_begin);
            }
            hb::mbar_wait(&acc_full[a], aph);
            tc_fence_after();
            const uint32_t tmem_acc = tmem_base + a * ACC_COLS + ((uint32_t)(quarter * 32) << 16);
            if constexpr (EPI != EPI_ATOMIC) {
                // Plain / bias / f / f' results leave through the TMA: the warp applies the tail in registers (lane = row,
                // as TMEM delivers it), writes its 32 x 32 block into a 128-byte-swizzled 4 KB tile with eight conflict-free
                // 16-byte stores per lane and hands the tile to one cp.async.bulk.tensor store - no transposing read-back, no
                // per-lane global stores, ragged edges clipped by the tensor map.
                uint8_t *stile = reinterpret_cast<uint8_t *>(epi_smem) + warp * 4096;
                const CUtensorMap *pmap_d = second ? &map_d1 : &map_d0;
                bool handed_back = false;
#pragma unroll 1
                for (int c = c_begin; c < c_end; c += 32) {
                    const int n = n0 + c;
                    if (n >= g.N || mw >= g.M) break;
                    float4 h4[8];
                    if (EPI == EPI_ACT_BWD) {                    // this lane's row of the block, chunk j at j ^ (lane % 8)
                        hb::mbar_wait(&h_bar[warp], h_phase);
                        h_phase ^= 1u;
#pragma unroll
                        for (int j = 0; j < 8; ++j) h4[j] = *reinterpret_cast<const float4 *>(htile + lane * 128 + ((j ^ (lane & 7)) << 4));
                        if (c + 32 < c_end && n + 32 < g.N) {    // next block's activations: in flight behind this block's work
                            fence_async_smem();                  // (the reads above before the async-proxy overwrite)
                            __syncwarp();
                            fetch_h(c + 32);
                        }
                    }
                    float bias_l = 0.0f;
                    if (EPI == EPI_BIAS || EPI == EPI_BIAS_ACT) bias_l = (n + lane < g.N) ? __ldg(g.bias + (size_t)(n + lane) * g.bias_stride) : 0.0f;
                    float v[32];
                    if (BN > 16) {
                        tmem_ld32(tmem_acc + (uint32_t)c, v);
                    } else {                                     // 16-wide tiles: the upper half of the block is clipped by the store
                        tmem_ld16(tmem_acc + (uint32_t)c, v);
#pragma unroll
                        for (int i = 16; i < 32; ++i) v[i] = 0.0f;
                    }
                    if (c + 32 >= c_end || n + 32 >= g.N) {      // last read of this accumulator: the MMA warp may reuse it
                        tc_fence_before();
                        if (lane == 0) {
                            if (PAIR) mbar_arrive_cluster(mapa_shared(hb::smem_u32(&acc_empty[a]), 0));
                            else hb::mbar_arrive(&acc_empty[a]);
                        }
                        handed_back = true;
                    }
                    if (EPI == EPI_BIAS || EPI == EPI_BIAS_ACT) {
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            float x = v[i] + __shfl_sync(0xffffffffu, bias_l, i);
                            if (EPI == EPI_BIAS_ACT) x = hb::act_fwd<ACT, false>(x);
                            v[i] = x;
                        }
                    } else if (EPI == EPI_ACT_BWD) {            // h = f(z): f'(z) from h
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float h[4] = {h4[j].x, h4[j].y, h4[j].z, h4[j].w};
#pragma unroll
                            for (int k = 0; k < 4; ++k) v[4 * j + k] *= hb::act_grad<ACT>(h[k]);
                        }
                    }
                    if ((g.N & 3) && n + 32 > g.N) {
                        // The TMA store writes whole 16-byte chunks: the chunk holding column N - 1 would also overwrite the
                        // columns behind it up to the next multiple of 4, which belong to the caller (the ones column
                        // behind an MLP's hidden activations).  A block whose ragged edge falls inside a chunk is stored
                        // per lane instead.
                        if (mw + lane < g.M) {
                            float *drow = g.D + (size_t)(mw + lane) * g.ldd + n;
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (n + j < g.N) drow[j] = v[j];
                        }
                        continue;
                    }
                    if (lane == 0) tma_store_wait_read();        // the previous block's store has read the tile
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 8; ++j)                  // 16-byte chunk j of row `lane` sits at chunk j ^ (lane % 8)
                        *reinterpret_cast<float4 *>(stile + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                            make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) tma_store_2d(pmap_d, n, mw, stile);
                }
                if (!handed_back) {
                    tc_fence_before();
                    if (lane == 0) {
                        if (PAIR) mbar_arrive_cluster(mapa_shared(hb::smem_u32(&acc_empty[a]), 0));
                        else hb::mbar_arrive(&acc_empty[a]);
                    }
                }
                continue;
            }
#pragma unroll 1
            for (int c = c_begin; c < c_end; c += 32) {
                const int n = n0 + c;
                if (n >= g.N || mw >= g.M) break;
                const int ncols = min(32, g.N - n), nrows = min(32, g.M - mw);
                const bool col_ok = lane < ncols;
                // readout mapping: 8 lanes x float4 per row, 4 rows per instruction (128-byte row segments)
                const int rr = lane >> 3, c4 = (lane & 7) * 4;
                const bool fast = (ncols == 32) && ((g.ldd & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.D) & 15u) == 0) &&
                                  (EPI != EPI_ACT_BWD || (((g.ldh & 3) == 0) && ((reinterpret_cast<uintptr_t>(g.H) & 15u) == 0)));
                float4 h4[8];                                  // f': forward activations, all loads in flight early
                float b4[4] = {0.f, 0.f, 0.f, 0.f};           // forward: this lane's four biases
                if (fast) {
                    if (EPI == EPI_ACT_BWD) {
#pragma unroll
                        for (int it = 0; it < 8; ++it) {
                            const int r = it * 4 + rr;
                            h4[it] = (r < nrows) ? __ldg(reinterpret_cast<const float4 *>(g.H + (size_t)(mw + r) * g.ldh + n + c4))
                                                 : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
                    }
                    if (EPI == EPI_BIAS || EPI == EPI_BIAS_ACT) {
#pragma unroll
                        for (int k = 0; k < 4; ++k) b4[k] = __ldg(g.bias + (size_t)(n + c4 + k) * g.bias_stride);
                    }
                }
                float v[32];
                tmem_ld16(tmem_acc + (uint32_t)c, v);
                if (BN > 16) tmem_ld16(tmem_acc + (uint32_t)(c + 16), v + 16);
                // transpose through the warp's padded tile: written with lane = row, read with lane = column group
#pragma unroll
                for (int i = 0; i < 32; ++i) tile[lane * 33 + i] = v[i];
                __syncwarp();
                if (fast) {
#pragma unroll
                    for (int it = 0; it < 8; ++it) {
                        const int r = it * 4 + rr;
                        if (r < nrows) {
                            const float *tt = tile + r * 33 + c4;
                            float x[4] = {tt[0], tt[1], tt[2], tt[3]};
                            if (EPI == EPI_BIAS || EPI == EPI_BIAS_ACT) {
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    x[k] += b4[k];
                                    if (EPI == EPI_BIAS_ACT) x[k] = hb::act_fwd<ACT, false>(x[k]);
                                }
                            } else if (EPI == EPI_ACT_BWD) {
                                const float h[4] = {h4[it].x, h4[it].y, h4[it].z, h4[it].w};
#pragma unroll
                                for (int k = 0; k < 4; ++k) x[k] *= hb::act_grad<ACT>(h[k]);
                            }
                            float *dst = g.D + (size_t)(mw + r) * g.ldd + n + c4;
                            if (EPI == EPI_ATOMIC) {      // one 16-byte vector reduction per lane (sm_90+)
                                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(x[0]), "f"(x[1]),
                                             "f"(x[2]), "f"(x[3])
                                             : "memory");
                            } else {
                                *reinterpret_cast<float4 *>(dst) = make_float4(x[0], x[1], x[2], x[3]);
                            }
                        }
                    }
                } else if (col_ok) {                           // ragged edge / unaligned: one column per lane
                    const float bias = (EPI == EPI_BIAS || EPI == EPI_BIAS_ACT) ? __ldg(g.bias + (size_t)(n + lane) * g.bias_stride) : 0.0f;
                    for (int r = 0; r < nrows; ++r) {
                        float x = tile[r * 33 + lane];
                        if (EPI == EPI_BIAS || EPI == EPI_BIAS_ACT) {
                            x += bias;
                            if (EPI == EPI_BIAS_ACT) x = hb::act_fwd<ACT, false>(x);
                        } else if (EPI == EPI_ACT_BWD) {
                            x *= hb::act_grad<ACT>(__ldg(g.H + (size_t)(mw + r) * g.ldh + n + lane));
                        }
                        float *dst = g.D + (size_t)(mw + r) * g.ldd + n + lane;
                        if (EPI == EPI_ATOMIC) atomicAdd(dst, x);
                        else *dst = x;
                    }
                }
                __syncwarp();
            }
            // every tcgen05.ld of this warp has completed (tcgen05.wait::ld inside tmem_ld16): hand the accumulator back
            tc_fence_before();
            if (lane == 0) {
                if (PAIR) mbar_arrive_cluster(mapa_shared(hb::smem_u32(&acc_empty[a]), 0));   // the leader's barrier
                else hb::mbar_arrive(&acc_empty[a]);
            }
        }
    }
    if (EPI != EPI_ATOMIC && warp < EPI_WARPS && lane == 0) tma_store_wait_all();      // this warp's last stores have left its tile
    __syncwarp();                    // single-lane roles (producer, MMA issuer) rejoin their warps before the aligned barrier
    tc_fence_before();
    if (PAIR) cluster_sync();        // the leader's MMAs read the peer's shared memory: leave together
    else __syncthreads();
    if (warp == MMA_WARP) {
        if (PAIR) tmem_dealloc_pair(tmem_base, TMEM_COLS);
        else tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// ---- host side --------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// 2-D fp32 tensor map over a row-major matrix [rows, cols] with leading dimension ld (floats).
// K-major operand: inner = contraction (cols), box = 32 x box_rows.
// MN-major operand: the matrix is [K rows, MN cols]; inner = MN (cols), box = 32 x 32.
int make_map(CUtensorMap *map, const float *base, int rows, int cols, int ld, int box_inner, int box_outer,
             bool mn_major) {
    EncodeTiledFn enc = encode_fn();
    if (!enc) {
        hb::set_error("cuTensorMapEncodeTiled is not available from this driver");
        return HB_ERR_UNSUPPORTED;
    }
    if ((reinterpret_cast<uintptr_t>(base) & 15u) || (ld % 4) != 0) {
        hb::set_error("TMA operand needs a 16-byte aligned base and a leading dimension that is a multiple of 4 floats "
                      "(base=%p ld=%d)", (const void *)base, ld);
        return HB_ERR_BAD_ARG;
    }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE,
                     mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        hb::set_error("cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%d box=%dx%d", (int)r, rows, cols, ld,
                      box_inner, box_outer);
        return HB_ERR_CUDA;
    }
    return HB_OK;
}

// tensor maps + tile list of one problem
template <int BN, bool A_MN, bool B_MN, int EPI, bool PAIR>
int setup_problem(const hb_gemm_desc *d, CUtensorMap *ma, CUtensorMap *mb, CUtensorMap *md, CUtensorMap *mh, GemmArgs *gp,
                  int auto_splits) {
    constexpr int BN_CTA = PAIR ? BN / 2 : BN;
    int rc;
    *mh = CUtensorMap{};
    if (EPI == EPI_ACT_BWD) {     // forward activations, read in the same 32 x 32 boxes as the output is written
        rc = make_map(mh, d->H, d->M, d->N, d->ldh, 32, 32, false);
        if (rc) return rc;
    }
    if (EPI != EPI_ATOMIC) {      // the output leaves through TMA stores of 32 x 32 boxes (clipped at M, N)
        rc = make_map(md, d->D, d->M, d->N, d->ldd, 32, 32, false);
        if (rc) return rc;
    } else {
        *md = CUtensorMap{};
    }
    // A: K-major  -> memory [M, K] ;  MN-major -> memory [K, M]
    rc = A_MN ? make_map(ma, d->A, d->K, d->M, d->lda, 32, 32, true) : make_map(ma, d->A, d->M, d->K, d->lda, BK, BM, false);
    if (rc) return rc;
    rc = B_MN ? make_map(mb, d->B, d->K, d->N, d->ldb, 32, 32, true) : make_map(mb, d->B, d->N, d->K, d->ldb, BK, BN_CTA, false);
    if (rc) return rc;
    GemmArgs &g = *gp;
    g.M = d->M, g.N = d->N, g.K = d->K;
    const int kb_total = (d->K + BK - 1) / BK;
    int splits = d->split_k > 0 ? d->split_k : 1;
    if (d->split_k == 0 && EPI == EPI_ATOMIC) splits = auto_splits;      // chosen for the launch as a whole (launch())
    if (splits > kb_total) splits = kb_total > 0 ? kb_total : 1;
    g.kb_per_split = (kb_total + splits - 1) / splits;
    splits = g.kb_per_split > 0 ? (kb_total + g.kb_per_split - 1) / g.kb_per_split : 1;
    g.D = d->D, g.ldd = d->ldd, g.bias = d->bias, g.bias_stride = d->bias_stride, g.H = d->H, g.ldh = d->ldh;
    g.snake = hb::g_gemm_snake;
    const int rows_per_tile = PAIR ? 2 * BM : BM;
    const int tiles_m = (d->M + rows_per_tile - 1) / rows_per_tile;
    g.tiles_m = tiles_m, g.tiles_n = (d->N + BN - 1) / BN, g.splits = splits;
    g.total_tiles = tiles_m * g.tiles_n * splits;
    return HB_OK;
}

// d1 may be null (one problem)
template <int BN, bool A_MN, bool B_MN, int EPI, bool PAIR, int ACT>
int launch(const hb_gemm_desc *d, const hb_gemm_desc *d1, cudaStream_t st) {
    constexpr size_t SMEM = smem_bytes_for<BN, PAIR, EPI>();
    static bool attr = false;
    auto kern = gemm_tf32_kernel<BN, A_MN, B_MN, EPI, PAIR, ACT>;
    if (!attr) {
        HB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM));
        attr = true;
    }
    alignas(64) CUtensorMap ma, mb, ma1, mb1, md, md1, mh, mh1;
    GemmArgs g, g1;
    // Automatic split-K (weight gradients): k ranges of about equal length over BOTH problems of the launch, about two
    // rounds of tile jobs over the SMs (SM pairs in pair mode) - one round when the outputs have only a few tiles, where
    // the atomic accumulation of a second round costs more than the shorter k ranges save.
    int auto_splits[2] = {1, 1};
    {
        const hb_gemm_desc *ds[2] = {d, d1};
        const int count = d1 ? 2 : 1, slots = PAIR ? hb::sm_count() / 2 : hb::sm_count(), rows = PAIR ? 2 * BM : BM;
        long long tiles_all = 0, work = 0;
        for (int i = 0; i < count; ++i) {
            const long long tiles = (long long)((ds[i]->M + rows - 1) / rows) * ((ds[i]->N + BN - 1) / BN);
            tiles_all += tiles, work += tiles * ((ds[i]->K + BK - 1) / BK);
        }
        const long long jobs = (tiles_all <= 2 * count ? 1 : 2) * slots;
        const double target = (double)work / (double)jobs;               // k-blocks per tile job
        for (int i = 0; i < count; ++i) {
            const int sp = (int)((double)((ds[i]->K + BK - 1) / BK) / (target > 1.0 ? target : 1.0) + 0.5);
            auto_splits[i] = sp < 1 ? 1 : sp;
        }
    }
    if (int rc = setup_problem<BN, A_MN, B_MN, EPI, PAIR>(d, &ma, &mb, &md, &mh, &g, auto_splits[0])) return rc;
    if (d1) {
        if (int rc = setup_problem<BN, A_MN, B_MN, EPI, PAIR>(d1, &ma1, &mb1, &md1, &mh1, &g1, auto_splits[1])) return rc;
    } else {
        ma1 = ma, mb1 = mb, md1 = md, mh1 = mh, g1 = g;
        g1.total_tiles = 0;
    }
    const int total_tiles = g.total_tiles + g1.total_tiles;
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute at[2];
    int nat = 0;
    at[nat].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[nat].val.programmaticStreamSerializationAllowed = hb::g_gemm_pdl ? 1 : 0;
    ++nat;
    int grid;
    if (PAIR) {
        const int pairs = hb::sm_count() / 2;
        grid = 2 * (total_tiles < pairs ? total_tiles : pairs);
        at[nat].id = cudaLaunchAttributeClusterDimension;
        at[nat].val.clusterDim.x = 2, at[nat].val.clusterDim.y = 1, at[nat].val.clusterDim.z = 1;
        ++nat;
    } else {
        grid = total_tiles < hb::sm_count() ? total_tiles : hb::sm_count();
    }
    cfg.gridDim = dim3(grid), cfg.blockDim = dim3(GEMM_THREADS), cfg.dynamicSmemBytes = SMEM, cfg.stream = st;
    cfg.attrs = at, cfg.numAttrs = nat;
    HB_CUDA(cudaLaunchKernelEx(&cfg, kern, ma, mb, g, ma1, mb1, g1, md, md1, mh, mh1));
    HB_CHECK_LAUNCH("gemm_tf32_kernel");
    return HB_OK;
}

int g_gemm_pair = 1;          // "gemm_pair" option: 0 disables the 2-CTA kernels

template <int BN, bool A_MN, bool B_MN, int EPI, int ACT = HB_ACT_ELU>
int launch_auto(const hb_gemm_desc *d, const hb_gemm_desc *d1, cudaStream_t st) {
    if constexpr (BN == 256) {
        if (g_gemm_pair && d->M > BM && (!d1 || d1->M > BM)) return launch<BN, A_MN, B_MN, EPI, true, ACT>(d, d1, st);
    }
    return launch<BN, A_MN, B_MN, EPI, false, ACT>(d, d1, st);
}

template <int BN, int EPI>
int dispatch_major(const hb_gemm_desc *d, const hb_gemm_desc *d1, cudaStream_t st) {
    if (!d->a_mn_major && !d->b_mn_major) return launch_auto<BN, false, false, EPI>(d, d1, st);
    if (d->b_mn_major) {
        if constexpr (BN < 128) {      // only N <= 64 picks these widths, and check_desc refuses an MN-major B there: not built
            hb::set_error("hb_gemm_tf32: MN-major B needs N > 64");
            return HB_ERR_BAD_ARG;
        } else {
            return d->a_mn_major ? launch_auto<BN, true, true, EPI>(d, d1, st) : launch_auto<BN, false, true, EPI>(d, d1, st);
        }
    }
    hb::set_error("hb_gemm_tf32: A MN-major with B K-major is not instantiated");
    return HB_ERR_UNSUPPORTED;
}

// The activation epilogues: ELU in every layout, the other activations in the layout of their GEMM in an MLP - the forward
// pass (A and B K-major) and the data gradient (A K-major, B = the weights MN-major).  An MN-major B has N > 64
// (check_desc), so the data gradient never runs on tiles narrower than 128.
template <int BN, int EPI>
int dispatch_act(const hb_gemm_desc *d, const hb_gemm_desc *d1, cudaStream_t st) {
    if (d->activation == HB_ACT_ELU) return dispatch_major<BN, EPI>(d, d1, st);
    constexpr bool B_MN = EPI == EPI_ACT_BWD;
    if (d->a_mn_major || (d->b_mn_major != 0) != B_MN) {
        hb::set_error("hb_gemm_tf32: activation %d is built for %s only", d->activation,
                      B_MN ? "A K-major with B MN-major (data gradient)" : "A and B K-major (forward)");
        return HB_ERR_UNSUPPORTED;
    }
    if constexpr (B_MN && BN < 128) {
        hb::set_error("hb_gemm_tf32: MN-major B needs N > 64");
        return HB_ERR_BAD_ARG;
    } else {
        HB_ACT_DISPATCH(d->activation, return (launch_auto<BN, false, B_MN, EPI, ACT>(d, d1, st)));
    }
}

template <int BN>
int dispatch_epi(const hb_gemm_desc *d, const hb_gemm_desc *d1, cudaStream_t st) {
    switch (d->epilogue) {
        case HB_EPI_STORE: return dispatch_major<BN, EPI_STORE>(d, d1, st);
        case HB_EPI_BIAS: return dispatch_major<BN, EPI_BIAS>(d, d1, st);
        case HB_EPI_BIAS_ACT: return dispatch_act<BN, EPI_BIAS_ACT>(d, d1, st);
        case HB_EPI_ACT_BWD: return dispatch_act<BN, EPI_ACT_BWD>(d, d1, st);
        case HB_EPI_ATOMIC_ADD: return dispatch_major<BN, EPI_ATOMIC>(d, d1, st);
    }
    hb::set_error("hb_gemm_tf32: unknown epilogue %d", d->epilogue);
    return HB_ERR_BAD_ARG;
}

// ---- 3xTF32: fp32-grade products on the TF32 tensor cores ---------------------------------------------
// x = hi + lo with hi = x rounded to TF32 (10 explicit mantissa bits) and lo = x - hi (exact in fp32, |lo| <= 2^-11 |x|):
//   a * b  =  a_hi b_hi + a_lo b_hi + a_hi b_lo  (+ a_lo b_lo, dropped: 2^-22 relative)
// The three partial products are ONE longer contraction: A' = [A_hi | A_lo | A_hi], B' = [B_hi | B_hi | B_lo] along K,
// so the tcgen05 kernel above runs unchanged (fused epilogues, split-K, pair mode) on K' = 3 K with the fp32
// accumulator in TMEM summing all three.  The split is a pre-pass into a caller-supplied workspace.
__device__ __forceinline__ float tf32_round(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}
// K-major operand [rows, K] (leading dimension ld) -> [rows, 3 * kp], kp = K rounded up to 4, zero padded
__global__ void __launch_bounds__(256)
split3_kmajor_kernel(const float *__restrict__ src, int ld, long long rows, int K, int kp, float *__restrict__ dst, int second_is_lo) {
    const long long quads = (long long)(kp >> 2);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * quads) return;
    const long long r = i / quads;
    const int c = (int)(i - r * quads) * 4;
    float x[4], hi[4], lo[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        x[k] = (c + k < K) ? __ldg(src + (size_t)r * ld + c + k) : 0.0f;
        hi[k] = tf32_round(x[k]), lo[k] = x[k] - hi[k];
    }
    float *row = dst + (size_t)r * 3 * kp + c;
    const float4 h4 = make_float4(hi[0], hi[1], hi[2], hi[3]), l4 = make_float4(lo[0], lo[1], lo[2], lo[3]);
    *reinterpret_cast<float4 *>(row) = h4;
    *reinterpret_cast<float4 *>(row + kp) = second_is_lo ? l4 : h4;
    *reinterpret_cast<float4 *>(row + 2 * kp) = second_is_lo ? h4 : l4;
}
// MN-major operand [K, cols] (leading dimension ld) -> [3 * kp, ldd]: the three parts stacked along K at the same
// pitch kp as a K-major partner (rows K..kp-1 of each part are zero)
__global__ void __launch_bounds__(256)
split3_mnmajor_kernel(const float *__restrict__ src, int ld, long long K, long long kp, int cols, float *__restrict__ dst, int ldd,
                      int second_is_lo) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= kp * ldd) return;
    const long long k = i / ldd;
    const int c = (int)(i - k * ldd);
    const float x = (c < cols && k < K) ? __ldg(src + (size_t)k * ld + c) : 0.0f;
    const float hi = tf32_round(x), lo = x - hi;
    dst[(size_t)k * ldd + c] = hi;
    dst[(size_t)(kp + k) * ldd + c] = second_is_lo ? lo : hi;
    dst[(size_t)(2 * kp + k) * ldd + c] = second_is_lo ? hi : lo;
}

inline long long pad4ll(long long v) { return (v + 3) / 4 * 4; }
long long split3_floats(long long rows, long long K, bool mn_major) {
    return mn_major ? 3 * pad4ll(K) * pad4ll(rows) : rows * 3 * pad4ll(K);
}

int gemm_tf32_dispatch(const hb_gemm_desc *d, cudaStream_t st);

// The tensor core adds each instruction's products (8 along K) into the TMEM accumulator with truncation, about
// 3e-8 relative per step (measured: 1.2e-5 over the ~400 steps of a K' = 3 * 1052 contraction, where exact accumulation of
// the same split operands gives 5e-7).  The fp32-grade mode therefore keeps accumulation chains SHORT: the contraction
// is cut into splits of CHAIN_KB k-blocks (16 accumulation steps), every split adds its partial tile to D with
// round-to-nearest fp32 reductions (red.global.add), and bias / f / f' run as a separate pass over D (libm accuracy).
constexpr int CHAIN_KB = 4;

template <int ACT>
__global__ void __launch_bounds__(256)
epilogue_inplace_kernel(float *__restrict__ D, int ldd, long long M, int N, int epi, const float *__restrict__ bias, int bias_stride,
                        const float *__restrict__ H, int ldh) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * N) return;
    const long long m = i / N;
    const int n = (int)(i - m * N);
    float x = D[(size_t)m * ldd + n];
    if (epi == EPI_BIAS || epi == EPI_BIAS_ACT) {
        x += __ldg(bias + (size_t)n * bias_stride);
        if (epi == EPI_BIAS_ACT) x = hb::act_fwd<ACT, true>(x);
    } else if (epi == EPI_ACT_BWD) {
        x *= hb::act_grad<ACT>(__ldg(H + (size_t)m * ldh + n));
    }
    D[(size_t)m * ldd + n] = x;
}

int gemm_3xtf32(const hb_gemm_desc *d, cudaStream_t st) {
    const long long fa = split3_floats(d->M, d->K, d->a_mn_major != 0), fb = split3_floats(d->N, d->K, d->b_mn_major != 0);
    HB_REQUIRE(d->workspace && hb::aligned16(d->workspace) && d->workspace_floats >= fa + fb,
               "hb_gemm_tf32: HB_GEMM_3XTF32 needs a 16-byte aligned workspace of %lld floats (hb_gemm_workspace_floats), got %lld",
               fa + fb, (long long)d->workspace_floats);
    const long long kp = pad4ll(d->K);
    HB_REQUIRE(3 * kp < (1ll << 31), "hb_gemm_tf32: contraction too long for the 3xTF32 form");
    float *wa = d->workspace, *wb = d->workspace + fa;
    hb_gemm_desc e = *d;
    e.precision = HB_GEMM_TF32, e.A = wa, e.B = wb, e.K = (int)(3 * kp);
    auto split = [&](const float *src, int ld, int rows, bool mn, float *dst, int second_is_lo, int &ld_out) {
        if (mn) {
            ld_out = (int)pad4ll(rows);
            const long long total = kp * ld_out;
            split3_mnmajor_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, ld, d->K, kp, rows, dst, ld_out, second_is_lo);
        } else {
            ld_out = (int)(3 * kp);
            const long long total = (long long)rows * (kp >> 2);
            split3_kmajor_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, ld, rows, d->K, (int)kp, dst, second_is_lo);
        }
    };
    split(d->A, d->lda, d->M, d->a_mn_major != 0, wa, 1, e.lda);       // A' = [hi | lo | hi]
    HB_CHECK_LAUNCH("split3 (A)");
    split(d->B, d->ldb, d->N, d->b_mn_major != 0, wb, 0, e.ldb);       // B' = [hi | hi | lo]
    HB_CHECK_LAUNCH("split3 (B)");
    // short accumulation chains: split-K with fp32 reductions into D, fused tails moved to a second pass
    const int kb_total = (e.K + BK - 1) / BK;
    e.split_k = (kb_total + CHAIN_KB - 1) / CHAIN_KB;
    e.epilogue = HB_EPI_ATOMIC_ADD;
    e.bias = nullptr, e.H = nullptr;
    if (d->epilogue != HB_EPI_ATOMIC_ADD)                               // D = ..., not D += ...: start from zero
        HB_CUDA(cudaMemset2DAsync(d->D, (size_t)d->ldd * 4, 0, (size_t)d->N * 4, (size_t)d->M, st));
    if (int rc = gemm_tf32_dispatch(&e, st)) return rc;
    if (d->epilogue == HB_EPI_BIAS || d->epilogue == HB_EPI_BIAS_ACT || d->epilogue == HB_EPI_ACT_BWD) {
        const long long total = (long long)d->M * d->N;
        HB_ACT_DISPATCH(d->activation, (epilogue_inplace_kernel<ACT><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
            d->D, d->ldd, d->M, d->N, d->epilogue, d->bias, d->bias_stride, d->H, d->ldh)));
        HB_CHECK_LAUNCH("epilogue_inplace_kernel");
    }
    return HB_OK;
}

}  // namespace

extern "C" int hb_gemm_set_pair_mode(int on) {
    g_gemm_pair = on;
    return HB_OK;
}

namespace {
static int check_desc(const hb_gemm_desc *d) {
    HB_REQUIRE(d && d->A && d->B && d->D, "hb_gemm_tf32: null descriptor/operand");
    HB_REQUIRE(d->M > 0 && d->N > 0 && d->K > 0, "hb_gemm_tf32: empty problem %dx%dx%d", d->M, d->N, d->K);
    HB_REQUIRE((d->epilogue != HB_EPI_BIAS && d->epilogue != HB_EPI_BIAS_ACT) || d->bias, "hb_gemm_tf32: bias epilogue without bias");
    HB_REQUIRE(d->epilogue != HB_EPI_ACT_BWD || d->H, "hb_gemm_tf32: activation backward epilogue without activations");
    HB_REQUIRE(d->activation >= 0 && d->activation < HB_ACT_COUNT, "hb_gemm_tf32: unknown activation %d (hb_activation)", d->activation);
    HB_REQUIRE(d->split_k <= 1 || d->epilogue == HB_EPI_ATOMIC_ADD, "hb_gemm_tf32: split-K needs the atomic epilogue");
    HB_REQUIRE(!d->b_mn_major || d->N > 64, "hb_gemm_tf32: MN-major B needs N > 64 (32-wide TMA boxes per 128-byte swizzle row)");
    return HB_OK;
}

// tile width of a problem: 16 / 64 / 128 / 256
static int pick_tile_n(const hb_gemm_desc *d) {
    // the widest UMMA N that does not waste more than half a tile ...
    if (d->N <= 16) return 16;
    if (d->N <= 64) return 64;
    if (d->N <= 128 || d->tile_n == 128) return 128;
    if (d->tile_n == 0 && d->epilogue != HB_EPI_ATOMIC_ADD) {
        // ... unless 128-wide tiles balance better over the SMs: rounds of the persistent tile loop x operand
        // bytes per tile (proportional to 128 + BN); e.g. M = 24576, N = 256 is 192 tiles = 2 rounds of 148 SMs at
        // BN = 256 but 3 rounds of half-size tiles at BN = 128
        const long long sms = hb::sm_count(), tm = (d->M + BM - 1) / BM;
        const long long t256 = tm * ((d->N + 255) / 256), t128 = tm * ((d->N + 127) / 128);
        long long c256 = ((t256 + sms - 1) / sms) * (128 + 256);
        const long long c128 = ((t128 + sms - 1) / sms) * (128 + 128);
        if (g_gemm_pair && d->M > BM) {      // 256-row pair tiles: half of B per CTA
            const long long tp = ((d->M + 2 * BM - 1) / (2 * BM)) * ((d->N + 255) / 256), pairs = sms / 2;
            c256 = ((tp + pairs - 1) / pairs) * (128 + 128);
        }
        if (c128 < c256) return 128;
    }
    return 256;
}

static int dispatch_tile(int bn, const hb_gemm_desc *d, const hb_gemm_desc *d1, cudaStream_t st) {
    switch (bn) {
        case 16: return dispatch_epi<16>(d, d1, st);
        case 64: return dispatch_epi<64>(d, d1, st);
        case 128: return dispatch_epi<128>(d, d1, st);
        default: return dispatch_epi<256>(d, d1, st);
    }
}

int gemm_tf32_dispatch(const hb_gemm_desc *d, cudaStream_t st) {
    if (int rc = check_desc(d)) return rc;
    return dispatch_tile(pick_tile_n(d), d, nullptr, st);
}

int gemm_tf32_dispatch_grouped(const hb_gemm_desc *d0, const hb_gemm_desc *d1, cudaStream_t st) {
    if (int rc = check_desc(d0)) return rc;
    if (int rc = check_desc(d1)) return rc;
    HB_REQUIRE(d0->epilogue == d1->epilogue && d0->activation == d1->activation && d0->a_mn_major == d1->a_mn_major &&
                   d0->b_mn_major == d1->b_mn_major,
               "hb_gemm_tf32_grouped: both problems must share epilogue and operand layouts");
    // one tile width for both: with two problems in flight there are enough tiles for the wide one whenever both are wide
    int bn0 = pick_tile_n(d0), bn1 = pick_tile_n(d1);
    if ((bn0 >= 128) != (bn1 >= 128) || (bn0 < 128 && bn0 != bn1)) {       // too different to share a kernel: two launches
        if (int rc = dispatch_tile(bn0, d0, nullptr, st)) return rc;
        return dispatch_tile(bn1, d1, nullptr, st);
    }
    const int bn = bn0 > bn1 ? bn0 : bn1;
    if (bn == 256 && (d0->N <= 128 || d1->N <= 128)) return dispatch_tile(128, d0, d1, st);
    return dispatch_tile(bn, d0, d1, st);
}
}  // namespace

extern "C" int64_t hb_gemm_workspace_floats(const hb_gemm_desc *d) {
    if (!d || d->precision != HB_GEMM_3XTF32) return 0;
    return split3_floats(d->M, d->K, d->a_mn_major != 0) + split3_floats(d->N, d->K, d->b_mn_major != 0);
}

extern "C" int hb_gemm_tf32_grouped(const hb_gemm_desc *d0, const hb_gemm_desc *d1, void *stream) {
    HB_REQUIRE(d0 && d1, "hb_gemm_tf32_grouped: null descriptor");
    if (d0->precision != HB_GEMM_TF32 || d1->precision != HB_GEMM_TF32) {      // the fp32-grade mode has its own passes
        if (int rc = hb_gemm_tf32(d0, stream)) return rc;
        return hb_gemm_tf32(d1, stream);
    }
    return gemm_tf32_dispatch_grouped(d0, d1, (cudaStream_t)stream);
}

extern "C" int hb_gemm_tf32(const hb_gemm_desc *d, void *stream) {
    HB_REQUIRE(d, "hb_gemm_tf32: null descriptor");
    HB_REQUIRE(d->precision == HB_GEMM_TF32 || d->precision == HB_GEMM_3XTF32, "hb_gemm_tf32: unknown precision %d", d->precision);
    if (d->precision == HB_GEMM_3XTF32) {
        HB_REQUIRE(d->A && d->B && d->D && d->M > 0 && d->N > 0 && d->K > 0, "hb_gemm_tf32: null operand / empty problem");
        HB_REQUIRE(d->activation >= 0 && d->activation < HB_ACT_COUNT, "hb_gemm_tf32: unknown activation %d (hb_activation)",
                   d->activation);
        return gemm_3xtf32(d, (cudaStream_t)stream);
    }
    return gemm_tf32_dispatch(d, (cudaStream_t)stream);
}
