// Micro-benchmark (go / no-go for a trunk with the activations as the N operand): the weight stream and the MMA schedule of a
// CTA pair that alternates between two independent groups of positions layer by layer (as net_pp_kernel.cuh), but with the
// operand roles swapped -- A = a 128 x 16 weight block (M = the 128 output channels), B = the group's activation rows
// (N = rows of this CTA, any multiple of 16) -- so that an MMA costs N / 2 cycles instead of 64 cycles per 128-row tile
// (tools/micro/mma_shapes.cu).  cta_group::1: every CTA streams ALL weights once per group = 576 KB per layer; the question is
// whether 148 SMs sustain that through a deep ring (7 x 16 KiB) next to the tensor pipe's operand reads, unicast or with the
// two CTAs of a pair loading half a stage each and multicasting it.  The epilogue is a stub (waits `epi_delay` cycles).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/nt_skeleton tools/micro/nt_skeleton.cu
#include <cstdlib>

#include "../../ultimate-tictactoe-alphazero_b200/csrc/tc_common.cuh"

using namespace uttt::tcx;

// cta_group::1 MMA and commits (the library's trunks issue cta_group::2 MMAs only)
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at the same shared-memory offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mcast(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(mask)
                 : "memory");
}

constexpr int LEAD = 11;
constexpr int BLOCK_BYTES = 4096, STAGE_BLOCKS = 4, STAGE_BYTES = STAGE_BLOCKS * BLOCK_BYTES, STAGES = 7;
constexpr int SPL = 72 / STAGE_BLOCKS;                  // weight stages per layer (+ 1 bias stage)
constexpr int LAYERS = 32;
constexpr int EPI_WARPS = 16, THREADS = (EPI_WARPS + 3) * 32;
constexpr int PR0 = 233, PR1 = 185;                     // rows per channel panel (= 1 mod 8: conflict-free transposed stores)
constexpr int A0_BYTES = 16 * PR0 * 16, A1_BYTES = 16 * PR1 * 16;
constexpr int CONST_ROWS = 208, CONST_BYTES = 2 * CONST_ROWS * 16;
constexpr int RING_OFF = (A0_BYTES + A1_BYTES + CONST_BYTES + 1023) / 1024 * 1024;
constexpr int BAR_OFF = RING_OFF + STAGES * STAGE_BYTES;
constexpr int SMEM_BYTES = BAR_OFF + 256;
static_assert(SMEM_BYTES <= 232448, "shared memory");

template <bool MCAST>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
nt_skeleton(const uint8_t* __restrict__ wq, const uint8_t* __restrict__ wbias, int N0, int N1, int epi_delay, long long* out) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank(), peer = rank ^ 1u;
    const uint32_t base = smem_u32(smem);
    const uint32_t sAct[2] = {base, base + A0_BYTES};
    const uint32_t panel[2] = {PR0 * 16, PR1 * 16};
    const uint32_t sConst = base + A0_BYTES + A1_BYTES, sRing = base + RING_OFF, bar = base + BAR_OFF;
    const uint32_t bar_full = bar, bar_empty = bar + 8 * STAGES, bar_accum = bar + 16 * STAGES, bar_act = bar_accum + 16;
    uint32_t* holder = reinterpret_cast<uint32_t*>(smem + BAR_OFF + 16 * STAGES + 32);
    const int N[2] = {N0, N1};
    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; i++) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, MCAST ? 4 : 2); }
        for (int g = 0; g < 2; g++) { mbar_init(bar_accum + 8 * g, 1); mbar_init(bar_act + 8 * g, EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == EPI_WARPS + 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(holder)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = threadIdx.x; i < RING_OFF / 16; i += THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem = *holder;

    if (warp < EPI_WARPS) {
        // stub epilogue: input "ready", then per layer and group: accumulator ready -> epi_delay cycles -> output published
        if (lane == 0) { mbar_arrive(bar_act); mbar_arrive(bar_act + 8); }
        for (int layer = 0; layer < LAYERS; layer++)
            for (int g = 0; g < 2; g++) {
                mbar_wait_spin<false>(bar_accum + 8 * g, (uint32_t)(layer & 1));
                tc_fence_after();
                float v[16];
                tmem_ld16(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(g * 256), v);
                tmem_ld_wait();
                long long t0 = clock64();
                while (clock64() - t0 < epi_delay) {}
                if (v[0] == 12345.f) out[200] = 1;
                tc_fence_before();
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_act + 8 * g);
            }
    } else if (warp == EPI_WARPS) {
        // weight producer: per layer and group one bias block + SPL stages (MCAST: this rank loads its half for both CTAs)
        int gn = 0;
        for (int layer = 0; layer < LAYERS; layer++)
            for (int g = 0; g < 2; g++)
                for (int st = 0; st <= SPL; st++, gn++) {
                    const int slot = gn % STAGES;
                    const uint32_t par = (uint32_t)((gn / STAGES) & 1);
                    mbar_wait(bar_empty + 8 * slot, par ^ 1u);
                    if (lane == 0) {
                        const uint8_t* src = st == 0 ? wbias + (size_t)layer * BLOCK_BYTES : wq + ((size_t)layer * SPL + st - 1) * STAGE_BYTES;
                        const uint32_t bytes = st == 0 ? BLOCK_BYTES : STAGE_BYTES;
                        mbar_expect_tx(bar_full + 8 * slot, bytes);
                        if (MCAST) {
                            const uint32_t half = bytes / 2;
                            asm volatile(
                                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
                                    sRing + slot * STAGE_BYTES + rank * half),
                                "l"(src + rank * half), "r"(half), "r"(bar_full + 8 * slot), "h"((uint16_t)3)
                                : "memory");
                        } else {
                            bulk_g2s(sRing + slot * STAGE_BYTES, src, bytes, bar_full + 8 * slot);
                        }
                    }
                    __syncwarp();
                }
    } else {
        // issuer of group g: A = weight block (M = 128 output channels, K = 16), B = the group's rows at the tap's shift
        const int g = warp - (EPI_WARPS + 1);
        const bool leader = elect_one();
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N[g] >> 3) << 17) | ((128u >> 4) << 24);
        const uint64_t b_desc = make_desc(sAct[g] + LEAD * 16, panel[g], 128);
        const uint64_t c_desc = make_desc(sConst, CONST_ROWS * 16, 128);
        const uint64_t a_desc = make_desc(sRing, 2048, 128);
        const uint32_t tmem_d = tmem + (uint32_t)(g * 256);
        const int panel16 = (int)(panel[g] / 16);
        // every issuer walks ALL stages in ring order (waits, and releases with a commit), but issues MMAs only for its own
        // group: a consumer that skipped the other group's stages would alias the barrier parities two ring turns apart
        int gn = 0;
        for (int layer = 0; layer < LAYERS; layer++) {
#pragma unroll 1
            for (int gg = 0; gg < 2; gg++) {
                const bool mine = gg == g;
                if (mine) {
                    mbar_wait_spin<false>(bar_act + 8 * g, (uint32_t)(layer & 1));
                    tc_fence_after();
                    if (g == 0 && leader && blockIdx.x == 0) out[layer] = clock64();
                }
#pragma unroll 1
                for (int st = 0; st <= SPL; st++, gn++) {
                    const int slot = gn % STAGES;
                    const uint32_t par = (uint32_t)((gn / STAGES) & 1);
                    mbar_wait_spin<false>(bar_full + 8 * slot, par);
                    tc_fence_after();
                    if (leader) {
                        if (mine) {
                            const uint64_t a_st = a_desc + (uint64_t)(uint32_t)(slot * (STAGE_BYTES / 16));
                            if (st == 0) {
                                umma_bf16(tmem_d, a_st, c_desc, idesc, 0u);
                            } else {
#pragma unroll
                                for (int ks = 0; ks < STAGE_BLOCKS; ks++) {
                                    const int m = STAGE_BLOCKS * (st - 1) + ks, q = m / 18, r = m % 18, tap = r >> 1, unit = q + 4 * (r & 1);
                                    const int off = (tap / 3 - 1) * 10 + (tap % 3 - 1) + 2 * unit * panel16;
                                    umma_bf16(tmem_d, a_st + (uint64_t)(ks * (BLOCK_BYTES / 16)), b_desc + (uint64_t)(int64_t)off, idesc, 1u);
                                }
                            }
                        }
                        if (MCAST) umma_commit_mcast(bar_empty + 8 * slot, (uint16_t)3);
                        else umma_commit(bar_empty + 8 * slot);
                        if (mine && st == SPL) umma_commit(bar_accum + 8 * g);
                    }
                    __syncwarp();
                }
            }
        }
        if (g == 0 && leader && blockIdx.x == 0) out[LAYERS] = clock64();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == EPI_WARPS + 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    (void)peer;
}

template <bool MCAST>
void run(const uint8_t* wq, const uint8_t* wb, int N0, int N1, int epi_delay, long long* d_out, int grid) {
    cudaFuncSetAttribute(nt_skeleton<MCAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    for (int rep = 0; rep < 2; rep++) nt_skeleton<MCAST><<<grid, THREADS, SMEM_BYTES>>>(wq, wb, N0, N1, epi_delay, d_out);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("error: %s\n", cudaGetErrorString(e)); exit(1); }
    long long h[LAYERS + 1];
    cudaMemcpy(h, d_out, sizeof(h), cudaMemcpyDeviceToHost);
    const double period = (double)(h[LAYERS] - h[2]) / (LAYERS - 2);
    const double floor_ = 73.0 * ((N0 > 94 ? N0 / 2.0 : 47.0) + (N1 > 94 ? N1 / 2.0 : 47.0));
    printf("N = %3d + %3d  epilogue %4d cycles  %s grid %3d: layer period %7.0f cycles (MMA floor %6.0f), weight stream %.1f B/clk/SM\n", N0, N1,
           epi_delay, MCAST ? "multicast" : "unicast  ", grid, period, floor_, 2.0 * 73 * 4096 / period);
}

int main() {
    uint8_t *wq, *wb;
    cudaMalloc(&wq, (size_t)LAYERS * 72 * BLOCK_BYTES);
    cudaMalloc(&wb, (size_t)(LAYERS + 1) * BLOCK_BYTES);
    cudaMemset(wq, 0, (size_t)LAYERS * 72 * BLOCK_BYTES);
    cudaMemset(wb, 0, (size_t)(LAYERS + 1) * BLOCK_BYTES);
    long long* d_out;
    cudaMalloc(&d_out, 256 * sizeof(long long));
    const int shapes[][2] = {{208, 160}, {160, 160}, {160, 112}, {112, 112}, {112, 64}, {64, 64}};
    for (int grid : {148, 2})
        for (auto& s : shapes)
            for (int delay : {3000}) {
                run<false>(wq, wb, s[0], s[1], delay, d_out, grid);
                run<true>(wq, wb, s[0], s[1], delay, d_out, grid);
            }
    run<false>(wq, wb, 208, 160, 5000, d_out, 148);
    run<true>(wq, wb, 208, 160, 5000, d_out, 148);
    return 0;
}
