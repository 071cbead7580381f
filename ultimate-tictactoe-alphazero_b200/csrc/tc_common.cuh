// tc_common.cuh -- PTX wrappers shared by the tensor-core trunk kernels (net_tc2.cu, net_pp.cu, net_auto.cu): UMMA shared-memory
// descriptors, mbarriers, bulk async copies, tcgen05 MMA / commit / TMEM loads, cluster (DSMEM) helpers, and the
// packed-math epilogue helpers.
#pragma once
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"

namespace uttt {
namespace tcx {

// K order of a 3x3 layer: 72 blocks of K = 16 (one MMA each).  Block m = 18*q + 2*tap + h multiplies tap `tap` of
// the 16 input channels of unit u = q + 4h (channels 16u .. 16u+15).  The order is channel-quarter-major: an epilogue
// warp writes units 0..3 (column half 0) or 4..7 (column half 1) in that order, so the blocks of quarter q only need
// the q-th 16-column chunk of every epilogue warp -- the next layer's MMAs start while the epilogue is still running.
// The pre-packed weights (pack_res_kernel, weights.cu) are stored in the same order, 4 KiB per block.
__host__ __device__ __forceinline__ int kblock_of(int tap, int unit) { return 18 * (unit & 3) + 2 * tap + (unit >> 2); }
// The inverse, as offsets of the A descriptor (16-byte units) from a tile's first row in channel panel 0.  Tap t of the
// 100-row position layout (row = 10 r + c) is the row shift 10 dy + dx:
__host__ __device__ __forceinline__ constexpr int tap_shift(int tap) { return (tap / 3 - 1) * 10 + (tap % 3 - 1); }
// K-block m reads that shift in the panel pair of its unit (panel16: bytes per channel panel / 16).
__host__ __device__ __forceinline__ constexpr int kblock_a_offset(int m, int panel16) {
    return tap_shift((m % 18) >> 1) + 2 * (m / 18 + 4 * ((m % 18) & 1)) * panel16;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// after the mbarrier.init of barriers that the peer CTA or the async proxy will signal
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// bounded wait; traps instead of hanging.  CLUSTER = true acquires at cluster scope (needed where an arrival
// comes from the peer CTA); ptxas then flushes L1 after the wait (CCTL.IVALL), so it is used only there.
template <bool CLUSTER = false>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t backoff_ns = 0) {
    uint32_t ok = 0;
    long long t0 = 0;
    for (uint32_t it = 0;; it++) {
        if (CLUSTER)
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(ok)
                : "r"(bar), "r"(parity)
                : "memory");
        else
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(ok)
                : "r"(bar), "r"(parity)
                : "memory");
        if (ok) return;
        if (backoff_ns) __nanosleep(backoff_ns);
        if ((it & 1023u) == 1023u) {
            long long now = clock64();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 4000000000ll) {
                printf("uttt trunk: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x,
                       threadIdx.x, bar, parity);
                __trap();
            }
        }
    }
}
// Lean wait for the waits on the critical path of a layer (issuer <- epilogue chunk, epilogue <- accumulator): no
// back-off sleep and no message.  POLL = false suspends in try_wait (the hardware parks the warp for a time slice: a
// dozen warps waiting this way cost no issue slots); POLL = true spins on test_wait -- lowest wake-up latency, but 16
// epilogue warps spinning through a whole MMA phase starve the single issuer thread (measured in net_pp.cu: every
// instruction of the issuer took 200-500 cycles), so it is reserved for short waits of single warps.
template <bool POLL>
__device__ __forceinline__ void mbar_wait_spin(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
#pragma unroll 1
    for (uint32_t it = 0; it < (1u << 26); it++) {
        if (POLL)
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(ok)
                : "r"(bar), "r"(parity)
                : "memory");
        else
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(ok)
                : "r"(bar), "r"(parity)
                : "memory");
        if (ok) return;
    }
    __trap();
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// shared memory of this CTA -> shared memory of a CTA of the cluster, by the async proxy; the bytes are counted on the
// destination CTA's mbarrier (complete_tx), so the receiver's tensor pipe may read them after a plain wait: no
// cluster-scope release on the sender (ptxas turns that into MEMBAR.ALL.GPU) and no acquire.cluster on the receiver.
__device__ __forceinline__ void bulk_s2peer(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t bar_cluster) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     dst_cluster),
                 "r"(src_cta), "r"(bytes), "r"(bar_cluster)
                 : "memory");
}
__device__ __forceinline__ void fence_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// cta_group::2: one MMA of M = 256 over the CTA pair (128 rows from each CTA's shared memory at the same offsets, the B
// operand split by N between the two CTAs); issued by the leader CTA only.  Instruction descriptor (kind::f16): D = f32
// (bit 4), A = B = bf16 (bits 7, 10), K-major A and B, N = 128, M = 256
constexpr uint32_t IDESC_M256_N128_BF16 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((256u >> 4) << 24);
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"(mask)
                 : "memory");
}
// arrive on a barrier of another CTA of the cluster with CTA-scope semantics (one SYNCS.ARRIVE.RED, no MEMBAR.GPU)
__device__ __forceinline__ void mbar_arrive_peer(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
    uint32_t* r = reinterpret_cast<uint32_t*>(v);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
    return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}
// v[0..3] += 4 fp32 values
__device__ __forceinline__ void f32x4_add(const uint4& q, float* v) {
    v[0] += __uint_as_float(q.x); v[1] += __uint_as_float(q.y); v[2] += __uint_as_float(q.z); v[3] += __uint_as_float(q.w);
}
// l[i] = x[i] - float(hi[i]) for 8 packed bf16 (exact: the difference of a float and its bf16 rounding)
__device__ __forceinline__ void bf16x8_residual(const uint4& hi, const float* x, float* l) {
    const uint32_t w[4] = {hi.x, hi.y, hi.z, hi.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        l[2 * i] = x[2 * i] - __uint_as_float(w[i] << 16);
        l[2 * i + 1] = x[2 * i + 1] - __uint_as_float(w[i] & 0xFFFF0000u);
    }
}
// ReLU fused into the conversion (F2FP.RELU): max(x,0) then round to bf16 / fp16 (saturating)
__device__ __forceinline__ uint32_t relu_bf16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__device__ __forceinline__ uint32_t relu_f16x2(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.satfinite.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__device__ __forceinline__ uint4 relu_pack8_bf16(const float* v) {
    return make_uint4(relu_bf16x2(v[0], v[1]), relu_bf16x2(v[2], v[3]), relu_bf16x2(v[4], v[5]), relu_bf16x2(v[6], v[7]));
}
__device__ __forceinline__ uint4 relu_pack8_f16(const float* v) {
    return make_uint4(relu_f16x2(v[0], v[1]), relu_f16x2(v[2], v[3]), relu_f16x2(v[4], v[5]), relu_f16x2(v[6], v[7]));
}
// v[0..7] += 8 fp16 values (FADD2 pairs)
__device__ __forceinline__ void f16x8_add2(const uint4& q, float* v) {
    const __half2* h = reinterpret_cast<const __half2*>(&q);
    float2* v2 = reinterpret_cast<float2*>(v);
#pragma unroll
    for (int i = 0; i < 4; i++) v2[i] = __fadd2_rn(v2[i], __half22float2(h[i]));
}
// diagnostics (dbg non-null): histogram of evaluator batch sizes, 16 per bucket, read by uttt_debug_batch_histogram.
// Every trunk kernel counts once per launch that evaluates a batch.
__device__ __forceinline__ void count_batch(long long* dbg, int n_pos) {
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0)
        atomicAdd(reinterpret_cast<unsigned long long*>(dbg) + 128 + min(n_pos >> 4, 63), 1ull);
}

}  // namespace tcx
}  // namespace uttt
