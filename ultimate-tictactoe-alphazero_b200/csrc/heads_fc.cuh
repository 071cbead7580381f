// heads_fc.cuh -- the fully connected part of the network heads as a block-level device function, used by
// heads_fc_kernel (net_fp32.cu) and by the tail of trunk_auto_kernel (net_auto.cu), so both give the same bits.
#pragma once
#include "tc_common.cuh"

namespace uttt {

constexpr int HEADS_P = 4;                                            // positions per call
constexpr int HEADS_THREADS = 512;                                    // threads that work (more may take part in the barriers)
constexpr int HEADS_CHUNKS = 3, HEADS_CHUNK_ROWS = 27;                // the FC inputs are streamed in 3 chunks of 27
// one chunk of NetWeights::heads_pack: policy_fc rows [27c, 27c+27) of input half 0, the same of half 1 ([in][81 out]),
// value_fc1 rows [27c, 27c+27) ([in][256 hidden]), padded to a multiple of 16 bytes
constexpr int HEADS_POL_FLOATS = HEADS_CHUNK_ROWS * 81;
constexpr int HEADS_CHUNK_FLOATS = (2 * HEADS_POL_FLOATS + HEADS_CHUNK_ROWS * 256 + 3) / 4 * 4;
constexpr int HEADS_CHUNK_BYTES = HEADS_CHUNK_FLOATS * 4;
constexpr int HEADS_PACK_FLOATS = HEADS_CHUNKS * HEADS_CHUNK_FLOATS;
constexpr int HEADS_F_OFF = HEADS_PACK_FLOATS;                        // [243 features][4 positions]
constexpr int HEADS_PART_OFF = HEADS_F_OFF + HEADS_P * 243;           // [2 halves][4][81] policy partial sums
constexpr int HEADS_HID_OFF = HEADS_PART_OFF + 2 * HEADS_P * 81;      // [4][256] value hidden units x value_fc2 weight
constexpr int HEADS_BAR_OFF = HEADS_HID_OFF + HEADS_P * 256;          // 3 mbarriers
constexpr int HEADS_SMEM_BYTES = HEADS_BAR_OFF * 4 + 8 * HEADS_CHUNKS + 8;
static_assert(HEADS_P == 4, "feature vectors are read as float4 over the positions");
static_assert(HEADS_CHUNK_BYTES % 16 == 0 && (HEADS_F_OFF * 4) % 16 == 0 && (HEADS_BAR_OFF * 4) % 8 == 0, "alignment");

struct HeadsFC {                      // built by uttt_upload_weights
    const float *pack, *pol_fc_b, *val_fc1_b, *val_fc2_w, *val_fc2_b;
};
__host__ __device__ inline HeadsFC heads_fc_of(const NetWeights& w) {
    return HeadsFC{w.heads_pack, w.pol_fc_b, w.val_fc1_b, w.val_fc2_w, w.val_fc2_b};
}

// policy_fc + softmax and value_fc1 + ReLU + value_fc2 + tanh (dual_network.py:106-108,115-119) of np <= HEADS_P
// positions, rows row0, row0 + row_step, ... of headfeat = [row][243] (the heads' 1x1 convolutions + BN + ReLU, computed
// in the trunk's last epilogue).
// The 135 KB of FC weights are what costs: read by every thread for itself they are L2-latency-bound (first version:
// 23 k cycles per block, ncu profiles/r1_heads_full.md).  Here one thread streams them into shared memory with three
// bulk async copies (an SM ingests 64 B/clk: ~2 k cycles) and the arithmetic of chunk c overlaps the copy of chunk c+1.
// Thread t < 162 owns policy output t % 81 over input half t / 81, thread 256 + j owns hidden unit j of value_fc1
// (one weight serves the 4 positions: features are read as float4 over the positions); then one warp per position does
// the softmax and one the value_fc2 reduction.  A position's arithmetic does not depend on its place in the call.
// EVERY thread of the block must call this (block-uniform arguments): it contains __syncthreads.
__device__ __forceinline__ void heads_fc_block(const HeadsFC& W, const float* headfeat, int row0, int row_step, int np,
                                               float* __restrict__ policy, float* __restrict__ value, int row_stride,
                                               float* sm /* HEADS_SMEM_BYTES, 16-byte aligned */) {
    const float4* f = reinterpret_cast<const float4*>(sm + HEADS_F_OFF);
    float (*part)[HEADS_P][81] = reinterpret_cast<float (*)[HEADS_P][81]>(sm + HEADS_PART_OFF);
    float (*hid)[256] = reinterpret_cast<float (*)[256]>(sm + HEADS_HID_OFF);
    const uint32_t bar = tcx::smem_u32(sm + HEADS_BAR_OFF);
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    // global loads first (they have nothing to wait for): this thread's share of the features, and the biases the last
    // phase needs (a dependent L2 round trip there would sit on the kernel's critical tail)
    constexpr int F_PER_THREAD = 4;                                     // covers HEADS_P * 243 = 972 values with >= 243 threads
    float fv_[F_PER_THREAD];
#pragma unroll
    for (int u = 0; u < F_PER_THREAD; u++) {
        const int i = t + u * (int)blockDim.x;
        const int p = i / 243, k = i - p * 243;
        fv_[u] = (i < HEADS_P * 243 && p < np) ? __ldcg(headfeat + (size_t)(row0 + p * row_step) * 243 + k) : 0.0f;
    }
    float pb[3] = {0.0f, 0.0f, 0.0f}, vb = 0.0f;
    if (warp < HEADS_P) {
#pragma unroll
        for (int k = 0; k < 3; k++)
            if (lane + 32 * k < 81) pb[k] = __ldg(W.pol_fc_b + lane + 32 * k);
    } else if (warp < 2 * HEADS_P) {
        vb = __ldg(W.val_fc2_b);
    }
    if (t == 0) {
        for (int c = 0; c < HEADS_CHUNKS; c++) tcx::mbar_init(bar + 8 * c, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tcx::fence_async_smem();            // earlier generic-proxy accesses to this shared memory precede the bulk copies
    __syncthreads();
    if (t == 0) {
        for (int c = 0; c < HEADS_CHUNKS; c++) {
            tcx::mbar_expect_tx(bar + 8 * c, HEADS_CHUNK_BYTES);
            tcx::bulk_g2s(tcx::smem_u32(sm + c * HEADS_CHUNK_FLOATS), W.pack + c * HEADS_CHUNK_FLOATS, HEADS_CHUNK_BYTES, bar + 8 * c);
        }
    }
#pragma unroll
    for (int u = 0; u < F_PER_THREAD; u++) {
        const int i = t + u * (int)blockDim.x;
        if (i < HEADS_P * 243) {
            const int p = i / 243, k = i - p * 243;
            sm[HEADS_F_OFF + k * HEADS_P + p] = fv_[u];
        }
    }
    __syncthreads();
    if (t < 162) {
        // policy_fc: output o over input half h
        const int h = t / 81, o = t - 81 * h;
        float ap[HEADS_P];
#pragma unroll
        for (int p = 0; p < HEADS_P; p++) ap[p] = 0.0f;
#pragma unroll 1
        for (int c = 0; c < HEADS_CHUNKS; c++) {
            tcx::mbar_wait(bar + 8 * c, 0);
            const float* wp = sm + c * HEADS_CHUNK_FLOATS + h * HEADS_POL_FLOATS + o;
            const float4* fp4 = f + h * 81 + c * HEADS_CHUNK_ROWS;
#pragma unroll 9
            for (int i = 0; i < HEADS_CHUNK_ROWS; i++) {
                const float xp = wp[i * 81];
                const float4 fp = fp4[i];
                ap[0] = fmaf(fp.x, xp, ap[0]); ap[1] = fmaf(fp.y, xp, ap[1]);
                ap[2] = fmaf(fp.z, xp, ap[2]); ap[3] = fmaf(fp.w, xp, ap[3]);
            }
        }
#pragma unroll
        for (int p = 0; p < HEADS_P; p++) part[h][p][o] = ap[p];
    } else if (t >= 256 && t < 512) {
        // value_fc1: hidden unit j (on its own warps, so the two FC layers run side by side)
        const int j = t - 256;
        const float b1 = __ldg(W.val_fc1_b + j), w2 = __ldg(W.val_fc2_w + j);
        float av[HEADS_P];
#pragma unroll
        for (int p = 0; p < HEADS_P; p++) av[p] = b1;
#pragma unroll 1
        for (int c = 0; c < HEADS_CHUNKS; c++) {
            tcx::mbar_wait(bar + 8 * c, 0);
            const float* wv = sm + c * HEADS_CHUNK_FLOATS + 2 * HEADS_POL_FLOATS + j;
            const float4* fv4 = f + 162 + c * HEADS_CHUNK_ROWS;
#pragma unroll 9
            for (int i = 0; i < HEADS_CHUNK_ROWS; i++) {
                const float xv = wv[i * 256];
                const float4 fv = fv4[i];
                av[0] = fmaf(fv.x, xv, av[0]); av[1] = fmaf(fv.y, xv, av[1]);
                av[2] = fmaf(fv.z, xv, av[2]); av[3] = fmaf(fv.w, xv, av[3]);
            }
        }
#pragma unroll
        for (int p = 0; p < HEADS_P; p++) hid[p][j] = fmaxf(av[p], 0.0f) * w2;
    }
    __syncthreads();
    if (warp < HEADS_P) {
        const int p = warp;
        if (p >= np) return;
        float lg[3], m = -INFINITY;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const int o = lane + 32 * k;
            lg[k] = (o < 81) ? (part[0][p][o] + part[1][p][o]) + pb[k] : -INFINITY;
            m = fmaxf(m, lg[k]);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, off));
        float e[3], s = 0.0f;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            e[k] = (lane + 32 * k < 81) ? expf(lg[k] - m) : 0.0f;
            s += e[k];
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, off);
        float* prow = policy + (size_t)(row0 + p * row_step) * row_stride * 81;
#pragma unroll
        for (int k = 0; k < 3; k++)
            if (lane + 32 * k < 81) prow[lane + 32 * k] = e[k] / s;
    } else if (warp < 2 * HEADS_P) {
        const int p = warp - HEADS_P;
        if (p >= np) return;
        float a = 0.0f;
#pragma unroll
        for (int k = 0; k < 8; k++) a += hid[p][lane + 32 * k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) a += __shfl_xor_sync(0xFFFFFFFFu, a, off);
        if (lane == 0) value[(size_t)(row0 + p * row_step) * row_stride] = tanhf(a + vb);
    }
}

}  // namespace uttt
