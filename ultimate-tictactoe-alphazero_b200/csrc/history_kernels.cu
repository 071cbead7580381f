// history_kernels.cu -- the self-play history as one contiguous buffer of fixed-size samples, built and consumed on the device.
//
// The reference's history is a Python list of [x (9,9,3) f32, pi (81,) f64, z int] per ply (self_play_cpp.py:56-99),
// ~1.7 KB per sample, pickled once per cycle.  On the device a finished cycle lies in per-game arrays padded to 81 plies
// (engine.cu: hist_states / hist_counts / hist_actions / hist_len / hist_final).  For the multi-GPU cycle (BASELINE config
// 5) every rank packs its played plies -- those that were full searches (hist_full: all of them without
// UTTT_SP_PLAYOUT_CAP) -- into 196-byte samples
//     bytes   0..31   packed position (8 x u32)
//     bytes  32..193  root visit counts by action id, u16[81]          (pi = counts / sum, self_play_cpp.py:63-83)
//     byte   194      z, int8: the label of self_play_cpp.py:95-99 (value of the final position, alternating from ply 0)
//     byte   195      ply
// so that ONE exact-length NCCL transfer per rank carries the whole cycle to the trainer rank, which expands the samples
// into the trainer's tensors (train_network.py:41-60) on its own GPU.  Both kernels are HBM-bound byte shuffling: a warp
// per sample, 32-bit coalesced accesses, grids sized from the sample count.
#include "tree_common.cuh"

namespace uttt {

constexpr int SAMPLE_WORDS = UTTT_SAMPLE_BYTES / 4;      // 49

// offsets[g] = number of samples of game g: its plies p < lens[g] with full[g*81 + p] = 1 (every ply without
// UTTT_SP_PLAYOUT_CAP).  One warp per game, one ballot per 32 plies.
__global__ void __launch_bounds__(128) count_samples_kernel(const int32_t* __restrict__ lens, const uint8_t* __restrict__ full,
                                                            int64_t n, int64_t* __restrict__ offsets) {
    const int64_t g = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= n) return;
    const int len = lens[g];
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int p = 32 * j + lane;
        cnt += __popc(__ballot_sync(FULL, p < len && full[(size_t)g * 81 + p] != 0));
    }
    if (lane == 0) offsets[g] = cnt;
}

// in place: offsets[g] = number of samples of the games before g (exclusive prefix sum of the counts); offsets[n] = total.
// One block; n is at most a few 10^4 games.
__global__ void __launch_bounds__(1024) scan_counts_kernel(int64_t n, int64_t* __restrict__ offsets) {
    __shared__ long long part[1024];
    const int t = threadIdx.x;
    const int64_t per = (n + 1023) / 1024, a = t * per, b = min(n, a + per);
    long long s = 0;
    for (int64_t i = a; i < b; i++) s += offsets[i];
    part[t] = s;
    __syncthreads();
    if (t == 0) {
        long long run = 0;
        for (int i = 0; i < 1024; i++) { long long v = part[i]; part[i] = run; run += v; }
        offsets[n] = run;
    }
    __syncthreads();
    long long run = part[t];
    for (int64_t i = a; i < b; i++) { const long long v = offsets[i]; offsets[i] = run; run += v; }
}

// game g's samples in ply order from offsets[g] on; every warp of the block takes the prefix over the game's 81 flags
// (3 ballots) that gives a ply its place among them
__global__ void __launch_bounds__(128) pack_samples_kernel(const PackedState* __restrict__ states, const uint16_t* __restrict__ counts,
                                                           const int32_t* __restrict__ lens, const uint8_t* __restrict__ full,
                                                           const int8_t* __restrict__ final_lose, const int64_t* __restrict__ offsets,
                                                           int64_t n_games, uint32_t* __restrict__ out, int64_t cap_samples) {
    const int64_t g = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (g >= n_games) return;
    const int len = lens[g];
    const int64_t base = offsets[g];
    uint32_t fm[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int p = 32 * j + lane;
        fm[j] = __ballot_sync(FULL, p < len && full[(size_t)g * 81 + p] != 0);
    }
    const int z0 = final_lose[g] ? -1 : 0;                               // self_play_cpp.py:95
    for (int ply = warp; ply < len; ply += 4) {
        const int j = ply >> 5;
        const uint32_t below = fm[j] & ((1u << (ply & 31)) - 1u);
        if (!((fm[j] >> (ply & 31)) & 1u)) continue;
        const int64_t idx = base + (j > 0 ? __popc(fm[0]) : 0) + (j > 1 ? __popc(fm[1]) : 0) + __popc(below);
        if (idx >= cap_samples) return;
        const size_t row = (size_t)g * 81 + (size_t)ply;
        const uint32_t* st = reinterpret_cast<const uint32_t*>(states + row);
        const uint16_t* cn = counts + row * 81;
        uint32_t* dst = out + (size_t)idx * SAMPLE_WORDS;
        const int z = (ply & 1) ? -z0 : z0;                              // :96-99
        for (int w = lane; w < SAMPLE_WORDS; w += 32) {
            uint32_t v;
            if (w < 8) v = st[w];
            else if (w < 48) v = (uint32_t)cn[2 * (w - 8)] | ((uint32_t)cn[2 * (w - 8) + 1] << 16);
            else v = (uint32_t)cn[80] | ((uint32_t)(uint8_t)(int8_t)z << 16) | ((uint32_t)ply << 24);
            dst[w] = v;
        }
    }
}

// samples -> the trainer's arrays: x (n,3,9,9) f32 NCHW (to_input_tensor + the transpose of train_network.py:49),
// policy (n,81) f32 = count / sum (fp32 division), value (n) f32
__global__ void __launch_bounds__(128) unpack_samples_kernel(const uint32_t* __restrict__ samples, int64_t n, float* __restrict__ x,
                                                             float* __restrict__ policy, float* __restrict__ value) {
    const int64_t i = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    const uint32_t* src = samples + (size_t)i * SAMPLE_WORDS;
    const uint32_t w0 = src[lane], w1 = (lane + 32 < SAMPLE_WORDS) ? src[lane + 32] : 0u;
    PackedState st;
#pragma unroll
    for (int k = 0; k < 8; k++) st.w[k] = __shfl_sync(FULL, w0, k);
    uint32_t lm[3];
    legal_mask(st, lm);
    // planes: lane 9*plane + R holds the 9-bit picture row R of plane (mover, opponent, legal)
    {
        const int plane = lane / 9, R = lane - 9 * plane;
        uint32_t xx[3];
#pragma unroll
        for (int j = 0; j < 3; j++) xx[j] = (plane == 0) ? st.w[j] : (plane == 1 ? st.w[3 + j] : lm[j]);
        const uint32_t rows = (lane < 27) ? picture_row(xx, R) : 0u;
        float* xo = x + (size_t)i * 243;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int e = lane + 32 * k;
            const int row = e / 9, C = e - 9 * row;
            const uint32_t m = __shfl_sync(FULL, rows, row & 31);
            if (e < 243) xo[e] = ((m >> C) & 1u) ? 1.0f : 0.0f;
        }
    }
    // counts: action a sits in word 8 + a/2 (half a%2); lane l holds words l and l + 32
    int tot = 0;
    float c[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const int a = lane + 32 * k;
        const int w = 8 + (a >> 1);
        const uint32_t lo = __shfl_sync(FULL, w0, w & 31), hi = __shfl_sync(FULL, w1, w & 31);
        const uint32_t word = (w < 32) ? lo : hi;
        const int v = (a < 81) ? (int)((word >> (16 * (a & 1))) & 0xFFFFu) : 0;
        c[k] = (float)v;
        tot += v;
    }
    tot = __reduce_add_sync(FULL, tot);
    const float inv_ok = tot > 0 ? 1.0f : 0.0f;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const int a = lane + 32 * k;
        if (a < 81) policy[(size_t)i * 81 + a] = inv_ok != 0.0f ? __fdiv_rn(c[k], (float)tot) : 0.0f;
    }
    const uint32_t tail = __shfl_sync(FULL, w1, 48 - 32);
    if (lane == 0) value[i] = (float)(int)(int8_t)((tail >> 16) & 0xFFu);
}

cudaError_t launch_scan_samples(const int32_t* lens, const uint8_t* full, int64_t n, int64_t* offsets, cudaStream_t s) {
    if (n > 0) count_samples_kernel<<<(unsigned)((n + 3) / 4), 128, 0, s>>>(lens, full, n, offsets);
    scan_counts_kernel<<<1, 1024, 0, s>>>(n, offsets);
    return cudaGetLastError();
}
cudaError_t launch_pack_samples(const PackedState* states, const uint16_t* counts, const int32_t* lens, const uint8_t* full,
                                const int8_t* final_lose, const int64_t* offsets, int64_t n_games, void* out, int64_t cap_samples,
                                cudaStream_t s) {
    if (n_games == 0) return cudaSuccess;
    pack_samples_kernel<<<(unsigned)n_games, 128, 0, s>>>(states, counts, lens, full, final_lose, offsets, n_games,
                                                         reinterpret_cast<uint32_t*>(out), cap_samples);
    return cudaGetLastError();
}
cudaError_t launch_unpack_samples(const void* samples, int64_t n, float* x, float* policy, float* value, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    unpack_samples_kernel<<<(unsigned)((n + 3) / 4), 128, 0, s>>>(reinterpret_cast<const uint32_t*>(samples), n, x, policy, value);
    return cudaGetLastError();
}

}  // namespace uttt
