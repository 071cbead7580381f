// net_tc2_kernel.cuh -- trunk_tc2_body: the residual trunk as a tcgen05 implicit GEMM where a thread-block CLUSTER of two
// CTAs (two SMs) shares one group of up to 5 positions, split by GEMM rows.  It runs inside trunk_auto_kernel (net_auto.cu:
// bf16 batches of up to one wave of groups) and trunk_x3_kernel (net_tc2.cu: split-bf16, any batch).
//
// Positions are padded to 100 GEMM rows; the activations stay in shared memory as no-swizzle K-major A panels, the
// pre-packed weights arrive by bulk copies, the accumulators live in TMEM and the epilogue writes the next layer's input
// in place.  The up-to-4 accumulator tiles of a group are divided between the two CTAs of a cluster (2+2, 2+1, 1+1 or
// 1+0).  Per CTA that halves the serial work of a forward pass -- the self-play rounds are latency-bound at the
// reference's 500-game cycle (about 345 queued leaves per round = 69 groups of 5: one CTA per group would use 69 of 148
// SMs, a CTA pair per group uses 138).
//
// The MMAs are cta_group::2 pair MMAs issued by the leader CTA (rank 0) for both CTAs (see Cfg).  The CTAs exchange the
// 11-row halo of the 3x3 taps at the split:
//   * the epilogue warp that owns the last 11 rows of rank 0 (first 11 rows of rank 1) pushes them into the peer's lead
//     (tail) margin with bulk shared->shared copies whose bytes complete on the peer's act_ready barrier of its boundary
//     tile (the peer's boundary warp announces them with expect_tx);
//   * before it overwrites the peer's margin it waits until the peer's boundary-tile MMAs of the current layer have
//     retired: they are the other half of a pair MMA, whose commit arrives on the accumulator barriers of both CTAs.
// Rank 1 issues no MMAs: its issuer warps forward its weight-stage and activation barriers to the leader.
//
// Warp roles (19 warps): 0-15 epilogue (2 tiles x 4 TMEM lane quarters x 2 column halves -- the epilogue is
// instruction-latency bound, so it wants warps, not wider threads), 16 weight producer, 17-18 MMA issuers.
#pragma once
#include <stdlib.h>

#include "tc_common.cuh"


namespace uttt {
namespace tc2 {

constexpr int POS_ROWS = 100;
constexpr int LEAD = 11;
constexpr int GROUP_LAYERS = NET_LAYERS + 1;     // conv_input runs as layer -1 through the same pipeline

// Two accumulator tiles per CTA (LOC_TILES): up to 5 positions per CTA pair (2+2 tiles), 8 weight stages of 16 KiB (this
// CTA's halves of 8 K-blocks).
// X3 = split-bf16 numerics ("bf16x3", UTTT_EVAL_NET_BF16X3): activations and weights are kept as bf16 hi + lo pairs
// (lo = bf16(x - hi)) and every K-block costs three MMAs, hi*hi + lo*hi + hi*lo, accumulated in fp32 in TMEM; the skip
// connection is kept in fp32.  That is ~16 mantissa bits per operand: the mode that meets the reference's fp32 forward
// (dual_network.py:89-121) within 1e-2 on random-init weights (SURVEY.md H1), at a third of the MMA rate.
// Shared memory then holds 32 activation panels (16 hi + 16 lo) and a ring of 3 stages of 6 K-blocks (hi + lo = 4 KiB each).
//
// The MMAs are cta_group::2 pair MMAs (M = 256: local tile t of the leader CTA and local tile t of its peer, issued by the
// leader only, as in net_pp_kernel.cuh) and the B operand is split by output channel: each CTA streams and stores HALF of
// every weight block.  Why: a cta_group::1 MMA of M = N = 128 reads 4 KiB of A and 4 KiB of B per 64 cycles = 128 B/clk,
// all the shared-memory bandwidth of an SM, so the weight stream (one-tile groups of the split-bf16 mode: 590 KB per layer)
// and the epilogue's stores slow the tensor pipe down (tools/micro/mma_shapes.cu, DESIGN.md section 9); a pair MMA reads
// 4 + 2 KiB per CTA.
template <bool X3 = false>
struct Cfg {
    static constexpr int LOC_TILES = 2;
    static constexpr int MAX_P = 5;
    static constexpr int AROWS = (LEAD + 128 * LOC_TILES + 11 + 7) / 8 * 8;
    static constexpr int PANEL_BYTES = AROWS * 16;
    static constexpr int ACT_PANELS = X3 ? 32 : 16;        // channel panels [ci/8][row][8] bf16 (X3: panels 16.. hold the lo parts)
    static constexpr int A_BYTES = (ACT_PANELS + 2) * PANEL_BYTES;      // + the constant panel pair of the bias MMA
    static constexpr int STAGES = X3 ? 3 : 8;
    // K-blocks (one K = 16 slice of a layer: 1 MMA per tile, X3: 3) per weight stage.  An issuer thread pays one barrier
    // wait and one commit per stage (200+ cycles each while the tensor pipe saturates shared memory): with 4-block stages
    // a CTA that owns ONE tile (batches of up to 148 positions) was issue-bound at ~93 cycles per MMA
    static constexpr int STAGE_BLOCKS = X3 ? 6 : 8;
    static constexpr int NCO = 64;                         // output channels of the B operand held by this CTA
    static constexpr int SUB_BYTES = 2 * NCO * 16;         // one [2 k-panels][NCO co][8] bf16 block
    static constexpr int BLOCK_BYTES = (X3 ? 2 : 1) * SUB_BYTES;   // (X3: hi block, then lo block)
    static constexpr int BIAS_BLOCK_BYTES = SUB_BYTES;     // the BN shift as one block: bf16 hi + lo (+ lo2) in k = 0, 1 (, 2)
    static constexpr int STAGE_BYTES = STAGE_BLOCKS * BLOCK_BYTES;
    static constexpr int STAGES_PER_LAYER = 72 / STAGE_BLOCKS;
    static constexpr int IN_STAGES = (9 + STAGE_BLOCKS - 1) / STAGE_BLOCKS;   // conv_input: 9 taps x (K=16: 3 real channels) in IN_STAGES * STAGE_BLOCKS tap slots
    static constexpr int GROUP_STAGES = (IN_STAGES + 1) + NET_LAYERS * (STAGES_PER_LAYER + 1);   // every layer starts with its bias block
    // TMEM holds two accumulators per tile (4 x 128 = 512 columns): the layers alternate between them, and the epilogue
    // publishes its output per 16-column chunk (NQ act_ready barriers per tile), so the MMAs of layer L+1 run while the
    // epilogue of layer L is still converting the other chunks.
    static constexpr int NQ = 4;
    static constexpr uint32_t ALT_COLS = 256u;                         // column offset of a tile's second accumulator
    static constexpr int BAR_OFF = A_BYTES + STAGES * STAGE_BYTES;
    static constexpr int HEAD_OFF = BAR_OFF + 256;                 // [128*LOC_TILES rows][4] floats: head partial sums
    static constexpr int SMEM_BYTES = HEAD_OFF + 128 * LOC_TILES * 16;
    static constexpr int EPI_WARPS = 8 * LOC_TILES;  // (tile, lane quarter, column half)
    static constexpr int THREADS = (EPI_WARPS + 1 + LOC_TILES) * 32;
    static constexpr int SKIP_ROWS = 128 * LOC_TILES;
    static constexpr int SKIP_U4 = X3 ? 2 : 1;             // 16-byte units per (panel, row) of the skip buffer: 8 fp16 / 8 fp32
    static constexpr uint32_t TMEM_COLS = 512u;
    static_assert(SMEM_BYTES <= 232448, "shared memory");
};

using namespace tcx;

// positions per CTA pair (= per group) for a batch of n_pos positions on n_pairs pairs
__host__ __device__ inline int group_positions(int n_pos, int n_pairs) {
    int P = (n_pos + n_pairs - 1) / n_pairs;
    P = P < 1 ? 1 : (P > Cfg<>::MAX_P ? Cfg<>::MAX_P : P);
    if (P == 4) P = 5;                                // 4 positions need the same 4 tiles as 5
    return P;
}

// the kernel body (a __device__ function: trunk_auto_kernel, net_auto.cu, puts it behind a device-side dispatch together
// with pp::trunk_pp_body; trunk_x3_kernel, net_tc2.cu, runs it once per group).  The caller has read the batch size and
// counted it (count_batch).
// The three weight arrays hold per-CTA halves, stage-major: [stage][2 ranks][STAGE_BLOCKS blocks]([hi, lo])[2][64][8].
template <bool X3>
__device__ __forceinline__ void trunk_tc2_body(const __nv_bfloat16* __restrict__ wq,   // [32 * 72 / STAGE_BLOCKS stages]...: 72 K-blocks per layer
                 const __nv_bfloat16* __restrict__ wq_in,// conv_input: [IN_STAGES]...: one K-block per tap (9 of IN_STAGES * STAGE_BLOCKS used)
                 const __nv_bfloat16* __restrict__ wq_bias,   // [33][2 ranks][1 block]...: per layer the BN shift as a K=16 B block
                 const __nv_bfloat16* __restrict__ planes,   // network input [rows][3][81] bf16
                 const float* __restrict__ headw,        // [3][128] policy conv (2) + value conv, BN scale folded; [384..386] shifts
                 float* headfeat,                        // out: [rows][243] = relu(policy conv)[2][81], relu(value conv)[81]
                 uint4* skip,                            // [gridDim][16 panels][256 rows] fp16x8 skip connection (X3: fp32x8)
                 long long* dbg,
                 int n_pos,                              // the batch size
                 const int* src_rows,                    // slot mode: position i of this CTA pair reads planes row src_rows[i], else null
                 int pos_base, bool solo) {              // solo: this CTA pair alone evaluates the n_pos positions that start
                                                         // at row pos_base of planes / headfeat (trunk_x3_kernel)
    using C = Cfg<X3>;
    constexpr int LOC_TILES = C::LOC_TILES, PANEL_BYTES = C::PANEL_BYTES, A_BYTES = C::A_BYTES,
                  STAGES = C::STAGES, BAR_OFF = C::BAR_OFF, EPI_WARPS = C::EPI_WARPS, THREADS = C::THREADS,
                  SKIP_ROWS = C::SKIP_ROWS, NQ = C::NQ, STAGE_BLOCKS = C::STAGE_BLOCKS, STAGE_BYTES = C::STAGE_BYTES,
                  STAGES_PER_LAYER = C::STAGES_PER_LAYER, IN_STAGES = C::IN_STAGES, GROUP_STAGES = C::GROUP_STAGES,
                  ACT_PANELS = C::ACT_PANELS, SKIP_U4 = C::SKIP_U4, BLOCK_BYTES = C::BLOCK_BYTES;
    extern __shared__ __align__(1024) uint8_t smem[];
    const long long t_entry = clock64();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const int n_pairs = solo ? 1 : (int)gridDim.x >> 1, pair = solo ? 0 : (int)blockIdx.x >> 1;
    const int P = group_positions(n_pos, n_pairs);
    const int T = (P * POS_ROWS + 127) / 128;         // tiles of the pair: 1..4
    const int T0 = (T + 1) >> 1;                      // rank 0 takes the first ceil(T/2) tiles
    const int tiles = (rank == 0) ? T0 : T - T0;      // this CTA's tiles (0..2)
    const int tile0 = (rank == 0) ? 0 : T0;           // first global tile of this CTA
    const int n_groups = (n_pos + P - 1) / P;
    if (pair >= n_groups) return;                     // both CTAs of the pair take the same branch
    const int T1 = T - T0;                            // tiles of rank 1 (<= T0)
    const bool has_peer = T1 > 0;

    uint8_t* sA = smem;
    const uint32_t sA_u = smem_u32(sA);
    const uint32_t sB_u = sA_u + A_BYTES;
    const uint32_t bar_u = sA_u + BAR_OFF;
    // barriers: full[STAGES], empty[STAGES], accum[LOC_TILES], act[LOC_TILES][NQ]; then the tmem base holder
    const uint32_t bar_full = bar_u, bar_empty = bar_u + 8 * STAGES, bar_accum = bar_u + 16 * STAGES,
                   bar_act = bar_accum + 8 * LOC_TILES;
    constexpr int N_BARS = 2 * STAGES + LOC_TILES * (1 + NQ);
    static_assert(8 * N_BARS + 4 <= 256, "barrier block");
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + BAR_OFF + 8 * N_BARS);
    // the tile of this CTA that touches the peer's rows, and the quarter-warp that owns the shared rows
    const int bnd_tile = (rank == 0) ? tiles - 1 : 0;
    const int bnd_quarter = (rank == 0) ? 3 : 0;

    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; i++) {
            // the leader's full barrier also counts the peer's forwarded "my half has landed"; a stage is released in
            // both CTAs by the multicast commits of the leader's T0 issuers
            mbar_init(bar_full + 8 * i, rank == 0 ? 2 : 1);
            mbar_init(bar_empty + 8 * i, T0);
        }
        for (int t = 0; t < LOC_TILES; t++) {
            mbar_init(bar_accum + 8 * t, 1);
            int c = 8 + (t > 0 ? 2 : 0) + (t < tiles - 1 ? 2 : 0);      // (the peer's halo rows arrive as transaction bytes)
            if (rank == 0 && t < T1) c += 1;                            // the peer's forwarded "my rows of tile pair t are in place"
            for (int q = 0; q < NQ; q++) mbar_init(bar_act + 8 * (t * NQ + q), c);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == EPI_WARPS + 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)),
                     "r"(C::TMEM_COLS)
                     : "memory");
        // (solo: the body runs again in this launch and allocates again -- a CTA that gave up its permit may not)
        if (!solo) asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    for (int i = threadIdx.x; i < A_BYTES / 16; i += THREADS) reinterpret_cast<uint4*>(sA)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    // constant panel 16: every row = (1, 1, 0, ..., 0).  One extra K=16 MMA per tile and layer multiplies it with the
    // layer's bias block (shift_hi, shift_lo in k = 0, 1), so the BatchNorm shift is added by the tensor pipe and the
    // epilogue has no bias loads or adds (measured: -20 % epilogue time).
    // (X3: (1, 1, 1, 0, ...): the shift comes as three bf16 terms)
    for (int i = threadIdx.x; i < C::AROWS; i += THREADS)
        reinterpret_cast<uint4*>(sA + (size_t)ACT_PANELS * PANEL_BYTES)[i] = make_uint4(0x3F803F80u, X3 ? 0x00003F80u : 0u, 0, 0);
    fence_async_all();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the peer's barriers and margins exist before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    const uint32_t peer = rank ^ 1u;
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) { dbg[192] = t_entry; dbg[193] = clock64(); }

    int iter = 0;
    for (int g = pair; g < n_groups; g += n_pairs, iter++) {
        if (warp < EPI_WARPS) {
            // ================= epilogue warps: (tile, TMEM lane quarter, 64-column half) =================
            const int lt = warp >> 3, quarter = warp & 3, chalf = (warp >> 2) & 1;
            if (lt >= tiles) continue;
            const int lr = lt * 128 + quarter * 32 + lane;            // local GEMM row
            const int gr = tile0 * 128 + lr;                          // row within the group
            const int pos = gr / POS_ROWS, idx = gr - pos * POS_ROWS;
            const int r = idx / 10, c = idx - 10 * r;
            const int gpos = g * P + pos;
            const bool valid = (pos < P) && (r < 9) && (c < 9) && (gpos < n_pos);
            float* hrow = headfeat + (size_t)(pos_base + gpos) * 243 + (size_t)(r * 9 + c);
            float4* hscr = reinterpret_cast<float4*>(smem + C::HEAD_OFF) + lr;
            uint4* srow_skip = skip + ((size_t)blockIdx.x * (16 * SKIP_ROWS) + (size_t)(chalf * 8) * SKIP_ROWS + (size_t)lr) * SKIP_U4;
            uint8_t* srow = sA + (size_t)(chalf * 8) * PANEL_BYTES + (size_t)(LEAD + lr) * 16;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(lt * 128 + chalf * 64);
            const bool nb_lo = (quarter == 0) && (lt > 0);
            const bool nb_hi = (quarter == 3) && (lt < tiles - 1);
            const bool bnd = has_peer && (lt == bnd_tile) && (quarter == bnd_quarter);
            // The 11 boundary rows of this CTA (rank 0: its last rows -> the peer's lead margin, rank 1: its first rows ->
            // the peer's tail margin) are pushed panel by panel with bulk shared->shared copies that count their bytes on
            // the peer's act_ready barrier; the peer's chalf-0 boundary warp announces them with expect_tx.
            constexpr uint32_t HALO_BYTES = 11 * 16;
            const uint32_t halo_src = sA_u + (uint32_t)(chalf * 8) * PANEL_BYTES +
                                      (uint32_t)(LEAD + ((rank == 0) ? (128 * tiles - 11) : 0)) * 16u;
            const uint32_t halo_dst = map_to_rank(sA_u + (uint32_t)(chalf * 8) * PANEL_BYTES +
                                                  (uint32_t)((rank == 0) ? 0 : (LEAD + 128 * T0)) * 16u, peer);
            const uint32_t peer_act = map_to_rank(bar_act + 8 * NQ * ((rank == 0) ? 0 : (T0 - 1)), peer);
            // publish rows of this warp (chunk barrier q of its tile and of the row neighbours); `tx` = bytes the peer
            // pushes into this CTA's margin for the same barrier phase
            auto publish = [&](int q, uint32_t tx) {
                if (bnd && chalf == 0) mbar_expect_tx(bar_act + 8 * (lt * NQ + q), tx);
                else mbar_arrive(bar_act + 8 * (lt * NQ + q));
                if (nb_lo) mbar_arrive(bar_act + 8 * ((lt - 1) * NQ + q));
                if (nb_hi) mbar_arrive(bar_act + 8 * ((lt + 1) * NQ + q));
            };
            auto push_halo = [&](int panel, int q) {       // panel relative to this warp's column half
                bulk_s2peer(halo_dst + (uint32_t)panel * PANEL_BYTES, halo_src + (uint32_t)panel * PANEL_BYTES, HALO_BYTES,
                            peer_act + 8u * (uint32_t)q);
            };
            const uint4 zero4 = make_uint4(0, 0, 0, 0);

            // prologue: the three input planes of this row go into channel panel 0 (channels 3..15 are zero): the
            // A operand of conv_input, which runs as "layer -1" on the tensor pipe with K = 16 per tap
            {
                uint4 pk = zero4;
                if (chalf == 0 && valid) {
                    const __nv_bfloat16* px = planes + (size_t)(src_rows ? src_rows[pos] : pos_base + gpos) * 243 + (size_t)(r * 9 + c);
                    uint32_t x0 = (uint32_t)__bfloat16_as_ushort(px[0]), x1 = (uint32_t)__bfloat16_as_ushort(px[81]),
                             x2 = (uint32_t)__bfloat16_as_ushort(px[162]);
                    pk = make_uint4(x0 | (x1 << 16), x2, 0u, 0u);
                }
                uint8_t* dst = sA + (size_t)chalf * PANEL_BYTES + (size_t)(LEAD + lr) * 16;
                *reinterpret_cast<uint4*>(dst) = pk;
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
#pragma unroll
                for (int q = 0; q < NQ; q++) publish(q, q == 0 ? 2 * HALO_BYTES : 0u);
                // input panel `chalf` of the boundary rows (halo_src / halo_dst point at panel 8*chalf)
                if (bnd) bulk_s2peer(halo_dst - (uint32_t)(chalf * 7) * PANEL_BYTES, halo_src - (uint32_t)(chalf * 7) * PANEL_BYTES,
                                     HALO_BYTES, peer_act);
            }

            // the last layer (heads' 1x1 convs instead of a write-back) is a separate instantiation of the body so that
            // its extra live registers do not burden the 32 common layers
            int layer = -1;
            auto epilogue_layer = [&](auto last_tag) {
                constexpr bool last = decltype(last_tag)::value;
                const uint32_t lpar = (uint32_t)((iter * GROUP_LAYERS + layer + 1) & 1);
                const uint32_t tsrc = taddr + lpar * C::ALT_COLS;       // this layer's accumulator
                const bool second = (layer >= 0) && (layer & 1) != 0;   // conv2 of a block: add the skip connection
                const bool keep = second || (layer < 0);                // output is the input of the next block: keep it as skip
                // the skip connection (8 x 16 B per thread) is fetched from L2 while the MMAs still run
                // (X3: fp32, 4 x 16 B per 16-column chunk; the chunks 0 and 1 are prefetched, 2 and 3 follow as 0 and 1 are used)
                uint4 sk[8];
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if constexpr (X3) sk[j] = (second && valid) ? srow_skip[(size_t)(j >> 1) * SKIP_ROWS * 2 + (j & 1)] : zero4;
                    else sk[j] = (second && valid) ? srow_skip[(size_t)j * SKIP_ROWS] : zero4;
                }
                mbar_wait_spin<false>(bar_accum + 8 * lt, lpar);
                if (nb_lo) mbar_wait_spin<false>(bar_accum + 8 * (lt - 1), lpar);
                if (nb_hi) mbar_wait_spin<false>(bar_accum + 8 * (lt + 1), lpar);
                // the peer's boundary-tile MMAs have retired: they are the other half of the pair MMAs of index 0 -- rank
                // 1's first tile -- or T0 - 1 -- rank 0's last tile --, whose multicast commits arrive on this CTA's barrier
                if (bnd) mbar_wait_spin<false>(bar_accum + 8 * ((rank == 0) ? 0 : T0 - 1), lpar);
                if (dbg && blockIdx.x == 0 && iter == 0 && threadIdx.x == 0 && layer >= 0) dbg[layer * 4 + 2] = clock64();
                const bool detail = dbg && blockIdx.x == 0 && iter == 0 && threadIdx.x == 0 && layer == 20;   // diagnostics: dbg[160..175]
                if (detail) dbg[160] = clock64();
                tc_fence_after();
                float va[16], vb[16];
                float h0 = 0.0f, h1 = 0.0f, h2 = 0.0f;               // last layer: the heads' 1x1 convolutions of this row
                tmem_ld16(tsrc, va);
#pragma unroll
                for (int ch = 0; ch < 4; ch++) {
                    float* v = (ch & 1) ? vb : va;
                    tmem_ld_wait();
                    if (detail && ch == 0) dbg[161] = clock64();
                    if (ch < 3) tmem_ld16(tsrc + (uint32_t)((ch + 1) * 16), (ch & 1) ? va : vb);
                    if constexpr (X3) {
#pragma unroll
                        for (int j = 0; j < 4; j++) f32x4_add(sk[4 * (ch & 1) + j], v + 4 * j);
                        if (ch < 2 && second && valid) {             // refill the four registers just consumed: chunk ch + 2
#pragma unroll
                            for (int j = 0; j < 4; j++)
                                sk[4 * (ch & 1) + j] = srow_skip[(size_t)(2 * (ch + 2) + (j >> 1)) * SKIP_ROWS * 2 + (j & 1)];
                        }
                    } else {
                        f16x8_add2(sk[2 * ch], v);
                        f16x8_add2(sk[2 * ch + 1], v + 8);
                    }
                    if constexpr (last) {
                        // the trunk output never leaves the SM: policy_conv / value_conv (1x1, dual_network.py:102,111)
                        // are three dot products over the channels this thread holds
                        const float* hw = headw + chalf * 64 + ch * 16;
#pragma unroll
                        for (int j = 0; j < 16; j++) {
                            float x = fmaxf(v[j], 0.0f);
                            h0 = fmaf(x, __ldg(hw + j), h0);
                            h1 = fmaf(x, __ldg(hw + 128 + j), h1);
                            h2 = fmaf(x, __ldg(hw + 256 + j), h2);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 2; j++) {
                            if constexpr (X3) {
                                // x = relu(v) = hi + lo (+ 2^-17 |x|): both halves feed the next layer's MMAs
                                float x[8], l[8];
#pragma unroll
                                for (int i = 0; i < 8; i++) x[i] = fmaxf(v[8 * j + i], 0.0f);
                                uint4 hi = pack8_bf16(x);
                                bf16x8_residual(hi, x, l);
                                uint4 lo = pack8_bf16(l);
                                if (!valid) hi = lo = zero4;                             // padding rows stay zero
                                *reinterpret_cast<uint4*>(srow + (size_t)(ch * 2 + j) * PANEL_BYTES) = hi;
                                *reinterpret_cast<uint4*>(srow + (size_t)(16 + ch * 2 + j) * PANEL_BYTES) = lo;
                                if (keep && valid) {
                                    uint4* d = srow_skip + (size_t)(ch * 2 + j) * SKIP_ROWS * 2;
                                    d[0] = make_uint4(__float_as_uint(x[0]), __float_as_uint(x[1]), __float_as_uint(x[2]), __float_as_uint(x[3]));
                                    d[1] = make_uint4(__float_as_uint(x[4]), __float_as_uint(x[5]), __float_as_uint(x[6]), __float_as_uint(x[7]));
                                }
                            } else {
                                uint4 pk = valid ? relu_pack8_bf16(v + 8 * j) : zero4;      // padding rows stay zero
                                *reinterpret_cast<uint4*>(srow + (size_t)(ch * 2 + j) * PANEL_BYTES) = pk;
                                if (keep && valid) srow_skip[(size_t)(ch * 2 + j) * SKIP_ROWS] = relu_pack8_f16(v + 8 * j);
                            }
                        }
                        // channels 16(4*chalf + ch) .. +15 of these rows are in place
                        if (detail && ch == 0) dbg[162] = clock64();
                        fence_async_smem();
                        tc_fence_before();
                        __syncwarp();
                        if (detail && ch == 0) dbg[163] = clock64();
                        if (lane == 0) {
                            publish(ch, (X3 ? 8 : 4) * HALO_BYTES);
                            if (bnd) {
                                push_halo(2 * ch, ch); push_halo(2 * ch + 1, ch);
                                if (X3) { push_halo(16 + 2 * ch, ch); push_halo(16 + 2 * ch + 1, ch); }
                            }
                            if (detail) dbg[164 + ch] = clock64();
                        }
                    }
                }
                if constexpr (last) {
                    // combine the two column halves of the row (two warps) and emit BN shift + ReLU of the head convs
                    if (chalf == 1) *hscr = make_float4(h0, h1, h2, 0.0f);
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + lt * 4 + quarter) : "memory");
                    if (chalf == 0 && valid) {
                        float4 o = *hscr;
                        hrow[0] = fmaxf(h0 + o.x + __ldg(headw + 384), 0.0f);
                        hrow[81] = fmaxf(h1 + o.y + __ldg(headw + 385), 0.0f);
                        hrow[162] = fmaxf(h2 + o.z + __ldg(headw + 386), 0.0f);
                    }
                }
                if (dbg && blockIdx.x == 0 && iter == 0 && threadIdx.x == 0 && layer >= 0) dbg[layer * 4 + 3] = clock64();
            };
#pragma unroll 1
            for (layer = -1; layer < NET_LAYERS - 1; layer++) epilogue_layer(std::false_type{});
            epilogue_layer(std::true_type{});          // layer == NET_LAYERS - 1
            tc_fence_before();
        } else if (warp == EPI_WARPS) {
            // ================= weight producer =================
            // (also in a CTA that owns no tile: the leader's pair MMAs read this CTA's half of every B operand)
            int gn = iter * GROUP_STAGES;
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++) {
                const int n_st = 1 + ((layer < 0) ? IN_STAGES : STAGES_PER_LAYER);
#pragma unroll 1
                for (int st = 0; st < n_st; st++, gn++) {
                    const int stage = gn % STAGES;
                    const uint32_t par = (uint32_t)((gn / STAGES) & 1);
                    mbar_wait(bar_empty + 8 * stage, par ^ 1u);
                    if (lane == 0) {
                        const __nv_bfloat16* src;
                        uint32_t bytes = STAGE_BYTES;
                        const int rk = (int)rank;          // per-CTA halves are stored stage-major: [stage][rank]
                        if (st == 0) { src = wq_bias + (size_t)((layer + 1) * 2 + rk) * (C::BIAS_BLOCK_BYTES / 2); bytes = C::BIAS_BLOCK_BYTES; }   // (sizes in bf16 elements)
                        else if (layer < 0) src = wq_in + (size_t)((st - 1) * 2 + rk) * (STAGE_BYTES / 2);
                        else src = wq + (size_t)((layer * STAGES_PER_LAYER + st - 1) * 2 + rk) * (STAGE_BYTES / 2);
                        mbar_expect_tx(bar_full + 8 * stage, bytes);
                        bulk_g2s(sB_u + stage * STAGE_BYTES, src, bytes, bar_full + 8 * stage);
                    }
                    __syncwarp();
                }
            }
        } else {
            // ================= MMA issuers: warp EPI_WARPS+1+t drives local accumulator tile t =================
            // One thread issues every MMA of a tile, and two tiles share the tensor pipe: the issuer has 128 cycles per
            // MMA before it becomes the bottleneck.  Its loop is therefore unrolled over the 18 weight stages of a layer
            // (all K-block offsets are immediates), keeps stage / parity as running counters and waits without back-off.
            const int lt = warp - (EPI_WARPS + 1);
            if (rank != 0) {
                // rank 1 has no MMAs to issue (the leader issues for the pair): its two issuer warps forward its barriers
                // to the leader with CTA-scope remote arrives (see net_pp_kernel.cuh).  Warp 0: "my half of weight stage i
                // has landed"; warp 1: "chunk q of my rows of tile pair t is in place".  Neither can be lapped: the
                // events they wait for need the leader's next MMAs, which need their arrive.
                if (lt == 0) {
                    int gn = iter * GROUP_STAGES;
#pragma unroll 1
                    for (int i = 0; i < GROUP_STAGES; i++, gn++) {
                        const int stage = gn % STAGES;
                        mbar_wait_spin<false>(bar_full + 8 * stage, (uint32_t)((gn / STAGES) & 1));
                        if (lane == 0) mbar_arrive_peer(map_to_rank(bar_full + 8 * stage, 0));
                        __syncwarp();
                    }
                } else if (lt == 1) {
#pragma unroll 1
                    for (int layer = -1; layer < NET_LAYERS; layer++) {
                        const uint32_t apar = (uint32_t)((iter * GROUP_LAYERS + layer + 1) & 1);
#pragma unroll 1
                        for (int q = 0; q < NQ; q++)
#pragma unroll 1
                            for (int t = 0; t < T1; t++) {
                                mbar_wait_spin<false>(bar_act + 8 * (t * NQ + q), apar);
                                if (lane == 0) mbar_arrive_peer(map_to_rank(bar_act + 8 * (t * NQ + q), 0));
                                __syncwarp();
                            }
                    }
                }
                continue;
            }
            if (lt >= tiles) continue;
            const bool leader = elect_one();
            const uint32_t a_tile = sA_u + (uint32_t)(LEAD + lt * 128) * 16u;
            const uint64_t a_desc = make_desc(a_tile, PANEL_BYTES, 128);         // + (row shift + panel offset) / 16: shared
            const uint64_t b_desc = make_desc(sB_u, C::NCO * 16, 128);           //   addresses are < 256 KiB, no carry
            const uint64_t bias_a = a_desc + (uint64_t)((uint32_t)ACT_PANELS * PANEL_BYTES / 16u);
            constexpr uint64_t A_LO = (uint64_t)(16u * PANEL_BYTES / 16u);      // X3: descriptor offset of the lo panels
            constexpr uint64_t B_BLK = (uint64_t)(BLOCK_BYTES / 16), B_LO = (uint64_t)(C::SUB_BYTES / 16); // per K-block / X3: of its lo half
            // one MMA of this tile and the peer's tile of the same index
            auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t acc) { umma_bf16_2sm(d, a, b, IDESC_M256_N128_BF16, acc); };
            auto commit_accum = [&]() {            // the layer's accumulator is complete when the MMAs issued so far retire
                umma_commit_2sm(bar_accum + 8 * lt, (uint16_t)3);                            // (in both CTAs)
            };
            int gn = iter * GROUP_STAGES;
            int stage = gn % STAGES;
            uint32_t par = (uint32_t)((gn / STAGES) & 1);
            uint64_t b_st = 0;
            // rows of chunk q are in place (own warps, row neighbours, and across the cluster for the boundary tile)
            auto wait_act = [&](int q, uint32_t apar) {
                mbar_wait_spin<false>(bar_act + 8 * (lt * NQ + q), apar);
                tc_fence_after();
            };
            auto next_stage = [&]() {              // waits for the next weight stage; b_st = descriptor of its first block
                mbar_wait_spin<false>(bar_full + 8 * stage, par);
                tc_fence_after();
                b_st = b_desc + (uint64_t)(uint32_t)(stage * (STAGE_BYTES / 16));
            };
            auto release_stage = [&]() {           // leader only: frees the stage when the MMAs issued so far retire
                umma_commit_2sm(bar_empty + 8 * stage, (uint16_t)3);                         // (in both CTAs)
            };
            auto advance = [&]() {
                if (++stage == STAGES) { stage = 0; par ^= 1u; }
            };
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++) {
                const uint32_t apar = (uint32_t)((iter * GROUP_LAYERS + layer + 1) & 1);
                const uint32_t tmem_d = tmem_base + (uint32_t)(lt * 128) + apar * C::ALT_COLS;
                // accumulator := BN shift (constant panel x bias block); starts the layer's accumulation.  With two
                // accumulators per tile this needs no activation: it is issued while the previous epilogue still runs.
                if (layer < 0) {
#pragma unroll
                    for (int q = 0; q < NQ; q++) wait_act(q, apar);
                    if (dbg && blockIdx.x == 0 && iter == 0 && lt == 0 && leader && layer >= 0) dbg[layer * 4 + 0] = clock64();
                }
                next_stage();
                if (leader) {
                    mma(tmem_d, bias_a, b_st, 0u);
                    release_stage();
                }
                advance();
                if (layer < 0) {
                    // conv_input: block j of stage s is tap 8s+j, K = 16 (channel panels 0,1)
#pragma unroll
                    for (int s = 0; s < IN_STAGES; s++) {
                        next_stage();
                        if (leader) {
#pragma unroll
                            for (int j = 0; j < STAGE_BLOCKS; j++) {
                                const int tap = STAGE_BLOCKS * s + j;
                                if (tap < 9) {
                                    const uint64_t a_tap = a_desc + (uint64_t)(int64_t)((tap / 3 - 1) * 10 + (tap % 3 - 1));
                                    mma(tmem_d, a_tap, b_st + (uint64_t)j * B_BLK, 1u);
                                    // (the input planes are exact in bf16: no lo part on the A side)
                                    if (X3) mma(tmem_d, a_tap, b_st + (uint64_t)j * B_BLK + B_LO, 1u);
                                }
                            }
                            release_stage();
                            if (s == IN_STAGES - 1) commit_accum();
                        }
                        advance();
                    }
                } else {
                    // stage s holds K-blocks 8s .. 8s+7 in the order of tcx::kblock_of (channel-quarter-major); the first
                    // block of quarter q waits for the epilogue's q-th chunk of the previous layer
#pragma unroll
                    for (int s = 0; s < STAGES_PER_LAYER; s++) {
                        next_stage();
#pragma unroll
                        for (int ks = 0; ks < STAGE_BLOCKS; ks++) {
                            const int m = STAGE_BLOCKS * s + ks, q = m / 18, r = m % 18, tap = r >> 1, unit = q + 4 * (r & 1);
                            if (r == 0) {
                                wait_act(q, apar);
                                if (q == 0 && dbg && blockIdx.x == 0 && iter == 0 && lt == 0 && leader) dbg[layer * 4 + 0] = clock64();
                                if (dbg && blockIdx.x == 0 && iter == 0 && lt == 0 && leader && layer == 21) dbg[168 + q] = clock64();
                            }
                            const int off = (tap / 3 - 1) * 10 + (tap % 3 - 1) + 2 * unit * (PANEL_BYTES / 16);
                            if (leader) {
                                const uint64_t a_k = a_desc + (uint64_t)(int64_t)off, b_k = b_st + (uint64_t)ks * B_BLK;
                                mma(tmem_d, a_k, b_k, 1u);
                                if (X3) {
                                    mma(tmem_d, a_k + A_LO, b_k, 1u);
                                    mma(tmem_d, a_k, b_k + B_LO, 1u);
                                }
                            }
                        }
                        if (leader) {
                            release_stage();
                            if (s == STAGES_PER_LAYER - 1) {
                                commit_accum();
                                if (dbg && blockIdx.x == 0 && iter == 0 && lt == 0) dbg[layer * 4 + 1] = clock64();
                                if (dbg && blockIdx.x == 0 && iter == 0 && lt == 0 && layer == 20) dbg[172] = clock64();
                            }
                        }
                        advance();
                    }
                }
            }
            __syncwarp();
        }
    }

    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) dbg[194] = clock64();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // nobody exits while the peer may still write its margins / barriers
    if (warp == EPI_WARPS + 1)
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::TMEM_COLS) : "memory");
    if (solo && threadIdx.x == 0) {     // the body runs again in this launch: leave no valid mbarrier objects behind
#pragma unroll
        for (int i = 0; i < N_BARS; i++) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar_u + 8 * i) : "memory");
    }
    if (dbg && blockIdx.x == 0 && threadIdx.x == 0) dbg[195] = clock64();
}

}  // namespace tc2
}  // namespace uttt
