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
// The pipeline pieces -- pair geometry, set-up and tear-down, the weight ring and its producer, rank 1's forwarders, the
// halo addresses, the epilogue's chunk conversion and heads -- are shared with pp::trunk_pp_body (trunk_pair.cuh).  What
// is this body's own is the schedule: two TMEM accumulators per tile, so the MMAs of layer L+1 start while the epilogue
// of layer L still runs, and an act_ready barrier per tile and 16-column chunk, on which the issuer waits quarter by
// quarter of the K loop.  The MMAs are cta_group::2 pair MMAs issued by the leader CTA (rank 0) for both CTAs (see Cfg);
// the 11 halo rows at the split are pushed into the peer's margin by the epilogue warp that owns them, after the peer's
// boundary-tile MMAs of the current layer have retired.
//
// Warp roles (19 warps): 0-15 epilogue (2 tiles x 4 TMEM lane quarters x 2 column halves -- the epilogue is
// instruction-latency bound, so it wants warps, not wider threads), 16 weight producer, 17-18 MMA issuers (rank 1:
// barrier forwarders).
#pragma once
#include "trunk_pair.cuh"


namespace uttt {
namespace tc2 {

using namespace tcx;
using tp::HALO_BYTES;
using tp::LEAD;

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
    static constexpr int AROWS = tp::a_rows(LOC_TILES);
    static constexpr int PANEL_BYTES = AROWS * 16;
    static constexpr int ACT_PANELS = X3 ? 32 : 16;        // channel panels [ci/8][row][8] bf16 (X3: panels 16.. hold the lo parts)
    static constexpr int A_BYTES = (ACT_PANELS + 2) * PANEL_BYTES;      // + the constant panel pair of the bias MMA
    static constexpr int NCO = 64;                         // output channels of the B operand held by this CTA
    static constexpr int SUB_BYTES = 2 * NCO * 16;         // one [2 k-panels][NCO co][8] bf16 block
    // Weight ring: 8 stages (X3: 3) of 8 K-blocks (X3: 6, hi block then lo block); the bias block is one block of
    // bf16 hi + lo (+ lo2) in k = 0, 1 (, 2).  K-blocks (one K = 16 slice of a layer: 1 MMA per tile, X3: 3) per weight
    // stage: an issuer thread pays one barrier wait and one commit per stage (200+ cycles each while the tensor pipe
    // saturates shared memory): with 4-block stages a CTA that owns ONE tile (batches of up to 148 positions) was
    // issue-bound at ~93 cycles per MMA
    using W = tp::Stream<X3 ? 3 : 8, X3 ? 6 : 8, (X3 ? 2 : 1) * SUB_BYTES, SUB_BYTES>;
    // TMEM holds two accumulators per tile (4 x 128 = 512 columns): the layers alternate between them, and the epilogue
    // publishes its output per 16-column chunk (NQ act_ready barriers per tile), so the MMAs of layer L+1 run while the
    // epilogue of layer L is still converting the other chunks.
    static constexpr int NQ = 4;
    static constexpr uint32_t ALT_COLS = 256u;                         // column offset of a tile's second accumulator
    static constexpr int BAR_OFF = A_BYTES + W::STAGES * W::STAGE_BYTES;
    static constexpr int HEAD_OFF = BAR_OFF + 256;                 // [128*LOC_TILES rows][4] floats: head partial sums
    static constexpr int SMEM_BYTES = HEAD_OFF + 128 * LOC_TILES * 16;
    static constexpr int EPI_WARPS = 8 * LOC_TILES;  // (tile, lane quarter, column half)
    static constexpr int THREADS = (EPI_WARPS + 1 + LOC_TILES) * 32;
    static constexpr int SKIP_ROWS = 128 * LOC_TILES;
    static constexpr int SKIP_U4 = X3 ? 2 : 1;             // 16-byte units per (panel, row) of the skip buffer: 8 fp16 / 8 fp32
    static_assert(SMEM_BYTES <= 232448, "shared memory");
};

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
                 int pos_base, bool solo) {              // solo: this CTA pair alone evaluates the n_pos positions that start
                                                         // at row pos_base of planes / headfeat (trunk_x3_kernel)
    using C = Cfg<X3>;
    using W = typename C::W;
    constexpr int LOC_TILES = C::LOC_TILES, PANEL_BYTES = C::PANEL_BYTES, EPI_WARPS = C::EPI_WARPS, SKIP_ROWS = C::SKIP_ROWS,
                  NQ = C::NQ, STAGE_BLOCKS = W::STAGE_BLOCKS;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const int n_pairs = solo ? 1 : (int)gridDim.x >> 1, pair = solo ? 0 : (int)blockIdx.x >> 1;
    const int P = group_positions(n_pos, n_pairs);
    const tp::Geo geo = tp::make_geo(P, rank);
    const int n_groups = (n_pos + P - 1) / P;
    if (pair >= n_groups) return;                     // both CTAs of the pair take the same branch

    uint8_t* sA = smem;
    const uint32_t sA_u = smem_u32(sA);
    const uint32_t sB_u = sA_u + C::A_BYTES;
    const uint32_t bar_u = sA_u + C::BAR_OFF;
    // barriers: the ring's full[STAGES], empty[STAGES], then accum[LOC_TILES], act[LOC_TILES][NQ]; then the tmem base holder
    const uint32_t bar_accum = bar_u + 16 * W::STAGES, bar_act = bar_accum + 8 * LOC_TILES;
    constexpr int N_BARS = 2 * W::STAGES + LOC_TILES * (1 + NQ);
    static_assert(8 * N_BARS + 4 <= 256, "barrier block");
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + C::BAR_OFF + 8 * N_BARS);

    if (threadIdx.x == 0) {
        tp::Ring<W>::init(bar_u, rank, geo.T0);       // a stage is released by the leader's T0 issuers
        for (int t = 0; t < LOC_TILES; t++) {
            mbar_init(bar_accum + 8 * t, 1);
            for (int q = 0; q < NQ; q++) mbar_init(bar_act + 8 * (t * NQ + q), tp::act_count(geo, t, rank));
        }
        fence_mbar_init();
    }
    // (solo: the body runs again in this launch and allocates again -- a CTA that gave up its permit may not)
    if (warp == EPI_WARPS + 1) tp::tmem_alloc(tmem_holder, !solo);
    tp::init_operands<X3, C::THREADS>(sA, C::A_BYTES, C::ACT_PANELS * PANEL_BYTES, C::AROWS);    // constant panel ACT_PANELS: the bias MMA's rows
    const uint32_t tmem_base = tp::setup_sync(tmem_holder);
    const uint32_t peer = rank ^ 1u;

    int iter = 0;
    for (int g = pair; g < n_groups; g += n_pairs, iter++) {
        if (warp < EPI_WARPS) {
            // ================= epilogue warps: (tile, TMEM lane quarter, 64-column half) =================
            const int lt = warp >> 3, quarter = warp & 3, chalf = (warp >> 2) & 1;
            if (lt >= geo.tiles) continue;
            const int lr = lt * 128 + quarter * 32 + lane;            // local GEMM row
            const tp::Row row = tp::row_of(geo, lt, quarter, lane, g * P, n_pos, rank);
            float* hrow = headfeat + (size_t)(pos_base + row.gpos) * 243 + (size_t)row.cell;
            float4* hscr = reinterpret_cast<float4*>(smem + C::HEAD_OFF) + lr;
            uint4* srow_skip = skip + ((size_t)blockIdx.x * (16 * SKIP_ROWS) + (size_t)(chalf * 8) * SKIP_ROWS + (size_t)lr) * C::SKIP_U4;
            uint8_t* srow = sA + (size_t)(chalf * 8) * PANEL_BYTES + (size_t)(LEAD + lr) * 16;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(lt * 128 + chalf * 64);
            // the boundary rows are pushed panel by panel (halo_src / halo_dst: panel 8 * chalf) and counted on the
            // peer's act_ready barrier of the same chunk
            const uint32_t panel0 = sA_u + (uint32_t)(chalf * 8) * PANEL_BYTES;
            const uint32_t halo_src = tp::halo_src(panel0, geo, rank), halo_dst = tp::halo_dst(panel0, geo, rank);
            const uint32_t peer_act = map_to_rank(bar_act + 8 * NQ * tp::peer_tile(geo, rank), peer);
            // rows of chunk q of this warp are in place; `tx` = bytes the peer pushes into this CTA's margin for the
            // same barrier phase
            auto publish = [&](int q, uint32_t tx) {
                tp::publish_rows(bar_act + 8 * q, 8 * NQ, row, lt, row.bnd && chalf == 0, tx);
            };
            auto push_halo = [&](int panel, int q) {       // panel relative to this warp's column half
                bulk_s2peer(halo_dst + (uint32_t)panel * PANEL_BYTES, halo_src + (uint32_t)panel * PANEL_BYTES, HALO_BYTES,
                            peer_act + 8u * (uint32_t)q);
            };

            tp::write_input_row(sA + (size_t)chalf * PANEL_BYTES + (size_t)(LEAD + lr) * 16, planes + (size_t)(pos_base + row.gpos) * 243 + (size_t)row.cell, chalf == 0 && row.valid);
            fence_async_smem();
            __syncwarp();
            if (lane == 0) {
#pragma unroll
                for (int q = 0; q < NQ; q++) publish(q, q == 0 ? 2 * HALO_BYTES : 0u);
                // input panel `chalf` of the boundary rows
                if (row.bnd) bulk_s2peer(halo_dst - (uint32_t)(chalf * 7) * PANEL_BYTES, halo_src - (uint32_t)(chalf * 7) * PANEL_BYTES,
                                         HALO_BYTES, peer_act);
            }

            // the last layer (heads' 1x1 convs instead of a write-back) is a separate instantiation of the body so that
            // its extra live registers do not burden the 32 common layers
            int layer = -1;
            auto epilogue_layer = [&](auto last_tag) {
                constexpr bool last = decltype(last_tag)::value;
                const uint32_t lpar = (uint32_t)((iter * tp::GROUP_LAYERS + layer + 1) & 1);
                const uint32_t tsrc = taddr + lpar * C::ALT_COLS;       // this layer's accumulator
                const bool second = (layer >= 0) && (layer & 1) != 0;   // conv2 of a block: add the skip connection
                const bool keep = second || (layer < 0);                // output is the input of the next block: keep it as skip
                uint4 sk[8];
                tp::skip_prefetch<X3, SKIP_ROWS>(sk, srow_skip, second && row.valid);
                tp::wait_rows_free(bar_accum, row, lt, tp::peer_tile(geo, rank), lpar);
                if (threadIdx.x == 0) tp::timeline(dbg, iter, layer, 2);
                tc_fence_after();
                float3 h = make_float3(0.0f, 0.0f, 0.0f);
                tp::for_each_chunk(tsrc, [&](int ch, float* v) {
                    tp::skip_add<X3, SKIP_ROWS>(sk, v, ch, srow_skip, second && row.valid);
                    if constexpr (decltype(last_tag)::value) {
                        tp::head_dots(h, v, headw + chalf * 64 + ch * 16);
                    } else {
                        // channels 16(4*chalf + ch) .. +15 of these rows are in place
                        tp::store_chunk<X3, SKIP_ROWS>(v, ch, srow, PANEL_BYTES, srow_skip, row.valid, keep);
                        fence_async_smem();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) {
                            publish(ch, (X3 ? 8 : 4) * HALO_BYTES);
                            if (row.bnd) {
                                push_halo(2 * ch, ch); push_halo(2 * ch + 1, ch);
                                if (X3) { push_halo(16 + 2 * ch, ch); push_halo(16 + 2 * ch + 1, ch); }
                            }
                        }
                    }
                });
                if constexpr (last) tp::head_store(h, hscr, chalf, 1 + lt * 4 + quarter, row.valid, hrow, headw);
                if (threadIdx.x == 0) tp::timeline(dbg, iter, layer, 3);
            };
#pragma unroll 1
            for (layer = -1; layer < NET_LAYERS - 1; layer++) epilogue_layer(std::false_type{});
            epilogue_layer(std::true_type{});          // layer == NET_LAYERS - 1
            tc_fence_before();
        } else if (warp == EPI_WARPS) {
            // ================= weight producer =================
            // (also in a CTA that owns no tile: the leader's pair MMAs read this CTA's half of every B operand)
            tp::Ring<W> ring(bar_u, iter * W::GROUP_STAGES);
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++)
#pragma unroll 1
                for (int st = 0; st < W::layer_stages(layer); st++) tp::produce_stage(ring, sB_u, wq, wq_in, wq_bias, layer, st, rank, lane);
        } else {
            // ================= MMA issuers: warp EPI_WARPS+1+t drives local accumulator tile t =================
            // One thread issues every MMA of a tile, and two tiles share the tensor pipe: the issuer has 128 cycles per
            // MMA before it becomes the bottleneck.  Its loop is therefore unrolled over the 18 weight stages of a layer
            // (all K-block offsets are immediates), keeps stage / parity as running counters and waits without back-off.
            const int lt = warp - (EPI_WARPS + 1);
            tp::Ring<W> ring(bar_u, iter * W::GROUP_STAGES);
            if (rank != 0) {
                // rank 1: warp 0 forwards "my half of weight stage i has landed", warp 1 "chunk q of my rows of tile pair
                // t is in place"
                if (lt == 0) {
                    tp::forward_stages(ring, W::GROUP_STAGES, lane);
                } else if (lt == 1) {
#pragma unroll 1
                    for (int layer = -1; layer < NET_LAYERS; layer++) {
                        const uint32_t apar = (uint32_t)((iter * tp::GROUP_LAYERS + layer + 1) & 1);
#pragma unroll 1
                        for (int q = 0; q < NQ; q++)
#pragma unroll 1
                            for (int t = 0; t < geo.T1; t++) tp::forward_to_leader(bar_act + 8 * (t * NQ + q), apar, lane);
                    }
                }
                continue;
            }
            if (lt >= geo.tiles) continue;
            const bool leader = elect_one();
            const uint32_t a_tile = sA_u + (uint32_t)(LEAD + lt * 128) * 16u;
            const uint64_t a_desc = make_desc(a_tile, PANEL_BYTES, 128);         // + (row shift + panel offset) / 16: shared
            const uint64_t b_desc = make_desc(sB_u, C::NCO * 16, 128);           //   addresses are < 256 KiB, no carry
            const uint64_t bias_a = a_desc + (uint64_t)((uint32_t)C::ACT_PANELS * PANEL_BYTES / 16u);
            constexpr uint64_t A_LO = (uint64_t)(16u * PANEL_BYTES / 16u);      // X3: descriptor offset of the lo panels
            constexpr uint64_t B_BLK = (uint64_t)(W::BLOCK_BYTES / 16), B_LO = (uint64_t)(C::SUB_BYTES / 16); // per K-block / X3: of its lo half
            // one MMA of this tile and the peer's tile of the same index
            auto mma = [&](uint32_t d, uint64_t a, uint64_t b, uint32_t acc) { umma_bf16_2sm(d, a, b, IDESC_M256_N128_BF16, acc); };
            auto commit_accum = [&]() {            // the layer's accumulator is complete when the MMAs issued so far retire
                umma_commit_2sm(bar_accum + 8 * lt, (uint16_t)3);                            // (in both CTAs)
            };
            // rows of chunk q are in place (own warps, row neighbours, and across the cluster for the boundary tile)
            auto wait_act = [&](int q, uint32_t apar) {
                mbar_wait_spin<false>(bar_act + 8 * (lt * NQ + q), apar);
                tc_fence_after();
            };
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++) {
                const uint32_t apar = (uint32_t)((iter * tp::GROUP_LAYERS + layer + 1) & 1);
                const uint32_t tmem_d = tmem_base + (uint32_t)(lt * 128) + apar * C::ALT_COLS;
                // accumulator := BN shift (constant panel x bias block); starts the layer's accumulation.  With two
                // accumulators per tile this needs no activation: it is issued while the previous epilogue still runs.
                if (layer < 0) {
#pragma unroll
                    for (int q = 0; q < NQ; q++) wait_act(q, apar);
                }
                uint64_t b_st = ring.next_stage(b_desc);
                if (leader) {
                    mma(tmem_d, bias_a, b_st, 0u);
                    ring.release_stage();
                }
                ring.advance();
                if (layer < 0) {
                    // conv_input: block j of stage s is tap STAGE_BLOCKS * s + j, K = 16 (channel panels 0,1)
#pragma unroll
                    for (int s = 0; s < W::IN_STAGES; s++) {
                        b_st = ring.next_stage(b_desc);
                        if (leader) {
#pragma unroll
                            for (int j = 0; j < STAGE_BLOCKS; j++) {
                                const int tap = STAGE_BLOCKS * s + j;
                                if (tap < 9) {
                                    const uint64_t a_tap = a_desc + (uint64_t)(int64_t)tap_shift(tap);
                                    mma(tmem_d, a_tap, b_st + (uint64_t)j * B_BLK, 1u);
                                    // (the input planes are exact in bf16: no lo part on the A side)
                                    if (X3) mma(tmem_d, a_tap, b_st + (uint64_t)j * B_BLK + B_LO, 1u);
                                }
                            }
                            ring.release_stage();
                            if (s == W::IN_STAGES - 1) commit_accum();
                        }
                        ring.advance();
                    }
                } else {
                    // stage s holds K-blocks STAGE_BLOCKS * s ... in the order of tcx::kblock_of (channel-quarter-major);
                    // the first block of quarter q waits for the epilogue's q-th chunk of the previous layer
#pragma unroll
                    for (int s = 0; s < W::STAGES_PER_LAYER; s++) {
                        b_st = ring.next_stage(b_desc);
#pragma unroll
                        for (int ks = 0; ks < STAGE_BLOCKS; ks++) {
                            const int m = STAGE_BLOCKS * s + ks;
                            if (m % 18 == 0) {
                                wait_act(m / 18, apar);
                                if (m == 0 && lt == 0 && leader) tp::timeline(dbg, iter, layer, 0);
                            }
                            if (leader) {
                                const uint64_t a_k = a_desc + (uint64_t)(int64_t)kblock_a_offset(m, PANEL_BYTES / 16),
                                               b_k = b_st + (uint64_t)ks * B_BLK;
                                mma(tmem_d, a_k, b_k, 1u);
                                if (X3) {
                                    mma(tmem_d, a_k + A_LO, b_k, 1u);
                                    mma(tmem_d, a_k, b_k + B_LO, 1u);
                                }
                            }
                        }
                        if (leader) {
                            ring.release_stage();
                            if (s == W::STAGES_PER_LAYER - 1) {
                                commit_accum();
                                if (lt == 0) tp::timeline(dbg, iter, layer, 1);
                            }
                        }
                        ring.advance();
                    }
                }
            }
            __syncwarp();
        }
    }

    tp::teardown(tmem_base, warp == EPI_WARPS + 1);
    if (solo && threadIdx.x == 0) {     // the body runs again in this launch: leave no valid mbarrier objects behind
#pragma unroll
        for (int i = 0; i < N_BARS; i++) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(bar_u + 8 * i) : "memory");
    }
}

}  // namespace tc2
}  // namespace uttt
