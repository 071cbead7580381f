// net_pp_kernel.cuh -- trunk_pp_body: the residual trunk with two independent groups of positions in flight per CTA
// pair and cta_group::2 MMAs.  It runs evaluator batches above one wave of 5-position groups (370 positions on 148 SMs):
// up to 7 positions per pair inside trunk_auto_kernel (net_auto.cu), more in trunk_pp_large_kernel (net_pp.cu); smaller
// batches run tc2::trunk_tc2_body (net_tc2_kernel.cuh).
//
// A thread-block cluster of two CTAs (positions padded to 100 GEMM rows, a group's rows split between the two CTAs, 11
// halo rows exchanged at the split; the pipeline pieces are shared with trunk_tc2_body, trunk_pair.cuh) alternates
// between two groups layer by layer:
//
//      tensor pipe :  MMA(A, L)   MMA(B, L)   MMA(A, L+1)   MMA(B, L+1)  ...
//      epilogue    :              epi(A, L)   epi(B, L)     epi(A, L+1)  ...
//
// so a layer's epilogue always has the other group's MMAs to hide behind.  Group A holds 5 positions (2 + 2 accumulator
// tiles), group B the rest of the pair's share (instantiation 1: up to 2 positions = 1 + 1 tiles, weight stages of a
// quarter layer; instantiation 2: up to 5 positions, stages of 8 K-blocks).  Rows are bit-identical to net_tc2_kernel.cuh: every accumulator
// sums its K-blocks in the order of tcx::kblock_of, whichever kernel and thread issued them.
//
// The MMAs are cta_group::2 pair MMAs (M = 256: tile t of the leader CTA and tile t of its peer, N = 128) issued by the
// leader CTA only; the B operand is split by output channel between the two CTAs, so each CTA streams and stores HALF of
// every layer's weights (2 KiB per K-block).  That matters because the weight stream bounds this design: an SM ingests
// at most 64 B/clk from L2 (tools/micro/l2stream.cu: same figure for 2 or 148 CTAs, unicast or multicast) and a ring slot
// stays occupied for about 2000 cycles (copy latency + MMA queue + retirement); with cta_group::1 MMAs every CTA streamed
// all weights once per group and the kernel was weight-stream-bound (19.9 k cycles per layer at 500 positions).
// Measured (B200, tools/pp_timeline.py): layer period 14.5 k cycles at 500 positions (MMA floor for 3 pair tiles:
// 3 x 72 x 64 = 13.8 k), 18.7 k at 740.  The peer CTA forwards "my half of stage i has landed" / "my rows of tile pair t
// are in place" to the leader's barriers with CTA-scope remote arrives (no cluster-scope fences in the layer loop).
// Each group's epilogue publishes once per layer, and the issuer waits for a group's whole input before its layer.
//
// Warp roles (19 warps): 0-15 epilogue ((tile, TMEM lane quarter, 64-column half), the same warps serve both groups),
// 16 weight producer, 17-18 leader: MMA issuers (one per local tile index; an issuer without a tile in a group still walks
// and releases that group's weight stages so the ring has one consumer count) / peer: barrier forwarders.
#pragma once
#include "trunk_pair.cuh"

namespace uttt {
namespace pp {

using namespace tcx;
using tp::HALO_BYTES;
using tp::LEAD;

constexpr int LT = 2;                           // accumulator tiles per CTA of group A (and the number of issuer warps)
constexpr int NG = 2;                           // groups in flight
constexpr int BIAS_BYTES = 2048;                // per CTA
constexpr int CONST_BYTES = 4096;
constexpr int EPI_WARPS = 8 * LT;
constexpr int THREADS = (EPI_WARPS + 1 + LT) * 32;
constexpr int SKIP_ROWS = 128 * LT;
constexpr uint32_t IDESC = IDESC_M256_N128_BF16; // cta_group::2: 128 rows of each CTA x all 128 output channels

// LTB = accumulator tiles per CTA of group B: 1 (B holds up to 2 positions: 7 per pair, a deeper weight ring) or
// 2 (B holds up to 5 positions: 10 per pair)
template <int LTB>
struct Cfg {
    static constexpr int MAX_PA = 5, MAX_PB = (LTB == 1) ? 2 : 5;
    static constexpr int PANEL_A = tp::a_rows(LT) * 16, PANEL_B = tp::a_rows(LTB) * 16;   // bytes per channel panel [row][8] bf16
    static constexpr int A_BYTES = 16 * PANEL_A, B_BYTES = 16 * PANEL_B;            // 16 channel panels per group
    static constexpr int CONST_OFF = A_BYTES + B_BYTES;   // [2][128][8] bf16: rows (1,1,0,...,0), the A operand of the bias MMA
    static constexpr int W_OFF = CONST_OFF + CONST_BYTES;
    // K-blocks (MMAs per tile pair) per weight stage: an issuer thread pays one barrier wait and one commit per stage,
    // 200+ cycles each while the tensor pipe saturates shared memory.  LTB = 1: group B is ONE tile pair, whose 72 MMAs
    // of a layer must be issued at 64 cycles each by one thread -- with a quarter of a layer (18 K-blocks, 36 KiB per CTA)
    // per stage that thread has 1152 cycles per stage for its two barrier operations and 18 MMA issues.  (Round 1 split
    // that tile's K loop over two threads and two accumulators instead: same speed, but other low bits than every other
    // batch band; handing one accumulator to and fro between two threads with tcgen05 fences is bit-identical but the
    // hand-over sits on the issue path: +3 % per cycle.)
    // Per CTA: its output-channel half of the stage's K-blocks, 2 KiB each; a ring of 3 (LTB = 2: 4) stages
    using W = tp::Stream<(LTB == 1) ? 3 : 4, (LTB == 1) ? 18 : 8, 2048, BIAS_BYTES>;
    static constexpr int BAR_OFF = W_OFF + W::STAGES * W::STAGE_BYTES;
    static constexpr int HEAD_OFF = BAR_OFF + 512;        // [128*LT rows][4] floats: head partial sums
    static constexpr int SMEM_BYTES = HEAD_OFF + 128 * LT * 16;
    static_assert(SMEM_BYTES <= 232448, "shared memory");
};

// positions per CTA pair and super-group (groups A + B) for a batch of n_pos positions on n_pairs pairs
template <int LTB>
__host__ __device__ inline int pair_positions(int n_pos, int n_pairs) {
    int P = (n_pos + n_pairs - 1) / n_pairs;
    return P < 1 ? 1 : (P > Cfg<LTB>::MAX_PA + Cfg<LTB>::MAX_PB ? Cfg<LTB>::MAX_PA + Cfg<LTB>::MAX_PB : P);
}

// the kernel body (see net_tc2_kernel.cuh): trunk_pp_large_kernel (net_pp.cu) runs LTB = 2, trunk_auto_kernel (net_auto.cu)
// LTB = 1.  The caller has read the batch size and counted it (count_batch).
template <int LTB>
__device__ __forceinline__ void trunk_pp_body(const __nv_bfloat16* __restrict__ wq,        // [32 * STAGES_PER_LAYER stages][2 ranks][STAGE_BLOCKS K-blocks][2][64][8] bf16
                const __nv_bfloat16* __restrict__ wq_in,     // conv_input: [IN_STAGES][2 ranks][STAGE_BLOCKS tap slots][2][64][8] bf16
                const __nv_bfloat16* __restrict__ wq_bias,   // [33][2 ranks][2][64][8] bf16: per layer the BN shift as a K=16 B block
                const __nv_bfloat16* __restrict__ planes,    // network input [rows][3][81] bf16
                const float* __restrict__ headw,             // [3][128] policy conv (2) + value conv; [384..386] shifts
                float* headfeat,                             // out: [rows][243]
                uint4* skip,                                 // [gridDim][NG][16 panels][256 rows] fp16x8 skip connection
                long long* dbg,
                int n_pos) {                                 // the batch size
    using C = Cfg<LTB>;
    using W = typename C::W;
    constexpr int STAGE_BLOCKS = W::STAGE_BLOCKS;
    constexpr int MAX_P = C::MAX_PA;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const uint32_t peer = rank ^ 1u;
    const int n_pairs = (int)gridDim.x >> 1, pair = (int)blockIdx.x >> 1;
    const int Ptot = pair_positions<LTB>(n_pos, n_pairs);     // positions per pair and super-group
    const int n_super = (n_pos + Ptot - 1) / Ptot;
    if (pair >= n_super) return;                              // both CTAs of the pair take the same branch
    const int PA = Ptot < MAX_P ? Ptot : MAX_P;
    const tp::Geo geo[NG] = {tp::make_geo(PA, rank), tp::make_geo(Ptot - PA, rank)};
    // groups the pair has (pair-level: both CTAs stream the weights of a group that exists); each walks the weight ring once
    const int n_streams = (geo[0].T0 > 0) + (geo[1].T0 > 0);

    uint8_t* sA = smem;
    const uint32_t sA_u = smem_u32(sA);
    const uint32_t sB_u = sA_u + C::W_OFF;
    // per group: offset of its activation buffer, bytes per channel panel
    auto grp_off = [](int g) { return (uint32_t)(g == 0 ? 0 : C::A_BYTES); };
    auto grp_panel = [](int g) { return (uint32_t)(g == 0 ? C::PANEL_A : C::PANEL_B); };
    const uint32_t bar_u = sA_u + C::BAR_OFF;
    // barriers: the ring's full[STAGES], empty[STAGES], then per group accum[LT], act[LT]; then the tmem base holder.  The
    // leader's full / act barriers also count an arrive forwarded by the peer ("my half of the stage has landed" / "my rows
    // of the tile pair are in place"), so its issuers wait on one barrier per event.
    const uint32_t bar_grp = bar_u + 16 * W::STAGES;
    constexpr int GRP_BARS = 2 * LT;
    auto bar_accum = [&](int g, int t) { return bar_grp + 8u * (uint32_t)(g * GRP_BARS + t); };
    auto bar_act = [&](int g, int t) { return bar_grp + 8u * (uint32_t)(g * GRP_BARS + LT + t); };
    static_assert(16 * W::STAGES + 8 * NG * GRP_BARS + 4 <= 512, "barrier block");
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + C::BAR_OFF + 16 * W::STAGES + 8 * NG * GRP_BARS);
    // timeline slot of (group, layer): layers 0..15 of both groups
    auto tl_slot = [](int g, int layer) { return (layer >= 0 && layer < 16) ? 16 * g + layer : -1; };

    if (threadIdx.x == 0) {
        tp::Ring<W>::init(bar_u, rank, LT);                   // a stage is released by the leader's LT issuers
        for (int g = 0; g < NG; g++) {
            for (int t = 0; t < LT; t++) {
                mbar_init(bar_accum(g, t), 1);
                mbar_init(bar_act(g, t), tp::act_count(geo[g], t, rank));
            }
        }
        fence_mbar_init();
    }
    if (warp == EPI_WARPS + 1) tp::tmem_alloc(tmem_holder, true);
    tp::init_operands<false, THREADS>(sA, C::W_OFF, C::CONST_OFF, 128);    // (the constant block's second panel stays zero)
    const uint32_t tmem_base = tp::setup_sync(tmem_holder);

    int iter = 0;
    for (int sg = pair; sg < n_super; sg += n_pairs, iter++) {
        const int ring0 = iter * n_streams * W::GROUP_STAGES;    // the ring position continues across super-groups
        if (warp < EPI_WARPS) {
            // ================= epilogue warps: (tile, TMEM lane quarter, 64-column half), both groups =================
            const int lt = warp >> 3, quarter = warp & 3, chalf = (warp >> 2) & 1;
            const int lr = lt * 128 + quarter * 32 + lane;                   // local GEMM row
            float4* hscr = reinterpret_cast<float4*>(smem + C::HEAD_OFF) + lr;

            // this thread's row in group g (recomputed per call: the epilogue is off the critical path here, registers are not)
            auto row_of = [&](int g) { return tp::row_of(geo[g], lt, quarter, lane, sg * Ptot + (g == 0 ? 0 : PA), n_pos, rank); };
            // the boundary rows of panels panel .. panel + n_panels - 1, counted on the peer's act_ready barrier
            auto push_halo = [&](int g, int panel, int n_panels) {
                const uint32_t PANEL_BYTES = grp_panel(g);
                const uint32_t base = sA_u + grp_off(g) + (uint32_t)panel * PANEL_BYTES;
                const uint32_t src = tp::halo_src(base, geo[g], rank), dst = tp::halo_dst(base, geo[g], rank);
                const uint32_t pbar = map_to_rank(bar_act(g, tp::peer_tile(geo[g], rank)), peer);
                for (int p = 0; p < n_panels; p++)
                    bulk_s2peer(dst + (uint32_t)p * PANEL_BYTES, src + (uint32_t)p * PANEL_BYTES, HALO_BYTES, pbar);
            };
            auto publish = [&](int g, const tp::Row& r, uint32_t tx) {
                tp::publish_rows(bar_act(g, 0), 8u, r, lt, r.bnd && chalf == 0, tx);
            };

#pragma unroll 1
            for (int g = 0; g < NG; g++) {
                if (lt >= geo[g].tiles) continue;
                const tp::Row r = row_of(g);
                tp::write_input_row(sA + grp_off(g) + (size_t)chalf * grp_panel(g) + (size_t)(LEAD + lr) * 16,
                                    planes + (size_t)r.gpos * 243 + (size_t)r.cell, chalf == 0 && r.valid);
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    publish(g, r, 2 * HALO_BYTES);
                    if (r.bnd) push_halo(g, chalf, 1);
                }
            }

            auto epilogue_layer = [&](int g, int layer, auto last_tag) {
                constexpr bool last = decltype(last_tag)::value;
                if (lt >= geo[g].tiles) return;
                const tp::Row r = row_of(g);
                const uint32_t lpar = (uint32_t)((iter * tp::GROUP_LAYERS + layer + 1) & 1);
                const bool second = (layer >= 0) && (layer & 1) != 0;   // conv2 of a block: add the skip connection
                const bool keep = second || (layer < 0);                // output is the input of the next block: keep it as skip
                uint4* srow_skip = skip + (size_t)(blockIdx.x * NG + g) * (16 * SKIP_ROWS) + (size_t)(chalf * 8) * SKIP_ROWS + (size_t)lr;
                const uint32_t PANEL_BYTES = grp_panel(g);
                uint8_t* srow = sA + grp_off(g) + (size_t)(chalf * 8) * PANEL_BYTES + (size_t)(LEAD + lr) * 16;
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((g * LT + lt) * 128 + chalf * 64);
                uint4 sk[8];
                tp::skip_prefetch<false, SKIP_ROWS>(sk, srow_skip, second && r.valid);
                tp::wait_rows_free(bar_accum(g, 0), r, lt, tp::peer_tile(geo[g], rank), lpar);
                if (threadIdx.x == 0) tp::timeline(dbg, iter, tl_slot(g, layer), 2);
                tc_fence_after();
                float3 h = make_float3(0.0f, 0.0f, 0.0f);
                tp::for_each_chunk(taddr, [&](int ch, float* v) {
                    tp::skip_add<false, SKIP_ROWS>(sk, v, ch, srow_skip, false);
                    if constexpr (decltype(last_tag)::value) tp::head_dots(h, v, headw + chalf * 64 + ch * 16);
                    else tp::store_chunk<false, SKIP_ROWS>(v, ch, srow, PANEL_BYTES, srow_skip, r.valid, keep);
                });
                if constexpr (!last) {
                    fence_async_smem();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        publish(g, r, 16 * HALO_BYTES);
                        if (r.bnd) push_halo(g, chalf * 8, 8);
                    }
                } else {
                    tc_fence_before();
                    tp::head_store(h, hscr, chalf, 1 + lt * 4 + quarter, r.valid, headfeat + (size_t)r.gpos * 243 + (size_t)r.cell, headw);
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + lt * 4 + quarter) : "memory");   // hscr is reused by the other group
                }
                if (threadIdx.x == 0) tp::timeline(dbg, iter, tl_slot(g, layer), 3);
            };
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS - 1; layer++) {
#pragma unroll 1
                for (int g = 0; g < NG; g++) epilogue_layer(g, layer, std::false_type{});
            }
#pragma unroll 1
            for (int g = 0; g < NG; g++) epilogue_layer(g, NET_LAYERS - 1, std::true_type{});
        } else if (n_streams == 0) {
            continue;
        } else if (warp == EPI_WARPS) {
            // ================= weight producer: this CTA's output-channel half of every layer, once per group =========
            tp::Ring<W> ring(bar_u, ring0);
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++) {
#pragma unroll 1
                for (int g = 0; g < NG; g++) {
                    if (geo[g].T0 == 0) continue;
#pragma unroll 1
                    for (int st = 0; st < W::layer_stages(layer); st++) tp::produce_stage(ring, sB_u, wq, wq_in, wq_bias, layer, st, rank, lane);
                }
            }
        } else if (rank != 0) {
            // ================= rank 1: warp EPI_WARPS+1 forwards "my half of weight stage i has landed", warp EPI_WARPS+2
            // "my rows of tile pair t of group g are in place"
            if (warp == EPI_WARPS + 1) {
                tp::forward_stages(tp::Ring<W>(bar_u, ring0), n_streams * W::GROUP_STAGES, lane);
            } else {
#pragma unroll 1
                for (int layer = -1; layer < NET_LAYERS; layer++) {
                    const uint32_t apar = (uint32_t)((iter * tp::GROUP_LAYERS + layer + 1) & 1);
#pragma unroll 1
                    for (int g = 0; g < NG; g++)
#pragma unroll 1
                        for (int t = 0; t < geo[g].T1; t++) tp::forward_to_leader(bar_act(g, t), apar, lane);
                }
            }
        } else {
            // ================= leader CTA: warp EPI_WARPS+1+t issues the pair MMAs (cta_group::2, M = 256: tile t of this CTA
            // and tile t of the peer) of both groups ==========
            const int lt = warp - (EPI_WARPS + 1);
            const bool leader = elect_one();
            const uint64_t b_desc = make_desc(sB_u, 1024, 128);           // this CTA's 64 output channels: [2 panels][64][8]
            const uint64_t bias_a = make_desc(sA_u + C::CONST_OFF, 2048, 128);
            tp::Ring<W> ring(bar_u, ring0);
            // per group, fixed for the kernel: does this thread issue for it, into which accumulator, from which rows
            bool g_stream[NG], g_issue[NG];
            uint32_t g_tmem[NG], g_act[NG], g_accum[NG];
            uint64_t g_adesc[NG];
            int g_panel16[NG];
#pragma unroll
            for (int g = 0; g < NG; g++) {
                const tp::Geo& G = geo[g];
                const int tile = lt;
                g_stream[g] = G.T0 > 0;
                g_issue[g] = tile < G.T0;
                g_tmem[g] = tmem_base + (uint32_t)((g * LT + tile) * 128);
                g_act[g] = bar_act(g, tile);
                g_accum[g] = bar_accum(g, tile);
                g_panel16[g] = (int)(grp_panel(g) / 16);
                g_adesc[g] = make_desc(sA_u + grp_off(g) + (uint32_t)(LEAD + tile * 128) * 16u, grp_panel(g), 128);
            }
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++) {
                const uint32_t apar = (uint32_t)((iter * tp::GROUP_LAYERS + layer + 1) & 1);
#pragma unroll
                for (int g = 0; g < NG; g++) {
                    if (!g_stream[g]) continue;                     // the pair does not have this group
                    const bool mine = g_issue[g];                   // otherwise: walk and release the stages only
                    const uint32_t tmem_d = g_tmem[g];
                    const uint64_t a_desc = g_adesc[g];
                    const int panel16 = g_panel16[g];
                    if (mine) {
                        // the layer's input rows are in place: this CTA's (own rows, row neighbours', the peer's halo) and
                        // the peer's (forwarded arrive)
                        mbar_wait_spin<false>(g_act[g], apar);
                        tc_fence_after();
                    }
                    if (lt == 0 && leader) tp::timeline(dbg, iter, tl_slot(g, layer), 0);
                    // accumulator := BN shift (constant rows x bias block); starts the layer's accumulation
                    uint64_t b_st = ring.next_stage(b_desc);
                    if (mine && leader) umma_bf16_2sm(tmem_d, bias_a, b_st, IDESC, 0u);
                    if (leader) ring.release_stage();
                    ring.advance();
                    if (layer < 0) {
                        // conv_input: block j of stage s is tap STAGE_BLOCKS * s + j, K = 16 (channel panels 0,1)
#pragma unroll
                        for (int s = 0; s < W::IN_STAGES; s++) {
                            b_st = ring.next_stage(b_desc);
                            if (mine && leader) {
#pragma unroll
                                for (int j = 0; j < STAGE_BLOCKS; j++) {
                                    const int tap = STAGE_BLOCKS * s + j;
                                    if (tap < 9)
                                        umma_bf16_2sm(tmem_d, a_desc + (uint64_t)(int64_t)tap_shift(tap), b_st + (uint64_t)(j * 128), IDESC, 1u);
                                }
                            }
                            if (leader) {
                                ring.release_stage();
                                if (mine && s == W::IN_STAGES - 1) umma_commit_2sm(g_accum[g], (uint16_t)3);
                            }
                            ring.advance();
                        }
                    } else {
                        // stage s holds K-blocks STAGE_BLOCKS * s ... in the order of tcx::kblock_of
#pragma unroll
                        for (int s = 0; s < W::STAGES_PER_LAYER; s++) {
                            b_st = ring.next_stage(b_desc);
                            if (mine && leader) {
#pragma unroll
                                for (int ks = 0; ks < STAGE_BLOCKS; ks++)
                                    umma_bf16_2sm(tmem_d, a_desc + (uint64_t)(int64_t)kblock_a_offset(STAGE_BLOCKS * s + ks, panel16),
                                                  b_st + (uint64_t)(ks * 128), IDESC, 1u);
                            }
                            if (leader) {
                                ring.release_stage();
                                if (mine && s == W::STAGES_PER_LAYER - 1) {
                                    umma_commit_2sm(g_accum[g], (uint16_t)3);
                                    if (lt == 0) tp::timeline(dbg, iter, tl_slot(g, layer), 1);
                                }
                            }
                            ring.advance();
                        }
                    }
                }
            }
            __syncwarp();
        }
    }

    tp::teardown(tmem_base, warp == EPI_WARPS + 1);
}

}  // namespace pp
}  // namespace uttt
