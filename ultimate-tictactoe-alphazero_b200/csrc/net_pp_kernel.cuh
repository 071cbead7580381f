// net_pp_kernel.cuh -- trunk_pp_body: the residual trunk with two independent groups of positions in flight per CTA
// pair and cta_group::2 MMAs.  It runs evaluator batches above one wave of 5-position groups (370 positions on 148 SMs):
// up to 7 positions per pair inside trunk_auto_kernel (net_auto.cu), more in trunk_pp_large_kernel (net_pp.cu); smaller
// batches run tc2::trunk_tc2_body (net_tc2_kernel.cuh).
//
// A thread-block cluster of two CTAs (as in net_tc2_kernel.cuh: positions padded to 100 GEMM rows, a group's rows split
// between the two CTAs, 11 halo rows exchanged at the split) alternates between two groups layer by layer:
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
//
// Warp roles (19 warps): 0-15 epilogue ((tile, TMEM lane quarter, 64-column half), the same warps serve both groups),
// 16 weight producer, 17-18 leader: MMA issuers (one per local tile index; an issuer without a tile in a group still walks
// and releases that group's weight stages so the ring has one consumer count) / peer: barrier forwarders.
#pragma once
#include "tc_common.cuh"

namespace uttt {
namespace pp {

using namespace tcx;

constexpr int POS_ROWS = 100;
constexpr int LEAD = 11;
constexpr int LT = 2;                           // accumulator tiles per CTA of group A (and the number of issuer warps)
constexpr int NG = 2;                           // groups in flight
constexpr int BIAS_BYTES = 2048;                // per CTA
constexpr int CONST_BYTES = 4096;
constexpr int EPI_WARPS = 8 * LT;
constexpr int THREADS = (EPI_WARPS + 1 + LT) * 32;
constexpr int SKIP_ROWS = 128 * LT;
constexpr int GROUP_LAYERS = NET_LAYERS + 1;    // conv_input runs as layer -1 through the same pipeline
constexpr uint32_t IDESC = IDESC_M256_N128_BF16; // cta_group::2: 128 rows of each CTA x all 128 output channels
constexpr int a_rows(int tiles) { return (LEAD + 128 * tiles + 11 + 7) / 8 * 8; }

// LTB = accumulator tiles per CTA of group B: 1 (B holds up to 2 positions: 7 per pair, a deeper weight ring) or
// 2 (B holds up to 5 positions: 10 per pair)
template <int LTB>
struct Cfg {
    static constexpr int MAX_PA = 5, MAX_PB = (LTB == 1) ? 2 : 5;
    static constexpr int PANEL_A = a_rows(LT) * 16, PANEL_B = a_rows(LTB) * 16;      // bytes per channel panel [row][8] bf16
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
    static constexpr int STAGE_BLOCKS = (LTB == 1) ? 18 : 8;
    static constexpr int STAGE_BYTES = STAGE_BLOCKS * 2048;       // per CTA: its output-channel half of the stage's K-blocks
    static constexpr int STAGES_PER_LAYER = 72 / STAGE_BLOCKS;
    static constexpr int IN_STAGES = (LTB == 1) ? 1 : 2;          // conv_input: 16 / 18 tap slots (9 used)
    static constexpr int STAGES = (LTB == 1) ? 3 : 4;
    static constexpr int BAR_OFF = W_OFF + STAGES * STAGE_BYTES;
    static constexpr int HEAD_OFF = BAR_OFF + 512;        // [128*LT rows][4] floats: head partial sums
    static constexpr int SMEM_BYTES = HEAD_OFF + 128 * LT * 16;
    static_assert(SMEM_BYTES <= 232448, "shared memory");
};

// geometry of one group inside its CTA pair (uniform per CTA)
struct Geo {
    int P;          // positions
    int T0;         // tiles of rank 0 (= MMA pair indices in use: rank 0 never has fewer tiles than rank 1)
    int T1;         // tiles of rank 1
    int tiles;      // tiles of this CTA
    int tile0;      // first tile of this CTA within the group
    int bnd_tile;   // local tile that touches the peer's rows
    bool has_peer;  // the other CTA holds rows of this group too
};
__device__ __forceinline__ Geo make_geo(int P, uint32_t rank) {
    Geo g;
    g.P = P;
    const int T = (P * POS_ROWS + 127) / 128;
    g.T0 = (T + 1) >> 1;
    g.T1 = T - g.T0;
    g.tiles = (rank == 0) ? g.T0 : T - g.T0;
    g.tile0 = (rank == 0) ? 0 : g.T0;
    g.has_peer = (T - g.T0) > 0;
    g.bnd_tile = (rank == 0) ? g.tiles - 1 : 0;
    return g;
}

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
                int n_pos,                                   // the batch size
                const int* src_rows) {                       // slot mode (net_auto.cu): position i of this pair reads planes row
                                                             // src_rows[i], else null
    using C = Cfg<LTB>;
    constexpr int STAGES = C::STAGES, BAR_OFF = C::BAR_OFF, HEAD_OFF = C::HEAD_OFF, CONST_OFF = C::CONST_OFF,
                  STAGE_BLOCKS = C::STAGE_BLOCKS, STAGE_BYTES = C::STAGE_BYTES, STAGES_PER_LAYER = C::STAGES_PER_LAYER,
                  IN_STAGES = C::IN_STAGES;
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
    const Geo geo[NG] = {make_geo(PA, rank), make_geo(Ptot - PA, rank)};
    const bool any_tiles = geo[0].T0 + geo[1].T0 > 0;         // pair-level: both CTAs stream the weights of a group that exists

    uint8_t* sA = smem;
    const uint32_t sA_u = smem_u32(sA);
    const uint32_t sB_u = sA_u + C::W_OFF;
    // per group: offset of its activation buffer, bytes per channel panel
    auto grp_off = [](int g) { return (uint32_t)(g == 0 ? 0 : C::A_BYTES); };
    auto grp_panel = [](int g) { return (uint32_t)(g == 0 ? C::PANEL_A : C::PANEL_B); };
    const uint32_t bar_u = sA_u + BAR_OFF;
    // barriers: full[STAGES], empty[STAGES], then per group accum[LT], act[LT]; then the tmem base holder.  The leader's
    // full / act barriers also count an arrive forwarded by the peer ("my half of the stage has landed" / "my rows of the
    // tile pair are in place"), so its issuers wait on one barrier per event.
    const uint32_t bar_full = bar_u, bar_empty = bar_u + 8 * STAGES, bar_grp = bar_u + 16 * STAGES;
    constexpr int GRP_BARS = 2 * LT;
    auto bar_accum = [&](int g, int t) { return bar_grp + 8u * (uint32_t)(g * GRP_BARS + t); };
    auto bar_act = [&](int g, int t) { return bar_grp + 8u * (uint32_t)(g * GRP_BARS + LT + t); };
    static_assert(16 * STAGES + 8 * NG * GRP_BARS + 4 <= 512, "barrier block");
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(smem + BAR_OFF + 16 * STAGES + 8 * NG * GRP_BARS);
    const int bnd_quarter = (rank == 0) ? 3 : 0;              // the quarter-warp that owns the rows next to the peer

    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; i++) {
            mbar_init(bar_full + 8 * i, rank == 0 ? 2 : 1);      // own producer (+ the peer's forwarded arrive)
            mbar_init(bar_empty + 8 * i, LT);                     // multicast commits of the leader's LT issuers
        }
        for (int g = 0; g < NG; g++) {
            for (int t = 0; t < LT; t++) {
                mbar_init(bar_accum(g, t), 1);
                // own 8 epilogue warps + the 2 boundary warps of each row neighbour (the peer's halo rows arrive as
                // transaction bytes) + on the leader the peer's forwarded arrive for its tile of the same index
                mbar_init(bar_act(g, t), 8 + (t > 0 ? 2 : 0) + (t < geo[g].tiles - 1 ? 2 : 0) + ((rank == 0 && t < geo[g].T1) ? 1 : 0));
            }
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == EPI_WARPS + 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_holder)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    for (int i = threadIdx.x; i < (C::A_BYTES + C::B_BYTES) / 16; i += THREADS) reinterpret_cast<uint4*>(sA)[i] = make_uint4(0, 0, 0, 0);
    // constant A block: every row = (1, 1, 0, ..., 0).  One extra K=16 MMA per tile and layer multiplies it with the
    // layer's bias block (shift_hi, shift_lo in k = 0, 1): the BatchNorm shift is added by the tensor pipe.
    for (int i = threadIdx.x; i < CONST_BYTES / 16; i += THREADS)
        reinterpret_cast<uint4*>(sA + CONST_OFF)[i] = (i < 128) ? make_uint4(0x3F803F80u, 0, 0, 0) : make_uint4(0, 0, 0, 0);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the peer's barriers and margins exist before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    int iter = 0;
    for (int sg = pair; sg < n_super; sg += n_pairs, iter++) {
        if (warp < EPI_WARPS) {
            // ================= epilogue warps: (tile, TMEM lane quarter, 64-column half), both groups =================
            const int lt = warp >> 3, quarter = warp & 3, chalf = (warp >> 2) & 1;
            const int lr = lt * 128 + quarter * 32 + lane;                   // local GEMM row
            const uint4 zero4 = make_uint4(0, 0, 0, 0);
            constexpr uint32_t HALO_BYTES = 11 * 16;
            float4* hscr = reinterpret_cast<float4*>(smem + HEAD_OFF) + lr;

            // everything a thread needs to know about its row in group g (recomputed per call: the epilogue is off the
            // critical path here, registers are not)
            struct Row {
                bool active, valid, nb_lo, nb_hi, bnd;
                int gpos, cell;
            };
            auto row_of = [&](int g) {
                Row r;
                const Geo& G = geo[g];
                r.active = lt < G.tiles;
                const int gr = G.tile0 * 128 + lr;                               // row within the group
                const int pos = gr / POS_ROWS, idx = gr - pos * POS_ROWS;
                const int rr = idx / 10, cc = idx - 10 * rr;
                r.gpos = sg * Ptot + (g == 0 ? 0 : PA) + pos;
                r.cell = rr * 9 + cc;
                r.valid = (pos < G.P) && (rr < 9) && (cc < 9) && (r.gpos < n_pos);
                r.nb_lo = (quarter == 0) && (lt > 0);
                r.nb_hi = (quarter == 3) && (lt < G.tiles - 1);
                r.bnd = G.has_peer && (lt == G.bnd_tile) && (quarter == bnd_quarter);
                return r;
            };
            // boundary rows of this CTA (rank 0: its last rows -> the peer's lead margin, rank 1: its first rows -> the
            // peer's tail margin), pushed panel by panel with bulk shared->shared copies that count their bytes on the
            // peer's act_ready barrier; the peer's chalf-0 boundary warp announces them with expect_tx
            auto push_halo = [&](int g, int panel, int n_panels) {
                const Geo& G = geo[g];
                const uint32_t PANEL_BYTES = grp_panel(g);
                const uint32_t base = sA_u + grp_off(g) + (uint32_t)panel * PANEL_BYTES;
                const uint32_t src = base + (uint32_t)(LEAD + ((rank == 0) ? (128 * G.tiles - 11) : 0)) * 16u;
                const uint32_t dst = map_to_rank(base + (uint32_t)((rank == 0) ? 0 : (LEAD + 128 * G.T0)) * 16u, peer);
                const uint32_t pbar = map_to_rank(bar_act(g, (rank == 0) ? 0 : (G.T0 - 1)), peer);
                for (int p = 0; p < n_panels; p++)
                    bulk_s2peer(dst + (uint32_t)p * PANEL_BYTES, src + (uint32_t)p * PANEL_BYTES, HALO_BYTES, pbar);
            };
            auto publish = [&](int g, const Row& r, uint32_t tx) {
                if (r.bnd && chalf == 0) mbar_expect_tx(bar_act(g, lt), tx);
                else mbar_arrive(bar_act(g, lt));
                if (r.nb_lo) mbar_arrive(bar_act(g, lt - 1));
                if (r.nb_hi) mbar_arrive(bar_act(g, lt + 1));
            };

            // prologue: the three input planes of a row go into channel panel 0 (channels 3..15 are zero): the A operand
            // of conv_input, which runs as "layer -1" on the tensor pipe with K = 16 per tap
#pragma unroll 1
            for (int g = 0; g < NG; g++) {
                const Row r = row_of(g);
                if (!r.active) continue;
                uint4 pk = zero4;
                if (chalf == 0 && r.valid) {
                    const __nv_bfloat16* px = planes + (size_t)(src_rows ? src_rows[r.gpos - sg * Ptot] : r.gpos) * 243 + (size_t)r.cell;
                    uint32_t x0 = (uint32_t)__bfloat16_as_ushort(px[0]), x1 = (uint32_t)__bfloat16_as_ushort(px[81]),
                             x2 = (uint32_t)__bfloat16_as_ushort(px[162]);
                    pk = make_uint4(x0 | (x1 << 16), x2, 0u, 0u);
                }
                *reinterpret_cast<uint4*>(sA + grp_off(g) + (size_t)chalf * grp_panel(g) + (size_t)(LEAD + lr) * 16) = pk;
                fence_async_smem();
                __syncwarp();
                if (lane == 0) {
                    publish(g, r, 2 * HALO_BYTES);
                    if (r.bnd) push_halo(g, chalf, 1);
                }
            }

            auto epilogue_layer = [&](int g, int layer, auto last_tag) {
                constexpr bool last = decltype(last_tag)::value;
                const Row r = row_of(g);
                if (!r.active) return;
                const uint32_t lpar = (uint32_t)((iter * GROUP_LAYERS + layer + 1) & 1);
                const bool second = (layer >= 0) && (layer & 1) != 0;   // conv2 of a block: add the skip connection
                const bool keep = second || (layer < 0);                // output is the input of the next block: keep it as skip
                uint4* srow_skip = skip + (size_t)(blockIdx.x * NG + g) * (16 * SKIP_ROWS) + (size_t)(chalf * 8) * SKIP_ROWS + (size_t)lr;
                const uint32_t PANEL_BYTES = grp_panel(g);
                uint8_t* srow = sA + grp_off(g) + (size_t)(chalf * 8) * PANEL_BYTES + (size_t)(LEAD + lr) * 16;
                const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((g * LT + lt) * 128 + chalf * 64);
                // the skip connection (8 x 16 B per thread) is fetched from L2 while the MMAs still run
                uint4 sk[8];
#pragma unroll
                for (int j = 0; j < 8; j++) sk[j] = (second && r.valid) ? srow_skip[(size_t)j * SKIP_ROWS] : zero4;
                mbar_wait_spin<false>(bar_accum(g, lt), lpar);
                if (r.nb_lo) mbar_wait_spin<false>(bar_accum(g, lt - 1), lpar);
                if (r.nb_hi) mbar_wait_spin<false>(bar_accum(g, lt + 1), lpar);
                // the peer's boundary tile has retired too: its MMAs are the other half of the pair MMAs of index 0 (rank 1's
                // first tile) / T0-1 (rank 0's last tile), whose commits arrive on this CTA's barrier of that index
                if (r.bnd) mbar_wait_spin<false>(bar_accum(g, (rank == 0) ? 0 : geo[g].T0 - 1), lpar);
                if (dbg && blockIdx.x == 0 && iter == 0 && threadIdx.x == 0 && layer >= 0 && layer < 16) dbg[(16 * g + layer) * 4 + 2] = clock64();
                tc_fence_after();
                float va[16], vb[16];
                float h0 = 0.0f, h1 = 0.0f, h2 = 0.0f;               // last layer: the heads' 1x1 convolutions of this row
                tmem_ld16(taddr, va);
#pragma unroll
                for (int ch = 0; ch < 4; ch++) {
                    float* v = (ch & 1) ? vb : va;
                    float* o = (ch & 1) ? va : vb;
                    tmem_ld_wait();
                    if (ch < 3) tmem_ld16(taddr + (uint32_t)((ch + 1) * 16), o);
                    f16x8_add2(sk[2 * ch], v);
                    f16x8_add2(sk[2 * ch + 1], v + 8);
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
                            uint4 pk = r.valid ? relu_pack8_bf16(v + 8 * j) : zero4;      // padding rows stay zero
                            *reinterpret_cast<uint4*>(srow + (size_t)(ch * 2 + j) * PANEL_BYTES) = pk;
                            if (keep && r.valid) srow_skip[(size_t)(ch * 2 + j) * SKIP_ROWS] = relu_pack8_f16(v + 8 * j);
                        }
                    }
                }
                if constexpr (!last) {
                    fence_async_smem();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        publish(g, r, 16 * HALO_BYTES);
                        if (r.bnd) push_halo(g, chalf * 8, 8);
                    }
                } else {
                    // combine the two column halves of the row (two warps) and emit BN shift + ReLU of the head convs
                    tc_fence_before();
                    if (chalf == 1) *hscr = make_float4(h0, h1, h2, 0.0f);
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + lt * 4 + quarter) : "memory");
                    if (chalf == 0 && r.valid) {
                        float4 o = *hscr;
                        float* hrow = headfeat + (size_t)r.gpos * 243 + (size_t)r.cell;
                        hrow[0] = fmaxf(h0 + o.x + __ldg(headw + 384), 0.0f);
                        hrow[81] = fmaxf(h1 + o.y + __ldg(headw + 385), 0.0f);
                        hrow[162] = fmaxf(h2 + o.z + __ldg(headw + 386), 0.0f);
                    }
                    asm volatile("bar.sync %0, 64;" ::"r"(1 + lt * 4 + quarter) : "memory");   // hscr is reused by the other group
                }
                if (dbg && blockIdx.x == 0 && iter == 0 && threadIdx.x == 0 && layer >= 0 && layer < 16) dbg[(16 * g + layer) * 4 + 3] = clock64();
            };
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS - 1; layer++) {
#pragma unroll 1
                for (int g = 0; g < NG; g++) epilogue_layer(g, layer, std::false_type{});
            }
#pragma unroll 1
            for (int g = 0; g < NG; g++) epilogue_layer(g, NET_LAYERS - 1, std::true_type{});
        } else if (warp == EPI_WARPS) {
            // ================= weight producer: this CTA's output-channel half of every layer, once per group =========
            if (!any_tiles) continue;
            int stage = 0;
            uint32_t par = 0;
            {
                // the ring position continues across super-groups
                int per_group = (IN_STAGES + 1) + NET_LAYERS * (STAGES_PER_LAYER + 1);
                int gn = iter * per_group * ((geo[0].T0 > 0) + (geo[1].T0 > 0));
                stage = gn % STAGES;
                par = (uint32_t)((gn / STAGES) & 1);
            }
#pragma unroll 1
            for (int layer = -1; layer < NET_LAYERS; layer++) {
                const int n_st = 1 + ((layer < 0) ? IN_STAGES : STAGES_PER_LAYER);
#pragma unroll 1
                for (int g = 0; g < NG; g++) {
                    if (geo[g].T0 == 0) continue;
#pragma unroll 1
                    for (int st = 0; st < n_st; st++) {
                        mbar_wait(bar_empty + 8 * stage, par ^ 1u);
                        if (lane == 0) {
                            const __nv_bfloat16* src;
                            uint32_t bytes = STAGE_BYTES;
                            if (st == 0) { src = wq_bias + (size_t)((layer + 1) * 2 + (int)rank) * (BIAS_BYTES / 2); bytes = BIAS_BYTES; }
                            else if (layer < 0) src = wq_in + (size_t)((st - 1) * 2 + (int)rank) * (STAGE_BYTES / 2);
                            else src = wq + (size_t)((layer * STAGES_PER_LAYER + st - 1) * 2 + (int)rank) * (STAGE_BYTES / 2);
                            mbar_expect_tx(bar_full + 8 * stage, bytes);
                            bulk_g2s(sB_u + stage * STAGE_BYTES, src, bytes, bar_full + 8 * stage);
                        }
                        __syncwarp();
                        if (++stage == STAGES) { stage = 0; par ^= 1u; }
                    }
                }
            }
        } else if (rank != 0) {
            // ================= rank 1 has no MMAs to issue (the leader issues for the pair): its two issuer warps forward
            // its barriers to the leader.  Warp EPI_WARPS+1: "my half of weight stage i has landed"; warp EPI_WARPS+2: "my
            // rows of tile pair t of group g are in place".  CTA-scope arrives on the leader's barriers (no MEMBAR.GPU): the
            // data they announce sit in THIS CTA's shared memory, fenced for the async proxy by their writers, and are read
            // by this CTA's tensor pipe when the leader's MMA executes.
            if (!any_tiles) continue;
            if (warp == EPI_WARPS + 1) {
                int stage = 0;
                uint32_t par = 0;
                {
                    int per_group = (IN_STAGES + 1) + NET_LAYERS * (STAGES_PER_LAYER + 1);
                    int gn = iter * per_group * ((geo[0].T0 > 0) + (geo[1].T0 > 0));
                    stage = gn % STAGES;
                    par = (uint32_t)((gn / STAGES) & 1);
                }
                const int total = ((geo[0].T0 > 0) + (geo[1].T0 > 0)) * ((IN_STAGES + 1) + NET_LAYERS * (STAGES_PER_LAYER + 1));
#pragma unroll 1
                for (int i = 0; i < total; i++) {
                    mbar_wait_spin<false>(bar_full + 8 * stage, par);
                    if (lane == 0) mbar_arrive_peer(map_to_rank(bar_full + 8 * stage, 0));
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; par ^= 1u; }
                }
            } else {
#pragma unroll 1
                for (int layer = -1; layer < NET_LAYERS; layer++) {
                    const uint32_t apar = (uint32_t)((iter * GROUP_LAYERS + layer + 1) & 1);
#pragma unroll 1
                    for (int g = 0; g < NG; g++) {
#pragma unroll 1
                        for (int t = 0; t < geo[g].T1; t++) {
                            mbar_wait_spin<false>(bar_act(g, t), apar);
                            if (lane == 0) mbar_arrive_peer(map_to_rank(bar_act(g, t), 0));
                            __syncwarp();
                        }
                    }
                }
            }
        } else {
            // ================= leader CTA: warp EPI_WARPS+1+t issues the pair MMAs (cta_group::2, M = 256: tile t of this CTA
            // and tile t of the peer) of both groups ==========
            if (!any_tiles) continue;
            const int lt = warp - (EPI_WARPS + 1);
            const bool leader = elect_one();
            const uint64_t b_desc = make_desc(sB_u, 1024, 128);           // this CTA's 64 output channels: [2 panels][64][8]
            const uint64_t bias_a = make_desc(sA_u + CONST_OFF, 2048, 128);
            int stage = 0;
            uint32_t par = 0;
            {
                int per_group = (IN_STAGES + 1) + NET_LAYERS * (STAGES_PER_LAYER + 1);
                int gn = iter * per_group * ((geo[0].T0 > 0) + (geo[1].T0 > 0));
                stage = gn % STAGES;
                par = (uint32_t)((gn / STAGES) & 1);
            }
            uint64_t b_st = 0;
            auto next_stage = [&]() {              // both halves of the next weight stage have landed; b_st = its first block
                mbar_wait_spin<false>(bar_full + 8 * stage, par);
                tc_fence_after();
                b_st = b_desc + (uint64_t)(uint32_t)(stage * (STAGE_BYTES / 16));
            };
            auto release_stage = [&]() {           // frees the stage in both CTAs when the MMAs issued so far retire
                umma_commit_2sm(bar_empty + 8 * stage, (uint16_t)3);
            };
            auto advance = [&]() {
                if (++stage == STAGES) { stage = 0; par ^= 1u; }
            };
            // per group, fixed for the kernel: does this thread issue for it, into which accumulator, from which rows
            bool g_stream[NG], g_issue[NG];
            uint32_t g_tmem[NG], g_act[NG], g_accum[NG];
            uint64_t g_adesc[NG];
            int g_panel16[NG];
#pragma unroll
            for (int g = 0; g < NG; g++) {
                const Geo& G = geo[g];
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
                const uint32_t apar = (uint32_t)((iter * GROUP_LAYERS + layer + 1) & 1);
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
                    if (dbg && blockIdx.x == 0 && iter == 0 && lt == 0 && leader && layer >= 0 && layer < 16) dbg[(16 * g + layer) * 4 + 0] = clock64();
                    // accumulator := BN shift (constant rows x bias block); starts the layer's accumulation
                    next_stage();
                    if (mine && leader) umma_bf16_2sm(tmem_d, bias_a, b_st, IDESC, 0u);
                    if (leader) release_stage();
                    advance();
                    if (layer < 0) {
                        // conv_input: block j of stage s is tap 8s+j, K = 16 (channel panels 0,1)
#pragma unroll
                        for (int s = 0; s < IN_STAGES; s++) {
                            next_stage();
                            if (mine && leader) {
#pragma unroll
                                for (int j = 0; j < STAGE_BLOCKS; j++) {
                                    const int tap = STAGE_BLOCKS * s + j;
                                    if (tap < 9)
                                        umma_bf16_2sm(tmem_d, a_desc + (uint64_t)(int64_t)((tap / 3 - 1) * 10 + (tap % 3 - 1)),
                                                      b_st + (uint64_t)(j * 128), IDESC, 1u);
                                }
                            }
                            if (leader) {
                                release_stage();
                                if (mine && s == IN_STAGES - 1) umma_commit_2sm(g_accum[g], (uint16_t)3);
                            }
                            advance();
                        }
                    } else {
                        // stage s holds K-blocks STAGE_BLOCKS * s ... in the order of tcx::kblock_of
#pragma unroll
                        for (int s = 0; s < STAGES_PER_LAYER; s++) {
                            next_stage();
                            if (mine && leader) {
#pragma unroll
                                for (int ks = 0; ks < STAGE_BLOCKS; ks++) {
                                    const int m = STAGE_BLOCKS * s + ks, q = m / 18, rr = m % 18, tap = rr >> 1, unit = q + 4 * (rr & 1);
                                    const int off = (tap / 3 - 1) * 10 + (tap % 3 - 1) + 2 * unit * panel16;
                                    umma_bf16_2sm(tmem_d, a_desc + (uint64_t)(int64_t)off, b_st + (uint64_t)(ks * 128), IDESC, 1u);
                                }
                            }
                            if (leader) {
                                release_stage();
                                if (mine && s == STAGES_PER_LAYER - 1) {
                                    umma_commit_2sm(g_accum[g], (uint16_t)3);
                                    if (dbg && blockIdx.x == 0 && iter == 0 && lt == 0 && layer < 16) dbg[(16 * g + layer) * 4 + 1] = clock64();
                                }
                            }
                            advance();
                        }
                    }
                }
            }
            __syncwarp();
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // nobody exits while the peer may still write its margins / barriers
    if (warp == EPI_WARPS + 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

}  // namespace pp
}  // namespace uttt
