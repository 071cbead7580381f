// trunk_pair.cuh -- the pieces of the CTA-pair trunk pipeline shared by its two schedules, tc2::trunk_tc2_body
// (net_tc2_kernel.cuh: next layer overlaps the epilogue) and pp::trunk_pp_body (net_pp_kernel.cuh: two groups alternate).
// Both run a group of positions on a cluster of two CTAs: positions padded to 100 GEMM rows, the group's accumulator tiles
// split between the CTAs (rank 0 takes the first ceil(T/2)), cta_group::2 MMAs issued by the leader (rank 0) for both,
// each CTA streaming its output-channel half of every weight block through a ring of stages, the 11 halo rows at the split
// pushed to the peer with bulk shared->shared copies, conv_input run as "layer -1" and the BN shift added by a bias MMA.
// Each body keeps its own schedule (its loops, warp roles and barrier counts); nothing here depends on which body calls it.
#pragma once
#include "tc_common.cuh"

namespace uttt {
namespace tp {

using namespace tcx;

constexpr int POS_ROWS = 100;                   // GEMM rows per position: row = 10 r + c (column 9 and rows 90..99 are zero)
constexpr int LEAD = 11;                        // margin rows before a CTA's first tile (the halo rows of its first row)
constexpr int HALO_ROWS = 11;                   // rows a 3x3 tap reaches across a tile boundary
constexpr uint32_t HALO_BYTES = HALO_ROWS * 16; // the halo rows of one channel panel
constexpr int GROUP_LAYERS = NET_LAYERS + 1;    // conv_input runs as layer -1 through the same pipeline
constexpr uint32_t TMEM_COLS = 512u;
// rows of a CTA's activation panel: lead margin, its tiles, tail margin
constexpr int a_rows(int tiles) { return (LEAD + 128 * tiles + HALO_ROWS + 7) / 8 * 8; }

// ---------------------------------------------------------------- pair geometry

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
    g.tiles = (rank == 0) ? g.T0 : g.T1;
    g.tile0 = (rank == 0) ? 0 : g.T0;
    g.has_peer = g.T1 > 0;
    g.bnd_tile = (rank == 0) ? g.tiles - 1 : 0;
    return g;
}
// the peer's tile next to this CTA's rows (rank 1's first, rank 0's last): its pair MMAs are the other half of this
// index's, so their multicast commits arrive on this CTA's accumulator barrier of that index
__device__ __forceinline__ int peer_tile(const Geo& G, uint32_t rank) { return (rank == 0) ? 0 : G.T0 - 1; }

// an epilogue thread's GEMM row: lane `lane` of TMEM lane quarter `quarter` of local tile lt
struct Row {
    int gpos;       // position in the batch
    int cell;       // 9 r + c
    bool valid;     // a real cell of a position of the batch (padding rows stay zero)
    bool nb_lo;     // the quarter-warp whose rows the previous tile's last taps read
    bool nb_hi;     // the quarter-warp whose rows the next tile's first taps read
    bool bnd;       // the quarter-warp whose rows the peer's boundary tile reads
};
__device__ __forceinline__ Row row_of(const Geo& G, int lt, int quarter, int lane, int pos0 /* the group's first position */,
                                      int n_pos, uint32_t rank) {
    Row w;
    const int gr = G.tile0 * 128 + lt * 128 + quarter * 32 + lane;     // row within the group
    const int pos = gr / POS_ROWS, idx = gr - pos * POS_ROWS;
    const int r = idx / 10, c = idx - 10 * r;
    w.gpos = pos0 + pos;
    w.cell = r * 9 + c;
    w.valid = (pos < G.P) && (r < 9) && (c < 9) && (w.gpos < n_pos);
    w.nb_lo = (quarter == 0) && (lt > 0);
    w.nb_hi = (quarter == 3) && (lt < G.tiles - 1);
    w.bnd = G.has_peer && (lt == G.bnd_tile) && (quarter == ((rank == 0) ? 3 : 0));
    return w;
}

// halo of one channel panel (`panel`: its address in this CTA's shared memory, the same offset in the peer's): rank 0
// sends its last 11 rows into the peer's lead margin, rank 1 its first 11 rows into the peer's tail margin
__device__ __forceinline__ uint32_t halo_src(uint32_t panel, const Geo& G, uint32_t rank) {
    return panel + (uint32_t)(LEAD + ((rank == 0) ? (128 * G.tiles - HALO_ROWS) : 0)) * 16u;
}
__device__ __forceinline__ uint32_t halo_dst(uint32_t panel, const Geo& G, uint32_t rank) {
    return map_to_rank(panel + (uint32_t)((rank == 0) ? 0 : (LEAD + 128 * G.T0)) * 16u, rank ^ 1u);
}

// ---------------------------------------------------------------- set-up and tear-down

// act_ready barrier of local tile t: its 8 epilogue warps + the 2 boundary warps of each row neighbour (the peer's halo
// rows arrive as transaction bytes) + on the leader the peer's forwarded "my rows of tile pair t are in place"
__device__ __forceinline__ uint32_t act_count(const Geo& G, int t, uint32_t rank) {
    return 8 + (t > 0 ? 2 : 0) + (t < G.tiles - 1 ? 2 : 0) + ((rank == 0 && t < G.T1) ? 1 : 0);
}
// one warp: the pair's 512 TMEM columns (relinquish: this CTA allocates no more in this launch)
__device__ __forceinline__ void tmem_alloc(uint32_t* holder, bool relinquish) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(holder)), "r"(TMEM_COLS)
                 : "memory");
    if (relinquish) asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
// all THREADS threads: zero the first `zero_bytes` of shared memory (activation panels: padding rows and margins stay
// zero), then write the A operand of the bias MMA: `rows` rows of (1, 1, 0, ..., 0) at `bias_off`.  One extra K=16 MMA per tile and layer
// multiplies it with the layer's bias block (shift_hi, shift_lo in k = 0, 1), so the BatchNorm shift is added by the
// tensor pipe and the epilogue has no bias loads or adds (measured: -20 % epilogue time).  X3: rows (1, 1, 1, 0, ...), the
// shift comes as three bf16 terms.
template <bool X3, int THREADS>
__device__ __forceinline__ void init_operands(uint8_t* smem, int zero_bytes, int bias_off, int rows) {
    for (int i = threadIdx.x; i < zero_bytes / 16; i += THREADS) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    for (int i = threadIdx.x; i < rows; i += THREADS)
        reinterpret_cast<uint4*>(smem + bias_off)[i] = make_uint4(0x3F803F80u, X3 ? 0x00003F80u : 0u, 0, 0);
}
// every thread, after the barrier inits and init_operands: the peer's barriers and margins exist before anyone signals
// them, the zeroed operands are visible to the tensor pipe.  Returns the TMEM base.
__device__ __forceinline__ uint32_t setup_sync(const uint32_t* tmem_holder) {
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    return *tmem_holder;
}
// every thread: nobody exits while the peer may still write its margins / barriers; `dealloc`: the warp that allocated
__device__ __forceinline__ void teardown(uint32_t tmem_base, bool dealloc) {
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (dealloc) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
}

// ---------------------------------------------------------------- weight stream

// One CTA's weight stream: per layer its bias block (the BN shift as one K=16 B block of BIAS_BYTES), then its 72 K-blocks
// (conv_input: one block per tap, 9 of IN_STAGES * STAGE_BLOCKS slots used) in stages of STAGE_BLOCKS blocks of
// BLOCK_BYTES, through a ring of STAGES slots.  The weights hold per-CTA halves, stage-major: [stage][2 ranks][STAGE_BLOCKS
// blocks], the bias blocks [33 layers][2 ranks].
template <int STAGES_, int STAGE_BLOCKS_, int BLOCK_BYTES_, int BIAS_BYTES_>
struct Stream {
    static constexpr int STAGES = STAGES_, STAGE_BLOCKS = STAGE_BLOCKS_, BLOCK_BYTES = BLOCK_BYTES_, BIAS_BYTES = BIAS_BYTES_;
    static constexpr int STAGE_BYTES = STAGE_BLOCKS * BLOCK_BYTES;
    static constexpr int STAGES_PER_LAYER = 72 / STAGE_BLOCKS;
    static constexpr int IN_STAGES = (9 + STAGE_BLOCKS - 1) / STAGE_BLOCKS;
    static constexpr int GROUP_STAGES = (IN_STAGES + 1) + NET_LAYERS * (STAGES_PER_LAYER + 1);   // ring slots per group
    static_assert(72 % STAGE_BLOCKS == 0, "a stage holds K-blocks of one layer");
    __device__ static int layer_stages(int layer) { return 1 + ((layer < 0) ? IN_STAGES : STAGES_PER_LAYER); }
};

// A cursor into the ring: slot `stage` in its use of parity `par`.  The producer, the issuers and rank 1's forwarder each
// walk the ring with their own, all starting a group at the same ring position (the slots used by the pair so far).
// Barriers at `bars`: full[STAGES], then empty[STAGES].
template <class S>
struct Ring {
    uint32_t bars;
    int stage;
    uint32_t par;
    __device__ __forceinline__ Ring(uint32_t bars_, int pos) : bars(bars_), stage(pos % S::STAGES), par((uint32_t)((pos / S::STAGES) & 1)) {}
    // full: the own producer (+ on the leader the peer's forwarded "my half has landed"); empty: the multicast commits of
    // the leader's `issuers` issuer threads
    __device__ static void init(uint32_t bars, uint32_t rank, uint32_t issuers) {
        for (int i = 0; i < S::STAGES; i++) {
            mbar_init(bars + 8 * i, rank == 0 ? 2 : 1);
            mbar_init(bars + 8 * (S::STAGES + i), issuers);
        }
    }
    __device__ __forceinline__ uint32_t full() const { return bars + 8u * (uint32_t)stage; }
    __device__ __forceinline__ uint32_t empty() const { return bars + 8u * (uint32_t)(S::STAGES + stage); }
    // issuer: waits until both halves of the slot have landed; returns the B descriptor of its first block
    __device__ __forceinline__ uint64_t next_stage(uint64_t b_desc) const {
        mbar_wait_spin<false>(full(), par);
        tc_fence_after();
        return b_desc + (uint64_t)(uint32_t)(stage * (S::STAGE_BYTES / 16));
    }
    // leader issuer: frees the slot in both CTAs when the MMAs issued so far retire
    __device__ __forceinline__ void release_stage() const { umma_commit_2sm(empty(), (uint16_t)3); }
    __device__ __forceinline__ void advance() {
        if (++stage == S::STAGES) { stage = 0; par ^= 1u; }
    }
};

// producer warp: stage st of layer `layer` (st = 0: the layer's bias block) of this CTA's weight half into the next slot
template <class S>
__device__ __forceinline__ void produce_stage(Ring<S>& ring, uint32_t sB_u, const __nv_bfloat16* wq, const __nv_bfloat16* wq_in,
                                              const __nv_bfloat16* wq_bias, int layer, int st, uint32_t rank, int lane) {
    mbar_wait(ring.empty(), ring.par ^ 1u);
    if (lane == 0) {
        const int rk = (int)rank;
        const __nv_bfloat16* src;                           // (offsets in bf16 elements)
        uint32_t bytes = S::STAGE_BYTES;
        if (st == 0) { src = wq_bias + (size_t)((layer + 1) * 2 + rk) * (S::BIAS_BYTES / 2); bytes = S::BIAS_BYTES; }
        else if (layer < 0) src = wq_in + (size_t)((st - 1) * 2 + rk) * (S::STAGE_BYTES / 2);
        else src = wq + (size_t)((layer * S::STAGES_PER_LAYER + st - 1) * 2 + rk) * (S::STAGE_BYTES / 2);
        mbar_expect_tx(ring.full(), bytes);
        bulk_g2s(sB_u + ring.stage * S::STAGE_BYTES, src, bytes, ring.full());
    }
    __syncwarp();
    ring.advance();
}

// Rank 1 issues no MMAs (the leader issues for the pair): its issuer warps forward its barriers to the leader's barrier
// of the same address with CTA-scope remote arrives (no MEMBAR.GPU): the data they announce sit in THIS CTA's shared
// memory, fenced for the async proxy by their writers, and are read by this CTA's tensor pipe when the leader's MMA
// executes.  Neither forwarder can be lapped: the events it waits for need the leader's next MMAs, which need its arrive.
__device__ __forceinline__ void forward_to_leader(uint32_t bar, uint32_t par, int lane) {
    mbar_wait_spin<false>(bar, par);
    if (lane == 0) mbar_arrive_peer(map_to_rank(bar, 0));
    __syncwarp();
}
// "my half of weight stage i has landed", for the next n slots
template <class S>
__device__ __forceinline__ void forward_stages(Ring<S> ring, int n, int lane) {
#pragma unroll 1
    for (int i = 0; i < n; i++) {
        forward_to_leader(ring.full(), ring.par, lane);
        ring.advance();
    }
}

// ---------------------------------------------------------------- epilogue

// prologue: the three input planes of a row (px: its cell in plane 0 of planes [rows][3][81]; load = false: zeros) into
// channel panel 0, channels 3..15 zero -- the A operand of conv_input, which runs with K = 16 per tap
__device__ __forceinline__ void write_input_row(uint8_t* dst, const __nv_bfloat16* px, bool load) {
    uint4 pk = make_uint4(0, 0, 0, 0);
    if (load) {
        uint32_t x0 = (uint32_t)__bfloat16_as_ushort(px[0]), x1 = (uint32_t)__bfloat16_as_ushort(px[81]),
                 x2 = (uint32_t)__bfloat16_as_ushort(px[162]);
        pk = make_uint4(x0 | (x1 << 16), x2, 0u, 0u);
    }
    *reinterpret_cast<uint4*>(dst) = pk;
}

// Before a thread overwrites its rows in place, every MMA that reads them has retired: its own tile's, its row
// neighbours' (their taps reach 11 rows into this tile) and, for the boundary rows, the peer's boundary tile's.
// accum0: the accumulator barrier of local tile 0 (tiles 8 bytes apart).
__device__ __forceinline__ void wait_rows_free(uint32_t accum0, const Row& w, int lt, int peer_t, uint32_t par) {
    mbar_wait_spin<false>(accum0 + 8u * (uint32_t)lt, par);
    if (w.nb_lo) mbar_wait_spin<false>(accum0 + 8u * (uint32_t)(lt - 1), par);
    if (w.nb_hi) mbar_wait_spin<false>(accum0 + 8u * (uint32_t)(lt + 1), par);
    if (w.bnd) mbar_wait_spin<false>(accum0 + 8u * (uint32_t)peer_t, par);
}
// lane 0: this warp's rows are in place, on the act_ready barrier act0 + stride * t of its own tile and of its row
// neighbours.  announce (the chalf-0 boundary warp): arrive with expect_tx of the `tx` bytes the peer pushes into this
// CTA's margin for the same barrier phase
__device__ __forceinline__ void publish_rows(uint32_t act0, uint32_t stride, const Row& w, int lt, bool announce, uint32_t tx) {
    if (announce) mbar_expect_tx(act0 + stride * (uint32_t)lt, tx);
    else mbar_arrive(act0 + stride * (uint32_t)lt);
    if (w.nb_lo) mbar_arrive(act0 + stride * (uint32_t)(lt - 1));
    if (w.nb_hi) mbar_arrive(act0 + stride * (uint32_t)(lt + 1));
}

// The 64 accumulator columns of a thread's row in 4 chunks of 16, each chunk's load overlapping the previous chunk's
// math: f(ch, v) with v = columns 16 ch .. 16 ch + 15.
template <class F>
__device__ __forceinline__ void for_each_chunk(uint32_t taddr, F&& f) {
    float va[16], vb[16];
    tmem_ld16(taddr, va);
#pragma unroll
    for (int ch = 0; ch < 4; ch++) {
        float* v = (ch & 1) ? vb : va;
        tmem_ld_wait();
        if (ch < 3) tmem_ld16(taddr + (uint32_t)((ch + 1) * 16), (ch & 1) ? va : vb);
        f(ch, v);
    }
}

// The skip connection of a row's 64 columns, srow_skip = [8 panels][SKIP_ROWS rows] fp16x8 (X3: fp32x8, 2 x 16 B), is
// fetched from L2 while the MMAs still run: 8 x 16 B per thread (X3: chunks 0 and 1; chunks 2 and 3 are refilled into
// the registers of 0 and 1 as those are used).
template <bool X3, int SKIP_ROWS>
__device__ __forceinline__ void skip_prefetch(uint4 (&sk)[8], const uint4* srow_skip, bool load) {
#pragma unroll
    for (int j = 0; j < 8; j++) {
        if constexpr (X3) sk[j] = load ? srow_skip[(size_t)(j >> 1) * SKIP_ROWS * 2 + (j & 1)] : make_uint4(0, 0, 0, 0);
        else sk[j] = load ? srow_skip[(size_t)j * SKIP_ROWS] : make_uint4(0, 0, 0, 0);
    }
}
// v (chunk ch) += its skip connection
template <bool X3, int SKIP_ROWS>
__device__ __forceinline__ void skip_add(uint4 (&sk)[8], float* v, int ch, const uint4* srow_skip, bool load) {
    if constexpr (X3) {
#pragma unroll
        for (int j = 0; j < 4; j++) f32x4_add(sk[4 * (ch & 1) + j], v + 4 * j);
        if (ch < 2 && load) {             // refill the four registers just consumed: chunk ch + 2
#pragma unroll
            for (int j = 0; j < 4; j++) sk[4 * (ch & 1) + j] = srow_skip[(size_t)(2 * (ch + 2) + (j >> 1)) * SKIP_ROWS * 2 + (j & 1)];
        }
    } else {
        f16x8_add2(sk[2 * ch], v);
        f16x8_add2(sk[2 * ch + 1], v + 8);
    }
}
// relu(v) of chunk ch as the next layer's input: bf16 into channel panels 2 ch, 2 ch + 1 of the row (srow: panel 0 of
// the thread's column half; X3: hi there, lo = bf16(x - hi) 16 panels further), and as the next block's skip connection
// (keep: fp16; X3: fp32)
template <bool X3, int SKIP_ROWS>
__device__ __forceinline__ void store_chunk(const float* v, int ch, uint8_t* srow, uint32_t panel_bytes, uint4* srow_skip, bool valid,
                                            bool keep) {
    const uint4 zero4 = make_uint4(0, 0, 0, 0);
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
            *reinterpret_cast<uint4*>(srow + (size_t)(ch * 2 + j) * panel_bytes) = hi;
            *reinterpret_cast<uint4*>(srow + (size_t)(16 + ch * 2 + j) * panel_bytes) = lo;
            if (keep && valid) {
                uint4* d = srow_skip + (size_t)(ch * 2 + j) * SKIP_ROWS * 2;
                d[0] = make_uint4(__float_as_uint(x[0]), __float_as_uint(x[1]), __float_as_uint(x[2]), __float_as_uint(x[3]));
                d[1] = make_uint4(__float_as_uint(x[4]), __float_as_uint(x[5]), __float_as_uint(x[6]), __float_as_uint(x[7]));
            }
        } else {
            uint4 pk = valid ? relu_pack8_bf16(v + 8 * j) : zero4;      // padding rows stay zero
            *reinterpret_cast<uint4*>(srow + (size_t)(ch * 2 + j) * panel_bytes) = pk;
            if (keep && valid) srow_skip[(size_t)(ch * 2 + j) * SKIP_ROWS] = relu_pack8_f16(v + 8 * j);
        }
    }
}

// Last layer: the trunk output never leaves the SM.  policy_conv / value_conv (1x1, dual_network.py:102,111) are three
// dot products over the channels this thread holds (hw: headw [3][128] at the channel of v[0]).
__device__ __forceinline__ void head_dots(float3& h, const float* v, const float* hw) {
#pragma unroll
    for (int j = 0; j < 16; j++) {
        float x = fmaxf(v[j], 0.0f);
        h.x = fmaf(x, __ldg(hw + j), h.x);
        h.y = fmaf(x, __ldg(hw + 128 + j), h.y);
        h.z = fmaf(x, __ldg(hw + 256 + j), h.z);
    }
}
// combine the two column halves of a row (its two warps, on named barrier bar_id) and write BN shift + ReLU of the head
// convs to hrow (headfeat [rows][243] at the row's cell; headw[384..386]: the shifts)
__device__ __forceinline__ void head_store(float3 h, float4* hscr, int chalf, int bar_id, bool valid, float* hrow, const float* headw) {
    if (chalf == 1) *hscr = make_float4(h.x, h.y, h.z, 0.0f);
    asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
    if (chalf == 0 && valid) {
        float4 o = *hscr;
        hrow[0] = fmaxf(h.x + o.x + __ldg(headw + 384), 0.0f);
        hrow[81] = fmaxf(h.y + o.y + __ldg(headw + 385), 0.0f);
        hrow[162] = fmaxf(h.z + o.z + __ldg(headw + 386), 0.0f);
    }
}

// diagnostics (dbg non-null): per-layer timeline of CTA 0's first group, read by uttt_debug_trunk_timeline
// (tools/trunk_timeline.py, tools/pp_timeline.py): dbg[4 * slot + k] = clock64() at event k of timeline slot `slot`
// (0: first MMA issued, 1: last MMA committed, 2: accumulators ready, 3: epilogue done); slots outside 0..31 are not
// recorded.  The caller picks one thread per event.
__device__ __forceinline__ void timeline(long long* dbg, int iter, int slot, int k) {
    if (dbg && blockIdx.x == 0 && iter == 0 && (unsigned)slot < 32u) dbg[4 * slot + k] = clock64();
}

}  // namespace tp
}  // namespace uttt
