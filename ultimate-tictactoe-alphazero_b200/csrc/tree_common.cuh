// tree_common.cuh -- helpers shared by the reference-exact (tree_kernels.cu) and throughput (tree_tp_kernels.cu)
// search kernels: node word accessors, warp-wide state load/store, Philox move sampling.
#pragma once
#include "common.cuh"

namespace uttt {

constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int WARPS_PER_BLOCK = 4;

struct TreeView {
    uint4* node;     // [node_cap]
    int32_t* path;   // [PATH_CAP]
};

__device__ __forceinline__ TreeView view_of(const TreeParams& P, int t) {
    TreeView v = {P.nodes + (size_t)t * (size_t)P.node_cap, P.path + (size_t)t * PATH_CAP};
    return v;
}

__device__ __forceinline__ uint4 make_node(int action, float p) {
    return make_uint4((uint32_t)action << 16, 0u, __float_as_uint(p), 0u);
}
__device__ __forceinline__ int node_n(const uint4& q) { return (int)(q.x & 0xFFFFu); }
__device__ __forceinline__ int node_action(const uint4& q) { return (int)((q.x >> 16) & 0x7Fu); }
__device__ __forceinline__ int node_vloss(const uint4& q) { return (int)(q.x >> 23); }
__device__ __forceinline__ uint32_t node_base(const uint4& q) { return q.w & 0xFFFFFu; }
__device__ __forceinline__ int node_cnt(const uint4& q) { return (int)(q.w >> 20); }

// a packed state is loaded by lanes 0..7 (one word each) and handed round by shuffles; the two halves are separate so
// that a kernel can issue several such loads before it consumes the first (one L2 round trip instead of one each)
__device__ __forceinline__ uint32_t warp_load_state_issue(const PackedState* p, int lane) {
    return (lane < 8) ? reinterpret_cast<const uint32_t*>(p)[lane] : 0u;
}
__device__ __forceinline__ PackedState warp_load_state_finish(uint32_t x) {
    PackedState s;
#pragma unroll
    for (int i = 0; i < 8; i++) s.w[i] = __shfl_sync(FULL, x, i);
    return s;
}
__device__ __forceinline__ PackedState warp_load_state(const PackedState* p, int lane) {
    return warp_load_state_finish(warp_load_state_issue(p, lane));
}
__device__ __forceinline__ void warp_store_state(PackedState* p, const PackedState& s, int lane) {
    uint32_t x = s.w[0];
#pragma unroll
    for (int i = 1; i < 8; i++) x = (lane == i) ? s.w[i] : x;
    if (lane < 8) reinterpret_cast<uint32_t*>(p)[lane] = x;
}

// fused leaf gather: bf16 CHW (3,9,9) planes of `st` (cpp/uttt_game.cpp:244-280 after the NHWC->NCHW transpose of
// pv_mcts_cpp.py:60).  Lane 9*plane + R builds the 9-bit picture row R of plane (mover, opponent, legal); every
// element is then one shuffle + shift, and each store instruction of the warp writes 64 contiguous bytes.
__device__ __forceinline__ void warp_write_planes(__nv_bfloat16* pl, const PackedState& st, const uint32_t lm[3], int lane) {
    int plane = lane / 9, R = lane - 9 * plane;
    uint32_t x[3];
#pragma unroll
    for (int j = 0; j < 3; j++) x[j] = (plane == 0) ? st.w[j] : (plane == 1 ? st.w[3 + j] : lm[j]);
    uint32_t rows = (lane < 27) ? picture_row(x, R) : 0u;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        int e = lane + 32 * k;
        int row = e / 9, C = e - 9 * row;
        uint32_t m = __shfl_sync(FULL, rows, row & 31);
        if (e < 243) pl[e] = __ushort_as_bfloat16(((m >> C) & 1u) ? (unsigned short)0x3F80 : (unsigned short)0);
    }
}

// UTTT_SP_RANDOM_SYMMETRY: the symmetry under which evaluation j of the tree's current move is made (0, the identity,
// without the flag).  Search calls key it with seed 0, the root's index (c.game) and ply 0.
__device__ __forceinline__ int leaf_symmetry(const TreeParams& P, const TreeCtl& c, int j) {
    if (!(P.flags & UTTT_SP_RANDOM_SYMMETRY)) return 0;
    return sym_draw(P.mode == MODE_SELFPLAY ? P.seed : 0u, c.game, (uint32_t)c.ply, (uint32_t)j);
}

// evaluator row `row` for leaf `st` (legal mask lm) under symmetry g: the row's position and planes are those of g(st)
__device__ __forceinline__ void warp_write_row(const TreeParams& P, int row, const PackedState& st, const uint32_t lm[3], int g,
                                               int lane) {
    if (g == 0) {
        warp_store_state(P.nn_states + row, st, lane);
        warp_write_planes(P.nn_planes + (size_t)row * 243, st, lm, lane);
        return;
    }
    PackedState gs;
    sym_state(st, g, gs);
    uint32_t glm[3];
    legal_mask(gs, glm);
    warp_store_state(P.nn_states + row, gs, lane);
    warp_write_planes(P.nn_planes + (size_t)row * 243, gs, glm, lane);
}

// one coalesced read of a policy row for the leaf it was evaluated for under symmetry g: lane l gets the priors of actions
// l, l + 32, l + 64 (p2: lanes < 17), i.e. row entries sigma_g(a)
__device__ __forceinline__ void warp_load_priors(const float* pol, int g, int lane, float& p0, float& p1, float& p2) {
    int e0 = lane, e1 = 32 + lane, e2 = 64 + lane;
    if (g != 0) { e0 = sym_action(e0, g); e1 = sym_action(e1, g); e2 = (lane < 17) ? sym_action(e2, g) : 0; }
    p0 = __ldg(pol + e0);
    p1 = __ldg(pol + e1);
    p2 = (lane < 17) ? __ldg(pol + e2) : 0.0f;
}

// Philox temperature-1 sampling over the root visit counts; returns the chosen action.
// SP_TEMPERATURE != 1 (self_play_cpp.py:27,62 -> cpp/uttt_mcts.cpp:183-216): T == 0 plays the first maximum of the visit
// counts (the reference's one-hot scores leave np.random.choice no choice); otherwise the move is drawn from
// n_i^(1/T) / sum with the same Philox draw as the T == 1 sampler (fp32 weights, a fixed-order warp scan)
__device__ __forceinline__ int sample_move_temperature(const TreeParams& P, const TreeView& T, const TreeCtl& c, const uint32_t lm[3],
                                                       int lane) {
    const int L = c.n_root;
    if (P.temperature == 0.0f) {
        int best = -1, besti = 0x7FFFFFFF;
        for (int i = lane; i < L; i += 32) {
            int n = node_n(T.node[1 + i]);
            if (n > best) { best = n; besti = i; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            int ob = __shfl_xor_sync(FULL, best, off), oi = __shfl_xor_sync(FULL, besti, off);
            if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
        }
        return nth_legal(lm, besti);
    }
    const float inv = __fdiv_rn(1.0f, P.temperature);
    Philox4 r = philox4x32(P.seed, 1u, (uint32_t)c.game, (uint32_t)(c.game >> 32), (uint32_t)c.ply, 0u);
    const float u = (float)(r.x >> 8) * (1.0f / 16777216.0f);          // [0, 1)
    // pass 1: total weight (same scan as pass 2, so the threshold u * total is consistent with the prefix sums)
    float total = 0.0f;
    for (int pass = 0; pass < 2; pass++) {
        float carry = 0.0f;
        const float thr = __fmul_rn(u, total);
        for (int base = 0; base < L; base += 32) {
            const int i = base + lane;
            float incl = (i < L) ? powf((float)node_n(T.node[1 + i]), inv) : 0.0f;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                float o = __shfl_up_sync(FULL, incl, off);
                if (lane >= off) incl = __fadd_rn(incl, o);
            }
            incl = __fadd_rn(incl, carry);
            if (pass == 1) {
                unsigned hit = __ballot_sync(FULL, (i < L) && (incl > thr));
                if (hit) return nth_legal(lm, base + (__ffs((int)hit) - 1));
            }
            carry = __shfl_sync(FULL, incl, 31);
        }
        total = carry;
    }
    // rounding left u * total >= every prefix sum: the last visited child
    int last = 0;
    for (int i = lane; i < L; i += 32)
        if (node_n(T.node[1 + i]) > 0) last = i;
    last = __reduce_max_sync(FULL, last);
    return nth_legal(lm, last);
}

__device__ __forceinline__ int sample_move(const TreeParams& P, const TreeView& T, const TreeCtl& c, const uint32_t lm[3], int lane) {
    if (P.temperature != 1.0f) return sample_move_temperature(P, T, c, lm, lane);
    int L = c.n_root;
    int tot = 0;
    for (int i = lane; i < L; i += 32) tot += node_n(T.node[1 + i]);
    tot = __reduce_add_sync(FULL, tot);
    Philox4 r = philox4x32(P.seed, 1u, (uint32_t)c.game, (uint32_t)(c.game >> 32), (uint32_t)c.ply, 0u);
    uint32_t pick = __umulhi(r.x, (uint32_t)tot);
    int carry = 0, chosen = -1;
    for (int base = 0; base < L && chosen < 0; base += 32) {
        int i = base + lane;
        int v = (i < L) ? node_n(T.node[1 + i]) : 0;
        int incl = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            int o = __shfl_up_sync(FULL, incl, off);
            if (lane >= off) incl += o;
        }
        incl += carry;
        unsigned hit = __ballot_sync(FULL, (i < L) && ((uint32_t)incl > pick));
        if (hit) chosen = base + (__ffs((int)hit) - 1);
        carry = __shfl_sync(FULL, incl, 31);
    }
    if (chosen < 0) chosen = 0;
    return nth_legal(lm, chosen);
}


}  // namespace uttt
