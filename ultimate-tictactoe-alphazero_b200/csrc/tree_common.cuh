// tree_common.cuh -- the warp pieces both search kernels are built from, the reference-exact (tree_kernels.cu) and the
// throughput (tree_tp_kernels.cu) round: node word accessors, warp-wide state load/store, the evaluator row, the prior
// normalisation, the PUCT descent, the leaf queue and the move decision with its Philox sampling.  None of them
// depends on which kernel calls it; each kernel keeps its own schedule (phases, apply step, backup, round loop).
#pragma once
#include "common.cuh"

namespace uttt {

constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int WARPS_PER_BLOCK = 4;
constexpr uint32_t LINK_PENDING = 0xFFFFFu;      // first_child marker: leaf queued, expansion outstanding (throughput mode)

struct TreeView {
    uint4* node;     // [node_cap]
};

__device__ __forceinline__ TreeView view_of(const TreeParams& P, int t) {
    TreeView v = {P.nodes + (size_t)t * (size_t)P.node_cap};
    return v;
}

// the recorded path of pending leaf j of tree t (the reference-exact mode has one pending leaf, j = 0)
__device__ __forceinline__ int32_t* leaf_path(const TreeParams& P, int t, int j) {
    return P.paths + ((size_t)t * TP_MAX_LEAVES + j) * PATH_CAP;
}
__device__ __forceinline__ PackedState* leaf_state(const TreeParams& P, int t, int j) {
    return P.leaf_state + (size_t)t * TP_MAX_LEAVES + j;
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

// UTTT_SP_MATCH: the network that evaluates the leaves of the tree's current move -- weight slot (game + ply) & 1, so slot 0
// moves first in even games and slot 1 in odd ones; 0 without the flag.  The ply does not change between queueing a leaf
// and applying its row, so the apply step finds the row in the queue it was written to.
__device__ __forceinline__ int leaf_net(const TreeParams& P, const TreeCtl& c) {
    return (P.flags & UTTT_SP_MATCH) ? (int)(((uint32_t)c.game + (uint32_t)c.ply) & 1u) : 0;
}
// the evaluator rows of that network
__device__ __forceinline__ const float* net_policy(const TreeParams& P, int net) { return net ? P.policy1 : P.policy; }
__device__ __forceinline__ const float* net_value(const TreeParams& P, int net) { return net ? P.value1 : P.value; }

// evaluator row `row` of network `net`'s queue for leaf `st` (legal mask lm) under symmetry g: the row's position and planes
// are those of g(st)
__device__ __forceinline__ void warp_write_row(const TreeParams& P, int net, int row, const PackedState& st, const uint32_t lm[3],
                                               int g, int lane) {
    PackedState* states = (net ? P.nn1_states : P.nn_states) + row;
    __nv_bfloat16* planes = (net ? P.nn1_planes : P.nn_planes) + (size_t)row * 243;
    if (g == 0) {
        warp_store_state(states, st, lane);
        warp_write_planes(planes, st, lm, lane);
        return;
    }
    PackedState gs;
    sym_state(st, g, gs);
    uint32_t glm[3];
    legal_mask(gs, glm);
    warp_store_state(states, gs, lane);
    warp_write_planes(planes, gs, glm, lane);
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

// priors of a leaf with legal mask lm (L legal actions) from its policy row: policy[legal] / sum in fp32, the sum taken
// serially over the legal actions in ascending id (cpp/uttt_mcts.cpp:144-163), uniform if it is not positive.  One
// coalesced read of the row, then one shuffle per addend (`a` is warp-uniform).  pr[q] is the prior of action
// lane + 32 q (meaningful where that action is legal).
__device__ __forceinline__ void legal_priors(const float* pol, int g, const uint32_t lm[3], int L, int lane, float pr[3]) {
    float p0, p1, p2;
    warp_load_priors(pol, g, lane, p0, p1, p2);
    float sum = 0.0f;
#pragma unroll
    for (int j = 0; j < 3; j++) {
        uint32_t m = lm[j];
        while (m) {
            int a = 27 * j + __ffs((int)m) - 1;
            m &= m - 1u;
            const float src = a < 32 ? p0 : (a < 64 ? p1 : p2);
            sum = __fadd_rn(sum, __shfl_sync(FULL, src, a & 31));
        }
    }
    const float uni = (L > 0) ? __fdiv_rn(1.0f, (float)L) : 0.0f;
    pr[0] = (sum > 0.0f) ? __fdiv_rn(p0, sum) : uni;
    pr[1] = (sum > 0.0f) ? __fdiv_rn(p1, sum) : uni;
    pr[2] = (sum > 0.0f) ? __fdiv_rn(p2, sum) : uni;
}

// queues leaf `st` (legal mask lm) for the evaluator as evaluation c.n_eval of the tree's current move, standing for k
// simulations, in the queue of the network to move (leaf_net); returns its row there
__device__ __forceinline__ int queue_leaf(const TreeParams& P, int t, TreeCtl& c, const PackedState& st, const uint32_t lm[3],
                                          int k, int lane) {
    const int net = leaf_net(P, c);
    int row = 0;
    if (lane == 0) {
        row = atomicAdd((net ? P.nn1_count : P.nn_count) + P.parity, 1);
        atomicAdd(P.counters + 4, 1ull);
        (net ? P.nn1_tree : P.nn_tree)[row] = t;
        (net ? P.nn1_k : P.nn_k)[row] = k;
    }
    row = __shfl_sync(FULL, row, 0);
    warp_write_row(P, net, row, st, lm, leaf_symmetry(P, c, c.n_eval), lane);
    c.n_eval += 1;
    return row;
}

enum : int { LEAF_UNEXPANDED = 0, LEAF_LOST = 1, LEAF_DRAWN = 2, LEAF_BLOCKED = 3 };

struct Descent {
    PackedState st;      // the position the descent ended on
    uint32_t lm[3];      // its legal mask
    int node, plen;      // its node, and the length of the path root..node
    int end;             // LEAF_UNEXPANDED, LEAF_LOST / LEAF_DRAWN (terminal), LEAF_BLOCKED (a child already queued)
};

// descend from the root by PUCT (cpp/uttt_mcts.cpp:15-32,57-81), recording the node path into `path`.  Children are
// read once (one 128-bit load each); lanes keep their first three in registers, longer lists (the reference-exact mode's
// k-fold duplicated lists, Q-M3) are re-read through L1.  A child with vl units of virtual loss counts as n + vl
// visits and w + vl lost value (the reference-exact mode sets none).
__device__ __forceinline__ Descent descend(const TreeView& T, const PackedState& root, int32_t* path, int lane) {
    Descent d;
    d.st = root;
    d.node = 0;
    d.plen = 1;
    d.end = LEAF_UNEXPANDED;
    if (lane == 0) path[0] = 0;
    uint32_t link = T.node[0].w;               // first_child | n_children<<20 of the current node
    for (;;) {
        const int L = legal_mask(d.st, d.lm);
        if (is_lose(d.st)) { d.end = LEAF_LOST; break; }
        if (L == 0) { d.end = LEAF_DRAWN; break; }
        const uint32_t cbase = link & 0xFFFFFu;
        if (cbase == 0u) break;
        if (cbase == LINK_PENDING) { d.end = LEAF_BLOCKED; break; }
        const int cnt = (int)(link >> 20);
        const uint4* ch = T.node + cbase;
        uint4 c0 = make_uint4(0, 0, 0, 0), c1 = c0, c2 = c0;
        int tot = 0;
        if (lane < cnt) { c0 = ch[lane]; tot += node_n(c0) + node_vloss(c0); }
        if (lane + 32 < cnt) { c1 = ch[lane + 32]; tot += node_n(c1) + node_vloss(c1); }
        if (lane + 64 < cnt) { c2 = ch[lane + 64]; tot += node_n(c2) + node_vloss(c2); }
        for (int i = lane + 96; i < cnt; i += 32) { const uint4 q = ch[i]; tot += node_n(q) + node_vloss(q); }
        tot = __reduce_add_sync(FULL, tot);
        const float sq = __fsqrt_rn((float)tot);
        float best = -1e9f;
        int besti = 0x7FFFFFFF;
        uint32_t bestx = 0u, bestlink = 0u;
        auto consider = [&](const uint4& q, int i) {
            const int vl = node_vloss(q), n = node_n(q) + vl;
            // unvisited child (most of a k-fold duplicated list): q = 0 and u = (p*sq)/1, so pucb = p*sq exactly --
            // the two IEEE divisions are only executed for visited children
            float s = __fmul_rn(__uint_as_float(q.z), sq);
            if (n > 0) {
                const float qv = __fdiv_rn(-__fadd_rn(__uint_as_float(q.y), (float)vl), (float)n);
                s = __fadd_rn(qv, __fdiv_rn(s, (float)(1 + n)));
            }
            if (s > best) { best = s; besti = i; bestx = q.x; bestlink = q.w; }
        };
        if (lane < cnt) consider(c0, lane);
        if (lane + 32 < cnt) consider(c1, lane + 32);
        if (lane + 64 < cnt) consider(c2, lane + 64);
        for (int i = lane + 96; i < cnt; i += 32) consider(ch[i], i);
        // first maximum wins (Q-M6): the largest score by one warp reduction on an order-preserving integer image of
        // the float (scores are never -0.0 or NaN: q + u with u >= +0), then the smallest child index among the lanes
        // that hold it, then that lane's node word -- 2 reductions + 2 shuffles instead of a 20-shuffle butterfly
        {
            const uint32_t fb = __float_as_uint(best);
            const uint32_t key = (fb & 0x80000000u) ? ~fb : (fb | 0x80000000u);
            const uint32_t kmax = __reduce_max_sync(FULL, key);
            besti = (int)__reduce_min_sync(FULL, key == kmax ? (uint32_t)besti : 0x7FFFFFFFu);
            const int src = besti & 31;                          // child i is held by lane i % 32
            // (a lane's own candidate is its FIRST maximum, so the winning lane's registers hold child besti)
            bestx = __shfl_sync(FULL, bestx, src);
            bestlink = __shfl_sync(FULL, bestlink, src);
        }
        d.node = (int)cbase + besti;
        link = bestlink;
        PackedState nx;
        next_state(d.st, (int)((bestx >> 16) & 0x7Fu), nx);
        d.st = nx;
        if (lane == 0) path[d.plen] = d.node;
        d.plen++;
    }
    return d;
}

// the legal-order index of the root child with the most visits, the first maximum (the same on every lane)
__device__ __forceinline__ int most_visited(const TreeView& T, int L, int lane) {
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
    return besti;
}

// The mover's value of the searched position: Q = -w / n of the most visited root child (the child sample_move plays
// at T = 0), exactly as descend computes it without virtual loss, and 0 for an unvisited child (descend's Q).  No
// virtual loss is outstanding when a move is decided: the reference-exact mode sets none, and the throughput round
// decides only in PHASE_SEARCH, which it enters after the tp_backup of every leaf it queued has removed that leaf's unit
// (terminal descents add none).
__device__ __forceinline__ float root_value(const TreeView& T, const TreeCtl& c, int lane) {
    const uint4 q = T.node[1 + most_visited(T, c.n_root, lane)];
    const int n = node_n(q);
    return n > 0 ? __fdiv_rn(-__uint_as_float(q.y), (float)n) : 0.0f;
}

// UTTT_SP_RESIGN: game g is a check game, never resigned, iff u < check fraction, u = (philox(key=(seed, 4),
// ctr=(g_lo, g_hi, 0, 0)).x >> 8) * 2^-24
__device__ __forceinline__ bool check_game(const TreeParams& P, uint64_t game) {
    const Philox4 r = philox4x32(P.seed, 4u, (uint32_t)game, (uint32_t)(game >> 32), 0u, 0u);
    return (float)(r.x >> 8) * (1.0f / 16777216.0f) < P.resign_check_fraction;
}

// Philox temperature-1 sampling over the root visit counts; returns the chosen action.
// SP_TEMPERATURE != 1 (self_play_cpp.py:27,62 -> cpp/uttt_mcts.cpp:183-216): T == 0 plays the first maximum of the visit
// counts (the reference's one-hot scores leave np.random.choice no choice); otherwise the move is drawn from
// n_i^(1/T) / sum with the same Philox draw as the T == 1 sampler (fp32 weights, a fixed-order warp scan)
__device__ __forceinline__ int sample_move_temperature(const TreeParams& P, const TreeView& T, const TreeCtl& c, const uint32_t lm[3],
                                                       int lane) {
    const int L = c.n_root;
    if (P.temperature == 0.0f) return nth_legal(lm, most_visited(T, L, lane));
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

// the move is decided (the simulation budget is spent).  Search: the root visit counts are the tree's output
// (cpp/uttt_mcts.cpp:177-180) and the tree is done.  Self-play: record the root value and the history row, sample the
// move, play it; when the game is over (lost or drawn, self_play_cpp.py:50-51,95) record it and claim the next game from
// counters[0].  With UTTT_SP_RESIGN, a mover at ply p >= 1 of a game that is not a check game resigns instead when its
// root value is below the threshold: only the value of ply p is recorded, and the game ends with p plies as one whose
// final position is lost for its mover.  Returns whether the tree goes on; if so `root` is the position of its next
// search, already stored in P.root[t].
__device__ __forceinline__ bool decide_move(const TreeParams& P, const TreeView& T, int t, TreeCtl& c, PackedState& root, int lane) {
    if (P.mode == MODE_SEARCH) {
        for (int i = lane; i < 81; i += 32) P.out_counts[(size_t)t * 81 + i] = (i < c.n_root) ? node_n(T.node[1 + i]) : 0;
        if (lane == 0) { P.out_n[t] = c.n_root; atomicAdd(P.counters + 6, 1ull); }
        c.phase = PHASE_DONE;
        return false;
    }
    uint32_t lm[3];
    legal_mask(root, lm);
    const size_t hrow = (size_t)c.game_idx * 81 + (size_t)c.ply;
    const float v = root_value(T, c, lane);
    if (lane == 0) P.hist_value[hrow] = v;
    const bool resign = (P.flags & UTTT_SP_RESIGN) && c.ply >= 1 && v < P.resign_threshold && !check_game(P, c.game);
    bool over = resign;
    if (!resign) {
        warp_store_state(P.hist_states + hrow, root, lane);
        for (int a = lane; a < 81; a += 32)
            P.hist_counts[hrow * 81 + a] = legal_bit(lm, a) ? (uint16_t)node_n(T.node[1 + legal_rank(lm, a)]) : (uint16_t)0;
        const int action = sample_move(P, T, c, lm, lane);
        if (lane == 0) P.hist_actions[hrow] = (uint8_t)action;
        PackedState nx;
        next_state(root, action, nx);
        root = nx;
        c.ply += 1;
        over = legal_mask(root, lm) == 0;
    }
    if (over) {
        if (lane == 0) {
            P.hist_len[c.game_idx] = c.ply;
            P.hist_final[c.game_idx] = (resign || is_lose(root)) ? 1 : 0;
            if (resign) P.hist_resigned[c.game_idx] = 1;
            atomicAdd(P.counters + 1, 1ull);
            atomicAdd(P.counters + 2, (unsigned long long)c.ply);
        }
        unsigned long long g = 0;
        if (lane == 0) g = atomicAdd(P.counters + 0, 1ull);
        g = __shfl_sync(FULL, g, 0);
        if ((int64_t)g >= P.n_games) { c.phase = PHASE_DONE; return false; }
        c.game = P.game0 + g;
        c.game_idx = (int32_t)g;
        c.ply = 0;
        init_state(root);
    }
    warp_store_state(P.root + t, root, lane);
    return true;
}


}  // namespace uttt
