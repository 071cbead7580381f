// tree_tp_kernels.cu -- "throughput" search: standard AlphaZero batched PUCT on the same SoA trees.
//
// Not in the reference (SURVEY.md N1): the reference has no virtual loss, no root noise and never evaluates
// the root.  This mode is what BASELINE.json's north_star asks for beyond the reference-exact mode:
//   * the root is evaluated by the network; Dirichlet(alpha) noise from the counter-based Philox stream
//     keyed by (seed, game, ply, child) -- (0, root index, 0, child) in a search call -- is mixed into its priors:
//     p = (1-eps) p + eps * eta (root_noise, tp_expand)
//   * up to m leaves per tree per round are collected with VIRTUAL LOSS (a per-node counter in the node word:
//     selection sees n+vl visits and w+vl lost value, so nothing has to be undone in floating point)
//   * every leaf is expanded once (no duplicated child lists), terminal values use the correct sign
//   * one warp still owns one tree, so there are no atomics on tree data and the result depends only on
//     (seed, m), never on scheduling.
// With m = 1 and eps = 0 it is plain sequential PUCT with an evaluated root (oracle/uttt_oracle.c: orc_az_search_hash);
// tests/tp_oracle.c restates the round for any m, with the noise taken from uttt_debug_root_noise.
// The round takes its descent, prior normalisation, leaf queue and move decision from tree_common.cuh, like the
// reference-exact round; its phases, expansion (tp_expand, with the root noise), backup (tp_backup, removing virtual
// loss) and round loop are its own.  tree_begin_kernel (tree_kernels.cu) starts its trees in PHASE_ROOT.
#include "tree_common.cuh"

namespace uttt {

// uniform in (0,1) from 24 random bits
__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// Gamma(alpha,1) sample, Marsaglia-Tsang with the alpha<1 boost; stream = Philox(seed,3 ; game, ply, child, attempt)
__device__ float gamma_sample(float alpha, uint32_t seed, uint64_t game, uint32_t ply, uint32_t child) {
    float a = alpha < 1.0f ? alpha + 1.0f : alpha;
    float d = a - 1.0f / 3.0f, c = rsqrtf(9.0f * d);
    float g = d;
    for (uint32_t attempt = 0; attempt < 64; attempt++) {
        Philox4 r = philox4x32(seed, 3u, (uint32_t)game, (uint32_t)(game >> 32) ^ (ply << 16), child, attempt);
        float u1 = u01(r.x), u2 = u01(r.y), u3 = u01(r.z);
        float x = sqrtf(-2.0f * logf(u1)) * cosf(6.283185307f * u2);       // Box-Muller
        float v = 1.0f + c * x;
        if (v <= 0.0f) continue;
        v = v * v * v;
        if (logf(u3) < 0.5f * x * x + d - d * v + d * logf(v)) { g = d * v; break; }
    }
    if (alpha < 1.0f) {
        Philox4 r = philox4x32(seed, 3u, (uint32_t)game, (uint32_t)(game >> 32) ^ (ply << 16), child, 0xFFFFu);
        g *= powf(u01(r.w), 1.0f / alpha);
    }
    return g;
}

// The root noise eta of a position with legal mask lm (L legal actions) under key (seed, game, ply): a Gamma(alpha) sample
// g_a = gamma_sample(alpha, seed, game, ply, a) for every legal action id a, their sum taken per lane (actions lane,
// lane + 32, lane + 64 in that order) and then by a shuffle-xor butterfly (offsets 16, 8, 4, 2, 1), and eta_a = g_a / sum,
// or 1 / L if the sum is not positive.  eta[q] is that of action lane + 32 q (0 where it is not legal).  tp_expand mixes it
// into an evaluated root; uttt_debug_root_noise and uttt_debug_dirichlet export it, so that a CPU check can take the
// draw from the device (it cannot restate logf / cosf / powf / rsqrtf bit for bit).
__device__ void root_noise(float alpha, uint32_t seed, uint64_t game, uint32_t ply, const uint32_t lm[3], int L, int lane,
                           float eta[3]) {
    float gsum = 0.0f, g[3] = {0.f, 0.f, 0.f};
    for (int q = 0, a = lane; a < 81; a += 32, q++)
        if (legal_bit(lm, a)) { g[q] = gamma_sample(alpha, seed, game, ply, (uint32_t)a); gsum += g[q]; }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) gsum += __shfl_xor_sync(FULL, gsum, off);
    const float uni = (L > 0) ? __fdiv_rn(1.0f, (float)L) : 0.0f;
#pragma unroll
    for (int q = 0; q < 3; q++) {
        const int a = lane + 32 * q;
        eta[q] = (a < 81 && legal_bit(lm, a)) ? (gsum > 0.0f ? __fdiv_rn(g[q], gsum) : uni) : 0.0f;
    }
}

// diagnostics (uttt_debug_dirichlet): out[g][a] = eta_a of root_noise for game game0 + g at ply 0 of a root whose legal
// actions are 0 .. n_children - 1 (a game's first root has all 81; tp_expand keys its draw by action id, so a root with
// other legal actions gets other draws -- uttt_debug_root_noise gives those)
__global__ void __launch_bounds__(128) dirichlet_kernel(uint32_t seed, uint64_t game0, int64_t n, int n_children, float alpha,
                                                        float* __restrict__ out) {
    const int64_t g = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= n) return;
    uint32_t lm[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int k = n_children - 27 * j;
        lm[j] = k >= 27 ? 0x7FFFFFFu : (k > 0 ? (1u << k) - 1u : 0u);
    }
    float eta[3];
    root_noise(alpha, seed, game0 + (uint64_t)g, 0u, lm, n_children, lane, eta);
    for (int q = 0, a = lane; a < n_children; a += 32, q++) out[g * n_children + a] = eta[q];
}
cudaError_t launch_dirichlet(uint32_t seed, uint64_t game0, int64_t n, int n_children, float alpha, float* out, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    dirichlet_kernel<<<(unsigned)((n + 3) / 4), 128, 0, s>>>(seed, game0, n, n_children, alpha, out);
    return cudaGetLastError();
}

// diagnostics (uttt_debug_root_noise): eta[i][a] = root_noise of position states[i] under key (seed, games[i], plies[i]),
// 0 for an illegal action
__global__ void __launch_bounds__(128) root_noise_kernel(uint32_t seed, float alpha, const PackedState* __restrict__ states,
                                                         const uint64_t* __restrict__ games, const int32_t* __restrict__ plies,
                                                         int64_t n, float* __restrict__ eta_out) {
    const int64_t i = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    const PackedState st = warp_load_state(states + i, lane);
    uint32_t lm[3];
    const int L = legal_mask(st, lm);
    float eta[3];
    root_noise(alpha, seed, games[i], (uint32_t)plies[i], lm, L, lane, eta);
    for (int q = 0, a = lane; a < 81; a += 32, q++) eta_out[i * 81 + a] = eta[q];
}
cudaError_t launch_root_noise(uint32_t seed, float alpha, const PackedState* states, const uint64_t* games, const int32_t* plies,
                              int64_t n, float* eta_out, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    root_noise_kernel<<<(unsigned)((n + 3) / 4), 128, 0, s>>>(seed, alpha, states, games, plies, n, eta_out);
    return cudaGetLastError();
}

struct TpAux {                 // per tree, per pending leaf
    int32_t path_len[TP_MAX_LEAVES];
    int32_t nn_row[TP_MAX_LEAVES];
};

// expansion of `leaf` from one policy row, evaluated under symmetry `sym`: masked, serially renormalised priors (the
// reference-exact mode's arithmetic), and for the root of a full search with eps > 0 the root noise mixed in as
// p = fma(1 - eps, p, eps * eta): eps * eta rounded, then one fused multiply-add (the form nvcc gave the plain expression).  The noise is keyed by
// (seed, game, ply) in self-play and by (0, root index, 0) in a search call, like leaf_symmetry.
__device__ void tp_expand(const TreeParams& P, const TreeView& T, TreeCtl& c, const PackedState& st, int leaf,
                          const float* pol, int sym, bool is_root, int lane) {
    uint32_t lm[3];
    int L = legal_mask(st, lm);
    int base = c.n_nodes;
    float pr[3];
    legal_priors(pol, sym, lm, L, lane, pr);
    const bool noise = is_root && P.dir_eps > 0.0f && full_search(P, c);      // a fast search gets none (KataGo)
    float eta[3] = {0.f, 0.f, 0.f};
    if (noise) root_noise(P.dir_alpha, P.mode == MODE_SELFPLAY ? P.seed : 0u, c.game, (uint32_t)c.ply, lm, L, lane, eta);
    const float keep = 1.0f - P.dir_eps;
#pragma unroll
    for (int q = 0; q < 3; q++) {
        const int a = lane + 32 * q;
        if (a < 81 && legal_bit(lm, a)) {
            float p = pr[q];
            if (noise) p = __fmaf_rn(keep, p, __fmul_rn(P.dir_eps, eta[q]));
            T.node[base + legal_rank(lm, a)] = make_node(a, p);
        }
    }
    if (lane == 0) T.node[leaf].w = (uint32_t)base | ((uint32_t)L << 20);
    c.n_nodes = base + L;
}

// value backup along a recorded path; removes one unit of virtual loss from every node of the path
__device__ void tp_backup(const TreeView& T, const int32_t* path, int plen, float v, bool had_vloss, int lane) {
    __syncwarp();
    for (int i = lane; i < plen; i += 32) {
        int node = path[i];
        bool flip = ((plen - 1 - i) & 1) != 0;
        uint2* nw = reinterpret_cast<uint2*>(T.node + node);
        uint2 q = *nw;
        q.y = __float_as_uint(__fadd_rn(__uint_as_float(q.y), flip ? -v : v));
        q.x += 1u;                                   // n += 1
        if (had_vloss) q.x -= (1u << 23);            // vl -= 1
        *nw = q;
    }
    __syncwarp();
}

// 5 blocks per SM (at most 102 registers): left to itself ptxas gives the inlined descent more registers, and fewer trees
// would be resident
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK, 5) tree_tp_round_kernel(TreeParams P) {
    int t = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) { P.nn_count[P.parity ^ 1] = 0; P.nn1_count[P.parity ^ 1] = 0; }
    if (t >= P.n_trees) return;
    TreeCtl c = P.ctl[t];
    if (c.phase == PHASE_DONE) return;
    TreeView T = view_of(P, t);
    TpAux* aux = reinterpret_cast<TpAux*>(P.tp_aux) + t;
    PackedState root = warp_load_state(P.root + t, lane);
    const int m = P.batch < TP_MAX_LEAVES ? P.batch : TP_MAX_LEAVES;

    // ---------------- apply what the evaluator returned for this tree
    if (c.phase == PHASE_ROOT_PENDING) {
        if (lane == 0) T.node[0] = make_uint4(0x7Fu << 16, 0u, 0u, 0u);
        __syncwarp();
        c.n_nodes = 1;
        tp_expand(P, T, c, root, 0, net_policy(P, leaf_net(P, c)) + (size_t)c.nn_row * 81, leaf_symmetry(P, c, 0), true, lane);
        uint32_t lm[3];
        c.n_root = legal_mask(root, lm);
        c.sims_left = move_sims(P, c);
        c.phase = PHASE_SEARCH;
        __syncwarp();
    } else if (c.phase == PHASE_PENDING) {
        for (int j = 0; j < c.pend_k; j++) {
            int plen = aux->path_len[j], row = aux->nn_row[j];
            const int32_t* path = leaf_path(P, t, j);
            int leaf = path[plen - 1];
            PackedState st = warp_load_state(leaf_state(P, t, j), lane);
            if (c.n_nodes + 81 > P.node_cap) {
                if (lane == 0) atomicExch(P.counters + 5, 1ull);
                c.phase = PHASE_DONE;
                if (lane == 0) P.ctl[t] = c;
                return;
            }
            tp_expand(P, T, c, st, leaf, net_policy(P, leaf_net(P, c)) + (size_t)row * 81, leaf_symmetry(P, c, c.n_eval - c.pend_k + j), false,
                      lane);
            tp_backup(T, path, plen, net_value(P, leaf_net(P, c))[row], true, lane);
        }
        c.sims_left -= c.pend_k;
        if (lane == 0) atomicAdd(P.counters + 3, (unsigned long long)c.pend_k);
        c.pend_k = 0;
        c.phase = PHASE_SEARCH;
    }

    // UTTT_SP_FORCED_PLAYOUTS' k for this round's descents and its move decision, which all belong to the move at c.ply
    // (a decided move ends the round's search: the next move starts by queueing its root)
    const float forced_k = ((P.flags & UTTT_SP_FORCED_PLAYOUTS) && full_search(P, c)) ? P.forced_k : 0.0f;
    for (int guard = 0; guard < 4; guard++) {
        if (c.phase == PHASE_SEARCH && c.sims_left <= 0) {
            if (!decide_move(P, T, t, c, root, forced_k, lane)) break;
            c.phase = PHASE_ROOT;
        }
        if (c.phase == PHASE_ROOT) {
            uint32_t lm[3];
            int L = legal_mask(root, lm);
            if (L == 0) {                                   // search mode on a finished position: empty result
                if (lane == 0) { P.out_n[t] = 0; atomicAdd(P.counters + 6, 1ull); }
                c.phase = PHASE_DONE;
                break;
            }
            c.n_eval = 0;                                   // the root is evaluation 0 of the move's search
            c.nn_row = queue_leaf(P, t, c, root, lm, 1, lane);
            c.phase = PHASE_ROOT_PENDING;
            break;
        }

        // ---------------- collect up to m leaves with virtual loss
        int want = c.sims_left < m ? c.sims_left : m;
        int got = 0, terminals = 0;
        while (got < want && got + terminals < c.sims_left && terminals < 2 * m) {
            int32_t* path = leaf_path(P, t, got);
            const Descent d = descend(T, root, path, forced_k, lane);
            if (d.end == LEAF_BLOCKED) break;       // the best line ends in a leaf already queued this round
            if (d.end != LEAF_UNEXPANDED) {
                // value for the mover of the terminal node: -1 lost, 0 draw (correct sign, unlike cpp/uttt_mcts.cpp:19-21)
                tp_backup(T, path, d.plen, d.end == LEAF_LOST ? -1.0f : 0.0f, false, lane);
                terminals++;
                continue;
            }
            // unexpanded leaf: mark it, add virtual loss along the path, queue it
            __syncwarp();
            for (int i = lane; i < d.plen; i += 32) T.node[path[i]].x += (1u << 23);
            if (lane == 0) T.node[d.node].w = LINK_PENDING;
            __syncwarp();
            int row = queue_leaf(P, t, c, d.st, d.lm, 1, lane);
            warp_store_state(leaf_state(P, t, got), d.st, lane);
            if (lane == 0) { aux->path_len[got] = d.plen; aux->nn_row[got] = row; }
            got++;
        }
        if (terminals) {
            c.sims_left -= terminals;
            if (lane == 0) atomicAdd(P.counters + 3, (unsigned long long)terminals);
        }
        if (got > 0) {
            c.pend_k = got;
            c.phase = PHASE_PENDING;
            break;
        }
        if (c.sims_left > 0) break;             // only terminals this round (bounded work): continue next round
    }
    if (lane == 0) P.ctl[t] = c;
}

cudaError_t launch_tree_tp_round(const TreeParams& p, cudaStream_t s) {
    tree_tp_round_kernel<<<ceil_div(p.n_trees, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, s>>>(p);
    return cudaGetLastError();
}

}  // namespace uttt
