// tree_kernels.cu -- PUCT search over structure-of-arrays trees resident in HBM.
//
// Replaces UTTT::Node / UTTT::pv_mcts_scores (cpp/uttt_mcts.cpp:10-196).  One warp owns one
// tree (atomics-free per-tree ownership); thousands of trees advance in lock-step "rounds":
//
//   tree_round:  [apply]   if the tree has an evaluated leaf waiting: masked + serially
//                          renormalised priors (:144-163), expansion (:35-44), k sequential
//                          backups (:47-54)
//                [select]  descend by PUCT (:57-81) with a warp-level first-max argmax until an
//                          unexpanded leaf (queue it for the evaluator, fused leaf gather) or a
//                          terminal node (back up immediately, :115-118, and descend again)
//                [move]    when the simulation budget is spent: root visit counts -> search
//                          output, or (self-play) temperature-1 sampling with Philox into the
//                          history buffers, advance the game, recycle the slot
//
// Reference-exact ("compat") semantics.  The reference queues the SAME leaf k = min(batch_size,
// sims_left) times between flushes because it has no virtual loss (SURVEY.md Q-M3/Q-M4); the
// loop is therefore equivalent to: evaluate the leaf once, append k copies of its child list,
// back the value up k times sequentially.  That equivalent form is what runs here, and
// oracle/uttt_oracle.c (which restates the literal queue/flush loop) checks it bit for bit.
// A node is ONE 16-byte word {n:16 | action:7, w (f32), p (f32), first_child:20 | n_children:12}: positions are
// recomputed by next_state() during the descent (the reference stores ~760 B per node), and a PUCT step
// is a single coalesced 128-bit load per child -- the chosen child's own word already carries where its
// children are, so the descent pays one L2 round trip per level.
//
// All float arithmetic on n/w/p uses explicit round-to-nearest intrinsics in the reference's
// operation order (no FMA contraction, no reassociation): cpp/setup.py:10 builds with -O3 only.
//
// The round is built from the warp pieces of tree_common.cuh (prior normalisation, descent, leaf queue, move decision),
// which the throughput round (tree_tp_kernels.cu) shares; its apply step, backup and round loop are its own.  This file
// also holds the begin kernel of both modes, the device hash evaluator and the scores / boltzman kernels.
#include "tree_common.cuh"

namespace uttt {

// cpp/uttt_mcts.cpp:92-103: root expanded up-front with the uniform prior 1/L (never evaluated, Q-M1)
__device__ void init_root(const TreeParams& P, const TreeView& T, TreeCtl& c, const PackedState& rs, int lane) {
    uint32_t lm[3];
    int L = legal_mask(rs, lm);
    if (P.flags & UTTT_SP_PYSEARCH) {
        // pv_mcts.py:133: the root starts as an unexpanded leaf; the first simulations queue the root itself
        if (lane == 0) T.node[0] = make_uint4(0x7Fu << 16, 0u, 0u, 0u);
        c.n_nodes = 1;
        c.n_root = L;
        c.sims_left = move_sims(P, c);
        c.path_len = 0;
        c.pend_k = 0;
        c.n_eval = 0;
        return;
    }
    float pu = (L > 0) ? __fdiv_rn(1.0f, (float)L) : 0.0f;
    if (lane == 0) T.node[0] = make_uint4(0x7Fu << 16, 0u, 0u, (L > 0 ? 1u : 0u) | ((uint32_t)L << 20));
    for (int a = lane; a < 81; a += 32)
        if (legal_bit(lm, a)) T.node[1 + legal_rank(lm, a)] = make_node(a, pu);
    c.n_nodes = 1 + L;
    c.n_root = L;
    c.sims_left = move_sims(P, c);
    c.path_len = 0;
    c.pend_k = 0;
    c.n_eval = 0;
}

// cpp/uttt_mcts.cpp:47-54, k sequential backups of the same path (values may differ per copy)
__device__ void backup(const TreeView& T, const int32_t* path, int plen, int k, const float* vals, int vstride, float v_single,
                       int lane) {
    __syncwarp();
    for (int i = lane; i < plen; i += 32) {
        int node = path[i];
        bool flip = ((plen - 1 - i) & 1) != 0;
        uint2* nw = reinterpret_cast<uint2*>(T.node + node);     // {n|action, w}
        uint2 q = *nw;
        float w = __uint_as_float(q.y);
        if (vals && vstride != 0) {
            for (int c = 0; c < k; c++) {
                float v = vals[(size_t)c * vstride];
                w = __fadd_rn(w, flip ? -v : v);
            }
        } else {
            // k identical values: still k sequential fp32 adds (w += v k times != w += k*v), but one load
            float v = vals ? vals[0] : v_single;
            v = flip ? -v : v;
            for (int c = 0; c < k; c++) w = __fadd_rn(w, v);
        }
        q.y = __float_as_uint(w);
        q.x += (uint32_t)k;                                       // n lives in the low 16 bits
        *nw = q;
    }
    __syncwarp();
}

// pv_mcts.py:46-48: np.sum over the float32 legal policies = numpy's pairwise summation, which for fewer than 128
// addends is: 8 running sums over the leading multiple of 8 (element i goes to sum i % 8), combined as
// ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the remaining addends one by one; fewer than 8 addends: serially from 0.
// lp0/lp1/lp2 hold the legal policies in legal order (rank lane, lane + 32, lane + 64).
__device__ float numpy_sum_f32(float lp0, float lp1, float lp2, int L, int lane) {
    auto at = [&](int i) {                                            // warp-uniform i
        const float src = i < 32 ? lp0 : (i < 64 ? lp1 : lp2);
        return __shfl_sync(FULL, src, i & 31);
    };
    if (L < 8) {
        float res = 0.0f;
        for (int i = 0; i < L; i++) res = __fadd_rn(res, at(i));
        return res;
    }
    const int nfull = L - (L % 8);
    float r = __shfl_sync(FULL, lp0, lane & 7);                        // lanes 0..7: the 8 running sums
    for (int b = 8; b < nfull; b += 8) {
        const float src = b < 32 ? lp0 : (b < 64 ? lp1 : lp2);         // (b + j) >> 5 == b >> 5 for j < 8
        r = __fadd_rn(r, __shfl_sync(FULL, src, (b + (lane & 7)) & 31));
    }
    float r0 = __shfl_sync(FULL, r, 0), r1 = __shfl_sync(FULL, r, 1), r2 = __shfl_sync(FULL, r, 2), r3 = __shfl_sync(FULL, r, 3);
    float r4 = __shfl_sync(FULL, r, 4), r5 = __shfl_sync(FULL, r, 5), r6 = __shfl_sync(FULL, r, 6), r7 = __shfl_sync(FULL, r, 7);
    float res = __fadd_rn(__fadd_rn(__fadd_rn(r0, r1), __fadd_rn(r2, r3)), __fadd_rn(__fadd_rn(r4, r5), __fadd_rn(r6, r7)));
    for (int i = nfull; i < L; i++) res = __fadd_rn(res, at(i));
    return res;
}

// pv_mcts.py:105-109,157-160 for the k queued copies of one leaf: every copy REPLACES the child list (one list survives),
// priors = policy[legal] / np.sum(policy[legal]) in float32 (pv_mcts.py:45-49), k sequential backups
__device__ void apply_leaf_py(const TreeParams& P, const TreeView& T, TreeCtl& c, const PackedState& st, const int32_t* path,
                              int lane) {
    uint32_t lm[3];
    int L = legal_mask(st, lm);
    int k = c.pend_k, plen = c.path_len;
    int leaf = path[plen - 1];
    int base = c.n_nodes;
    if (base + L > P.node_cap) {
        if (lane == 0) atomicExch(P.counters + 5, 1ull);
        c.phase = PHASE_DONE;
        return;
    }
    size_t row = (size_t)c.nn_row * (size_t)P.row_stride;
    float p0, p1, p2;
    warp_load_priors(net_policy(P, leaf_net(P, c)) + row * 81, leaf_symmetry(P, c, c.n_eval - 1), lane, p0, p1, p2);
    // legal policies in legal order: rank i sits in lane i % 32, register i / 32
    float lp[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int i = lane + 32 * j;
        const int a = (i < L) ? nth_legal(lm, i) : 0;
        const float v0 = __shfl_sync(FULL, p0, a & 31), v1 = __shfl_sync(FULL, p1, a & 31), v2 = __shfl_sync(FULL, p2, a & 31);
        lp[j] = (i < L) ? (a < 32 ? v0 : (a < 64 ? v1 : v2)) : 0.0f;
    }
    const float sum = numpy_sum_f32(lp[0], lp[1], lp[2], L, lane);
    const float uni = (L > 0) ? __fdiv_rn(1.0f, (float)L) : 0.0f;      // pv_mcts.py:50-56 (float64 there; unreachable with a softmax)
#pragma unroll
    for (int j = 0; j < 3; j++) {
        const int i = lane + 32 * j;
        if (i < L) T.node[base + i] = make_node(nth_legal(lm, i), (sum > 0.0f) ? __fdiv_rn(lp[j], sum) : uni);
    }
    if (lane == 0) T.node[leaf].w = (uint32_t)base | ((uint32_t)L << 20);
    c.n_nodes = base + L;
    backup(T, path, plen, k, net_value(P, leaf_net(P, c)) + row, 0, 0.0f, lane);
    c.sims_left -= k;
    c.pend_k = 0;
    if (lane == 0) atomicAdd(P.counters + 3, (unsigned long long)k);
}

// cpp/uttt_mcts.cpp:138-167 for the k queued copies of one leaf
__device__ void apply_leaf(const TreeParams& P, const TreeView& T, TreeCtl& c, const PackedState& st, const int32_t* path,
                           int lane) {
    uint32_t lm[3];
    int L = legal_mask(st, lm);
    int k = c.pend_k, plen = c.path_len;
    int leaf = path[plen - 1];
    int base = c.n_nodes;
    if (base + k * L > P.node_cap) {          // cannot happen with node_cap = 1 + 81 + 81*max_sims
        if (lane == 0) atomicExch(P.counters + 5, 1ull);
        c.phase = PHASE_DONE;
        return;
    }
    size_t row = (size_t)c.nn_row * (size_t)P.row_stride;
    const int g = leaf_symmetry(P, c, c.n_eval - 1);
    for (int cp = 0; cp < k; cp++) {
        float pr[3];
        legal_priors(net_policy(P, leaf_net(P, c)) + (row + (size_t)cp * P.copy_stride) * 81, g, lm, L, lane, pr);
        int reps = (P.copy_stride == 0) ? k : 1;       // identical rows: write all k copies at once
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const int a = lane + 32 * q;
            if (a < 81 && legal_bit(lm, a)) {
                int r = legal_rank(lm, a);
                for (int c2 = 0; c2 < reps; c2++) T.node[base + (cp + c2) * L + r] = make_node(a, pr[q]);
            }
        }
        if (P.copy_stride == 0) break;
    }
    if (lane == 0) T.node[leaf].w = (uint32_t)base | ((uint32_t)(k * L) << 20);
    c.n_nodes = base + k * L;
    backup(T, path, plen, k, net_value(P, leaf_net(P, c)) + row, P.copy_stride, 0.0f, lane);
    c.sims_left -= k;
    c.pend_k = 0;
    if (lane == 0) atomicAdd(P.counters + 3, (unsigned long long)k);
}

// both search modes: reset the evaluator queue and give every tree its root.  Self-play slot t starts game slot0 + t
// (a game's moves do not depend on its slot); later games are claimed from counters[0] as slots finish, which the
// host starts at the number of slots before the lanes fork.  Search mode keys UTTT_SP_RANDOM_SYMMETRY's draw and the
// root noise by the root's index.
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) tree_begin_kernel(TreeParams P) {
    int t = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (blockIdx.x == 0 && threadIdx.x == 0) { P.nn_count[0] = 0; P.nn_count[1] = 0; P.nn1_count[0] = 0; P.nn1_count[1] = 0; }
    if (t >= P.n_trees) return;
    TreeView T = view_of(P, t);
    TreeCtl c = P.ctl[t];
    c.ply = 0; c.game = 0; c.game_idx = -1; c.nn_row = 0; c.n_eval = 0;
    PackedState rs;
    if (P.mode == MODE_SELFPLAY) {
        unsigned long long g = (unsigned long long)(P.slot0 + t);
        if ((int64_t)g >= P.n_games) {
            c.phase = PHASE_DONE;
            if (lane == 0) P.ctl[t] = c;
            return;
        }
        c.game = P.game0 + g;
        c.game_idx = (int32_t)g;
        init_state(rs);
        warp_store_state(P.root + t, rs, lane);
    } else {
        c.game = (uint64_t)t;
        rs = warp_load_state(P.root + t, lane);
    }
    if (P.flags & UTTT_SP_THROUGHPUT) {
        c.phase = PHASE_ROOT;                // the first round queues the root for evaluation
    } else {
        init_root(P, T, c, rs, lane);
        if (c.n_root == 0) {                 // cpp/uttt_mcts.cpp:96-98: no legal move -> empty result
            c.phase = PHASE_DONE;
            if (lane == 0) { P.out_n[t] = 0; atomicAdd(P.counters + 6, 1ull); }
        } else {
            c.phase = PHASE_SEARCH;
        }
    }
    if (lane == 0) P.ctl[t] = c;
}

// 7 blocks per SM (at most 73 registers): left to itself ptxas gives the inlined pieces more registers, and spills
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK, 7) tree_round_kernel(TreeParams P) {
    pdl_trigger();          // the evaluator kernel behind this one may be scheduled now (it waits for this grid's results)
    pdl_wait();             // the previous round's evaluator has finished: policy / value rows are visible
    int t = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    // the other parity's counters were consumed by the previous round's evaluator passes: reset them
    if (blockIdx.x == 0 && threadIdx.x == 0) { P.nn_count[P.parity ^ 1] = 0; P.nn1_count[P.parity ^ 1] = 0; }
    if (t >= P.n_trees) return;
    // the control block, the pending leaf and the root position have nothing to wait for: one L2 round trip for the three
    const uint32_t leaf_raw = warp_load_state_issue(leaf_state(P, t, 0), lane);
    const uint32_t root_raw = warp_load_state_issue(P.root + t, lane);
    TreeCtl c = P.ctl[t];
    if (c.phase == PHASE_DONE) return;
    TreeView T = view_of(P, t);
    int32_t* path = leaf_path(P, t, 0);

    if (c.phase == PHASE_PENDING) {
        if (P.flags & UTTT_SP_PYSEARCH) apply_leaf_py(P, T, c, warp_load_state_finish(leaf_raw), path, lane);
        else apply_leaf(P, T, c, warp_load_state_finish(leaf_raw), path, lane);
        if (c.phase == PHASE_DONE) {
            if (lane == 0) P.ctl[t] = c;
            return;
        }
        c.phase = PHASE_SEARCH;
    }

    PackedState root = warp_load_state_finish(root_raw);
    int n_terminal = 0;
    for (;;) {
        if (c.sims_left <= 0) {
            if (!decide_move(P, T, t, c, root, 0.0f, lane)) break;
            __syncwarp();
            init_root(P, T, c, root, lane);
            __syncwarp();
        }

        const Descent d = descend(T, root, path, 0.0f, lane);
        if (d.end != LEAF_UNEXPANDED) {
            // cpp/uttt_mcts.cpp:19-21,115-118: the reference backs up -value with value = -1 for a lost
            // mover, i.e. +1 lands on the lost node itself (inverted sign, Q-M2); draws back up -0.0f.
            const bool lost = d.end == LEAF_LOST;
            float v = lost ? 1.0f : -0.0f;
            if (P.flags & UTTT_SP_CORRECT_TERMINAL_SIGN) v = lost ? -1.0f : 0.0f;
            backup(T, path, d.plen, 1, nullptr, 0, v, lane);
            c.sims_left -= 1;
            if (lane == 0) atomicAdd(P.counters + 3, 1ull);
            // Every tree of the batch waits for the slowest warp of the round: bound the work of one round.  The
            // remaining simulations simply continue next round (same order, same results).
            if (++n_terminal >= P.max_terminal && c.sims_left > 0) { c.phase = PHASE_SEARCH; break; }
            continue;
        }

        // ---------------- queue the leaf for the evaluator; fused leaf gather (cpp/uttt_game.cpp:244-280)
        const int k = min(P.batch, c.sims_left);                      // cpp/uttt_mcts.cpp:127 flush rule
        warp_store_state(leaf_state(P, t, 0), d.st, lane);
        c.nn_row = queue_leaf(P, t, c, d.st, d.lm, k, lane);
        c.phase = PHASE_PENDING;
        c.pend_k = k;
        c.path_len = d.plen;
        break;
    }
    if (lane == 0) P.ctl[t] = c;
}

// Deterministic integer-hash evaluator on the device (the "oracle evaluator" of the parity tests):
// identical arithmetic to orc_hash_eval in oracle/uttt_oracle.c.
__global__ void __launch_bounds__(128) hash_eval_kernel(const PackedState* __restrict__ states, const int32_t* __restrict__ count,
                                                        float* __restrict__ policy, float* __restrict__ value) {
    int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (row >= *count) return;
    PackedState st = warp_load_state(states + row, lane);
    uint32_t h = state_hash(st);
    for (int a = lane; a < 81; a += 32) {
        float num = (float)((mix32(h + (uint32_t)a) & 0xFFFFu) + 1u);
        policy[(size_t)row * 81 + a] = __fdiv_rn(__fdiv_rn(num, 65536.0f), 81.0f);
    }
    if (lane == 0) value[row] = __fdiv_rn(__fsub_rn((float)(int)(mix32(h ^ 0xABCDu) & 0xFFFFu), 32768.0f), 32768.0f);
}

// cpp/uttt_mcts.cpp:177-193: counts -> scores (one-hot at the first maximum for T==0, boltzman otherwise)
__global__ void scores_kernel(const int32_t* __restrict__ counts, const int32_t* __restrict__ nn, int n_trees,
                              float temperature, float* __restrict__ scores) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_trees) return;
    int n = nn[t];
    const int32_t* c = counts + (size_t)t * 81;
    float* s = scores + (size_t)t * 81;
    if (temperature == 0.0f) {
        int best = 0;
        for (int i = 1; i < n; i++)
            if ((float)c[i] > (float)c[best]) best = i;
        for (int i = 0; i < n; i++) s[i] = (i == best) ? 1.0f : 0.0f;
    } else {
        float inv = __fdiv_rn(1.0f, temperature), sum = 0.0f;
        for (int i = 0; i < n; i++) {
            float x = (float)c[i];
            float v = (inv == 1.0f) ? x : powf(x, inv);     // powf(x, 1) == x exactly
            s[i] = v;
            sum = __fadd_rn(sum, v);
        }
        if (sum > 0.0f)
            for (int i = 0; i < n; i++) s[i] = __fdiv_rn(s[i], sum);
    }
    for (int i = n; i < 81; i++) s[i] = 0.0f;
}

// cpp/uttt_mcts.cpp:199-216
__global__ void boltzman_kernel(const float* __restrict__ xs, int n, float temperature, float* __restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    float inv = __fdiv_rn(1.0f, temperature), sum = 0.0f;
    for (int i = 0; i < n; i++) {
        float v = (inv == 1.0f) ? xs[i] : powf(xs[i], inv);
        out[i] = v;
        sum = __fadd_rn(sum, v);
    }
    if (sum > 0.0f)
        for (int i = 0; i < n; i++) out[i] = __fdiv_rn(out[i], sum);
}

cudaError_t launch_tree_begin(const TreeParams& p, cudaStream_t s) {
    tree_begin_kernel<<<ceil_div(p.n_trees, WARPS_PER_BLOCK), 32 * WARPS_PER_BLOCK, 0, s>>>(p);
    return cudaGetLastError();
}
cudaError_t launch_tree_round(const TreeParams& p, cudaStream_t s) {
    return launch_pdl(tree_round_kernel, dim3(ceil_div(p.n_trees, WARPS_PER_BLOCK)), dim3(32 * WARPS_PER_BLOCK), 0, s, p);
}
cudaError_t launch_hash_eval(const PackedState* states, const int32_t* count, int max_rows, float* policy, float* value,
                             cudaStream_t s) {
    hash_eval_kernel<<<ceil_div(max_rows, 4), 128, 0, s>>>(states, count, policy, value);
    return cudaGetLastError();
}
cudaError_t launch_scores(const int32_t* counts, const int32_t* n, int n_trees, float temperature, float* scores,
                          cudaStream_t s) {
    scores_kernel<<<ceil_div(n_trees, 128), 128, 0, s>>>(counts, n, n_trees, temperature, scores);
    return cudaGetLastError();
}
cudaError_t launch_boltzman(const float* xs, int n, float temperature, float* out, cudaStream_t s) {
    boltzman_kernel<<<1, 32, 0, s>>>(xs, n, temperature, out);
    return cudaGetLastError();
}

}  // namespace uttt
