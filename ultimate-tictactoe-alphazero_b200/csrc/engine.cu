// engine.cu -- host side of libuttt_b200.so: the engine object (HBM arenas for trees, evaluator
// queues, network weights, history buffers) and the C-ABI entry points for the network forward,
// the batched search and the self-play loop.
//
// Reference call stack replaced (SURVEY.md section 3.2):
//   self_play_cpp.self_play -> play -> pv_mcts_scores_cpp -> uttt_cpp.pv_mcts_scores
//     -> C++ MCTS -> Python inference callback -> DualNetwork.forward
// Here every game of a self-play cycle is a slot on the device; one "round" is
//   tree_round kernel (apply previous evaluation, select next leaf, gather planes)
//   -> evaluator (trunk_auto_kernel: tensor-core trunk + heads in one launch; or the fp32 kernels / hash evaluator)
// (a match between two networks, UTTT_SP_MATCH, runs a second evaluator pass per round: slot 1's weights on slot 1's queue)
// enqueued back to back on one stream; the host keeps two windows of CHECK_EVERY rounds in flight and reads the
// progress counters of a window while the next one runs.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"

using namespace uttt;

namespace {

constexpr int CHECK_EVERY = 8;             // rounds per host progress check (self-play: per window)
constexpr int N_LANES = 2;
constexpr int N_WINDOWS = 2;           // self-play keeps two windows of CHECK_EVERY rounds in flight
constexpr int EV_PER_ROUND = 8;        // events of one lane's round: before the tree round, then 3 per evaluator pass (2 passes)
constexpr int EV_POOL = N_WINDOWS * CHECK_EVERY * EV_PER_ROUND * N_LANES;

__global__ void set_int_kernel(int32_t* p, int32_t v) { *p = v; }
__global__ void set_u64_kernel(unsigned long long* p, unsigned long long v) { *p = v; }

template <typename T>
cudaError_t dmalloc(T** p, size_t n) { return cudaMalloc((void**)p, n * sizeof(T)); }

}  // namespace

struct uttt_engine {
    uttt_config cfg;
    int n_sm;
    int node_cap;
    int rows_per_slot;      // evaluator rows per slot (max_batch: throughput mode queues up to that many leaves)
    cudaStream_t stream;
    cudaStream_t lane_stream[N_LANES];
    cudaEvent_t ev_fork, ev_join[N_LANES], ev_win[N_WINDOWS][N_LANES];
    // uttt_net_forward runs on the CALLER's stream but works in the engine's evaluator buffers: ev_fwd marks the end of the
    // last forward (the engine's own streams wait for it before they touch those buffers), ev_idle the point the engine's
    // stream had reached when a forward started (the forward waits for it)
    cudaEvent_t ev_fwd, ev_idle;
    bool fwd_pending;
    TreeParams tp;          // device pointers (n_trees / mode / sims set per call)
    float* policy;          // [n_slots*max_batch][81]
    float* value;           // [n_slots*max_batch]
    float* scores;          // [n_slots][81]
    float* act_a;           // [n_slots][81][128] fp32
    float* act_b;
    float* headfeat;        // [rows][243] head 1x1-conv outputs written by the tensor-core trunk
    float* tc_resid;        // [n_sm][32][512][4] fp32 residual stream of the tensor-core trunk (per CTA)
    int32_t* fwd_count;     // device int for uttt_net_forward
    int64_t* hist_offsets;  // [max_games + 1] exclusive prefix sums of the games' sample counts (uttt_selfplay_pack)
    long long* tc_dbg;      // [32][4] clock64 timeline of trunk CTA 0, then [64] histogram of batch sizes (diagnostics)
    int prof_level;         // self-play kernel timing: 2 = tree / trunk / heads events every round, 1 = trunk only, 0 = none
    int prof_sample;        // level 1: the trunk is bracketed in every prof_sample-th window of rounds only (see uttt_set_profile_level)
    int64_t prof_sampled_launches, prof_sampled_evals;      // trunk launches with events in the last run, positions they evaluated
    int lane_threshold;     // slots from which self-play splits into two overlapped lanes
    bool last_forced;       // the last self-play run had UTTT_SP_FORCED_PLAYOUTS: its policy targets are in tp.hist_target
    NetWeights w;           // weight slot 0
    NetWeights w1;          // weight slot 1 (UTTT_SP_MATCH), allocated by its first upload
    // slot 1's evaluator queue, the same per-row arrays as slot 0's (e->tp.nn_*, policy, value, headfeat); allocated by the
    // first slot-1 upload or match run, so that an engine that never plays a match keeps its footprint.  act_a / act_b /
    // tc_resid are scratch that both passes of a round share (they run one after the other on a lane's stream).
    struct {
        PackedState* states; __nv_bfloat16* planes; int32_t *tree, *k; float *policy, *value, *headfeat;
    } q1;
    unsigned long long* h_counters;   // pinned [8 * (1 + N_WINDOWS)]: [0..7] general use, then one copy per self-play window
    int32_t* h_count;                 // pinned [2]
    // step-wise search state
    int s_n_roots, s_sims, s_batch, s_round, s_pending, s_per_copy, s_have_results;
    // profiling of the last self-play run
    cudaEvent_t ev[EV_POOL];
    double prof_ms[4];
    int64_t prof_launches[4];
    std::vector<void*> allocs;
    // diagnostics (uttt_debug_trace): every evaluated leaf with the rows its tree is about to consume -- what
    // tests/test_gpu_replay.py and tests/test_gpu_throughput_oracle.py feed to the CPU searches
    uttt_progress_fn progress_cb;     // self-play: called when the number of finished games changed (per window of rounds)
    void* progress_user;
    bool trace_on;
    struct TraceRec { int32_t tree, game_idx, ply, round; float value; uint32_t state[8]; float policy[81]; };
    std::vector<TraceRec> trace;
};

namespace {

template <typename T>
int ealloc(uttt_engine* e, T** p, size_t n) {
    UTTT_CUDA_OK(dmalloc(p, n ? n : 1));
    e->allocs.push_back((void*)*p);
    return 0;
}

// the buffers one evaluator invocation works on (the whole engine, or one lane's slice of it) and the queue it reads
struct EvalBufs {
    PackedState* nn_states;
    __nv_bfloat16* nn_planes;
    int32_t *nn_tree, *nn_k;
    float *policy, *value, *act_a, *act_b, *resid, *headfeat;
};

// net 0: slot 0's queue; net 1: slot 1's (q1, allocated)
EvalBufs bufs_of(uttt_engine* e, size_t first_slot, int lane, int net = 0) {
    EvalBufs b;
    size_t first_row = first_slot * (size_t)e->rows_per_slot;
    b.nn_states = (net ? e->q1.states : e->tp.nn_states) + first_row;
    b.nn_planes = (net ? e->q1.planes : e->tp.nn_planes) + first_row * 243;
    b.nn_tree = (net ? e->q1.tree : e->tp.nn_tree) + first_row;
    b.nn_k = (net ? e->q1.k : e->tp.nn_k) + first_row;
    b.policy = (net ? e->q1.policy : e->policy) + first_slot * e->cfg.max_batch * 81;
    b.value = (net ? e->q1.value : e->value) + first_slot * e->cfg.max_batch;
    b.act_a = e->act_a + first_row * 81 * 128;
    b.act_b = e->act_b + first_row * 81 * 128;
    b.headfeat = (net ? e->q1.headfeat : e->headfeat) + first_row * 243;
    b.resid = e->tc_resid + (size_t)lane * e->n_sm * 512 * 64;     // fp16 panels: 128 KiB per CTA
    return b;
}

// self-play lane `lane` runs the slots [first, first + n_trees): its slice of the trees and of the evaluator queues (p),
// and of the evaluator's buffers of each network (b[net]; net 1 only with `match`)
void lane_of(uttt_engine* e, size_t first, int n_trees, int lane, bool match, TreeParams& p, EvalBufs b[2]) {
    b[0] = bufs_of(e, first, lane, 0);
    p = e->tp;
    p.n_trees = n_trees;
    p.slot0 = (int32_t)first;
    p.root += first; p.ctl += first;
    p.nodes += first * (size_t)e->node_cap;
    p.leaf_state += first * TP_MAX_LEAVES; p.paths += first * TP_MAX_LEAVES * PATH_CAP; p.tp_aux += first * 2 * TP_MAX_LEAVES;
    p.nn_states = b[0].nn_states; p.nn_planes = b[0].nn_planes; p.nn_tree = b[0].nn_tree; p.nn_k = b[0].nn_k;
    p.nn_count += 2 * lane;
    p.nn1_count += 2 * lane;
    p.policy = b[0].policy;
    p.value = b[0].value;
    if (match) {
        b[1] = bufs_of(e, first, lane, 1);
        p.nn1_states = b[1].nn_states; p.nn1_planes = b[1].nn_planes; p.nn1_tree = b[1].nn_tree; p.nn1_k = b[1].nn_k;
        p.policy1 = b[1].policy;
        p.value1 = b[1].value;
    }
}

// slot 1's evaluator queue (q1), on first use
int alloc_queue1(uttt_engine* e) {
    if (e->q1.states) return 0;
    const size_t S = (size_t)e->cfg.n_slots, R = S * (size_t)e->rows_per_slot;
    auto al = [&](auto** p, size_t n) -> int {
        UTTT_CUDA_OK(cudaMalloc((void**)p, (n ? n : 1) * sizeof(**p)));
        e->allocs.push_back((void*)*p);
        return 0;
    };
    decltype(e->q1) q;
    if (al(&q.planes, R * 243 + 8) || al(&q.tree, R) || al(&q.k, R) || al(&q.policy, S * e->cfg.max_batch * 81) ||
        al(&q.value, S * e->cfg.max_batch) || al(&q.headfeat, R * 243) || al(&q.states, R))
        return 1;
    e->q1 = q;
    return 0;
}

// work about to be enqueued on `s` touches the evaluator buffers / weights: order it behind an unfinished uttt_net_forward
int wait_for_forward(uttt_engine* e, cudaStream_t s) {
    if (e->fwd_pending) {
        UTTT_CUDA_OK(cudaStreamWaitEvent(s, e->ev_fwd, 0));
        e->fwd_pending = false;
    }
    return 0;
}

// one evaluator pass: the network `w` over the queue whose rows are b's and whose length is *count
int run_evaluator(uttt_engine* e, const NetWeights& w, const EvalBufs& b, int evaluator, const int32_t* count, int max_rows,
                  cudaStream_t s, cudaEvent_t* ev3 /* optional: [0] before trunk, [1] after trunk, [2] after heads */) {
    if (evaluator == UTTT_EVAL_HASH) {
        if (ev3) cudaEventRecord(ev3[0], s);
        UTTT_CUDA_OK(launch_hash_eval(b.nn_states, count, max_rows, b.policy, b.value, s));
        if (ev3) { cudaEventRecord(ev3[1], s); cudaEventRecord(ev3[2], s); }
        e->prof_launches[1] += 1;
        return 0;
    }
    UTTT_CHECK(w.loaded, "network weights not uploaded (uttt_upload_weights)");
    bool heads_fused = false;
    if (evaluator == UTTT_EVAL_NET_FP32) {
        if (ev3) cudaEventRecord(ev3[0], s);
        UTTT_CUDA_OK(launch_trunk_fp32(w, b.nn_planes, count, max_rows, b.act_a, b.act_b, s));
        e->prof_launches[1] += 1 + 2 * NET_BLOCKS;
    } else if (evaluator == UTTT_EVAL_NET_BF16X3) {
        // split-bf16 numerics: one launch for any batch (groups of <= 5 positions per CTA pair, several waves if needed);
        // the heads' FC layers follow as their own kernel (1 % of a round here: the trunk issues 3x the MMAs)
        if (ev3) cudaEventRecord(ev3[0], s);
        UTTT_CUDA_OK(launch_trunk_x3(w, b.nn_planes, b.headfeat, count, max_rows, b.resid, e->n_sm, s, e->tc_dbg));
        e->prof_launches[1] += 1;
    } else if (evaluator == UTTT_EVAL_NET_BF16) {
        // conv_input runs inside the trunk kernels (tensor pipe, "layer -1").  The queue length is only known on the
        // device: small batches (one wave of CTA pairs) are latency-bound -> one group per pair with the next layer
        // overlapping the epilogue, larger ones are throughput-bound -> two groups in flight with cta_group::2 MMAs.
        // trunk_auto_kernel makes that choice inside one launch (net_auto.cu).  Counted as ONE trunk launch per round.
        if (ev3) cudaEventRecord(ev3[0], s);
        // batches above 7 positions per CTA pair (only possible when max_rows allows them) are left to the
        // 10-positions-per-pair kernel; if no batch can exceed that, the heads' FC layers run in the tail of trunk_auto_kernel
        heads_fused = max_rows <= trunk_pp_cap1(e->n_sm);
        UTTT_CUDA_OK(launch_trunk_auto(w, b.nn_planes, b.headfeat, count, max_rows, b.resid, e->n_sm, s, e->tc_dbg,
                                       heads_fused ? b.policy : nullptr, heads_fused ? b.value : nullptr));
        if (!heads_fused)
            UTTT_CUDA_OK(launch_trunk_pp_large(w, b.nn_planes, b.headfeat, count, max_rows, b.resid, e->n_sm, s, e->tc_dbg));
        e->prof_launches[1] += 1;
    } else {
        UTTT_CHECK(false, "evaluator %d cannot run on the device", evaluator);
    }
    if (ev3) cudaEventRecord(ev3[1], s);
    if (heads_fused) {
        if (ev3 && e->prof_level >= 2) cudaEventRecord(ev3[2], s);
        return 0;
    }
    if (evaluator == UTTT_EVAL_NET_BF16 || evaluator == UTTT_EVAL_NET_BF16X3)
        UTTT_CUDA_OK(launch_heads_fc(w, b.headfeat, count, max_rows, b.policy, b.value, 1, s));
    else
        UTTT_CUDA_OK(launch_heads(w, b.act_a, nullptr, count, max_rows, b.policy, b.value, 1, s));
    e->prof_launches[2] += 1;
    if (ev3 && e->prof_level >= 2) cudaEventRecord(ev3[2], s);
    return 0;
}

// uttt_debug_trace: after the evaluator pass of round `round` over queue b, record (tree, game, ply, round, leaf state,
// policy row, value) of every leaf queued there: the untransformed leaf and its row in the leaf's own action ids
// (UTTT_SP_RANDOM_SYMMETRY: entry a = row entry sigma_g(a)), i.e. exactly what the tree consumes.  The row's owner:
// reference-exact mode, a PHASE_PENDING tree's row nn_row with leaf 0, evaluation n_eval - 1; throughput mode, a
// PHASE_ROOT_PENDING tree's row nn_row with its root, evaluation 0, or a PHASE_PENDING tree's rows tp_aux[t][1][j] (j <
// pend_k) with leaf j, evaluation n_eval - pend_k + j.  Synchronises the stream (diagnostics only).
int trace_round(uttt_engine* e, const TreeParams& p, const EvalBufs& b, const int32_t* count, int64_t round, cudaStream_t s) {
    UTTT_CUDA_OK(cudaStreamSynchronize(s));
    int32_t n_rows = 0;
    UTTT_CUDA_OK(cudaMemcpy(&n_rows, count, sizeof(n_rows), cudaMemcpyDeviceToHost));
    if (n_rows == 0) return 0;
    const bool tp = (p.flags & UTTT_SP_THROUGHPUT) != 0;
    const size_t T = (size_t)p.n_trees;
    std::vector<int32_t> trees((size_t)n_rows);
    UTTT_CUDA_OK(cudaMemcpy(trees.data(), b.nn_tree, (size_t)n_rows * 4, cudaMemcpyDeviceToHost));
    std::vector<float> pol((size_t)n_rows * 81), val((size_t)n_rows);
    std::vector<TreeCtl> ctl(T);
    std::vector<PackedState> leaf(T * TP_MAX_LEAVES), root(T);
    std::vector<int32_t> aux(T * 2 * TP_MAX_LEAVES);       // [t][0][j] path length, [t][1][j] row of pending leaf j
    UTTT_CUDA_OK(cudaMemcpy(leaf.data(), p.leaf_state, leaf.size() * sizeof(PackedState), cudaMemcpyDeviceToHost));
    UTTT_CUDA_OK(cudaMemcpy(root.data(), p.root, root.size() * sizeof(PackedState), cudaMemcpyDeviceToHost));
    UTTT_CUDA_OK(cudaMemcpy(aux.data(), p.tp_aux, aux.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
    UTTT_CUDA_OK(cudaMemcpy(pol.data(), b.policy, pol.size() * 4, cudaMemcpyDeviceToHost));
    UTTT_CUDA_OK(cudaMemcpy(val.data(), b.value, val.size() * 4, cudaMemcpyDeviceToHost));
    UTTT_CUDA_OK(cudaMemcpy(ctl.data(), p.ctl, ctl.size() * sizeof(TreeCtl), cudaMemcpyDeviceToHost));
    for (int r = 0; r < n_rows; r++) {
        const int t = trees[r];
        UTTT_CHECK(t >= 0 && t < p.n_trees, "trace: row %d does not belong to a pending tree", r);
        const TreeCtl& c = ctl[(size_t)t];
        const PackedState* st = nullptr;
        int j_eval = 0;
        if (!tp && c.phase == PHASE_PENDING && c.nn_row == r) {
            st = &leaf[(size_t)t * TP_MAX_LEAVES];
            j_eval = c.n_eval - 1;
        } else if (tp && c.phase == PHASE_ROOT_PENDING && c.nn_row == r) {
            st = &root[(size_t)t];
            j_eval = 0;
        } else if (tp && c.phase == PHASE_PENDING) {
            for (int j = 0; j < c.pend_k && j < TP_MAX_LEAVES; j++)
                if (aux[((size_t)t * 2 + 1) * TP_MAX_LEAVES + j] == r) {
                    st = &leaf[(size_t)t * TP_MAX_LEAVES + j];
                    j_eval = c.n_eval - c.pend_k + j;
                    break;
                }
        }
        UTTT_CHECK(st != nullptr, "trace: row %d does not belong to a pending tree", r);
        uttt_engine::TraceRec rec;
        rec.tree = p.slot0 + t;
        rec.game_idx = (p.mode == MODE_SELFPLAY) ? c.game_idx : p.slot0 + t;
        rec.ply = (p.mode == MODE_SELFPLAY) ? c.ply : 0;
        rec.round = (int32_t)round;
        rec.value = val[r];
        memcpy(rec.state, st, 32);
        const int g = (p.flags & UTTT_SP_RANDOM_SYMMETRY)
                          ? sym_draw(p.mode == MODE_SELFPLAY ? p.seed : 0u, c.game, (uint32_t)c.ply, (uint32_t)j_eval)
                          : 0;
        for (int a = 0; a < 81; a++) rec.policy[a] = pol[(size_t)r * 81 + sym_action(a, g)];
        e->trace.push_back(rec);
    }
    return 0;
}

int check_search_args(uttt_engine* e, int n_roots, int sims, int batch) {
    UTTT_CHECK(e != nullptr, "null engine");
    UTTT_CHECK(n_roots >= 0 && n_roots <= e->cfg.n_slots, "n_roots %d exceeds n_slots %d", n_roots, e->cfg.n_slots);
    UTTT_CHECK(sims >= 1 && sims <= e->cfg.max_sims, "evaluate_count %d outside [1, max_sims=%d]", sims, e->cfg.max_sims);
    UTTT_CHECK(batch >= 1 && batch <= e->cfg.max_batch, "batch_size %d outside [1, max_batch=%d]", batch, e->cfg.max_batch);
    return 0;
}

}  // namespace

extern "C" {

int uttt_create(const uttt_config* cfg, uttt_engine** out) {
    UTTT_CHECK(cfg && out, "null argument");
    UTTT_CHECK(cfg->n_slots >= 1 && cfg->max_sims >= 1 && cfg->max_batch >= 1 && cfg->max_games >= 0,
               "bad config (n_slots=%d max_sims=%d max_batch=%d)", cfg->n_slots, cfg->max_sims, cfg->max_batch);
    // node word limits: n in 16 bits, first_child in 20 bits, n_children (<= 81*batch) in 12 bits
    UTTT_CHECK(cfg->max_sims <= 12000 && cfg->max_batch <= 50, "max_sims <= 12000 and max_batch <= 50 supported");
    if (uttt_device_check(cfg->device)) return 1;
    UTTT_CUDA_OK(cudaSetDevice(cfg->device));
    uttt_engine* e = new uttt_engine();
    memset(&e->tp, 0, sizeof(e->tp));
    memset(&e->w, 0, sizeof(e->w));
    memset(&e->w1, 0, sizeof(e->w1));
    memset(&e->q1, 0, sizeof(e->q1));
    e->cfg = *cfg;
    e->trace_on = false;
    e->progress_cb = nullptr;
    e->progress_user = nullptr;
    e->prof_level = getenv("UTTT_PROFILE") ? atoi(getenv("UTTT_PROFILE")) : 1;
    e->prof_sample = getenv("UTTT_PROFILE_SAMPLE") ? atoi(getenv("UTTT_PROFILE_SAMPLE")) : 4;
    if (e->prof_sample < 1) e->prof_sample = 1;
    e->lane_threshold = getenv("UTTT_LANE_THRESHOLD") ? atoi(getenv("UTTT_LANE_THRESHOLD")) : 1024;
    UTTT_CUDA_OK(net_fp32_init());
    UTTT_CUDA_OK(trunk_tc2_init());
    UTTT_CUDA_OK(trunk_pp_init());
    UTTT_CUDA_OK(trunk_auto_init());
    cudaDeviceProp prop;
    UTTT_CUDA_OK(cudaGetDeviceProperties(&prop, cfg->device));
    e->n_sm = prop.multiProcessorCount;
    // worst case per tree: root + 81 root children + (sum of k over evaluations <= sims) * 81
    e->node_cap = 1 + 81 + 81 * cfg->max_sims;
    e->rows_per_slot = cfg->max_batch < TP_MAX_LEAVES ? cfg->max_batch : TP_MAX_LEAVES;
    UTTT_CUDA_OK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    size_t S = (size_t)cfg->n_slots, NC = (size_t)e->node_cap, G = (size_t)cfg->max_games;
    size_t R = S * (size_t)e->rows_per_slot;      // evaluator row capacity
    TreeParams& t = e->tp;
    t.node_cap = e->node_cap;
    if (ealloc(e, &t.root, S) || ealloc(e, &t.leaf_state, S * TP_MAX_LEAVES) ||
        ealloc(e, &t.paths, S * TP_MAX_LEAVES * PATH_CAP) || ealloc(e, &t.tp_aux, S * 2 * TP_MAX_LEAVES) || ealloc(e, &t.ctl, S) ||
        ealloc(e, &t.nodes, S * NC) ||
        ealloc(e, &t.nn_states, R) || ealloc(e, &t.nn_planes, R * 243 + 8) || ealloc(e, &t.nn_tree, R) ||
        ealloc(e, &t.nn_k, R) || ealloc(e, &t.nn_count, 4 * N_LANES) || ealloc(e, &t.out_counts, S * 81) ||
        ealloc(e, &t.out_n, S) || ealloc(e, &t.counters, 8) || ealloc(e, &t.hist_states, G * 81) ||
        ealloc(e, &t.hist_counts, G * 81 * 81) || ealloc(e, &t.hist_actions, G * 81) || ealloc(e, &t.hist_len, G) ||
        ealloc(e, &t.hist_final, G) || ealloc(e, &t.hist_value, G * 81) || ealloc(e, &t.hist_resigned, G) ||
        ealloc(e, &t.hist_full, G * 81) ||
        ealloc(e, &e->policy, S * cfg->max_batch * 81) ||
        ealloc(e, &e->value, S * cfg->max_batch) || ealloc(e, &e->scores, S * 81) ||
        ealloc(e, &e->headfeat, R * 243) || ealloc(e, &e->act_a, R * 81 * 128) || ealloc(e, &e->act_b, R * 81 * 128) ||
        ealloc(e, &e->tc_resid, (size_t)N_LANES * e->n_sm * 512 * 64) || ealloc(e, &e->fwd_count, 1) || ealloc(e, &e->tc_dbg, 128 + 64) ||
        ealloc(e, &e->hist_offsets, G + 1)) {
        uttt_destroy(e);
        return 1;
    }
    UTTT_CUDA_OK(cudaMemset(t.ctl, 0, S * sizeof(TreeCtl)));
    UTTT_CUDA_OK(cudaMemset(e->tc_dbg, 0, (128 + 64) * sizeof(long long)));
    UTTT_CUDA_OK(cudaMemset(t.nn_count, 0, 4 * N_LANES * sizeof(int32_t)));
    t.nn1_count = t.nn_count + 2 * N_LANES;         // slot 1's queue lengths: [lane][parity] behind slot 0's
    for (int i = 0; i < N_LANES; i++) {
        UTTT_CUDA_OK(cudaStreamCreateWithFlags(&e->lane_stream[i], cudaStreamNonBlocking));
        UTTT_CUDA_OK(cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming));
        for (int w = 0; w < N_WINDOWS; w++) UTTT_CUDA_OK(cudaEventCreateWithFlags(&e->ev_win[w][i], cudaEventDisableTiming));
    }
    UTTT_CUDA_OK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    UTTT_CUDA_OK(cudaEventCreateWithFlags(&e->ev_fwd, cudaEventDisableTiming));
    UTTT_CUDA_OK(cudaEventCreateWithFlags(&e->ev_idle, cudaEventDisableTiming));
    e->fwd_pending = false;
    UTTT_CUDA_OK(cudaMallocHost((void**)&e->h_counters, 8 * (1 + N_WINDOWS) * sizeof(unsigned long long)));
    UTTT_CUDA_OK(cudaMallocHost((void**)&e->h_count, 2 * sizeof(int32_t)));
    for (int i = 0; i < EV_POOL; i++) UTTT_CUDA_OK(cudaEventCreate(&e->ev[i]));
    t.policy = e->policy;
    t.value = e->value;
    t.max_terminal = getenv("UTTT_MAX_TERMINAL") ? atoi(getenv("UTTT_MAX_TERMINAL")) : 4;   // measured on the 500-game cycle: 2..4 best, 8: +0.8 %, 50: +8 %
    t.dir_alpha = 0.3f;
    t.dir_eps = 0.25f;
    t.temperature = 1.0f;
    t.resign_threshold = -0.95f;
    t.resign_check_fraction = 0.1f;
    t.fast_sims = 8;
    t.full_fraction = 0.25f;
    t.forced_k = 2.0f;
    e->last_forced = false;
    *out = e;
    return 0;
}

int uttt_destroy(uttt_engine* e) {
    if (!e) return 0;
    cudaSetDevice(e->cfg.device);
    cudaDeviceSynchronize();
    for (void* p : e->allocs) cudaFree(p);
    release_weights(e->w);
    release_weights(e->w1);
    if (e->h_counters) cudaFreeHost(e->h_counters);
    if (e->h_count) cudaFreeHost(e->h_count);
    for (int i = 0; i < EV_POOL; i++) if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    if (e->stream) cudaStreamDestroy(e->stream);
    for (int i = 0; i < N_LANES; i++) {
        if (e->lane_stream[i]) cudaStreamDestroy(e->lane_stream[i]);
        if (e->ev_join[i]) cudaEventDestroy(e->ev_join[i]);
        for (int w = 0; w < N_WINDOWS; w++) if (e->ev_win[w][i]) cudaEventDestroy(e->ev_win[w][i]);
    }
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->ev_fwd) cudaEventDestroy(e->ev_fwd);
    if (e->ev_idle) cudaEventDestroy(e->ev_idle);
    delete e;
    return 0;
}

// ---------------------------------------------------------------------------- weights
static int upload_impl(uttt_engine* e, int slot, const uttt_weights* w, int on_device, const float* const* res_tab,
                       const float* const (*res_bn_tab)[4]) {
    UTTT_CHECK(slot == 0 || slot == 1, "weight slot %d: must be 0 or 1", slot);
    UTTT_CHECK(e && w, "null argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    if (e->fwd_pending) {          // (the upload is synchronous and partly uses blocking copies: wait on the host)
        UTTT_CUDA_OK(cudaEventSynchronize(e->ev_fwd));
        e->fwd_pending = false;
    }
    if (slot == 1 && alloc_queue1(e)) return 1;
    return upload_weights(slot ? e->w1 : e->w, w, on_device, res_tab, res_bn_tab, e->stream);
}

int uttt_upload_weights_slot(uttt_engine* e, int slot, const uttt_weights* w, int on_device) {
    return upload_impl(e, slot, w, on_device, nullptr, nullptr);
}

int uttt_upload_weights_scattered_slot(uttt_engine* e, int slot, const uttt_weights_scattered* w, int on_device) {
    UTTT_CHECK(slot == 0 || slot == 1, "weight slot %d: must be 0 or 1", slot);
    UTTT_CHECK(e && w, "null argument");
    return upload_impl(e, slot, &w->small, on_device, w->res_conv_w, w->res_bn);
}

int uttt_upload_weights(uttt_engine* e, const uttt_weights* w, int on_device) {
    return uttt_upload_weights_slot(e, 0, w, on_device);
}

int uttt_upload_weights_scattered(uttt_engine* e, const uttt_weights_scattered* w, int on_device) {
    return uttt_upload_weights_scattered_slot(e, 0, w, on_device);
}

int uttt_net_forward(uttt_engine* e, const uint32_t* states_dev, int64_t n, int mode, float* policy_dev,
                     float* value_dev, void* stream) {
    UTTT_CHECK(e && (n == 0 || (states_dev && policy_dev && value_dev)), "null argument");
    UTTT_CHECK(mode == UTTT_EVAL_NET_BF16 || mode == UTTT_EVAL_NET_FP32 || mode == UTTT_EVAL_NET_BF16X3,
               "mode must be UTTT_EVAL_NET_BF16, _BF16X3 or _FP32");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    cudaStream_t s = (cudaStream_t)stream;
    // the engine's own stream may still be uploading weights or finishing a search in the same buffers
    UTTT_CUDA_OK(cudaEventRecord(e->ev_idle, e->stream));
    UTTT_CUDA_OK(cudaStreamWaitEvent(s, e->ev_idle, 0));
    for (int64_t off = 0; off < n; off += e->cfg.n_slots) {
        int m = (int)((n - off < e->cfg.n_slots) ? (n - off) : e->cfg.n_slots);
        if (uttt_game_gather_planes(states_dev + off * 8, e->tp.nn_planes, m, s)) return 1;
        set_int_kernel<<<1, 1, 0, s>>>(e->fwd_count, m);
        if (run_evaluator(e, e->w, bufs_of(e, 0, 0), mode, e->fwd_count, m, s, nullptr)) return 1;
        UTTT_CUDA_OK(cudaMemcpyAsync(policy_dev + off * 81, e->policy, (size_t)m * 81 * sizeof(float),
                                     cudaMemcpyDeviceToDevice, s));
        UTTT_CUDA_OK(cudaMemcpyAsync(value_dev + off, e->value, (size_t)m * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    UTTT_CUDA_OK(cudaEventRecord(e->ev_fwd, s));
    e->fwd_pending = true;
    return 0;
}

// ---------------------------------------------------------------------------- search
static int mcts_begin_impl(uttt_engine* e, const uint32_t* roots, int32_t n_roots, int32_t sims, int32_t batch, int32_t flags) {
    if (check_search_args(e, n_roots, sims, batch)) return 1;
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    TreeParams& t = e->tp;
    t.n_trees = n_roots; t.sims = sims; t.batch = batch; t.mode = MODE_SEARCH; t.flags = flags;
    t.parity = 0; t.row_stride = 1; t.copy_stride = 0;
    e->s_n_roots = n_roots; e->s_sims = sims; e->s_batch = batch; e->s_round = 0; e->s_pending = 0;
    e->s_per_copy = 0; e->s_have_results = 0;
    if (n_roots == 0) return 0;
    if (wait_for_forward(e, e->stream)) return 1;
    UTTT_CUDA_OK(cudaMemcpyAsync(t.root, roots, (size_t)n_roots * 32, cudaMemcpyHostToDevice, e->stream));
    UTTT_CUDA_OK(cudaMemsetAsync(t.counters, 0, 8 * sizeof(unsigned long long), e->stream));
    UTTT_CUDA_OK(launch_tree_begin(t, e->stream));
    return 0;
}

int uttt_mcts_begin(uttt_engine* e, const uint32_t* roots, int32_t n_roots, int32_t sims, int32_t batch) {
    return mcts_begin_impl(e, roots, n_roots, sims, batch, 0);
}

int uttt_mcts_advance(uttt_engine* e, int32_t* n_pending) {
    UTTT_CHECK(e && n_pending, "null argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    TreeParams& t = e->tp;
    if (e->s_n_roots == 0) { *n_pending = 0; return 0; }
    UTTT_CHECK(e->s_pending == 0 || e->s_have_results, "pending leaves have no results yet (uttt_mcts_put_results)");
    // a round may queue nothing although trees are still searching (bounded terminal work per round): keep going
    for (;;) {
        t.parity = e->s_round & 1;
        UTTT_CUDA_OK(launch_tree_round(t, e->stream));
        UTTT_CUDA_OK(cudaMemcpyAsync(e->h_count, t.nn_count + t.parity, sizeof(int32_t), cudaMemcpyDeviceToHost, e->stream));
        UTTT_CUDA_OK(cudaMemcpyAsync(e->h_counters, t.counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                                     e->stream));
        UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
        UTTT_CHECK(e->h_counters[5] == 0, "tree node arena overflow (node_cap=%d)", e->node_cap);
        e->s_round++;
        if (e->h_count[0] > 0 || (int64_t)e->h_counters[6] >= e->s_n_roots) break;
        UTTT_CHECK(e->s_round < 64 * (e->s_sims + 3), "search did not finish");
    }
    e->s_pending = e->h_count[0];
    e->s_have_results = 0;
    *n_pending = e->s_pending;
    return 0;
}

int uttt_mcts_get_leaves(uttt_engine* e, uint32_t* states, int32_t* k, int32_t* tree) {
    UTTT_CHECK(e, "null engine");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    int n = e->s_pending;
    if (n == 0) return 0;
    if (states) UTTT_CUDA_OK(cudaMemcpyAsync(states, e->tp.nn_states, (size_t)n * 32, cudaMemcpyDeviceToHost, e->stream));
    if (k) UTTT_CUDA_OK(cudaMemcpyAsync(k, e->tp.nn_k, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    if (tree) UTTT_CUDA_OK(cudaMemcpyAsync(tree, e->tp.nn_tree, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
    return 0;
}

int uttt_mcts_put_results(uttt_engine* e, const float* policy, const float* value, int per_copy) {
    UTTT_CHECK(e && policy && value, "null argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    int n = e->s_pending;
    size_t rows = per_copy ? (size_t)n * e->cfg.max_batch : (size_t)n;
    UTTT_CUDA_OK(cudaMemcpyAsync(e->policy, policy, rows * 81 * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    UTTT_CUDA_OK(cudaMemcpyAsync(e->value, value, rows * sizeof(float), cudaMemcpyHostToDevice, e->stream));
    e->tp.row_stride = per_copy ? e->cfg.max_batch : 1;
    e->tp.copy_stride = per_copy ? 1 : 0;
    e->s_have_results = 1;
    return 0;
}

int uttt_mcts_finish(uttt_engine* e, float temperature, float* scores, int32_t* counts, int32_t* n_scores) {
    UTTT_CHECK(e, "null engine");
    int n = e->s_n_roots;
    if (n == 0) return 0;
    UTTT_CUDA_OK(launch_scores(e->tp.out_counts, e->tp.out_n, n, temperature, e->scores, e->stream));
    if (scores) UTTT_CUDA_OK(cudaMemcpyAsync(scores, e->scores, (size_t)n * 81 * 4, cudaMemcpyDeviceToHost, e->stream));
    if (counts) UTTT_CUDA_OK(cudaMemcpyAsync(counts, e->tp.out_counts, (size_t)n * 81 * 4, cudaMemcpyDeviceToHost, e->stream));
    if (n_scores) UTTT_CUDA_OK(cudaMemcpyAsync(n_scores, e->tp.out_n, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
    UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
    return 0;
}

int uttt_mcts_search(uttt_engine* e, const uint32_t* roots, int32_t n_roots, int32_t sims, int32_t batch,
                     float temperature, int32_t evaluator, int32_t flags, float* scores, int32_t* counts,
                     int32_t* n_scores) {
    UTTT_CHECK(evaluator == UTTT_EVAL_NET_BF16 || evaluator == UTTT_EVAL_NET_FP32 || evaluator == UTTT_EVAL_HASH ||
                   evaluator == UTTT_EVAL_NET_BF16X3,
               "uttt_mcts_search needs a device evaluator; use the step-wise calls for UTTT_EVAL_HOST");
    const bool tp = (flags & UTTT_SP_THROUGHPUT) != 0;
    UTTT_CHECK(!tp || batch <= TP_MAX_LEAVES, "throughput mode: at most %d leaves per tree per round", TP_MAX_LEAVES);
    UTTT_CHECK(!(tp && (flags & UTTT_SP_PYSEARCH)), "UTTT_SP_PYSEARCH and UTTT_SP_THROUGHPUT exclude each other");
    UTTT_CHECK(!(flags & UTTT_SP_MATCH), "UTTT_SP_MATCH is a self-play mode (uttt_selfplay_run*), not a search option");
    UTTT_CHECK(!(flags & UTTT_SP_RESIGN), "UTTT_SP_RESIGN is a self-play mode (uttt_selfplay_run*), not a search option");
    UTTT_CHECK(!(flags & UTTT_SP_PLAYOUT_CAP), "UTTT_SP_PLAYOUT_CAP is a self-play mode (uttt_selfplay_run*), not a search option");
    UTTT_CHECK(!(flags & UTTT_SP_FORCED_PLAYOUTS),
               "UTTT_SP_FORCED_PLAYOUTS is a self-play mode (uttt_selfplay_run*), not a search option");
    if (mcts_begin_impl(e, roots, n_roots, sims, batch, flags)) return 1;     // uploads roots, runs the begin kernel
    if (n_roots == 0) return 0;
    TreeParams& t = e->tp;
    // rounds are enqueued without host synchronisation; the tree kernel ignores finished trees.
    // Upper bound on rounds: every round retires >= 1 simulation of every unfinished tree (+ root evaluation).
    const int rows = tp ? n_roots * batch : n_roots;
    const EvalBufs bufs = bufs_of(e, 0, 0);
    int max_rounds = sims + 3;
    int r = 0;
    while (r < max_rounds) {
        int stop = (r + CHECK_EVERY < max_rounds) ? r + CHECK_EVERY : max_rounds;
        for (; r < stop; r++) {
            t.parity = r & 1;
            UTTT_CUDA_OK(tp ? launch_tree_tp_round(t, e->stream) : launch_tree_round(t, e->stream));
            if (run_evaluator(e, e->w, bufs, evaluator, t.nn_count + t.parity, rows, e->stream, nullptr)) return 1;
            if (e->trace_on && trace_round(e, t, bufs, t.nn_count + t.parity, r, e->stream)) return 1;
        }
        UTTT_CUDA_OK(cudaMemcpyAsync(e->h_count, t.nn_count + ((r - 1) & 1), sizeof(int32_t), cudaMemcpyDeviceToHost,
                                     e->stream));
        UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
        // rounds may queue nothing (bounded terminal work per round): finished trees are counted on the device
        UTTT_CUDA_OK(cudaMemcpyAsync(e->h_counters, t.counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                                     e->stream));
        UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
        if ((int64_t)e->h_counters[6] >= n_roots) break;
        if (r >= max_rounds) max_rounds += CHECK_EVERY;
        UTTT_CHECK(max_rounds < 64 * (sims + 3), "search did not finish");
    }
    UTTT_CUDA_OK(cudaMemcpyAsync(e->h_counters, t.counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
    UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
    UTTT_CHECK(e->h_counters[5] == 0, "tree node arena overflow (node_cap=%d)", e->node_cap);
    e->s_n_roots = n_roots;
    return uttt_mcts_finish(e, temperature, scores, counts, n_scores);
}

int uttt_set_root_noise(uttt_engine* e, float alpha, float eps) {
    UTTT_CHECK(e && alpha > 0.0f && eps >= 0.0f && eps <= 1.0f, "bad root-noise parameters");
    e->tp.dir_alpha = alpha;
    e->tp.dir_eps = eps;
    return 0;
}

int uttt_debug_dirichlet(uint32_t seed, uint64_t game0, int64_t n, int32_t n_children, float alpha, float* out_dev, void* stream) {
    UTTT_CHECK(n >= 0 && n_children >= 1 && n_children <= 81 && alpha > 0.0f && (n == 0 || out_dev), "bad argument");
    UTTT_CUDA_OK(launch_dirichlet(seed, game0, n, n_children, alpha, out_dev, (cudaStream_t)stream));
    return 0;
}

int uttt_debug_root_noise(uint32_t seed, float alpha, const uint32_t* states_dev, const uint64_t* games_dev,
                          const int32_t* plies_dev, int64_t n, float* eta_dev, void* stream) {
    UTTT_CHECK(n >= 0 && alpha > 0.0f && (n == 0 || (states_dev && games_dev && plies_dev && eta_dev)), "bad argument");
    UTTT_CUDA_OK(launch_root_noise(seed, alpha, reinterpret_cast<const PackedState*>(states_dev), games_dev, plies_dev, n, eta_dev,
                                   (cudaStream_t)stream));
    return 0;
}

int uttt_set_progress_callback(uttt_engine* e, uttt_progress_fn fn, void* user) {
    UTTT_CHECK(e != nullptr, "null engine");
    e->progress_cb = fn;
    e->progress_user = user;
    return 0;
}

int uttt_set_selfplay_temperature(uttt_engine* e, float temperature) {
    UTTT_CHECK(e && temperature >= 0.0f && temperature == temperature, "bad temperature");
    e->tp.temperature = temperature;
    return 0;
}

int uttt_boltzman(const float* xs, int32_t n, float temperature, float* out) {
    UTTT_CHECK(xs && out && n >= 0, "bad argument");
    UTTT_CHECK(temperature != 0.0f, "temperature must be non-zero");
    if (n == 0) return 0;
    float *dx = nullptr, *dy = nullptr;
    UTTT_CUDA_OK(cudaMalloc((void**)&dx, n * sizeof(float)));
    UTTT_CUDA_OK(cudaMalloc((void**)&dy, n * sizeof(float)));
    UTTT_CUDA_OK(cudaMemcpy(dx, xs, n * sizeof(float), cudaMemcpyHostToDevice));
    UTTT_CUDA_OK(launch_boltzman(dx, n, temperature, dy, 0));
    UTTT_CUDA_OK(cudaMemcpy(out, dy, n * sizeof(float), cudaMemcpyDeviceToHost));
    cudaFree(dx);
    cudaFree(dy);
    return 0;
}

// ---------------------------------------------------------------------------- self-play
int uttt_selfplay_run_device(uttt_engine* e, int64_t n_games, uint64_t game0, int32_t sims, int32_t batch,
                             uint32_t seed, int32_t evaluator, int32_t flags, int64_t* stats, void* stream) {
    UTTT_CHECK(e != nullptr, "null engine");
    UTTT_CHECK(n_games >= 0 && n_games <= e->cfg.max_games, "n_games %lld exceeds max_games %lld", (long long)n_games,
               (long long)e->cfg.max_games);
    UTTT_CHECK(evaluator == UTTT_EVAL_NET_BF16 || evaluator == UTTT_EVAL_NET_FP32 || evaluator == UTTT_EVAL_HASH ||
                   evaluator == UTTT_EVAL_NET_BF16X3,
               "self-play needs a device evaluator");
    int n_trees = (int)((n_games < e->cfg.n_slots) ? n_games : e->cfg.n_slots);
    if (check_search_args(e, n_trees, sims, batch)) return 1;
    const bool match = (flags & UTTT_SP_MATCH) != 0;
    UTTT_CHECK(match || !(flags & UTTT_SP_PYSEARCH),
               "UTTT_SP_PYSEARCH is a search option (uttt_mcts_search) and a match option (UTTT_SP_MATCH), not a self-play mode");
    const bool tp = (flags & UTTT_SP_THROUGHPUT) != 0;
    UTTT_CHECK(!(tp && (flags & UTTT_SP_PYSEARCH)), "UTTT_SP_PYSEARCH and UTTT_SP_THROUGHPUT exclude each other");
    UTTT_CHECK(!tp || batch <= TP_MAX_LEAVES, "throughput mode: at most %d leaves per tree per round", TP_MAX_LEAVES);
    // under the reference's inverted terminal sign (tree_kernels.cu, round kernel) a move that wins at once backs up as
    // a loss, so a root value says nothing a resignation could rest on
    UTTT_CHECK(!(flags & UTTT_SP_RESIGN) || tp || (flags & UTTT_SP_CORRECT_TERMINAL_SIGN),
               "UTTT_SP_RESIGN needs terminal values of the correct sign: add UTTT_SP_CORRECT_TERMINAL_SIGN or use UTTT_SP_THROUGHPUT");
    if (flags & UTTT_SP_PLAYOUT_CAP) {
        UTTT_CHECK(!match, "UTTT_SP_PLAYOUT_CAP and UTTT_SP_MATCH exclude each other (a match records no training targets)");
        UTTT_CHECK(e->tp.fast_sims <= sims, "UTTT_SP_PLAYOUT_CAP: fast_sims %d exceeds evaluate_count %d", e->tp.fast_sims, sims);
    }
    const bool forced = (flags & UTTT_SP_FORCED_PLAYOUTS) != 0;
    if (forced) {
        // the reference-exact root is uniform and never noised: forcing its children is not what the rule is for
        UTTT_CHECK(tp, "UTTT_SP_FORCED_PLAYOUTS needs UTTT_SP_THROUGHPUT");
        UTTT_CHECK(!match, "UTTT_SP_FORCED_PLAYOUTS and UTTT_SP_MATCH exclude each other (a match records no training targets)");
    }
    UTTT_CHECK(!match || evaluator == UTTT_EVAL_HASH || e->w1.loaded,
               "UTTT_SP_MATCH: weight slot 1 was never uploaded (uttt_upload_weights_slot(e, 1, ...))");
    const int rows_per_tree = tp ? batch : 1;
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    if (match && alloc_queue1(e)) return 1;
    // the policy targets on first use, so that an engine that never uses the flag keeps its footprint
    if (forced && !e->tp.hist_target && ealloc(e, &e->tp.hist_target, (size_t)e->cfg.max_games * 81 * 81)) return 1;
    e->last_forced = forced;
    cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
    for (int i = 0; i < 4; i++) { e->prof_ms[i] = 0.0; e->prof_launches[i] = 0; }
    e->prof_sampled_launches = e->prof_sampled_evals = 0;
    if (stats) stats[0] = stats[1] = stats[2] = stats[3] = 0;
    if (n_games == 0) return 0;
    if (wait_for_forward(e, s)) return 1;
    TreeParams& t = e->tp;
    t.sims = sims; t.batch = batch; t.mode = MODE_SELFPLAY; t.flags = flags;
    t.parity = 0; t.row_stride = 1; t.copy_stride = 0;
    t.seed = seed; t.game0 = game0; t.n_games = n_games;
    // Two lanes (halves of the slots) run on two streams: each lane is the sequential chain
    // tree_round -> conv_input -> trunk -> heads, so one lane's tree/heads work runs in the shadow of the
    // other lane's trunk (the tree blocks fit beside a trunk CTA on an SM).  Lanes share only the atomic
    // game/progress counters and the history buffers (disjoint rows).
    // (worth it only when half a batch still fills the machine; small batches are latency-bound)
    const int n_lanes = (n_trees >= e->lane_threshold) ? N_LANES : 1;
    // A match runs two evaluator passes per round and lane, slot 0's network on slot 0's queue, then slot 1's on slot 1's:
    // each is the usual chain of programmatic dependent launches, so the second trunk launch follows the first pass's
    // last kernel (which, like every kernel of the chain, waits for its predecessor before it touches memory) and reuses
    // its scratch.  A pass whose queue is empty costs its launches only: the kernels read the count and exit.
    const int n_nets = match ? 2 : 1;
    TreeParams lane_tp[N_LANES];
    EvalBufs lane_bufs[N_LANES][2];
    int lane_trees[N_LANES];
    for (int l = 0; l < n_lanes; l++) {
        size_t first = (size_t)l * (size_t)(n_trees / n_lanes);
        lane_trees[l] = (l == n_lanes - 1) ? n_trees - (int)first : n_trees / n_lanes;
        lane_of(e, first, lane_trees[l], l, match, lane_tp[l], lane_bufs[l]);
    }
    UTTT_CUDA_OK(cudaMemsetAsync(t.counters, 0, 8 * sizeof(unsigned long long), s));
    // (counters[0] = next game to hand out: the first n_trees games are assigned by tree_begin; set here, before the lanes
    // fork, so that no lane's begin kernel races with another lane's first recycled slot)
    set_u64_kernel<<<1, 1, 0, s>>>(t.counters, (unsigned long long)n_trees);
    UTTT_CUDA_OK(cudaMemsetAsync(t.hist_len, 0, (size_t)n_games * sizeof(int32_t), s));
    UTTT_CUDA_OK(cudaMemsetAsync(t.hist_resigned, 0, (size_t)n_games, s));
    UTTT_CUDA_OK(cudaEventRecord(e->ev_fork, s));
    cudaStream_t ls[N_LANES];
    for (int l = 0; l < n_lanes; l++) {
        ls[l] = (n_lanes == 1) ? s : e->lane_stream[l];
        if (n_lanes > 1) UTTT_CUDA_OK(cudaStreamWaitEvent(ls[l], e->ev_fork, 0));
        UTTT_CUDA_OK(launch_tree_begin(lane_tp[l], ls[l]));
        e->prof_launches[0] += 1;
    }
    // every round retires >= 1 simulation of every live slot: hard upper bound on rounds
    int64_t waves = (n_games + n_trees - 1) / n_trees;
    int64_t max_rounds = waves * 82 * (int64_t)(sims + 3) * (tp ? 4 : 1) + CHECK_EVERY;
    int64_t r = 0, reported = 0;
    bool done = false;
    // Two windows of CHECK_EVERY rounds are kept in flight: window w+1 is enqueued before the host waits for window w,
    // so the GPU never idles while the host reads the progress counters and the per-kernel event times (one window at
    // a time, that wait cost ~230 us of GPU idle time per window = 4 % of a 500-game cycle).  The price is up to one
    // extra window of rounds after the last game ended (every kernel of such a round exits at once).
    // Level 1 brackets the trunk launches of every prof_sample-th window only: the two event records per round cost 1.6 % of a
    // 500-game cycle (183 k -> 180 k moves/s, with or without programmatic dependent launch); the positions those launches
    // evaluated come from the evaluation counter in the windows' progress copies.
    int64_t n_enqueued = 0;
    bool win_sampled[N_WINDOWS] = {};
    unsigned long long last_evals = 0;
    auto enqueue_window = [&](int slot) -> int {
        const bool sampled = e->prof_level >= 2 || (e->prof_level == 1 && n_enqueued % e->prof_sample == 0);
        win_sampled[slot] = sampled;
        n_enqueued++;
        for (int i = 0; i < CHECK_EVERY; i++, r++) {
            for (int l = 0; l < n_lanes; l++) {
                cudaEvent_t* ev = e->ev + EV_PER_ROUND * ((slot * CHECK_EVERY + i) * N_LANES + l);
                lane_tp[l].parity = (int)(r & 1);
                if (e->prof_level >= 2) cudaEventRecord(ev[0], ls[l]);
                UTTT_CUDA_OK(tp ? launch_tree_tp_round(lane_tp[l], ls[l]) : launch_tree_round(lane_tp[l], ls[l]));
                e->prof_launches[0] += 1;
                for (int net = 0; net < n_nets; net++) {
                    const int32_t* count = (net ? lane_tp[l].nn1_count : lane_tp[l].nn_count) + lane_tp[l].parity;
                    if (run_evaluator(e, net ? e->w1 : e->w, lane_bufs[l][net], evaluator, count, lane_trees[l] * rows_per_tree,
                                      ls[l], sampled ? ev + 1 + 3 * net : nullptr))
                        return 1;
                }
                for (int net = 0; net < n_nets && e->trace_on; net++)
                    if (trace_round(e, lane_tp[l], lane_bufs[l][net],
                                    (net ? lane_tp[l].nn1_count : lane_tp[l].nn_count) + lane_tp[l].parity, r, ls[l]))
                        return 1;
            }
        }
        UTTT_CUDA_OK(cudaMemcpyAsync(e->h_counters + 8 * (1 + slot), t.counters, 8 * sizeof(unsigned long long),
                                     cudaMemcpyDeviceToHost, ls[0]));
        for (int l = 0; l < n_lanes; l++) UTTT_CUDA_OK(cudaEventRecord(e->ev_win[slot][l], ls[l]));
        return 0;
    };
    auto retire_window = [&](int slot) -> int {
        for (int l = 0; l < n_lanes; l++) UTTT_CUDA_OK(cudaEventSynchronize(e->ev_win[slot][l]));
        for (int i = 0; i < CHECK_EVERY; i++) {
            for (int l = 0; l < n_lanes; l++) {
                float ms = 0.f;
                cudaEvent_t* ev = e->ev + EV_PER_ROUND * ((slot * CHECK_EVERY + i) * N_LANES + l);
                for (int net = 0; net < n_nets; net++) {       // pass `net`: [1 + 3 net] trunk [2 + 3 net] heads [3 + 3 net]
                    cudaEvent_t* p = ev + 3 * net;
                    if (win_sampled[slot]) { cudaEventElapsedTime(&ms, p[1], p[2]); e->prof_ms[1] += ms; e->prof_sampled_launches += 1; }
                    if (e->prof_level >= 2) { cudaEventElapsedTime(&ms, p[2], p[3]); e->prof_ms[2] += ms; }
                }
                if (e->prof_level >= 2) {
                    cudaEventElapsedTime(&ms, ev[0], ev[1]); e->prof_ms[0] += ms;
                    cudaEventElapsedTime(&ms, ev[0], ev[3 * n_nets]); e->prof_ms[3] += ms;
                }
            }
        }
        const unsigned long long* hc = e->h_counters + 8 * (1 + slot);
        // (every leaf queued by a tree round of this window was evaluated by a trunk launch of this window)
        if (win_sampled[slot]) e->prof_sampled_evals += (int64_t)(hc[4] - last_evals);
        last_evals = hc[4];
        UTTT_CHECK(hc[5] == 0, "tree node arena overflow (node_cap=%d)", e->node_cap);
        // lane 0's copy may predate lane 1's last rounds: "done" only ever lags, never leads
        done = (int64_t)hc[1] >= n_games;
        if (e->progress_cb && (int64_t)hc[1] != reported) {
            reported = (int64_t)hc[1];
            e->progress_cb(reported < n_games ? reported : n_games, n_games, e->progress_user);
        }
        return 0;
    };
    int head = 0, in_flight = 0;                 // windows are retired in the order they were enqueued
    while (!done && (r < max_rounds || in_flight > 0)) {
        while (in_flight < N_WINDOWS && r < max_rounds) {
            if (enqueue_window((head + in_flight) % N_WINDOWS)) return 1;
            in_flight++;
        }
        if (retire_window(head)) return 1;
        head = (head + 1) % N_WINDOWS;
        in_flight--;
    }
    while (in_flight > 0) {                      // the window enqueued behind the one that saw the last game end
        bool was_done = done;
        if (retire_window(head)) return 1;
        done = done || was_done;
        head = (head + 1) % N_WINDOWS;
        in_flight--;
    }
    if (n_lanes > 1) {          // join: the caller's stream continues after both lanes
        for (int l = 0; l < n_lanes; l++) {
            UTTT_CUDA_OK(cudaEventRecord(e->ev_join[l], ls[l]));
            UTTT_CUDA_OK(cudaStreamWaitEvent(s, e->ev_join[l], 0));
        }
    }
    UTTT_CUDA_OK(cudaMemcpy(e->h_counters, t.counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    UTTT_CHECK(done, "self-play did not finish within %lld rounds", (long long)max_rounds);
    e->prof_launches[3] = e->prof_launches[0] + e->prof_launches[1] + e->prof_launches[2];
    if (stats) {
        stats[0] = (int64_t)e->h_counters[2];
        stats[1] = (int64_t)e->h_counters[3];
        stats[2] = (int64_t)e->h_counters[4];
        stats[3] = r;
    }
    return 0;
}

int uttt_selfplay_fetch(uttt_engine* e, int64_t n_games, uint32_t* hist_states, uint16_t* hist_counts,
                        uint8_t* hist_actions, int32_t* hist_len, int8_t* hist_final) {
    UTTT_CHECK(e && n_games <= e->cfg.max_games, "bad argument");
    if (n_games <= 0) return 0;
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    size_t G = (size_t)n_games;
    cudaStream_t s = e->stream;
    const TreeParams& t = e->tp;
    if (hist_states) UTTT_CUDA_OK(cudaMemcpyAsync(hist_states, t.hist_states, G * 81 * 32, cudaMemcpyDeviceToHost, s));
    if (hist_counts) UTTT_CUDA_OK(cudaMemcpyAsync(hist_counts, t.hist_counts, G * 81 * 81 * 2, cudaMemcpyDeviceToHost, s));
    if (hist_actions) UTTT_CUDA_OK(cudaMemcpyAsync(hist_actions, t.hist_actions, G * 81, cudaMemcpyDeviceToHost, s));
    if (hist_len) UTTT_CUDA_OK(cudaMemcpyAsync(hist_len, t.hist_len, G * 4, cudaMemcpyDeviceToHost, s));
    if (hist_final) UTTT_CUDA_OK(cudaMemcpyAsync(hist_final, t.hist_final, G, cudaMemcpyDeviceToHost, s));
    UTTT_CUDA_OK(cudaStreamSynchronize(s));
    return 0;
}

int uttt_set_resign(uttt_engine* e, float threshold, float check_fraction) {
    UTTT_CHECK(threshold >= -1.0f && threshold <= 1.0f, "resign threshold %g: must be a number in [-1, 1]", (double)threshold);
    UTTT_CHECK(check_fraction >= 0.0f && check_fraction <= 1.0f, "resign check fraction %g: must be in [0, 1]",
               (double)check_fraction);
    UTTT_CHECK(e != nullptr, "null engine");
    e->tp.resign_threshold = threshold;
    e->tp.resign_check_fraction = check_fraction;
    return 0;
}

int uttt_selfplay_fetch_values(uttt_engine* e, int64_t n_games, float* hist_value, int8_t* hist_resigned) {
    UTTT_CHECK(e && n_games <= e->cfg.max_games, "bad argument");
    if (n_games <= 0) return 0;
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    const size_t G = (size_t)n_games;
    cudaStream_t s = e->stream;
    if (hist_value) UTTT_CUDA_OK(cudaMemcpyAsync(hist_value, e->tp.hist_value, G * 81 * sizeof(float), cudaMemcpyDeviceToHost, s));
    if (hist_resigned) UTTT_CUDA_OK(cudaMemcpyAsync(hist_resigned, e->tp.hist_resigned, G, cudaMemcpyDeviceToHost, s));
    UTTT_CUDA_OK(cudaStreamSynchronize(s));
    return 0;
}

int uttt_set_playout_cap(uttt_engine* e, int32_t fast_sims, float full_fraction) {
    UTTT_CHECK(full_fraction >= 0.0f && full_fraction <= 1.0f, "playout cap full fraction %g: must be in [0, 1]", (double)full_fraction);
    UTTT_CHECK(fast_sims >= 1, "playout cap fast_sims %d: must be at least 1", fast_sims);
    UTTT_CHECK(e != nullptr, "null engine");
    UTTT_CHECK(fast_sims <= e->cfg.max_sims, "playout cap fast_sims %d exceeds the engine's max_sims %d", fast_sims, e->cfg.max_sims);
    e->tp.fast_sims = fast_sims;
    e->tp.full_fraction = full_fraction;
    return 0;
}

int uttt_selfplay_fetch_full(uttt_engine* e, int64_t n_games, uint8_t* hist_full) {
    UTTT_CHECK(e && n_games <= e->cfg.max_games && (hist_full || n_games <= 0), "bad argument");
    if (n_games <= 0) return 0;
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    UTTT_CUDA_OK(cudaMemcpyAsync(hist_full, e->tp.hist_full, (size_t)n_games * 81, cudaMemcpyDeviceToHost, e->stream));
    UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
    return 0;
}

int uttt_set_forced_playouts(uttt_engine* e, float k) {
    UTTT_CHECK(k > 0.0f && k <= 100.0f, "forced playouts k %g: must be in (0, 100]", (double)k);
    UTTT_CHECK(e != nullptr, "null engine");
    e->tp.forced_k = k;
    return 0;
}

int uttt_selfplay_fetch_target(uttt_engine* e, int64_t n_games, uint16_t* hist_target) {
    UTTT_CHECK(e && n_games <= e->cfg.max_games && (hist_target || n_games <= 0), "bad argument");
    if (n_games <= 0) return 0;
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    const uint16_t* src = e->last_forced ? e->tp.hist_target : e->tp.hist_counts;
    UTTT_CUDA_OK(cudaMemcpyAsync(hist_target, src, (size_t)n_games * 81 * 81 * 2, cudaMemcpyDeviceToHost, e->stream));
    UTTT_CUDA_OK(cudaStreamSynchronize(e->stream));
    return 0;
}

int uttt_selfplay_pack(uttt_engine* e, int64_t n_games, void* out_dev, int64_t cap_samples, int64_t* n_samples_out, void* stream) {
    UTTT_CHECK(e && n_samples_out && n_games >= 0 && n_games <= e->cfg.max_games && (out_dev || cap_samples == 0), "bad argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    cudaStream_t s = stream ? (cudaStream_t)stream : e->stream;
    const TreeParams& t = e->tp;
    *n_samples_out = 0;
    if (n_games == 0) return 0;
    UTTT_CUDA_OK(launch_scan_samples(t.hist_len, t.hist_full, n_games, e->hist_offsets, s));
    long long total = 0;
    UTTT_CUDA_OK(cudaMemcpyAsync(&total, e->hist_offsets + n_games, sizeof(total), cudaMemcpyDeviceToHost, s));
    UTTT_CUDA_OK(cudaStreamSynchronize(s));
    UTTT_CHECK(total <= cap_samples, "sample buffer too small: %lld samples, room for %lld", total, (long long)cap_samples);
    // policy target counts: the pruned ones of a run with UTTT_SP_FORCED_PLAYOUTS, the visit counts otherwise
    const uint16_t* counts = e->last_forced ? t.hist_target : t.hist_counts;
    UTTT_CUDA_OK(launch_pack_samples(t.hist_states, counts, t.hist_len, t.hist_full, t.hist_final, e->hist_offsets, n_games,
                                     out_dev, cap_samples, s));
    *n_samples_out = total;
    return 0;
}

int uttt_samples_unpack(const void* samples_dev, int64_t n, float* x_dev, float* policy_dev, float* value_dev, void* stream) {
    UTTT_CHECK(n >= 0 && (n == 0 || (samples_dev && x_dev && policy_dev && value_dev)), "bad argument");
    UTTT_CUDA_OK(launch_unpack_samples(samples_dev, n, x_dev, policy_dev, value_dev, (cudaStream_t)stream));
    return 0;
}

int uttt_selfplay_run(uttt_engine* e, int64_t n_games, uint64_t game0, int32_t sims, int32_t batch, uint32_t seed,
                      int32_t evaluator, int32_t flags, uint32_t* hist_states, uint16_t* hist_counts,
                      uint8_t* hist_actions, int32_t* hist_len, int8_t* hist_final, int64_t* stats) {
    if (uttt_selfplay_run_device(e, n_games, game0, sims, batch, seed, evaluator, flags, stats, nullptr)) return 1;
    return uttt_selfplay_fetch(e, n_games, hist_states, hist_counts, hist_actions, hist_len, hist_final);
}

int uttt_debug_trunk_timeline(uttt_engine* e, int64_t* out128) {
    UTTT_CHECK(e && out128, "null argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    UTTT_CUDA_OK(cudaDeviceSynchronize());
    UTTT_CUDA_OK(cudaMemcpy(out128, e->tc_dbg, 128 * sizeof(long long), cudaMemcpyDeviceToHost));
    return 0;
}

int uttt_debug_batch_histogram(uttt_engine* e, int64_t* out64, int32_t reset) {
    UTTT_CHECK(e && out64, "null argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    UTTT_CUDA_OK(cudaDeviceSynchronize());
    UTTT_CUDA_OK(cudaMemcpy(out64, e->tc_dbg + 128, 64 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (reset) UTTT_CUDA_OK(cudaMemset(e->tc_dbg + 128, 0, 64 * sizeof(long long)));
    return 0;
}

int uttt_debug_trace(uttt_engine* e, int enable) {
    UTTT_CHECK(e != nullptr, "null engine");
    e->trace_on = enable != 0;
    e->trace.clear();
    return 0;
}

int uttt_debug_trace_read(uttt_engine* e, int64_t cap, int64_t* n_out, int32_t* meta, uint32_t* states, float* policy,
                          float* value) {
    UTTT_CHECK(e && n_out, "null argument");
    const int64_t n = (int64_t)e->trace.size();
    *n_out = n;
    if (cap <= 0) return 0;
    UTTT_CHECK(cap >= n && meta && states && policy && value, "trace buffers too small (%lld records)", (long long)n);
    for (int64_t i = 0; i < n; i++) {
        const uttt_engine::TraceRec& r = e->trace[(size_t)i];
        meta[4 * i] = r.tree; meta[4 * i + 1] = r.game_idx; meta[4 * i + 2] = r.ply; meta[4 * i + 3] = r.round;
        memcpy(states + 8 * i, r.state, 32);
        memcpy(policy + 81 * i, r.policy, 81 * 4);
        value[i] = r.value;
    }
    return 0;
}

int uttt_debug_counters(uttt_engine* e, uint64_t* out8) {
    UTTT_CHECK(e && out8, "null argument");
    UTTT_CUDA_OK(cudaSetDevice(e->cfg.device));
    UTTT_CUDA_OK(cudaDeviceSynchronize());
    UTTT_CUDA_OK(cudaMemcpy(out8, e->tp.counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return 0;
}

int uttt_set_profile_level(uttt_engine* e, int level) {
    UTTT_CHECK(e != nullptr, "null engine");
    UTTT_CHECK(level >= 0 && level <= 2, "profile level %d outside [0, 2]", level);
    e->prof_level = level;
    return 0;
}

int uttt_last_run_profile(uttt_engine* e, int kind, double* ms_out, int64_t* launches_out) {
    UTTT_CHECK(e && kind >= 0 && kind < 6, "bad argument");
    if (kind < 4) {
        if (ms_out) *ms_out = e->prof_ms[kind];
        if (launches_out) *launches_out = e->prof_launches[kind];
    } else {            // the trunk launches that were bracketed by events: 4 -> (their ms, their number), 5 -> (their ms, positions)
        if (ms_out) *ms_out = e->prof_ms[1];
        if (launches_out) *launches_out = kind == 4 ? e->prof_sampled_launches : e->prof_sampled_evals;
    }
    return 0;
}

}  // extern "C"
