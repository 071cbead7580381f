// common.cuh -- shared declarations of libuttt_b200.so (internal).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/uttt_b200.h"
#include "uttt_rules.cuh"

namespace uttt {

void set_error(const char* fmt, ...);

#define UTTT_CUDA_OK(expr)                                                                   \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            ::uttt::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return 1;                                                                        \
        }                                                                                    \
    } while (0)

#define UTTT_CHECK(cond, ...)               \
    do {                                    \
        if (!(cond)) {                      \
            ::uttt::set_error(__VA_ARGS__); \
            return 2;                       \
        }                                   \
    } while (0)

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Programmatic dependent launch (the round loop is tree_round -> trunk -> tree_round -> ...: each kernel needs the previous
// one's output from its first instruction, but its blocks can be scheduled and resident while the previous kernel drains,
// which hides the launch latency of the boundary).  A kernel launched through launch_pdl may start before its predecessor
// in the stream has finished: it must execute pdl_wait() before touching anything the predecessor writes, and may call
// pdl_trigger() to let its own successor be scheduled early.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

// ---------------------------------------------------------------- network geometry
constexpr int NET_C = 128;        // DN_FILTERS          dual_network.py:12
constexpr int NET_BLOCKS = 16;    // DN_RESIDUAL_NUM     dual_network.py:13
constexpr int NET_LAYERS = 2 * NET_BLOCKS;
constexpr int NET_CELLS = 81;
constexpr int NET_ACTIONS = 81;   // DN_OUTPUT_SIZE      dual_network.py:15

// ---------------------------------------------------------------- tree storage
constexpr int PATH_CAP = 96;      // root + at most 81 plies

enum : int32_t { PHASE_DONE = 0, PHASE_SEARCH = 1, PHASE_PENDING = 2, PHASE_ROOT = 3, PHASE_ROOT_PENDING = 4 };
constexpr int TP_MAX_LEAVES = 16;   // throughput mode: leaves per tree per round
enum : int32_t { MODE_SEARCH = 0, MODE_SELFPLAY = 1 };

struct alignas(16) TreeCtl {
    int32_t phase;
    int32_t sims_left;
    int32_t n_nodes;
    int32_t path_len;
    int32_t pend_k;
    int32_t nn_row;
    int32_t n_root;
    int32_t ply;
    uint64_t game;      // absolute game id (self-play)
    int32_t game_idx;   // index into the history buffers
    int32_t n_eval;     // evaluations queued by the current move's search (keys UTTT_SP_RANDOM_SYMMETRY's draw)
};

struct TreeParams {
    int32_t n_trees, node_cap, sims, batch, mode, flags;
    int32_t slot0;            // global index of this lane's first slot (self-play: slot s starts with game game0 + s)
    int32_t max_terminal;     // terminal descents one tree may retire per round (the rest continues next round)
    PackedState* root;        // [n_trees]
    // per tree up to TP_MAX_LEAVES pending leaves (the reference-exact mode has one, leaf 0): position and node path
    PackedState* leaf_state;  // [n_trees][TP_MAX_LEAVES]
    int32_t* paths;           // [n_trees][TP_MAX_LEAVES][PATH_CAP]
    int32_t* tp_aux;          // [n_trees][2][TP_MAX_LEAVES]: throughput mode's path lengths, evaluator rows
    float dir_alpha, dir_eps; // Dirichlet root noise
    float temperature;        // self-play move sampling (SP_TEMPERATURE, self_play_cpp.py:27); 1 = the reference's setting
    TreeCtl* ctl;             // [n_trees]
    // nodes, [n_trees][node_cap], 16 B each: {n:16 | action<<16, w, p, first_child:20 | n_children<<20}
    uint4* nodes;
    // evaluator queue (rows are compacted with an atomic counter, double-buffered by round parity)
    PackedState* nn_states;   // [rows]
    __nv_bfloat16* nn_planes; // [rows][3*81]
    int32_t* nn_tree;         // [rows]
    int32_t* nn_k;            // [rows]
    int32_t* nn_count;        // [2]
    int32_t parity;
    const float* policy;      // [(row*row_stride + copy*copy_stride)][81]
    const float* value;
    int32_t row_stride, copy_stride;
    // UTTT_SP_MATCH: the queue of weight slot 1 (same layout as the one above, which is slot 0's), for the leaves of the
    // moves that slot 1's network plays; nn1_count is always valid (the tree kernels reset it), the rest only in a match
    PackedState* nn1_states;
    __nv_bfloat16* nn1_planes;
    int32_t* nn1_tree;
    int32_t* nn1_k;
    int32_t* nn1_count;       // [2]
    const float* policy1;
    const float* value1;
    // search outputs
    int32_t* out_counts;      // [n_trees][81]
    int32_t* out_n;           // [n_trees]
    // self-play
    uint32_t seed;
    uint64_t game0;
    int64_t n_games;
    unsigned long long* counters;  // [0] next game, [1] finished games, [2] plies, [3] sims, [4] evals, [5] overflow flag
    PackedState* hist_states;      // [n_games][81]
    uint16_t* hist_counts;         // [n_games][81][81]
    uint8_t* hist_actions;         // [n_games][81]
    int32_t* hist_len;             // [n_games]
    int8_t* hist_final;            // [n_games]
    float* hist_value;             // [n_games][81]: the mover's root value of every decided move
    int8_t* hist_resigned;         // [n_games]
    float resign_threshold;        // UTTT_SP_RESIGN (uttt_set_resign)
    float resign_check_fraction;
};

// kernels' host launchers (each returns cudaGetLastError of the launch)
cudaError_t launch_tree_begin(const TreeParams& p, cudaStream_t s);
cudaError_t launch_tree_round(const TreeParams& p, cudaStream_t s);
cudaError_t launch_tree_tp_round(const TreeParams& p, cudaStream_t s);
cudaError_t launch_hash_eval(const PackedState* states, const int32_t* count, int max_rows, float* policy, float* value,
                             cudaStream_t s);
cudaError_t launch_scores(const int32_t* counts, const int32_t* n, int n_trees, float temperature,
                          float* scores, cudaStream_t s);
cudaError_t launch_dirichlet(uint32_t seed, uint64_t game0, int64_t n, int n_children, float alpha, float* out, cudaStream_t s);
cudaError_t launch_boltzman(const float* xs, int n, float temperature, float* out, cudaStream_t s);

// history as fixed-size samples (history_kernels.cu)
cudaError_t launch_scan_lens(const int32_t* lens, int64_t n, int64_t* offsets, cudaStream_t s);
cudaError_t launch_pack_samples(const PackedState* states, const uint16_t* counts, const int32_t* lens, const int8_t* final_lose,
                                const int64_t* offsets, int64_t n_games, void* out, int64_t cap_samples, cudaStream_t s);
cudaError_t launch_unpack_samples(const void* samples, int64_t n, float* x, float* policy, float* value, cudaStream_t s);

// ---------------------------------------------------------------- network
struct NetWeights {
    // every array is a region of `block`, one allocation per engine laid out and filled by weights.cu
    // fp32 path: folded BN (scale into the weights, shift separate); layout [layer][tap][cin][cout]
    float* conv_in_w;     // [9][3][128]
    float* conv_in_b;     // [128]
    float* res_w;         // [32][9][128][128]
    float* res_b;         // [32][128]
    // bf16 tensor-core path: the B operand of one K=16 MMA is a block [2 k-panels][cout 128][8] (UMMA canonical K-major,
    // no swizzle): 72 per residual layer in the order of tcx::kblock_of, conv_input as a K=16-per-tap layer (one block
    // per tap, channels 3..15 zero), and per layer (conv_input's and the 32 trunk layers') the BN shift as one block
    // (hi, lo in k = 0, 1).  The MMAs are cta_group::2: every block is split by output channel between the two CTAs of a
    // pair, and a CTA's share of a weight stage is contiguous: [stage][cta rank 2][blocks][2 k-panels][64 co][8]
    __nv_bfloat16* res_w_2sm;        // [32*9 stages][2][8 blocks]...
    __nv_bfloat16* conv_in_w_2sm;    // [2 stages][2][8 taps]... (16 tap slots, 9 used)
    __nv_bfloat16* bias_blk_2sm;     // [33][2][1 block]...
    // the 7-positions-per-pair instantiation (the 500-game cycle's batches) streams a quarter of a layer per stage
    __nv_bfloat16* res_w_2sm18;      // [32*4 stages][2][18 blocks]...
    __nv_bfloat16* conv_in_w_2sm18;  // [1 stage][2][18 tap slots (9 used)]...
    // split-bf16 ("bf16x3"), what trunk_x3_kernel (cta_group::2 MMAs) streams: per-CTA halves in stages of 6 K-blocks,
    // every block followed by its lo part, lo = bf16(w - hi)
    __nv_bfloat16* res_w_x3p;        // [32*12 stages][2 ranks][6 blocks][hi, lo][2 k-panels][64][8]
    __nv_bfloat16* conv_in_w_x3p;    // [2 stages][2 ranks][6 tap slots (9 of 12 used)][hi, lo][2][64][8]
    __nv_bfloat16* bias_blk_x3p;     // [33][2 ranks][2][64][8]: shift as three bf16 terms in k = 0, 1, 2
    // heads (fp32)
    float* head_w;          // [3][128] policy conv (2 rows) + value conv, BN scale folded; [384..386] BN shifts
    float* pol_fc_w;        // [162 in][81 out] + pol_fc_b [81]
    float* pol_fc_b;
    float* val_fc1_w;       // [81 in][256 out] + val_fc1_b [256]; val_fc2_w [256] + val_fc2_b [1]
    float* val_fc1_b; float* val_fc2_w; float* val_fc2_b;
    float* heads_pack;      // policy_fc / value_fc1 weights in the chunk order of heads_fc.cuh (bulk-copied to shared memory)
    float* raw_res;         // staging of an upload: the caller's residual convolutions and BN vectors as they are
    float* raw_res_bn;
    uint8_t* block;         // null before the first upload
    bool loaded;
};

// weights.cu: fold and pack a checkpoint into w on stream s (the device is set, nothing else uses w meanwhile; returns when
// done).  res_tab / res_bn_tab (optional): the 32 residual convolutions and their 32 x 4 BatchNorm vectors as separate
// tensors, each in host or device memory.  release_weights frees the allocation.
int upload_weights(NetWeights& w, const uttt_weights* src, int on_device, const float* const* res_tab,
                   const float* const (*res_bn_tab)[4], cudaStream_t s);
void release_weights(NetWeights& w);

// dynamic shared-memory limits of the network kernels, one function per file (net_fp32.cu, net_tc2.cu, net_pp.cu,
// net_auto.cu); they act on the current device, so uttt_create calls them for every engine
cudaError_t net_fp32_init();
cudaError_t trunk_tc2_init();
cudaError_t trunk_pp_init();
cudaError_t trunk_auto_init();
// trunk input: bf16 planes [rows][3][81]; output: final trunk activations [rows][81][128] (fp32 or bf16)
cudaError_t launch_conv_input(const NetWeights& w, const __nv_bfloat16* planes, const int32_t* count, int max_rows,
                              float* out, cudaStream_t s);
cudaError_t launch_trunk_fp32(const NetWeights& w, const __nv_bfloat16* planes, const int32_t* count, int max_rows,
                              float* act_a, float* act_b, cudaStream_t s);
// planes: network input [rows][3][81] bf16; headfeat: [rows][243] output of the heads' 1x1 convs (computed in the
// trunk's last epilogue); resid: per-CTA fp16 skip panels
cudaError_t launch_heads_fc(const NetWeights& w, const float* headfeat, const int32_t* count, int max_rows, float* policy,
                            float* value, int row_stride, cudaStream_t s);
cudaError_t launch_heads(const NetWeights& w, const float* act_f32, const __nv_bfloat16* act_bf16,
                         const int32_t* count, int max_rows, float* policy, float* value, int row_stride,
                         cudaStream_t s);
// split-bf16 numerics (UTTT_EVAL_NET_BF16X3, net_tc2.cu): any batch size in one launch; skip: [n_sm][16][256] fp32x8
cudaError_t launch_trunk_x3(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count,
                            int max_rows, float* skip, int n_sm, cudaStream_t s, long long* dbg);
// two groups of positions per CTA pair in flight (net_pp.cu): batches of more than trunk_pp_cap1 positions
int trunk_pp_cap1(int n_sm);         // largest batch of trunk_auto_kernel (7 positions per CTA pair)
cudaError_t launch_trunk_pp_large(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count,
                                  int max_rows, float* skip, int n_sm, cudaStream_t s, long long* dbg);
// one launch for every batch up to trunk_pp_cap1: device-side choice between the bodies of net_tc2_kernel.cuh and net_pp_kernel.cuh
// (policy / value non-null: the heads' FC layers run in the kernel's tail; requires max_rows <= trunk_pp_cap1)
cudaError_t launch_trunk_auto(const NetWeights& w, const __nv_bfloat16* planes, float* headfeat, const int32_t* count, int max_rows,
                              float* skip, int n_sm, cudaStream_t s, long long* dbg, float* policy, float* value);

}  // namespace uttt
