/*
 * uttt_b200.h -- C ABI of libuttt_b200.so, the B200 (sm_100a) self-play engine for
 * Ultimate Tic-Tac-Toe.  This is the drop-in boundary: every entry point replaces a
 * piece of the reference's pybind11 module `uttt_cpp` (cpp/python_bindings.cpp:49-107)
 * or of the Python glue that drives it (pv_mcts_cpp.py, self_play_cpp.py).
 * Citations are <file>:<line> in the reference repository.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; uttt_last_error()
 *     returns a message for the calling thread's last failure.
 *   - "packed state" = 8 x uint32 (32 B), see csrc/uttt_rules.cuh:
 *       w0..w2 mover stones, w3..w5 opponent stones (3 sub-boards/word, 9 bits each),
 *       w6 = main_board_pieces | main_board_enemy_pieces<<9 | (active_board+1)<<18, w7 = 0.
 *   - "legal mask" = 4 x uint32 per state: words 0..2 hold 27 action bits each
 *     (action id = 27*word + bit = 9*board + cell), word 3 = number of legal moves.
 *   - *_dev pointers are CUDA device pointers owned by the caller (e.g. torch tensors);
 *     `stream` is a cudaStream_t (NULL = default stream); device calls are asynchronous
 *     on that stream unless stated otherwise.
 *   - there is no CPU fallback: device entry points fail if no sm_100 GPU is present.
 */
#ifndef UTTT_B200_H
#define UTTT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UTTT_ABI_VERSION 1

/* evaluators for search / self-play */
#define UTTT_EVAL_NET_BF16 0 /* DualNetwork forward, tcgen05 bf16 implicit-GEMM trunk          */
#define UTTT_EVAL_NET_FP32 1 /* DualNetwork forward, fp32 CUDA-core trunk ("parity" numerics)  */
#define UTTT_EVAL_HASH     2 /* deterministic integer-hash evaluator (search parity oracle mode) */
#define UTTT_EVAL_HOST     3 /* caller evaluates leaves (uttt_mcts_get_leaves/put_results)     */
#define UTTT_EVAL_NET_BF16X3 4 /* DualNetwork forward, tcgen05 trunk with split-bf16 operands (hi*hi + lo*hi + hi*lo,
                                  fp32 accumulation and skip connection): within 1e-2 of the fp32 reference forward
                                  (dual_network.py:89-121) on random-init weights, 3x the MMAs of _BF16 */

/* self-play flags */
#define UTTT_SP_CORRECT_TERMINAL_SIGN 1 /* opt out of the reference's inverted terminal sign (cpp/uttt_mcts.cpp:19-21) */
#define UTTT_SP_THROUGHPUT 2            /* standard AlphaZero search instead of the reference-exact one: evaluated root
                                           with Dirichlet noise, virtual loss, `batch_size` = leaves per tree per round
                                           (<= 16), single expansion per leaf, correct terminal sign (not in the reference) */

#define UTTT_SP_PYSEARCH 4              /* uttt_mcts_search, and uttt_selfplay_run* together with UTTT_SP_MATCH: the
                                           semantics of the reference's pure-Python search (pv_mcts.py:74-180, used by its
                                           gating match evaluate_network.py:73-75) instead of the C++ one's: the root is
                                           evaluated like any leaf, a flush's k expansions of a leaf replace each other (one
                                           child list), priors are normalised with numpy's float32 pairwise sum.  Excludes
                                           UTTT_SP_THROUGHPUT. */
#define UTTT_SP_RANDOM_SYMMETRY 8       /* uttt_mcts_search and uttt_selfplay_run*, any search mode and device evaluator:
                                           every leaf is evaluated under a board symmetry g drawn at random (AlphaGo Zero's
                                           evaluation-time augmentation) and the policy is mapped back.  Symmetry
                                           g = 4f + r (0..7) of the 9x9 picture (R, C) of uttt_state_encode (action
                                           9b + c at R = 3(b/3) + c/3, C = 3(b%3) + c%3): transpose (R,C) -> (C,R) if f,
                                           then numpy.rot90(picture, k=r); stones, main-board flags and the forced board
                                           move with it (see uttt_state_symmetry).  The evaluator sees g(leaf); the prior
                                           of legal action a is read from row entry sigma_g(a), everything else is
                                           unchanged.  g = philox4x32(key=(seed, 2), ctr=(game_lo, game_hi, ply, j)).x >> 29
                                           with j = 0, 1, ... the evaluations of that move's search in the order its tree
                                           queues them (reference-exact and _PYSEARCH: a leaf's k queued copies are one
                                           evaluation; _THROUGHPUT: the root is j = 0).  uttt_mcts_search keys it with
                                           seed 0, game = root index in the call, ply 0.  g depends on neither slot nor
                                           batch position, so runs stay reproducible. */
#define UTTT_SP_MATCH 16                /* uttt_selfplay_run* only: a match between the networks of weight slots 0 and 1
                                           (uttt_upload_weights_slot).  Colour rule: in game g (the absolute id, game0 +
                                           index) the position at ply p is searched with the network of slot (g + p) & 1,
                                           i.e. slot 0 moves first in even games and slot 1 in odd ones (the reference's
                                           evaluate_network.py:80-85); the rule keys on g, so a match split over calls by
                                           game0 is the same match.  Everything else is self-play as without the flag
                                           (search flags, temperature, Philox move draw, history).  The history is the
                                           result: the point of slot 0 in game g is 0.5 if hist_final[g] == 0 (a draw),
                                           else 1 if the last mover, slot (g + hist_len[g] - 1) & 1, is slot 0 and 0 if
                                           not.  Fails if a network evaluator is asked for and slot 1 was never uploaded
                                           (the hash evaluator reads no weights). */
#define UTTT_SP_RESIGN 32               /* uttt_selfplay_run* only, alone or with UTTT_SP_MATCH: resignation (AlphaGo Zero).
                                           Every decided move records v, its mover's root value: -w/n of the root child
                                           with the most visits (the first maximum in legal order), 0 if that child is
                                           unvisited -- with or without the flag (uttt_selfplay_fetch_values).  Game g
                                           (absolute id) is a check game iff u < check_fraction, u = (philox4x32(
                                           key=(seed, 4), ctr=(g_lo, g_hi, 0, 0)).x >> 8) * 2^-24; a check game is never
                                           resigned.  In any other game the mover at ply p >= 1 resigns when v < threshold
                                           (uttt_set_resign): v goes to hist_value row p, rows p of hist_states / _counts
                                           / _actions are not written, hist_len = p, hist_final = 1 (the final position is
                                           lost for its mover, the resigner), hist_resigned = 1, and the slot goes on to
                                           the next game as after a natural end.  A resigned game is therefore the first
                                           p plies of the same game played out, and its labels, packed samples and match
                                           points give the resigner's opponent the win.  Needs terminal values of the
                                           correct sign: UTTT_SP_THROUGHPUT or UTTT_SP_CORRECT_TERMINAL_SIGN. */
#define UTTT_SP_PLAYOUT_CAP 64          /* uttt_selfplay_run* only, any search mode, alone or with UTTT_SP_RANDOM_SYMMETRY,
                                           UTTT_SP_RESIGN or UTTT_SP_CORRECT_TERMINAL_SIGN: playout cap randomization
                                           (KataGo, Wu 2019, section 3.1).  The move at ply p of game g (absolute id) is a
                                           full search iff u < full_fraction, u = (philox4x32(key=(seed, 5), ctr=(g_lo,
                                           g_hi, p, 0)).x >> 8) * 2^-24 compared in fp32; a full search spends
                                           evaluate_count simulations, a fast search fast_sims (uttt_set_playout_cap).  In
                                           the throughput mode a fast search mixes no Dirichlet noise into its root
                                           priors; a full search keeps it.  Everything else about a move is the same for
                                           both kinds: temperature and Philox move draw, symmetry draws, root value and the
                                           resignation rule, and rows of hist_states / _counts / _actions.  hist_full[g*81
                                           + p] (uttt_selfplay_fetch_full) is 1 for a full search and 0 for a fast one,
                                           written for every decided move that is not a resignation, and 1 for every move
                                           without the flag.  Only full-search plies become packed samples
                                           (uttt_selfplay_pack).  Fails with fast_sims > evaluate_count and with
                                           UTTT_SP_MATCH (a match records no training targets). */
#define UTTT_SP_FORCED_PLAYOUTS 128     /* uttt_selfplay_run* only, with UTTT_SP_THROUGHPUT, alone or with
                                           UTTT_SP_RANDOM_SYMMETRY, UTTT_SP_RESIGN or UTTT_SP_PLAYOUT_CAP: forced playouts
                                           and policy target pruning (KataGo, Wu 2019, section 3.2).  It applies to every
                                           full search of the run (every move without UTTT_SP_PLAYOUT_CAP, the full ones
                                           with it); a fast search neither forces nor prunes.  It does not depend on the
                                           root noise's eps.  k = forced_k (uttt_set_forced_playouts, default 2).  All
                                           arithmetic is IEEE fp32, correctly rounded, in the order written, without FMA.
                                           Forcing (the PUCT step at the root only): N = sum of (n + vl) over the root's
                                           children, virtual loss included; a root child with m = n + vl and stored prior
                                           p (the noised one where noise is mixed in) is forced iff m >= 1 and (float)m <
                                           F, F = sqrt((k * p) * (float)N); a forced child scores 1e20f, so the first
                                           maximum picks the forced child with the smallest index.  Pruning (when the move
                                           is decided; no virtual loss is outstanding): N = sum of n, sq = sqrt((float)N),
                                           c* = the first child with the most visits, S* = q* + (p* * sq) / (float)(1 +
                                           n*) with q* = -w* / n*.  Every other child c with n >= 1: q = -w / n, F as
                                           above with this N, R = min(n, (int)F); r is the largest value in [0, R] with
                                           score(n - j) < S* for every j in 1..r, score(m) = q + (p * sq) / (float)(1 +
                                           m); the child's target is t = n - r, and 0 if r >= 1 and n - r == 1 (a child
                                           reduced to a single playout is pruned outright).  c* keeps t = n*, an
                                           unvisited child 0.  hist_counts keeps the raw visit counts; hist_target[g*81 +
                                           p][a] (uttt_selfplay_fetch_target) holds t, and equals the counts on a fast
                                           ply.  The move is drawn from t (the same Philox draw, temperature rule and
                                           legal order as from the counts; T = 0 still plays c*); the root value and
                                           resignation use the raw (n, w) of c*, which pruning never changes.  Packed
                                           samples carry t as their policy counts.  Fails without UTTT_SP_THROUGHPUT (the
                                           reference-exact root is uniform and never noised) and with UTTT_SP_MATCH (a
                                           match records no training targets). */

typedef struct uttt_engine uttt_engine;

const char *uttt_last_error(void);
int uttt_abi_version(void);
/* 0 iff `device` exists and is compute capability 10.x */
int uttt_device_check(int device);

/* ------------------------------------------------------------------------------------------
 * Single-state helpers (host arithmetic on ONE packed state; back the `uttt_cpp.State`
 * object of the Python shim -- cpp/python_bindings.cpp:54-74).  Not a device fallback:
 * every batch / search / self-play entry point below runs on the GPU only.
 * ---------------------------------------------------------------------------------------- */
int uttt_state_init(uint32_t *state);                                             /* cpp/uttt_game.cpp:9-19   */
int uttt_state_next(const uint32_t *state, int action, uint32_t *out);            /* cpp/uttt_game.cpp:97-145 */
int uttt_state_legal_actions(const uint32_t *state, int32_t *out81, int *n_out);  /* cpp/uttt_game.cpp:148-191 */
/* bit0 is_lose, bit1 is_draw, bit2 is_done, bit3 is_first_player (cpp/uttt_game.cpp:77-94) */
int uttt_state_flags(const uint32_t *state, int *flags_out);
int uttt_state_encode(const uint32_t *state, float *out243);                      /* cpp/uttt_game.cpp:244-280 */
int uttt_state_to_string(const uint32_t *state, char *buf, int cap, int *len_out);/* cpp/uttt_game.cpp:194-241 */
/* out = the image of the position under board symmetry g (0..7, numbering of UTTT_SP_RANDOM_SYMMETRY);
 * action_map81 (may be NULL): [a] = sigma_g(a), the action at the image of action a's cell */
int uttt_state_symmetry(const uint32_t *state, int g, uint32_t *out, int32_t *action_map81);

/* ------------------------------------------------------------------------------------------
 * Rules kernels over arrays of packed states in HBM (replace UTTT::State, cpp/uttt_game.cpp)
 * ---------------------------------------------------------------------------------------- */
/* out[i] = next(states[i], actions[i])                      cpp/uttt_game.cpp:97-145 */
int uttt_game_step(const uint32_t *states_dev, const int32_t *actions_dev, uint32_t *out_dev,
                   int64_t n, void *stream);
/* masks[i] = legal mask (4 words), status[i] = 0 ongoing / 1 lose / 2 draw
 *                                                            cpp/uttt_game.cpp:77-89,148-191 */
int uttt_game_legal_mask(const uint32_t *states_dev, uint32_t *masks_dev, uint8_t *status_dev,
                         int64_t n, void *stream);
/* planes[i] = float[9*9*3] HWC exactly as State::to_input_tensor   cpp/uttt_game.cpp:244-280 */
int uttt_game_encode(const uint32_t *states_dev, float *planes_dev, int64_t n, void *stream);
/* leaf gather: planes[i] = bf16[3*9*9] CHW, the network's input batch
 *                                     (pv_mcts_cpp.py:47-60: reshape + stack + NHWC->NCHW) */
int uttt_game_gather_planes(const uint32_t *states_dev, void *planes_bf16_dev, int64_t n, void *stream);
/* n random playouts from the initial position, game ids game0..game0+n-1; action at ply t =
 * legal[ philox4x32(key=(seed,0), ctr=(game_lo,game_hi,t,0)).x % n_legal ]; outputs per game:
 * FNV-1a(64) digest over (action, legal mask, main flags/active) per ply + final state,
 * ply count, result (0 draw / 1 first player won / 2 second player won). */
int uttt_game_playout(uint32_t seed, uint64_t game0, int64_t n, uint64_t *digests_dev,
                      int32_t *plies_dev, int32_t *results_dev, void *stream);

/* ------------------------------------------------------------------------------------------
 * Engine: trees, network weights, self-play slots -- all resident in HBM
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t device;        /* CUDA device ordinal */
    int32_t n_slots;       /* concurrent trees / games */
    int32_t max_sims;      /* largest evaluate_count that will be requested */
    int32_t max_batch;     /* largest batch_size that will be requested */
    int64_t max_games;     /* capacity of the self-play history buffers (games per run) */
} uttt_config;

int uttt_create(const uttt_config *cfg, uttt_engine **out);
int uttt_destroy(uttt_engine *e);

/* DualNetwork parameters (dual_network.py:47-75), fp32, PyTorch layouts, eval-mode BatchNorm.
 * All pointers are device pointers if on_device != 0, else host pointers.
 * bn arrays are [4][C]: weight, bias, running_mean, running_var (eps = 1e-5).            */
typedef struct {
    const float *conv_input_w;   /* (128,3,3,3)      */
    const float *bn_input;       /* [4][128]         */
    const float *res_conv_w;     /* (16,2,128,128,3,3): block, conv1/conv2, out, in, ky, kx */
    const float *res_bn;         /* (16,2,4,128)     */
    const float *policy_conv_w;  /* (2,128)          */
    const float *policy_bn;      /* [4][2]           */
    const float *policy_fc_w;    /* (81,162)         */
    const float *policy_fc_b;    /* (81)             */
    const float *value_conv_w;   /* (1,128)          */
    const float *value_bn;       /* [4][1]           */
    const float *value_fc1_w;    /* (256,81)         */
    const float *value_fc1_b;    /* (256)            */
    const float *value_fc2_w;    /* (1,256)          */
    const float *value_fc2_b;    /* (1)              */
} uttt_weights;

/* folds BatchNorm, repacks to the tensor-core layouts; synchronous */
int uttt_upload_weights(uttt_engine *e, const uttt_weights *w, int on_device);

/* The same upload straight from a state_dict (torch.load('./model/best.pth'), self_play_cpp.py:110-112): the 32
 * residual convolutions `residual_blocks.{b}.conv{1,2}.weight` (index 2*b + j, each (128,128,3,3)) and their
 * BatchNorm vectors `residual_blocks.{b}.bn{1,2}.{weight,bias,running_mean,running_var}` (128 each) are read from
 * the caller's 160 tensors where they lie (pinned host memory -> one DMA each, no host-side concatenation);
 * `small` holds the remaining 12 arrays as in uttt_weights (its res_conv_w / res_bn are ignored); `on_device` describes
 * `small` only: each of the 160 tensors may lie in host or device memory (copied with cudaMemcpyDefault).            */
typedef struct {
    uttt_weights small;
    const float *res_conv_w[32];
    const float *res_bn[32][4];
} uttt_weights_scattered;
int uttt_upload_weights_scattered(uttt_engine *e, const uttt_weights_scattered *w, int on_device);

/* Weight slots: slot 0 is what uttt_upload_weights / _scattered write and what every evaluator reads; slot 1 is a second
 * network, read only by the moves UTTT_SP_MATCH gives it.  slot must be 0 or 1.  The first upload to slot 1 allocates its
 * weights and a second evaluator queue (about 1.8 KB per evaluator row); uttt_destroy frees them. */
int uttt_upload_weights_slot(uttt_engine *e, int slot, const uttt_weights *w, int on_device);
int uttt_upload_weights_scattered_slot(uttt_engine *e, int slot, const uttt_weights_scattered *w, int on_device);

/* DualNetwork.forward on n packed states (dual_network.py:89-121 behind pv_mcts_cpp.py:37-78):
 * policy[n][81] (softmax over all 81 actions), value[n].  mode = UTTT_EVAL_NET_BF16 / _BF16X3 / _FP32. */
int uttt_net_forward(uttt_engine *e, const uint32_t *states_dev, int64_t n, int mode,
                     float *policy_dev, float *value_dev, void *stream);

/* ---- search: UTTT::pv_mcts_scores (cpp/uttt_mcts.cpp:84-196) over n_roots independent trees ----
 * Synchronous.  roots/scores/counts/n_scores are HOST pointers.
 * scores[i][0..n_scores[i]) follow legal_actions(root i) order; counts are the raw visit counts. */
int uttt_mcts_search(uttt_engine *e, const uint32_t *roots, int32_t n_roots, int32_t evaluate_count,
                     int32_t batch_size, float temperature, int32_t evaluator, int32_t flags,
                     float *scores /* n*81 */, int32_t *counts /* n*81 */, int32_t *n_scores /* n */);
/* Dirichlet root noise of the throughput mode: p = (1-eps) p + eps * Dir(alpha); defaults alpha 0.3, eps 0.25
 * (AlphaZero's settings; the reference has no noise).  eps = 0 disables it.  It is mixed into the evaluated root of every
 * full search (every move without UTTT_SP_PLAYOUT_CAP) as p' = fma(1 - eps, p, eps * eta) in IEEE fp32: 1 - eps and
 * eps * eta correctly rounded, then one fused multiply-add (one rounding); p is the root's renormalised prior, eta the draw
 * of uttt_debug_root_noise for the root position under key (seed, game, ply): uttt_selfplay_run* keys it with its seed,
 * the game and the ply, uttt_mcts_search with seed 0, game = root index in the call and ply 0 (like
 * UTTT_SP_RANDOM_SYMMETRY), so a search's result does not depend on what the engine ran before. */
int uttt_set_root_noise(uttt_engine *e, float alpha, float eps);

/* SP_TEMPERATURE of the self-play loop (self_play_cpp.py:27,62 -> cpp/uttt_mcts.cpp:183-216); default 1 (the reference's
 * setting: moves drawn in proportion to the visit counts).  0: the first maximum of the visit counts is played; otherwise
 * moves are drawn from n^(1/T) / sum.  The history always holds the raw visit counts. */
int uttt_set_selfplay_temperature(uttt_engine *e, float temperature);

/* diagnostics: the root-noise sampler alone -- out[g][0..n_children) = the Dirichlet(alpha) draw of game game0 + g at ply 0
 * for a root whose legal actions are 0 .. n_children - 1 (Philox key (seed, 3), counter (game, ply, child, attempt));
 * the draw the throughput mode mixes into a game's first root when n_children = 81 */
int uttt_debug_dirichlet(uint32_t seed, uint64_t game0, int64_t n, int32_t n_children, float alpha, float *out_dev,
                         void *stream);
/* diagnostics: the root noise the throughput mode mixes into the root priors of position states_dev[i] under key (seed,
 * games_dev[i], plies_dev[i]) -- eta_dev[i][a] (DEVICE pointers, n rows of 81): for each legal action id a a Gamma(alpha)
 * sample g_a (Marsaglia-Tsang on the Philox stream above), eta_a = g_a / sum of the g (summed in the device's fixed
 * order), or 1 / (number of legal actions) if that sum is not positive; 0 for an illegal action.  Exactly the draw of
 * uttt_set_root_noise, from the same device function. */
int uttt_debug_root_noise(uint32_t seed, float alpha, const uint32_t *states_dev, const uint64_t *games_dev,
                          const int32_t *plies_dev, int64_t n, float *eta_dev, void *stream);

/* step-wise form for a caller-side evaluator (python_bindings.cpp:11-47 `wrap_python_inference`) */
int uttt_mcts_begin(uttt_engine *e, const uint32_t *roots, int32_t n_roots, int32_t evaluate_count,
                    int32_t batch_size);
/* applies the results put since the last call, then descends every unfinished tree to its next
 * unevaluated leaf; *n_pending = number of leaves now waiting (0 => search finished) */
int uttt_mcts_advance(uttt_engine *e, int32_t *n_pending);
/* pending leaves: packed states, k = number of queued copies of that leaf (cpp/uttt_mcts.cpp:121-127), tree id */
int uttt_mcts_get_leaves(uttt_engine *e, uint32_t *states /* n_pending*8 */, int32_t *k /* n_pending */,
                         int32_t *tree /* n_pending */);
/* results for pending leaf i: per_copy==0 -> policy[i][81], value[i];
 * per_copy!=0 -> policy[i][max_batch][81], value[i][max_batch] (row c feeds queued copy c) */
int uttt_mcts_put_results(uttt_engine *e, const float *policy, const float *value, int per_copy);
int uttt_mcts_finish(uttt_engine *e, float temperature, float *scores, int32_t *counts, int32_t *n_scores);

/* cpp/uttt_mcts.cpp:199-216 on the device (fp32; bit-identical to the reference for T == 1) */
int uttt_boltzman(const float *xs, int32_t n, float temperature, float *out);

/* ---- self-play: self_play_cpp.py:34-130 for n_games games, all concurrent on the device ----
 * Game ids game0..game0+n_games-1.  Per ply of game g (row g*81 + ply):
 *   hist_states  packed state the move was chosen in                (self_play_cpp.py:56-59: x)
 *   hist_counts  root visit counts by action id, uint16[81]          (self_play_cpp.py:63-83: pi = counts/sum)
 *   hist_actions sampled action: pick = floor(philox(key=(seed,1),ctr=(g_lo,g_hi,ply,0)).x * sum / 2^32)
 *                over the counts in legal order                      (self_play_cpp.py:86)
 * hist_len[g] = plies, hist_final[g] = 1 if the final position is_lose (z0 = -1) else 0
 *                                                                    (self_play_cpp.py:95-99)
 * All hist_* pointers are HOST pointers (pinned memory recommended).  Synchronous.
 * stats (may be NULL): [0] plies, [1] simulations, [2] evaluated leaves, [3] tree rounds */
int uttt_selfplay_run(uttt_engine *e, int64_t n_games, uint64_t game0, int32_t evaluate_count,
                      int32_t batch_size, uint32_t seed, int32_t evaluator, int32_t flags,
                      uint32_t *hist_states, uint16_t *hist_counts, uint8_t *hist_actions,
                      int32_t *hist_len, int8_t *hist_final, int64_t *stats);

/* progress of a running uttt_selfplay_run*: `fn(finished games, n_games, user)` is called on the calling thread whenever the
 * host sees the count of finished games change (once per window of 8 rounds) -- what the reference prints per game
 * (self_play_cpp.py:121).  NULL removes it. */
typedef void (*uttt_progress_fn)(int64_t done, int64_t total, void *user);
int uttt_set_progress_callback(uttt_engine *e, uttt_progress_fn fn, void *user);

/* device-resident variant for benchmarking / multi-GPU pipelines: runs the same loop but leaves
 * the history in the engine's HBM buffers; uttt_selfplay_fetch copies it out afterwards. */
int uttt_selfplay_run_device(uttt_engine *e, int64_t n_games, uint64_t game0, int32_t evaluate_count,
                             int32_t batch_size, uint32_t seed, int32_t evaluator, int32_t flags,
                             int64_t *stats, void *stream);
int uttt_selfplay_fetch(uttt_engine *e, int64_t n_games, uint32_t *hist_states, uint16_t *hist_counts,
                        uint8_t *hist_actions, int32_t *hist_len, int8_t *hist_final);

/* UTTT_SP_RESIGN's threshold (a number in [-1, 1]; default -0.95) and the fraction of check games (in [0, 1]; default
 * 0.1).  Fails on a NaN or out-of-range value. */
int uttt_set_resign(uttt_engine *e, float threshold, float check_fraction);
/* the root values of the last uttt_selfplay_run*, like uttt_selfplay_fetch: hist_value[g*81 + ply] = v of every decided
 * move (rows 0..hist_len-1, and row hist_len of a resigned game; later rows are unspecified), hist_resigned[g] = 1 if
 * game g resigned.  HOST pointers, either may be NULL.  Synchronous. */
int uttt_selfplay_fetch_values(uttt_engine *e, int64_t n_games, float *hist_value /* n*81 */, int8_t *hist_resigned /* n */);

/* UTTT_SP_PLAYOUT_CAP's fast-search budget (1 <= fast_sims <= the engine's max_sims; default 8) and the probability of a
 * full search (in [0, 1]; default 0.25): KataGo's ratio at the reference's 50 simulations, and its p.  Fails on a NaN or
 * out-of-range value. */
int uttt_set_playout_cap(uttt_engine *e, int32_t fast_sims, float full_fraction);
/* the search kinds of the last uttt_selfplay_run*, like uttt_selfplay_fetch: hist_full[g*81 + ply] = 1 for a full search,
 * 0 for a fast one (rows 0..hist_len-1; later rows are unspecified).  HOST pointer.  Synchronous. */
int uttt_selfplay_fetch_full(uttt_engine *e, int64_t n_games, uint8_t *hist_full /* n*81 */);

/* UTTT_SP_FORCED_PLAYOUTS's k (finite, in (0, 100]; default 2, KataGo's).  Fails on any other value. */
int uttt_set_forced_playouts(uttt_engine *e, float k);
/* the policy target counts of the last uttt_selfplay_run*, like uttt_selfplay_fetch's hist_counts: hist_target[(g*81 +
 * ply)*81 + a] = t of UTTT_SP_FORCED_PLAYOUTS, or a copy of the visit counts if that run had no such flag.  HOST pointer.
 * Synchronous. */
int uttt_selfplay_fetch_target(uttt_engine *e, int64_t n_games, uint16_t *hist_target /* n*81*81 */);

/* The history of the last uttt_selfplay_run_device as ONE contiguous device buffer of fixed-size samples (one per played
 * ply with hist_full = 1, i.e. every played ply without UTTT_SP_PLAYOUT_CAP; game-major, ply order): bytes 0..31 packed
 * position, 32..193 policy target counts u16[81] (the visit counts without UTTT_SP_FORCED_PLAYOUTS), 194 z (int8, the label of
 * self_play_cpp.py:95-99), 195 ply.  This is what a rank sends to the trainer rank in the multi-GPU cycle (one
 * exact-length transfer instead of the ~1.7 KB/sample pickle of self_play_cpp.py:125-130).
 * uttt_selfplay_pack: out_dev must hold cap_samples samples; *n_samples_out (HOST) = samples written; synchronises `stream`.
 * uttt_samples_unpack (no engine needed): samples -> x (n,3,9,9) f32, policy (n,81) f32 = counts / sum, value (n) f32:
 * the arrays train_network.py:41-60 builds from the pickle (policy in fp32 instead of the pickle's float64). */
#define UTTT_SAMPLE_BYTES 196
int uttt_selfplay_pack(uttt_engine *e, int64_t n_games, void *out_dev, int64_t cap_samples, int64_t *n_samples_out,
                       void *stream);
int uttt_samples_unpack(const void *samples_dev, int64_t n, float *x_dev, float *policy_dev, float *value_dev,
                        void *stream);

/* timing of the engine's own kernels during the last uttt_selfplay_run*: CUDA-event ms on the
 * launching stream and launch counts; kind: 0 tree kernels, 1 trunk, 2 heads, 3 everything (ms: of the launches that were
 * bracketed by events, see uttt_set_profile_level; counts: of all launches); 4: the bracketed trunk launches (their ms,
 * their number), 5: the same ms and the number of positions those launches evaluated.  A match (UTTT_SP_MATCH) runs two
 * evaluator passes per round: both are counted and bracketed. */
int uttt_last_run_profile(uttt_engine *e, int kind, double *ms_out, int64_t *launches_out);

/* which of those kernels are bracketed by CUDA events during self-play (an event between two dependent kernels costs
 * about 1 us of GPU idle time): 0 none, 1 the trunk only, and only in
 * every 4th window of 8 rounds (default: what the roofline needs -- a uniform sample of the launches; UTTT_PROFILE_SAMPLE=1
 * brackets every launch), 2 tree / trunk / heads in every round (kind 0, 2, 3 of uttt_last_run_profile report 0 ms below
 * level 2).  Launch counts are always kept. */
int uttt_set_profile_level(uttt_engine *e, int level);

/* diagnostics: clock64 timeline of CTA 0 of the last tensor-core trunk launch, [32 layers][4]:
 * MMA start, MMA issue done, accumulators ready (epilogue start), epilogue done */
int uttt_debug_trunk_timeline(uttt_engine *e, int64_t *out128);

/* diagnostics: how many tensor-core trunk launches evaluated n positions, 64 buckets of 16 (bucket 63 = 1008 and
 * more), accumulated since creation or the last call with reset != 0 */
int uttt_debug_batch_histogram(uttt_engine *e, int64_t *out64, int32_t reset);

/* diagnostics: the device counters of the last search / self-play run: [2] plies, [3] simulations, [4] evaluated leaves,
 * [5] node-arena overflow flag, [6] finished trees (search), [1] finished games (self-play) */
int uttt_debug_counters(uttt_engine *e, uint64_t *out8);

/* diagnostics for the parity tests: while enabled, uttt_mcts_search and uttt_selfplay_run* (every search mode; a match
 * records the rows of both networks' evaluator passes) record every evaluated leaf with the evaluator rows its tree is
 * about to consume -- (tree, game index, ply, round), packed leaf state, policy[81], value -- in evaluation order (the
 * throughput mode: a move's root, then its leaves in the order they were queued); `round` numbers the rounds of the call
 * from 0.  The host synchronises after every round.  `enable` also clears the log.
 * uttt_debug_trace_read: *n_out = records; with cap >= *n_out the arrays meta[n][4], states[n][8], policy[n][81],
 * value[n] (HOST pointers) are filled; cap = 0 only asks for the size.  With UTTT_SP_RANDOM_SYMMETRY a record holds the
 * untransformed leaf and its row mapped back into the leaf's own action ids.  Feeding these rows to the reference's
 * UTTT::pv_mcts_scores (cpp/uttt_mcts.cpp:84-196) must reproduce the engine's scores bit for bit. */
int uttt_debug_trace(uttt_engine *e, int enable);
int uttt_debug_trace_read(uttt_engine *e, int64_t cap, int64_t *n_out, int32_t *meta, uint32_t *states,
                          float *policy, float *value);

#ifdef __cplusplus
}
#endif
#endif
