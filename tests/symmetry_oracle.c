/*
 * symmetry_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * Independent restatement of UTTT_SP_RANDOM_SYMMETRY (include/uttt_b200.h) on the oracle's [9][9] arrays, linked
 * against oracle/uttt_oracle.c (which it leaves as it is):
 *   - orc_symmetry / orc_symmetry_action compute the image of a position and of an action from picture coordinates
 *     (transpose if g >= 4, then numpy.rot90 by g % 4 of the 9x9 picture), not from bitboards;
 *   - the *_sym searches are the oracle's hash-evaluator searches in which a leaf's evaluation is
 *     hash_eval(g(leaf)) read back through sigma_g, with g = philox4x32(key=(seed, 2), ctr=(game, ply, j)).x >> 29 and
 *     j the evaluation's index within the move's search (a flush of k copies of a leaf is one evaluation).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "../oracle/uttt_oracle.h"

/* defined in oracle/uttt_oracle.c (pv_mcts.py:74-180 with a caller-side evaluator) */
int orc_py_mcts_counts(orc_eval_fn eval, void *ctx, const orc_state *root_state, int evaluate_count, int batch_size,
                       int *counts_out);

/* (R, C) of the 9x9 picture -> its image: transpose if g >= 4, then rot90 (counter-clockwise) g % 4 times; a rot90 of an
 * n x n picture moves (R, C) to (n-1-C, R) */
static void sym_rc(int g, int n, int *R, int *C) {
    int r = *R, c = *C;
    if (g >= 4) { int t = r; r = c; c = t; }
    for (int k = 0; k < g % 4; k++) { int t = r; r = n - 1 - c; c = t; }
    *R = r; *C = c;
}

int orc_symmetry_action(int a, int g) {
    int b = a / 9, c = a % 9;
    int R = 3 * (b / 3) + c / 3, C = 3 * (b % 3) + c % 3;
    sym_rc(g, 9, &R, &C);
    return (3 * (R / 3) + C / 3) * 9 + 3 * (R % 3) + C % 3;
}

static int sym_board(int b, int g) {
    int R = b / 3, C = b % 3;
    sym_rc(g, 3, &R, &C);
    return 3 * R + C;
}

void orc_symmetry(const orc_state *s, int g, orc_state *out) {
    memset(out, 0, sizeof(*out));
    for (int a = 0; a < 81; a++) {
        int na = orc_symmetry_action(a, g);
        out->pieces[na / 9][na % 9] = s->pieces[a / 9][a % 9];
        out->enemy[na / 9][na % 9] = s->enemy[a / 9][a % 9];
    }
    for (int b = 0; b < 9; b++) {
        out->main_pieces[sym_board(b, g)] = s->main_pieces[b];
        out->main_enemy[sym_board(b, g)] = s->main_enemy[b];
    }
    out->active = s->active < 0 ? -1 : sym_board(s->active, g);
}

int orc_symmetry_draw(uint32_t seed, uint64_t game, uint32_t ply, uint32_t j) {
    uint32_t r[4];
    orc_philox4x32(seed, 2u, (uint32_t)game, (uint32_t)(game >> 32), ply, j, r);
    return (int)(r[0] >> 29);
}

/* hash evaluation of the position's image, row entry a = the image's entry sigma_g(a) */
typedef struct { uint32_t seed; uint64_t game; uint32_t ply, j; } sym_ctx;

static void sym_eval(sym_ctx *x, const orc_state *s, float *pol, float *val) {
    int g = orc_symmetry_draw(x->seed, x->game, x->ply, x->j);
    orc_state gs;
    float gp[81];
    orc_symmetry(s, g, &gs);
    orc_hash_eval(&gs, gp, val);
    for (int a = 0; a < 81; a++) pol[a] = gp[orc_symmetry_action(a, g)];
}

static void sym_eval_cb(void *ctx, const orc_state *st, int n, float *pol, float *val) {
    sym_ctx *x = (sym_ctx *)ctx;
    for (int i = 0; i < n; i++) sym_eval(x, &st[i], pol + 81 * i, val + i);
    x->j++;                                       /* one flush = one evaluation */
}

/* the C++ search (cpp/uttt_mcts.cpp:84-196) */
int orc_pv_mcts_scores_hash_sym(const orc_state *root, uint32_t seed, uint64_t game, uint32_t ply, float temperature,
                                int evaluate_count, int batch_size, float *scores_out, int *counts_out) {
    sym_ctx x = {seed, game, ply, 0};
    return orc_pv_mcts_scores(sym_eval_cb, &x, root, temperature, evaluate_count, batch_size, scores_out, counts_out, NULL);
}

/* the pure-Python search (pv_mcts.py:74-180): the root is evaluation 0 */
int orc_py_mcts_counts_hash_sym(const orc_state *root, uint32_t seed, uint64_t game, uint32_t ply, int evaluate_count,
                                int batch_size, int *counts_out) {
    sym_ctx x = {seed, game, ply, 0};
    return orc_py_mcts_counts(sym_eval_cb, &x, root, evaluate_count, batch_size, counts_out);
}

/* orc_selfplay_hash with the C++ search above, keyed by (seed, game, ply) */
int orc_selfplay_hash_sym(uint32_t seed, uint64_t game, int sims, int batch, uint32_t *states, uint16_t *counts,
                          uint8_t *actions) {
    orc_state s;
    orc_init(&s);
    int t = 0;
    while (!orc_is_done(&s)) {
        int legal[81], cnt[81];
        float scores[81];
        int nl = orc_legal_actions(&s, legal);
        orc_pv_mcts_scores_hash_sym(&s, seed, game, (uint32_t)t, 1.0f, sims, batch, scores, cnt);
        int total = 0;
        for (int i = 0; i < nl; i++) total += cnt[i];
        uint32_t r[4];
        orc_philox4x32(seed, 1u, (uint32_t)game, (uint32_t)(game >> 32), (uint32_t)t, 0u, r);
        uint32_t pick = (uint32_t)(((uint64_t)r[0] * (uint64_t)total) >> 32);
        int idx = 0, acc = 0;
        for (int i = 0; i < nl; i++) {
            acc += cnt[i];
            if ((uint32_t)acc > pick) { idx = i; break; }
        }
        orc_pack(&s, states + 8 * t);
        for (int a = 0; a < 81; a++) counts[81 * t + a] = 0;
        for (int i = 0; i < nl; i++) counts[81 * t + legal[i]] = (uint16_t)cnt[i];
        actions[t] = (uint8_t)legal[idx];
        orc_state nx;
        orc_next(&s, legal[idx], &nx);
        s = nx;
        t++;
    }
    return t;
}

/* orc_az_search_hash (the throughput mode with one leaf per round and no root noise) restated with the symmetric
 * evaluation: the root is evaluation 0, leaves follow in the order they are reached */
typedef struct az_node {
    orc_state state;
    float p, w;
    int n, n_child;
    struct az_node *child;
} az_node;

static void az_free(az_node *nd) {
    for (int i = 0; i < nd->n_child; i++) az_free(&nd->child[i]);
    free(nd->child);
}

/* evaluates and expands nd; returns the value of the evaluation */
static float az_expand(az_node *nd, sym_ctx *x) {
    float pol[81], v;
    sym_eval(x, &nd->state, pol, &v);
    x->j++;
    int legal[81];
    int nl = orc_legal_actions(&nd->state, legal);
    float sum = 0.0f;
    for (int k = 0; k < nl; k++) sum += pol[legal[k]];
    nd->child = (az_node *)calloc((size_t)(nl > 0 ? nl : 1), sizeof(az_node));
    nd->n_child = nl;
    for (int k = 0; k < nl; k++) {
        orc_next(&nd->state, legal[k], &nd->child[k].state);
        nd->child[k].p = (sum > 0) ? pol[legal[k]] / sum : 1.0f / (float)nl;
    }
    return v;
}

/* PUCT with C = 1, first maximum wins (cpp/uttt_mcts.cpp:57-81) */
static az_node *az_select(az_node *nd) {
    int total = 0;
    for (int i = 0; i < nd->n_child; i++) total += nd->child[i].n;
    float sq = sqrtf((float)total), best = -1e9f;
    az_node *b = NULL;
    for (int i = 0; i < nd->n_child; i++) {
        az_node *c = &nd->child[i];
        float q = (c->n > 0) ? (-c->w / (float)c->n) : 0.0f;
        float s = q + c->p * sq / (float)(1 + c->n);
        if (s > best) { best = s; b = c; }
    }
    return b;
}

int orc_az_search_hash_sym(const orc_state *root_state, uint64_t game, int sims, int *counts_out) {
    int tmp[81];
    if (orc_is_lose(root_state) || orc_legal_actions(root_state, tmp) == 0) return 0;
    sym_ctx x = {0u, game, 0u, 0u};
    az_node root;
    memset(&root, 0, sizeof(root));
    root.state = *root_state;
    az_expand(&root, &x);                          /* evaluated root; its value is not backed up */
    for (int i = 0; i < sims; i++) {
        az_node *path[128];
        int plen = 0;
        az_node *nd = &root;
        float v;
        for (;;) {
            path[plen++] = nd;
            if (orc_is_done(&nd->state)) { v = orc_is_lose(&nd->state) ? -1.0f : 0.0f; break; }
            if (nd->n_child == 0) { v = az_expand(nd, &x); break; }
            nd = az_select(nd);
        }
        for (int k = plen - 1; k >= 0; k--) {      /* cpp/uttt_mcts.cpp:47-54 */
            path[k]->w += v;
            path[k]->n += 1;
            v = -v;
        }
    }
    for (int k = 0; k < root.n_child; k++) counts_out[k] = root.child[k].n;
    int n = root.n_child;
    az_free(&root);
    return n;
}
