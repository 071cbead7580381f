/*
 * forced_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * UTTT_SP_FORCED_PLAYOUTS (include/uttt_b200.h) restated on the CPU.  This file compiles oracle/uttt_oracle.c into
 * itself (unchanged, so that its node type, PUCT arithmetic, expansion and backup are the very ones the existing checks
 * rest on) and adds:
 *   - orc_prune_targets: the policy target pruning of one root, from its children's (n, w, p) in legal order;
 *   - orc_az_search_forced_root_hash: orc_az_search_hash (the throughput mode with one leaf per round and no root
 *     noise, hash evaluator) with the forcing rule in its root PUCT step, returning the root children's raw (n, w) and
 *     their pruned targets in legal order.
 * Every float operation is a single correctly rounded fp32 operation in the header's order (-std=c11 turns FMA
 * contraction off).
 */
#include "../oracle/uttt_oracle.c"

void orc_prune_targets(int nc, const int *n, const float *w, const float *p, float k, int *t_out) {
    int tot = 0, cs = 0;
    for (int i = 0; i < nc; i++) {
        tot += n[i];
        if (n[i] > n[cs]) cs = i;                       /* c*: the first maximum */
        t_out[i] = n[i];
    }
    if (nc == 0 || n[cs] == 0) return;
    const float sq = sqrtf((float)tot);
    const float best = -w[cs] / (float)n[cs] + (p[cs] * sq) / (float)(1 + n[cs]);
    for (int i = 0; i < nc; i++) {
        if (i == cs || n[i] == 0) continue;
        const float q = -w[i] / (float)n[i], u = p[i] * sq;
        const int f = (int)sqrtf((k * p[i]) * (float)tot);
        const int cap = n[i] < f ? n[i] : f;
        int r = 0;
        while (r < cap && q + u / (float)(1 + n[i] - (r + 1)) < best) r++;
        t_out[i] = (r >= 1 && n[i] - r == 1) ? 0 : n[i] - r;
    }
}

/* next_child_node with the forcing rule: a child with n >= 1 and (float)n < sqrt((k * p) * (float)N) scores 1e20f */
static orc_node *next_child_node_forced(orc_node *nd, float k) {
    int total_n = 0;
    for (int i = 0; i < nd->n_child; i++) total_n += nd->child[i]->n;
    float sqrt_total = sqrtf((float)total_n);
    float max_pucb = -1e9f;
    orc_node *best = NULL;
    for (int i = 0; i < nd->n_child; i++) {
        orc_node *c = nd->child[i];
        float q = (c->n > 0) ? (-c->w / (float)c->n) : 0.0f;
        float u = c->p * sqrt_total / (float)(1 + c->n);
        float pucb = q + u;
        if (c->n >= 1 && (float)c->n < sqrtf((k * c->p) * (float)total_n)) pucb = 1e20f;
        if (pucb > max_pucb) { max_pucb = pucb; best = c; }
    }
    return best;
}

int orc_az_search_forced_root_hash(const orc_state *root_state, int sims, float k, int *n_out, float *w_out, int *t_out) {
    int tmp[81];
    if (orc_is_lose(root_state) || orc_legal_actions(root_state, tmp) == 0) return 0;
    float pol[81], val;
    orc_node *root = node_new(root_state, 0.0f);
    orc_hash_eval(root_state, pol, &val);
    az_expand(root, pol);
    for (int i = 0; i < sims; i++) {
        orc_node *path[ORC_MAX_PATH];
        int plen = 0;
        orc_node *nd = root;
        float v;
        for (;;) {
            path[plen++] = nd;
            if (orc_is_done(&nd->state)) { v = orc_is_lose(&nd->state) ? -1.0f : 0.0f; break; }
            if (nd->n_child == 0) {
                orc_hash_eval(&nd->state, pol, &v);
                az_expand(nd, pol);
                break;
            }
            nd = (nd == root) ? next_child_node_forced(nd, k) : next_child_node(nd);
        }
        backpropagate(path, plen, v);
    }
    float p[81];
    for (int c = 0; c < root->n_child; c++) { n_out[c] = root->child[c]->n; w_out[c] = root->child[c]->w; p[c] = root->child[c]->p; }
    int n = root->n_child;
    orc_prune_targets(n, n_out, w_out, p, k, t_out);
    node_free(root);
    return n;
}
