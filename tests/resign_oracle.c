/*
 * resign_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * The root value that UTTT_SP_RESIGN records (include/uttt_b200.h) needs the root children's (n, w), which the
 * oracle's searches do not return.  This file compiles oracle/uttt_oracle.c into itself (unchanged, so that its node
 * type, PUCT step and backup are the very ones the existing checks rest on) and adds, beside its searches:
 *   - orc_pv_mcts_root_hash: the reference-exact search (cpp/uttt_mcts.cpp:84-196, the oracle's literal queue / flush
 *     loop) under the hash evaluator, with the reference's inverted terminal sign or, with correct_sign, the correct one
 *     (UTTT_SP_CORRECT_TERMINAL_SIGN: -1 for a lost mover, 0 for a draw);
 *   - orc_az_search_root_hash: orc_az_search_hash (the throughput mode with one leaf per round and no root noise);
 * both returning the root children's visit counts and summed values in legal order.
 */
#include "../oracle/uttt_oracle.c"

/* search_leaf with the terminal sign chosen by the caller */
static orc_node *search_leaf_sign(orc_node *nd, orc_node **path, int *plen, float *value, int correct_sign) {
    for (;;) {
        path[(*plen)++] = nd;
        if (orc_is_done(&nd->state)) {
            float v = orc_is_lose(&nd->state) ? -1.0f : 0.0f;
            *value = correct_sign ? v : -v;
            return nd;
        }
        if (nd->n_child == 0) { *value = 0.0f; return nd; }
        nd = next_child_node(nd);
    }
}

int orc_pv_mcts_root_hash(const orc_state *root_state, int evaluate_count, int batch_size, int correct_sign, int *n_out,
                          float *w_out) {
    int root_legal[81];
    int nroot = orc_legal_actions(root_state, root_legal);
    if (nroot == 0) return 0;
    orc_node *root = node_new(root_state, 0.0f);
    float init_pol[81];
    float uniform = 1.0f / (float)nroot;
    for (int i = 0; i < nroot; i++) init_pol[i] = uniform;
    expand(root, init_pol, nroot);

    int qcap = batch_size > 0 ? batch_size : 1;
    orc_node **q_leaf = (orc_node **)malloc(sizeof(orc_node *) * (size_t)qcap);
    orc_node **q_path = (orc_node **)malloc(sizeof(orc_node *) * (size_t)qcap * ORC_MAX_PATH);
    int *q_plen = (int *)malloc(sizeof(int) * (size_t)qcap);
    orc_state *bstates = (orc_state *)malloc(sizeof(orc_state) * (size_t)qcap);
    float *bpol = (float *)malloc(sizeof(float) * 81 * (size_t)qcap);
    float *bval = (float *)malloc(sizeof(float) * (size_t)qcap);
    int nq = 0;
    for (int i = 0; i < evaluate_count; i++) {
        orc_node *path[ORC_MAX_PATH];
        int plen = 0;
        float value;
        orc_node *leaf = search_leaf_sign(root, path, &plen, &value, correct_sign);
        if (orc_is_done(&leaf->state)) {
            backpropagate(path, plen, value);
            continue;
        }
        if (leaf->n == 0 && leaf->n_child == 0) {
            q_leaf[nq] = leaf;
            memcpy(q_path + (size_t)nq * ORC_MAX_PATH, path, sizeof(orc_node *) * (size_t)plen);
            q_plen[nq] = plen;
            nq++;
        }
        if ((nq >= batch_size || i == evaluate_count - 1) && nq > 0) {
            for (int j = 0; j < nq; j++) bstates[j] = q_leaf[j]->state;
            hash_eval_cb(NULL, bstates, nq, bpol, bval);
            for (int j = 0; j < nq; j++) {
                orc_node *lf = q_leaf[j];
                int legal[81];
                int nl = orc_legal_actions(&lf->state, legal);
                float lp[81];
                float sum = 0.0f;
                for (int k = 0; k < nl; k++) {
                    lp[k] = bpol[81 * j + legal[k]];
                    sum += lp[k];
                }
                for (int k = 0; k < nl; k++) lp[k] = (sum > 0) ? lp[k] / sum : (nl == 0 ? 0.0f : 1.0f / (float)nl);
                expand(lf, lp, nl);
                backpropagate(q_path + (size_t)j * ORC_MAX_PATH, q_plen[j], bval[j]);
            }
            nq = 0;
        }
    }
    for (int i = 0; i < root->n_child; i++) { n_out[i] = root->child[i]->n; w_out[i] = root->child[i]->w; }
    int n = root->n_child;
    node_free(root);
    free(q_leaf); free(q_path); free(q_plen); free(bstates); free(bpol); free(bval);
    return n;
}

int orc_az_search_root_hash(const orc_state *root_state, int sims, int *n_out, float *w_out) {
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
            nd = next_child_node(nd);
        }
        backpropagate(path, plen, v);
    }
    for (int k = 0; k < root->n_child; k++) { n_out[k] = root->child[k]->n; w_out[k] = root->child[k]->w; }
    int n = root->n_child;
    node_free(root);
    return n;
}
