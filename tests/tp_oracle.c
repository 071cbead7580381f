/*
 * tp_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * One move's search of the throughput mode (UTTT_SP_THROUGHPUT, tree_tp_round_kernel) restated on the CPU for any number
 * m = 1..16 of leaves per tree per round.  This file compiles oracle/uttt_oracle.c into itself (its rules, hash evaluator
 * and Philox stream) and is linked with tests/symmetry_oracle.c (its board symmetries and symmetry draw).  The round:
 *   - round 0 queues the root (evaluation 0); round 1 expands it from its row and, with eta != NULL, mixes the root
 *     noise into its priors: p = fma(1 - eps, p, eps * eta[a]) (one rounding for the multiply-add);
 *   - every round then collects up to min(m, sims_left) leaves: a descent by PUCT in which a child with vl units of
 *     virtual loss counts as n + vl visits and w + vl lost value (forced_k > 0: the root's forcing rule, N with virtual
 *     loss); a descent that ends on a terminal position is backed up at once (-1 lost, 0 drawn, no virtual loss); an
 *     unexpanded leaf gets one unit of virtual loss on every node of its path, is marked pending and queued.  Collection
 *     stops when a descent ends on a pending leaf (blocked), when got + terminals == sims_left or terminals == 2m (the
 *     terminal guard), or when m leaves are queued; a round of terminals only goes on in the next round;
 *   - the next round expands and backs up the pending leaves in queue order (removing their virtual loss), then collects;
 *   - when the budget is spent the move is decided: the root children's (n, w, p) in legal order, the policy targets
 *     (forced_k > 0: the pruning of UTTT_SP_FORCED_PLAYOUTS, else the counts) and the root value -w/n of the first most
 *     visited child.  No virtual loss may be outstanding then; the oracle checks it.
 * Evaluations are the hash evaluator, optionally under the symmetry g = orc_symmetry_draw(seed, game, ply, j) of
 * evaluation j, or recorded rows (policy in the leaf's own action ids, value) consumed in evaluation order.
 * Every float operation is a single correctly rounded fp32 operation in the order written (-std=c11: no FMA contraction;
 * the one fused multiply-add of the noise mix is an explicit fmaf).
 */
#include "../oracle/uttt_oracle.c"

/* tests/symmetry_oracle.c */
void orc_symmetry(const orc_state *s, int g, orc_state *out);
int orc_symmetry_action(int a, int g);
int orc_symmetry_draw(uint32_t seed, uint64_t game, uint32_t ply, uint32_t j);

#define TP_MAX_M 16

typedef struct {
    int action, n, vl, first, cnt, pending;      /* first/cnt: children (cnt = 0: unexpanded) */
    float w, p;
} tp_node;

typedef struct {
    tp_node *node;
    int n_nodes, cap;
    /* evaluator */
    int sym;
    uint32_t seed, ply;
    uint64_t game;
    int n_rows, used;
    const float *row_pol, *row_val;
    int n_eval;
    /* output: queued positions */
    int leaf_cap, n_leaves;
    uint32_t *leaf_states;
    int *leaf_round;
} tp_search;

enum { TP_UNEXPANDED = 0, TP_LOST = 1, TP_DRAWN = 2, TP_BLOCKED = 3 };

/* evaluation s->n_eval of the move: leaf st -> policy row in st's own action ids, value */
static int tp_eval(tp_search *s, const orc_state *st, float *pol, float *val) {
    const int j = s->n_eval++;
    if (s->n_rows >= 0) {
        if (s->used >= s->n_rows) return 0;
        memcpy(pol, s->row_pol + 81 * (size_t)s->used, 81 * sizeof(float));
        *val = s->row_val[s->used++];
        return 1;
    }
    int g = s->sym ? orc_symmetry_draw(s->seed, s->game, s->ply, (uint32_t)j) : 0;
    orc_state gs;
    float gp[81];
    orc_symmetry(st, g, &gs);
    orc_hash_eval(&gs, gp, val);
    for (int a = 0; a < 81; a++) pol[a] = gp[orc_symmetry_action(a, g)];
    return 1;
}

static int tp_queue(tp_search *s, const orc_state *st, int round) {
    if (s->n_leaves >= s->leaf_cap) return 0;
    orc_pack(st, s->leaf_states + 8 * (size_t)s->n_leaves);
    s->leaf_round[s->n_leaves++] = round;
    return 1;
}

/* expansion of node nd (position st) from its row: priors pol[legal] / sum, the sum taken serially over the legal
 * actions in ascending id, uniform 1/L if it is not positive; with eta the root noise is mixed in */
static void tp_expand(tp_search *s, int nd, const orc_state *st, const float *pol, const float *eta, float eps) {
    int legal[81];
    int L = orc_legal_actions(st, legal);
    float sum = 0.0f;
    for (int k = 0; k < L; k++) sum = sum + pol[legal[k]];
    const float uni = 1.0f / (float)L, keep = 1.0f - eps;
    const int base = s->n_nodes;
    for (int k = 0; k < L; k++) {
        tp_node *c = &s->node[base + k];
        memset(c, 0, sizeof(*c));
        c->action = legal[k];
        float p = (sum > 0.0f) ? pol[legal[k]] / sum : uni;
        if (eta) p = fmaf(keep, p, eps * eta[legal[k]]);
        c->p = p;
    }
    s->node[nd].first = base;
    s->node[nd].cnt = L;
    s->n_nodes = base + L;
}

/* descent from the root; path[0..*plen) the node path, *st the position it ended on */
static int tp_descend(tp_search *s, const orc_state *root, int *path, int *plen, orc_state *st, float forced_k) {
    *st = *root;
    int nd = 0;
    *plen = 0;
    path[(*plen)++] = 0;
    for (;;) {
        int legal[81];
        if (orc_is_lose(st)) return TP_LOST;
        if (orc_legal_actions(st, legal) == 0) return TP_DRAWN;
        const tp_node *x = &s->node[nd];
        if (x->pending) return TP_BLOCKED;
        if (x->cnt == 0) return TP_UNEXPANDED;
        int tot = 0;
        for (int i = 0; i < x->cnt; i++) tot += s->node[x->first + i].n + s->node[x->first + i].vl;
        const float sq = sqrtf((float)tot);
        const int force = forced_k > 0.0f && *plen == 1;
        float best = -1e9f;
        int besti = 0;
        for (int i = 0; i < x->cnt; i++) {
            const tp_node *c = &s->node[x->first + i];
            const int n = c->n + c->vl;
            float sc = c->p * sq;
            if (n > 0) {
                const float q = -(c->w + (float)c->vl) / (float)n;
                sc = q + sc / (float)(1 + n);
                if (force && (float)n < sqrtf((forced_k * c->p) * (float)tot)) sc = 1e20f;
            }
            if (sc > best) { best = sc; besti = i; }
        }
        nd = x->first + besti;
        orc_state nx;
        orc_next(st, s->node[nd].action, &nx);
        *st = nx;
        path[(*plen)++] = nd;
    }
}

/* value v for the mover of the path's last node, alternating sign towards the root; n += 1, vl -= had_vloss */
static void tp_backup(tp_search *s, const int *path, int plen, float v, int had_vloss) {
    for (int i = plen - 1; i >= 0; i--) {
        tp_node *x = &s->node[path[i]];
        x->w = x->w + (((plen - 1 - i) & 1) ? -v : v);
        x->n += 1;
        x->vl -= had_vloss;
    }
}

/* the policy targets of UTTT_SP_FORCED_PLAYOUTS from the root children's raw (n, w, p) in legal order */
static void tp_prune(int L, const int *n, const float *w, const float *p, float k, int *t) {
    int tot = 0, cs = 0;
    for (int i = 0; i < L; i++) {
        tot += n[i];
        if (n[i] > n[cs]) cs = i;
        t[i] = n[i];
    }
    if (L == 0 || n[cs] == 0) return;
    const float sq = sqrtf((float)tot);
    const float best = -w[cs] / (float)n[cs] + (p[cs] * sq) / (float)(1 + n[cs]);
    for (int i = 0; i < L; i++) {
        if (i == cs || n[i] == 0) continue;
        const float q = -w[i] / (float)n[i], u = p[i] * sq;
        const int f = (int)sqrtf((k * p[i]) * (float)tot);
        const int cap = n[i] < f ? n[i] : f;
        int r = 0;
        while (r < cap && q + u / (float)(n[i] - r) < best) r++;
        t[i] = (r >= 1 && n[i] - r == 1) ? 0 : n[i] - r;
    }
}

/*
 * One move's search of root_state.  sims >= 1, m in 1..16, forced_k (0: off), eta[81] by action id (NULL: no noise) with
 * eps; evaluator: n_rows >= 0 recorded rows row_pol[n_rows][81], row_val[n_rows], else the hash evaluator (sym: under
 * the symmetry keyed (seed, game, ply)).  Outputs the root children's n, w, p, targets t in legal order and *value;
 * leaf_states[leaf_cap][8] / leaf_round[leaf_cap] the queued positions (the root first) with the round each was queued
 * in, *n_leaves of them; cov[6] = rounds, blocked stops, terminal backups, terminal-guard stops, terminal-only rounds,
 * evaluations.  Returns the number of root children (0: a finished root, nothing queued), or -1 when recorded rows run
 * out, -2 when leaf_cap is too small, -3 when virtual loss is outstanding at the decision, -4 on bad arguments.
 */
int orc_tp_search(const orc_state *root_state, int sims, int m, float forced_k, const float *eta, float eps, int sym,
                  uint32_t seed, uint64_t game, uint32_t ply, int n_rows, const float *row_pol, const float *row_val,
                  int *n_out, float *w_out, float *p_out, int *t_out, float *value, int leaf_cap, uint32_t *leaf_states,
                  int *leaf_round, int *n_leaves, int *cov) {
    for (int i = 0; i < 6; i++) cov[i] = 0;
    *n_leaves = 0;
    *value = 0.0f;
    if (sims < 1 || m < 1 || m > TP_MAX_M) return -4;
    int tmp[81];
    if (orc_legal_actions(root_state, tmp) == 0) return 0;
    tp_search s;
    memset(&s, 0, sizeof(s));
    s.cap = 1 + 81 * (sims + 1);
    s.node = (tp_node *)calloc((size_t)s.cap, sizeof(tp_node));
    s.sym = sym; s.seed = seed; s.game = game; s.ply = ply;
    s.n_rows = n_rows; s.row_pol = row_pol; s.row_val = row_val;
    s.leaf_cap = leaf_cap; s.leaf_states = leaf_states; s.leaf_round = leaf_round;
    int rc = 0;
    s.n_nodes = 1;

    /* round 0: the root is queued; round 1: it is expanded */
    float pol[81], v;
    if (!tp_queue(&s, root_state, 0)) { rc = -2; goto out; }
    if (!tp_eval(&s, root_state, pol, &v)) { rc = -1; goto out; }
    tp_expand(&s, 0, root_state, pol, eta, eps);
    int round = 1, sims_left = sims;
    int paths[TP_MAX_M][ORC_MAX_PATH], plens[TP_MAX_M];
    orc_state pend[TP_MAX_M];
    int pend_node[TP_MAX_M];
    while (sims_left > 0) {
        const int want = sims_left < m ? sims_left : m;
        int got = 0, terminals = 0, blocked = 0;
        while (got < want && got + terminals < sims_left && terminals < 2 * m) {
            int path[ORC_MAX_PATH], plen;
            orc_state st;
            const int end = tp_descend(&s, root_state, path, &plen, &st, forced_k);
            if (end == TP_BLOCKED) { blocked = 1; break; }
            if (end != TP_UNEXPANDED) {
                tp_backup(&s, path, plen, end == TP_LOST ? -1.0f : 0.0f, 0);
                terminals++;
                continue;
            }
            for (int i = 0; i < plen; i++) s.node[path[i]].vl += 1;
            s.node[path[plen - 1]].pending = 1;
            memcpy(paths[got], path, sizeof(int) * (size_t)plen);
            plens[got] = plen;
            pend[got] = st;
            pend_node[got] = path[plen - 1];
            if (!tp_queue(&s, &st, round)) { rc = -2; goto out; }
            got++;
        }
        cov[1] += blocked;
        cov[2] += terminals;
        cov[3] += (!blocked && got < want);
        sims_left -= terminals;
        if (got > 0) {
            round++;                                 /* the evaluator runs; the next round applies its rows in queue order */
            for (int j = 0; j < got; j++) {
                if (!tp_eval(&s, &pend[j], pol, &v)) { rc = -1; goto out; }
                s.node[pend_node[j]].pending = 0;
                tp_expand(&s, pend_node[j], &pend[j], pol, NULL, 0.0f);
                tp_backup(&s, paths[j], plens[j], v, 1);
            }
            sims_left -= got;
        } else if (sims_left > 0) {
            cov[4] += 1;                             /* terminals only: the search goes on in the next round */
            round++;
        }
    }
    cov[0] = round;
    for (int i = 0; i < s.n_nodes; i++)
        if (s.node[i].vl != 0 || s.node[i].pending) { rc = -3; goto out; }
    {
        const tp_node *r = &s.node[0];
        int cs = 0;
        for (int i = 0; i < r->cnt; i++) {
            const tp_node *c = &s.node[r->first + i];
            n_out[i] = c->n; w_out[i] = c->w; p_out[i] = c->p;
            if (c->n > n_out[cs]) cs = i;
        }
        *value = n_out[cs] > 0 ? -w_out[cs] / (float)n_out[cs] : 0.0f;
        if (forced_k > 0.0f) tp_prune(r->cnt, n_out, w_out, p_out, forced_k, t_out);
        else for (int i = 0; i < r->cnt; i++) t_out[i] = n_out[i];
        rc = r->cnt;
    }
out:
    cov[5] = s.n_eval;
    *n_leaves = s.n_leaves;
    free(s.node);
    return rc;
}
