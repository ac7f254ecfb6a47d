/* TEST INFRASTRUCTURE: the Gumbel search of include/harmonies_b200.h ("Gumbel search") restated on the C oracle.
 * The oracle is included whole, so the tree, the expansion and the evaluators are exactly those of hzo_search; only the
 * descent differs.  Built by tests/gumbel_oracle.py. */
#include <float.h>

#include "../oracle/hz_oracle.c"

/* mctx's get_sequence_of_considered_visits(m, n) (seq_halving.py) */
void hzo_considered_visits(int m, int n, int32_t *seq) {
    if (m <= 1) {
        for (int i = 0; i < n; i++) seq[i] = i;
        return;
    }
    int log2max = (int)ceil(log2((double)m));
    int visits[64] = {0}, len = 0, nc = m;
    while (len < n) {
        int extra = (int)((double)n / (double)(log2max * nc));
        if (extra < 1) extra = 1;
        for (int x = 0; x < extra; x++) {
            for (int i = 0; i < nc && len < n; i++) seq[len++] = visits[i];
            for (int i = 0; i < nc; i++) visits[i]++;
        }
        nc = nc / 2 > 2 ? nc / 2 : 2;
    }
}

/* completed-Q transform of node nd: lg[k] = logit, sg[k] = sigma of its edge k; sums in edge order */
static void gumbel_sigma(const otree *t, const onode *nd, double vhat, double c_visit, double c_scale, double *lg, double *sg,
                         int *out_mx, int *out_ns) {
    const oedge *E = &t->edges[nd->first_edge];
    const int ne = nd->n_edges;
    double sp = 0.0;
    int mx = 0, ns = 0;
    for (int k = 0; k < ne; k++) { sp += (double)E[k].P; if (E[k].N > mx) mx = E[k].N; ns += E[k].N; }
    double spi = 0.0, spq = 0.0;
    for (int k = 0; k < ne; k++)
        if (E[k].N > 0) {
            double pi = fmax((double)E[k].P / sp, (double)FLT_MIN);
            spi += pi;
            spq += pi * (E[k].W / (double)E[k].N);
        }
    double vmix = (vhat + (double)ns * (spi > 0.0 ? spq / spi : 0.0)) / (1.0 + (double)ns);
    double qmin = INFINITY, qmax = -INFINITY;
    for (int k = 0; k < ne; k++) {
        double q = E[k].N > 0 ? E[k].W / (double)E[k].N : vmix;
        sg[k] = q;
        qmin = fmin(qmin, q); qmax = fmax(qmax, q);
    }
    double span = fmax(qmax - qmin, 1e-8), vs = (c_visit + (double)mx) * c_scale;
    for (int k = 0; k < ne; k++) {
        lg[k] = log((double)fmaxf(E[k].P, FLT_MIN));
        sg[k] = vs * ((sg[k] - qmin) / span);
    }
    *out_mx = mx; *out_ns = ns;
}

static double gumbel_g(uint64_t skey, int action, double scale) {
    uint64_t z = rand64(skey ^ HZ_GUMBEL_SALT, (uint64_t)action);
    return scale * -log(-log(((double)(z >> 11) + 0.5) * 0x1p-53));
}

/* root scores at considered visit cv (-inf off the considered set) */
static void root_scores(const otree *t, const onode *nd, uint64_t skey, double scale, int cv, const double *lg,
                        const double *sg, double *sc) {
    const oedge *E = &t->edges[nd->first_edge];
    double mlg = -INFINITY;
    for (int k = 0; k < nd->n_edges; k++) mlg = fmax(mlg, lg[k]);
    for (int k = 0; k < nd->n_edges; k++)
        sc[k] = E[k].N == cv ? fmax(-1e9, gumbel_g(skey, E[k].action, scale) + (lg[k] - mlg) + sg[k]) : -INFINITY;
}

static void softmax_z(int ne, const double *lg, const double *sg, double *p) {
    double zm = -INFINITY, s = 0.0;
    for (int k = 0; k < ne; k++) zm = fmax(zm, lg[k] + sg[k]);
    for (int k = 0; k < ne; k++) { p[k] = exp(lg[k] + sg[k] - zm); s += p[k]; }
    for (int k = 0; k < ne; k++) p[k] /= s;
}

/* first strict maximum; *gap = min(*gap, smallest non-zero distance from the winner to another finite score) */
static int argmax_gap(const double *sc, int n, double *gap) {
    int b = -1;
    for (int k = 0; k < n; k++) if (sc[k] > -INFINITY && (b < 0 || sc[k] > sc[b])) b = k;
    if (b < 0) return -1;
    for (int k = 0; k < n; k++) {
        if (k == b || !(sc[k] > -INFINITY)) continue;
        double d = sc[b] - sc[k];
        if (d != 0.0 && d < *gap) *gap = d;
    }
    return b;
}

/* hzo_search with the Gumbel descent (m = max_considered, n = num_sims of the table; c_visit, c_scale, scale as the
 * library's fp32 arguments).  Also returns the root's policy target [143], the played action, vhat(root) and the
 * smallest non-zero score gap of all decisions of the search (INFINITY when no decision had two distinct scores). */
int hzo_search_gumbel(const uint32_t *root, uint64_t search_key, int sims, int key_mode, int m, int n, float c_visit_f,
                      float c_scale_f, float scale_f, hzo_eval_fn eval, void *user, int32_t *outN, double *outW, float *outP,
                      int32_t *out_child, int32_t *out_nodes, int32_t *out_edges, hzo_tree_dump *dump, float *out_policy,
                      int32_t *out_action, float *out_root_value, double *out_gap) {
    geometry();
    if (!eval) eval = fake_eval;
    const double c_visit = c_visit_f, c_scale = c_scale_f, scale = scale_f;
    otree t;
    t.cap_nodes = 1 + 69 * sims; t.cap_edges = 69 * sims + 1;
    int tsize = 1; while (tsize < 2 * t.cap_nodes) tsize <<= 1;
    t.table_mask = tsize - 1;
    t.nodes = (onode *)malloc(sizeof(onode) * (size_t)t.cap_nodes);
    t.edges = (oedge *)malloc(sizeof(oedge) * (size_t)t.cap_edges);
    t.table = (int *)malloc(sizeof(int) * (size_t)tsize);
    float *vhat = (float *)calloc((size_t)t.cap_nodes, sizeof(float));
    int *path = (int *)malloc(sizeof(int) * (size_t)(sims + 2));
    int32_t *table = (int32_t *)malloc(sizeof(int32_t) * (size_t)(m + 1) * (size_t)n);
    for (int k = 0; k <= m; k++) hzo_considered_visits(k, n, table + (size_t)k * n);
    for (int i = 0; i < tsize; i++) t.table[i] = -1;
    t.n_nodes = 0; t.n_edges = 0; t.key_mode = key_mode;
    int was_new, rc = 0;
    double gap = INFINITY, lg[HZ_ACTION_SIZE], sg[HZ_ACTION_SIZE], sc[HZ_ACTION_SIZE];
    tree_find_or_add(&t, root, key_hash(root, key_mode), &was_new);

    for (int sim = 0; sim < sims && rc == 0; sim++) {
        int cur = 0, depth = 0;
        while (t.nodes[cur].n_edges > 0) {
            onode *nd = &t.nodes[cur];
            int mx, ns, ne = nd->n_edges;
            gumbel_sigma(&t, nd, (double)vhat[cur], c_visit, c_scale, lg, sg, &mx, &ns);
            if (depth == 0) {
                int kc = m < ne ? m : ne, i = ns < n - 1 ? ns : n - 1;
                root_scores(&t, nd, search_key, scale, table[(size_t)kc * n + i], lg, sg, sc);
            } else {
                softmax_z(ne, lg, sg, sc);
                for (int k = 0; k < ne; k++) sc[k] -= (double)t.edges[nd->first_edge + k].N / (1.0 + (double)ns);
            }
            int b = argmax_gap(sc, ne, &gap);
            if (b < 0 && depth == 0) b = 0;
            if (b < 0) break;
            path[depth++] = nd->first_edge + b;
            cur = t.edges[nd->first_edge + b].child;
        }
        onode *leaf = &t.nodes[cur];
        ostate ls; unpack(leaf->w, &ls);
        double value;
        if (!is_over(&ls)) {
            float policy[HZ_ACTION_SIZE];
            eval(leaf->w, policy, &value, user);
            int acts[HZ_ACTION_SIZE], k = legal_actions(&ls, acts);
            int first = t.n_edges, cnt = 0;
            for (int i = 0; i < k; i++) {
                ostate cs = ls;
                cs.key = search_key; cs.event = ((uint32_t)sim << 8) | (uint32_t)acts[i];
                if (apply_action(&cs, acts[i], HZ_NO_DRAW) != HZ_MOVE_OK) continue;
                cs.key = ls.key; cs.event = ls.event;
                uint32_t cw[32]; pack(&cs, cw);
                uint64_t h = key_hash(cw, key_mode);
                if (h == leaf->hash) continue;
                int child = tree_find_or_add(&t, cw, h, &was_new);
                leaf = &t.nodes[cur];
                if (child < 0 || t.n_edges == t.cap_edges) { rc = -1; break; }
                oedge *e = &t.edges[t.n_edges++];
                e->child = child; e->N = 0; e->V = 0; e->W = 0.0; e->P = policy[acts[i]];
                e->action = acts[i]; e->mover = leaf->player;
                cnt++;
            }
            leaf->first_edge = first; leaf->n_edges = cnt;
            vhat[cur] = (float)value;                                /* the evaluator's fp32 value */
        } else {
            int oc = outcome(&ls);
            value = oc == 0 ? 0.0 : (leaf->player == 0 ? (double)oc : -(double)oc);
        }
        for (int d = depth - 1; d >= 0; d--) {
            oedge *e = &t.edges[path[d]];
            double dir = e->mover == t.nodes[cur].player ? 1.0 : -1.0;
            e->N += 1; e->W += value * dir;
        }
    }
    for (int a = 0; a < HZ_ACTION_SIZE; a++) {
        if (outN) outN[a] = 0;
        if (outW) outW[a] = 0.0;
        if (outP) outP[a] = 0.0f;
        if (out_child) out_child[a] = -1;
        if (out_policy) out_policy[a] = 0.0f;
    }
    const onode *r = &t.nodes[0];
    for (int k = 0; k < r->n_edges; k++) {
        oedge *e = &t.edges[r->first_edge + k];
        if (outN) outN[e->action] = e->N;
        if (outW) outW[e->action] = e->W;
        if (outP) outP[e->action] = e->P;
        if (out_child) out_child[e->action] = e->child;
    }
    int action = -1;
    float rv = 0.0f;
    if (r->n_edges > 0) {                                        /* hz_tree_gumbel_root */
        int mx, ns;
        double p[HZ_ACTION_SIZE];
        gumbel_sigma(&t, r, (double)vhat[0], c_visit, c_scale, lg, sg, &mx, &ns);
        root_scores(&t, r, search_key, scale, mx, lg, sg, sc);
        int b = argmax_gap(sc, r->n_edges, &gap);
        if (b < 0) b = 0;
        action = t.edges[r->first_edge + b].action;
        softmax_z(r->n_edges, lg, sg, p);
        if (out_policy)
            for (int k = 0; k < r->n_edges; k++) out_policy[t.edges[r->first_edge + k].action] = (float)p[k];
        rv = vhat[0];
    }
    if (out_action) *out_action = action;
    if (out_root_value) *out_root_value = rv;
    if (out_gap) *out_gap = gap;
    if (out_nodes) *out_nodes = t.n_nodes;
    if (out_edges) *out_edges = t.n_edges;
    dump_tree(&t, dump);
    free(t.nodes); free(t.edges); free(t.table); free(path); free(vhat); free(table);
    return rc;
}
