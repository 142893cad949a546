/* Exact 2-passenger pool: minimum-cost maximum-cardinality pair matching.  TEST INFRASTRUCTURE ONLY.
 *
 * A literal sequential O(n^3) primal-dual blossom algorithm (Edmonds / Galil), restated from the van Rantwijk
 * formulation that networkx ships as max_weight_matching (no max-cardinality flag), on a dense n x n weight table.
 * Edge candidates, plans and costs are those of pool_pairs_oracle (pool_oracle.c); the weight of an edge is
 * K - cost with K = floor(n/2) * 3 * 2^22 + 1, which exceeds floor(n/2) * (c_max - c_min) for every cost in
 * [0, 3 * 2^22] (three stand distances of at most 2^22): one more pair always outweighs any cost saving, so the
 * maximum-weight matching is a maximum-cardinality matching of minimum total cost.  Duals are kept doubled, as in
 * networkx (slack = u_i + u_j - 2 w_ij), so every quantity stays an even int64.
 *
 * Vertices are 0..n-1, blossoms n..2n-1; blossom children form a circular linked list (cnext / cprev) with the edge
 * to the next child stored on the child (cex in this child, cey in the next one). */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int n;
    const int64_t *W;                       /* n x n weights, 0 = no edge */
    int *mate, *label, *lex, *ley, *inb, *bpar, *bbase, *bfirst, *nchild, *cnext, *cprev, *cex, *cey, *bex, *bey;
    int *queue, qn, *freeb, nfree, *tmp;
    int64_t *dual;
} Bl;

static int64_t slack(const Bl *m, int v, int w) { return m->dual[v] + m->dual[w] - 2 * m->W[(int64_t)v * m->n + w]; }

static void push_leaves(Bl *m, int b) {
    if (b < m->n) { m->queue[m->qn++] = b; return; }
    for (int v = 0; v < m->n; v++) if (m->inb[v] == b) m->queue[m->qn++] = v;
}

static void assign_label(Bl *m, int w, int t, int v) {
    int b = m->inb[w];
    m->label[w] = m->label[b] = t;
    m->lex[w] = m->lex[b] = v;
    m->ley[w] = m->ley[b] = v >= 0 ? w : -1;
    m->bex[w] = m->bex[b] = -1;
    m->bey[w] = m->bey[b] = -1;
    if (t == 1) push_leaves(m, b);
    else { int base = m->bbase[b]; assign_label(m, m->mate[base], 1, base); }
}

static int scan_blossom(Bl *m, int v, int w) {
    int np = 0, base = -1;
    while (v != -1) {
        int b = m->inb[v];
        if (m->label[b] & 4) { base = m->bbase[b]; break; }
        m->tmp[np++] = b;
        m->label[b] = 5;
        if (m->lex[b] == -1) v = -1;
        else { v = m->lex[b]; b = m->inb[v]; v = m->lex[b]; }
        if (w != -1) { int t = v; v = w; w = t; }
    }
    for (int i = 0; i < np; i++) m->label[m->tmp[i]] = 1;
    return base;
}

static void add_blossom(Bl *m, int base, int v, int w) {
    const int n = m->n;
    int bb = m->inb[base], bv = m->inb[v], bw = m->inb[w];
    int b = m->freeb[--m->nfree];
    m->bbase[b] = base; m->bpar[b] = -1; m->bpar[bb] = b;
    /* tmp holds the children, tmp + 2n the edge x, tmp + 4n the edge y */
    int *ch = m->tmp, *ex = m->tmp + 2 * n, *ey = m->tmp + 4 * n, k = 0;
    while (bv != bb) {                       /* v side, from v towards the base */
        m->bpar[bv] = b;
        ch[k] = bv; ex[k] = m->lex[bv]; ey[k] = m->ley[bv]; k++;
        bv = m->inb[m->lex[bv]];
    }
    int L = 0;
    int *c2 = m->tmp + 6 * n, *x2 = m->tmp + 8 * n, *y2 = m->tmp + 10 * n;
    c2[L] = bb;
    for (int i = k - 1; i >= 0; i--) { c2[L + 1] = ch[i]; x2[L] = ex[i]; y2[L] = ey[i]; L++; }
    x2[L] = v; y2[L] = w;                    /* edge from the last v-side child to the first w-side one */
    L++;
    while (bw != bb) {
        m->bpar[bw] = b;
        c2[L] = bw; x2[L] = m->ley[bw]; y2[L] = m->lex[bw]; L++;
        bw = m->inb[m->lex[bw]];
    }
    for (int i = 0; i < L; i++) {
        int c = c2[i], d = c2[(i + 1) % L];
        m->cnext[c] = d; m->cprev[d] = c; m->cex[c] = x2[i]; m->cey[c] = y2[i];
    }
    m->bfirst[b] = bb; m->nchild[b] = L;
    m->label[b] = 1; m->lex[b] = m->lex[bb]; m->ley[b] = m->ley[bb]; m->dual[b] = 0;
    for (int u = 0; u < n; u++) {
        int t = m->inb[u];
        if (t != b && m->bpar[t] == b) {
            if (m->label[t] == 2) m->queue[m->qn++] = u;
            m->inb[u] = b;
        }
    }
    int64_t best = -1; int bi = -1, bj = -1;
    for (int i = 0; i < n; i++) {
        if (m->inb[i] != b) continue;
        for (int j = 0; j < n; j++) {
            if (m->W[(int64_t)i * n + j] == 0 || m->inb[j] == b || m->label[m->inb[j]] != 1) continue;
            int64_t s = slack(m, i, j);
            if (bi < 0 || s < best) { best = s; bi = i; bj = j; }
        }
    }
    for (int i = 0; i < L; i++) { m->bex[c2[i]] = -1; m->bey[c2[i]] = -1; }
    m->bex[b] = bi; m->bey[b] = bj;
}

static int is_leaf_of(const Bl *m, int v, int s) {
    for (int t = v; t != -1; t = m->bpar[t]) if (t == s) return 1;
    return 0;
}

static void expand_blossom(Bl *m, int b, int endstage) {
    const int n = m->n;
    int c = m->bfirst[b];
    for (int i = 0; i < m->nchild[b]; i++, c = m->cnext[c]) {
        m->bpar[c] = -1;
        if (c >= n) {
            if (endstage && m->dual[c] == 0) expand_blossom(m, c, endstage);
            else for (int v = 0; v < n; v++) if (is_leaf_of(m, v, c)) m->inb[v] = c;
        } else {
            m->inb[c] = c;
        }
    }
    if (!endstage && m->label[b] == 2) {
        const int L = m->nchild[b];
        int entry = m->inb[m->ley[b]];
        int j = 0;
        for (c = m->bfirst[b]; c != entry; c = m->cnext[c]) j++;
        int jstep;
        if (j & 1) { j -= L; jstep = 1; } else jstep = -1;
        int v = m->lex[b], w = m->ley[b], p, q;
        while (j != 0) {
            if (jstep == 1) { p = m->cex[c]; q = m->cey[c]; }
            else { q = m->cex[m->cprev[c]]; p = m->cey[m->cprev[c]]; }
            (void)p;
            m->label[w] = 0; m->label[q] = 0;
            assign_label(m, w, 2, v);
            j += jstep; c = jstep == 1 ? m->cnext[c] : m->cprev[c];
            if (jstep == 1) { v = m->cex[c]; w = m->cey[c]; }
            else { w = m->cex[m->cprev[c]]; v = m->cey[m->cprev[c]]; }
            j += jstep; c = jstep == 1 ? m->cnext[c] : m->cprev[c];
        }
        int bw = c;
        m->label[w] = m->label[bw] = 2;
        m->lex[w] = m->lex[bw] = v; m->ley[w] = m->ley[bw] = w;
        m->bex[bw] = m->bey[bw] = -1;
        c = jstep == 1 ? m->cnext[c] : m->cprev[c];
        while (c != entry) {
            int bv = c;
            if (m->label[bv] == 1) { c = jstep == 1 ? m->cnext[c] : m->cprev[c]; continue; }
            int u = bv;
            if (bv >= n) {
                u = -1;
                for (int x = 0; x < n; x++) if (m->label[x] && m->inb[x] == bv) { u = x; break; }
            }
            if (u >= 0 && m->label[u]) {
                m->label[u] = 0;
                m->label[m->mate[m->bbase[bv]]] = 0;
                assign_label(m, u, 2, m->lex[u]);
            }
            c = jstep == 1 ? m->cnext[c] : m->cprev[c];
        }
    }
    m->label[b] = 0; m->lex[b] = m->ley[b] = -1; m->bex[b] = m->bey[b] = -1;
    m->bpar[b] = -1; m->bbase[b] = -1; m->dual[b] = 0;
    m->freeb[m->nfree++] = b;
}

static void augment_blossom(Bl *m, int b, int v) {
    const int n = m->n;
    int t = v;
    while (m->bpar[t] != b) t = m->bpar[t];
    if (t >= n) augment_blossom(m, t, v);
    const int L = m->nchild[b];
    int i = 0, c;
    for (c = m->bfirst[b]; c != t; c = m->cnext[c]) i++;
    int j = i, jstep;
    if (i & 1) { j -= L; jstep = 1; } else jstep = -1;
    while (j != 0) {
        int w, x;
        j += jstep; c = jstep == 1 ? m->cnext[c] : m->cprev[c];
        if (jstep == 1) { w = m->cex[c]; x = m->cey[c]; }
        else { x = m->cex[m->cprev[c]]; w = m->cey[m->cprev[c]]; }
        if (c >= n) augment_blossom(m, c, w);
        j += jstep; c = jstep == 1 ? m->cnext[c] : m->cprev[c];
        if (c >= n) augment_blossom(m, c, x);
        m->mate[w] = x; m->mate[x] = w;
    }
    m->bfirst[b] = t;
    m->bbase[b] = m->bbase[t];
}

static void augment_matching(Bl *m, int v, int w) {
    for (int side = 0; side < 2; side++) {
        int s = side ? w : v, j = side ? v : w;
        for (;;) {
            int bs = m->inb[s];
            if (bs >= m->n) augment_blossom(m, bs, s);
            m->mate[s] = j;
            if (m->lex[bs] == -1) break;
            int t = m->lex[bs], bt = m->inb[t];
            s = m->lex[bt]; j = m->ley[bt];
            if (bt >= m->n) augment_blossom(m, bt, j);
            m->mate[j] = s;
        }
    }
}

/* max-weight matching of the dense weights W (0 = no edge, else > 0); mate[v] = partner or -1 */
static int blossom(int n, const int64_t *W, int *mate_out) {
    Bl M, *m = &M;
    memset(m, 0, sizeof M);
    m->n = n; m->W = W;
    const int N2 = 2 * n > 0 ? 2 * n : 1;
    int *ints = (int *)malloc(sizeof(int) * (size_t)N2 * 30);
    int64_t *duals = (int64_t *)calloc((size_t)N2, sizeof(int64_t));
    if (!ints || !duals) { free(ints); free(duals); return -1; }
    int *p = ints;
    m->mate = mate_out;
    m->label = p; p += N2; m->lex = p; p += N2; m->ley = p; p += N2; m->inb = p; p += N2; m->bpar = p; p += N2;
    m->bbase = p; p += N2; m->bfirst = p; p += N2; m->nchild = p; p += N2; m->cnext = p; p += N2; m->cprev = p; p += N2;
    m->cex = p; p += N2; m->cey = p; p += N2; m->bex = p; p += N2; m->bey = p; p += N2; m->queue = p; p += N2 * 2;
    m->freeb = p; p += N2; m->tmp = p;           /* 12 n scratch */
    m->dual = duals;
    int64_t maxw = 0;
    for (int64_t k = 0; k < (int64_t)n * n; k++) if (W[k] > maxw) maxw = W[k];
    for (int v = 0; v < 2 * n; v++) {
        m->label[v] = 0; m->lex[v] = m->ley[v] = -1; m->bpar[v] = -1; m->bex[v] = m->bey[v] = -1;
        m->bbase[v] = v < n ? v : -1; m->inb[v] = v; m->nchild[v] = 0;
    }
    for (int v = 0; v < n; v++) { m->mate[v] = -1; m->dual[v] = maxw; }
    m->nfree = 0;
    for (int b = 2 * n - 1; b >= n; b--) m->freeb[m->nfree++] = b;
    for (;;) {
        for (int b = 0; b < 2 * n; b++) { m->label[b] = 0; m->lex[b] = m->ley[b] = -1; m->bex[b] = m->bey[b] = -1; }
        m->qn = 0;
        for (int v = 0; v < n; v++)
            if (m->mate[v] == -1 && m->label[m->inb[v]] == 0) assign_label(m, v, 1, -1);
        int augmented = 0;
        for (;;) {
            while (m->qn > 0 && !augmented) {
                int v = m->queue[--m->qn];
                for (int w = 0; w < n; w++) {
                    if (W[(int64_t)v * n + w] == 0) continue;
                    int bv = m->inb[v], bw = m->inb[w];
                    if (bv == bw) continue;
                    int64_t ks = slack(m, v, w);
                    if (ks <= 0) {
                        if (m->label[bw] == 0) assign_label(m, w, 2, v);
                        else if (m->label[bw] == 1) {
                            int base = scan_blossom(m, v, w);
                            if (base != -1) add_blossom(m, base, v, w);
                            else { augment_matching(m, v, w); augmented = 1; break; }
                        } else if (m->label[w] == 0) { m->label[w] = 2; m->lex[w] = v; m->ley[w] = w; }
                    } else if (m->label[bw] == 1) {
                        if (m->bex[bv] == -1 || ks < slack(m, m->bex[bv], m->bey[bv])) { m->bex[bv] = v; m->bey[bv] = w; }
                    } else if (m->label[w] == 0) {
                        if (m->bex[w] == -1 || ks < slack(m, m->bex[w], m->bey[w])) { m->bex[w] = v; m->bey[w] = w; }
                    }
                }
            }
            if (augmented) break;
            int dtype = 1, de_v = -1, de_w = -1, dblossom = -1;
            int64_t delta = INT64_MAX;
            for (int v = 0; v < n; v++) if (m->dual[v] < delta) delta = m->dual[v];
            for (int v = 0; v < n; v++)
                if (m->label[m->inb[v]] == 0 && m->bex[v] != -1) {
                    int64_t d = slack(m, m->bex[v], m->bey[v]);
                    if (d < delta) { delta = d; dtype = 2; de_v = m->bex[v]; de_w = m->bey[v]; }
                }
            for (int b = 0; b < 2 * n; b++)
                if (m->bbase[b] != -1 && m->bpar[b] == -1 && m->label[b] == 1 && m->bex[b] != -1) {
                    int64_t d = slack(m, m->bex[b], m->bey[b]) / 2;
                    if (d < delta) { delta = d; dtype = 3; de_v = m->bex[b]; de_w = m->bey[b]; }
                }
            for (int b = n; b < 2 * n; b++)
                if (m->bbase[b] != -1 && m->bpar[b] == -1 && m->label[b] == 2 && m->dual[b] < delta) {
                    delta = m->dual[b]; dtype = 4; dblossom = b;
                }
            for (int v = 0; v < n; v++) {
                int l = m->label[m->inb[v]];
                if (l == 1) m->dual[v] -= delta; else if (l == 2) m->dual[v] += delta;
            }
            for (int b = n; b < 2 * n; b++)
                if (m->bbase[b] != -1 && m->bpar[b] == -1) {
                    if (m->label[b] == 1) m->dual[b] += delta; else if (m->label[b] == 2) m->dual[b] -= delta;
                }
            if (dtype == 1) break;
            if (dtype == 2 || dtype == 3) { (void)de_w; m->queue[m->qn++] = de_v; }
            else expand_blossom(m, dblossom, 0);
        }
        if (!augmented) break;
        for (int b = n; b < 2 * n; b++)
            if (m->bbase[b] != -1 && m->bpar[b] == -1 && m->label[b] == 1 && m->dual[b] == 0) expand_blossom(m, b, 1);
    }
    free(ints); free(duals);
    return 0;
}

/* candidate (A picked up first, then B) as pool_pairs_oracle accepts it; returns 1 with plan / cost when accepted */
static int candidate(const int32_t *from, const int32_t *to, const int32_t *dist, int S, int accept_all, double max_loss,
                     int A, int B, int *plan, int *cost) {
#define DD(x, y) dist[(int64_t)(x) * S + (y)]
    if (A == B || from[A] < 0 || from[B] < 0) return 0;
    int ok = accept_all != 0;
    int cost1 = DD(from[A], from[B]) + DD(from[B], to[A]) + DD(to[A], to[B]);
    int cost2 = DD(from[A], from[B]) + DD(from[B], to[B]) + DD(to[B], to[A]);
    if (DD(from[B], to[A]) + DD(to[A], to[B]) < DD(from[B], to[B]) * max_loss &&
        DD(from[A], from[B]) + DD(from[B], to[A]) < DD(from[A], to[A]) * max_loss) ok = 1;
    if (cost2 < DD(from[A], to[A]) * max_loss) ok = 1;
#undef DD
    if (!ok) return 0;
    *plan = cost1 < cost2 ? 1 : 0;
    *cost = cost1 < cost2 ? cost1 : cost2;
    return 1;
}

static int cmp_row(const void *a, const void *b) {
    const int64_t *x = (const int64_t *)a, *y = (const int64_t *)b;
    return x[0] < y[0] ? -1 : x[0] > y[0] ? 1 : (x[1] < y[1] ? -1 : x[1] > y[1]);
}

/* Returns 0; -1 on allocation failure; -2 when a live row names a stand outside the table (the instance is
 * withdrawn).  out: rows [custA, custB, plan, cost] in (cost, A*n+B) order, at most n/2 of them. */
int pairs_exact_oracle(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int S, int accept_all,
                       double max_loss, int32_t *out, int32_t *n_pairs_out, int64_t *total_out) {
    for (int i = 0; i < n; i++)
        if (from[i] >= 0 && (from[i] >= S || to[i] < 0 || to[i] >= S)) return -2;
    const int64_t K = (int64_t)(n / 2) * 3 * (1 << 22) + 1;
    int64_t *W = (int64_t *)calloc((size_t)(n > 0 ? n : 1) * (n > 0 ? n : 1), sizeof(int64_t));
    int32_t *pref = (int32_t *)malloc(sizeof(int32_t) * 3 * (size_t)(n > 0 ? n : 1) * (n > 0 ? n : 1));
    int *mate = (int *)malloc(sizeof(int) * (size_t)(n > 0 ? n : 1));
    int64_t *rows = (int64_t *)malloc(sizeof(int64_t) * 2 * (size_t)(n / 2 + 1));
    if (!W || !pref || !mate || !rows) { free(W); free(pref); free(mate); free(rows); return -1; }
    for (int i = 0; i < n; i++)
        for (int j = i + 1; j < n; j++) {
            int p1 = 0, c1 = 0, p2 = 0, c2 = 0;
            int a1 = candidate(from, to, dist, S, accept_all, max_loss, i, j, &p1, &c1);
            int a2 = candidate(from, to, dist, S, accept_all, max_loss, j, i, &p2, &c2);
            if (!a1 && !a2) continue;
            /* preferred candidate: smallest (cost, A*n+B); (i, j) has the smaller key at equal cost */
            int use1 = a1 && (!a2 || c1 <= c2);
            int32_t *r = pref + 3 * ((int64_t)i * n + j);
            r[0] = use1 ? i : j; r[1] = use1 ? p1 : p2; r[2] = use1 ? c1 : c2;
            W[(int64_t)i * n + j] = W[(int64_t)j * n + i] = K - r[2];
        }
    int rc = blossom(n, W, mate);
    if (rc == 0) {
        int m = 0;
        int64_t total = 0;
        for (int i = 0; i < n; i++) {
            int j = mate[i];
            if (j <= i) continue;
            const int32_t *r = pref + 3 * ((int64_t)i * n + j);
            int A = r[0], B = A == i ? j : i;
            rows[2 * m] = r[2]; rows[2 * m + 1] = (int64_t)A * n + B;
            total += r[2];
            m++;
        }
        qsort(rows, (size_t)m, 2 * sizeof(int64_t), cmp_row);
        for (int k = 0; k < m; k++) {
            int A = (int)(rows[2 * k + 1] / n), B = (int)(rows[2 * k + 1] % n);
            int i = A < B ? A : B, j = A < B ? B : A;
            out[4 * k] = A; out[4 * k + 1] = B; out[4 * k + 2] = pref[3 * ((int64_t)i * n + j) + 1]; out[4 * k + 3] = (int32_t)rows[2 * k];
        }
        *n_pairs_out = m;
        *total_out = total;
    }
    free(W); free(pref); free(mate); free(rows);
    return rc;
}
