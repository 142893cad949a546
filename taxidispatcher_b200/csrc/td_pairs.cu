// td_pairs.cu -- exact 2-passenger pool: minimum-cost maximum-cardinality pair matching, batched, one CTA per instance;
// and the Simulator's greedy 2-passenger pool over the same batch layout and edges (pairs_greedy_kernel, at the end).
//
// The greedy of Simulator.findPool (td_pool.cu, pool_pairs_*) stable-sorts the accepted candidates by cost and scans them
// for disjoint pairs.  Its exact counterpart (the ILP of the reference's pool_optimum.py / pool_opt_min.py, where every
// customer sits in exactly one pair) is a general -- non-bipartite -- matching problem.  This file solves it with the
// O(n^3) primal-dual weighted blossom algorithm (Edmonds / Galil) in the van Rantwijk formulation that networkx ships
// as max_weight_matching: stages, S/T labels, per-blossom least-slack edges and the four dual step cases.
//
// Graph.  Vertex i = customer i of the instance; {i, j} is an edge when at least one of the ordered candidates (i, j),
// (j, i) is accepted exactly as pool_pairs_enum_kernel accepts it; its cost is the smaller accepted candidate cost.
// Costs are recomputed from the stand table staged in shared memory -- nothing of size n^2 is stored.
//
// Objective.  Edge weight w = K - cost with K = floor(n/2) * 3 * 2^22 + 1.  A cost is at most three stand distances of
// at most 2^22, so K > floor(n/2) * (c_max - c_min) + c_max: a matching with one more pair always weighs more, and the
// maximum-weight matching is a maximum-cardinality matching of minimum total cost.  Duals are doubled as in networkx
// (slack = u_i + u_j - 2 w_ij) and all arithmetic is int64; K < 2^35 at n = 4096, so every dual and slack stays far
// below the 2^39 the packed reduction keys leave for them.
//
// Parallel split.  The O(n) loops run block-parallel with (value, index) min-reductions, so the result never depends on
// timing: the neighbour scan of a vertex that became S (slack, least-slack edge refresh, tight-edge search), the least-
// slack edge of a new blossom, the four delta minima and the dual update.  Tree, blossom and augmentation surgery is
// sequential, done by thread 0.  State is O(n) per instance in a global workspace slice (see DESIGN.md section 12).
#include "td_common.cuh"
#include <cmath>

namespace td {

constexpr int kPairsThreads = 256;
constexpr int kPairsMaxStands = 128;
constexpr int kPairsMaxDist = 1 << 22;
constexpr unsigned long long kNone = ~0ull;

// per-instance workspace slice; every array is sized by n_max so that slices have one stride
struct PairsWs {
    int *mate, *label, *lex, *ley, *inb, *bpar, *bbase, *bfirst, *nchild, *cnext, *cprev, *cex, *cey, *bex, *bey;
    int *queue, *freeb, *stk, *tmp, *leaves;
    long long *dual;
    unsigned long long *keys;
    size_t bytes;
};

// the same 256-byte aligned slicing as Carver, callable from the kernel that finds its own slice
struct PairsCarver {
    char *base; size_t off;
    template <typename T> __host__ __device__ T *take(size_t count) {
        off = (off + 255) & ~size_t(255);
        T *p = reinterpret_cast<T *>(base + off);
        off += count * sizeof(T);
        return p;
    }
};

__host__ __device__ static PairsWs carve_pairs(void *base, int n_max) {
    PairsCarver c{static_cast<char *>(base), 0};
    PairsWs w;
    const size_t N = n_max > 0 ? size_t(n_max) : 1, N2 = 2 * N;
    int **two[] = {&w.label, &w.lex, &w.ley, &w.inb, &w.bpar, &w.bbase, &w.bfirst, &w.nchild, &w.cnext, &w.cprev, &w.cex,
                   &w.cey, &w.bex, &w.bey, &w.queue, &w.freeb};
    for (int **p : two) *p = c.take<int>(N2);
    w.mate = c.take<int>(N);
    w.stk = c.take<int>(2 * N2);
    w.tmp = c.take<int>(6 * N2);
    w.leaves = c.take<int>(N);
    w.dual = c.take<long long>(N2);
    w.keys = c.take<unsigned long long>(N);
    w.bytes = (c.off + 255) & ~size_t(255);
    return w;
}

// what defines the edges of an instance; shared by the exact kernel and the greedy batch kernel
struct PairsEdges {
    int S, accept_all;
    double max_loss;
    const int32_t *dist, *from, *to;   // shared memory
};

struct PairsCtx : PairsEdges {
    PairsWs w;
    int n, qn, nfree;
    long long K;
};

// accepted candidate (A first picked up, then B) -> cost, or -1; plan as in pool_pairs_enum_kernel
__device__ __forceinline__ int candidate(const PairsEdges &m, int A, int B, int *plan) {
    const int S = m.S, fa = m.from[A], ta = m.to[A], fb = m.from[B], tb = m.to[B];
    const int32_t *d = m.dist;
    const int dab = d[fa * S + fb];
    const int cost1 = dab + d[fb * S + ta] + d[ta * S + tb];
    const int cost2 = dab + d[fb * S + tb] + d[tb * S + ta];
    if (!m.accept_all) {
        const double dB = double(d[fb * S + tb]), dA = double(d[fa * S + ta]);
        const bool plan1 = double(d[fb * S + ta] + d[ta * S + tb]) < __dmul_rn(dB, m.max_loss) &&
                           double(dab + d[fb * S + ta]) < __dmul_rn(dA, m.max_loss);
        const bool plan2 = double(cost2) < __dmul_rn(dA, m.max_loss);
        if (!(plan1 || plan2)) return -1;
    }
    *plan = cost1 < cost2 ? 1 : 0;
    return cost1 < cost2 ? cost1 : cost2;
}

// edge {i, j}: the cost of the preferred accepted candidate (smallest (cost, A*n+B)), or -1 when there is no edge
__device__ __forceinline__ int edge_cost(const PairsEdges &m, int i, int j, int *A_out = nullptr, int *plan_out = nullptr) {
    if (i == j || m.from[i] < 0 || m.from[j] < 0) return -1;
    const int lo = i < j ? i : j, hi = i < j ? j : i;
    int p1 = 0, p2 = 0;
    const int c1 = candidate(m, lo, hi, &p1), c2 = candidate(m, hi, lo, &p2);
    if (c1 < 0 && c2 < 0) return -1;
    const bool first = c1 >= 0 && (c2 < 0 || c1 <= c2);      // (lo, hi) has the smaller A*n+B at equal cost
    if (A_out) *A_out = first ? lo : hi;
    if (plan_out) *plan_out = first ? p1 : p2;
    return first ? c1 : c2;
}

__device__ __forceinline__ long long slack_c(const PairsCtx &m, int v, int w, int cost) {
    return m.w.dual[v] + m.w.dual[w] - 2 * (m.K - cost);
}

__device__ __forceinline__ long long slack(const PairsCtx &m, int v, int w) { return slack_c(m, v, w, edge_cost(m, v, w)); }

__device__ __forceinline__ unsigned long long block_min(unsigned long long v, unsigned long long *red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o; o >>= 1) { const unsigned long long x = __shfl_xor_sync(0xffffffffu, v, o); v = x < v ? x : v; }
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        v = lane < int(blockDim.x >> 5) ? red[lane] : kNone;
        for (int o = 16; o; o >>= 1) { const unsigned long long x = __shfl_xor_sync(0xffffffffu, v, o); v = x < v ? x : v; }
        if (lane == 0) red[32] = v;
    }
    __syncthreads();
    v = red[32];
    __syncthreads();
    return v;
}

// ---- sequential surgery (thread 0) ----------------------------------------------------------------------------------
__device__ void push_leaves(PairsCtx &m, int b) {
    if (b < m.n) { m.w.queue[m.qn++] = b; return; }
    for (int v = 0; v < m.n; ++v) if (m.w.inb[v] == b) m.w.queue[m.qn++] = v;
}

__device__ void assign_label(PairsCtx &m, int w, int t, int v) {
    PairsWs &s = m.w;
    for (;;) {
        const int b = s.inb[w];
        s.label[w] = s.label[b] = t;
        s.lex[w] = s.lex[b] = v;
        s.ley[w] = s.ley[b] = v >= 0 ? w : -1;
        s.bex[w] = s.bex[b] = -1;
        s.bey[w] = s.bey[b] = -1;
        if (t == 1) { push_leaves(m, b); return; }
        const int base = s.bbase[b];                 // a T-blossom's base is matched: its mate becomes S
        w = s.mate[base]; t = 1; v = base;
    }
}

__device__ int scan_blossom(PairsCtx &m, int v, int w) {
    PairsWs &s = m.w;
    int np = 0, base = -1;
    while (v != -1) {
        int b = s.inb[v];
        if (s.label[b] & 4) { base = s.bbase[b]; break; }
        s.tmp[np++] = b;
        s.label[b] = 5;
        if (s.lex[b] == -1) v = -1;
        else { v = s.lex[b]; b = s.inb[v]; v = s.lex[b]; }
        if (w != -1) { const int t = v; v = w; w = t; }
    }
    for (int i = 0; i < np; ++i) s.label[s.tmp[i]] = 1;
    return base;
}

// builds blossom b over the cycle base .. v - w .. base; returns its leaf count (the leaves are listed in s.leaves)
__device__ int add_blossom(PairsCtx &m, int base, int v, int w, int *b_out) {
    PairsWs &s = m.w;
    const int n = m.n;
    int bb = s.inb[base], bv = s.inb[v], bw = s.inb[w];
    const int b = s.freeb[--m.nfree];
    s.bbase[b] = base; s.bpar[b] = -1; s.bpar[bb] = b;
    int *ch = s.tmp, *ex = s.tmp + 2 * n, *ey = s.tmp + 4 * n, *c2 = s.tmp + 6 * n, *x2 = s.tmp + 8 * n, *y2 = s.tmp + 10 * n;
    int k = 0;
    while (bv != bb) {
        s.bpar[bv] = b;
        ch[k] = bv; ex[k] = s.lex[bv]; ey[k] = s.ley[bv]; ++k;
        bv = s.inb[s.lex[bv]];
    }
    int L = 0;
    c2[0] = bb;
    for (int i = k - 1; i >= 0; --i) { c2[L + 1] = ch[i]; x2[L] = ex[i]; y2[L] = ey[i]; ++L; }
    x2[L] = v; y2[L] = w; ++L;
    while (bw != bb) {
        s.bpar[bw] = b;
        c2[L] = bw; x2[L] = s.ley[bw]; y2[L] = s.lex[bw]; ++L;
        bw = s.inb[s.lex[bw]];
    }
    for (int i = 0; i < L; ++i) {
        const int c = c2[i], d = c2[i + 1 < L ? i + 1 : 0];
        s.cnext[c] = d; s.cprev[d] = c; s.cex[c] = x2[i]; s.cey[c] = y2[i];
        s.bex[c] = s.bey[c] = -1;
    }
    s.bfirst[b] = bb; s.nchild[b] = L;
    s.label[b] = 1; s.lex[b] = s.lex[bb]; s.ley[b] = s.ley[bb]; s.dual[b] = 0;
    int nl = 0;
    for (int u = 0; u < n; ++u) {
        const int t = s.inb[u];
        if (t != b && s.bpar[t] == b) {
            if (s.label[t] == 2) s.queue[m.qn++] = u;
            s.inb[u] = b;
            s.leaves[nl++] = u;
        }
    }
    *b_out = b;
    return nl;
}

// expands top-level blossom b; at the end of a stage (endstage) sub-blossoms with zero dual are expanded too
__device__ void expand_blossom(PairsCtx &m, int b, bool endstage) {
    PairsWs &s = m.w;
    const int n = m.n;
    // new top-level blossom of every leaf: the highest node below b on its parent chain that stays a blossom
    for (int v = 0; v < n; ++v) {
        if (s.inb[v] != b) continue;
        int top = v;
        for (int t = v; t != b; t = s.bpar[t])
            if (t < n || !endstage || s.dual[t] != 0) top = t;
        s.inb[v] = top;
    }
    // release b (and, at the end of a stage, its zero-dual descendants): their children become top level
    int sp = 0;
    s.stk[sp++] = b;
    while (sp) {
        const int x = s.stk[--sp];
        int c = s.bfirst[x];
        for (int i = 0; i < s.nchild[x]; ++i, c = s.cnext[c]) {
            s.bpar[c] = -1;
            if (c >= n && endstage && s.dual[c] == 0) s.stk[sp++] = c;
        }
        if (x != b) { s.label[x] = 0; s.lex[x] = s.ley[x] = -1; s.bex[x] = s.bey[x] = -1; s.bbase[x] = -1; s.freeb[m.nfree++] = x; }
    }
    if (!endstage && s.label[b] == 2) {
        // relabel the even-length path from the entry child to the base; the other children lose their labels
        const int L = s.nchild[b];
        const int entry = s.inb[s.ley[b]];
        int j = 0, c;
        for (c = s.bfirst[b]; c != entry; c = s.cnext[c]) ++j;
        int jstep;
        if (j & 1) { j -= L; jstep = 1; } else jstep = -1;
        int v = s.lex[b], w = s.ley[b];
        while (j != 0) {
            const int q = jstep == 1 ? s.cey[c] : s.cex[s.cprev[c]];
            s.label[w] = 0; s.label[q] = 0;
            assign_label(m, w, 2, v);
            j += jstep; c = jstep == 1 ? s.cnext[c] : s.cprev[c];
            if (jstep == 1) { v = s.cex[c]; w = s.cey[c]; }
            else { w = s.cex[s.cprev[c]]; v = s.cey[s.cprev[c]]; }
            j += jstep; c = jstep == 1 ? s.cnext[c] : s.cprev[c];
        }
        const int bw = c;
        s.label[w] = s.label[bw] = 2;
        s.lex[w] = s.lex[bw] = v; s.ley[w] = s.ley[bw] = w;
        s.bex[bw] = s.bey[bw] = -1;
        c = jstep == 1 ? s.cnext[c] : s.cprev[c];
        while (c != entry) {
            const int bv = c;
            c = jstep == 1 ? s.cnext[c] : s.cprev[c];
            if (s.label[bv] == 1) continue;
            int u = bv;
            if (bv >= n) {
                u = -1;
                for (int x = 0; x < n; ++x) if (s.label[x] && s.inb[x] == bv) { u = x; break; }
            }
            if (u >= 0 && s.label[u]) {
                s.label[u] = 0;
                s.label[s.mate[s.bbase[bv]]] = 0;
                assign_label(m, u, 2, s.lex[u]);
            }
        }
    }
    s.label[b] = 0; s.lex[b] = s.ley[b] = -1; s.bex[b] = s.bey[b] = -1;
    s.bpar[b] = -1; s.bbase[b] = -1; s.dual[b] = 0;
    s.freeb[m.nfree++] = b;
}

// flips the alternating path inside blossom b so that vertex v becomes its base; sub-blossoms are independent of the
// parent's path, so they are handled from a work list instead of by recursion
__device__ void augment_blossom(PairsCtx &m, int b0, int v0) {
    PairsWs &s = m.w;
    const int n = m.n;
    int sp = 0;
    s.stk[sp++] = b0; s.stk[sp++] = v0;
    while (sp) {
        const int v = s.stk[--sp], b = s.stk[--sp];
        int t = v;
        while (s.bpar[t] != b) t = s.bpar[t];
        if (t >= n) { s.stk[sp++] = t; s.stk[sp++] = v; }
        const int L = s.nchild[b];
        int i = 0, c;
        for (c = s.bfirst[b]; c != t; c = s.cnext[c]) ++i;
        int j = i, jstep;
        if (i & 1) { j -= L; jstep = 1; } else jstep = -1;
        while (j != 0) {
            int w, x;
            j += jstep; c = jstep == 1 ? s.cnext[c] : s.cprev[c];
            if (jstep == 1) { w = s.cex[c]; x = s.cey[c]; }
            else { x = s.cex[s.cprev[c]]; w = s.cey[s.cprev[c]]; }
            if (c >= n) { s.stk[sp++] = c; s.stk[sp++] = w; }
            j += jstep; c = jstep == 1 ? s.cnext[c] : s.cprev[c];
            if (c >= n) { s.stk[sp++] = c; s.stk[sp++] = x; }
            s.mate[w] = x; s.mate[x] = w;
        }
        s.bfirst[b] = t;
        s.bbase[b] = v;
    }
}

__device__ void augment_matching(PairsCtx &m, int v, int w) {
    PairsWs &s = m.w;
    for (int side = 0; side < 2; ++side) {
        int a = side ? w : v, j = side ? v : w;
        for (;;) {
            const int bs = s.inb[a];
            if (bs >= m.n) augment_blossom(m, bs, a);
            s.mate[a] = j;
            if (s.lex[bs] == -1) break;
            const int t = s.lex[bs], bt = s.inb[t];
            a = s.lex[bt]; j = s.ley[bt];
            if (bt >= m.n) augment_blossom(m, bt, j);
            s.mate[j] = a;
        }
    }
}

// ---- the kernels ------------------------------------------------------------------------------------------------------
// Stages instance blockIdx.x (the stand table, its from / to) in shared memory and returns its size.  A withdrawn
// instance (bad size or offset, a live row whose stand lies outside the table, a table entry outside [0, 2^22]) gets its
// outputs here and -1 back; the neighbours are unaffected.  The `to` of a removed row (from < 0) is never read.
__device__ int stage_instance(const int32_t *__restrict__ from, const int32_t *__restrict__ to,
                              const int32_t *__restrict__ sizes, const int64_t *__restrict__ offsets, int n_max,
                              const int32_t *__restrict__ dist, int S, int32_t *s_dist, int32_t *s_from, int32_t *s_to,
                              int32_t *rows, int32_t *n_pairs_out, long long *cost_out, int *s_bad) {
    const int tid = threadIdx.x, inst = blockIdx.x;
    const int n = sizes[inst];
    const long long off = offsets[inst];
    if (tid == 0) *s_bad = (n < 0 || n > n_max || off < 0) ? 1 : 0;
    __syncthreads();
    if (!*s_bad) {
        for (int k = tid; k < S * S; k += blockDim.x) {
            const int d = dist[k];
            if (d < 0 || d > kPairsMaxDist) *s_bad = 1;
            s_dist[k] = d;
        }
        for (int i = tid; i < n; i += blockDim.x) {
            const int f = from[off + i], t = f >= 0 ? to[off + i] : -1;
            if (f >= 0 && (f >= S || t < 0 || t >= S)) *s_bad = 1;
            s_from[i] = f; s_to[i] = t;
        }
    }
    __syncthreads();
    if (*s_bad) {
        const int rows_cap = n_max / 2;
        for (int k = tid; k < rows_cap * 4; k += blockDim.x) rows[k] = -1;
        if (tid == 0) { n_pairs_out[inst] = -1; cost_out[inst] = LLONG_MIN; }
        return -1;
    }
    return n;
}

// Key layouts of the min-reductions: edge keys (slack << 24 | v << 12 | w), delta keys (delta << 16 | type << 13 | index).
__device__ __forceinline__ unsigned long long edge_key(long long sl, int v, int w) {
    return (unsigned long long)sl << 24 | (unsigned long long)v << 12 | unsigned(w);
}

__global__ void __launch_bounds__(kPairsThreads)
pairs_exact_kernel(const int32_t *__restrict__ from, const int32_t *__restrict__ to, const int32_t *__restrict__ sizes,
                   const int64_t *__restrict__ offsets, int n_max, const int32_t *__restrict__ dist, int S, int accept_all,
                   double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, long long *cost_out, char *workspace,
                   size_t stride) {
    extern __shared__ int32_t smem[];
    __shared__ unsigned long long red[33];
    __shared__ int s_bad, s_v, s_aug, s_newb, s_nleaf, s_m;
    __shared__ long long s_total;
    const int tid = threadIdx.x, inst = blockIdx.x;
    const int rows_cap = n_max / 2;
    int32_t *rows = pairs_out + size_t(inst) * rows_cap * 4;
    int32_t *s_dist = smem, *s_from = smem + S * S, *s_to = s_from + (n_max > 0 ? n_max : 1);
    const int n = stage_instance(from, to, sizes, offsets, n_max, dist, S, s_dist, s_from, s_to, rows, n_pairs_out, cost_out,
                                 &s_bad);
    if (n < 0) return;

    PairsCtx m;
    m.w = carve_pairs(workspace + size_t(inst) * stride, n_max);
    m.n = n; m.S = S; m.accept_all = accept_all; m.max_loss = max_loss;
    m.K = (long long)(n / 2) * 3 * (1ll << 22) + 1;
    m.dist = s_dist; m.from = s_from; m.to = s_to;
    m.qn = 0; m.nfree = n;
    PairsWs &s = m.w;

    // largest weight = K - the cheapest edge (networkx starts every vertex dual there)
    unsigned long long cmin = kNone;
    for (long long k = tid; k < (long long)n * n; k += blockDim.x) {
        const int i = int(k / n), j = int(k - (long long)i * n);
        if (i < j) {
            const int c = edge_cost(m, i, j);
            if (c >= 0 && (unsigned long long)c < cmin) cmin = (unsigned long long)c;
        }
    }
    cmin = block_min(cmin, red);
    const long long maxw = cmin == kNone ? 0 : m.K - (long long)cmin;
    for (int v = tid; v < 2 * n; v += blockDim.x) {
        s.label[v] = 0; s.lex[v] = s.ley[v] = -1; s.bpar[v] = -1; s.bex[v] = s.bey[v] = -1;
        s.bbase[v] = v < n ? v : -1; s.inb[v] = v; s.nchild[v] = 0;
        s.dual[v] = v < n ? maxw : 0;
        if (v < n) { s.mate[v] = -1; s.freeb[v] = 2 * n - 1 - v; }
    }
    __syncthreads();

    for (;;) {                                                 // stages: each ends with one augmentation or the optimum
        for (int b = tid; b < 2 * n; b += blockDim.x) { s.label[b] = 0; s.lex[b] = s.ley[b] = -1; s.bex[b] = s.bey[b] = -1; }
        __syncthreads();
        if (tid == 0) {
            m.qn = 0;
            for (int v = 0; v < n; ++v)
                if (s.mate[v] == -1 && s.label[s.inb[v]] == 0) assign_label(m, v, 1, -1);
            s_aug = 0;
        }
        __syncthreads();
        for (;;) {
            // ---- scan the S-vertices of the queue (LIFO, as networkx) ----
            for (;;) {
                if (tid == 0) { s_v = (m.qn > 0 && !s_aug) ? s.queue[--m.qn] : -1; }
                __syncthreads();
                const int v = s_v;
                if (v < 0) break;
                const int bv = s.inb[v];
                // pass 1: least-slack refresh for non-tight edges, first actionable tight edge
                unsigned long long ss = kNone, tight = kNone;
                for (int w = tid; w < n; w += blockDim.x) {
                    const int c = edge_cost(m, v, w);
                    if (c < 0) continue;
                    const int bw = s.inb[w];
                    if (bw == bv) continue;
                    const long long ks = slack_c(m, v, w, c);
                    if (ks <= 0) {
                        if (!(s.label[bw] == 2 && s.label[w] != 0) && (unsigned long long)w < tight) tight = w;
                    } else if (s.label[bw] == 1) {
                        const unsigned long long k = edge_key(ks, v, w);
                        ss = k < ss ? k : ss;
                    } else if (s.label[w] == 0) {
                        if (s.bex[w] == -1 || ks < slack(m, s.bex[w], s.bey[w])) { s.bex[w] = v; s.bey[w] = w; }
                    }
                }
                ss = block_min(ss, red);
                tight = block_min(tight, red);
                if (tid == 0 && ss != kNone) {
                    const int w = int(ss & 4095);
                    const long long ks = (long long)(ss >> 24);
                    if (s.bex[bv] == -1 || ks < slack(m, s.bex[bv], s.bey[bv])) { s.bex[bv] = v; s.bey[bv] = w; }
                }
                // tight edges in index order, each handled with the labels of the moment
                while (tight != kNone) {
                    const int w = int(tight);
                    if (tid == 0) {
                        s_newb = -1;
                        const int bv2 = s.inb[v], bw = s.inb[w];
                        if (bv2 != bw) {
                            if (s.label[bw] == 0) assign_label(m, w, 2, v);
                            else if (s.label[bw] == 1) {
                                const int base = scan_blossom(m, v, w);
                                if (base != -1) { int b; s_nleaf = add_blossom(m, base, v, w, &b); s_newb = b; }
                                else { augment_matching(m, v, w); s_aug = 1; }
                            } else if (s.label[w] == 0) { s.label[w] = 2; s.lex[w] = v; s.ley[w] = w; }
                        }
                    }
                    __syncthreads();
                    const int nb = s_newb;
                    if (nb >= 0) {                             // least-slack edge from the new blossom to another S-blossom
                        const long long work = (long long)s_nleaf * n;
                        unsigned long long best = kNone;
                        for (long long k = tid; k < work; k += blockDim.x) {
                            const int i = s.leaves[int(k / n)], j = int(k % n);
                            if (s.inb[j] == nb || s.label[s.inb[j]] != 1) continue;
                            const int c = edge_cost(m, i, j);
                            if (c < 0) continue;
                            const unsigned long long key = edge_key(slack_c(m, i, j, c), i, j);
                            best = key < best ? key : best;
                        }
                        best = block_min(best, red);
                        if (tid == 0 && best != kNone) { s.bex[nb] = int((best >> 12) & 4095); s.bey[nb] = int(best & 4095); }
                    }
                    if (s_aug) break;
                    // next actionable tight edge after w
                    unsigned long long nt = kNone;
                    const int bvn = s.inb[v];
                    for (int x = w + 1 + tid; x < n; x += blockDim.x) {
                        const int c = edge_cost(m, v, x);
                        if (c < 0) continue;
                        const int bx = s.inb[x];
                        if (bx == bvn || slack_c(m, v, x, c) > 0) continue;
                        if (!(s.label[bx] == 2 && s.label[x] != 0)) { nt = x; break; }
                    }
                    tight = block_min(nt, red);
                }
                __syncthreads();
                if (s_aug) break;
            }
            if (s_aug) break;
            // ---- dual step: the smallest of the four deltas, ties to the lower case, then the lower index ----
            unsigned long long dk = kNone;
            for (int v = tid; v < n; v += blockDim.x) {
                const unsigned long long k1 = (unsigned long long)s.dual[v] << 16 | 1ull << 13;
                dk = k1 < dk ? k1 : dk;
                if (s.label[s.inb[v]] == 0 && s.bex[v] != -1) {
                    const unsigned long long k2 = (unsigned long long)slack(m, s.bex[v], s.bey[v]) << 16 | 2ull << 13 | unsigned(v);
                    dk = k2 < dk ? k2 : dk;
                }
            }
            for (int b = tid; b < 2 * n; b += blockDim.x) {
                if (s.bbase[b] == -1 || s.bpar[b] != -1) continue;
                if (s.label[b] == 1 && s.bex[b] != -1) {
                    const unsigned long long k3 = (unsigned long long)(slack(m, s.bex[b], s.bey[b]) / 2) << 16 | 3ull << 13 | unsigned(b);
                    dk = k3 < dk ? k3 : dk;
                }
                if (b >= n && s.label[b] == 2) {
                    const unsigned long long k4 = (unsigned long long)s.dual[b] << 16 | 4ull << 13 | unsigned(b);
                    dk = k4 < dk ? k4 : dk;
                }
            }
            dk = block_min(dk, red);
            if (dk == kNone) break;                            // no vertex at all (n = 0): nothing to match
            const long long delta = (long long)(dk >> 16);
            const int dtype = int((dk >> 13) & 7), didx = int(dk & 8191);
            for (int v = tid; v < n; v += blockDim.x) {
                const int l = s.label[s.inb[v]];
                if (l == 1) s.dual[v] -= delta; else if (l == 2) s.dual[v] += delta;
            }
            for (int b = n + tid; b < 2 * n; b += blockDim.x)
                if (s.bbase[b] != -1 && s.bpar[b] == -1) {
                    if (s.label[b] == 1) s.dual[b] += delta; else if (s.label[b] == 2) s.dual[b] -= delta;
                }
            __syncthreads();
            if (dtype == 1) break;                             // a free vertex reached dual 0: optimum
            if (tid == 0) {
                if (dtype == 2 || dtype == 3) s.queue[m.qn++] = s.bex[didx];
                else expand_blossom(m, didx, false);
            }
            __syncthreads();
        }
        __syncthreads();
        if (!s_aug) break;
        if (tid == 0)
            for (int b = n; b < 2 * n; ++b)
                if (s.bbase[b] != -1 && s.bpar[b] == -1 && s.label[b] == 1 && s.dual[b] == 0) expand_blossom(m, b, true);
        __syncthreads();
    }

    // ---- output: the preferred row of every pair, in (cost, A*n+B) order ----
    if (tid == 0) { s_m = 0; s_total = 0; }
    __syncthreads();
    long long part = 0;
    for (int i = tid; i < n; i += blockDim.x) {
        const int j = s.mate[i];
        if (j <= i) continue;
        int A, plan;
        const int c = edge_cost(m, i, j, &A, &plan);
        const int B = A == i ? j : i;
        const int slot = atomicAdd(&s_m, 1);
        s.keys[slot] = (unsigned long long)c << 26 | (unsigned long long)plan << 25 | (unsigned long long)(A * n + B);
        part += c;
    }
    atomicAdd(reinterpret_cast<unsigned long long *>(&s_total), (unsigned long long)part);
    __syncthreads();
    const int npairs = s_m;
    for (int k = tid; k < npairs; k += blockDim.x) {
        const unsigned long long me = s.keys[k], mine = me & ~(1ull << 25);
        int rank = 0;
        for (int q = 0; q < npairs; ++q) rank += (s.keys[q] & ~(1ull << 25)) < mine;
        const int ab = int(me & ((1u << 25) - 1));
        int32_t *r = rows + size_t(rank) * 4;
        r[0] = ab / n; r[1] = ab % n; r[2] = int((me >> 25) & 1); r[3] = int(me >> 26);
    }
    for (int k = npairs * 4 + tid; k < rows_cap * 4; k += blockDim.x) rows[k] = -1;
    if (tid == 0) { n_pairs_out[inst] = npairs; cost_out[inst] = s_total; }
}

// ---- the greedy of Simulator.findPool, batched (see DESIGN.md section 14) ---------------------------------------------
// td_pool_pairs stable-sorts the accepted ordered candidates by cost and keeps every pair whose customers are both still
// free.  Per unordered pair only its preferred candidate (smallest (cost, A*n+B), edge_cost) can be kept, so this is the
// greedy matching under the strict edge order key = cost << 24 | A*n+B (cost <= 3 * 2^22 < 2^24, A*n+B < 2^24).  With
// distinct keys it equals dominance rounds: an edge that is the smallest live edge at both ends is kept by the scan
// (every smaller edge misses both ends), and removing its two customers leaves the scan of the rest unchanged.  Every
// live customer caches its smallest live edge; a round keeps all mutual bests, then rescans only the customers whose
// cached partner died.  A round that keeps nothing means no live edge is left (the smallest one is always mutual).
__device__ __forceinline__ unsigned long long greedy_key(const PairsEdges &e, int n, int i, int j) {
    int A;
    const int c = edge_cost(e, i, j, &A);
    return c < 0 ? kNone : (unsigned long long)c << 24 | unsigned(A * n + (A == i ? j : i));
}

__device__ __forceinline__ int key_partner(unsigned long long key, int n, int i) {
    const int ab = int(key & 0xffffff), A = ab / n;
    return A == i ? ab - A * n : A;
}

__global__ void __launch_bounds__(1024)
pairs_greedy_kernel(const int32_t *__restrict__ from, const int32_t *__restrict__ to, const int32_t *__restrict__ sizes,
                    const int64_t *__restrict__ offsets, int n_max, const int32_t *__restrict__ dist, int S, int accept_all,
                    double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, long long *cost_out) {
    extern __shared__ unsigned long long smem64[];
    __shared__ int s_bad, s_m, s_nlive, s_nscan;
    __shared__ long long s_total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5, inst = blockIdx.x;
    const int rows_cap = n_max / 2, N = n_max > 0 ? n_max : 1;
    int32_t *rows = pairs_out + size_t(inst) * rows_cap * 4;
    unsigned long long *best = smem64, *kept = best + N;               // kept: n_max / 2 + 1 keys
    int32_t *s_dist = reinterpret_cast<int32_t *>(kept + N / 2 + 1), *s_from = s_dist + S * S, *s_to = s_from + N;
    int32_t *live = s_to + N, *live_next = s_to + 2 * N, *scan = s_to + 3 * N;
    uint8_t *alive = reinterpret_cast<uint8_t *>(s_to + 4 * N);
    const int n = stage_instance(from, to, sizes, offsets, n_max, dist, S, s_dist, s_from, s_to, rows, n_pairs_out, cost_out,
                                 &s_bad);
    if (n < 0) return;
    PairsEdges e;
    e.S = S; e.accept_all = accept_all; e.max_loss = max_loss; e.dist = s_dist; e.from = s_from; e.to = s_to;

    // every customer that is not a removed row is live and scans once
    if (tid == 0) { s_m = 0; s_total = 0; s_nlive = 0; }
    __syncthreads();
    for (int i = tid; i < n; i += blockDim.x) {
        alive[i] = s_from[i] >= 0;
        if (alive[i]) { const int k = atomicAdd(&s_nlive, 1); live[k] = i; scan[k] = i; }
    }
    __syncthreads();
    int nlive = s_nlive, nscan = nlive, kept_before = 0;
    for (;;) {
        // rescan: one warp per customer, min over the live list (its order does not matter to a minimum).  A customer
        // left out of the list is dead or had no live edge when it last scanned, so it has no edge to anyone live now.
        for (int k = warp; k < nscan; k += nwarps) {
            const int i = scan[k];
            unsigned long long b = kNone;
            for (int q = lane; q < nlive; q += 32) {
                const int j = live[q];
                if (j == i) continue;
                const unsigned long long key = greedy_key(e, n, i, j);
                b = key < b ? key : b;
            }
            b = warp_min_u64(b);
            if (lane == 0) best[i] = b;
        }
        __syncthreads();
        // keep every mutual best; the customer with the lower index records the pair
        if (tid == 0) { s_nlive = 0; s_nscan = 0; }
        for (int k = tid; k < nlive; k += blockDim.x) {
            const int i = live[k];
            const unsigned long long b = best[i];
            if (b == kNone) continue;
            const int p = key_partner(b, n, i);
            if (best[p] != b) continue;
            alive[i] = 0;
            if (i < p) kept[atomicAdd(&s_m, 1)] = b;
        }
        __syncthreads();
        if (s_m == kept_before) break;                                 // no mutual best: no live edge is left
        kept_before = s_m;
        // next live list: customers that are alive and still have an edge; rescan those whose partner died
        for (int k = tid; k < nlive; k += blockDim.x) {
            const int i = live[k];
            const unsigned long long b = best[i];
            if (!alive[i] || b == kNone) continue;
            live_next[atomicAdd(&s_nlive, 1)] = i;
            if (!alive[key_partner(b, n, i)]) scan[atomicAdd(&s_nscan, 1)] = i;
        }
        __syncthreads();
        int32_t *const t = live; live = live_next; live_next = t;
        nlive = s_nlive;
        nscan = s_nscan;
    }

    // ---- output: the kept pairs in key order (rank counting), i.e. td_pool_pairs' scan order ----
    const int npairs = s_m;
    long long part = 0;
    for (int k = tid; k < npairs; k += blockDim.x) {
        const unsigned long long me = kept[k];
        int rank = 0;
        for (int q = 0; q < npairs; ++q) rank += kept[q] < me;
        const int ab = int(me & 0xffffff), A = ab / n, B = ab - A * n;
        int plan = 0;
        edge_cost(e, A, B, nullptr, &plan);
        int32_t *r = rows + size_t(rank) * 4;
        r[0] = A; r[1] = B; r[2] = plan; r[3] = int(me >> 24);
        part += int(me >> 24);
    }
    atomicAdd(reinterpret_cast<unsigned long long *>(&s_total), (unsigned long long)part);
    for (int k = npairs * 4 + tid; k < rows_cap * 4; k += blockDim.x) rows[k] = -1;
    __syncthreads();
    if (tid == 0) { n_pairs_out[inst] = npairs; cost_out[inst] = s_total; }
}

static size_t pairs_stride(int n_max) { return carve_pairs(nullptr, n_max).bytes; }

static size_t pairs_smem(int n_max, int S) { return (size_t(S) * S + 2 * size_t(n_max > 0 ? n_max : 1)) * sizeof(int32_t); }

// best (n_max keys), kept (n_max / 2 + 1 keys), the stand table, from, to, two live lists, the rescan list, alive bytes
static size_t greedy_smem(int n_max, int S) {
    const size_t N = n_max > 0 ? size_t(n_max) : 1;
    return (N + N / 2 + 1) * sizeof(unsigned long long) + (size_t(S) * S + 5 * N) * sizeof(int32_t) + N;
}

// the argument checks of both batch entry points, in this order, before any device lookup; kNothingToLaunch for batch 0
constexpr int kNothingToLaunch = 1;
static_assert(TD_PAIRS_EXACT_MAX_N == TD_PAIRS_BATCH_MAX_N, "both pair kernels take the same instance sizes");
static int check_pairs_batch(const int32_t *from, const int32_t *to, const int32_t *sizes, const int64_t *offsets, int batch,
                             int n_max, const int32_t *dist, int n_stands, int accept_all, double max_loss,
                             const int32_t *pairs_out, const int32_t *n_pairs_out, const int64_t *cost_out) {
    if (batch < 0 || n_max < 0 || n_max > TD_PAIRS_BATCH_MAX_N) return TD_ERR_INVALID;
    if (n_stands < 1 || n_stands > kPairsMaxStands) return TD_ERR_INVALID;
    if (!accept_all && !std::isfinite(max_loss)) return TD_ERR_INVALID;
    if (batch == 0) return have_device() ? kNothingToLaunch : TD_ERR_NO_DEVICE;
    if (!from || !to || !sizes || !offsets || !dist || !n_pairs_out || !cost_out || (n_max >= 2 && !pairs_out)) return TD_ERR_INVALID;
    return TD_OK;
}

}  // namespace td

extern "C" size_t td_pool_pairs_exact_workspace_bytes(int batch, int n_max) {
    if (batch < 0 || n_max < 0 || n_max > TD_PAIRS_EXACT_MAX_N) return 0;
    return size_t(batch) * td::pairs_stride(n_max);
}

extern "C" int td_pool_pairs_batch(const int32_t *from, const int32_t *to, const int32_t *sizes, const int64_t *offsets,
                                   int batch, int n_max, const int32_t *dist, int n_stands, int accept_all, double max_loss,
                                   int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out, void *stream) {
    using namespace td;
    const int rc = check_pairs_batch(from, to, sizes, offsets, batch, n_max, dist, n_stands, accept_all, max_loss, pairs_out,
                                     n_pairs_out, cost_out);
    if (rc != TD_OK) return rc == kNothingToLaunch ? TD_OK : rc;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t smem = greedy_smem(n_max, n_stands);
    // small instances: several CTAs of 256 threads per SM; large ones: one warp per rescanned customer on 32 warps
    const int threads = n_max > 512 ? 1024 : 256;
    TD_CUDA_TRY(cudaFuncSetAttribute(pairs_greedy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    pairs_greedy_kernel<<<batch, threads, smem, st>>>(from, to, sizes, offsets, n_max, dist, n_stands, accept_all, max_loss,
                                                      pairs_out, n_pairs_out, reinterpret_cast<long long *>(cost_out));
    TD_LAUNCH_CHECK();
    return TD_OK;
}

extern "C" int td_pool_pairs_exact_batch(const int32_t *from, const int32_t *to, const int32_t *sizes, const int64_t *offsets,
                                         int batch, int n_max, const int32_t *dist, int n_stands, int accept_all,
                                         double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out,
                                         void *workspace, size_t workspace_bytes, void *stream) {
    using namespace td;
    const int rc = check_pairs_batch(from, to, sizes, offsets, batch, n_max, dist, n_stands, accept_all, max_loss, pairs_out,
                                     n_pairs_out, cost_out);
    if (rc != TD_OK) return rc == kNothingToLaunch ? TD_OK : rc;
    if (!workspace || workspace_bytes < td_pool_pairs_exact_workspace_bytes(batch, n_max)) return TD_ERR_WORKSPACE;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t smem = pairs_smem(n_max, n_stands);
    TD_CUDA_TRY(cudaFuncSetAttribute(pairs_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    pairs_exact_kernel<<<batch, kPairsThreads, smem, st>>>(from, to, sizes, offsets, n_max, dist, n_stands, accept_all, max_loss,
                                                           pairs_out, n_pairs_out, reinterpret_cast<long long *>(cost_out),
                                                           static_cast<char *>(workspace), pairs_stride(n_max));
    TD_LAUNCH_CHECK();
    return TD_OK;
}
