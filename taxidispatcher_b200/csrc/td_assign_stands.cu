// td_assign_stands.cu -- exact stand-derived assignment as a stand-to-stand transportation problem, batched.
//
// calculate_cost (split.py:123-136, Simulator.java:493-520) gives every cab at stand a the same row and every customer at
// stand b the same column: cell = C(a, b) = dist[a][b] (fill when cutoff >= 0 and dist >= cutoff), padded to
// n = max(cabs, customers) with constant `fill` rows or columns.  The optimum of that n x n assignment is therefore the
// optimum of the S x S transportation problem with supplies = cabs per stand, demands = customers per stand and arc costs
// C(a, b), plus (n - min(cabs, customers)) * fill for the padding.  Nothing of size n^2 is formed.
//
// Four launches per call, all asynchronous:
//   stands_count_kernel   one CTA per (instance, side, chunk): per-chunk stand histograms and the stand-range check.
//   stands_solve_kernel   one warp per instance: successive shortest paths over the <= 2S stand nodes.  The spare side
//                         (the one with more members; cabs when balanced) is the source side, so its potentials stay <= 0
//                         and are 0 at every stand that keeps a spare member.  Dense Dijkstra on reduced costs with int64
//                         potentials that start from the column minima, ties broken by (label, side, stand): no atomics
//                         decide a path.  Bottleneck augmentation along the one shortest path found.
//   stands_expand_kernel  one CTA per (instance, chunk), customers first, then cabs: index-order ranks per stand from the
//                         chunk histograms, a prefix over earlier chunks and warps and a warp match within each 32-group;
//                         customers scatter themselves to their partner cab's slot, cabs read it back (the expansion rule
//                         of include/taxidispatch.h).
#include "td_common.cuh"

namespace td {

constexpr int kStandsChunks = 64;        // chunks per side per instance at most (the histogram slots of the workspace)
constexpr int kStandsChunkMin = 4096;    // elements per chunk at least: small instances take one chunk
constexpr int kStandsThreads = 512;      // count / expansion CTA
constexpr int kStandsWarps = kStandsThreads / 32;
constexpr long long kStandsInf = 1ll << 54;   // labels stay far below: reduced path lengths are < 2S * 2^33

struct StandsWs {
    int *hist;     // [batch][2][kStandsChunks][S + 1]   (entry S: stand indices outside the table)
    int *meta;     // [batch][5][S]  cab count, cab matched, cab start (prefix of counts), customer count, customer matched
    int *seg;      // [batch][S + 1] start of each customer stand's flow segment
    int *seg_a;    // [batch][S * S] cab stand of the segment entry (increasing a)
    int *seg_cp;   // [batch][S * S] first customer rank at stand b that this cab stand receives
    int *seg_rp;   // [batch][S * S] first cab rank at stand a that goes to stand b
    int *state;    // [batch] 1 = solved, 0 = withdrawn
    int *slot;     // [batch][n_max] customer index per cab slot (cabs sorted by (stand, index))
    size_t bytes;
};

struct StandsCarver {
    char *base; size_t off;
    template <typename T> __host__ __device__ T *take(size_t count) {
        off = (off + 255) & ~size_t(255);
        T *p = reinterpret_cast<T *>(base + off);
        off += count * sizeof(T);
        return p;
    }
};

__host__ __device__ static StandsWs carve_stands(void *base, int batch, int S, int n_max) {
    StandsCarver c{static_cast<char *>(base), 0};
    const size_t B = batch > 0 ? size_t(batch) : 1, s = size_t(S);
    StandsWs w;
    w.hist = c.take<int>(B * 2 * kStandsChunks * (s + 1));
    w.meta = c.take<int>(B * 5 * s);
    w.seg = c.take<int>(B * (s + 1));
    w.seg_a = c.take<int>(B * s * s);
    w.seg_cp = c.take<int>(B * s * s);
    w.seg_rp = c.take<int>(B * s * s);
    w.state = c.take<int>(B);
    w.slot = c.take<int>(B * size_t(n_max > 0 ? n_max : 1));
    w.bytes = (c.off + 255) & ~size_t(255);
    return w;
}

__device__ __forceinline__ bool stands_inst_ok(int nc, int nd, long long co, long long uo, int n_max) {
    return nc >= 0 && nd >= 0 && (nc > nd ? nc : nd) <= n_max && co >= 0 && uo >= 0;
}

// chunk c of a side with m elements, split into nch chunks of at least kStandsChunkMin (32-aligned)
__device__ __forceinline__ void stands_chunk(long long m, int nch, int c, long long *lo, long long *hi) {
    long long L = (m + nch - 1) / nch;
    L = (L + 31) & ~31ll;
    if (L < kStandsChunkMin) L = kStandsChunkMin;
    *lo = (long long)c * L < m ? (long long)c * L : m;
    *hi = *lo + L < m ? *lo + L : m;
}

// warp w's contiguous share of [lo, hi)
__device__ __forceinline__ void stands_warp_range(long long lo, long long hi, int w, long long *a, long long *b) {
    long long W = (hi - lo + kStandsWarps - 1) / kStandsWarps;
    W = (W + 31) & ~31ll;
    *a = lo + w * W < hi ? lo + w * W : hi;
    *b = *a + W < hi ? *a + W : hi;
}

__device__ __forceinline__ int32_t stands_cell(const int32_t *dist, int S, int a, int b, int32_t fill, int32_t cutoff) {
    const int32_t d = __ldg(dist + a * S + b);
    return (cutoff >= 0 && d >= cutoff) ? fill : d;
}

// per-warp histograms of this CTA's chunk into wh[kStandsWarps][S]; returns the out-of-table count (thread 0 only)
__device__ int stands_warp_hist(const int32_t *idx, long long lo, long long hi, int S, int *wh, int *bad_s) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int k = threadIdx.x; k < kStandsWarps * S; k += blockDim.x) wh[k] = 0;
    if (threadIdx.x == 0) *bad_s = 0;
    __syncthreads();
    long long a, b;
    stands_warp_range(lo, hi, warp, &a, &b);
    int bad = 0;
    int *mine = wh + warp * S;
    for (long long e = a + lane; e < b; e += 32) {
        const int x = __ldg(idx + e);
        if (unsigned(x) < unsigned(S)) atomicAdd(mine + x, 1);
        else ++bad;
    }
    for (int o = 16; o > 0; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
    if (lane == 0 && bad) atomicAdd(bad_s, bad);
    __syncthreads();
    return *bad_s;
}

__global__ void __launch_bounds__(kStandsThreads)
stands_count_kernel(const int32_t *__restrict__ cab_to, const int64_t *__restrict__ cab_off, const int32_t *__restrict__ n_c,
                    const int32_t *__restrict__ cust_from, const int64_t *__restrict__ cust_off,
                    const int32_t *__restrict__ n_d, int S, int n_max, int nch, StandsWs ws) {
    extern __shared__ int sm_count[];
    const int inst = blockIdx.x / nch, c = blockIdx.x % nch, side = blockIdx.y;
    int *out = ws.hist + ((size_t(inst) * 2 + side) * kStandsChunks + c) * (S + 1);
    const int nc = n_c[inst], nd = n_d[inst];
    const long long co = cab_off[inst], uo = cust_off[inst];
    if (!stands_inst_ok(nc, nd, co, uo, n_max)) {
        for (int s = threadIdx.x; s <= S; s += blockDim.x) out[s] = 0;
        return;
    }
    const int32_t *idx = side ? cust_from + uo : cab_to + co;
    long long lo, hi;
    stands_chunk(side ? nd : nc, nch, c, &lo, &hi);
    int *wh = sm_count;
    const int bad = stands_warp_hist(idx, lo, hi, S, wh, wh + kStandsWarps * S);
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
        int t = 0;
        for (int w = 0; w < kStandsWarps; ++w) t += wh[w * S + s];
        out[s] = t;
    }
    if (threadIdx.x == 0) out[S] = bad;
}

// ---- the transportation solve: one warp per instance -------------------------------------------------------------------
struct StandsSmem {
    int32_t *K, *F;                 // [S][ld] arc costs and flows, source side x major
    long long *lab_p, *lab_q, *al, *be;
    int *par_p, *par_q, *cnt_p, *cnt_q, *res_p, *res_q;
    unsigned char *done_p, *done_q;
};

__host__ __device__ inline int stands_ld(int S) { return S | 1; }   // odd stride: row and column walks hit distinct banks

__host__ __device__ inline size_t stands_solve_smem(int S) {
    return size_t(2) * S * stands_ld(S) * 4 + size_t(4) * S * 8 + size_t(6) * S * 4 + size_t(2) * S + 16;
}

__global__ void __launch_bounds__(32)
stands_solve_kernel(const int32_t *__restrict__ dist, int S, int32_t fill, int32_t cutoff, const int32_t *__restrict__ n_c,
                    const int64_t *__restrict__ cab_off, const int32_t *__restrict__ n_d,
                    const int64_t *__restrict__ cust_off, int n_max, int nch, int32_t *__restrict__ col_of_row,
                    int32_t *__restrict__ cost_of_row, int64_t *__restrict__ objective, int64_t *__restrict__ u_out,
                    int64_t *__restrict__ v_out, int32_t *__restrict__ stats, StandsWs ws) {
    extern __shared__ __align__(16) unsigned char sm_solve[];
    const int inst = blockIdx.x, lane = threadIdx.x, ld = stands_ld(S);
    StandsSmem m;
    {
        unsigned char *p = sm_solve;
        m.lab_p = reinterpret_cast<long long *>(p); p += size_t(S) * 8;
        m.lab_q = reinterpret_cast<long long *>(p); p += size_t(S) * 8;
        m.al = reinterpret_cast<long long *>(p); p += size_t(S) * 8;
        m.be = reinterpret_cast<long long *>(p); p += size_t(S) * 8;
        m.K = reinterpret_cast<int32_t *>(p); p += size_t(S) * ld * 4;
        m.F = reinterpret_cast<int32_t *>(p); p += size_t(S) * ld * 4;
        int **ints[] = {&m.par_p, &m.par_q, &m.cnt_p, &m.cnt_q, &m.res_p, &m.res_q};
        for (int **q : ints) { *q = reinterpret_cast<int *>(p); p += size_t(S) * 4; }
        m.done_p = p; p += S;
        m.done_q = p;
    }
    const int nc = n_c[inst], nd = n_d[inst];
    const long long co = cab_off[inst], uo = cust_off[inst];
    const size_t row0 = size_t(inst) * n_max;
    bool ok = stands_inst_ok(nc, nd, co, uo, n_max);
    // stand counts: sums of the chunk histograms (cabs into res_p, customers into res_q for now)
    int bad = 0;
    for (int s = lane; s <= S; s += 32) {
        int t0 = 0, t1 = 0;
        if (ok) {
            const int *h = ws.hist + size_t(inst) * 2 * kStandsChunks * (S + 1);
            for (int c = 0; c < nch; ++c) { t0 += h[c * (S + 1) + s]; t1 += h[(kStandsChunks + c) * (S + 1) + s]; }
        }
        if (s == S) bad = t0 + t1;
        else { m.res_p[s] = t0; m.res_q[s] = t1; }
    }
    for (int o = 16; o > 0; o >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, o);
    ok = ok && bad == 0;
    if (!ok) {                                              // withdrawn: INT64_MIN, -1 slots, 0 potentials
        if (lane == 0) { objective[inst] = INT64_MIN; ws.state[inst] = 0; if (stats) { stats[2 * inst] = 0; stats[2 * inst + 1] = 0; } }
        for (int k = lane; k < n_max; k += 32) { col_of_row[row0 + k] = -1; if (cost_of_row) cost_of_row[row0 + k] = -1; }
        for (int s = lane; s < S; s += 32) { if (u_out) u_out[size_t(inst) * S + s] = 0; if (v_out) v_out[size_t(inst) * S + s] = 0; }
        return;
    }
    const int n = nc > nd ? nc : nd;
    for (int k = n + lane; k < n_max; k += 32) { col_of_row[row0 + k] = -1; if (cost_of_row) cost_of_row[row0 + k] = -1; }
    // orientation: sources (x) = the side with more members, sinks (y) = the other; K(x, y) = C of the (cab, customer) pair
    const bool tr = nc < nd;
    __syncwarp();
    for (int s = lane; s < S; s += 32) {
        const int cab = m.res_p[s], cust = m.res_q[s];
        m.cnt_p[s] = tr ? cust : cab;
        m.cnt_q[s] = tr ? cab : cust;
    }
    __syncwarp();
    for (int k = lane; k < S * S; k += 32) {
        const int x = k / S, y = k % S;
        int32_t c = 0;
        if (m.cnt_p[x] > 0 && m.cnt_q[y] > 0) c = tr ? stands_cell(dist, S, y, x, fill, cutoff) : stands_cell(dist, S, x, y, fill, cutoff);
        m.K[x * ld + y] = c;
        m.F[x * ld + y] = 0;
    }
    __syncwarp();
    long long total = 0;
    for (int s = lane; s < S; s += 32) {
        m.res_p[s] = m.cnt_p[s];
        m.res_q[s] = m.cnt_q[s];
        m.al[s] = 0;
        long long mn = 0;
        if (m.cnt_q[s] > 0) {                               // column minimum over the source stands with members
            mn = LLONG_MAX;
            for (int x = 0; x < S; ++x)
                if (m.cnt_p[x] > 0 && m.K[x * ld + s] < mn) mn = m.K[x * ld + s];
            if (mn == LLONG_MAX) mn = 0;
        }
        m.be[s] = mn;
        total += m.cnt_q[s];
    }
    for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(0xffffffffu, total, o);
    if (nc == 0 || nd == 0) total = 0;
    __syncwarp();

    long long flow = 0;
    int phases = 0, augs = 0;
    while (flow < total) {
        for (int s = lane; s < S; s += 32) {
            m.lab_p[s] = (m.cnt_p[s] > 0 && m.res_p[s] > 0) ? 0 : kStandsInf;
            m.par_p[s] = -1;
            m.done_p[s] = m.cnt_p[s] == 0;
            m.lab_q[s] = kStandsInf;
            m.par_q[s] = -1;
            m.done_q[s] = m.cnt_q[s] == 0;
        }
        __syncwarp();
        int sink = -1;
        long long D = 0;
        for (;;) {
            unsigned long long best = ~0ull;
            for (int s = lane; s < S; s += 32) {
                if (!m.done_p[s] && m.lab_p[s] < kStandsInf) {
                    const unsigned long long k = (unsigned long long)m.lab_p[s] << 9 | unsigned(s);
                    best = k < best ? k : best;
                }
                if (!m.done_q[s] && m.lab_q[s] < kStandsInf) {
                    const unsigned long long k = (unsigned long long)m.lab_q[s] << 9 | unsigned(256 + s);
                    best = k < best ? k : best;
                }
            }
            best = warp_min_u64(best);
            if (best == ~0ull) break;                       // unreachable sink: cannot happen on a complete table
            const int z = int(best & 511);
            const long long L = (long long)(best >> 9);
            __syncwarp();
            if (z >= 256) {
                const int y = z - 256;
                if (m.res_q[y] > 0) { sink = y; D = L; break; }
                if (lane == 0) m.done_q[y] = 1;
                const long long by = m.be[y];
                for (int x = lane; x < S; x += 32) {        // backward arcs: flow from x to y can be taken back
                    if (m.done_p[x] || m.F[x * ld + y] <= 0) continue;
                    const long long nl = L - ((long long)m.K[x * ld + y] - m.al[x] - by);
                    if (nl < m.lab_p[x]) { m.lab_p[x] = nl; m.par_p[x] = y; }
                }
            } else {
                const int x = z;
                if (lane == 0) m.done_p[x] = 1;
                const long long ax = m.al[x];
                for (int y = lane; y < S; y += 32) {
                    if (m.done_q[y]) continue;
                    const long long nl = L + ((long long)m.K[x * ld + y] - ax - m.be[y]);
                    if (nl < m.lab_q[y]) { m.lab_q[y] = nl; m.par_q[y] = x; }
                }
            }
            __syncwarp();
        }
        if (sink < 0) break;
        for (int s = lane; s < S; s += 32) {
            if (m.cnt_p[s] > 0) m.al[s] -= m.lab_p[s] < D ? m.lab_p[s] : D;
            if (m.cnt_q[s] > 0) m.be[s] += m.lab_q[s] < D ? m.lab_q[s] : D;
        }
        __syncwarp();
        long long d = 0;
        if (lane == 0) {
            d = m.res_q[sink];
            for (int y = sink;;) {
                const int x = m.par_q[y], py = m.par_p[x];
                if (py < 0) { d = m.res_p[x] < d ? m.res_p[x] : d; break; }
                d = m.F[x * ld + py] < d ? m.F[x * ld + py] : d;
                y = py;
            }
            for (int y = sink;;) {
                const int x = m.par_q[y], py = m.par_p[x];
                m.F[x * ld + y] += int(d);
                if (py < 0) { m.res_p[x] -= int(d); break; }
                m.F[x * ld + py] -= int(d);
                y = py;
            }
            m.res_q[sink] -= int(d);
        }
        d = __shfl_sync(0xffffffffu, d, 0);
        flow += d;
        ++phases;
        ++augs;
        __syncwarp();
    }

    // objective, potentials, stats
    long long obj = 0;
    for (int k = lane; k < S * S; k += 32) {
        const int x = k / S, y = k % S;
        obj += (long long)m.F[x * ld + y] * m.K[x * ld + y];
    }
    for (int o = 16; o > 0; o >>= 1) obj += __shfl_xor_sync(0xffffffffu, obj, o);
    if (lane == 0) {
        objective[inst] = obj + (long long)(n - (nc < nd ? nc : nd)) * fill;
        ws.state[inst] = 1;
        if (stats) { stats[2 * inst] = phases; stats[2 * inst + 1] = augs; }
    }
    for (int s = lane; s < S; s += 32) {
        if (u_out) u_out[size_t(inst) * S + s] = tr ? m.be[s] : m.al[s];
        if (v_out) v_out[size_t(inst) * S + s] = tr ? m.al[s] : m.be[s];
    }
    // expansion tables in (cab stand a, customer stand b) terms; f(a, b) = F of the oriented pair
    auto f = [&](int a, int b) -> int { return tr ? m.F[b * ld + a] : m.F[a * ld + b]; };
    int *meta = ws.meta + size_t(inst) * 5 * S;
    int *seg = ws.seg + size_t(inst) * (S + 1);
    int *seg_a = ws.seg_a + size_t(inst) * S * S, *seg_cp = ws.seg_cp + size_t(inst) * S * S;
    int *seg_rp = ws.seg_rp + size_t(inst) * S * S;
    __syncwarp();
    // K is free now: K[a][b] := first cab rank at stand a that goes to stand b (row prefix of the flows)
    for (int a = lane; a < S; a += 32) {
        int run = 0;
        for (int b = 0; b < S; ++b) { const int fab = f(a, b); m.K[a * ld + b] = run; run += fab; }
        meta[S + a] = run;                                  // cabs of stand a that got a customer
        meta[a] = tr ? m.cnt_q[a] : m.cnt_p[a];
        meta[3 * S + a] = tr ? m.cnt_p[a] : m.cnt_q[a];
    }
    for (int b = lane; b < S; b += 32) {
        int nnz = 0, in = 0;
        for (int a = 0; a < S; ++a) { const int fab = f(a, b); nnz += fab > 0; in += fab; }
        meta[4 * S + b] = in;                               // customers of stand b that got a cab
        m.par_q[b] = nnz;
    }
    __syncwarp();
    if (lane == 0) {
        int run = 0, start = 0;
        for (int s = 0; s < S; ++s) {
            seg[s] = start; start += m.par_q[s];
            meta[2 * S + s] = run; run += meta[s];
        }
        seg[S] = start;
    }
    __syncwarp();
    for (int b = lane; b < S; b += 32) {
        int e = seg[b], cp = 0;
        for (int a = 0; a < S; ++a) {
            const int fab = f(a, b);
            if (fab > 0) { seg_a[e] = a; seg_cp[e] = cp; seg_rp[e] = m.K[a * ld + b]; ++e; cp += fab; }
        }
    }
}

// ---- expansion -------------------------------------------------------------------------------------------------------
// kCabs == false: customers scatter themselves into the slot of their partner cab, unmatched customers fill the padding
// rows nc.. in index order.  kCabs == true: cabs read their partner from that slot, unmatched cabs take columns nd.. in
// index order.
template <bool kCabs>
__global__ void __launch_bounds__(kStandsThreads)
stands_expand_kernel(const int32_t *__restrict__ dist, int S, int32_t fill, int32_t cutoff,
                     const int32_t *__restrict__ cab_to, const int64_t *__restrict__ cab_off, const int32_t *__restrict__ n_c,
                     const int32_t *__restrict__ cust_from, const int64_t *__restrict__ cust_off,
                     const int32_t *__restrict__ n_d, int n_max, int nch, int32_t *__restrict__ col_of_row,
                     int32_t *__restrict__ cost_of_row, StandsWs ws) {
    extern __shared__ int sm_exp[];
    const int inst = blockIdx.x / nch, c = blockIdx.x % nch;
    if (ws.state[inst] != 1) return;
    const int nc = n_c[inst], nd = n_d[inst];
    const int m_side = kCabs ? nc : nd;
    long long lo, hi;
    stands_chunk(m_side, nch, c, &lo, &hi);
    if (lo >= hi) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int32_t *idx = kCabs ? cab_to + cab_off[inst] : cust_from + cust_off[inst];
    const int32_t *cust = cust_from + cust_off[inst];
    const int *meta = ws.meta + size_t(inst) * 5 * S;
    const int *matched = meta + (kCabs ? S : 4 * S);
    const int *seg = ws.seg + size_t(inst) * (S + 1);
    const int *seg_a = ws.seg_a + size_t(inst) * S * S, *seg_cp = ws.seg_cp + size_t(inst) * S * S;
    const int *seg_rp = ws.seg_rp + size_t(inst) * S * S;
    int *slot = ws.slot + size_t(inst) * n_max;
    int32_t *col = col_of_row + size_t(inst) * n_max;
    int32_t *cost = cost_of_row ? cost_of_row + size_t(inst) * n_max : nullptr;

    int *wh = sm_exp;                                       // [warps][S]: histogram, then running rank base
    int *bad_s = wh + kStandsWarps * S;
    int *ubase = bad_s + 1;                                 // [warps] unmatched members before each warp
    stands_warp_hist(idx, lo, hi, S, wh, bad_s);
    // rank base per (warp, stand): earlier chunks + earlier warps of this chunk
    const int *h = ws.hist + (size_t(inst) * 2 + (kCabs ? 0 : 1)) * kStandsChunks * (S + 1);
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
        int run = 0;
        for (int cc = 0; cc < c; ++cc) run += h[cc * (S + 1) + s];
        for (int w = 0; w < kStandsWarps; ++w) { const int t = wh[w * S + s]; wh[w * S + s] = run; run += t; }
    }
    __syncthreads();
    {   // members past their stand's matched count, before this warp's range: sum over stands of max(0, base - matched)
        int u = 0;
        for (int s = lane; s < S; s += 32) { const int e = wh[warp * S + s] - matched[s]; u += e > 0 ? e : 0; }
        for (int o = 16; o > 0; o >>= 1) u += __shfl_xor_sync(0xffffffffu, u, o);
        if (lane == 0) ubase[warp] = u;
    }
    __syncwarp();
    int unmatched = ubase[warp];
    int *base = wh + warp * S;
    long long a0, a1;
    stands_warp_range(lo, hi, warp, &a0, &a1);
    const unsigned lt = (1u << lane) - 1u;
    for (long long g = a0; g < a1; g += 32) {
        const long long e = g + lane;
        const bool valid = e < a1;
        const int x = valid ? __ldg(idx + e) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, x);
        const int r = valid ? base[x] + __popc(peers & lt) : 0;
        __syncwarp();
        if (valid && lane == __ffs(peers) - 1) base[x] += __popc(peers);
        __syncwarp();
        const bool spare = valid && r >= matched[valid ? x : 0];
        const unsigned sb = __ballot_sync(0xffffffffu, spare);
        const int ord = unmatched + __popc(sb & lt);
        unmatched += __popc(sb);
        if (!valid) continue;
        if (kCabs) {
            const int i = int(e);
            if (spare) {
                col[i] = nd + ord;
                if (cost) cost[i] = fill;
            } else {
                const int j = slot[meta[2 * S + x] + r];
                col[i] = j;
                if (cost) cost[i] = stands_cell(dist, S, x, __ldg(cust + j), fill, cutoff);
            }
        } else {
            const int j = int(e);
            if (spare) {
                col[nc + ord] = j;
                if (cost) cost[nc + ord] = fill;
            } else {                                        // the cab stand whose customer-rank range holds r
                int lo_e = seg[x], hi_e = seg[x + 1] - 1;
                while (lo_e < hi_e) {
                    const int mid = (lo_e + hi_e + 1) >> 1;
                    if (seg_cp[mid] <= r) lo_e = mid; else hi_e = mid - 1;
                }
                const int a = seg_a[lo_e];
                slot[meta[2 * S + a] + seg_rp[lo_e] + (r - seg_cp[lo_e])] = j;
            }
        }
    }
}

static size_t stands_expand_smem(int S) { return (size_t(kStandsWarps) * S + 1 + kStandsWarps) * 4; }

}  // namespace td

extern "C" size_t td_assign_stands_workspace_bytes(int batch, int n_stands, int n_max) {
    if (batch < 0 || n_stands < 1 || n_stands > TD_STANDS_MAX_S || n_max < 0) return 0;
    return td::carve_stands(nullptr, batch, n_stands, n_max).bytes;
}

extern "C" int td_assign_stands_batch(const int32_t *dist, int n_stands, int32_t fill, int32_t cutoff,
                                      const int32_t *cab_to, const int64_t *cab_off, const int32_t *n_c,
                                      const int32_t *cust_from, const int64_t *cust_off, const int32_t *n_d,
                                      int batch, int n_max, int32_t *col_of_row, int32_t *cost_of_row,
                                      int64_t *objective, int64_t *u, int64_t *v, int32_t *stats,
                                      void *workspace, size_t workspace_bytes, void *stream) {
    using namespace td;
    if (batch < 0 || n_stands < 1 || n_stands > TD_STANDS_MAX_S || n_max < 0) return TD_ERR_INVALID;
    if (batch == 0) return TD_OK;
    if (!dist || !cab_to || !cab_off || !n_c || !cust_from || !cust_off || !n_d || !col_of_row || !objective || !workspace)
        return TD_ERR_INVALID;
    if (workspace_bytes < td_assign_stands_workspace_bytes(batch, n_stands, n_max)) return TD_ERR_WORKSPACE;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const StandsWs ws = carve_stands(workspace, batch, n_stands, n_max);
    const int S = n_stands;
    const long long want = (n_max + kStandsChunkMin - 1) / kStandsChunkMin;
    const int nch = int(want < 1 ? 1 : want > kStandsChunks ? kStandsChunks : want);
    const size_t esm = stands_expand_smem(S);
    stands_count_kernel<<<dim3(unsigned(batch) * nch, 2), kStandsThreads, esm, st>>>(cab_to, cab_off, n_c, cust_from, cust_off,
                                                                                    n_d, S, n_max, nch, ws);
    TD_LAUNCH_CHECK();
    const size_t ssm = stands_solve_smem(S);
    TD_CUDA_TRY(cudaFuncSetAttribute(stands_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(ssm)));
    stands_solve_kernel<<<batch, 32, ssm, st>>>(dist, S, fill, cutoff, n_c, cab_off, n_d, cust_off, n_max, nch, col_of_row,
                                                cost_of_row, objective, u, v, stats, ws);
    TD_LAUNCH_CHECK();
    stands_expand_kernel<false><<<unsigned(batch) * nch, kStandsThreads, esm, st>>>(
        dist, S, fill, cutoff, cab_to, cab_off, n_c, cust_from, cust_off, n_d, n_max, nch, col_of_row, cost_of_row, ws);
    TD_LAUNCH_CHECK();
    stands_expand_kernel<true><<<unsigned(batch) * nch, kStandsThreads, esm, st>>>(
        dist, S, fill, cutoff, cab_to, cab_off, n_c, cust_from, cust_off, n_d, n_max, nch, col_of_row, cost_of_row, ws);
    TD_LAUNCH_CHECK();
    return TD_OK;
}
