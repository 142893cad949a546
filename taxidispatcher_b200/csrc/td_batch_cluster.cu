// td_batch_cluster.cu -- batches of mid-size and large assignment and LCM instances, one thread-block cluster of K CTAs
// per instance.  Two storage forms of the same two kernels (template parameter kGlobal):
//
//   DSMEM form   (td_*_batch_cluster, n <= TD_BATCH_CLUSTER_MAX_N = 640): the n x n matrix is cut into K blocks, one per
//                CTA of a portable cluster (K in {1, 2, 4, 8}), and staged in the CTAs' shared memory.  K is the smallest
//                count whose block fits one CTA next to its O(n) state: 232 -> 1, 300 -> 2, 400 -> 4, 640 -> 8.
//   global form  (td_*_batch_large, n <= TD_BATCH_LARGE_MAX_N = 2048): the matrix stays in global memory (L2 / HBM) and
//                only the O(n) state is on chip.  K is the smallest of {4, 8} with ceil(n_max / K) <= 256, so a thread
//                owns at most one column (assignment) or one row (LCM): 4 up to 1024, 8 up to 2048.
//
// What the single-CTA routines read from their own shared memory -- the row minima, the lowest asking column of a row,
// the level minimum of a Dijkstra step, the rows that join the tree, the LCM arg-min -- is reduced or gathered across the
// cluster through distributed shared memory in both forms.  K depends on n_max only.
//
// What one CTA of the global form reads from the matrix per step:
//   assignment  row minima: one warp per row over the CTA's columns (coalesced row segments); column minima and the
//               greedy: thread t walks down its column j0 + t (one coalesced row segment per row across the CTA); a
//               Dijkstra step: the row segment [j0, j0 + B) of every row that joined the tree in the previous step.
//   LCM         the initial row minima: one warp per owned row, the whole row; per iteration: the whole row of every
//               owned row whose cached minimum sat in the picked column (one warp per row).  The mask is not written:
//               a cell reads as mask_value when its row or its column has been picked (flags in shared memory), which is
//               exactly the value the literal algorithm wrote there.
//
// Both kernels run the SAME algorithm as the single-CTA ones, step for step, in both forms, so they return the same
// results:
//   assignment  the matching, both potential vectors and the objective of assign_small_solve (td_assign.cu) for every
//               n <= 232, and results that depend neither on K, nor on the storage form, nor on n_max, nor on the
//               instance's slot in the batch;
//   LCM         the literal trace (rows, cols, n_pairs, total, last_min) of td_lcm / td_lcm_batch for every params.
//
// Every CTA of a cluster takes the same path (also when an instance is withdrawn) and ends with cluster.sync(), so no
// CTA leaves while another one may still read or write its shared memory.
#include "td_common.cuh"
#include <stdio.h>

namespace cg = cooperative_groups;

namespace td {

constexpr int kClThreads = 256;
constexpr int kClWarps = kClThreads / 32;
constexpr int kClMaxK = 8;                           // portable cluster size
constexpr size_t kClSmemLimit = 227 * 1024;          // shared memory of one CTA (dynamic + static) on sm_100
constexpr size_t kClStaticReserve = 1024;            // the kernels' static __shared__ variables stay below this

__host__ __device__ constexpr int cl_block(int n_max, int k) { return (n_max + k - 1) / k; }
__host__ __device__ constexpr size_t cl_align16(size_t b) { return (b + 15) & ~size_t(15); }

// ---- exact assignment: CTA k owns the columns [k*B, min(n, (k+1)*B)) ------------------------------------------------
// Shared memory of one CTA (n_max rows, B columns):
//   c      [n_max][B] int32   the cost block of the CTA's columns (DSMEM form only; the global form reads the matrix)
//   u      [n_max]    int64   row potentials (replicated)
//   mate   [n_max]    int32   column of row i, -1: free (replicated)
//   tr     [n_max]    int32   rows of the current tree in join order; the rows of one level are a contiguous run (replicated)
//   xa, xb [n_max]    int32   cluster exchange: partial row minima / lowest asking columns; path of the flip
//   p, way [B]        int32   row of the column, predecessor column on the alternating path (the CTA's columns)
//   stage  [B]        int32   rows of the CTA's columns that join the tree in this step, in column order
//   slots             int64 delta[8], int64 obj[8], int32 cnt[8], int32 jfree[8]: values pushed by every CTA of the cluster
struct AsgClLayout {
    size_t c, u, mate, tr, xa, xb, p, way, stage, slots, bytes;
};
__host__ __device__ inline AsgClLayout asg_cl_layout(int n_max, int B, bool global) {
    AsgClLayout L;
    size_t o = 0;
    L.c = o; o = cl_align16(o + (global ? 0 : size_t(n_max) * B * 4));
    L.u = o; o = cl_align16(o + size_t(n_max) * 8);
    L.mate = o; o = cl_align16(o + size_t(n_max) * 4);
    L.tr = o; o = cl_align16(o + size_t(n_max) * 4);
    L.xa = o; o = cl_align16(o + size_t(n_max) * 4);
    L.xb = o; o = cl_align16(o + size_t(n_max) * 4);
    L.p = o; o = cl_align16(o + size_t(B) * 4);
    L.way = o; o = cl_align16(o + size_t(B) * 4);
    L.stage = o; o = cl_align16(o + size_t(B) * 4);
    L.slots = o; o = cl_align16(o + kClMaxK * (8 + 8 + 4 + 4));
    L.bytes = o;
    return L;
}

__device__ __forceinline__ long long block_min_ll(long long x, long long *s_red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const long long y = __shfl_xor_sync(0xffffffffu, x, o); x = y < x ? y : x; }
    __syncthreads();                         // s_red is free (its previous readers are done)
    if (lane == 0) s_red[w] = x;
    __syncthreads();
    long long m = s_red[0];
#pragma unroll
    for (int k = 1; k < kClWarps; ++k) m = s_red[k] < m ? s_red[k] : m;
    return m;
}

__device__ __forceinline__ long long block_sum_ll(long long x, long long *s_red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    __syncthreads();
    if (lane == 0) s_red[w] = x;
    __syncthreads();
    long long s = 0;
#pragma unroll
    for (int k = 0; k < kClWarps; ++k) s += s_red[k];
    return s;
}

template <bool kGlobal>
__global__ void __launch_bounds__(kClThreads, 1)
assign_cluster_kernel(const int32_t *__restrict__ costs, const int32_t *__restrict__ sizes, const int64_t *__restrict__ offsets,
                      int n_max, int B, int32_t *col_of_row_out, long long *objective_out, long long *u_out, long long *v_out) {
    extern __shared__ __align__(16) unsigned char csm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int K = int(cluster.num_blocks());
    const int rank = int(cluster.block_rank());
    const int b = blockIdx.x / K;
    const int n = sizes[b];
    const long long off = offsets[b];
    const size_t o = size_t(b) * n_max;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const long long kInf = LLONG_MAX / 4;
    __shared__ long long s_red[kClWarps];
    __shared__ int s_wcnt[kClWarps], s_jfree, s_progress, s_len;

    const bool bad = n < 0 || n > n_max || off < 0 || (off & 3) != 0;
    if (bad || n == 0) {                     // withdrawn or empty: the same path in every CTA
        if (rank == 0) {
            for (int k = t; k < n_max; k += kClThreads) {
                col_of_row_out[o + k] = -1;
                if (u_out) u_out[o + k] = 0;
                if (v_out) v_out[o + k] = 0;
            }
            if (t == 0) objective_out[b] = bad ? LLONG_MIN : 0;
        }
        cluster.sync();
        return;
    }
    const AsgClLayout L = asg_cl_layout(n_max, B, kGlobal);
    int32_t *c = reinterpret_cast<int32_t *>(csm + L.c);
    long long *u = reinterpret_cast<long long *>(csm + L.u);
    int *mate = reinterpret_cast<int *>(csm + L.mate);
    int *tr = reinterpret_cast<int *>(csm + L.tr);
    int *xa = reinterpret_cast<int *>(csm + L.xa);
    int *xb = reinterpret_cast<int *>(csm + L.xb);
    int *p = reinterpret_cast<int *>(csm + L.p);
    int *way = reinterpret_cast<int *>(csm + L.way);
    int *stage = reinterpret_cast<int *>(csm + L.stage);
    long long *slot_delta = reinterpret_cast<long long *>(csm + L.slots);
    long long *slot_obj = slot_delta + kClMaxK;
    int *slot_cnt = reinterpret_cast<int *>(slot_obj + kClMaxK);
    int *slot_jfree = slot_cnt + kClMaxK;

    const int j0 = rank * B;
    const int nloc = n - j0 < 0 ? 0 : (n - j0 < B ? n - j0 : B);
    const bool own = t < nloc;               // thread t owns column j0 + t
    const int32_t *src = costs + off;
    // cost[i][j0 + jl]: the staged block, or the matrix itself
    auto cst = [&](int i, int jl) -> int32_t {
        if constexpr (kGlobal) return __ldg(src + size_t(i) * n + j0 + jl);
        else return c[i * B + jl];
    };
    // row minima: partial over the CTA's columns -> xa, then the minimum of the K partials (order-free: the same value)
    if constexpr (kGlobal) {
        for (int i = w; i < n; i += kClWarps) {
            int m = INT_MAX;
            for (int jl = lane; jl < nloc; jl += 32) { const int v0 = cst(i, jl); m = v0 < m ? v0 : m; }
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) { const int y = __shfl_xor_sync(0xffffffffu, m, s); m = y < m ? y : m; }
            if (lane == 0) xa[i] = m;
        }
    } else {
        for (int e = t; e < n * nloc; e += kClThreads) {
            const int i = e / nloc, jl = e - i * nloc;
            c[i * B + jl] = __ldg(src + size_t(i) * n + j0 + jl);
        }
        __syncthreads();
        for (int i = t; i < n; i += kClThreads) {
            int m = INT_MAX;
            for (int jl = 0; jl < nloc; ++jl) { const int v0 = c[i * B + ((jl + i) % nloc)]; m = v0 < m ? v0 : m; }
            xa[i] = m;
        }
    }
    cluster.sync();
    for (int i = t; i < n; i += kClThreads) {
        int m = INT_MAX;
        for (int k = 0; k < K; ++k) { const int v0 = cluster.map_shared_rank(xa, k)[i]; m = v0 < m ? v0 : m; }
        u[i] = m;
        mate[i] = -1;
    }
    if (own) p[t] = -1;
    __syncthreads();
    // column minima of the row-reduced costs -> v (the column's own)
    long long v = 0;
    if (own) {
        long long m = kInf;
        for (int i = 0; i < n; ++i) { const long long r = (long long)cst(i, t) - u[i]; m = r < m ? r : m; }
        v = m;
    }
    // greedy matching on tight cells, as assign_small_solve: every free column asks for the lowest free row that is tight
    // with it, every asked row accepts the lowest asking column (the minimum over the cluster of the CTAs' lowest ones).
    // Round r collects in xb / xa alternately: a buffer is written again only after the next cluster.sync, which every
    // CTA reaches after its reads of that buffer (xa's row-minimum reads end before round 0's barrier).
    for (int round = 0; round < 4; ++round) {
        int *ask = (round & 1) ? xa : xb;
        __syncthreads();                     // everybody has read s_progress of the previous round
        for (int i = t; i < n; i += kClThreads) ask[i] = INT_MAX;
        if (t == 0) s_progress = 0;
        __syncthreads();
        if (own && p[t] < 0) {
            int pick = -1;
            for (int i = 0; i < n && pick < 0; ++i)
                if (mate[i] < 0 && (long long)cst(i, t) - u[i] - v == 0) pick = i;
            if (pick >= 0) atomicMin(&ask[pick], j0 + t);
        }
        cluster.sync();
        for (int i = t; i < n; i += kClThreads) {
            if (mate[i] >= 0) continue;
            int got = INT_MAX;
            for (int k = 0; k < K; ++k) { const int a = cluster.map_shared_rank(ask, k)[i]; got = a < got ? a : got; }
            if (got != INT_MAX) {
                mate[i] = got;
                if (got >= j0 && got < j0 + nloc) p[got - j0] = i;
                s_progress = 1;
            }
        }
        __syncthreads();
        if (!s_progress) break;              // the same in every CTA: computed from the same exchanged minima
    }
    __syncthreads();
    // ---- augment every row that is still free: level-wise Dijkstra, as assign_small_solve ------------------------------
    // A step: relax the rows that joined in the previous step (list order = global column order) -> cluster minimum of the
    // distances (delta, barrier A) -> dual update -> the columns at delta join; their rows are appended to tr in global
    // column order (counts and staged rows pushed, barrier B).  Slots written before A are read between A and B, slots
    // written before B are read between B and the next A: one buffer each suffices.
    for (int i = 0; i < n; ++i) {
        if (mate[i] >= 0) continue;          // uniform: mate[] is replicated and read after a barrier
        long long minv = kInf;
        bool used = false;
        if (own) way[t] = -1;
        if (t == 0) tr[0] = i;
        __syncthreads();
        int lo = 0, hi = 1;                  // tr[lo, hi): the rows relaxed in this step; tr[0, hi): every row of the tree
        int jend;
        for (;;) {
            long long key = kInf;
            if (own && !used) {
                for (int k = lo; k < hi; ++k) {
                    const int r = tr[k];
                    const long long cur = (long long)cst(r, t) - u[r] - v;
                    if (cur < minv) { minv = cur; way[t] = r == i ? -1 : mate[r]; }
                }
                key = minv;
            }
            const long long lmin = block_min_ll(key, s_red);
            if (t < K) cluster.map_shared_rank(slot_delta, t)[rank] = lmin;
            cluster.sync();                                                        // A
            long long delta = slot_delta[0];
            for (int k = 1; k < K; ++k) delta = slot_delta[k] < delta ? slot_delta[k] : delta;
            const bool joins = own && !used && minv == delta;
            if (own) {
                if (used) v -= delta;
                else minv -= delta;
            }
            for (int k = t; k < hi; k += kClThreads) u[tr[k]] += delta;         // the tree's rows (the root included)
            const bool matched = joins && p[t] >= 0;
            const unsigned ball = __ballot_sync(0xffffffffu, matched);
            if (lane == 0) s_wcnt[w] = __popc(ball);
            if (t == 0) s_jfree = INT_MAX;
            __syncthreads();
            if (joins) {
                used = true;
                if (!matched) atomicMin(&s_jfree, j0 + t);
                else {
                    int pos = __popc(ball & ((1u << lane) - 1));
                    for (int k = 0; k < w; ++k) pos += s_wcnt[k];
                    stage[pos] = p[t];
                }
            }
            __syncthreads();
            if (t < K) {
                int cnt = 0;
                for (int k = 0; k < kClWarps; ++k) cnt += s_wcnt[k];
                cluster.map_shared_rank(slot_cnt, t)[rank] = cnt;
                cluster.map_shared_rank(slot_jfree, t)[rank] = s_jfree;
            }
            cluster.sync();                                                        // B
            int jfree = INT_MAX, base = hi;
            for (int k = 0; k < K; ++k) {
                const int cnt = slot_cnt[k];
                jfree = slot_jfree[k] < jfree ? slot_jfree[k] : jfree;
                if (cnt > 0) {
                    const int *rs = cluster.map_shared_rank(stage, k);
                    for (int x = t; x < cnt; x += kClThreads) tr[base + x] = rs[x];
                }
                base += cnt;
            }
            __syncthreads();
            lo = hi;
            hi = base;
            if (jfree != INT_MAX) { jend = jfree; break; }   // a free column at this level: augment (the smallest one)
        }
        // flip the alternating path.  Every CTA walks it (way / p of other CTAs through DSMEM, reads only), the cluster
        // barrier ends all reads, then every CTA applies it to its mate[] and to the p[] of its own columns.
        if (t == 0) {
            int j = jend, len = 0;
            for (;;) {
                const int oj = j / B;
                const int jp = cluster.map_shared_rank(way, oj)[j - oj * B];
                int r = i;
                if (jp >= 0) { const int op = jp / B; r = cluster.map_shared_rank(p, op)[jp - op * B]; }
                xa[len] = r; xb[len] = j; ++len;
                if (jp < 0) break;
                j = jp;
            }
            s_len = len;
        }
        cluster.sync();
        const int len = s_len;
        for (int k = t; k < len; k += kClThreads) {
            const int r = xa[k], j = xb[k];
            mate[r] = j;
            if (j >= j0 && j < j0 + nloc) p[j - j0] = r;
        }
        __syncthreads();
    }
    // ---- results: CTA k writes the rows and columns of its range; the objective is summed over the cluster --------------
    for (int k = t; k < nloc; k += kClThreads) {
        col_of_row_out[o + j0 + k] = mate[j0 + k];
        if (u_out) u_out[o + j0 + k] = u[j0 + k];
    }
    if (own && v_out) v_out[o + j0 + t] = v;
    if (rank == K - 1)
        for (int k = n + t; k < n_max; k += kClThreads) {
            col_of_row_out[o + k] = -1;
            if (u_out) u_out[o + k] = 0;
            if (v_out) v_out[o + k] = 0;
        }
    const long long part = block_sum_ll(own ? (long long)cst(p[t], t) : 0, s_red);
    if (t == 0) cluster.map_shared_rank(slot_obj, 0)[rank] = part;
    cluster.sync();                          // the last remote access of the cluster
    if (rank == 0 && t == 0) {
        long long tot = 0;
        for (int k = 0; k < K; ++k) tot += slot_obj[k];
        objective_out[b] = tot;
    }
}

// ---- LCM: CTA k owns the rows [k*R, min(n, (k+1)*R)) of the working array ---------------------------------------------
// Shared memory: rk [R] uint64 (cached row minimum keys), d [R][n_max] int32 (DSMEM form: the CTA's rows, overwritten with
// the mask like the reference does), stale [R] int32, slots [2][8] uint64 (every CTA's local arg-min, double-buffered by
// iteration parity: one cluster.sync per iteration), and in the global form the picked flags cpick [n_max] and rpick [R]
// uint8 (column / owned row picked: its cells read as mask_value).
__host__ __device__ inline size_t lcm_cl_bytes(int n_max, int R, bool global) {
    return cl_align16(size_t(R) * 8) + cl_align16(global ? 0 : size_t(R) * n_max * 4) + cl_align16(size_t(R) * 4) +
           2 * kClMaxK * 8 + (global ? cl_align16(size_t(n_max)) + cl_align16(size_t(R)) : 0);
}

template <bool kGlobal>
__global__ void __launch_bounds__(kClThreads, 1)
lcm_cluster_kernel(const int32_t *__restrict__ costs, const int32_t *__restrict__ sizes, const int64_t *__restrict__ offsets,
                   int n_max, int R, td_lcm_params prm, int32_t *rows_out, int32_t *cols_out, int32_t *n_pairs_out,
                   long long *total_out, int32_t *last_min_out) {
    extern __shared__ __align__(16) unsigned char csm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int K = int(cluster.num_blocks());
    const int rank = int(cluster.block_rank());
    const int b = blockIdx.x / K;
    const int n = sizes[b];
    const long long off = offsets[b];
    const size_t o = size_t(b) * n_max;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    __shared__ unsigned long long s_min[kClWarps];
    __shared__ int s_nstale;
    const bool bad = n < 0 || n > n_max || off < 0 || (off & 3) != 0;
    if (bad) {
        if (rank == 0) {
            for (int k = t; k < n_max; k += kClThreads) { rows_out[o + k] = -1; cols_out[o + k] = -1; }
            if (t == 0) {
                n_pairs_out[b] = -1; total_out[b] = LLONG_MIN;
                if (last_min_out) last_min_out[b] = INT32_MIN;
            }
        }
        cluster.sync();
        return;
    }
    unsigned long long *rk = reinterpret_cast<unsigned long long *>(csm);                          // [R]
    int32_t *d = reinterpret_cast<int32_t *>(csm + cl_align16(size_t(R) * 8));                     // [R][n]
    int *stale = reinterpret_cast<int *>(reinterpret_cast<unsigned char *>(d) +
                                         cl_align16(kGlobal ? 0 : size_t(R) * n_max * 4));          // [R]
    unsigned long long *slot = reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(stale) +
                                                                      cl_align16(size_t(R) * 4));   // [2][8]
    unsigned char *cpick = reinterpret_cast<unsigned char *>(slot + 2 * kClMaxK);                    // [n_max]
    unsigned char *rpick = cpick + cl_align16(size_t(n_max));                                        // [R]
    const int i0 = rank * R;
    const int nloc = n - i0 < 0 ? 0 : (n - i0 < R ? n - i0 : R);
    const int32_t *src = costs + off + size_t(i0) * n;
    // the minimum key of owned row il (one warp): the working array's cells, or the matrix with the picked rows and
    // columns reading as mask_value
    auto row_min = [&](int il) -> uint64_t {
        const int ig = i0 + il;
        uint64_t best = kKeyInf;
        for (int j = lane; j < n; j += 32) {
            int32_t x;
            if constexpr (kGlobal) x = (rpick[il] || cpick[j]) ? prm.mask_value : __ldg(src + size_t(il) * n + j);
            else x = d[il * n + j];
            const uint64_t k = pack_key(x, uint32_t(ig * n + j));
            best = k < best ? k : best;
        }
        return warp_min_u64(best);
    };
    if constexpr (kGlobal) {
        for (int k = t; k < n; k += kClThreads) cpick[k] = 0;
        for (int k = t; k < nloc; k += kClThreads) rpick[k] = 0;
    } else {
        for (int k = t; k < nloc * n; k += kClThreads) d[k] = __ldg(src + k);
    }
    __syncthreads();
    for (int il = w; il < nloc; il += kClWarps) { const uint64_t k = row_min(il); if (lane == 0) rk[il] = k; }
    const int iters = (prm.max_iters < 0 || prm.max_iters > n) ? n : prm.max_iters;
    long long total = 0;
    int pairs = 0;
    int32_t last_min = INT32_MAX;
    for (int it = 0; it < iters; ++it) {
        unsigned long long *sl = slot + (it & 1) * kClMaxK;
        __syncthreads();                                  // rk complete
        uint64_t m = t < nloc ? rk[t] : kKeyInf;
        m = warp_min_u64(m);
        if (lane == 0) s_min[w] = m;
        if (t == 0) s_nstale = 0;
        __syncthreads();
        if (t < K) {
            uint64_t g = s_min[0];
#pragma unroll
            for (int k = 1; k < kClWarps; ++k) g = s_min[k] < g ? s_min[k] : g;
            cluster.map_shared_rank(sl, t)[rank] = g;     // push the CTA's arg-min to every CTA
        }
        cluster.sync();
        uint64_t g = sl[0];
        for (int k = 1; k < K; ++k) g = sl[k] < g ? sl[k] : g;
        const int32_t v = key_value(g);
        last_min = v;
        if (prm.stop_above != INT32_MAX && v > prm.stop_above) break;
        if (prm.stop_at_value != INT32_MAX && v >= prm.stop_at_value) break;
        const int e = int(key_index(g)), r = e / n, cc = e - r * n;
        if (rank == 0 && t == 0) { rows_out[o + pairs] = r; cols_out[o + pairs] = cc; }
        ++pairs;
        if (prm.sum_below == INT32_MAX || v < prm.sum_below) total += v;
        if constexpr (kGlobal) {                          // flag row r (its owner) and column cc (every CTA)
            if (t == 0) {
                cpick[cc] = 1;
                if (r >= i0 && r < i0 + nloc) rpick[r - i0] = 1;
            }
        } else if (r >= i0 && r < i0 + nloc) {            // the owner masks row r
            for (int j = t; j < n; j += kClThreads) d[(r - i0) * n + j] = prm.mask_value;
        }
        if (t < nloc) {                                   // every CTA masks column cc in its rows
            const int ig = i0 + t;
            if constexpr (!kGlobal) d[t * n + cc] = prm.mask_value;
            const uint64_t k = rk[t];
            if (ig == r) rk[t] = pack_key(prm.mask_value, uint32_t(r * n));
            else if (int(key_index(k)) - ig * n == cc) stale[atomicAdd(&s_nstale, 1)] = t;
            else { const uint64_t km = pack_key(prm.mask_value, uint32_t(ig * n + cc)); rk[t] = km < k ? km : k; }
        }
        __syncthreads();                                  // mask written, stale list complete
        const int ns = s_nstale;
        for (int s = w; s < ns; s += kClWarps) {
            const int il = stale[s];
            const uint64_t k = row_min(il);
            if (lane == 0) rk[il] = k;
        }
        if (prm.residual_size > 0 && n - pairs == prm.residual_size) break;
    }
    if (rank == 0) {
        for (int k = pairs + t; k < n_max; k += kClThreads) { rows_out[o + k] = -1; cols_out[o + k] = -1; }
        if (t == 0) {
            n_pairs_out[b] = pairs; total_out[b] = total;
            if (last_min_out) last_min_out[b] = last_min;
        }
    }
    cluster.sync();
}

// ---- host side ----------------------------------------------------------------------------------------------------------
// DSMEM form: the smallest cluster whose per-CTA block fits next to its O(n) state.  Global form: the smallest of {4, 8}
// that leaves at most one column / row per thread.  Both depend on n_max only.
template <typename Bytes>
static int cluster_ctas(int n_max, bool global, Bytes bytes) {
    if (global) return cl_block(n_max, 4) <= kClThreads ? 4 : 8;
    for (int k = 1; k <= kClMaxK; k *= 2)
        if (bytes(n_max, cl_block(n_max, k), false) + kClStaticReserve <= kClSmemLimit) return k;
    return 0;
}
static size_t asg_cl_bytes(int n_max, int B, bool global) { return asg_cl_layout(n_max, B, global).bytes; }

template <typename... Exp, typename... Act>
static int launch_clusters(void (*kernel)(Exp...), const char *name, int batch, int k, size_t smem, cudaStream_t st,
                           Act... args) {
    if (k == 0 || (long long)batch * k > INT_MAX) return TD_ERR_INVALID;
    TD_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(batch * k));
    cfg.blockDim = dim3(kClThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = unsigned(k);
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int active = 0;
    TD_CUDA_TRY(cudaOccupancyMaxActiveClusters(&active, kernel, &cfg));
    if (active <= 0) {                       // such a cluster can never be resident: refuse instead of hanging
        char what[160];
        snprintf(what, sizeof what, "%s: no cluster of %d CTAs x %zu B of shared memory fits this device", name, k, smem);
        set_cuda_error(cudaErrorInvalidConfiguration, what);
        return TD_ERR_CUDA;
    }
    TD_CUDA_TRY(cudaLaunchKernelEx(&cfg, kernel, args...));
    TD_LAUNCH_CHECK();
    return TD_OK;
}

// The argument rules of the four entry points; they differ in the storage form and its size limit only.
template <bool kGlobal>
static int assign_batch(const char *name, int max_n, const int32_t *costs, const int32_t *sizes, const int64_t *offsets,
                        int batch, int n_max, int32_t *col_of_row_out, int64_t *objective_out, int64_t *u_out,
                        int64_t *v_out, void *stream) {
    if (batch < 0 || n_max < 0 || n_max > max_n) return TD_ERR_INVALID;
    if (batch == 0) return TD_OK;
    if (!costs || !sizes || !offsets || !col_of_row_out || !objective_out) return TD_ERR_INVALID;
    if ((reinterpret_cast<uintptr_t>(costs) & 15) != 0) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    const int k = cluster_ctas(n_max, kGlobal, asg_cl_bytes);
    const int B = k ? cl_block(n_max, k) : 0;
    return launch_clusters(assign_cluster_kernel<kGlobal>, name, batch, k, asg_cl_bytes(n_max, B, kGlobal),
                           static_cast<cudaStream_t>(stream), costs, sizes, offsets, n_max, B, col_of_row_out,
                           reinterpret_cast<long long *>(objective_out), reinterpret_cast<long long *>(u_out),
                           reinterpret_cast<long long *>(v_out));
}

template <bool kGlobal>
static int lcm_batch(const char *name, int max_n, const int32_t *costs, const int32_t *sizes, const int64_t *offsets,
                     int batch, int n_max, const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out,
                     int32_t *n_pairs_out, int64_t *total_out, int32_t *last_min_out, void *stream) {
    if (batch < 0 || n_max < 0 || n_max > max_n) return TD_ERR_INVALID;
    if (batch == 0) return TD_OK;
    if (!costs || !sizes || !offsets || !params || !rows_out || !cols_out || !n_pairs_out || !total_out) return TD_ERR_INVALID;
    if ((reinterpret_cast<uintptr_t>(costs) & 15) != 0) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    const int k = cluster_ctas(n_max, kGlobal, lcm_cl_bytes);
    const int R = k ? cl_block(n_max, k) : 0;
    return launch_clusters(lcm_cluster_kernel<kGlobal>, name, batch, k, lcm_cl_bytes(n_max, R, kGlobal),
                           static_cast<cudaStream_t>(stream), costs, sizes, offsets, n_max, R, *params, rows_out, cols_out,
                           n_pairs_out, reinterpret_cast<long long *>(total_out), last_min_out);
}

}  // namespace td

extern "C" int td_assign_exact_batch_cluster(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch,
                                             int n_max, int32_t *col_of_row_out, int64_t *objective_out, int64_t *u_out,
                                             int64_t *v_out, void *stream) {
    return td::assign_batch<false>("td_assign_exact_batch_cluster", TD_BATCH_CLUSTER_MAX_N, costs, sizes, offsets, batch,
                                   n_max, col_of_row_out, objective_out, u_out, v_out, stream);
}

extern "C" int td_lcm_batch_cluster(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                                    const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out, int32_t *n_pairs_out,
                                    int64_t *total_out, int32_t *last_min_out, void *stream) {
    return td::lcm_batch<false>("td_lcm_batch_cluster", TD_BATCH_CLUSTER_MAX_N, costs, sizes, offsets, batch, n_max, params,
                                rows_out, cols_out, n_pairs_out, total_out, last_min_out, stream);
}

extern "C" int td_assign_exact_batch_large(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch,
                                           int n_max, int32_t *col_of_row_out, int64_t *objective_out, int64_t *u_out,
                                           int64_t *v_out, void *stream) {
    return td::assign_batch<true>("td_assign_exact_batch_large", TD_BATCH_LARGE_MAX_N, costs, sizes, offsets, batch, n_max,
                                  col_of_row_out, objective_out, u_out, v_out, stream);
}

extern "C" int td_lcm_batch_large(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                                  const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out, int32_t *n_pairs_out,
                                  int64_t *total_out, int32_t *last_min_out, void *stream) {
    return td::lcm_batch<true>("td_lcm_batch_large", TD_BATCH_LARGE_MAX_N, costs, sizes, offsets, batch, n_max, params,
                               rows_out, cols_out, n_pairs_out, total_out, last_min_out, stream);
}
