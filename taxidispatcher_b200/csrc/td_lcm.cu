// td_lcm.cu -- K3: the LCM ("lowest cost method") greedy, bit-exact trace.
//
// Replaces heuristic.py:24-33, split.py:161-175, greedy_opt.py:61-82, simulate.py:76-97 and
// Simulator.LCM (Simulator.java:523-549).  The reference repeats n times: first-index argmin of
// the whole n*n array, then overwrite that row and column with a mask VALUE.
//
// The sequential chain is replaced by an equivalent parallel greedy.  Under the strict total
// order key(i,j) = (cost, i*n+j) the literal algorithm picks, each iteration, the smallest FREE
// cell (as long as the mask value does not win the argmin -- see the tail rule below).  A free
// cell that is simultaneously the smallest free cell of its row and of its column ("locally
// dominant") is picked by the sequential greedy no matter what happens elsewhere, so every round
// selects ALL dominant cells at once; the picks of all rounds sorted by key ARE the sequential
// trace.  The global minimum is always dominant, so every round makes progress.
//
//   lcm_transpose        cost^T, so that column minima are contiguous scans as well
//   lcm_rounds (coop)    per-row / per-column cached minima; round = select (thread per row) ->
//                        grid sync -> rescan stale lines (warp per line) -> grid sync
//   lcm_rank_sort        picks -> ascending key order (= pick order of the reference)
//   lcm_finalize         stop rules (greedy_opt.py:69, Simulator.java:538,545), totals
//                        (split.py:167) and the "mask is a value" tail (SURVEY.md section 4 trap 4)
//
// Tail rule.  Masked cells hold mask_value and keep taking part in the argmin.  After t >= 1
// picks the smallest masked cell in first-index order is (0,0) if row 0 has been masked, else
// (0, min masked column).  The first time that (mask_value, that index) beats the smallest free
// key, the literal algorithm re-selects a masked cell; this masks row 0, after which cell (0,0)
// wins every remaining iteration.  lcm_finalize reproduces exactly that.
//
// Algorithmic bytes: 4*n^2 (every cost read once).  Actual traffic is higher (transpose + stale
// rescans) but L2-resident at n = 2000 (16 MB); the kernel is latency/sync-bound, not HBM-bound.
#include "td_common.cuh"
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace td {

struct LcmCtrl {
    unsigned long long gmin[3];  // smallest cached row key over free rows, one slot per round mod 3
    unsigned int n_picked;
    unsigned int rounds;
    unsigned long long g_final;  // gmin at termination (kKeyInf when no free row is left)
};

constexpr int kLcmThreads = 512;

__global__ void lcm_transpose_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, int n) {
    __shared__ int32_t tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int i = by + r, j = bx + threadIdx.x;
        if (i < n && j < n) tile[r][threadIdx.x] = in[size_t(i) * n + j];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int j = bx + r, i = by + threadIdx.x;
        if (i < n && j < n) out[size_t(j) * n + i] = tile[threadIdx.x][r];
    }
}

// min key over the still-free entries of one contiguous line (a row of cost or of cost^T).
// The rounds are latency-bound (a line is 8 KB at n = 2000 and comes from L2), so the scan keeps as many
// loads in flight as it can: 4 x 16-byte cost loads + 4 x 4-byte flag loads per lane per trip when the
// line is 16-byte aligned (n % 4 == 0), 4 scalar loads per trip otherwise.
template <bool kIsRow>
__device__ __forceinline__ uint64_t scan_line(const int32_t *__restrict__ line, int n, int fixed,
                                              const uint8_t *other_free, int lane, bool vec) {
    uint64_t best = kKeyInf;
    auto key_of = [&](int32_t v, int t) -> uint64_t {
        return pack_key(v, kIsRow ? uint32_t(fixed) * n + t : uint32_t(t) * n + fixed);
    };
    if (vec) {
        const int nq = n >> 2;   // int4 groups
        for (int g0 = lane; g0 < nq; g0 += 128) {
            int4 c[4];
            uchar4 f[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int gq = g0 + 32 * u;
                if (gq < nq) {
                    c[u] = *reinterpret_cast<const int4 *>(line + 4 * gq);
                    f[u] = *reinterpret_cast<const uchar4 *>(other_free + 4 * gq);
                } else {
                    f[u] = make_uchar4(0, 0, 0, 0);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int t = 4 * (g0 + 32 * u);
                if (f[u].x) { const uint64_t k = key_of(c[u].x, t); best = k < best ? k : best; }
                if (f[u].y) { const uint64_t k = key_of(c[u].y, t + 1); best = k < best ? k : best; }
                if (f[u].z) { const uint64_t k = key_of(c[u].z, t + 2); best = k < best ? k : best; }
                if (f[u].w) { const uint64_t k = key_of(c[u].w, t + 3); best = k < best ? k : best; }
            }
        }
        return warp_min_u64(best);
    }
    int t = lane;
    for (; t + 96 < n; t += 128) {  // 4 independent loads in flight per lane
        int32_t v0 = line[t], v1 = line[t + 32], v2 = line[t + 64], v3 = line[t + 96];
        uint8_t f0 = other_free[t], f1 = other_free[t + 32], f2 = other_free[t + 64], f3 = other_free[t + 96];
        uint64_t k0 = key_of(v0, t), k1 = key_of(v1, t + 32), k2 = key_of(v2, t + 64), k3 = key_of(v3, t + 96);
        if (f0 && k0 < best) best = k0;
        if (f1 && k1 < best) best = k1;
        if (f2 && k2 < best) best = k2;
        if (f3 && k3 < best) best = k3;
    }
    for (; t < n; t += 32) {
        if (other_free[t]) {
            uint64_t k = key_of(line[t], t);
            if (k < best) best = k;
        }
    }
    return warp_min_u64(best);
}

__global__ void __launch_bounds__(kLcmThreads)
lcm_rounds_kernel(const int32_t *__restrict__ cost, const int32_t *__restrict__ costT, int n, int vec,
                  td_lcm_params prm, unsigned long long *rowkey, unsigned long long *colkey,
                  uint8_t *rowfree, uint8_t *colfree, unsigned long long *picked, LcmCtrl *ctrl) {
    cg::grid_group grid = cg::this_grid();
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nthreads = gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    const int gwarp = tid >> 5;
    const int nwarps = nthreads >> 5;
    __shared__ unsigned long long s_min[kLcmThreads / 32];

    // ---- init: everything free, all caches computed ------------------------------------------
    for (int i = tid; i < n; i += nthreads) { rowfree[i] = 1; colfree[i] = 1; }
    if (tid == 0) {
        ctrl->gmin[0] = ctrl->gmin[1] = ctrl->gmin[2] = kKeyInf;
        ctrl->n_picked = 0; ctrl->rounds = 0; ctrl->g_final = kKeyInf;
    }
    grid.sync();
    for (int l = gwarp; l < 2 * n; l += nwarps) {
        if (l < n) {
            uint64_t k = scan_line<true>(cost + size_t(l) * n, n, l, colfree, lane, vec != 0);
            if (lane == 0) rowkey[l] = k;
        } else {
            int j = l - n;
            uint64_t k = scan_line<false>(costT + size_t(j) * n, n, j, rowfree, lane, vec != 0);
            if (lane == 0) colkey[j] = k;
        }
    }
    grid.sync();

    for (unsigned round = 0;; ++round) {
        // ---- select: row i takes its cached cell iff that cell is also its column's minimum ----
        for (int i = tid; i < n; i += nthreads) {
            if (!rowfree[i]) continue;
            unsigned long long k = rowkey[i];
            if (k == kKeyInf) continue;
            int j = int(key_index(k) - uint32_t(i) * n);
            if (colkey[j] == k) {
                unsigned slot = atomicAdd(&ctrl->n_picked, 1u);
                picked[slot] = k;
                rowfree[i] = 0;
                colfree[j] = 0;
            }
        }
        if (tid == 0) ctrl->gmin[(round + 1) % 3] = kKeyInf;
        grid.sync();
        // ---- refresh stale caches (cached partner was just taken); track the global free minimum
        unsigned long long wmin = kKeyInf;
        for (int l = gwarp; l < 2 * n; l += nwarps) {
            if (l < n) {
                if (!rowfree[l]) continue;
                unsigned long long k = rowkey[l];
                if (k != kKeyInf && !colfree[key_index(k) - uint32_t(l) * n]) {
                    k = scan_line<true>(cost + size_t(l) * n, n, l, colfree, lane, vec != 0);
                    if (lane == 0) rowkey[l] = k;
                }
                if (k < wmin) wmin = k;
            } else {
                int j = l - n;
                if (!colfree[j]) continue;
                unsigned long long k = colkey[j];
                if (k != kKeyInf && !rowfree[(key_index(k) - uint32_t(j)) / uint32_t(n)]) {
                    k = scan_line<false>(costT + size_t(j) * n, n, j, rowfree, lane, vec != 0);
                    if (lane == 0) colkey[j] = k;
                }
            }
        }
        if (lane == 0) s_min[threadIdx.x >> 5] = wmin;
        __syncthreads();
        if (threadIdx.x < 32) {
            unsigned long long v = threadIdx.x < (kLcmThreads / 32) ? s_min[threadIdx.x] : kKeyInf;
            v = warp_min_u64(v);
            if (threadIdx.x == 0 && v != kKeyInf) atomicMin(&ctrl->gmin[round % 3], v);
        }
        grid.sync();
        // ---- termination: nothing free, or the smallest free value can never be recorded ------
        const unsigned long long g = ctrl->gmin[round % 3];
        bool done = (g == kKeyInf);
        if (!done) {
            const int32_t v = key_value(g);
            if (prm.stop_above != INT32_MAX && v > prm.stop_above) done = true;
            if (prm.stop_at_value != INT32_MAX && v >= prm.stop_at_value) done = true;
            if (v > prm.mask_value) done = true;  // a masked cell wins every later argmin
        }
        if (done) {
            if (tid == 0) { ctrl->g_final = g; ctrl->rounds = round + 1; }
            break;
        }
    }
}

// Small / medium instances (the state fits in shared memory: 18 n bytes): every CTA keeps a FULL replica of
// the cached minima and of the free flags.  The selection and the staleness test are then pure shared-memory
// work that every CTA repeats identically (no communication), the rescans of the stale lines are split over
// the CTAs, and ONE grid.sync per round publishes the refreshed minima, which every CTA then pulls into its
// replica.  Half the barriers and none of the dependent global round trips of the generic kernel.
__global__ void __launch_bounds__(kLcmThreads)
lcm_rounds_smem_kernel(const int32_t *__restrict__ cost, const int32_t *__restrict__ costT, int n, int vec,
                       td_lcm_params prm, unsigned long long *gkey /* 2n: rows then columns */,
                       unsigned long long *picked, LcmCtrl *ctrl) {
    cg::grid_group grid = cg::this_grid();
    extern __shared__ __align__(16) unsigned char lsm[];
    unsigned long long *rk = reinterpret_cast<unsigned long long *>(lsm);          // row minima
    unsigned long long *ck = rk + n;                                                // column minima
    const int nf = (n + 15) & ~15;
    uint8_t *rf = reinterpret_cast<uint8_t *>(ck + n);                              // row free flags
    uint8_t *cf = rf + nf;                                                          // column free flags
    int *mine = reinterpret_cast<int *>(cf + nf);                                   // stale lines this CTA rescans (<= 2n)
    __shared__ int s_nmine;
    __shared__ unsigned long long s_min[kLcmThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = kLcmThreads / 32;
    const int G = gridDim.x, b = blockIdx.x;
    const bool v = vec != 0;

    for (int i = tid; i < n; i += kLcmThreads) { rf[i] = 1; cf[i] = 1; }
    if (b == 0 && tid == 0) { ctrl->n_picked = 0; ctrl->rounds = 0; ctrl->g_final = kKeyInf; }
    __syncthreads();
    // initial minima: line l belongs to CTA l % G
    for (int l = b + G * warp; l < 2 * n; l += G * nw) {
        const unsigned long long k = l < n ? scan_line<true>(cost + size_t(l) * n, n, l, cf, lane, v)
                                           : scan_line<false>(costT + size_t(l - n) * n, n, l - n, rf, lane, v);
        if (lane == 0) gkey[l] = k;
    }
    grid.sync();
    for (int l = tid; l < 2 * n; l += kLcmThreads) { const unsigned long long k = __ldcg(gkey + l); if (l < n) rk[l] = k; else ck[l - n] = k; }
    __syncthreads();

    auto stale = [&](int l) -> bool {   // free line whose cached partner has been taken
        if (l < n) { const unsigned long long k = rk[l]; return rf[l] && k != kKeyInf && !cf[key_index(k) - uint32_t(l) * n]; }
        const int j = l - n;
        const unsigned long long k = ck[j];
        return cf[j] && k != kKeyInf && !rf[(key_index(k) - uint32_t(j)) / uint32_t(n)];
    };
    for (unsigned round = 0;; ++round) {
        // ---- select (replicated): row i takes its cached cell iff it is also its column's minimum ----
        for (int i = tid; i < n; i += kLcmThreads) {
            if (!rf[i]) continue;
            const unsigned long long k = rk[i];
            if (k == kKeyInf) continue;
            const int j = int(key_index(k) - uint32_t(i) * n);
            if (ck[j] == k) {
                rf[i] = 0; cf[j] = 0;
                if (b == 0) picked[atomicAdd(&ctrl->n_picked, 1u)] = k;
            }
        }
        if (tid == 0) s_nmine = 0;
        __syncthreads();
        // ---- stale lines: this CTA rescans those with l % G == b ----
        for (int l = b + G * tid; l < 2 * n; l += G * kLcmThreads)   // the lines with l % G == b, no division
            if (stale(l)) mine[atomicAdd(&s_nmine, 1)] = l;
        __syncthreads();
        const int nm = s_nmine;
        for (int t = warp; t < nm; t += nw) {
            const int l = mine[t];
            const unsigned long long k = l < n ? scan_line<true>(cost + size_t(l) * n, n, l, cf, lane, v)
                                               : scan_line<false>(costT + size_t(l - n) * n, n, l - n, rf, lane, v);
            if (lane == 0) __stcg(gkey + l, k);
        }
        grid.sync();
        // ---- pull the refreshed minima into the replica (the predicate still sees the old keys) ----
        for (int l = tid; l < 2 * n; l += kLcmThreads)
            if (stale(l)) { const unsigned long long k = __ldcg(gkey + l); if (l < n) rk[l] = k; else ck[l - n] = k; }
        __syncthreads();
        // ---- smallest free key (replicated) -> termination ----
        unsigned long long m = kKeyInf;
        for (int i = tid; i < n; i += kLcmThreads) if (rf[i] && rk[i] < m) m = rk[i];
        m = warp_min_u64(m);
        if (lane == 0) s_min[warp] = m;
        __syncthreads();
        unsigned long long g = s_min[0];
        for (int w2 = 1; w2 < nw; ++w2) g = s_min[w2] < g ? s_min[w2] : g;
        __syncthreads();
        bool done = (g == kKeyInf);
        if (!done) {
            const int32_t val = key_value(g);
            if (prm.stop_above != INT32_MAX && val > prm.stop_above) done = true;
            if (prm.stop_at_value != INT32_MAX && val >= prm.stop_at_value) done = true;
            if (val > prm.mask_value) done = true;  // a masked cell wins every later argmin
        }
        if (done) {
            if (b == 0 && tid == 0) { ctrl->g_final = g; ctrl->rounds = round + 1; }
            break;
        }
    }
}

// ascending key order by counting smaller keys (P <= n picks; keys are unique)
__global__ void lcm_rank_sort_kernel(const unsigned long long *__restrict__ picked,
                                     unsigned long long *__restrict__ sorted, const LcmCtrl *ctrl) {
    __shared__ unsigned long long tile[1024];
    const int P = int(ctrl->n_picked);
    const int base = blockIdx.x * blockDim.x;
    if (base >= P) return;
    const int me = base + threadIdx.x;
    const unsigned long long mine = me < P ? picked[me] : kKeyInf;
    int rank = 0;
    for (int t0 = 0; t0 < P; t0 += 1024) {
        __syncthreads();
        for (int t = threadIdx.x; t < 1024; t += blockDim.x) tile[t] = (t0 + t < P) ? picked[t0 + t] : kKeyInf;
        __syncthreads();
        const int m = (P - t0) < 1024 ? (P - t0) : 1024;
        for (int t = 0; t < m; ++t) rank += tile[t] < mine;
    }
    if (me < P) sorted[rank] = mine;
}

constexpr int kFinThreads = 1024;

// Walks the sorted picks exactly like the literal loop would, in parallel.
__global__ void __launch_bounds__(kFinThreads)
lcm_finalize_kernel(const unsigned long long *__restrict__ sorted, int n, td_lcm_params prm, const LcmCtrl *ctrl,
                    int32_t *rows_out, int32_t *cols_out, int32_t *n_pairs_out, long long *total_out,
                    int32_t *last_min_out) {
    __shared__ int s_has0[kFinThreads];
    __shared__ int s_minc[kFinThreads];
    __shared__ int s_event;       // first index at which the literal loop leaves the "free pick" regime
    __shared__ long long s_sum[kFinThreads / 32];
    const int tid = threadIdx.x;
    const int P = int(ctrl->n_picked);
    const int iters = (prm.max_iters < 0 || prm.max_iters > n) ? n : prm.max_iters;
    const int chunk = (P + kFinThreads - 1) / kFinThreads;
    const int lo = min(tid * chunk, P), hi = min(lo + chunk, P);

    // exclusive prefix of (row 0 masked?, smallest masked column) over the sorted picks
    int has0 = 0, minc = INT_MAX;
    for (int t = lo; t < hi; ++t) {
        uint32_t idx = key_index(sorted[t]);
        int r = int(idx / uint32_t(n)), c = int(idx - uint32_t(r) * n);
        has0 |= (r == 0);
        minc = c < minc ? c : minc;
    }
    s_has0[tid] = has0; s_minc[tid] = minc;
    if (tid == 0) s_event = INT_MAX;
    __syncthreads();
    if (tid == 0) {  // serial exclusive scan over 1024 aggregates
        int h = 0, m = INT_MAX;
        for (int t = 0; t < kFinThreads; ++t) {
            int nh = h | s_has0[t], nm = min(m, s_minc[t]);
            s_has0[t] = h; s_minc[t] = m; h = nh; m = nm;
        }
    }
    __syncthreads();
    has0 = s_has0[tid]; minc = s_minc[tid];
    // first index t where (a) a masked cell beats sorted[t], or (b) sorted[t] trips a stop rule
    int ev = INT_MAX;
    for (int t = lo; t < hi; ++t) {
        const unsigned long long fk = sorted[t];
        const int32_t v = key_value(fk);
        bool hit = false;
        if (t >= 1) {
            unsigned long long mk = pack_key(prm.mask_value, has0 ? 0u : uint32_t(minc));
            if (mk < fk) hit = true;
        }
        if (prm.stop_above != INT32_MAX && v > prm.stop_above) hit = true;
        if (prm.stop_at_value != INT32_MAX && v >= prm.stop_at_value) hit = true;
        if (hit) { ev = t; break; }
        uint32_t idx = key_index(fk);
        int r = int(idx / uint32_t(n)), c = int(idx - uint32_t(r) * n);
        has0 |= (r == 0);
        minc = c < minc ? c : minc;
    }
    if (ev != INT_MAX) atomicMin(&s_event, ev);
    __syncthreads();
    // free-pick regime covers iterations [0, t_free)
    int t_free = min(s_event, P);
    t_free = min(t_free, iters);
    int pairs_cap = INT_MAX;  // Simulator.java:545 -- break once n - pairs == residual_size
    if (prm.residual_size > 0 && n - prm.residual_size >= 1) pairs_cap = n - prm.residual_size;
    bool residual_hit = false;
    if (t_free >= pairs_cap) { t_free = pairs_cap; residual_hit = true; }

    long long sum = 0;
    for (int t = tid; t < t_free; t += kFinThreads) {
        const unsigned long long fk = sorted[t];
        uint32_t idx = key_index(fk);
        int r = int(idx / uint32_t(n));
        rows_out[t] = r;
        cols_out[t] = int(idx - uint32_t(r) * n);
        const int32_t v = key_value(fk);
        if (prm.sum_below == INT32_MAX || v < prm.sum_below) sum += v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((tid & 31) == 0) s_sum[tid >> 5] = sum;
    __syncthreads();
    if (tid != 0) return;
    long long total = 0;
    for (int w = 0; w < kFinThreads / 32; ++w) total += s_sum[w];
    int pairs = t_free;
    int32_t last_min = t_free > 0 ? key_value(sorted[t_free - 1]) : INT32_MAX;
    if (!residual_hit && t_free < iters) {
        // state after t_free free picks
        int h = 0, m = INT_MAX;
        {   // recompute the prefix state at t_free (cheap: at most one chunk beyond a stored prefix)
            int owner = chunk > 0 ? min(t_free / chunk, kFinThreads - 1) : 0;
            h = s_has0[owner]; m = s_minc[owner];
            for (int t = owner * chunk; t < t_free; ++t) {
                uint32_t idx = key_index(sorted[t]);
                int r = int(idx / uint32_t(n)), c = int(idx - uint32_t(r) * n);
                h |= (r == 0); m = min(m, c);
            }
        }
        // candidate of iteration t_free: smallest free key (a remaining pick, or the minimum left
        // behind when the rounds stopped) against the smallest masked cell
        unsigned long long fk = t_free < P ? sorted[t_free] : ctrl->g_final;
        unsigned long long mk = t_free >= 1 ? pack_key(prm.mask_value, h ? 0u : uint32_t(m)) : kKeyInf;
        unsigned long long cand = fk < mk ? fk : mk;
        if (cand != kKeyInf) {
            int32_t v = key_value(cand);
            last_min = v;
            bool stop = (prm.stop_above != INT32_MAX && v > prm.stop_above) ||
                        (prm.stop_at_value != INT32_MAX && v >= prm.stop_at_value);
            if (!stop) {
                // only a masked cell can get here (a free key that passes the stop rules and beats
                // the mask would have been part of the free regime)
                int t = t_free;
                int col0 = h ? 0 : m;  // first degenerate pick is (0, col0); all later ones are (0,0)
                while (t < iters) {
                    rows_out[t] = 0;
                    cols_out[t] = (t == t_free) ? col0 : 0;
                    if (prm.sum_below == INT32_MAX || v < prm.sum_below) total += v;
                    ++t; ++pairs;
                    if (pairs >= pairs_cap) break;
                }
            }
        }
    }
    *n_pairs_out = pairs;
    *total_out = total;
    if (last_min_out) *last_min_out = last_min;
}

// ---- batches of small instances: one CTA per instance, the literal array algorithm in shared memory ---------------------
// The working array d (n x n, n <= TD_BATCH_MAX_N) lives in shared memory and is overwritten with mask_value exactly like the
// reference does, so "the mask is a value" holds by construction.  rk[i] caches row i's minimum key (value, i*n + j); the
// whole-array first-index argmin is the block minimum of rk.  After row r and column c are masked:
//   row r                   -> (mask, r*n + 0)             (every cell of the row is the mask now)
//   a row cached at column c -> rescanned, one warp per row  (its minimum just changed to something unknown)
//   every other row          -> min(rk[i], (mask, i*n + c))  (only cell c changed, and it was not the minimum)
constexpr int kLcmBatchThreads = 256;

__device__ __forceinline__ uint64_t lcm_row_min(const int32_t *d, int n, int i, int lane) {
    uint64_t best = kKeyInf;
    for (int j = lane; j < n; j += 32) { const uint64_t k = pack_key(d[i * n + j], uint32_t(i * n + j)); best = k < best ? k : best; }
    return warp_min_u64(best);
}

__global__ void __launch_bounds__(kLcmBatchThreads)
lcm_batch_kernel(const int32_t *__restrict__ costs, const int32_t *__restrict__ sizes, const int64_t *__restrict__ offsets,
                 int n_max, td_lcm_params prm, int32_t *rows_out, int32_t *cols_out, int32_t *n_pairs_out,
                 long long *total_out, int32_t *last_min_out) {
    extern __shared__ __align__(16) unsigned char lbs[];
    const int b = blockIdx.x;
    const int n = sizes[b];
    const long long off = offsets[b];
    const size_t o = size_t(b) * n_max;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    constexpr int nw = kLcmBatchThreads / 32;
    const bool bad = n < 0 || n > n_max || off < 0 || (off & 3) != 0;
    if (bad) {
        for (int k = t; k < n_max; k += kLcmBatchThreads) { rows_out[o + k] = -1; cols_out[o + k] = -1; }
        if (t == 0) {
            n_pairs_out[b] = -1; total_out[b] = LLONG_MIN;
            if (last_min_out) last_min_out[b] = INT32_MIN;
        }
        return;
    }
    unsigned long long *rk = reinterpret_cast<unsigned long long *>(lbs);      // [n]
    int32_t *d = reinterpret_cast<int32_t *>(rk + n_max);                     // [n][n]
    int *stale = reinterpret_cast<int *>(d + size_t(n_max) * n_max);          // rows to rescan [n]
    __shared__ unsigned long long s_min[nw];
    __shared__ int s_nstale;
    const int32_t *src = costs + off;
    for (int k = t; k < n * n; k += kLcmBatchThreads) d[k] = __ldg(src + k);
    __syncthreads();
    for (int i = w; i < n; i += nw) { const uint64_t k = lcm_row_min(d, n, i, lane); if (lane == 0) rk[i] = k; }
    const int iters = (prm.max_iters < 0 || prm.max_iters > n) ? n : prm.max_iters;
    long long total = 0;
    int pairs = 0;
    int32_t last_min = INT32_MAX;
    for (int it = 0; it < iters; ++it) {
        __syncthreads();                                  // rk complete
        uint64_t m = t < n ? rk[t] : kKeyInf;
        m = warp_min_u64(m);
        if (lane == 0) s_min[w] = m;
        if (t == 0) s_nstale = 0;
        __syncthreads();
        uint64_t g = s_min[0];
#pragma unroll
        for (int k = 1; k < nw; ++k) g = s_min[k] < g ? s_min[k] : g;
        const int32_t v = key_value(g);
        last_min = v;
        if (prm.stop_above != INT32_MAX && v > prm.stop_above) break;
        if (prm.stop_at_value != INT32_MAX && v >= prm.stop_at_value) break;
        const int e = int(key_index(g)), r = e / n, c = e - r * n;
        if (t == 0) { rows_out[o + pairs] = r; cols_out[o + pairs] = c; }
        ++pairs;
        if (prm.sum_below == INT32_MAX || v < prm.sum_below) total += v;
        if (t < n) {
            d[r * n + t] = prm.mask_value;
            d[t * n + c] = prm.mask_value;
            const uint64_t k = rk[t];
            if (t == r) rk[t] = pack_key(prm.mask_value, uint32_t(r * n));
            else if (int(key_index(k)) - t * n == c) stale[atomicAdd(&s_nstale, 1)] = t;
            else { const uint64_t km = pack_key(prm.mask_value, uint32_t(t * n + c)); rk[t] = km < k ? km : k; }
        }
        __syncthreads();                                  // mask written, stale list complete
        const int ns = s_nstale;
        for (int s = w; s < ns; s += nw) { const int i = stale[s]; const uint64_t k = lcm_row_min(d, n, i, lane); if (lane == 0) rk[i] = k; }
        if (prm.residual_size > 0 && n - pairs == prm.residual_size) break;
    }
    for (int k = pairs + t; k < n_max; k += kLcmBatchThreads) { rows_out[o + k] = -1; cols_out[o + k] = -1; }
    if (t == 0) {
        n_pairs_out[b] = pairs; total_out[b] = total;
        if (last_min_out) last_min_out[b] = last_min;
    }
}

static size_t lcm_batch_smem_bytes(int n_max) {
    return size_t(n_max) * 8 + size_t(n_max) * n_max * 4 + size_t(n_max) * 4;
}

struct LcmWorkspace {
    int32_t *costT;
    unsigned long long *rowkey, *colkey, *picked, *sorted, *gkey2;
    uint8_t *rowfree, *colfree;
    LcmCtrl *ctrl;
    size_t bytes;
};

static LcmWorkspace carve_lcm(void *ws, int n) {
    Carver c(ws);
    LcmWorkspace w;
    w.costT = c.take<int32_t>(size_t(n) * n);
    w.rowkey = c.take<unsigned long long>(n);
    w.colkey = c.take<unsigned long long>(n);
    w.picked = c.take<unsigned long long>(n);
    w.sorted = c.take<unsigned long long>(n);
    w.gkey2 = c.take<unsigned long long>(size_t(2) * n);
    w.rowfree = c.take<uint8_t>(n);
    w.colfree = c.take<uint8_t>(n);
    w.ctrl = c.take<LcmCtrl>(1);
    w.bytes = c.used();
    return w;
}

}  // namespace td

extern "C" size_t td_lcm_workspace_bytes(int n) {
    if (n <= 0) return 256;
    return td::carve_lcm(nullptr, n).bytes;
}

extern "C" int td_lcm(const int32_t *cost, int n, const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out,
                      int32_t *n_pairs_out, int64_t *total_out, int32_t *last_min_out, void *workspace,
                      size_t workspace_bytes, void *stream) {
    using namespace td;
    if (n < 0 || !params || !n_pairs_out || !total_out) return TD_ERR_INVALID;
    if (n > 65535) return TD_ERR_INVALID;  // flat index n*n must fit the 32-bit half of the key
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n == 0) {
        TD_CUDA_TRY(cudaMemsetAsync(n_pairs_out, 0, sizeof(int32_t), st));
        TD_CUDA_TRY(cudaMemsetAsync(total_out, 0, sizeof(int64_t), st));
        return TD_OK;
    }
    if (!cost || !rows_out || !cols_out || !workspace) return TD_ERR_INVALID;
    if (workspace_bytes < td_lcm_workspace_bytes(n)) return TD_ERR_WORKSPACE;
    LcmWorkspace w = carve_lcm(workspace, n);

    dim3 tb(32, 8), tg((n + 31) / 32, (n + 31) / 32);
    lcm_transpose_kernel<<<tg, tb, 0, st>>>(cost, w.costT, n);
    TD_LAUNCH_CHECK();

    td_lcm_params prm = *params;
    const int32_t *costT = w.costT;
    // 16-byte loads need aligned lines: n % 4 == 0 and aligned bases (the flag arrays are 16-byte aligned)
    int vec = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(cost) & 15) == 0) ? 1 : 0;
    const size_t smem_need = size_t(n) * 16 + 2 * size_t((n + 15) & ~15) + size_t(2 * n) * 4 + 64;
    if (smem_need <= 200 * 1024 && !getenv("TD_LCM_GENERIC")) {
        // replicated-state kernel: one CTA per SM at most, never more CTAs than a quarter of the lines
        TD_CUDA_TRY(cudaFuncSetAttribute(lcm_rounds_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(200 * 1024)));
        int grid = device_sm_count();
        const int cap_grid = (2 * n + 3) / 4;
        if (grid > cap_grid) grid = cap_grid < 1 ? 1 : cap_grid;
        unsigned long long *gkey = w.gkey2;
        void *args[] = {(void *)&cost, (void *)&costT, (void *)&n, (void *)&vec, (void *)&prm, (void *)&gkey, (void *)&w.picked,
                        (void *)&w.ctrl};
        ProfScope prof(TD_PROF_LCM, st);
        TD_CUDA_TRY(cudaLaunchCooperativeKernel((void *)lcm_rounds_smem_kernel, dim3(grid), dim3(kLcmThreads), args, smem_need, st));
    } else {
        int per_sm = 0;
        TD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lcm_rounds_kernel, kLcmThreads, 0));
        if (per_sm < 1) return TD_ERR_CUDA;
        per_sm = per_sm > 2 ? 2 : per_sm;
        int grid = device_sm_count() * per_sm;
        // no point in more warps than lines to scan (2n); keeps grid.sync cheap for small n
        int need = (2 * n * 32 + kLcmThreads - 1) / kLcmThreads;
        if (grid > need) grid = need < 1 ? 1 : need;
        void *args[] = {(void *)&cost, (void *)&costT, (void *)&n, (void *)&vec, (void *)&prm, (void *)&w.rowkey, (void *)&w.colkey,
                        (void *)&w.rowfree, (void *)&w.colfree, (void *)&w.picked, (void *)&w.ctrl};
        ProfScope prof(TD_PROF_LCM, st);
        TD_CUDA_TRY(cudaLaunchCooperativeKernel((void *)lcm_rounds_kernel, dim3(grid), dim3(kLcmThreads), args, 0, st));
    }
    count_launch();

    lcm_rank_sort_kernel<<<(n + 255) / 256, 256, 0, st>>>(w.picked, w.sorted, w.ctrl);
    TD_LAUNCH_CHECK();
    lcm_finalize_kernel<<<1, kFinThreads, 0, st>>>(w.sorted, n, prm, w.ctrl, rows_out, cols_out, n_pairs_out,
                                                   reinterpret_cast<long long *>(total_out), last_min_out);
    TD_LAUNCH_CHECK();
    return TD_OK;
}

extern "C" int td_lcm_batch(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                            const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out, int32_t *n_pairs_out,
                            int64_t *total_out, int32_t *last_min_out, void *stream) {
    using namespace td;
    if (batch < 0 || n_max < 0 || n_max > TD_BATCH_MAX_N) return TD_ERR_INVALID;
    if (batch == 0) return TD_OK;
    if (!costs || !sizes || !offsets || !params || !rows_out || !cols_out || !n_pairs_out || !total_out) return TD_ERR_INVALID;
    if ((reinterpret_cast<uintptr_t>(costs) & 15) != 0) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t smem = lcm_batch_smem_bytes(n_max);
    TD_CUDA_TRY(cudaFuncSetAttribute(lcm_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    lcm_batch_kernel<<<batch, kLcmBatchThreads, smem, st>>>(costs, sizes, offsets, n_max, *params, rows_out, cols_out, n_pairs_out,
                                                            reinterpret_cast<long long *>(total_out), last_min_out);
    TD_LAUNCH_CHECK();
    return TD_OK;
}
