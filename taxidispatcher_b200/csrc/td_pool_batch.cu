// td_pool_batch.cu -- the whole `findpool` job (every logical shard of pool_n.c + the merge of findpool.c:83-108) for a
// batch of small demand sets in one launch (see DESIGN.md section 15).
//
// Grid: one CTA per (instance, logical shard).  The shards are independent by definition, exactly like the reference's
// pool_n processes.  A CTA stages the stand table and the instance's customers in shared memory, enumerates the pickup
// tuples of its leaders with the wait rule (pool_n.c:153-177) and evaluates all drop-off orders of each (pool_n.c:101-151).
// Every tuple with a feasible order materialises ONE 64-bit key into the CTA's workspace slice:
//     key = cost << 36 | p0 << 27 | p1 << 18 | p2 << 9 | p3      (unused pickup slots 0)
// n <= 512 gives 9 bits per customer and cost <= 7 * 2^22 < 2^25, so the key is exact for every accepted table.  Its
// order is (cost, lexicographic pickup tuple) = the order of a stable sort by cost of pool_n.c's enumeration; the drop-off
// order is not in the key: a tuple keeps its best order under (cost, lexicographic permutation index) only, as pool_enum
// does, and that order is recomputed at emission.  The greedy scan of removeDuplicates (pool_n.c:187-207) is then run as
// dominance rounds (DESIGN.md section 7): a record whose key is the minimum at all of its customers is kept, its customers
// die, the rest is compacted, repeat.  Equal to stable sort + scan because the keys are distinct.
//
// The CTA that finishes its instance last (atomic ticket after a fence, the pattern of pool_build_lists_kernel) merges the
// shard survivors in shard order with the same rounds: key (cost << 32 | position) for K = 4 and position for K < 4 (the
// findpool.c sort column quirk, SURVEY.md section 4 trap 8), and writes the rows.
#include "td_pool_common.cuh"

namespace td {

constexpr int kPBThreads = 256;
constexpr int kPBWarps = kPBThreads / 32;
constexpr int kPBMaxStands = 128;
constexpr int kPBCustBits = 9;
constexpr int kPBKeptCap = TD_POOL_BATCH_MAX_N / 2 + 1;   // kept plans of one shard or one merge are customer-disjoint
constexpr int kPBQueue = 64;                              // per-warp ring of K = 4 pickup tuples awaiting evaluation
static_assert(TD_POOL_BATCH_MAX_N <= (1 << kPBCustBits), "a customer index must fit the key");

struct PBMeta {                 // per (instance, shard), in the workspace
    int count;                  // survivors at the start of the shard's record slice, sorted by key
    int overflow;               // the slice was too small: no survivors
    long long needed;           // materialised records of the shard
};

struct PBWs {
    unsigned int *ticket;       // [batch]: shard CTAs of the instance that have finished
    PBMeta *meta;               // [batch * n_shards]
    unsigned long long *mlive;  // [batch * n_shards * kPBKeptCap]: the merge's live list
    unsigned long long *recs;   // [batch * n_shards * records_per_shard]
    size_t bytes;
};

__host__ __device__ static PBWs carve_pb(void *base, int batch, int n_shards, long long rps) {
    char *p = static_cast<char *>(base);
    size_t off = 0;
    auto take = [&](size_t bytes) { off = (off + 255) & ~size_t(255); char *r = p + off; off += bytes; return r; };
    PBWs w;
    const size_t slots = size_t(batch) * n_shards;
    w.ticket = reinterpret_cast<unsigned int *>(take(size_t(batch) * sizeof(unsigned int)));
    w.meta = reinterpret_cast<PBMeta *>(take(slots * sizeof(PBMeta)));
    w.mlive = reinterpret_cast<unsigned long long *>(take(slots * kPBKeptCap * 8));
    w.recs = reinterpret_cast<unsigned long long *>(take(slots * size_t(rps) * 8));
    w.bytes = (off + 255) & ~size_t(255);
    return w;
}

__device__ __forceinline__ unsigned long long tuple_rank(int p0, int p1, int p2, int p3) {
    return (unsigned long long)p0 << 27 | (unsigned long long)p1 << 18 | (unsigned)p2 << 9 | (unsigned)p3;
}
__device__ __forceinline__ void key_tuple(unsigned long long key, int p[4]) {
    p[0] = int(key >> 27) & 511; p[1] = int(key >> 18) & 511; p[2] = int(key >> 9) & 511; p[3] = int(key) & 511;
}

// All K! drop-off orders of the pickup tuple p (pool_n.c:101-151).  cust / D are in the fixed point of the evaluation
// (x32 for K = 4, see eval4s).  best = cost << 5 | permutation index of the best feasible order under (cost, index).
template <int K>
__device__ __forceinline__ void eval_tuple(const int p[4], const int4 *cust, const int32_t *D, int S, int &nfeas, int &best) {
    const int4 c0 = cust[p[0]], c1 = cust[p[1]];
    const int a01 = D[c0.x * S + c1.x];
    if (K == 2) {
        const int sl0 = c0.z - a01, sl1 = c1.z;
        const int e0 = D[c1.x * S + c0.y], e1 = D[c1.x * S + c1.y];
        const int t01 = D[c0.y * S + c1.y], t10 = D[c1.y * S + c0.y];
        // perm 0: drop 0 then 1; perm 1: drop 1 then 0
        const bool okA = e0 <= sl0 && e0 + t01 <= sl1;
        const bool okB = e1 <= sl1 && e1 + t10 <= sl0;
        const int kA = ((a01 + e0 + t01) << kPermBits) | 0, kB = ((a01 + e1 + t10) << kPermBits) | 1;
        nfeas = int(okA) + int(okB);
        best = INT_MAX;
        if (okA) best = kA;
        if (okB && kB < best) best = kB;
    } else if (K == 3) {
        const int4 c2 = cust[p[2]];
        const int a12 = D[c1.x * S + c2.x];
        int e[3], t[3][3], sl[3];
        e[0] = D[c2.x * S + c0.y]; e[1] = D[c2.x * S + c1.y]; e[2] = D[c2.x * S + c2.y];
        t[0][0] = t[1][1] = t[2][2] = 0;
        t[0][1] = D[c0.y * S + c1.y]; t[1][0] = D[c1.y * S + c0.y];
        t[0][2] = D[c0.y * S + c2.y]; t[2][0] = D[c2.y * S + c0.y];
        t[1][2] = D[c1.y * S + c2.y]; t[2][1] = D[c2.y * S + c1.y];
        sl[2] = c2.z; sl[1] = c1.z - a12; sl[0] = c0.z - a01 - a12;
        eval3(e, t, sl, a01 + a12, nfeas, best);
    } else {
        const int4 c2 = cust[p[2]], c3 = cust[p[3]];
        const int a12 = D[c1.x * S + c2.x], a23 = D[c2.x * S + c3.x];
        const int4 c[4] = {c0, c1, c2, c3};
        int e[4], t[4][4], sl[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            e[i] = D[c3.x * S + c[i].y];
#pragma unroll
            for (int j = 0; j < 4; ++j) t[i][j] = i == j ? 0 : D[c[i].y * S + c[j].y];
        }
        sl[3] = c3.z; sl[2] = c2.z - a23; sl[1] = c1.z - a12 - a23; sl[0] = c0.z - a01 - a12 - a23;
        eval4s(e, t, sl, nfeas, best);
        if (nfeas > 0) best += a01 + a12 + a23;   // pickup legs (multiples of 32): best = 32 * plan cost + permutation index
    }
}

// Greedy disjoint scan in key order over live[0, m) as dominance rounds; the kept keys go to s_kept (unsorted), their
// count is returned.  cust_of(key, c) gives the K customers of a key.  The live list is compacted in place.
template <int K, class CustOf>
__device__ int dominance_rounds(unsigned long long *live, int m, int n, CustOf cust_of, unsigned long long *s_min,
                                uint8_t *s_dead, unsigned long long *s_kept, int *s_nk, int *s_cnt) {
    const int tid = threadIdx.x;
    for (int c = tid; c < n; c += blockDim.x) s_dead[c] = 0;
    if (tid == 0) *s_nk = 0;
    __syncthreads();
    while (m > 0) {
        for (int c = tid; c < n; c += blockDim.x) s_min[c] = ~0ull;
        __syncthreads();
        for (int i = tid; i < m; i += blockDim.x) {
            const unsigned long long key = live[i];
            int c[4];
            cust_of(key, c);
#pragma unroll
            for (int j = 0; j < K; ++j) atomicMin(&s_min[c[j]], key);
        }
        __syncthreads();
        for (int i = tid; i < m; i += blockDim.x) {
            const unsigned long long key = live[i];
            int c[4];
            cust_of(key, c);
            bool dom = true;
#pragma unroll
            for (int j = 0; j < K; ++j) dom = dom && s_min[c[j]] == key;
            if (dom) {
                const int k = atomicAdd(s_nk, 1);
                if (k < kPBKeptCap) s_kept[k] = key;
#pragma unroll
                for (int j = 0; j < K; ++j) s_dead[c[j]] = 1;
            }
        }
        if (tid == 0) *s_cnt = 0;
        __syncthreads();
        // every thread reads its element of a chunk before any write of that chunk: writes land at or below it
        for (int base = 0; base < m; base += blockDim.x) {
            const int i = base + tid;
            bool keep = false;
            unsigned long long key = 0;
            if (i < m) {
                key = live[i];
                int c[4];
                cust_of(key, c);
                keep = true;
#pragma unroll
                for (int j = 0; j < K; ++j) keep = keep && !s_dead[c[j]];
            }
            __syncthreads();
            if (keep) live[atomicAdd(s_cnt, 1)] = key;
        }
        __syncthreads();
        m = *s_cnt;
        __syncthreads();
    }
    return *s_nk < kPBKeptCap ? *s_nk : kPBKeptCap;
}

// the kept keys in ascending order: dst[rank] = key
__device__ __forceinline__ void sort_kept(const unsigned long long *s_kept, int nk, unsigned long long *dst) {
    for (int i = threadIdx.x; i < nk; i += blockDim.x) {
        const unsigned long long me = s_kept[i];
        int rank = 0;
        for (int q = 0; q < nk; ++q) rank += s_kept[q] < me;
        dst[rank] = me;
    }
}

template <int K>
__global__ void __launch_bounds__(kPBThreads, 2)   // 76 registers for K = 4 without spills (the default heuristic stops at 64 and spills)
pool_batch_kernel(const int32_t *__restrict__ demand, const int32_t *__restrict__ sizes, const int64_t *__restrict__ offsets,
                  int n_max, const int32_t *__restrict__ dist, int S, int n_shards, int32_t *plans_out, int32_t *n_plans_out,
                  long long *evaluated_out, long long *feasible_out, int32_t *kept_out, long long *needed_out, PBWs ws,
                  long long rps) {
    constexpr int SH = K == 4 ? kSh4 : 0;   // fixed point of the evaluation (eval4s)
    extern __shared__ __align__(16) unsigned char smem[];
    const int N = n_max > 0 ? n_max : 1;
    int32_t *s_dist = reinterpret_cast<int32_t *>(smem);
    int4 *s_cust = reinterpret_cast<int4 *>(smem + ((size_t(S) * S * 4 + 15) & ~size_t(15)));
    unsigned long long *s_min = reinterpret_cast<unsigned long long *>(s_cust + N);
    unsigned long long *s_kept = s_min + N;
    unsigned long long *s_queue = s_kept + kPBKeptCap;
    uint8_t *s_dead = reinterpret_cast<uint8_t *>(s_queue + kPBWarps * kPBQueue);
    __shared__ int s_bad, s_nk, s_cnt, s_item;
    __shared__ bool s_last;
    __shared__ unsigned long long s_nrec, s_eval, s_feas;
    __shared__ int s_pre[65];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.x / n_shards, shard = blockIdx.x - b * n_shards;
    const int rows_cap = n_max / K + 1;
    const size_t slot = size_t(b) * n_shards + shard;
    const int n = sizes[b];
    const long long off = offsets[b];
    if (tid == 0) { s_bad = (n < 0 || n > n_max || off < 0) ? 1 : 0; s_nrec = 0; s_eval = 0; s_feas = 0; s_item = 0; }
    __syncthreads();
    if (!s_bad) {
        for (int k = tid; k < S * S; k += blockDim.x) {
            const int d = dist[k];
            if (d < 0 || d > kDistLimit) s_bad = 1;
            s_dist[k] = d << SH;
        }
        for (int c = tid; c < n; c += blockDim.x) {
            const int32_t *r = demand + (off + c) * 5;
            const int f = r[1], t = r[2], w = r[3], l = r[4];
            if (f < 0 || f >= S || t < 0 || t >= S) { s_bad = 1; continue; }
            // clamping thr to +-2^25 changes no comparison (a ride is at most 7 * 2^22) and keeps the slacks from wrapping
            int thr = pool_detour_thr(dist[f * S + t], l);
            thr = thr > (1 << 25) ? (1 << 25) : (thr < -(1 << 25) ? -(1 << 25) : thr);
            s_cust[c] = scale_cust_rt(make_int4(f, t, thr, w), SH);
        }
    }
    __syncthreads();
    long long *ev_out = evaluated_out + slot, *fe_out = feasible_out + slot;
    if (s_bad) {
        // every CTA of the instance reads the same inputs and comes to the same decision; shard 0 writes the instance
        if (tid == 0) { *ev_out = 0; *fe_out = 0; kept_out[slot] = 0; }
        if (shard == 0) {
            int32_t *rows = plans_out + size_t(b) * rows_cap * TD_POOL_REC_W;
            for (int k = tid; k < rows_cap * TD_POOL_REC_W; k += blockDim.x) rows[k] = -1;
            if (tid == 0) { n_plans_out[b] = -1; needed_out[b] = 0; }
        }
        return;
    }

    // ---- enumeration (pool_n.c:226-229 shard rule, :153-177 pickups, :101-151 drop-offs) ----
    const int step = n / n_shards + 1, start = step * shard, stop = min(n, start + step);
    const int n_lead = start < n ? stop - start : 0;
    const int32_t *D = s_dist;
    const int4 *cust = s_cust;
    unsigned long long *recs = ws.recs + slot * size_t(rps);
    unsigned long long my_eval = 0, my_feas = 0;
    const unsigned lt_mask = (1u << lane) - 1;
    // warp-collective: materialise the keys of the lanes with has; the counter runs on past the slice (needed_out)
    auto emit = [&](bool has, unsigned long long key) {
        const unsigned ball = __ballot_sync(0xffffffffu, has);
        if (!ball) return;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&s_nrec, (unsigned long long)__popc(ball));
        base = __shfl_sync(0xffffffffu, base, 0);
        const unsigned long long pos = base + __popc(ball & lt_mask);
        if (has && pos < (unsigned long long)rps) recs[pos] = key;
    };
    auto next_item = [&]() {
        int it = 0;
        if (lane == 0) it = atomicAdd(&s_item, 1);
        return __shfl_sync(0xffffffffu, it, 0);
    };
    if (K == 2) {
        // item = leader, lanes over the second pickup
        for (int it = next_item(); it < n_lead; it = next_item()) {
            const int p0 = start + it;
            const int4 c0 = cust[p0];
            if (c0.w < 0) continue;                                    // pool_n.c:172 at level 0
            for (int b1 = 0; b1 < n; b1 += 32) {
                const int p1 = b1 + lane;
                bool valid = p1 < n && p1 != p0;
                if (valid) valid = (D[c0.x * S + cust[p1].x] >> SH) <= cust[p1].w;
                int nfeas = 0, best = INT_MAX;
                if (valid) {
                    const int p[4] = {p0, p1, 0, 0};
                    eval_tuple<K>(p, cust, D, S, nfeas, best);
                    my_eval += 2;
                    my_feas += nfeas;
                }
                emit(nfeas > 0, (unsigned long long)(best >> kPermBits) << 36 | tuple_rank(p0, p1, 0, 0));
            }
        }
    } else {
        unsigned long long *queue = s_queue + warp * kPBQueue;
        int q_head = 0, q_cnt = 0;                                     // warp-uniform
        auto eval_queue = [&](int take) {
            int nfeas = 0, best = INT_MAX;
            unsigned long long rank = 0;
            if (lane < take) {
                rank = queue[(q_head + lane) & (kPBQueue - 1)];
                int p[4];
                key_tuple(rank, p);
                eval_tuple<K>(p, cust, D, S, nfeas, best);
                my_feas += nfeas;
            }
            emit(nfeas > 0, (unsigned long long)(best >> kPermBits) << 36 | rank);
            q_head = (q_head + take) & (kPBQueue - 1);
            q_cnt -= take;
            __syncwarp();
        };
        // item = (leader, second pickup); lanes over the third pickup.  K = 3 evaluates in place, K = 4 walks the last
        // pickups of every valid third one over the lanes and queues the tuples, evaluated 32 at a time
        const int n_items = n_lead * n;
        for (int it = next_item(); it < n_items; it = next_item()) {
            const int p0 = start + it / n, p1 = it - (it / n) * n;
            const int4 c0 = cust[p0], c1 = cust[p1];
            if (c0.w < 0 || p1 == p0) continue;
            const int a01 = D[c0.x * S + c1.x];
            if ((a01 >> SH) > c1.w) continue;                          // pool_n.c:172
            for (int b2 = 0; b2 < n; b2 += 32) {
                const int p2 = b2 + lane;
                bool valid = p2 < n && p2 != p0 && p2 != p1;
                int w2 = 0;
                if (valid) {
                    w2 = a01 + D[c1.x * S + cust[p2].x];
                    valid = (w2 >> SH) <= cust[p2].w;
                }
                if (K == 3) {
                    int nfeas = 0, best = INT_MAX;
                    if (valid) {
                        const int p[4] = {p0, p1, p2, 0};
                        eval_tuple<K>(p, cust, D, S, nfeas, best);
                        my_eval += 6;
                        my_feas += nfeas;
                    }
                    emit(nfeas > 0, (unsigned long long)(best >> kPermBits) << 36 | tuple_rank(p0, p1, p2, 0));
                    continue;
                }
                unsigned m2 = __ballot_sync(0xffffffffu, valid);
                while (m2) {
                    const int l2 = __ffs(m2) - 1;
                    m2 &= m2 - 1;
                    const int q2 = b2 + l2, w2q = __shfl_sync(0xffffffffu, w2, l2), f2 = cust[q2].x;
                    const unsigned long long ent = tuple_rank(p0, p1, q2, 0);
                    for (int b3 = 0; b3 < n; b3 += 32) {
                        const int p3 = b3 + lane;
                        bool v3 = p3 < n && p3 != p0 && p3 != p1 && p3 != q2;
                        if (v3) v3 = ((w2q + D[f2 * S + cust[p3].x]) >> SH) <= cust[p3].w;
                        my_eval += v3 ? 24 : 0;
                        const unsigned ball = __ballot_sync(0xffffffffu, v3);
                        if (v3) queue[(q_head + q_cnt + __popc(ball & lt_mask)) & (kPBQueue - 1)] = ent | unsigned(p3);
                        q_cnt += __popc(ball);
                        __syncwarp();
                        if (q_cnt >= 32) eval_queue(32);
                    }
                }
            }
        }
        if (K == 4)
            while (q_cnt > 0) eval_queue(q_cnt < 32 ? q_cnt : 32);
    }
    atomicAdd(&s_eval, my_eval);
    atomicAdd(&s_feas, my_feas);
    __syncthreads();

    // ---- this shard's greedy (pool_n.c:187-207) ----
    const unsigned long long needed = s_nrec;
    const bool overflow = needed > (unsigned long long)rps;
    int nk = 0;
    if (!overflow) {
        auto cust_of = [](unsigned long long key, int c[4]) { key_tuple(key, c); };
        nk = dominance_rounds<K>(recs, int(needed), n, cust_of, s_min, s_dead, s_kept, &s_nk, &s_cnt);
        __syncthreads();
        sort_kept(s_kept, nk, recs);                                   // survivors at the start of the slice
    }
    if (tid == 0) {
        *ev_out = (long long)s_eval;
        *fe_out = (long long)s_feas;
        kept_out[slot] = overflow ? -1 : nk;
        PBMeta me;
        me.count = nk; me.overflow = overflow ? 1 : 0; me.needed = (long long)needed;
        ws.meta[slot] = me;
    }
    __threadfence();                                                   // survivors and meta before the ticket
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&ws.ticket[b], 1u) == unsigned(n_shards - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();

    // ---- the last CTA of the instance: merge in shard order (findpool.c:83-108) and write the rows ----
    int32_t *rows = plans_out + size_t(b) * rows_cap * TD_POOL_REC_W;
    const PBMeta *meta = ws.meta + size_t(b) * n_shards;
    if (tid == 0) {
        int run = 0, any_over = 0;
        long long need = 0;
        for (int s = 0; s < n_shards; ++s) {
            const int cnt = __ldcg(&meta[s].count), ov = __ldcg(&meta[s].overflow);
            const long long nd = __ldcg(&meta[s].needed);
            s_pre[s] = run;
            run += cnt;
            any_over |= ov;
            need = nd > need ? nd : need;
        }
        s_pre[n_shards] = run;
        s_bad = any_over;
        needed_out[b] = need;
    }
    __syncthreads();
    if (s_bad) {
        for (int k = tid; k < rows_cap * TD_POOL_REC_W; k += blockDim.x) rows[k] = -1;
        if (tid == 0) n_plans_out[b] = -2;
        return;
    }
    const int total = s_pre[n_shards];
    const unsigned long long *inst_recs = ws.recs + size_t(b) * n_shards * size_t(rps);
    // survivor key at concatenation position pos
    auto surv = [&](int pos) {
        int s = 0;
        while (s_pre[s + 1] <= pos) ++s;
        return __ldcg(inst_recs + size_t(s) * rps + (pos - s_pre[s]));
    };
    unsigned long long *mlive = ws.mlive + size_t(b) * n_shards * kPBKeptCap;
    for (int pos = tid; pos < total; pos += blockDim.x)
        mlive[pos] = (K == 4 ? (surv(pos) >> 36) << 32 : 0ull) | unsigned(pos);
    __syncthreads();
    auto cust_of_pos = [&](unsigned long long key, int c[4]) { key_tuple(surv(int(key & 0xffffffffu)), c); };
    const int m = dominance_rounds<K>(mlive, total, n, cust_of_pos, s_min, s_dead, s_kept, &s_nk, &s_cnt);
    __syncthreads();
    // rows in merge order: pool_n.c:123-134 layout, the best drop-off order recomputed
    for (int i = tid; i < m; i += blockDim.x) {
        const unsigned long long me = s_kept[i];
        int rank = 0;
        for (int q = 0; q < m; ++q) rank += s_kept[q] < me;
        const unsigned long long key = surv(int(me & 0xffffffffu));
        int p[4];
        key_tuple(key, p);
        int nfeas = 0, best = 0;
        eval_tuple<K>(p, cust, D, S, nfeas, best);
        int perm = best & 31, used = 0;
        int32_t *r = rows + size_t(rank) * TD_POOL_REC_W;
        for (int d = 0; d < K; ++d) {                                  // lexicographic permutation index -> drop order
            const int fact = (K - 1 - d) == 3 ? 6 : ((K - 1 - d) == 2 ? 2 : 1);   // (K - 1 - d)!
            int digit = perm / fact;
            perm -= digit * fact;
            int q = 0;
            while ((used >> q) & 1 || digit-- > 0) ++q;                 // the digit-th passenger not yet dropped
            used |= 1 << q;
            r[d] = p[d];
            r[K + d] = q == 0 ? p[0] : (q == 1 ? p[1] : (q == 2 ? p[2] : p[3]));
        }
        for (int j = 2 * K; j < 8; ++j) r[j] = 0;
        r[8] = int(key >> 36);
    }
    for (int k = m * TD_POOL_REC_W + tid; k < rows_cap * TD_POOL_REC_W; k += blockDim.x) rows[k] = -1;
    if (tid == 0) n_plans_out[b] = m;
}

static size_t pb_smem(int n_max, int S) {
    const size_t N = n_max > 0 ? size_t(n_max) : 1;
    return ((size_t(S) * S * 4 + 15) & ~size_t(15)) + N * 16 + N * 8 + size_t(kPBKeptCap) * 8 +
           size_t(kPBWarps) * kPBQueue * 8 + N;
}

constexpr int kNothingToLaunch = 1;
static int check_pool_batch(const int32_t *demand, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                            const int32_t *dist, int n_stands, int pool_size, int n_shards, const int32_t *plans_out,
                            const int32_t *n_plans_out, const int64_t *evaluated_out, const int64_t *feasible_out,
                            const int32_t *kept_out, const int64_t *needed_out, int64_t records_per_shard) {
    if (batch < 0 || n_max < 0 || n_max > TD_POOL_BATCH_MAX_N) return TD_ERR_INVALID;
    if (pool_size < 2 || pool_size > TD_POOL_MAX_IN_POOL || n_shards < 1 || n_shards > 64) return TD_ERR_INVALID;
    if (n_stands < 1 || n_stands > kPBMaxStands || records_per_shard < 0 || records_per_shard > INT_MAX) return TD_ERR_INVALID;
    if (int64_t(batch) * n_shards > INT_MAX) return TD_ERR_INVALID;
    if (batch == 0) return have_device() ? kNothingToLaunch : TD_ERR_NO_DEVICE;
    if (!demand || !sizes || !offsets || !dist || !plans_out || !n_plans_out || !evaluated_out || !feasible_out || !kept_out ||
        !needed_out)
        return TD_ERR_INVALID;
    return TD_OK;
}

}  // namespace td

extern "C" size_t td_pool_batch_workspace_bytes(int batch, int n_shards, int64_t records_per_shard) {
    if (batch < 0 || n_shards < 1 || n_shards > 64 || records_per_shard < 0 || records_per_shard > INT_MAX) return 0;
    return td::carve_pb(nullptr, batch, n_shards, records_per_shard).bytes;
}

extern "C" int td_pool_find_all_batch(const int32_t *demand, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                                      const int32_t *dist, int n_stands, int pool_size, int n_shards, int32_t *plans_out,
                                      int32_t *n_plans_out, int64_t *evaluated_out, int64_t *feasible_out, int32_t *kept_out,
                                      int64_t *needed_out, void *workspace, size_t workspace_bytes, int64_t records_per_shard,
                                      void *stream) {
    using namespace td;
    const int rc = check_pool_batch(demand, sizes, offsets, batch, n_max, dist, n_stands, pool_size, n_shards, plans_out,
                                    n_plans_out, evaluated_out, feasible_out, kept_out, needed_out, records_per_shard);
    if (rc != TD_OK) return rc == kNothingToLaunch ? TD_OK : rc;
    if (!workspace || workspace_bytes < td_pool_batch_workspace_bytes(batch, n_shards, records_per_shard)) return TD_ERR_WORKSPACE;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const PBWs ws = carve_pb(workspace, batch, n_shards, records_per_shard);
    TD_CUDA_TRY(cudaMemsetAsync(ws.ticket, 0, size_t(batch) * sizeof(unsigned int), st));
    const size_t smem = pb_smem(n_max, n_stands);
    const unsigned grid = unsigned(batch) * unsigned(n_shards);
    long long *ev = reinterpret_cast<long long *>(evaluated_out), *fe = reinterpret_cast<long long *>(feasible_out);
    long long *nd = reinterpret_cast<long long *>(needed_out);
#define TD_PB_LAUNCH(K)                                                                                                    \
    do {                                                                                                                   \
        TD_CUDA_TRY(cudaFuncSetAttribute(pool_batch_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));    \
        pool_batch_kernel<K><<<grid, kPBThreads, smem, st>>>(demand, sizes, offsets, n_max, dist, n_stands, n_shards,       \
                                                             plans_out, n_plans_out, ev, fe, kept_out, nd, ws,              \
                                                             (long long)records_per_shard);                                 \
    } while (0)
    if (pool_size == 2) TD_PB_LAUNCH(2);
    else if (pool_size == 3) TD_PB_LAUNCH(3);
    else TD_PB_LAUNCH(4);
#undef TD_PB_LAUNCH
    TD_LAUNCH_CHECK();
    return TD_OK;
}
