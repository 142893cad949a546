// td_pool.cu -- K4: the 2..4-passenger pool finder.
//
// Replaces one pool_n process of the reference (pool_n.c:209-238):
//   findPool        pool_n.c:153-177   ordered pickup tuples, cumulative-wait pruning
//   drop_customers  pool_n.c:101-151   all K! drop-off orders, per-passenger detour test
//   removeDuplicates pool_n.c:187-207  sort by cost (stable => ties by enumeration rank), greedy
//                                      scan keeping plans that share no customer with a kept one
//   shard rule      pool_n.c:226-229   leading customer in [step*t, min(n, step*t+step)), step = n/S + 1
// and findpool.c:83-108 (merge of the shard outputs) in td_pool_merge.
//
// Formal statement: SURVEY.md section 8(a).  Notation: customer c has from F, to T, max wait W,
// max loss L (percent); D = stand distance table; thr[c] = floor(D(F,T) * (1 + L/100.0)) in IEEE
// fp64 -- the reference's int-vs-double compare `ride > D*(1+L/100.0)` (pool_n.c:115-116) is
// exactly `ride > thr` for integer ride.
//
// Kernels
//   pool_prepare       one launch for the three independent input passes: per customer {F, T, thr, W} (pool_prep_cust),
//                      the stand-table check + its copy in the fixed point of the evaluation (pool_check_table), and the
//                      shortest-path closure D* of the table for the K = 4 pruning bounds (pool_closure: Floyd-Warshall,
//                      one CTA, cells in registers)
//   pool_build_lists   per stand s: customers ordered by slack(s,c) = W[c] - D(s,F[c]) descending
//                      (counting sort, 64 buckets) + cnt[s][w] = #{c : slack >= w}.  The wait rule
//                      "cumulative pickup distance w + D(s,F[c]) <= W[c]" turns into "c is in the
//                      first cnt[s][w] entries of list[s]": the next pickup level is a contiguous
//                      prefix, no search, no test.
//   (item offsets)     work items = (leader, position in list[F[leader]]) for K >= 3, leader for K = 2; computed by the
//                      CTA of pool_build_lists that finishes last
//   pool_enum<K>       one warp per item; outer pickup levels are warp-uniform loops, the LAST
//                      pickup level is spread over the 32 lanes; each lane evaluates all K! drop-off
//                      orders of its tuple in registers (fully unrolled, shared prefixes CSE'd).
//                      Stand distances and customer records are staged in shared memory.
//                      Every tuple materialises at most ONE record: its best feasible order under
//                      (cost, permutation index).  The other feasible orders of the same tuple
//                      cover the same customers with a larger key, so they can never survive the
//                      greedy scan; they are counted (stats.feasible) but not stored.
//   pool_select (coop) parallel greedy = rounds of "locally dominant" plans: a live plan whose key
//                      (cost, rank) is the minimum over all live plans at each of its customers is
//                      kept by the sequential scan regardless of anything else; keep all of them,
//                      kill their customers, compact, repeat.  Equal to sort + greedy scan because
//                      the key order is strict.  rank = (p0,p1,..,perm) lexicographic = the
//                      enumeration order of pool_n.c, i.e. the tie order of a stable sort by cost.
//                      Records are processed in ascending cost bands (the cheap plans kill most customers before the
//                      bulk of the list is looked at), the active list is fragmented over the CTAs, and a warp folds
//                      the keys of consecutive records that share a customer into ONE atomicMin (per-run minima).
//                      Record format: when every plan cost provably fits beside the customers packed with
//                      cb = ceil(log2 n) bits each (key64_fits, decided on the device from max W + max thr before the
//                      enumeration), a record IS its 8-byte single-level key (cost | p0 | p1 | p2 | p3 | perm); otherwise
//                      it is a 16-byte PoolRec and the keys come from rec_key1 / rec_hi.  Kept plans are PoolRec either way.
//   pool_emit         kept plans in key order -> 9-int records of pool_n.c:123-134
//   pool_merge         findpool.c:83-108: the shard outputs are sorted runs, so the global order is a rank by binary
//                      searches (bitonic sort for rows in any other order), then the same dominance rounds in shared memory
//
// Roofline: the enumeration is INT32-issue + shared-memory-lookup bound; compulsory HBM traffic is
// ~0.4 B per plan.  SURVEY.md section 8(d) defines the logical bytes used for the HBM-fraction
// figure: 80 B per evaluated plan (4 customers x the 5-int32 demand record) + 36 B per feasible plan.
#include "td_pool_common.cuh"
#include <string.h>
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace td {

constexpr int kTbl = 64;          // budget table entries per stand
constexpr int kEnumThreads = 256;
constexpr int kEnumThreadsWide = 1024;  // one CTA per SM (big staged tables): 32 warps instead of 8
constexpr int kIoffSmem = 2048;          // leaders whose item offsets are staged in shared memory
constexpr size_t kEnumIoffBytes = (size_t(kIoffSmem) + 4) * 4;
constexpr size_t kEnumWarpBytes = 256 * 4 + 3 * 32 * 16 + 64 * 8;   // histogram + staging A, B, C + tuple queue
constexpr int kChunk = 128;       // records reserved per atomic
constexpr int kSelThreads = 512;
constexpr int kCustBits = 14;     // TD_POOL_MAX_CUSTOMERS = 16384

struct PoolRec {                  // 16 bytes
    unsigned long long rank;      // p0 | p1 | p2 | p3 | perm  (unused pickup slots are 0)
    int32_t cost;                 // < 0: hole (unused slot of a reserved chunk)
    int32_t pad;
};

constexpr int kMaxSlots = 64;     // logical shards handled by one call
constexpr int kBuckets = 256;     // cost histogram resolution (last bucket: cost >= 255)
constexpr int kMaxBands = 8;      // cost bands of the selection; band sizes grow 4x from kBand0
// Measured on config 3 (B200, 8 shards / 1 shard per call, select in us): 4096 x4: 917 / 294, 32768 x3: 720 / 259,
// 65536 x4: 706 / 252, 131072 x4: 791 / 301, 262144 x4: 805 / 311 -- a first band of 65 536 records keeps the number of
// grid-wide phases down without letting the last band (most of the records, few of them live) grow
constexpr unsigned kBand0 = 65536;

struct PoolCtrl {
    // ---- persistent over the passes of one call ----
    unsigned long long tstamp[32];  // %globaltimer at the phase boundaries of pool_select (diagnostics)
    unsigned long long evaluated[kMaxSlots], feasible[kMaxSlots];  // per logical shard of this call
    unsigned int n_kept[kMaxSlots];
    unsigned int total_rounds;
    unsigned int n_items;         // work items of the enumeration (set once by pool_build_lists)
    unsigned int closure_ok;      // pool_closure: the shortest-path closure of the stand table is usable as a lower bound
    unsigned int bad_input;       // a stand index outside the table, or (K = 4) a stand distance above kDistLimit (the x32
                                  // fixed-point evaluation would overflow): the call reports TD_ERR_INVALID / count -1
    unsigned int lists_done;      // CTAs of pool_build_lists that have finished (the last one computes the item offsets)
    unsigned int pass_begin_marker;  // ---- everything below is zeroed before every enumeration pass ----
    unsigned int n_records;       // slots reserved in the record list
    unsigned int item_counter;
    unsigned int overflow;
    unsigned int rounds;
    int band_hi[kMaxSlots][kMaxBands];           // exclusive cost bound of band b for each logical shard
    unsigned int band_cnt[kMaxSlots][kMaxBands]; // records of shard s in band b (from the histogram)
    unsigned int band_off[kMaxBands + 1];        // start of band b in the band-partitioned record list
    unsigned int band_cur[kMaxBands];            // write cursors of the partition pass
    unsigned int act_cnt[kMaxBands][2];          // live in-band records, ping-pong between rounds
    unsigned long long hist[kMaxSlots][kBuckets];   // plans per min(cost, kBuckets-1), filled by pool_enum (64-bit: the
                                                    // counts include plans beyond the materialised cost window)
    // ---- set once per call by pool_prepare / pool_build_lists, outside the per-pass reset (see key64_fits) ----
    int max_wait, max_thr;        // max(W, 0) and max(thr, 0) over the customers
    unsigned int key64;           // 1: the record list holds 8-byte keys, 0 (a zeroed block, td_pool_pairs): PoolRec
};

// Bits per customer index in the single-level key (selection) and in the 8-byte records: cb = ceil(log2 n), at least 1.
__host__ __device__ __forceinline__ int key_cb(int n) {
    int cb = 1;
    while ((1 << cb) < n) ++cb;
    return cb;
}

// The 8-byte record format: (cost, p0, p1, p2, p3, perm) packed as cost | cb bits x 4 | kPermBits, i.e. the single-level key
// of the selection itself.  It is exact when every materialised cost is below 2^(64 - 4 cb - kPermBits), and that follows
// from the input alone.  A plan's cost is its pickup legs plus its drop-off legs.  The pickup legs are at most W of its last
// pickup: the wait rule admits a pickup only while the cumulative pickup distance is within its W.  The drop-off legs are at
// most the ride of the passenger dropped last, which the detour rule bounds by its thr.  So every feasible plan costs at
// most max(W, 0) + max(thr, 0) over the customers, and costs are never negative (pool_check_table refuses negative table
// entries for every K), so the cost field needs no sign.  n <= 16384 leaves at least 3 cost bits.
__device__ __forceinline__ unsigned key64_fits(int n, int max_wait, int max_thr) {
    const int cost_bits = 64 - 4 * key_cb(n) - kPermBits;
    if (cost_bits < 1) return 0u;
    if (cost_bits >= 33) return 1u;
    return (unsigned long long)max_wait + (unsigned long long)max_thr < (1ull << cost_bits) ? 1u : 0u;
}
constexpr unsigned long long kKeyHole = ~0ull;   // no valid key: perm <= 23 never fills the permutation field

__device__ __forceinline__ unsigned long long make_rank(int p0, int p1, int p2, int p3, int perm) {
    return ((((((unsigned long long)p0 << kCustBits) | (unsigned)p1) << kCustBits | (unsigned)p2) << kCustBits |
             (unsigned)p3) << kPermBits) | (unsigned)perm;
}
__device__ __forceinline__ void split_rank(unsigned long long r, int p[4], int &perm) {
    perm = int(r & ((1u << kPermBits) - 1)); r >>= kPermBits;
    const unsigned m = (1u << kCustBits) - 1;
    p[3] = int(r & m); r >>= kCustBits;
    p[2] = int(r & m); r >>= kCustBits;
    p[1] = int(r & m); r >>= kCustBits;
    p[0] = int(r & m);
}
// Single-level key: (cost, rank) in ONE 64-bit word, rank repacked with cb = key_cb(n) bits per customer.  Exact when
// cost < 2^(64 - 4 cb - kPermBits).  Order-preserving: lexicographic (cost, p0, p1, p2, p3, perm).
__device__ __forceinline__ unsigned long long pack_key1(int cost, unsigned long long rank, int cb) {
    const unsigned m = (1u << kCustBits) - 1;
    const unsigned perm = unsigned(rank) & ((1u << kPermBits) - 1); rank >>= kPermBits;
    const unsigned p3 = unsigned(rank) & m; rank >>= kCustBits;
    const unsigned p2 = unsigned(rank) & m; rank >>= kCustBits;
    const unsigned p1 = unsigned(rank) & m; rank >>= kCustBits;
    const unsigned p0 = unsigned(rank) & m;
    unsigned long long k = (unsigned long long)(unsigned)cost;
    k = (k << cb) | p0; k = (k << cb) | p1; k = (k << cb) | p2; k = (k << cb) | p3;
    return (k << kPermBits) | perm;
}

// ---- prep ----------------------------------------------------------------------------------------
__device__ __forceinline__ void pool_prep_cust(int c, const int32_t *__restrict__ demand, int n, const int32_t *__restrict__ dist,
                                               int S, int4 *cust, int4 *cust_s, int sh, PoolCtrl *ctrl) {
    int w_pos = 0, thr_pos = 0;
    if (c < n) {
        int f = demand[c * 5 + 1], t = demand[c * 5 + 2];
        const int w = demand[c * 5 + 3], l = demand[c * 5 + 4];
        if (f < 0 || f >= S || t < 0 || t >= S) {   // pool_n.c:106-134 would index cost[][] out of bounds: refuse the input
            ctrl->bad_input = 1;
            f = 0; t = 0;
        }
        const int d = dist[size_t(f) * S + t];
        const int thr = pool_detour_thr(d, l);
        cust[c] = make_int4(f, t, thr, w);
        cust_s[c] = scale_cust_rt(make_int4(f, t, thr, w), sh);   // the enumeration's staged copy (fixed point of its evaluation)
        w_pos = w > 0 ? w : 0;
        thr_pos = thr > 0 ? thr : 0;
    }
    // the cost bound of the 8-byte records (key64_fits); the whole CTA prepares customers, so every lane is here
    w_pos = __reduce_max_sync(0xffffffffu, w_pos);
    thr_pos = __reduce_max_sync(0xffffffffu, thr_pos);
    if ((threadIdx.x & 31) == 0) {
        if (w_pos) atomicMax(&ctrl->max_wait, w_pos);
        if (thr_pos) atomicMax(&ctrl->max_thr, thr_pos);
    }
}

// one CTA per stand: counting sort of the customers reachable from this stand by slack, descending
__global__ void __launch_bounds__(256)
pool_build_lists_kernel(const int4 *__restrict__ cust, int n, const int32_t *__restrict__ dist, int S,
                        int32_t *list, int32_t *slack_out, int32_t *cnt, int start, int stop, int pool_size,
                        unsigned int *item_off, PoolCtrl *ctrl) {
    __shared__ int hist[kTbl];
    __shared__ int offs[kTbl];
    const int s = blockIdx.x;
    for (int b = threadIdx.x; b < kTbl; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        const int4 r = cust[c];
        const int sl = r.w - dist[size_t(s) * S + r.x];
        if (sl >= 0) atomicAdd(&hist[sl < kTbl ? sl : kTbl - 1], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int b = kTbl - 1; b >= 0; --b) {  // descending slack: bucket b starts after all larger buckets
            offs[b] = run;
            run += hist[b];
            cnt[size_t(s) * kTbl + b] = run;   // #{c : slack >= b}
        }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
        const int4 r = cust[c];
        const int sl = r.w - dist[size_t(s) * S + r.x];
        if (sl >= 0) {
            const int pos = atomicAdd(&offs[sl < kTbl ? sl : kTbl - 1], 1);
            list[size_t(s) * n + pos] = c;
            slack_out[size_t(s) * n + pos] = sl;
        }
    }
    // ---- items per leader (exclusive prefix; K >= 3: one item per (leader, first-level candidate)), by the CTA that
    // finishes last: it needs cnt[] of every stand, and a kernel of its own would cost a launch for a few microseconds
    __shared__ bool s_last;
    __shared__ unsigned s_part[256];
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();                                         // this CTA's cnt[] before the ticket
        s_last = atomicAdd(&ctrl->lists_done, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int nl = stop - start;
    const int chunk = (nl + 255) / 256;
    const int lo = min(int(threadIdx.x) * chunk, nl), hi = min(lo + chunk, nl);
    auto items_of = [&](int p0) -> unsigned {
        const int4 r = cust[p0];
        if (r.w < 0) return 0u;                                  // pool_n.c:172 at level 0
        return pool_size >= 3 ? unsigned(__ldcg(cnt + size_t(r.x) * kTbl + 0)) : 1u;   // written by other CTAs: L2
    };
    unsigned sum = 0;
    for (int t = lo; t < hi; ++t) sum += items_of(start + t);
    s_part[threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.x < 32) {   // exclusive scan of the 256 partial sums: 8 per lane, warp scan of the lane sums
        unsigned mine = 0;
        for (int k = 0; k < 8; ++k) mine += s_part[threadIdx.x * 8 + k];
        unsigned incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if (threadIdx.x >= o) incl += v; }
        unsigned acc = incl - mine;
        for (int k = 0; k < 8; ++k) { const unsigned v = s_part[threadIdx.x * 8 + k]; s_part[threadIdx.x * 8 + k] = acc; acc += v; }
        if (threadIdx.x == 31) {
            item_off[nl] = incl; ctrl->n_items = incl;
            ctrl->key64 = key64_fits(n, ctrl->max_wait, ctrl->max_thr);   // pool_prepare has ended: the maxima are final
        }
    }
    __syncthreads();
    unsigned run = s_part[threadIdx.x];
    for (int t = lo; t < hi; ++t) { item_off[t] = run; run += items_of(start + t); }
}


// Stand-table check for every pool size: a negative entry (plan costs could go negative -- a negative cost marks a hole
// in the record list) or an entry above kDistLimit is refused with TD_ERR_INVALID, never clamped.
__device__ __forceinline__ void pool_check_table(int block, int blocks, const int32_t *__restrict__ dist, long long cells,
                                                 PoolCtrl *ctrl, int32_t *dist_s, int sh) {
    int bad = 0;
    for (long long i = block * (long long)blockDim.x + threadIdx.x; i < cells; i += (long long)blocks * blockDim.x) {
        const int v = dist[i];
        bad |= (v < 0) | (v > kDistLimit);
        if (dist_s) dist_s[i] = v << sh;       // the copy the enumeration stages by bulk copy (small tables only)
    }
    if (__syncthreads_or(bad) && threadIdx.x == 0) ctrl->bad_input = 1;
}

// Shortest-path closure D* of the stand table (Floyd-Warshall in shared memory, one CTA, S <= kPfMaxStands).
// Every walk a -> ... -> b over the table is at least D*(a,b) long when no entry is negative, so
//   ride(j) >= (pickup legs from j to the current last pickup) + D*(F_last, T_j)
// at every pickup level: a pickup prefix whose bound already exceeds thr_j for one of its passengers cannot become
// feasible whatever is picked up later and whatever the drop-off order is (pool_n.c:105-120 rejects every one of its
// leaves, one at a time).  pool_enum<4> uses the bound to skip those leaves; they are still COUNTED (pool_n.c:103).
// On metric tables (|i-j|, pool_n.c:179-185) D* == D.  A table with a negative entry switches the bound off.
constexpr int kPfMaxStands = 128;
template <int T>
__device__ __forceinline__ void closure_steps(int S, int32_t *s_d, int32_t *s_line) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    constexpr int kBig = 1 << 28;
    int d[T][T];
#pragma unroll
    for (int a = 0; a < T; ++a)
#pragma unroll
        for (int b = 0; b < T; ++b) {
            const int r = ty + 16 * a, c = tx + 16 * b;
            d[a][b] = (r < S && c < S) ? s_d[r * S + c] : kBig;
        }
    for (int k = 0; k < S; ++k) {
        int32_t *row = s_line + (k & 1) * 2 * kPfMaxStands, *col = row + kPfMaxStands;
        const int ka = k >> 4, kt = k & 15;
#pragma unroll
        for (int a = 0; a < T; ++a)
#pragma unroll
            for (int b = 0; b < T; ++b) {
                if (a == ka && ty == kt && tx + 16 * b < S) row[tx + 16 * b] = d[a][b];
                if (b == ka && tx == kt && ty + 16 * a < S) col[ty + 16 * a] = d[a][b];
            }
        __syncthreads();
        int rk[T], kc[T];
#pragma unroll
        for (int a = 0; a < T; ++a) { rk[a] = ty + 16 * a < S ? col[ty + 16 * a] : kBig; kc[a] = tx + 16 * a < S ? row[tx + 16 * a] : kBig; }
#pragma unroll
        for (int a = 0; a < T; ++a)
#pragma unroll
            for (int b = 0; b < T; ++b) d[a][b] = min(d[a][b], rk[a] + kc[b]);
    }
#pragma unroll
    for (int a = 0; a < T; ++a)
#pragma unroll
        for (int b = 0; b < T; ++b) {
            const int r = ty + 16 * a, c = tx + 16 * b;
            if (r < S && c < S) s_d[r * S + c] = d[a][b];
        }
}

__device__ __forceinline__ void pool_closure(const int32_t *__restrict__ dist, int S, int32_t *__restrict__ dclose, int sh, PoolCtrl *ctrl) {
    extern __shared__ int32_t s_d[];
    __shared__ int32_t s_line[2][2][kPfMaxStands];
    const int cells = S * S;
    int neg = 0;
    for (int i = threadIdx.x; i < cells; i += blockDim.x) {
        int v = dist[i];
        neg |= v < 0;
        v = v > (1 << 28) ? (1 << 28) : v;             // sums of two entries stay below 2^30
        if (i / S == i % S) v = 0;                     // the empty walk
        s_d[i] = v;
    }
    neg = __syncthreads_or(neg);
    // 16 x 16 thread tile over the table, every thread keeps its T x T cells in registers.  Row k and column k do not
    // change in step k (d(k,k) = 0, entries >= 0), so their owners publish them after step k - 1 into a double-buffered
    // line pair: one block barrier and 2T shared-memory loads per step instead of two loads and a store per cell.
    if (S <= 64) closure_steps<4>(S, s_d, s_line[0][0]);
    else closure_steps<8>(S, s_d, s_line[0][0]);
    __syncthreads();
    for (int i = threadIdx.x; i < cells; i += blockDim.x) dclose[i] = (s_d[i] > kDistLimit ? kDistLimit : s_d[i]) << sh;   // D* <= D <= limit on accepted tables
    if (threadIdx.x == 0) ctrl->closure_ok = neg ? 0u : 1u;
}

// The three independent input passes of a call in ONE launch (a launch costs more than any of them): CTA 0 computes the
// closure (the longest, so it starts first), the next check_blocks CTAs check / scale the stand table, the rest prepare the
// customer records.
__global__ void __launch_bounds__(256)
pool_prepare_kernel(const int32_t *__restrict__ demand, int n, const int32_t *__restrict__ dist, int S, int4 *cust, int4 *cust_s,
                    int sh, PoolCtrl *ctrl, int32_t *dist_s, int32_t *dclose, int closure_blocks, int check_blocks) {
    const int b = blockIdx.x;
    if (b < closure_blocks) pool_closure(dist, S, dclose, sh, ctrl);
    else if (b < closure_blocks + check_blocks) pool_check_table(b - closure_blocks, check_blocks, dist, (long long)S * S, ctrl, dist_s, sh);
    else pool_prep_cust((b - closure_blocks - check_blocks) * blockDim.x + threadIdx.x, demand, n, dist, S, cust, cust_s, sh, ctrl);
}

// ---- enumeration ---------------------------------------------------------------------------------
struct EnumArgs {
    // cust_s, dist_s, dclose: copies in the fixed point of the evaluation (staged by bulk copy)
    const int4 *cust; const int4 *cust_s; const int32_t *dist; const int32_t *dist_s; const int32_t *dclose; const int32_t *list; const int32_t *slack; const int32_t *cnt;
    const unsigned int *item_off; PoolRec *recs; PoolCtrl *ctrl;   // recs: PoolRec or, when ctrl->key64, 8-byte keys
    int n, S, start, stop; unsigned int cap;                       // cap: records of either format
    int cb;                       // key_cb(n)
    int step, shard_begin;        // leader p0 belongs to call slot p0 / step - shard_begin
    // multi-pass support (large inputs): only plans with cost in [cost_lo, cost_hi) are materialised, customers
    // whose alive flag is 0 (taken by an earlier cost window) are pruned at every pickup level
    int cost_lo, cost_hi;
    const uint8_t *alive;         // [shard_count x n] or NULL (first pass: everybody is free)
    int count_stats;              // accumulate evaluated / feasible (first pass only)
    int item_stride;              // > 1: sampling pass -- every item_stride-th item, histogram only
    unsigned int ioff_bytes;      // shared memory reserved for the staged item offsets (multiple of 16)
};

template <bool kDistSmem, int SH>
struct DistView {   // staged copies are pre-scaled by 2^SH; the global table is scaled at the load
    const int32_t *p; int S;
    __device__ __forceinline__ int operator()(int a, int b) const {
        return kDistSmem ? p[a * S + b] : (__ldg(p + size_t(a) * S + b) << SH);
    }
};

// customer record {from, to, thr, wait} with the detour threshold in the fixed point of the evaluation:
// (clamped thr) * 2^SH + (2^SH - 1).  The clamp keeps every comparison exact because no ride exceeds 7 * kDistLimit.
template <int SH>
__device__ __forceinline__ int4 scale_cust(int4 c) {
    if (SH > 0) {
        const int lim = 1 << 25;
        const int z = c.z > lim ? lim : (c.z < -lim ? -lim : c.z);
        c.z = (z << SH) | ((1 << SH) - 1);
    }
    return c;
}
template <bool kCustSmem, int SH>
struct CustView {
    const int4 *p;
    __device__ __forceinline__ int4 operator[](int i) const { return kCustSmem ? p[i] : scale_cust<SH>(p[i]); }
};

// candidates of the next pickup level from stand s with cumulative wait w: prefix length of list[s]
__device__ __forceinline__ int cand_count(const int32_t *cnt, int s, int w) {
    return cnt[s * kTbl + (w < 0 ? 0 : (w < kTbl ? w : kTbl - 1))];
}

struct WarpOut {  // per-warp slice of the record list
    unsigned base, used;
    bool dead;    // the list overflowed: this warp stops materialising (counters and histogram stay exact)
};

// The record format (key64_fits), set by pool_build_lists before the enumeration and constant during it: loaded where a
// record is written (read-only path, an L1 hit) rather than kept in a register across the enumeration loops.
__device__ __forceinline__ bool rec_key64(const EnumArgs &a) { return __ldg(&a.ctrl->key64) != 0u; }
__device__ __forceinline__ void mark_hole(const EnumArgs &a, bool k64, unsigned pos) {
    if (k64) reinterpret_cast<unsigned long long *>(a.recs)[pos] = kKeyHole;
    else a.recs[pos].cost = -1;
}

__device__ __forceinline__ void emit_records(const EnumArgs &a, WarpOut &wo, bool has, unsigned long long rank, int cost,
                                             int lane, unsigned *whist) {
    has = has && cost >= a.cost_lo;                 // earlier windows are done
    if (has) atomicAdd(&whist[cost < 0 ? 0 : (cost < kBuckets ? cost : kBuckets - 1)], 1u);
    has = has && cost < a.cost_hi && a.item_stride == 1;
    const unsigned ball = __ballot_sync(0xffffffffu, has);
    if (ball == 0 || wo.dead) return;
    const unsigned need = __popc(ball);
    if (wo.used + need > kChunk) {
        // abandon the rest of the current chunk (mark holes) and reserve a new one
        if (wo.base != 0xffffffffu)
            for (unsigned t = wo.used + lane; t < kChunk; t += 32) mark_hole(a, rec_key64(a), wo.base + t);
        unsigned nb = 0xffffffffu;
        // once the list has overflowed nobody reserves any more (the counter must not run away and wrap)
        if (lane == 0 && *reinterpret_cast<volatile unsigned *>(&a.ctrl->overflow) == 0)
            nb = atomicAdd(&a.ctrl->n_records, unsigned(kChunk));
        nb = __shfl_sync(0xffffffffu, nb, 0);
        if ((unsigned long long)nb + kChunk > (unsigned long long)a.cap) {
            if (lane == 0) a.ctrl->overflow = 1;
            wo.base = 0xffffffffu; wo.used = kChunk; wo.dead = true;
            return;
        }
        wo.base = nb; wo.used = 0;
    }
    if (wo.base == 0xffffffffu) return;
    if (has) {
        const unsigned pos = wo.base + wo.used + __popc(ball & ((1u << lane) - 1));
        if (rec_key64(a)) {
            reinterpret_cast<unsigned long long *>(a.recs)[pos] = pack_key1(cost, rank, a.cb);
        } else {
            PoolRec r; r.rank = rank; r.cost = cost; r.pad = 0;
            *reinterpret_cast<int4 *>(a.recs + pos) = *reinterpret_cast<int4 *>(&r);
        }
    }
    wo.used += need;
}

// kPF (K = 4 with the stand table in shared memory): the closure D* is staged next to the table and the lower bound of
// pool_closure prunes pickup prefixes at the third and at the last pickup level.
// kThr: threads per CTA.  256 when several CTAs fit an SM; when the staged tables leave room for ONE CTA only (5000 customers:
// 80 KB of customer records), a 768-thread CTA keeps 24 warps per SM busy instead of 8 (ncu r02n: 11 % warps active, 40 % issue).
template <int K, bool kDistSmem, bool kCustSmem, bool kPF, int kThr>
__global__ void __launch_bounds__(kThr, kThr == 256 ? 4 : 1)   // 64 registers: four 256-thread CTAs (32 warps) per SM
pool_enum_kernel(EnumArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const size_t dist_b = (size_t(a.S) * a.S * 4 + 15) & ~size_t(15);
    int32_t *s_dist = reinterpret_cast<int32_t *>(smem_raw);
    int32_t *s_dc = reinterpret_cast<int32_t *>(smem_raw + (kDistSmem ? dist_b : 0));
    int4 *s_cust = reinterpret_cast<int4 *>(smem_raw + (kDistSmem ? dist_b : 0) + (kPF ? dist_b : 0));
    constexpr int SH = (K == 4) ? kSh4 : 0;   // fixed-point shift of the K = 4 evaluation (eval4s)
    if (a.ctrl->bad_input) return;   // refused input (pool_prep_cust / pool_check_table): uniform, set before this launch
    // The tables are staged by the TMA engine: the prep kernels left copies in the fixed point of the evaluation, one
    // elected thread arms an mbarrier with the byte count and issues one 1-D bulk copy per table (cp.async.bulk,
    // global -> shared, completion counted on the barrier); every thread then waits on the barrier's phase.
    if (kDistSmem || kCustSmem) {
        __shared__ __align__(8) unsigned long long s_mbar;
        const unsigned bar = static_cast<unsigned>(__cvta_generic_to_shared(&s_mbar));
        const unsigned cust_bytes = (unsigned(a.n) * 16u + 15u) & ~15u;
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned total = (kDistSmem ? unsigned(dist_b) : 0u) + (kPF ? unsigned(dist_b) : 0u) + (kCustSmem ? cust_bytes : 0u);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
            auto bulk = [&](void *dst, const void *src, unsigned bytes) {
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(dst))), "l"(src), "r"(bytes), "r"(bar) : "memory");
            };
            if (kDistSmem) bulk(s_dist, a.dist_s, unsigned(dist_b));
            if (kPF) bulk(s_dc, a.dclose, unsigned(dist_b));
            if (kCustSmem) bulk(s_cust, a.cust_s, cust_bytes);
        }
        unsigned done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(bar) : "memory");
    }
    // everything else in shared memory is carved from the dynamic allocation too (a 768-thread CTA needs 68 KB of it, the
    // static limit is 48 KB): item offsets per leader (searched once per work item), then per warp {cost histogram, batch
    // staging A / B, tuple queue}
    unsigned char *sm_rest = smem_raw + (kDistSmem ? dist_b : 0) + (kPF ? dist_b : 0) + (kCustSmem ? ((size_t(a.n) * 16 + 15) & ~size_t(15)) : 0);
    unsigned *s_ioff = reinterpret_cast<unsigned *>(sm_rest);               // [kIoffSmem + 1]
    unsigned char *sm_warp = sm_rest + a.ioff_bytes + size_t(threadIdx.x >> 5) * kEnumWarpBytes;
    const bool ioff_smem = (a.stop - a.start) <= kIoffSmem;
    if (ioff_smem)
        for (int i = threadIdx.x; i <= a.stop - a.start; i += kThr) s_ioff[i] = a.item_off[i];
    const unsigned *ioff = ioff_smem ? s_ioff : a.item_off;
    __syncthreads();
    const DistView<kDistSmem, SH> D{kDistSmem ? s_dist : a.dist, a.S};
    const DistView<true, SH> Dc{s_dc, a.S};            // only used when kPF
    const CustView<kCustSmem, SH> cust{kCustSmem ? s_cust : a.cust};
    const bool pf = kPF && a.ctrl->closure_ok != 0;
    const int lane = threadIdx.x & 31;
    const unsigned lt_mask = (1u << lane) - 1;
    const int n = a.n;
    const unsigned n_items = a.ctrl->n_items;
    const int n_lead = a.stop - a.start;
    unsigned long long my_eval = 0, my_feas = 0;
    int cur_slot = -1;
    WarpOut wo{0xffffffffu, unsigned(kChunk), false};
    unsigned *whist = reinterpret_cast<unsigned *>(sm_warp);            // [kBuckets] per-warp cost histogram of the warp's current shard
    // K = 4: per-warp staging of the current batch of third pickups {p2, F2, wait so far, slack of p0} / {slack of p1,
    // slack of p2, T2, end of its last-pickup range}, and the queue of pickup tuples that passed the bound
    int4 *stA = reinterpret_cast<int4 *>(sm_warp + kBuckets * 4);          // [32]
    int4 *stB = stA + 32;                                                   // [32]
    int4 *stC = stB + 32;                                                   // [32] closure distances between the drop-off stands
    unsigned long long *queue = reinterpret_cast<unsigned long long *>(stC + 32);   // [64]
    for (int b = lane; b < kBuckets; b += 32) whist[b] = 0;
    __syncwarp();
    auto flush_counts = [&]() {
        __syncwarp();
        if (cur_slot >= 0)
            for (int b = lane; b < kBuckets; b += 32) {
                const unsigned v = whist[b];
                if (v) { atomicAdd(&a.ctrl->hist[cur_slot][b], (unsigned long long)v); whist[b] = 0; }
            }
        __syncwarp();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            my_eval += __shfl_xor_sync(0xffffffffu, my_eval, o);
            my_feas += __shfl_xor_sync(0xffffffffu, my_feas, o);
        }
        if (lane == 0 && cur_slot >= 0 && a.count_stats) {
            if (my_eval) atomicAdd(&a.ctrl->evaluated[cur_slot], my_eval);
            if (my_feas) atomicAdd(&a.ctrl->feasible[cur_slot], my_feas);
        }
        my_eval = 0; my_feas = 0;
    };

    // ---- K = 4: queue of surviving pickup tuples; a full batch of 32 is evaluated at a time ----------------------
    int q_head = 0, q_cnt = 0;                        // warp-uniform ring state (64 entries, q_cnt < 32 between pushes)
    constexpr unsigned kCM = (1u << kCustBits) - 1;
    // all 24 drop-off orders of up to 32 queued tuples, one per lane; every tuple materialises its best feasible order
    auto eval_queue = [&](int take) {
        int nfeas = 0, best = INT_MAX;
        unsigned long long rank = 0;
        if (lane < take) {
            const unsigned long long ent = queue[(q_head + lane) & 63];
            const int q3 = int(unsigned(ent) & kCM), q2 = int(unsigned(ent >> kCustBits) & kCM);
            const int q1 = int(unsigned(ent >> (2 * kCustBits)) & kCM), q0 = int(unsigned(ent >> (3 * kCustBits)) & kCM);
            const int4 c0 = cust[q0], c1 = cust[q1], c2 = cust[q2], c3 = cust[q3];
            const int a01 = D(c0.x, c1.x), a12 = D(c1.x, c2.x), a23 = D(c2.x, c3.x);
            int e[4], t[4][4], sl[4];
            e[0] = D(c3.x, c0.y); e[1] = D(c3.x, c1.y); e[2] = D(c3.x, c2.y); e[3] = D(c3.x, c3.y);
            t[0][0] = t[1][1] = t[2][2] = t[3][3] = 0;
            t[0][1] = D(c0.y, c1.y); t[1][0] = D(c1.y, c0.y);
            t[0][2] = D(c0.y, c2.y); t[2][0] = D(c2.y, c0.y);
            t[1][2] = D(c1.y, c2.y); t[2][1] = D(c2.y, c1.y);
            t[0][3] = D(c0.y, c3.y); t[3][0] = D(c3.y, c0.y);
            t[1][3] = D(c1.y, c3.y); t[3][1] = D(c3.y, c1.y);
            t[2][3] = D(c2.y, c3.y); t[3][2] = D(c3.y, c2.y);
            sl[3] = c3.z; sl[2] = c2.z - a23; sl[1] = c1.z - a12 - a23; sl[0] = c0.z - a01 - a12 - a23;
            eval4s(e, t, sl, nfeas, best);
            my_feas += nfeas;
            if (nfeas > 0) best += a01 + a12 + a23;   // pickup legs (multiples of 32): best = 32 * plan cost + permutation index
            rank = make_rank(q0, q1, q2, q3, best & 31);
        }
        emit_records(a, wo, nfeas > 0, rank, best >> kPermBits, lane, whist);
        q_head = (q_head + take) & 63;
        q_cnt -= take;
        __syncwarp();
    };

    for (;;) {
        // (requesting the next item ahead of time to hide the atomic's latency was measured and dropped: a warp then
        // sits on an item while others idle at the tail -- 8 shards 0.60 -> 0.62 ms, one shard 0.13 -> 0.17 ms)
        unsigned item = 0;
        if (lane == 0) item = atomicAdd(&a.ctrl->item_counter, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        // K = 4 walks the (leader, second pickup) pairs twice: first everything but the first batch of 32 third pickups,
        // then the first batches alone.  The work is the same, but the units handed out last are at most a third of a
        // big pair, which cuts the tail of the launch (a big pair alone runs ~0.25 ms of a 1.7 ms kernel).
        const unsigned n_units = (K == 4) ? 2u * n_items : n_items;
        const bool done = item >= (n_units + unsigned(a.item_stride) - 1) / unsigned(a.item_stride);
        item *= unsigned(a.item_stride);
        const bool first_batch_only = (K == 4) && item >= n_items;
        if (first_batch_only) item -= n_items;
        int lo = 0;
        if (!done) {   // leader = last index with item_off[idx] <= item
            int hi = n_lead;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (ioff[mid] <= item) lo = mid; else hi = mid;
            }
        }
        const int p0 = a.start + lo;
        const int slot = done ? -2 : p0 / a.step - a.shard_begin;
        if (slot != cur_slot) {   // the per-warp counters, histogram and tuple queue belong to one logical shard at a time
            if (K == 4)
                while (q_cnt > 0) eval_queue(q_cnt < 32 ? q_cnt : 32);
            flush_counts();
            cur_slot = slot;
        }
        if (done) break;
        const int4 c0 = cust[p0];
        const uint8_t *al = a.alive ? a.alive + size_t(slot) * n : nullptr;
        if (al && !al[p0]) continue;

        if (K == 2) {
            // lanes over p1
            const int n1 = cand_count(a.cnt, c0.x, 0);
            for (int t1 = lane; t1 < ((n1 + 31) & ~31); t1 += 32) {
                bool valid = t1 < n1;
                int p1 = 0;
                if (valid) { p1 = a.list[size_t(c0.x) * n + t1]; valid = p1 != p0 && (!al || al[p1]); }
                int nfeas = 0, best = INT_MAX;
                if (valid) {
                    const int4 c1 = cust[p1];
                    const int a01 = D(c0.x, c1.x);
                    const int sl0 = c0.z - a01, sl1 = c1.z;
                    const int e0 = D(c1.x, c0.y), e1 = D(c1.x, c1.y);
                    const int t01 = D(c0.y, c1.y), t10 = D(c1.y, c0.y);
                    // perm 0: drop 0 then 1; perm 1: drop 1 then 0
                    const bool okA = e0 <= sl0 && e0 + t01 <= sl1;
                    const bool okB = e1 <= sl1 && e1 + t10 <= sl0;
                    const int kA = ((a01 + e0 + t01) << kPermBits) | 0, kB = ((a01 + e1 + t10) << kPermBits) | 1;
                    nfeas = int(okA) + int(okB);
                    if (okA) best = kA;
                    if (okB && kB < best) best = kB;
                    my_eval += 2;
                    my_feas += nfeas;
                }
                emit_records(a, wo, nfeas > 0, make_rank(p0, p1, 0, 0, best & 31), best >> kPermBits, lane, whist);
            }
            continue;
        }

        const int t1 = int(item - ioff[lo]);
        const int p1 = a.list[size_t(c0.x) * n + t1];
        if (p1 == p0 || (al && !al[p1])) continue;
        const int4 c1 = cust[p1];
        const int a01 = D(c0.x, c1.x);  // <= W[p1] by construction of the prefix

        if (K == 3) {
            const int t01 = D(c0.y, c1.y), t10 = D(c1.y, c0.y);
            const int n2 = cand_count(a.cnt, c1.x, a01);
            for (int t2 = lane; t2 < ((n2 + 31) & ~31); t2 += 32) {
                bool valid = t2 < n2;
                int p2 = 0;
                if (valid) {
                    p2 = a.list[size_t(c1.x) * n + t2];
                    valid = p2 != p0 && p2 != p1 && (a01 < kTbl || a.slack[size_t(c1.x) * n + t2] >= a01) && (!al || al[p2]);
                }
                int nfeas = 0, best = INT_MAX;
                if (valid) {
                    const int4 c2 = cust[p2];
                    const int a12 = D(c1.x, c2.x);
                    int e[3], t[3][3], sl[3];
                    e[0] = D(c2.x, c0.y); e[1] = D(c2.x, c1.y); e[2] = D(c2.x, c2.y);
                    t[0][0] = t[1][1] = t[2][2] = 0;
                    t[0][1] = t01; t[1][0] = t10;
                    t[0][2] = D(c0.y, c2.y); t[2][0] = D(c2.y, c0.y);
                    t[1][2] = D(c1.y, c2.y); t[2][1] = D(c2.y, c1.y);
                    sl[2] = c2.z; sl[1] = c1.z - a12; sl[0] = c0.z - a01 - a12;
                    eval3(e, t, sl, a01 + a12, nfeas, best);
                    my_eval += 6;
                    my_feas += nfeas;
                }
                emit_records(a, wo, nfeas > 0, make_rank(p0, p1, p2, 0, best & 31), best >> kPermBits, lane, whist);
            }
            continue;
        }

        // K == 4: the (third pickup, last pickup) pairs of the item are flattened over the lanes.  Per batch of 32 third
        // pickups: lane l prepares candidate b2 + l (validity, slacks, length n3 of its last-pickup prefix, the bound at
        // this level), a warp scan turns the lengths into offsets, and every lane then walks flat pair indices f, f + 32,
        // ...  A pair that passes the bound is pushed on the warp's queue; whenever 32 tuples are queued they are
        // evaluated, one per lane (all 24 drop-off orders).  a01 and every D() below are in the x32 fixed point of eval4s.
        const int a01u = a01 >> SH;
        const int n2 = cand_count(a.cnt, c1.x, a01u);
        // Second necessary condition (next to "every passenger reaches his drop-off within his slack"): among the
        // passengers on board, the one dropped LAST has every other drop-off on his way -- for some l and every other j on
        // board,  D*(F_last, T_j) + D*(T_j, T_l) <= slack_l  (the drop route to T_l passes T_j first, every leg of it is at
        // least the closure distance, and later pickups only lengthen it by the triangle inequality of the closure).
        // Checked on the first two passengers per item, on the first three per third pickup (together these prune 57 %
        // of the last-pickup walks of config 3) and again per tuple with the last pickup stand (36 % fewer evaluations).
        const int tc01 = pf ? Dc(c0.y, c1.y) : 0, tc10 = pf ? Dc(c1.y, c0.y) : 0;
        bool item_ok = true;
        if (pf) {
            const int f0 = Dc(c1.x, c0.y), f1 = Dc(c1.x, c1.y), z0 = c0.z - a01;
            item_ok = f0 <= z0 && f1 <= c1.z && (f1 + tc10 <= z0 || f0 + tc01 <= c1.z);
        }
        const unsigned long long ent01 = (((unsigned long long)unsigned(p0) << kCustBits) | unsigned(p1)) << (2 * kCustBits);
        unsigned my_tuples = 0;                        // valid pickup tuples seen by this lane (x 24 leaves each)
        for (int b2 = first_batch_only ? 0 : 32; b2 < (first_batch_only ? (n2 < 32 ? n2 : 32) : n2); b2 += 32) {
            const int t2 = b2 + lane;
            int n3l = 0;
            int4 A = make_int4(-1, 0, 0, 0), B = make_int4(0, 0, 0, 0), C = make_int4(0, 0, 0, 0);
            if (t2 < n2) {
                const int p2l = a.list[size_t(c1.x) * n + t2];
                bool ok = p2l != p0 && p2l != p1 && (!al || al[p2l]);
                if (ok && a01u >= kTbl) ok = a.slack[size_t(c1.x) * n + t2] >= a01u;
                if (ok) {
                    const int4 c2 = cust[p2l];
                    const int a12 = D(c1.x, c2.x);
                    const int w2 = a01 + a12;
                    n3l = cand_count(a.cnt, c2.x, w2 >> SH);
                    A = make_int4(p2l, c2.x, w2, c0.z - w2);
                    B = make_int4(c1.z - a12, c2.z, c2.y, 0);
                    bool keep = true;
                    if (pf) {
                        const int d0 = Dc(c2.x, c0.y), d1 = Dc(c2.x, c1.y), d2 = Dc(c2.x, c2.y);
                        C = make_int4(Dc(c0.y, c2.y), Dc(c2.y, c0.y), Dc(c1.y, c2.y), Dc(c2.y, c1.y));   // tc02, tc20, tc12, tc21
                        keep = item_ok && d0 <= A.w && d1 <= B.x && d2 <= B.y &&
                               ((d1 + tc10 <= A.w && d2 + C.y <= A.w) || (d0 + tc01 <= B.x && d2 + C.w <= B.x) ||
                                (d0 + C.x <= B.y && d1 + C.z <= B.y));
                    }
                    if (!keep && (w2 >> SH) < kTbl) {
                        // no last pickup and no drop-off order can make (p0, p1, p2) feasible.  Its leaves are counted, not
                        // visited: the last-pickup candidates are exactly the customers with slack >= wait so far at F2
                        // (the list prefix of length n3l), minus the three that are already on board.
                        const int lim = 1 << 25;
                        auto on_list = [&](const int4 c) { return (c.w < lim ? c.w : lim) * (1 << SH) - D(c2.x, c.x) >= w2 ? 1 : 0; };
                        my_tuples += unsigned(n3l - on_list(c0) - on_list(c1) - on_list(c2));
                        n3l = 0;
                    }
                }
            }
            int incl = n3l;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            B.w = incl;
            __syncwarp();
            stA[lane] = A;
            stB[lane] = B;
            stC[lane] = C;
            __syncwarp();
            int sidx = 0, prev_end = 0;                // this lane's position in the batch: ranges are visited in order
            for (int f0 = 0; f0 < total; f0 += 32) {
                const int f = f0 + lane;
                bool valid = f < total;
                int p3 = 0;
                int4 sa = A, sb = B;
                if (valid) {
                    int end = stB[sidx].w;
                    while (end <= f) { prev_end = end; end = stB[++sidx].w; }
                    sa = stA[sidx]; sb = stB[sidx];
                    const int t3 = f - prev_end;
                    const int w2u = sa.z >> SH;
                    p3 = a.list[size_t(sa.y) * n + t3];
                    valid = p3 != p0 && p3 != p1 && p3 != sa.x && (w2u < kTbl || a.slack[size_t(sa.y) * n + t3] >= w2u) &&
                            (!al || al[p3]);
                }
                bool pass = valid;
                if (valid) {
                    ++my_tuples;
                    if (pf) {
                        const int4 c3 = cust[p3];
                        const int4 sc = stC[sidx];
                        const int a23 = D(sa.y, c3.x);
                        const int e0 = Dc(c3.x, c0.y), e1 = Dc(c3.x, c1.y), e2 = Dc(c3.x, sb.z);
                        const int x0 = sa.w - a23, x1 = sb.x - a23, x2 = sb.y - a23;
                        pass = e0 <= x0 && e1 <= x1 && e2 <= x2 && Dc(c3.x, c3.y) <= c3.z &&
                               ((e1 + tc10 <= x0 && e2 + sc.y <= x0) || (e0 + tc01 <= x1 && e2 + sc.w <= x1) ||
                                (e0 + sc.x <= x2 && e1 + sc.z <= x2));
                    }
                }
                const unsigned ball = __ballot_sync(0xffffffffu, pass);
                if (pass)
                    queue[(q_head + q_cnt + __popc(ball & lt_mask)) & 63] =
                        ent01 | ((unsigned long long)unsigned(sa.x) << kCustBits) | unsigned(p3);
                q_cnt += __popc(ball);
                __syncwarp();
                if (q_cnt >= 32) eval_queue(32);
            }
        }
        my_eval += 24ull * my_tuples;
    }
    // close the last chunk (the queue was drained and the counters published when the item loop ended)
    if (wo.base != 0xffffffffu)
        for (unsigned t = wo.used + lane; t < kChunk; t += 32) mark_hole(a, rec_key64(a), wo.base + t);
}

// ---- selection -----------------------------------------------------------------------------------
struct SelArgs {
    PoolRec *list[2]; PoolRec *act[2]; PoolCtrl *ctrl;
    unsigned long long *best_hi[2]; unsigned int *best_lo[2]; uint8_t *alive; PoolRec *kept;
    int n, K;
    int n_slots, step, shard_begin, keep_cap;   // per-slot state lives at [slot * n + customer]
    unsigned int step_inv;                      // ceil(2^32 / step): p0 / step == umulhi(p0, step_inv) for p0, step <= 2^14 (p0 * step < 2^32)
    int first_pass;                             // 1: every customer starts free; 0: keep alive[] from the earlier windows
    int cost_hi;                                // records with cost >= cost_hi were counted in hist but not materialised
    unsigned int band0, band_growth;            // records of the first cost band, growth factor of the band sizes
    unsigned int frag_cap;                      // records per CTA fragment of act[] (see the filter step)
};

// Minimum of `key` over the run of consecutive lanes that hold the same cell (any lanes with an equal cell may be
// folded in: every one of them is a valid contribution to that cell).  Returns true on the first lane of a run -- the one
// that issues the atomic for it.  Emission order survives the partition and the compaction in runs, so consecutive
// records share the leader, mostly the second pickup and often the third: one atomic per run instead of one per record
// (same-address atomics serialise in L2).  Every lane of the warp must call it.
__device__ __forceinline__ unsigned long long sel_warp_min(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w < v ? w : v;
    }
    return v;
}

constexpr int kRunMinLive = 12;   // live records in a warp's batch from which the run minima are taken
__device__ __forceinline__ bool sel_run_min(int cell, unsigned long long &key, bool live, unsigned ball, unsigned lane) {
    // dead lanes (key = ~0) take the cell of the nearest live lane below them, so that they do not cut a run in two
    const unsigned below = ball & ((1u << lane) - 1);
    const int filled = __shfl_sync(0xffffffffu, cell, below ? 31 - __clz(below) : int(lane));
    if (!live) cell = below ? filled : -1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int oc = __shfl_down_sync(0xffffffffu, cell, o);
        const unsigned long long ok = __shfl_down_sync(0xffffffffu, key, o);
        if (lane + o < 32 && oc == cell && ok < key) key = ok;
    }
    const int pc = __shfl_up_sync(0xffffffffu, cell, 1);
    return lane == 0 || pc != cell;
}

__device__ __forceinline__ unsigned long long rec_hi(const PoolRec &r) {
    return ((unsigned long long)(unsigned)r.cost << 32) | (r.rank >> 32);
}
// Single-level key of a PoolRec (pack_key1).  Usable when every materialised cost is below 2^(64 - 4 cb - 5) (config 3:
// cb = 10, costs below 2^19); it removes the second-level pass, one grid barrier and the best_lo lookups from every
// dominance round.
__device__ __forceinline__ unsigned long long rec_key1(const PoolRec &r, int cb) { return pack_key1(r.cost, r.rank, cb); }

// The two formats of the record list, for the passes of pool_select_body.  Both give a record's cost, customers and
// first-level key; kept plans are stored as PoolRec either way (pool_emit reads those).
struct RecFmt16 {                  // PoolRec: any cost; single-level or two-level keys, decided from the histogram
    using R = PoolRec;
    static constexpr bool kSingle = false;
    static constexpr int kPartPer = 4, kFiltPer = 4;
    __device__ static bool hole(const R &r) { return r.cost < 0; }
    __device__ static R make_hole() { PoolRec r; r.rank = 0; r.cost = -1; r.pad = 0; return r; }
    __device__ static int cost(const R &r, int) { return r.cost; }
    __device__ static int lead(const R &r, int) { return int(r.rank >> (3 * kCustBits + kPermBits)); }
    __device__ static void cust(const R &r, int, int p[4]) { int perm; split_rank(r.rank, p, perm); }
    __device__ static unsigned long long key(const R &r, int cb, bool single) { return single ? rec_key1(r, cb) : rec_hi(r); }
    __device__ static unsigned key_lo(const R &r) { return unsigned(r.rank); }
    __device__ static PoolRec rec(const R &r, int) { return r; }
};
struct RecFmt8 {                   // the single-level key itself (key64_fits): no repacking, no second level
    using R = unsigned long long;
    static constexpr bool kSingle = true;
    static constexpr int kPartPer = 4, kFiltPer = 4;
    __device__ static bool hole(const R &r) { return r == kKeyHole; }
    __device__ static R make_hole() { return kKeyHole; }
    __device__ static int cost(const R &r, int cb) { return int(r >> (4 * cb + kPermBits)); }
    __device__ static int lead(const R &r, int cb) { return int(r >> (3 * cb + kPermBits)) & ((1 << cb) - 1); }
    __device__ static void cust(const R &r, int cb, int p[4]) {
        const unsigned m = (1u << cb) - 1;
        p[3] = int(unsigned(r >> kPermBits) & m);
        p[2] = int(unsigned(r >> (cb + kPermBits)) & m);
        p[1] = int(unsigned(r >> (2 * cb + kPermBits)) & m);
        p[0] = int(unsigned(r >> (3 * cb + kPermBits)) & m);
    }
    __device__ static unsigned long long key(const R &r, int, bool) { return r; }
    __device__ static unsigned key_lo(const R &) { return 0u; }
    __device__ static PoolRec rec(const R &r, int cb) {
        int p[4];
        cust(r, cb, p);
        PoolRec o; o.rank = make_rank(p[0], p[1], p[2], p[3], int(unsigned(r) & ((1u << kPermBits) - 1))); o.cost = cost(r, cb); o.pad = 0;
        return o;
    }
};

// Selection = the reference's sort-by-cost + greedy scan (pool_n.c:187-207), done as dominance rounds.
// Cost is the leading key, so the scan over records with cost < t is a prefix of the whole scan:
// records are processed in ascending COST BANDS (sizes grow 4x; bounds per shard from the cost
// histogram that pool_enum accumulates).
//   partition   one streaming pass moves every record into its band's segment (exact sizes are known)
//   per band    (1) filter: records of the band whose customers are all still free go to the active list,
//                   first-level key minima are taken on the fly;
//               (2) dominance rounds on the active list only (all shards of the call together; plans of
//                   different shards never interact because their state is indexed by shard).
// Each record is read ~3 times in total; the rounds touch only the live in-band records
// (config 3: ~0.3 M record visits per shard instead of ~7.5 M x 3 passes on the unbanded list).
// F: the record format (RecFmt16 / RecFmt8) of list[], act[]; kept[] is PoolRec either way.
template <class F>
__device__ __forceinline__ void pool_select_body(const SelArgs &a) {
    using R = typename F::R;
    cg::grid_group grid = cg::this_grid();
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned nthreads = gridDim.x * blockDim.x;
    const unsigned lane = threadIdx.x & 31;
    const int K = a.K;
    const int n = a.n;
    PoolCtrl *ctrl = a.ctrl;
    if (tid == 0) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ctrl->tstamp[31] = t; }
    __shared__ int s_band_hi[kMaxSlots][kMaxBands];
    const unsigned n_state = unsigned(n) * unsigned(a.n_slots);
    for (unsigned c = tid; c < n_state; c += nthreads) {
        if (a.first_pass) a.alive[c] = 1;
        a.best_hi[0][c] = a.best_hi[1][c] = ~0ull;
        a.best_lo[0][c] = a.best_lo[1][c] = ~0u;
    }
    if (int(blockIdx.x) < a.n_slots) {   // band bounds of shard blockIdx.x: cumulative histogram against 4x growing targets
        __shared__ unsigned s_hist[kBuckets];
        const int sl = int(blockIdx.x);
        for (int bkt = threadIdx.x; bkt < kBuckets; bkt += blockDim.x) s_hist[bkt] = bkt < a.cost_hi ? unsigned(ctrl->hist[sl][bkt]) : 0u;   // materialised records: < 2^32
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long cum = 0, target = a.band0;
            unsigned in_band = 0;
            int band = 0;
            for (int bkt = 0; bkt < kBuckets; ++bkt) {
                const unsigned h = s_hist[bkt];
                cum += h; in_band += h;
                if (band < kMaxBands - 1 && bkt < kBuckets - 1 && cum >= target) {
                    ctrl->band_hi[sl][band] = bkt + 1;
                    ctrl->band_cnt[sl][band] = in_band;
                    atomicAdd(&ctrl->band_off[band + 1], in_band);   // sizes first, prefix below
                    ++band; in_band = 0; target = cum * (unsigned long long)a.band_growth;
                }
            }
            ctrl->band_hi[sl][band] = INT_MAX;
            ctrl->band_cnt[sl][band] = in_band;
            atomicAdd(&ctrl->band_off[band + 1], in_band);
            for (int b2 = band + 1; b2 < kMaxBands; ++b2) { ctrl->band_hi[sl][b2] = INT_MAX; ctrl->band_cnt[sl][b2] = 0; }
        }
    }
    grid.sync();
    if (tid == 0) {
        unsigned run = 0;
        for (int b2 = 0; b2 < kMaxBands; ++b2) {   // band_off[b+1] holds size(b): turn into offsets
            const unsigned sz = ctrl->band_off[b2 + 1];
            ctrl->band_off[b2] = run; ctrl->band_cur[b2] = run;
            run += sz;
        }
        ctrl->band_off[kMaxBands] = run;
    }
    grid.sync();
    for (int i = threadIdx.x; i < a.n_slots * kMaxBands; i += blockDim.x) s_band_hi[i / kMaxBands][i % kMaxBands] = ctrl->band_hi[i / kMaxBands][i % kMaxBands];
    __syncthreads();
    // p0 / step without a division per record (step_inv == 0: step is 1)
    auto slot_of = [&](int p0) -> int { return (a.step_inv ? int(__umulhi(unsigned(p0), a.step_inv)) : p0) - a.shard_begin; };
    // single-level keys when every materialised cost fits beside the repacked rank (8-byte records: always; PoolRec:
    // uniform, from the histogram)
    const int cb = key_cb(n);
    const int cost_bits = 64 - 4 * cb - kPermBits;
    bool single_key = F::kSingle || cost_bits >= 1;
    if (!F::kSingle && single_key) {
        const int lim = cost_bits >= 31 ? kBuckets - 1 : (int)min((long long)kBuckets - 1, 1ll << cost_bits);
        // every bucket at or above the limit (and the open-ended last bucket) must be empty
        for (int sl = 0; sl < a.n_slots && single_key; ++sl)
            for (int bkt = lim; bkt < kBuckets && bkt < a.cost_hi; ++bkt)
                if (ctrl->hist[sl][bkt] != 0) { single_key = false; break; }
        if (single_key)
            for (int sl = 0; sl < a.n_slots && single_key; ++sl)
                if ((kBuckets - 1) < a.cost_hi && ctrl->hist[sl][kBuckets - 1] != 0) single_key = false;
    }
    int ts_i = 0;
    auto stamp = [&]() {
        if (tid == 0 && ts_i < 32) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); ctrl->tstamp[ts_i] = t; }
        ++ts_i;
    };
    stamp();

    // ---- partition pass: list[0] (emission order, with holes) -> list[1] (band segments) ------------------
    // Block-aggregated: a CTA classifies kPartPer records per thread, counts them per band in shared memory,
    // reserves one contiguous range per band with ONE global atomic each, then scatters.
    {
        constexpr int kPartPer = F::kPartPer;
        __shared__ unsigned s_bcnt[kMaxBands], s_bbase[kMaxBands];
        const unsigned cnt = ctrl->overflow ? 0u : ctrl->n_records;
        const R *src = reinterpret_cast<const R *>(a.list[0]);
        R *dst = reinterpret_cast<R *>(a.list[1]);
        const unsigned chunk = blockDim.x * kPartPer;
        for (unsigned base = blockIdx.x * chunk; base < cnt; base += gridDim.x * chunk) {
            if (threadIdx.x < kMaxBands) s_bcnt[threadIdx.x] = 0;
            __syncthreads();
            R r[kPartPer];
            int band[kPartPer];
            unsigned lrank[kPartPer];
#pragma unroll
            for (int u = 0; u < kPartPer; ++u) {
                const unsigned i = base + u * blockDim.x + threadIdx.x;
                band[u] = -1;
                r[u] = i < cnt ? src[i] : F::make_hole();
            }
#pragma unroll
            for (int u = 0; u < kPartPer; ++u) {
                if (F::hole(r[u])) continue;
                const int slot = slot_of(F::lead(r[u], cb));
                const int cost = F::cost(r[u], cb);
                int bsel = 0;
                while (cost >= s_band_hi[slot][bsel]) ++bsel;
                band[u] = bsel;
            }
#pragma unroll
            for (int u = 0; u < kPartPer; ++u) {   // one shared-memory atomic per distinct band per warp
                const unsigned peers = __match_any_sync(0xffffffffu, band[u]);
                unsigned wbase = 0;
                const int leader = __ffs(peers) - 1;
                if (band[u] >= 0 && int(lane) == leader) wbase = atomicAdd(&s_bcnt[band[u]], __popc(peers));
                wbase = __shfl_sync(0xffffffffu, wbase, leader);
                lrank[u] = wbase + __popc(peers & ((1u << lane) - 1));
            }
            __syncthreads();
            if (threadIdx.x < kMaxBands && s_bcnt[threadIdx.x])
                s_bbase[threadIdx.x] = atomicAdd(&ctrl->band_cur[threadIdx.x], s_bcnt[threadIdx.x]);
            __syncthreads();
#pragma unroll
            for (int u = 0; u < kPartPer; ++u)
                if (band[u] >= 0) dst[s_bbase[band[u]] + lrank[u]] = r[u];
        }
    }
    grid.sync();
    stamp();

    unsigned rounds = 0, par = 0;
    for (int band = 0; band < kMaxBands; ++band) {
        const unsigned b0 = ctrl->band_off[band], b1 = ctrl->band_off[band + 1];
        if (b0 == b1) continue;   // uniform: nothing in this band
        // ---- filter: live records of the band -> active list, first-level minima on the fly -------------------
        // The active list is FRAGMENTED over the CTAs: a CTA appends the live records of its chunks to its own fragment
        // (shared-memory cursor: no block barrier and no global atomic with a return value inside the loops) and every
        // later pass of the band works on that fragment.  Only the totals (termination test), alive[] and the
        // per-customer minima are shared through global memory.
        __shared__ unsigned s_cnt;               // records in this CTA's fragment of the list being written
        // frag_cap counts PoolRec: an 8-byte fragment starts at the same byte and holds twice the records
        const size_t frag = size_t(blockIdx.x) * a.frag_cap * (sizeof(PoolRec) / sizeof(R));
        unsigned my_cnt = 0;
        {
            constexpr int kFiltPer = F::kFiltPer;
            const R *src = reinterpret_cast<const R *>(a.list[1]);
            R *act = reinterpret_cast<R *>(a.act[0]) + frag;
            // records per thread and chunk: fewer for a small band, so that its live records (and with them the work of
            // the rounds, which stay on the fragments) spread over more CTAs
            const unsigned want = (b1 - b0 + nthreads - 1) / nthreads;
            const int per = want >= unsigned(kFiltPer) ? kFiltPer : (want < 1u ? 1 : int(want));
            const unsigned chunk = blockDim.x * per;
            __syncthreads();
            if (threadIdx.x == 0) s_cnt = 0;
            __syncthreads();
            for (unsigned base = b0 + blockIdx.x * chunk; base < b1; base += gridDim.x * chunk) {
                R r[kFiltPer];
                bool live[kFiltPer];
                int p[kFiltPer][4];
#pragma unroll
                for (int u = 0; u < kFiltPer; ++u) {
                    const unsigned i = base + u * blockDim.x + threadIdx.x;
                    live[u] = u < per && i < b1;
                    if (live[u]) r[u] = src[i];
                }
#pragma unroll
                for (int u = 0; u < kFiltPer; ++u) {
                    if (!live[u]) continue;
                    F::cust(r[u], cb, p[u]);
                    const int so = slot_of(p[u][0]) * n;
                    uint8_t fl[4];                       // the four flags are loaded together (no short-circuit chain)
#pragma unroll
                    for (int q = 0; q < 4; ++q) { p[u][q] += so; fl[q] = q < K ? a.alive[p[u][q]] : uint8_t(1); }
                    live[u] = fl[0] && fl[1] && fl[2] && fl[3];
                }
#pragma unroll
                for (int u = 0; u < kFiltPer; ++u) {   // warp-aggregated shared-memory cursor
                    const unsigned ball = __ballot_sync(0xffffffffu, live[u]);
                    if (ball == 0) continue;
                    unsigned wbase = 0;
                    if (lane == 0) wbase = atomicAdd(&s_cnt, __popc(ball));
                    wbase = __shfl_sync(0xffffffffu, wbase, 0);
                    const unsigned long long hi = live[u] ? F::key(r[u], cb, single_key) : ~0ull;
                    unsigned long long rmin[3];
                    bool head[3];
#pragma unroll
                    for (int q = 0; q < 3; ++q) { rmin[q] = hi; head[q] = q < K; }
                    if (band == 0 && __popc(ball) >= kRunMinLive) {   // uniform.  First band, dense survivors: per-run minima
                                                                      // (sel_run_min); the later bands' survivors are sparse
#pragma unroll
                        for (int q = 0; q < 3; ++q)
                            if (q < K) head[q] = sel_run_min(live[u] ? p[u][q] : -1, rmin[q], live[u], ball, lane);
                    } else {                                 // sparse survivors: only the leader's cell is worth a reduction
                        const int cell0 = live[u] ? p[u][0] : -1;
                        const int lead = __ffs(ball) - 1;
                        const int lead_cell = __shfl_sync(0xffffffffu, cell0, lead);
                        if (__all_sync(0xffffffffu, !live[u] || cell0 == lead_cell)) {
                            rmin[0] = sel_warp_min(hi);
                            head[0] = int(lane) == lead;
                        }
                    }
                    if (live[u]) {
                        act[wbase + __popc(ball & ((1u << lane) - 1))] = r[u];
                        // the test spares most of the atomics; the four current minima are loaded TOGETHER before the first
                        // atomic -- behind an atomic the compiler may not hoist the next load, which made this four dependent
                        // L2 round trips per live record.  A stale (larger) value only costs a redundant atomic.
                        unsigned long long cur4[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) cur4[q] = q < K ? a.best_hi[par][p[u][q]] : 0ull;
#pragma unroll
                        for (int q = 0; q < 3; ++q)
                            if (head[q] && rmin[q] < cur4[q]) atomicMin(&a.best_hi[par][p[u][q]], rmin[q]);
                        if (3 < K && hi < cur4[3]) atomicMin(&a.best_hi[par][p[u][3]], hi);
                    }
                }
            }
            __syncthreads();
            my_cnt = s_cnt;
            if (threadIdx.x == 0 && my_cnt) atomicAdd(&ctrl->act_cnt[band][0], my_cnt);
        }
        grid.sync();
        stamp();
        // ---- dominance rounds on the active list (all shards of the call at once) --------------------------------
        unsigned al = 0;
        for (unsigned r = 0;; ++r) {
            if (r > 0) {   // pass A: drop the plans killed by the previous round, compact, first-level minima
                const R *src = reinterpret_cast<const R *>(a.act[al]) + frag;
                R *dst = reinterpret_cast<R *>(a.act[al ^ 1]) + frag;
                __syncthreads();
                if (threadIdx.x == 0) s_cnt = 0;
                __syncthreads();
                for (unsigned base = 0; base < my_cnt; base += blockDim.x) {
                    const unsigned i = base + threadIdx.x;
                    bool live = false;
                    R rec;
                    int p[4];
                    if (i < my_cnt) {
                        rec = src[i];
                        F::cust(rec, cb, p);
                        const int so = slot_of(p[0]) * n;
                        uint8_t fl[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) { p[q] += so; fl[q] = q < K ? a.alive[p[q]] : uint8_t(1); }
                        live = fl[0] && fl[1] && fl[2] && fl[3];
                    }
                    const unsigned ball = __ballot_sync(0xffffffffu, live);
                    if (ball == 0) continue;
                    unsigned wbase = 0;
                    if (lane == 0) wbase = atomicAdd(&s_cnt, __popc(ball));
                    wbase = __shfl_sync(0xffffffffu, wbase, 0);
                    const unsigned long long hi = live ? F::key(rec, cb, single_key) : ~0ull;
                    unsigned long long rmin[3];
                    bool head[3];
#pragma unroll
                    const bool dense = __popc(ball) >= kRunMinLive;
                    for (int q = 0; q < 3; ++q) {           // see the filter
                        rmin[q] = hi;
                        head[q] = q < K && ((q > 0 && !dense) || sel_run_min(live ? p[q] : -1, rmin[q], live, ball, lane));
                    }
                    if (live) {
                        dst[wbase + __popc(ball & ((1u << lane) - 1))] = rec;
                        unsigned long long cur4[4];          // loaded together, see the filter
#pragma unroll
                        for (int q = 0; q < 4; ++q) cur4[q] = q < K ? a.best_hi[par][p[q]] : 0ull;
#pragma unroll
                        for (int q = 0; q < 3; ++q)
                            if (head[q] && rmin[q] < cur4[q]) atomicMin(&a.best_hi[par][p[q]], rmin[q]);
                        if (3 < K && hi < cur4[3]) atomicMin(&a.best_hi[par][p[3]], hi);
                    }
                }
                __syncthreads();
                my_cnt = s_cnt;
                if (threadIdx.x == 0 && my_cnt) atomicAdd(&ctrl->act_cnt[band][al ^ 1], my_cnt);
                grid.sync();
                al ^= 1;
            }
            const unsigned n_act = ctrl->act_cnt[band][al];
            if (n_act == 0) break;
            const R *cur = reinterpret_cast<const R *>(a.act[al]) + frag;
            // pass B: second-level minimum among the plans that tie on the first level (two-level keys only)
            if (!single_key)
            for (unsigned i = threadIdx.x; i < my_cnt; i += blockDim.x) {
                const R rec = cur[i];
                int p[4];
                F::cust(rec, cb, p);
                const int so = slot_of(p[0]) * n;
                const unsigned long long hi = F::key(rec, cb, false);
                const unsigned lo = F::key_lo(rec);
                for (int q = 0; q < K; ++q)
                    if (a.best_hi[par][so + p[q]] == hi && lo < a.best_lo[par][so + p[q]]) atomicMin(&a.best_lo[par][so + p[q]], lo);
            }
            if (tid == 0) ctrl->act_cnt[band][al ^ 1] = 0;   // target of the next round's pass A
            if (!single_key) grid.sync();
            // pass C: keep the plans that hold the minimum at every one of their customers
            for (unsigned i = threadIdx.x; i < my_cnt; i += blockDim.x) {
                const R rec = cur[i];
                int p[4];
                F::cust(rec, cb, p);
                const int slot = slot_of(p[0]);
                const int so = slot * n;
                const unsigned long long hi = F::key(rec, cb, single_key);
                const unsigned lo = F::key_lo(rec);
                unsigned long long bh[4];
                unsigned bl[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {            // loaded together, then compared
                    bh[q] = q < K ? a.best_hi[par][so + p[q]] : hi;
                    bl[q] = (q < K && !single_key) ? a.best_lo[par][so + p[q]] : lo;
                }
                const bool dom = bh[0] == hi && bh[1] == hi && bh[2] == hi && bh[3] == hi &&
                                 bl[0] == lo && bl[1] == lo && bl[2] == lo && bl[3] == lo;
                if (dom) {
                    const unsigned pos = atomicAdd(&ctrl->n_kept[slot], 1u);
                    a.kept[size_t(slot) * a.keep_cap + pos] = F::rec(rec, cb);
                    for (int q = 0; q < K; ++q) a.alive[so + p[q]] = 0;
                }
            }
            // reset the other parity's minima for the next round (nobody reads them in this round)
            for (unsigned c = tid; c < n_state; c += nthreads) { a.best_hi[par ^ 1][c] = ~0ull; a.best_lo[par ^ 1][c] = ~0u; }
            grid.sync();
            par ^= 1;
            ++rounds;
        }
        stamp();
    }
    if (tid == 0) { ctrl->rounds = rounds; ctrl->total_rounds += rounds; }
}

__global__ void __launch_bounds__(kSelThreads, 2)   // 64 registers: two CTAs per SM keep the streaming passes fed
pool_select_kernel(SelArgs a) {
    // The record list overflowed (asynchronous single pass) or the input was refused: the histogram kept counting, so the
    // band sizes exceed what was materialised -- nothing below may run.  Both flags are final when the enumeration has
    // ended, every thread of the grid sees the same values and leaves before the first barrier; pool_emit reports -1.
    // The record format is uniform as well (set by pool_build_lists; 0 in td_pool_pairs' zeroed block).
    if (a.ctrl->overflow || a.ctrl->bad_input) return;
    if (a.ctrl->key64) pool_select_body<RecFmt8>(a);
    else pool_select_body<RecFmt16>(a);
}

// kept plans -> ascending (cost, rank) -> pool_n.c:123-134 records
__global__ void __launch_bounds__(1024)
pool_emit_kernel(const PoolRec *__restrict__ kept_all, const PoolCtrl *ctrl, int K, int keep_cap, int32_t *plans_all,
                 int32_t cap, int32_t *counts_out, int headed) {
    // headed: every shard's block is (cap + 1) rows, row 0 is a header {count, evaluated lo, hi, feasible lo, hi, 0, 0, 0, 0}
    // -- the block travels through ONE collective with its count and its counters (td_pool_find_shards_headed)
    const int slot = blockIdx.x;
    const PoolRec *kept = kept_all + size_t(slot) * keep_cap;
    int32_t *block = plans_all + size_t(slot) * (cap + (headed ? 1 : 0)) * TD_POOL_REC_W;
    int32_t *plans_out = block + (headed ? TD_POOL_REC_W : 0);
    const int m = int(ctrl->n_kept[slot]);
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const PoolRec me = kept[i];
        int rank = 0;
        for (int j = 0; j < m; ++j) {
            const PoolRec o = kept[j];
            rank += (o.cost < me.cost) || (o.cost == me.cost && o.rank < me.rank);
        }
        if (rank < cap) {
            int p[4], perm;
            split_rank(me.rank, p, perm);
            // decode the lexicographic permutation index into the drop-off order
            int q[4] = {0, 0, 0, 0};
            bool used[4] = {false, false, false, false};
            int fact = 1;
            for (int f = 2; f < K; ++f) fact *= f;  // (K-1)!
            int rem = perm;
            for (int lvl = 0; lvl < K; ++lvl) {
                int idx = rem / fact; rem -= idx * fact;
                if (K - 1 - lvl > 0) fact /= (K - 1 - lvl);
                int c = 0;
                for (int cand = 0; cand < K; ++cand) {
                    if (used[cand]) continue;
                    if (c == idx) { q[lvl] = cand; used[cand] = true; break; }
                    ++c;
                }
            }
            int32_t *row = plans_out + size_t(rank) * TD_POOL_REC_W;
            for (int t = 0; t < TD_POOL_REC_W; ++t) row[t] = 0;
            for (int t = 0; t < K; ++t) { row[t] = p[t]; row[t + K] = p[q[t]]; }
            row[8] = me.cost;
        }
    }
    if (threadIdx.x == 0) {
        const int count = (ctrl->overflow || ctrl->bad_input) ? -1 : m;  // -1: record list overflowed / unsupported input
        if (counts_out) counts_out[slot] = count;
        if (headed) {
            const unsigned long long ev = ctrl->evaluated[slot], fe = ctrl->feasible[slot];
            block[0] = count;
            block[1] = int32_t(unsigned(ev)); block[2] = int32_t(unsigned(ev >> 32));
            block[3] = int32_t(unsigned(fe)); block[4] = int32_t(unsigned(fe >> 32));
            block[5] = block[6] = block[7] = block[8] = 0;
        }
    }
}

// ---- merge (findpool.c:83-108) ---------------------------------------------------------------
// One CTA.  Valid rows are compacted first (padded layout: slot s holds `cap` rows after `headed` header rows, row r of
// the slot is valid iff r < count(s); slot_shard[slot] = logical shard, concatenation order = shard order).  Scan order =
// (column 8, concatenation position) for K == 4, concatenation position otherwise (see header: findpool.c sorts on a
// column it never filled for K < 4).  Then the same dominance rounds as pool_select on the small list.
//
// Up to kMergeFast valid rows (config 3: 678; 5000 customers: ~5000 of the 8 x 1250 possible) everything after the
// compaction runs in shared memory: a bitonic sort of the 64-bit scan keys, dominance rounds with the SORTED POSITION as
// a 32-bit key (native shared-memory atomicMin on a per-customer table), a block scan for the output positions.
// More rows take the general path (ranks by counting, state in the global workspace).
// The rows may come from a caller, and both paths index a per-customer table with their customers: a valid row with a
// customer outside [0, n) makes the merge write *n_plans_out = -1 and return before any such indexing.
constexpr int kMergeSlots = 64;   // pool_merge ranks by binary search when it has at most this many (sorted) slots
constexpr int kMergeFast = 8192;
__global__ void __launch_bounds__(1024)
pool_merge_kernel(const int32_t *__restrict__ plans, int n_slots, int n, int K, const int32_t *__restrict__ counts, int cap,
                  int headed, int fast_cap, const int32_t *__restrict__ slot_shard, unsigned long long *ckey /* total */,
                  int32_t *crow /* total */, int32_t *order_key /* total */, int32_t *owner /* n */, uint8_t *state /* total */,
                  int32_t *plans_out, int32_t *n_plans_out) {
    extern __shared__ __align__(16) unsigned char msm[];   // fast path: keys | rows | customers (4 x u16) [fast_cap each] | owner[n] | state[fast_cap]
    __shared__ int s_m, s_live;
    __shared__ unsigned long long tile[1024];
    __shared__ int s_scan[1024];
    const int tid = threadIdx.x;
    const int slot_rows = cap + headed;
    const int total = n_slots * cap;
    auto row_ptr = [&](int ridx) { return plans + size_t(ridx) * TD_POOL_REC_W; };   // ridx: row index in the padded layout
    // Compaction.  Up to kMergeSlots slots: slot-major order (offsets = prefix sums of the counts), so that every slot's
    // rows stay a contiguous run -- the producer (pool_emit) writes them in ascending (cost, rank) order and the merge
    // below then needs no sort, only a rank by binary searches.  More slots: arrival order, sorted afterwards.
    __shared__ int s_off[kMergeSlots + 1];
    __shared__ int s_unsorted, s_bad;
    const bool by_slot = n_slots <= kMergeSlots;
    auto count_of = [&](int slot) { return counts ? counts[slot] : (headed ? plans[size_t(slot) * slot_rows * TD_POOL_REC_W] : cap); };
    if (tid == 0) { s_m = 0; s_unsorted = 0; s_bad = 0; }
    if (by_slot && tid < 32) {   // one warp: exclusive scan of the (clamped) counts
        int run = 0;
        for (int b0 = 0; b0 < n_slots; b0 += 32) {
            const int slot = b0 + tid;
            int c = slot < n_slots ? count_of(slot) : 0;
            c = c < 0 ? 0 : (c > cap ? cap : c);
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (tid >= o) incl += v; }
            if (slot < n_slots) s_off[slot] = run + incl - c;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (tid == 0) s_off[n_slots] = run;
    }
    __syncthreads();
    for (int base = 0; base < total; base += blockDim.x) {
        const int i = base + tid;
        bool ok = false;
        long long pos = 0;
        int ridx = 0, slot = 0, r = 0;
        if (i < total) {
            slot = i / cap; r = i % cap;
            const int cnt = count_of(slot);
            ok = r < cnt;
            pos = (long long)(slot_shard ? slot_shard[slot] : slot) * cap + r;
            ridx = slot * slot_rows + headed + r;
        }
        if (ok) {
            const int c = by_slot ? s_off[slot] + r : atomicAdd(&s_m, 1);
            const unsigned long long costpart = K == TD_POOL_MAX_IN_POOL ? (unsigned long long)(unsigned)row_ptr(ridx)[8] : 0ull;
            ckey[c] = (costpart << 32) | (unsigned long long)pos;   // pos < 2^32 (total <= 2^24 rows)
            crow[c] = ridx;
            bool bad = false;
            for (int q = 0; q < K; ++q) bad = bad || unsigned(row_ptr(ridx)[q]) >= unsigned(n);
            if (bad) s_bad = 1;
            // a slot whose rows do not ascend (a caller's own rows) sends the merge through the sort
            if (by_slot && K == TD_POOL_MAX_IN_POOL && r > 0 && (unsigned)row_ptr(ridx - 1)[8] > (unsigned)costpart) s_unsorted = 1;
        }
    }
    __syncthreads();
    if (s_bad) { if (tid == 0) *n_plans_out = -1; return; }   // uniform: read after the barrier
    if (by_slot && tid == 0) s_m = s_off[n_slots];
    __syncthreads();
    const int m = s_m;
    if (m == 0) { if (tid == 0) *n_plans_out = 0; return; }

    if (m <= fast_cap) {   // fast_cap: power of two, the arrays below hold that many rows (0: no fast path)
        unsigned long long *keys = reinterpret_cast<unsigned long long *>(msm);
        int *rows = reinterpret_cast<int *>(msm + size_t(fast_cap) * 8);
        ushort4 *cu = reinterpret_cast<ushort4 *>(rows + fast_cap);   // customers of the row at sorted position i (n <= 16384)
        int *own = reinterpret_cast<int *>(cu + fast_cap);
        uint8_t *st = reinterpret_cast<uint8_t *>(own + n);
        int P = 1;
        while (P < m) P <<= 1;
        if (by_slot && !s_unsorted) {
            // every slot is an ascending run: sorted position = own index in the run + the number of smaller keys in every
            // other run (binary searches in shared memory; keys are unique) -- no sort, two block barriers
            unsigned long long *ukeys = reinterpret_cast<unsigned long long *>(cu);   // cu[] is filled after this step
            for (int i = tid; i < m; i += blockDim.x) ukeys[i] = ckey[i];
            __syncthreads();
            for (int i = tid; i < m; i += blockDim.x) {
                const unsigned long long key = ukeys[i];
                int rank = 0;
                for (int sl = 0; sl < n_slots; ++sl) {
                    int lo = s_off[sl], hi = s_off[sl + 1];
                    if (i >= lo && i < hi) { rank += i - lo; continue; }
                    const int first = lo;
                    while (lo < hi) {   // lower bound of key in ukeys[lo, hi)
                        const int mid = (lo + hi) >> 1;
                        if (ukeys[mid] < key) lo = mid + 1; else hi = mid;
                    }
                    rank += lo - first;
                }
                keys[rank] = key;
                rows[rank] = crow[i];
            }
            __syncthreads();
        } else {
        for (int i = tid; i < P; i += blockDim.x) {
            keys[i] = i < m ? ckey[i] : ~0ull;
            rows[i] = i < m ? crow[i] : -1;
        }
        __syncthreads();
        for (int k = 2; k <= P; k <<= 1)                       // bitonic sort, ascending; keys are unique
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = tid; i < P; i += blockDim.x) {
                    const int l = i ^ j;
                    if (l > i) {
                        const unsigned long long a = keys[i], b2 = keys[l];
                        const bool up = (i & k) == 0;
                        if ((a > b2) == up) {
                            keys[i] = b2; keys[l] = a;
                            const int t = rows[i]; rows[i] = rows[l]; rows[l] = t;
                        }
                    }
                }
                __syncthreads();
            }
        }
        for (int i = tid; i < m; i += blockDim.x) {
            st[i] = 0;
            const int32_t *row = row_ptr(rows[i]);
            ushort4 c4 = make_ushort4(0, 0, 0, 0);
            c4.x = (unsigned short)row[0]; c4.y = (unsigned short)row[1];
            if (K > 2) c4.z = (unsigned short)row[2];
            if (K > 3) c4.w = (unsigned short)row[3];
            cu[i] = c4;
        }
        auto cust_of = [&](const ushort4 c4, int q) -> int { return q == 0 ? c4.x : q == 1 ? c4.y : q == 2 ? c4.z : c4.w; };
        for (;;) {   // dominance rounds: sorted position = scan rank
            for (int c = tid; c < n; c += blockDim.x) own[c] = INT_MAX;
            if (tid == 0) s_live = 0;
            __syncthreads();
            for (int i = tid; i < m; i += blockDim.x)
                if (st[i] == 0) {
                    s_live = 1;
                    const ushort4 c4 = cu[i];
                    for (int q = 0; q < K; ++q) atomicMin(&own[cust_of(c4, q)], i);
                }
            __syncthreads();
            if (!s_live) break;
            for (int i = tid; i < m; i += blockDim.x)
                if (st[i] == 0) {
                    const ushort4 c4 = cu[i];
                    bool dom = true;
                    for (int q = 0; q < K; ++q) dom = dom && own[cust_of(c4, q)] == i;
                    if (dom) st[i] = 1;
                }
            __syncthreads();
            for (int i = tid; i < m; i += blockDim.x)   // customers of kept plans are taken
                if (st[i] == 1) {
                    const ushort4 c4 = cu[i];
                    for (int q = 0; q < K; ++q) own[cust_of(c4, q)] = -1;
                }
            __syncthreads();
            for (int i = tid; i < m; i += blockDim.x)
                if (st[i] == 0) {
                    const ushort4 c4 = cu[i];
                    bool hit = false;
                    for (int q = 0; q < K; ++q) hit = hit || own[cust_of(c4, q)] == -1;
                    if (hit) st[i] = 2;
                }
            __syncthreads();
        }
        // output position of a kept row = number of kept rows before it in the sorted order (block scan over chunks)
        const int per = (m + blockDim.x - 1) / blockDim.x;
        const int lo = min(tid * per, m), hi = min(lo + per, m);
        int cnt = 0;
        for (int i = lo; i < hi; ++i) cnt += st[i] == 1;
        s_scan[tid] = cnt;
        __syncthreads();
        if (tid < 32) {   // exclusive scan of the 1024 chunk counts: 32 per lane, warp scan of the lane sums
            int run = 0;
            for (int k2 = 0; k2 < 32; ++k2) run += s_scan[tid * 32 + k2];
            int incl = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (tid >= o) incl += v; }
            int acc = incl - run;
            for (int k2 = 0; k2 < 32; ++k2) { const int v = s_scan[tid * 32 + k2]; s_scan[tid * 32 + k2] = acc; acc += v; }
            if (tid == 31) *n_plans_out = incl;
        }
        __syncthreads();
        int pos = s_scan[tid];
        for (int i = lo; i < hi; ++i)
            if (st[i] == 1) {
                const int32_t *row = row_ptr(rows[i]);
                for (int t = 0; t < TD_POOL_REC_W; ++t) plans_out[size_t(pos) * TD_POOL_REC_W + t] = row[t];
                ++pos;
            }
        return;
    }

    // ---- general path: rank = number of smaller keys (keys are unique) -----------------------------------------------
    for (int base = 0; base < m; base += blockDim.x) {
        const int me = base + tid;
        const unsigned long long mine = me < m ? ckey[me] : ~0ull;
        int rank = 0;
        for (int t0 = 0; t0 < m; t0 += 1024) {
            __syncthreads();
            tile[tid] = (t0 + tid < m) ? ckey[t0 + tid] : ~0ull;
            __syncthreads();
            const int lim = (m - t0) < 1024 ? (m - t0) : 1024;
            for (int t = 0; t < lim; ++t) rank += tile[t] < mine;
        }
        if (me < m) { order_key[me] = rank; state[me] = 0; }
    }
    __syncthreads();
    for (;;) {
        for (int c = tid; c < n; c += blockDim.x) owner[c] = INT_MAX;
        if (tid == 0) s_live = 0;
        __syncthreads();
        for (int i = tid; i < m; i += blockDim.x)
            if (state[i] == 0) {
                s_live = 1;
                const int32_t *row = row_ptr(crow[i]);
                for (int q = 0; q < K; ++q) atomicMin(&owner[row[q]], order_key[i]);
            }
        __syncthreads();
        if (!s_live) break;
        for (int i = tid; i < m; i += blockDim.x)
            if (state[i] == 0) {
                const int32_t *row = row_ptr(crow[i]);
                bool dom = true;
                for (int q = 0; q < K; ++q) dom = dom && owner[row[q]] == order_key[i];
                if (dom) state[i] = 1;
            }
        __syncthreads();
        // customers of kept plans are taken: every other live plan touching them dies
        for (int i = tid; i < m; i += blockDim.x)
            if (state[i] == 1) {
                const int32_t *row = row_ptr(crow[i]);
                for (int q = 0; q < K; ++q) owner[row[q]] = -1;
            }
        __syncthreads();
        for (int i = tid; i < m; i += blockDim.x)
            if (state[i] == 0) {
                const int32_t *row = row_ptr(crow[i]);
                bool hit = false;
                for (int q = 0; q < K; ++q) hit = hit || owner[row[q]] == -1;
                if (hit) state[i] = 2;
            }
        __syncthreads();
    }
    // kept rows in scan order: position = number of kept rows with a smaller scan rank
    if (tid == 0) s_m = 0;
    __syncthreads();
    for (int i = tid; i < m; i += blockDim.x)
        if (state[i] == 1) {
            int pos = 0;
            for (int j = 0; j < m; ++j) pos += (state[j] == 1 && order_key[j] < order_key[i]);
            const int32_t *row = row_ptr(crow[i]);
            for (int t = 0; t < TD_POOL_REC_W; ++t) plans_out[size_t(pos) * TD_POOL_REC_W + t] = row[t];
            atomicAdd(&s_m, 1);
        }
    __syncthreads();
    if (tid == 0) *n_plans_out = s_m;
}

// ---- 2-passenger pool of the Simulator (Simulator.java:681-758; pool.c:64-131) -----------------------
// Every ordered pair (A,B), A != B, is a candidate: A is picked up first, then B; cost1 = B dropped last,
// cost2 = A dropped last; the cheaper one is the pair's plan (ties -> A ends, Simulator.java:711-718).
// The Simulator initialises plan1 = plan2 = true (:691), so its loss tests are dead and EVERY pair is kept
// (SURVEY.md section 4 trap 6, the golden log was produced that way); accept_all = 0 applies the tests as
// written (:701-707, the pool.c behaviour).  Selection = stable sort by cost + greedy disjoint scan
// (:727-739) = the same dominance rounds with rank = A * n + B (TimSort is stable, candidates are A-major).
__global__ void __launch_bounds__(256)
pool_pairs_enum_kernel(const int32_t *__restrict__ from, const int32_t *__restrict__ to, int n,
                       const int32_t *__restrict__ dist, int S, int accept_all, double max_loss, PoolRec *recs,
                       PoolCtrl *ctrl) {
    __shared__ unsigned s_hist[kBuckets];
    for (int b = threadIdx.x; b < kBuckets; b += blockDim.x) s_hist[b] = 0;
    __syncthreads();
    const long long total = (long long)n * n;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int A = int(idx / n), B = int(idx - (long long)A * n);
        PoolRec r; r.rank = 0; r.cost = -1; r.pad = 0;
        const int fa = from[A], ta = to[A], fb = from[B], tb = to[B];
        if (A != B && fa >= 0 && fb >= 0) {                       // id == -1 rows are skipped (:688)
            const int dab = dist[size_t(fa) * S + fb];
            const int cost1 = dab + dist[size_t(fb) * S + ta] + dist[size_t(ta) * S + tb];
            const int cost2 = dab + dist[size_t(fb) * S + tb] + dist[size_t(tb) * S + ta];
            bool ok = accept_all != 0;
            if (!ok) {
                const double dB = double(dist[size_t(fb) * S + tb]), dA = double(dist[size_t(fa) * S + ta]);
                const bool plan1 = double(dist[size_t(fb) * S + ta] + dist[size_t(ta) * S + tb]) < __dmul_rn(dB, max_loss) &&
                                   double(dab + dist[size_t(fb) * S + ta]) < __dmul_rn(dA, max_loss);
                const bool plan2 = double(cost2) < __dmul_rn(dA, max_loss);
                ok = plan1 || plan2;
            }
            if (ok) {
                const int plan = cost1 < cost2 ? 1 : 0;             // CLNT_B_ENDS = 1, CLNT_A_ENDS = 0
                r.cost = cost1 < cost2 ? cost1 : cost2;
                r.rank = make_rank(A, B, 0, 0, plan);
                atomicAdd(&s_hist[r.cost < kBuckets ? r.cost : kBuckets - 1], 1u);
            }
        }
        recs[idx] = r;                                              // dense layout, holes have cost -1
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kBuckets; b += blockDim.x)
        if (s_hist[b]) atomicAdd(&ctrl->hist[0][b], (unsigned long long)s_hist[b]);
    if (blockIdx.x == 0 && threadIdx.x == 0) ctrl->n_records = unsigned(total);
}

// kept pairs in (cost, A*n+B) order -> rows [custA, custB, plan, cost]
__global__ void __launch_bounds__(1024)
pool_pairs_emit_kernel(const PoolRec *__restrict__ kept, const PoolCtrl *ctrl, int32_t *pairs_out, int32_t cap,
                       int32_t *n_pairs_out) {
    const int m = int(ctrl->n_kept[0]);
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const PoolRec me = kept[i];
        int rank = 0;
        for (int j = 0; j < m; ++j) {
            const PoolRec o = kept[j];
            rank += (o.cost < me.cost) || (o.cost == me.cost && o.rank < me.rank);
        }
        if (rank < cap) {
            int p[4], plan;
            split_rank(me.rank, p, plan);
            int32_t *row = pairs_out + size_t(rank) * 4;
            row[0] = p[0]; row[1] = p[1]; row[2] = plan; row[3] = me.cost;
        }
    }
    if (threadIdx.x == 0) *n_pairs_out = m;
}

struct PoolWorkspace {
    int4 *cust, *cust_s; int32_t *list, *slack, *cnt, *dclose, *dist_s; unsigned int *item_off; PoolRec *recs[2]; PoolRec *act[2]; PoolRec *kept;
    unsigned long long *best_hi[2]; unsigned int *best_lo[2]; uint8_t *alive; PoolCtrl *ctrl; size_t bytes;
};

// act[] is cut into one fragment per CTA of pool_select (at most kSelMaxGrid CTAs): a CTA filters whole chunks of
// kSelThreads * 4 records, so its fragment holds its share of the list plus one chunk
constexpr int kSelMaxGrid = 640;
constexpr size_t kActSlack = size_t(kSelMaxGrid) * (kSelThreads * 4 + 1);
static unsigned sel_frag_cap(int64_t max_records, int grid) { return unsigned(max_records / grid) + kSelThreads * 4 + 1; }

static PoolWorkspace carve_pool(void *ws, int n, int S, int n_slots, int64_t max_records) {
    Carver c(ws);
    PoolWorkspace w;
    const size_t nn = n > 0 ? n : 1;
    const size_t ns = nn * size_t(n_slots > 0 ? n_slots : 1);
    w.ctrl = c.take<PoolCtrl>(1);
    w.cust = c.take<int4>(nn);
    w.list = c.take<int32_t>(size_t(S) * nn);
    w.slack = c.take<int32_t>(size_t(S) * nn);
    w.cnt = c.take<int32_t>(size_t(S) * kTbl);
    w.dclose = c.take<int32_t>(S <= kPfMaxStands ? size_t(S) * S + 4 : 1);   // + 4: bulk copies move whole 16-byte units
    w.dist_s = c.take<int32_t>(S <= kPfMaxStands ? size_t(S) * S + 4 : 1);
    w.cust_s = c.take<int4>(nn);
    w.item_off = c.take<unsigned int>(nn + 2);
    w.recs[0] = c.take<PoolRec>(size_t(max_records));
    w.recs[1] = c.take<PoolRec>(size_t(max_records));
    w.act[0] = c.take<PoolRec>(size_t(max_records) + kActSlack);   // fragmented over the CTAs of pool_select
    w.act[1] = c.take<PoolRec>(size_t(max_records) + kActSlack);
    w.kept = c.take<PoolRec>(size_t(n_slots > 0 ? n_slots : 1) * (nn / 2 + 1));
    w.best_hi[0] = c.take<unsigned long long>(ns);
    w.best_hi[1] = c.take<unsigned long long>(ns);
    w.best_lo[0] = c.take<unsigned int>(ns);
    w.best_lo[1] = c.take<unsigned int>(ns);
    w.alive = c.take<uint8_t>(ns);
    w.bytes = c.used();
    return w;
}

// chunked reservation can strand up to one chunk per resident warp
static int64_t record_slack() { return int64_t(kChunk) * 148 * 64; }

#define TDH_RC_LOCAL(expr)      \
    do {                        \
        int _rc = (expr);       \
        if (_rc != TD_OK) return _rc; \
    } while (0)

template <int K>
static int launch_enum(EnumArgs a, int sms, bool closure, cudaStream_t st) {
    const size_t dist_b = (size_t(a.S) * a.S * 4 + 15) & ~size_t(15);
    const size_t cust_b = size_t(a.n) * 16;
    const bool ds = dist_b <= 64 * 1024;
    const bool pf = K == 4 && ds && closure;          // the closure table is staged next to the distance table
    const bool cs = cust_b <= (pf && dist_b > 32 * 1024 ? 48 * 1024 : 96 * 1024);
    const size_t tables = (ds ? dist_b : 0) + (pf ? dist_b : 0) + (cs ? ((cust_b + 15) & ~size_t(15)) : 0);
    const int n_lead = a.stop - a.start;
    a.ioff_bytes = unsigned(((size_t(n_lead <= kIoffSmem ? n_lead : 0) + 1) * 4 + 15) & ~size_t(15));   // staged only when they fit
#define TD_ENUM_LAUNCH(DS, CS, PF, THR, FORCE)                                                                           \
    do {                                                                                                                 \
        auto kern = pool_enum_kernel<K, DS, CS, PF, THR>;                                                                \
        const size_t smem = tables + a.ioff_bytes + size_t(THR / 32) * kEnumWarpBytes;                                   \
        TD_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(224 * 1024)));           \
        TD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THR, smem));                            \
        if (per_sm < 1) break;                                          /* does not fit: the caller tries the next   */ \
        if (!(FORCE) && THR == kEnumThreads && per_sm == 1 && K == 4 && !getenv("TD_ENUM_NARROW")) break;   /* wide CTA */ \
        kern<<<sms * (per_sm > 4 ? 4 : per_sm), THR, smem, st>>>(a);   /* resident CTAs only: a CTA that starts     */ \
        launched = true;                                                /* late finds the queue empty                */ \
    } while (0)
#define TD_ENUM_CASE(DS, CS, PF)                                                                                         \
    do {                                                                                                                 \
        int per_sm = 0;                                                                                                  \
        bool launched = false;                                                                                           \
        TD_ENUM_LAUNCH(DS, CS, PF, kEnumThreads, false);                                                                 \
        if (!launched) TD_ENUM_LAUNCH(DS, CS, PF, (K == 4 ? kEnumThreadsWide : kEnumThreads), false);                    \
        if (!launched) TD_ENUM_LAUNCH(DS, CS, PF, kEnumThreads, true);   /* big tables: the wide CTA's stages do not fit */ \
        if (!launched) return TD_ERR_CUDA;                                                                               \
    } while (0)
    if (pf) { if (cs) TD_ENUM_CASE(true, true, (K == 4)); else TD_ENUM_CASE(true, false, (K == 4)); }
    else if (ds && cs) TD_ENUM_CASE(true, true, false);
    else if (ds) TD_ENUM_CASE(true, false, false);
    else if (cs) TD_ENUM_CASE(false, true, false);
    else TD_ENUM_CASE(false, false, false);
#undef TD_ENUM_LAUNCH
#undef TD_ENUM_CASE
    TD_LAUNCH_CHECK();
    return TD_OK;
}

}  // namespace td

extern "C" size_t td_pool_shards_workspace_bytes(int n, int n_stands, int pool_size, int shard_count, int64_t max_feasible) {
    (void)pool_size;
    if (n < 0 || n_stands < 0 || max_feasible < 0 || shard_count < 1) return 0;
    return td::carve_pool(nullptr, n, n_stands, shard_count, max_feasible + td::record_slack()).bytes;
}

extern "C" size_t td_pool_workspace_bytes(int n, int n_stands, int pool_size, int64_t max_feasible) {
    return td_pool_shards_workspace_bytes(n, n_stands, pool_size, 1, max_feasible);
}

static int pool_find_shards_impl(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                                 int shard_begin, int shard_count, int n_shards, int32_t *plans_out, int32_t cap,
                                 int32_t *counts_out, td_pool_stats *stats, void *workspace, size_t workspace_bytes,
                                 int64_t max_feasible, void *stream, int headed);

extern "C" int td_pool_find_shards(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                                   int shard_begin, int shard_count, int n_shards, int32_t *plans_out, int32_t cap,
                                   int32_t *counts_out, td_pool_stats *stats, void *workspace, size_t workspace_bytes,
                                   int64_t max_feasible, void *stream) {
    if (!counts_out) return TD_ERR_INVALID;
    return pool_find_shards_impl(demand, n, dist, n_stands, pool_size, shard_begin, shard_count, n_shards, plans_out, cap, counts_out,
                                 stats, workspace, workspace_bytes, max_feasible, stream, 0);
}

extern "C" int td_pool_find_shards_headed(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                                          int shard_begin, int shard_count, int n_shards, int32_t *blocks_out, int32_t cap,
                                          void *workspace, size_t workspace_bytes, int64_t max_feasible, void *stream) {
    if (!blocks_out) return TD_ERR_INVALID;
    return pool_find_shards_impl(demand, n, dist, n_stands, pool_size, shard_begin, shard_count, n_shards, blocks_out, cap, nullptr,
                                 nullptr, workspace, workspace_bytes, max_feasible, stream, 1);
}

static int pool_find_shards_impl(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                                 int shard_begin, int shard_count, int n_shards, int32_t *plans_out, int32_t cap,
                                 int32_t *counts_out, td_pool_stats *stats, void *workspace, size_t workspace_bytes,
                                 int64_t max_feasible, void *stream, int headed) {
    using namespace td;
    if (pool_size < 2 || pool_size > TD_POOL_MAX_IN_POOL || n < 0 || n > TD_POOL_MAX_CUSTOMERS || n_stands <= 0 ||
        n_shards < 1 || shard_begin < 0 || shard_count < 1 || shard_count > kMaxSlots || shard_begin + shard_count > n_shards ||
        cap < 0 || (!counts_out && !headed) || max_feasible < 0)
        return TD_ERR_INVALID;
    if (n_stands > 32767) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (stats) memset(stats, 0, sizeof(*stats) * shard_count);
    const int step = n / n_shards + 1;                                        // pool_n.c:226
    const int start = step * shard_begin;                                     // pool_n.c:227
    const long long stop64 = (long long)step * (shard_begin + shard_count);
    const int stop = stop64 > n ? n : int(stop64);                            // pool_n.c:228
    if (n == 0 || start >= n) {
        if (counts_out) TD_CUDA_TRY(cudaMemsetAsync(counts_out, 0, sizeof(int32_t) * shard_count, st));
        if (headed && plans_out)   // empty blocks: header count 0
            TD_CUDA_TRY(cudaMemsetAsync(plans_out, 0, sizeof(int32_t) * size_t(shard_count) * (cap + 1) * TD_POOL_REC_W, st));
        if (stats) TD_CUDA_TRY(cudaStreamSynchronize(st));
        return TD_OK;
    }
    if (!demand || !dist || !workspace || (cap > 0 && !plans_out)) return TD_ERR_INVALID;
    if (workspace_bytes < td_pool_shards_workspace_bytes(n, n_stands, pool_size, shard_count, max_feasible)) return TD_ERR_WORKSPACE;
    const int64_t rec_cap64 = max_feasible + record_slack();
    if (rec_cap64 > 0xfffffff0ll) return TD_ERR_INVALID;
    PoolWorkspace w = carve_pool(workspace, n, n_stands, shard_count, rec_cap64);
    const int keep_cap = n / 2 + 1;

    TD_CUDA_TRY(cudaMemsetAsync(w.ctrl, 0, sizeof(PoolCtrl), st));
    const int sh = pool_size == 4 ? kSh4 : 0;                                  // fixed point of the enumeration's evaluation
    const bool closure = pool_size == 4 && n_stands <= kPfMaxStands;
    {
        const long long cells = (long long)n_stands * n_stands;
        const long long want = (cells + 256 * 16 - 1) / (256 * 16);
        const int check_blocks = int(want < 1 ? 1 : (want > 4LL * device_sm_count() ? 4LL * device_sm_count() : want));
        const size_t cl_smem = closure ? size_t(n_stands) * n_stands * 4 : 0;
        TD_CUDA_TRY(cudaFuncSetAttribute(pool_prepare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(64 * 1024)));
        pool_prepare_kernel<<<(closure ? 1 : 0) + check_blocks + (n + 255) / 256, 256, cl_smem, st>>>(
            demand, n, dist, n_stands, w.cust, w.cust_s, sh, w.ctrl, n_stands <= kPfMaxStands ? w.dist_s : nullptr, w.dclose,
            closure ? 1 : 0, check_blocks);
        TD_LAUNCH_CHECK();
    }
    pool_build_lists_kernel<<<n_stands, 256, 0, st>>>(w.cust, n, dist, n_stands, w.list, w.slack, w.cnt, start, stop, pool_size,
                                                      w.item_off, w.ctrl);
    TD_LAUNCH_CHECK();

    const int sms = device_sm_count();
    int sel_per_sm = 0;
    TD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sel_per_sm, pool_select_kernel, kSelThreads, 0));
    if (sel_per_sm < 1) return TD_ERR_CUDA;
    sel_per_sm = sel_per_sm > 4 ? 4 : sel_per_sm;
    if (const char *e = getenv("TD_SEL_PER_SM")) { const int v = atoi(e); if (v >= 1 && v <= sel_per_sm) sel_per_sm = v; }
    while (sel_per_sm > 1 && sms * sel_per_sm > kSelMaxGrid) --sel_per_sm;
    if (sms * sel_per_sm < shard_count || sms * sel_per_sm > kSelMaxGrid) return TD_ERR_INVALID;

    // the per-pass part of the control block (from pass_begin_marker to the per-call tail that starts at max_wait)
    const size_t pass_off = offsetof(PoolCtrl, pass_begin_marker);
    auto reset_pass = [&]() -> int {
        TD_CUDA_TRY(cudaMemsetAsync(reinterpret_cast<char *>(w.ctrl) + pass_off, 0, offsetof(PoolCtrl, max_wait) - pass_off, st));
        return TD_OK;
    };
    auto run_enum = [&](int cost_lo, int cost_hi, bool use_alive, bool count_stats, int stride) -> int {
        EnumArgs ea;
        ea.cust = w.cust; ea.cust_s = w.cust_s; ea.dist = dist; ea.dist_s = w.dist_s; ea.dclose = w.dclose; ea.list = w.list; ea.slack = w.slack; ea.cnt = w.cnt; ea.item_off = w.item_off;
        ea.recs = w.recs[0]; ea.ctrl = w.ctrl; ea.n = n; ea.S = n_stands; ea.start = start; ea.stop = stop;
        ea.cap = unsigned(rec_cap64); ea.step = step; ea.shard_begin = shard_begin; ea.cb = key_cb(n);
        ea.cost_lo = cost_lo; ea.cost_hi = cost_hi; ea.alive = use_alive ? w.alive : nullptr;
        ea.count_stats = count_stats ? 1 : 0; ea.item_stride = stride;
        ProfScope prof(TD_PROF_POOL_ENUM, st);
        return pool_size == 4 ? launch_enum<4>(ea, sms, closure, st) : pool_size == 3 ? launch_enum<3>(ea, sms, false, st)
                                                                                        : launch_enum<2>(ea, sms, false, st);
    };
    auto run_select = [&](bool first, int window_hi) -> int {
        SelArgs sa;
        sa.list[0] = w.recs[0]; sa.list[1] = w.recs[1]; sa.act[0] = w.act[0]; sa.act[1] = w.act[1]; sa.ctrl = w.ctrl;
        sa.best_hi[0] = w.best_hi[0]; sa.best_hi[1] = w.best_hi[1]; sa.best_lo[0] = w.best_lo[0]; sa.best_lo[1] = w.best_lo[1];
        sa.alive = w.alive; sa.kept = w.kept; sa.n = n; sa.K = pool_size;
        sa.n_slots = shard_count; sa.step = step; sa.shard_begin = shard_begin; sa.keep_cap = keep_cap;
        sa.step_inv = step > 1 ? unsigned(((1ull << 32) + unsigned(step) - 1) / unsigned(step)) : 0u;
        sa.first_pass = first ? 1 : 0;
        sa.cost_hi = window_hi;
        sa.frag_cap = sel_frag_cap(rec_cap64, sms * sel_per_sm);
        sa.band0 = kBand0; sa.band_growth = 4;
        if (const char *e = getenv("TD_SEL_BAND0")) sa.band0 = unsigned(atoi(e));
        if (const char *e = getenv("TD_SEL_GROWTH")) sa.band_growth = unsigned(atoi(e));
        void *sargs[] = {(void *)&sa};
        {
            ProfScope prof(TD_PROF_POOL_SELECT, st);
            TD_CUDA_TRY(cudaLaunchCooperativeKernel((void *)pool_select_kernel, dim3(sms * sel_per_sm), dim3(kSelThreads), sargs, 0, st));
        }
        count_launch();
        return TD_OK;
    };

    static thread_local PoolCtrl h;
    int passes = 0;
    if (!stats) {
        // asynchronous single pass: no host round trip; an overflow is reported through counts_out[s] = -1
        int rc = run_enum(INT_MIN, INT_MAX, false, true, 1);
        if (rc != TD_OK) return rc;
        rc = run_select(true, INT_MAX);
        if (rc != TD_OK) return rc;
        pool_emit_kernel<<<shard_count, 1024, 0, st>>>(w.kept, w.ctrl, pool_size, keep_cap, plans_out, cap, counts_out, headed);
        TD_LAUNCH_CHECK();
        return TD_OK;
    }

    // synchronous path: cost windows.  Window 0 tries to take everything; when the record list would overflow,
    // the histogram (which keeps counting after an overflow) tells where to cut, and later windows only
    // enumerate customers that are still free.
    unsigned n_items_host = 0;
    TD_CUDA_TRY(cudaMemcpyAsync(&n_items_host, &w.ctrl->n_items, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    TD_CUDA_TRY(cudaStreamSynchronize(st));
    const double budget = 0.9 * double(max_feasible);
    auto cut_from_hist = [&](int lo_bucket, double scale) -> int {   // largest cost bound whose cumulative count fits
        double cum = 0;
        int hi = lo_bucket;
        for (int bkt = lo_bucket; bkt < kBuckets - 1; ++bkt) {
            double c = 0;
            for (int sl = 0; sl < shard_count; ++sl) c += h.hist[sl][bkt];
            if (cum + c * scale > budget) break;
            cum += c * scale;
            hi = bkt + 1;
        }
        return hi;
    };
    int cost_lo = INT_MIN;
    bool first_select = true, stats_counted = false;
    for (int guard = 0; guard < 4 * kBuckets; ++guard) {
        int cost_hi = INT_MAX;
        const bool use_alive = !first_select;
        // big inputs: a 1/64 sampling pass estimates the histogram so that the full pass does not overflow
        const bool sample = (long long)n_items_host > (1ll << 18);
        if (sample) {
            TDH_RC_LOCAL(reset_pass());
            int rc = run_enum(cost_lo, INT_MAX, use_alive, false, 64);
            if (rc != TD_OK) return rc;
            ++passes;
            TD_CUDA_TRY(cudaMemcpyAsync(&h, w.ctrl, sizeof h, cudaMemcpyDeviceToHost, st));
            TD_CUDA_TRY(cudaStreamSynchronize(st));
            if (h.bad_input) return TD_ERR_INVALID;   // a stand distance above 2^22 (K = 4 fixed-point evaluation)
            double tot = 0;
            for (int sl = 0; sl < shard_count; ++sl) for (int bkt = 0; bkt < kBuckets; ++bkt) tot += h.hist[sl][bkt];
            if (tot * 64.0 * 1.3 > budget) {
                const int lo_b = cost_lo == INT_MIN ? 0 : (cost_lo < kBuckets ? cost_lo : kBuckets - 1);
                const int cut = cut_from_hist(lo_b, 64.0 * 1.3);
                if (cut > lo_b) cost_hi = cut;   // else: a single cost level is too big for the estimate, try anyway
            }
        }
        for (;;) {   // full pass, shrinking the window if it still overflows
            TDH_RC_LOCAL(reset_pass());
            int rc = run_enum(cost_lo, cost_hi, use_alive, !stats_counted, 1);
            if (rc != TD_OK) return rc;
            ++passes;
            stats_counted = true;
            TD_CUDA_TRY(cudaMemcpyAsync(&h, w.ctrl, sizeof h, cudaMemcpyDeviceToHost, st));
            TD_CUDA_TRY(cudaStreamSynchronize(st));
            if (h.bad_input) return TD_ERR_INVALID;   // a stand distance above 2^22 (K = 4 fixed-point evaluation)
            if (!h.overflow) break;
            const int lo_b = cost_lo == INT_MIN ? 0 : (cost_lo < kBuckets ? cost_lo : kBuckets - 1);
            const int cut = cut_from_hist(lo_b, 1.0);
            if (cut <= lo_b || (cost_hi != INT_MAX && cut >= cost_hi)) {
                // one cost level alone exceeds the record capacity: the caller has to provide a bigger workspace
                for (int sl = 0; sl < shard_count; ++sl) {
                    stats[sl].evaluated = int64_t(h.evaluated[sl]); stats[sl].feasible = int64_t(h.feasible[sl]);
                    stats[sl].passes = passes;
                }
                return TD_ERR_CAPACITY;
            }
            cost_hi = cut;
        }
        int rc = run_select(first_select, cost_hi);
        if (rc != TD_OK) return rc;
        first_select = false;
        if (cost_hi == INT_MAX) break;
        cost_lo = cost_hi;
    }
    pool_emit_kernel<<<shard_count, 1024, 0, st>>>(w.kept, w.ctrl, pool_size, keep_cap, plans_out, cap, counts_out, headed);
    TD_LAUNCH_CHECK();
    TD_CUDA_TRY(cudaMemcpyAsync(&h, w.ctrl, offsetof(PoolCtrl, pass_begin_marker), cudaMemcpyDeviceToHost, st));
    TD_CUDA_TRY(cudaStreamSynchronize(st));
    bool over_cap = false;
    for (int sl = 0; sl < shard_count; ++sl) {
        stats[sl].evaluated = int64_t(h.evaluated[sl]);
        stats[sl].feasible = int64_t(h.feasible[sl]);
        stats[sl].kept = h.n_kept[sl];
        stats[sl].rounds = int32_t(h.total_rounds);
        stats[sl].passes = passes;
        over_cap = over_cap || int64_t(h.n_kept[sl]) > cap;
    }
    return over_cap ? TD_ERR_CAPACITY : TD_OK;
}

extern "C" size_t td_pool_read_stats_bytes(void) { return offsetof(td::PoolCtrl, rounds) + sizeof(unsigned int); }

extern "C" int td_pool_read_stats(const void *workspace, int shard_count, td_pool_stats *stats, int *overflow_out,
                                  void *stream) {
    using namespace td;
    if (!workspace || shard_count < 1 || shard_count > kMaxSlots || !stats) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    static thread_local PoolCtrl h;
    const PoolCtrl *ctrl = Carver(const_cast<void *>(workspace)).take<PoolCtrl>(1);
    const size_t head = offsetof(PoolCtrl, rounds) + sizeof(unsigned int);
    TD_CUDA_TRY(cudaMemcpyAsync(&h, ctrl, head, cudaMemcpyDeviceToHost, st));
    TD_CUDA_TRY(cudaStreamSynchronize(st));
    for (int s = 0; s < shard_count; ++s) {
        stats[s].evaluated = int64_t(h.evaluated[s]);
        stats[s].feasible = int64_t(h.feasible[s]);
        stats[s].kept = h.n_kept[s];
        stats[s].rounds = int32_t(h.total_rounds);
        stats[s].passes = 1;
    }
    if (overflow_out) *overflow_out = (h.overflow || h.bad_input) ? 1 : 0;   // either way: repeat through the synchronous entry point
    return TD_OK;
}

extern "C" int td_pool_find(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size, int shard,
                            int n_shards, int32_t *plans_out, int32_t cap, int32_t *n_plans_out, td_pool_stats *stats,
                            void *workspace, size_t workspace_bytes, int64_t max_feasible, void *stream) {
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return TD_ERR_INVALID;
    return td_pool_find_shards(demand, n, dist, n_stands, pool_size, shard, 1, n_shards, plans_out, cap, n_plans_out, stats,
                               workspace, workspace_bytes, max_feasible, stream);
}

extern "C" size_t td_pool_pairs_workspace_bytes(int n) {
    if (n < 0) return 0;
    return td::carve_pool(nullptr, n, 1, 1, int64_t(n) * n + 16).bytes;
}

extern "C" int td_pool_pairs(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                             int accept_all, double max_loss, int32_t *pairs_out, int32_t cap, int32_t *n_pairs_out,
                             void *workspace, size_t workspace_bytes, void *stream) {
    using namespace td;
    if (n < 0 || n > TD_POOL_MAX_CUSTOMERS || n_stands <= 0 || cap < 0 || !n_pairs_out) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n < 2) { TD_CUDA_TRY(cudaMemsetAsync(n_pairs_out, 0, sizeof(int32_t), st)); return TD_OK; }
    if (!from || !to || !dist || !workspace || (cap > 0 && !pairs_out)) return TD_ERR_INVALID;
    if (workspace_bytes < td_pool_pairs_workspace_bytes(n)) return TD_ERR_WORKSPACE;
    const int64_t recs = int64_t(n) * n + 16;
    PoolWorkspace w = carve_pool(workspace, n, 1, 1, recs);
    TD_CUDA_TRY(cudaMemsetAsync(w.ctrl, 0, sizeof(PoolCtrl), st));
    const int sms = device_sm_count();
    pool_pairs_enum_kernel<<<sms * 8, 256, 0, st>>>(from, to, n, dist, n_stands, accept_all, max_loss, w.recs[0], w.ctrl);
    TD_LAUNCH_CHECK();
    SelArgs sa;
    sa.list[0] = w.recs[0]; sa.list[1] = w.recs[1]; sa.act[0] = w.act[0]; sa.act[1] = w.act[1]; sa.ctrl = w.ctrl;
    sa.best_hi[0] = w.best_hi[0]; sa.best_hi[1] = w.best_hi[1]; sa.best_lo[0] = w.best_lo[0]; sa.best_lo[1] = w.best_lo[1];
    sa.alive = w.alive; sa.kept = w.kept; sa.n = n; sa.K = 2;
    sa.n_slots = 1; sa.step = n + 1; sa.shard_begin = 0; sa.keep_cap = n / 2 + 1; sa.first_pass = 1; sa.cost_hi = INT_MAX;
    sa.band0 = kBand0; sa.band_growth = 4;
    sa.step_inv = unsigned(((1ull << 32) + unsigned(n + 1) - 1) / unsigned(n + 1));   // n >= 2 here
    int per_sm = 0;
    TD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pool_select_kernel, kSelThreads, 0));
    if (per_sm < 1) return TD_ERR_CUDA;
    per_sm = per_sm > 4 ? 4 : per_sm;
    while (per_sm > 1 && sms * per_sm > kSelMaxGrid) --per_sm;
    if (sms * per_sm > kSelMaxGrid) return TD_ERR_INVALID;
    sa.frag_cap = sel_frag_cap(recs, sms * per_sm);
    void *sargs[] = {(void *)&sa};
    {
        ProfScope prof(TD_PROF_POOL_SELECT, st);
        TD_CUDA_TRY(cudaLaunchCooperativeKernel((void *)pool_select_kernel, dim3(sms * per_sm), dim3(kSelThreads), sargs, 0, st));
    }
    count_launch();
    pool_pairs_emit_kernel<<<1, 1024, 0, st>>>(w.kept, w.ctrl, pairs_out, cap, n_pairs_out);
    TD_LAUNCH_CHECK();
    return TD_OK;
}

namespace td {
struct MergeWs { unsigned long long *ckey; int32_t *crow, *order_key, *owner; uint8_t *state; size_t bytes; };
static MergeWs carve_merge(void *ws, int total, int n) {
    Carver c(ws);
    MergeWs w;
    const size_t t = total > 0 ? total : 1;
    w.ckey = c.take<unsigned long long>(t);
    w.crow = c.take<int32_t>(t);
    w.order_key = c.take<int32_t>(t);
    w.owner = c.take<int32_t>(n > 0 ? n : 1);
    w.state = c.take<uint8_t>(t);
    w.bytes = c.used();
    return w;
}
}  // namespace td

extern "C" size_t td_pool_merge_workspace_bytes(int total_plans, int n) { return td::carve_merge(nullptr, total_plans, n).bytes; }

namespace td {
static int launch_merge(const int32_t *plans, int n_slots, int cap, int headed, const int32_t *counts, const int32_t *slot_shard,
                        int n, int pool_size, int32_t *plans_out, int32_t *n_plans_out, void *workspace, cudaStream_t st) {
    const int total = n_slots * cap;
    MergeWs w = carve_merge(workspace, total, n);
    // fast path capacity: the largest power of two (<= kMergeFast) whose arrays fit beside the per-customer table
    int fast_cap = 0;
    if (n <= TD_POOL_MAX_CUSTOMERS)
        for (fast_cap = kMergeFast; fast_cap >= 256 && size_t(fast_cap) * 21 + size_t(n) * 4 + 16 > 200 * 1024; fast_cap >>= 1) {}
    if (fast_cap < 256) fast_cap = 0;
    const size_t smem = fast_cap ? size_t(fast_cap) * 21 + size_t(n) * 4 + 16 : 0;   // keys + rows + customers + state + owner
    if (smem) TD_CUDA_TRY(cudaFuncSetAttribute(pool_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    pool_merge_kernel<<<1, 1024, smem, st>>>(plans, n_slots, n, pool_size, counts, cap, headed, fast_cap, slot_shard, w.ckey, w.crow,
                                             w.order_key, w.owner, w.state, plans_out, n_plans_out);
    TD_LAUNCH_CHECK();
    return TD_OK;
}
}  // namespace td

extern "C" int td_pool_merge(const int32_t *shard_plans, int total_plans, int n, int pool_size, int32_t *plans_out,
                             int32_t *n_plans_out, void *workspace, size_t workspace_bytes, void *stream) {
    using namespace td;
    if (total_plans < 0 || total_plans > (1 << 24) || n < 0 || pool_size < 2 || pool_size > TD_POOL_MAX_IN_POOL || !n_plans_out) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (total_plans == 0) { TD_CUDA_TRY(cudaMemsetAsync(n_plans_out, 0, sizeof(int32_t), st)); return TD_OK; }
    if (!shard_plans || !plans_out || !workspace) return TD_ERR_INVALID;
    if (workspace_bytes < td_pool_merge_workspace_bytes(total_plans, n)) return TD_ERR_WORKSPACE;
    return launch_merge(shard_plans, 1, total_plans, 0, nullptr, nullptr, n, pool_size, plans_out, n_plans_out, workspace, st);   // one slot, every row valid
}

extern "C" int td_pool_merge_padded(const int32_t *slot_plans, const int32_t *slot_counts, const int32_t *slot_shard,
                                    int n_slots, int cap, int n, int pool_size, int32_t *plans_out, int32_t *n_plans_out,
                                    void *workspace, size_t workspace_bytes, void *stream) {
    using namespace td;
    if (n_slots < 0 || cap < 1 || n < 0 || pool_size < 2 || pool_size > TD_POOL_MAX_IN_POOL || !n_plans_out) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long total64 = (long long)n_slots * cap;
    if (total64 > (1 << 24)) return TD_ERR_INVALID;
    const int total = int(total64);
    if (total == 0) { TD_CUDA_TRY(cudaMemsetAsync(n_plans_out, 0, sizeof(int32_t), st)); return TD_OK; }
    if (!slot_plans || !slot_counts || !plans_out || !workspace) return TD_ERR_INVALID;
    if (workspace_bytes < td_pool_merge_workspace_bytes(total, n)) return TD_ERR_WORKSPACE;
    return launch_merge(slot_plans, n_slots, cap, 0, slot_counts, slot_shard, n, pool_size, plans_out, n_plans_out, workspace, st);
}

extern "C" int td_pool_merge_headed(const int32_t *blocks, const int32_t *slot_shard, int n_slots, int cap, int n, int pool_size,
                                    int32_t *plans_out, int32_t *n_plans_out, void *workspace, size_t workspace_bytes,
                                    void *stream) {
    using namespace td;
    if (n_slots < 0 || cap < 1 || n < 0 || pool_size < 2 || pool_size > TD_POOL_MAX_IN_POOL || !n_plans_out) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long total64 = (long long)n_slots * cap;
    if (total64 > (1 << 24)) return TD_ERR_INVALID;
    const int total = int(total64);
    if (total == 0) { TD_CUDA_TRY(cudaMemsetAsync(n_plans_out, 0, sizeof(int32_t), st)); return TD_OK; }
    if (!blocks || !plans_out || !workspace) return TD_ERR_INVALID;
    if (workspace_bytes < td_pool_merge_workspace_bytes(total, n)) return TD_ERR_WORKSPACE;
    return launch_merge(blocks, n_slots, cap, 1, nullptr, slot_shard, n, pool_size, plans_out, n_plans_out, workspace, st);
}
