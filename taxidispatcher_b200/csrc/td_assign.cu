// td_assign.cu -- K2: exact balanced n x n assignment (minimum-cost perfect matching).
//
// Replaces the model build + cvxopt.glpk.ilp call of the reference (solver.py:11-27,
// python.py:6-25, procedure.py:14-29, split.py:139-155, heuristic.py:7-17,37): minimise
// sum c[i][j] x[n*i+j] with every row sum and column sum equal to 1, x binary.  The dense
// 2n x n^2 constraint matrix of solver.py:15-19 (3.5 GB at n = 600) is never materialised.
//
// Method: primal-dual shortest augmenting paths with integer potentials, organised so that every
// step is a bandwidth-bound sweep over whole cost rows and the number of grid-wide steps depends
// on the number of distinct reduced path lengths, not on n:
//
//   init      v_j = min_i c_ij ; u_i = min_j (c_ij - v_j) ; greedy matching on tight cells
//             (each row proposes a tight free column picked by a row hash, lowest row wins; up to 8 rounds,
//             the losers rescan only their own rows).  From here on  r_ij = c_ij - u_i - v_j >= 0
//             and matched cells have r = 0.
//   phase     multi-source Dijkstra from ALL free rows at once.  Costs are integers, so the
//             priority queue is a sequence of levels (Dial): one level = (a) every row that
//             entered the forest at the previous level relaxes all unsettled columns with one
//             coalesced pass over its cost row, (b) all columns at the new minimum distance
//             are settled together; matched ones pull their mate row into the forest, free ones
//             are sinks.  A phase goes on until 2 % of its trees own a sink (distances stay exact and
//             every settled node takes part in the dual update, so all forest edges become tight);
//             potentials are updated (u_i += D - d_i on forest rows, v_j -= D - dist_j on settled
//             columns) and one augmenting path per tree is flipped (trees are vertex-disjoint
//             because every column has one predecessor and every matched row one parent column).
//   carry     after a deep phase the trees that were not augmented stay: their rows are at distance 0
//             under the new potentials, so the next phase relaxes them in ONE bandwidth-bound sweep
//             at level 0 instead of re-discovering them tight edge by tight edge; the free rows
//             themselves are never rescanned (their column minima are cached, see P0).
//   finish    objective = sum c[i][mate(i)] in int64; optional dense x in the reference layout.
//
// Exactness: potentials stay feasible and matched cells stay tight through every step, so when
// the matching is perfect, complementary slackness gives optimality for any integer costs
// (ties included) -- no epsilon, no scaling, no price wars on the reference's tiny cost ranges.
// The matching itself is deterministic: every choice among ties is a minimum over an order that
// does not depend on scheduling.
//
// Data path (n % 4 == 0): cost rows are staged through a per-warp ring of 3 x 4 KB shared-memory
// stages filled by 16-byte cp.async copies (192 KB per CTA, no registers held by loads in flight),
// the arithmetic is 32-bit whenever 4 max|c| + 2 sum(D) + level < 2^30, and sweep units (256-column
// tile x up to 64 rows) are handed out dynamically.  Other shapes / magnitudes take the register-staged
// 64-bit sweeps (sweep_rows, row_min_reduced).
//
// Everything runs in ONE cooperative persistent kernel (one 512-thread CTA per SM);
// steps are separated by grid.sync().  Algorithmic bytes: 4n bytes per row relaxed; the solver
// reports rows_scanned so achieved GB/s = 4 n rows_scanned / time.
// Diagnostics (environment, read per call): TD_ASSIGN_PROF=1 prints in-kernel timers; TD_ASSIGN_DEEP
// (per-mille of trees per phase), TD_ASSIGN_CARRY, TD_ASSIGN_CARRY_MIN, TD_ASSIGN_WIDE override the defaults.
#include "td_common.cuh"
#include <string.h>
#include <stdio.h>
#include <stdlib.h>

namespace cg = cooperative_groups;

namespace td {

constexpr int kAsgThreads = 512;
constexpr int kRowBits = 24;                       // predecessor row in the low bits of the packed key
constexpr unsigned long long kDistInf = ~0ull;
constexpr long long kRowInf = (1ll << 62);
constexpr int kGreedyRounds = 8;    // upper bound; the loop stops early when a round stops paying

struct AsgCtrl {
    unsigned long long gmin[3];
    unsigned int fcount[2];
    unsigned int nsinks;
    unsigned int free_after_init;
    unsigned int phases, levels, augment, pad;
    unsigned long long rows_scanned;
    unsigned long long stale_cells;   // cells re-read to refresh cached level-0 distances
    long long sfree;                  // sum of the phase lengths D: every still-free row has u = u_init + sfree
    unsigned long long cabs;          // max |c_ij| (init sweep); bounds every potential: |v| <= cabs + sfree, |u| <= 2 cabs + sfree
    unsigned long long narrow_levels; // relaxation sweeps that ran on the 32-bit path
    unsigned int ncarry, pad4;        // rows of surviving trees that open the next phase
    unsigned int ticket[4];           // dynamic unit hand-out of the ring sweeps (slot rotates like gmin)
    unsigned int nstale, ndone;       // ndone: trees (free rows) that own a sink in the current phase
    unsigned long long t_prof[24];     // ns spent by CTA 0 in: scan, sync, settle, sync, phase start, augment (diagnostics)
    long long objective;
    int status;
    int pad2;
};

struct AsgArgs {
    const int32_t *cost; int n;
    long long *u, *v, *drow, *uinit, *vinit;
    unsigned long long *base0;        // per column: min over the FREE rows of (c - u_init - v_init), packed with the row
    int32_t *stale;
    int32_t *vmin; int32_t *mate_r, *mate_c, *root, *claim, *prop, *argcol;
    unsigned long long *distpred; uint8_t *settled;
    int32_t *frontier[2]; long long *fbase[2]; int32_t *carry; long long *cbase; int32_t *sinks;   // fbase = (distance - u) of the frontier row, same slot
    AsgCtrl *ctrl;
    int32_t *col_of_row_out; long long *objective_out; uint8_t *x_out;
    int max_phases;
    int nr;                           // rows 0..nr-1 are real; rows nr..n-1 are constant padding rows (nr == n: balanced)
    int32_t *col_tmp; int32_t *cost_t;   // rect with padding COLUMNS: solved on the transposed matrix
    int greedy_rounds;                // proposal rounds of the greedy initial matching
    int prof;                         // TD_ASSIGN_PROF: in-kernel timers
    int force_wide;                   // diagnostics / tests: always use the 64-bit relaxation
    int carry_min_levels;             // ... only after a phase of at least this many levels
    int carry_forest;                 // keep the trees that were not augmented into the next phase (see P0)
    int deep_permille;                // a phase goes on until this share (per 1000) of its trees has reached a sink
};

// The predecessor row sits in the low bits through a bijective scramble of [0, 2^24): among rows that offer a column
// the same distance the winner is then spread over the trees instead of always being the lowest row index, which
// keeps the trees of a phase balanced (far more of them reach a sink of their own on the reference's degenerate costs).
#ifndef TD_ASG_SCRAMBLE
#define TD_ASG_SCRAMBLE 1
#endif
constexpr unsigned kRowMask = (1u << kRowBits) - 1;
__device__ __forceinline__ unsigned scramble_row(int row) {
    return TD_ASG_SCRAMBLE ? (unsigned(row) * 0x3779b1u) & kRowMask : unsigned(row);
}
__device__ __forceinline__ unsigned long long pack_dp(long long dist, int row) {
    return ((unsigned long long)dist << kRowBits) | scramble_row(row);
}
__device__ __forceinline__ long long dp_dist(unsigned long long k) { return (long long)(k >> kRowBits); }
__device__ __forceinline__ int dp_row(unsigned long long k) {
    const unsigned r = unsigned(k) & kRowMask;
    return int(TD_ASG_SCRAMBLE ? (r * 0x8b2f51u) & kRowMask : r);
}

// One warp relaxes a 256-column tile for a strided group of rows.  rows == nullptr: rows are 0..nrows-1.
// kMode 0: column minima of the raw costs (init);  kMode 1: Dijkstra relaxation.
template <int kMode, bool kVec>
__device__ __forceinline__ void sweep_rows(const AsgArgs &a, const int32_t *rows, int nrows, int gwarp, int nwarps,
                                           int lane, unsigned long long &block_min) {
    const int n = a.n;
    const int tiles = (n + 255) >> 8;
    int groups = nwarps / tiles;
    groups = groups < 1 ? 1 : (groups > nrows ? nrows : groups);
    const int units = tiles * groups;
    int cmx = INT_MIN;   // kMode 0: largest cost seen by this lane
    for (int unit = gwarp; unit < units; unit += nwarps) {
        const int tile = unit % tiles, grp = unit / tiles;
        const int j0 = (tile << 8) + (kVec ? lane * 4 : lane);
        // column slots of this lane: kVec -> {j0..j0+3, j0+128..j0+131}; scalar -> j0 + 32*k
        int col[8];
        bool act[8];
        long long vj[8];
        unsigned long long best[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            col[k] = kVec ? j0 + (k & 3) + ((k >> 2) << 7) : j0 + (k << 5);
            act[k] = col[k] < n;
            if (kMode == 1) {
                act[k] = act[k] && !a.settled[act[k] ? col[k] : 0];
                vj[k] = act[k] ? a.v[col[k]] : 0;
            } else {
                vj[k] = 0;
            }
            best[k] = kDistInf;
        }
        // 4 rows per trip: all index / potential / cost loads are issued before any is consumed
        for (int r = grp; r < nrows; r += 4 * groups) {
            int ri[4];
            long long base[4];
            int4 lo[4], hi[4];
            int cs[4][8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int rr = r + q * groups;
                ri[q] = rr < nrows ? (rows ? rows[rr] : rr) : -1;
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (ri[q] < 0) continue;
                const int32_t *line = a.cost + size_t(ri[q]) * n;
                if (kVec) {
                    lo[q] = (j0 < n) ? ld_stream_int4(reinterpret_cast<const int4 *>(line + j0)) : make_int4(0, 0, 0, 0);
                    hi[q] = (j0 + 128 < n) ? ld_stream_int4(reinterpret_cast<const int4 *>(line + j0 + 128)) : make_int4(0, 0, 0, 0);
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k) cs[q][k] = col[k] < n ? __ldg(line + col[k]) : 0;
                }
                if (kMode == 1) base[q] = a.drow[ri[q]] - a.u[ri[q]];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (ri[q] < 0) continue;
                int c[8];
                if (kVec) {
                    c[0] = lo[q].x; c[1] = lo[q].y; c[2] = lo[q].z; c[3] = lo[q].w;
                    c[4] = hi[q].x; c[5] = hi[q].y; c[6] = hi[q].z; c[7] = hi[q].w;
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k) c[k] = cs[q][k];
                }
                if (kMode == 0) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        // order-preserving bias so that negative costs work too
                        const unsigned long long key = (unsigned long long)(unsigned(c[k]) ^ 0x80000000u);
                        best[k] = key < best[k] ? key : best[k];
                        cmx = c[k] > cmx ? c[k] : cmx;
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const unsigned long long key = pack_dp(base[q] + c[k] - vj[k], ri[q]);
                        best[k] = key < best[k] ? key : best[k];
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (!act[k] || best[k] == kDistInf) continue;
            if (kMode == 0) {
                const int32_t val = int32_t(unsigned(best[k]) ^ 0x80000000u);
                if (val < a.vmin[col[k]]) atomicMin(&a.vmin[col[k]], val);
            } else {
                if (best[k] < a.distpred[col[k]]) atomicMin(&a.distpred[col[k]], best[k]);
                block_min = best[k] < block_min ? best[k] : block_min;
            }
        }
    }
    if (kMode == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const int other = __shfl_xor_sync(0xffffffffu, cmx, o); cmx = other > cmx ? other : cmx; }
        if (lane == 0 && cmx != INT_MIN) atomicMax(&a.ctrl->cabs, (unsigned long long)(cmx < 0 ? -(long long)cmx : (long long)cmx));
    }
}

// ---- cp.async staging --------------------------------------------------------------------------------------------
// A register-staged sweep keeps 4 KB per warp in flight (64 KB per SM at 128 registers per thread), which caps it at
// ~2.5-4 TB/s on B200: the loaded HBM latency is ~2 us.  Here every warp owns a ring of kAsgStages stages of 4 cost-row
// segments (4 x 1 KB) in shared memory, filled with 16-byte cp.async copies that occupy no registers; each lane reads
// back exactly the bytes it copied, so no barrier is needed -- cp.async.wait_group is the only synchronisation.
constexpr int kAsgStages = 3;
constexpr int kAsgStageBytes = 4 * 1024;                                    // 4 rows x 256 columns x int32
constexpr int kAsgRingBytes = (kAsgThreads / 32) * kAsgStages * kAsgStageBytes;   // 192 KB per CTA

__device__ __forceinline__ void cp_async16(unsigned smem_addr, const void *g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(kPending) : "memory"); }
__device__ __forceinline__ int4 lds_int4(unsigned smem_addr) {
    int4 r;
    asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(smem_addr) : "memory");
    return r;
}

// Tie-breaking of the greedy initial matching (ring passes).  A row with many equally good columns must not always ask
// for the same one, so every row starts its cyclic column order at its own 256-column tile and its own lane:
// across tiles the smallest tile_rot wins (atomicMin), inside a tile the first tied lane at or after (hash & 31), inside
// the lane the first tied slot at or after ((hash >> 5) & 7).
__device__ __forceinline__ unsigned row_hash(int i) { return unsigned(i) * 2654435761u; }
__device__ __forceinline__ int pick_lane(unsigned ballot, unsigned h) {
    const unsigned r = h & 31u;
    return int((unsigned(__ffs(__funnelshift_r(ballot, ballot, r)) - 1) + r) & 31u);   // ballot != 0
}
__device__ __forceinline__ int pick_slot(unsigned mask8, unsigned h) {   // first set bit at or after (h >> 5) & 7, cyclic
    const unsigned s = (h >> 5) & 7u;
    return int((unsigned(__ffs(((mask8 | (mask8 << 8)) >> s) & 0xffu) - 1) + s) & 7u);   // mask8 != 0
}
__device__ __forceinline__ unsigned tile_rot(int col, unsigned h, int n) {
    const unsigned tiles = unsigned(n + 255) >> 8;
    const unsigned off = __umulhi(h, tiles) << 8;
    return unsigned(col) >= off ? unsigned(col) - off : unsigned(col) + (tiles << 8) - off;
}
__device__ __forceinline__ int tile_unrot(unsigned rot, unsigned h, int n) {
    const unsigned tiles = unsigned(n + 255) >> 8;
    const unsigned c = rot + (__umulhi(h, tiles) << 8);
    return int(c >= (tiles << 8) ? c - (tiles << 8) : c);
}

__device__ __forceinline__ int warp_min_i32(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const int other = __shfl_xor_sync(0xffffffffu, v, o); v = other < v ? other : v; }
    return v;
}
__device__ __forceinline__ unsigned warp_min_u32(unsigned v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned other = __shfl_xor_sync(0xffffffffu, v, o); v = other < v ? other : v; }
    return v;
}

// Generic tile sweep through the cp.async ring (n % 4 == 0).  A unit = one 256-column tile x one chunk of consecutive
// positions of the row list (rows == nullptr: the list is 0..nrows-1); units are numbered chunk-major so that warps
// working at the same time read neighbouring segments of the same cost rows.  The first nwarps units are assigned
// statically (small sweeps need no atomics); the rest are handed out through *ticket, because with a static split the
// slowest warp of a bandwidth-bound sweep finishes 2-3x later than the average one (ncu: two thirds of the samples of a
// full-matrix sweep were barrier waits).  Results do not depend on which warp runs which unit.
// unit_begin(j0) sets up the lane's column state, row_fn(pos, row, aux, c[8]) consumes one row (all 32 lanes call it
// together, so it may shuffle), unit_end(j0) publishes.  aux[pos] (optional, e.g. the row's distance - potential) is
// fetched one trip ahead, like the row ids, so no load on the path depends on another one.
__device__ __forceinline__ int ring_chunk_rows(int nrows, int tiles, int nwarps) {
    // Small sweeps are latency-bound: one unit per warp, all static.  Once a warp would get more than 16 rows the sweep
    // is bandwidth-bound and is cut into ~4 units per warp (16..64 rows each) for the dynamic hand-out.
    int groups = nwarps / tiles;
    groups = groups < 1 ? 1 : groups;
    const int per = (nrows + groups - 1) / groups;
    if (per <= 16) return per;
    int r = ((per + 3) / 4 + 3) & ~3;
    return r < 16 ? 16 : (r > 64 ? 64 : r);
}

template <typename UB, typename RF, typename UE>
__device__ __forceinline__ void ring_sweep(const int32_t *__restrict__ cost, int n, const int32_t *__restrict__ rows,
                                           const long long *__restrict__ aux, int nrows, int gwarp, int nwarps, int lane,
                                           unsigned ring, unsigned *ticket, UB unit_begin, RF row_fn, UE unit_end) {
    if (nrows <= 0) return;
    const int tiles = (n + 255) >> 8;
    const int chunk_rows = ring_chunk_rows(nrows, tiles, nwarps);
    const int chunks = (nrows + chunk_rows - 1) / chunk_rows;
    const long long units = (long long)tiles * chunks;
    const unsigned my = ring + unsigned(lane) * 16u;
    long long unit = gwarp;
    while (unit < units) {
        const int tile = int(unit % tiles), chunk = int(unit / tiles);
        const int j0 = (tile << 8) + lane * 4;
        const bool lo_in = j0 < n, hi_in = j0 + 128 < n;
        unit_begin(j0);
        const int p0 = chunk * chunk_rows;
        const int my_rows = (nrows - p0) < chunk_rows ? (nrows - p0) : chunk_rows;
        const int ntrips = (my_rows + 3) >> 2;
        const int32_t *cbase = cost + j0;
        auto issue = [&](int trip, const int (&r)[4]) {
            const unsigned st = my + unsigned(trip % kAsgStages) * kAsgStageBytes;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (r[q] < 0) continue;
                const int32_t *line = cbase + size_t(r[q]) * n;
                if (lo_in) cp_async16(st + q * 1024, line);
                if (hi_in) cp_async16(st + q * 1024 + 512, line + 128);
            }
            cp_async_commit();   // possibly empty: keeps the group count uniform
        };
        auto ids_of = [&](int trip, int (&r)[4]) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = 4 * trip + q;
                r[q] = e < my_rows ? (rows ? rows[p0 + e] : p0 + e) : -1;
            }
        };
        auto aux_of = [&](int trip, int (&x)[4]) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = 4 * trip + q;
                x[q] = (aux && e < my_rows) ? int(aux[p0 + e]) : 0;
            }
        };
        int ids[4], cur[4], ax[4];
        ids_of(0, cur);
        issue(0, cur);
#pragma unroll
        for (int t = 1; t < kAsgStages; ++t) { ids_of(t, ids); issue(t, ids); }
        ids_of(kAsgStages, ids);
        aux_of(0, ax);
        for (int trip = 0; trip < ntrips; ++trip) {
            cp_async_wait<kAsgStages - 1>();
            const unsigned st = my + unsigned(trip % kAsgStages) * kAsgStageBytes;
            const int last_q = my_rows - 4 * trip;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q >= last_q) continue;   // warp-uniform
                const int4 lo = lo_in ? lds_int4(st + q * 1024) : make_int4(0, 0, 0, 0);
                const int4 hi = hi_in ? lds_int4(st + q * 1024 + 512) : make_int4(0, 0, 0, 0);
                const int c[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
                row_fn(p0 + 4 * trip + q, cur[q], ax[q], c);
            }
            issue(trip + kAsgStages, ids);   // refills the stage just consumed (its ids were fetched a trip ago)
            ids_of(trip + kAsgStages + 1, ids);
            ids_of(trip + 1, cur);
            aux_of(trip + 1, ax);
        }
        cp_async_wait<0>();
        unit_end(j0);
        if (units <= nwarps) break;   // everything was assigned statically
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(ticket, 1u);
        unit = (long long)nwarps + __shfl_sync(0xffffffffu, t, 0);
    }
}

// warp per row: minimum and first argmin column of (c_ij - v_j); optionally restricted to free, tight columns
// Ties are broken by the column's cyclic distance from a row-dependent offset, so that rows with
// many equally good columns spread their proposals instead of all asking for the same few.
__device__ __forceinline__ unsigned row_offset(int i, int n) { return unsigned((unsigned(i) * 2654435761u) % unsigned(n)); }

template <bool kVec>
__device__ __forceinline__ unsigned long long row_min_reduced(const AsgArgs &a, int i, int lane, bool tight_free_only,
                                                              long long ui) {
    const int n = a.n;
    const unsigned off = row_offset(i, n);
    auto rot = [&](int j) -> unsigned { const unsigned d = unsigned(j) + unsigned(n) - off; return d >= unsigned(n) ? d - unsigned(n) : d; };
    const int32_t *line = a.cost + size_t(i) * n;
    unsigned long long best = kDistInf;
    if (kVec) {
        // 4 x 16-byte loads in flight per lane (a warp-per-row scan is latency-bound otherwise)
        for (int j0 = lane * 4; j0 < n; j0 += 512) {
            int4 q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + 128 * u;
                q[u] = j < n ? ld_stream_int4(reinterpret_cast<const int4 *>(line + j)) : make_int4(0, 0, 0, 0);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int j = j0 + 128 * u;
                if (j >= n) continue;
                const int c[4] = {q[u].x, q[u].y, q[u].z, q[u].w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const long long red = (long long)c[k] - a.v[j + k];
                    if (tight_free_only) {
                        if (red == ui && a.mate_c[j + k] < 0) { const unsigned long long key = rot(j + k); best = key < best ? key : best; }
                    } else {
                        const unsigned long long key = ((unsigned long long)red << 32) | rot(j + k);
                        best = key < best ? key : best;
                    }
                }
            }
        }
    } else {
        for (int j = lane; j < n; j += 32) {
            const long long red = (long long)__ldg(line + j) - a.v[j];
            if (tight_free_only) {
                if (red == ui && a.mate_c[j] < 0) { const unsigned long long key = rot(j); best = key < best ? key : best; }
            } else {
                const unsigned long long key = ((unsigned long long)red << 32) | rot(j);
                best = key < best ? key : best;
            }
        }
    }
    return warp_min_u64(best);
}

template <bool kVec>
__global__ void __launch_bounds__(kAsgThreads)
assign_kernel(AsgArgs a) {
    cg::grid_group grid = cg::this_grid();
    const int n = a.n;
    const int nr = a.nr;              // real rows; the padding rows nr..n-1 never search, they take the leftover columns
    const bool rect = nr < n;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nthreads = gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    const int gwarp = tid >> 5, nwarps = nthreads >> 5;
    __shared__ unsigned long long s_red[kAsgThreads / 32];
    __shared__ unsigned s_push[kAsgThreads / 32], s_push_base;
    extern __shared__ __align__(1024) unsigned char s_ring[];   // kVec only: per-warp cp.async ring
    const unsigned ring = unsigned(__cvta_generic_to_shared(s_ring)) + unsigned(threadIdx.x >> 5) * (kAsgStages * kAsgStageBytes);
    AsgCtrl *ctrl = a.ctrl;
    unsigned long long t_last = 0;
    const bool prof = a.prof != 0;   // the timers are read-modify-writes on CTA 0's path to every barrier: off by default
    auto tick = [&](int k) {   // thread 0 only: accumulate wall time since the previous tick into bucket k
        if (prof && tid == 0) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (k >= 0) ctrl->t_prof[k] += t - t_last;
            t_last = t;
        }
    };

    // ================= init =====================================================================
    for (int j = tid; j < n; j += nthreads) { a.vmin[j] = INT_MAX; a.mate_c[j] = -1; a.prop[j] = INT_MAX; }
    for (int i = tid; i < n; i += nthreads) { a.mate_r[i] = -1; }
    if (tid == 0) {
        ctrl->fcount[0] = ctrl->fcount[1] = 0; ctrl->nsinks = 0; ctrl->phases = ctrl->levels = ctrl->augment = 0;
        ctrl->rows_scanned = 0; ctrl->status = TD_OK; ctrl->gmin[0] = ctrl->gmin[1] = ctrl->gmin[2] = kDistInf;
    }
    grid.sync();
    tick(-1);
    // column slots of a lane inside a 256-column tile (ring sweeps): j0..j0+3 and j0+128..j0+131
    auto slot_col = [](int j0, int k) { return j0 + (k & 3) + ((k >> 2) << 7); };
    {   // column minima (and max |c| for the 32-bit guard)
        if (kVec) {
            int best[8];
            int cmx = 0;
            ring_sweep(a.cost, n, nullptr, nullptr, n, gwarp, nwarps, lane, ring, &ctrl->ticket[0],
                       [&](int) {
#pragma unroll
                           for (int k = 0; k < 8; ++k) best[k] = INT_MAX;
                       },
                       [&](int, int, int, const int (&c)[8]) {
#pragma unroll
                           for (int k = 0; k < 8; ++k) { best[k] = c[k] < best[k] ? c[k] : best[k]; cmx = c[k] > cmx ? c[k] : cmx; }
                       },
                       [&](int j0) {
#pragma unroll
                           for (int k = 0; k < 8; ++k) {
                               const int col = slot_col(j0, k);
                               if (col < n && best[k] < a.vmin[col]) atomicMin(&a.vmin[col], best[k]);
                           }
                       });
            cmx = -warp_min_i32(-cmx);
            if (lane == 0 && cmx > 0) atomicMax(&ctrl->cabs, (unsigned long long)cmx);
        } else {
            unsigned long long dummy = kDistInf;
            sweep_rows<0, kVec>(a, nullptr, n, gwarp, nwarps, lane, dummy);
        }
    }
    grid.sync();
    tick(6);
    {
        int vmn = 0;
        // rectangular instance: no column reduction -- a column that stays without a real row must keep v = 0
        for (int j = tid; j < n; j += nthreads) { const int m = a.vmin[j]; a.v[j] = rect ? 0 : m; vmn = m < vmn ? m : vmn; }
        if (vmn < 0) atomicMax(&ctrl->cabs, (unsigned long long)(-(long long)vmn));
        for (int i = tid; i < n; i += nthreads) a.distpred[i] = kDistInf;   // per-row (minimum, argmin) keys of the next pass
    }
    grid.sync();
    // c - v and u - (c - v) stay inside 32 bits when max |c| < 2^29; otherwise the 64-bit row scans are used
    const bool init_ring = kVec && ctrl->cabs < (1ull << 29);
    // row minima of the column-reduced costs; every row proposes its first argmin column (cyclic order from a
    // row-dependent offset, so that rows with many equally good columns spread their proposals)
    if (init_ring) {
        int nv[8], uj0 = 0;
        bool in[8];
        ring_sweep(a.cost, n, nullptr, nullptr, nr, gwarp, nwarps, lane, ring, &ctrl->ticket[1],
                   [&](int j0) {
                       uj0 = j0;
#pragma unroll
                       for (int k = 0; k < 8; ++k) { const int col = slot_col(j0, k); in[k] = col < n; nv[k] = in[k] ? -int(a.v[col]) : 0; }
                   },
                   [&](int, int i, int, const int (&c)[8]) {
                       int val[8], lm = INT_MAX;
#pragma unroll
                       for (int k = 0; k < 8; ++k) { val[k] = in[k] ? c[k] + nv[k] : INT_MAX; lm = val[k] < lm ? val[k] : lm; }
                       const int m = warp_min_i32(lm);
                       const unsigned h = row_hash(i);
                       if (lane == pick_lane(__ballot_sync(0xffffffffu, lm == m), h)) {
                           unsigned mask = 0;
#pragma unroll
                           for (int k = 0; k < 8; ++k) mask |= val[k] == m ? (1u << k) : 0u;
                           const int col = slot_col(uj0, pick_slot(mask, h));
                           atomicMin(&a.distpred[i], ((unsigned long long)unsigned(m) << 32) | tile_rot(col, h, n));
                       }
                   },
                   [&](int) {});
        grid.sync();
        for (int i = tid; i < nr; i += nthreads) {
            const unsigned long long k = a.distpred[i];
            a.u[i] = (long long)(k >> 32);
            const int j = tile_unrot(unsigned(k), row_hash(i), n);
            a.argcol[i] = j;
            atomicMin(&a.prop[j], i);
        }
    } else {
        for (int i = gwarp; i < nr; i += nwarps) {
            const unsigned long long k = row_min_reduced<kVec>(a, i, lane, false, 0);
            if (lane == 0) {
                a.u[i] = (long long)(k >> 32);
                const int j = int((unsigned(k) + row_offset(i, n)) % unsigned(n));
                a.argcol[i] = j;
                atomicMin(&a.prop[j], i);
            }
        }
    }
    grid.sync();
    tick(7);
    unsigned prev_lost = 0xffffffffu / 32u;
    for (int round = 0;; ++round) {
        // accept: the lowest proposing row takes the column; the others are listed (row, u) for the next round
        const int lst = round & 1;
        for (int base = blockIdx.x * blockDim.x; base < n; base += nthreads) {
            const int i = base + threadIdx.x;
            bool lost = false;
            if (i < nr && a.mate_r[i] < 0) {
                const int j = a.argcol[i];
                if (j >= 0 && a.prop[j] == i) { a.mate_r[i] = j; a.mate_c[j] = i; }
                else lost = true;
            }
            if (init_ring) {
                const unsigned ball = __ballot_sync(0xffffffffu, lost);
                unsigned wb = 0;
                if (lane == 0 && ball) wb = atomicAdd(&ctrl->fcount[lst], __popc(ball));
                wb = __shfl_sync(0xffffffffu, wb, 0);
                if (lost) {
                    const unsigned slot_i = wb + __popc(ball & ((1u << lane) - 1));
                    a.frontier[lst][slot_i] = i;
                    a.fbase[lst][slot_i] = a.u[i];
                    a.claim[i] = -1;   // = UINT_MAX: no tight free column found yet
                }
            }
        }
        grid.sync();
        if (round == a.greedy_rounds - 1) break;
        if (init_ring) {   // stop early when nobody lost, or when a round matched fewer than 5 % of its losers
            const unsigned nl = ctrl->fcount[lst];
            if (nl == 0 || (round >= 3 && nl * 20u > prev_lost * 19u)) break;
            prev_lost = nl;
        } else if (round >= 3) {
            break;   // the 64-bit fallback path rescans whole rows per loser: four rounds
        }
        for (int j = tid; j < n; j += nthreads) a.prop[j] = INT_MAX;
        if (tid == 0) { ctrl->fcount[lst ^ 1] = 0; ctrl->ticket[lst] = 0; }
        grid.sync();
        // losers look for their first tight column that is still free
        if (init_ring) {
            const int nlost = int(ctrl->fcount[lst]);
            int nv[8], uj0 = 0;
            bool in[8];
            ring_sweep(a.cost, n, a.frontier[lst], a.fbase[lst], nlost, gwarp, nwarps, lane, ring, &ctrl->ticket[lst],
                       [&](int j0) {
                           uj0 = j0;
#pragma unroll
                           for (int k = 0; k < 8; ++k) {
                               const int col = slot_col(j0, k);
                               in[k] = col < n && a.mate_c[col < n ? col : 0] < 0;
                               nv[k] = in[k] ? -int(a.v[col]) : 0;
                           }
                       },
                       [&](int, int i, int ui, const int (&c)[8]) {
                           bool tight[8], any = false;
#pragma unroll
                           for (int k = 0; k < 8; ++k) { tight[k] = in[k] && c[k] + nv[k] == ui; any = any || tight[k]; }
                           const unsigned ball = __ballot_sync(0xffffffffu, any);
                           if (ball == 0) return;
                           const unsigned h = row_hash(i);
                           if (lane == pick_lane(ball, h)) {
                               unsigned mask = 0;
#pragma unroll
                               for (int k = 0; k < 8; ++k) mask |= tight[k] ? (1u << k) : 0u;
                               const int col = slot_col(uj0, pick_slot(mask, h));
                               atomicMin(reinterpret_cast<unsigned *>(&a.claim[i]), tile_rot(col, h, n));
                           }
                       },
                       [&](int) {});
            grid.sync();
            for (int t = tid; t < nlost; t += nthreads) {
                const int i = a.frontier[lst][t];
                const unsigned cand = unsigned(a.claim[i]);
                const int j = cand == 0xffffffffu ? -1 : tile_unrot(cand, row_hash(i), n);
                a.argcol[i] = j;
                if (j >= 0) atomicMin(&a.prop[j], i);
            }
        } else {
            for (int i = gwarp; i < nr; i += nwarps) {
                if (a.mate_r[i] >= 0) continue;
                const unsigned long long k = row_min_reduced<kVec>(a, i, lane, true, a.u[i]);
                if (lane == 0) {
                    const int j = (k == kDistInf) ? -1 : int((unsigned(k) + row_offset(i, n)) % unsigned(n));
                    a.argcol[i] = j;
                    if (j >= 0) atomicMin(&a.prop[j], i);
                }
            }
        }
        grid.sync();
    }
    if (tid == 0) { ctrl->fcount[0] = ctrl->fcount[1] = 0; ctrl->ticket[0] = ctrl->ticket[1] = ctrl->ticket[2] = 0; }
    grid.sync();

    for (int i = tid; i < n; i += nthreads) { a.uinit[i] = a.u[i]; a.vinit[i] = a.v[i]; }
    // ================= phases ===================================================================
    bool first_phase = true;
    bool keep_forest = false;
    for (int phase = 0;; ++phase) {
        // ---- P0: reset search state, frontier = all free rows ---------------------------------
        tick(-1);
        if (tid == 0) { ctrl->nsinks = 0; ctrl->ndone = 0; }
        // Trees that were not augmented survive into this phase (carry_forest): after the dual update all their edges
        // are tight, so their rows sit at distance 0 and their columns stay settled with the same predecessors; the
        // rows are relaxed again in ONE bandwidth-bound sweep at level 0 instead of being re-discovered tight edge by
        // tight edge over dozens of latency-bound levels.  The end of the previous phase left drow = 0 / settled = 1 /
        // distpred = (0, predecessor) on exactly those nodes.
        const bool carried = keep_forest;   // decided at the end of the previous phase
        for (int j = tid; j < n; j += nthreads) {
            if (!carried || !a.settled[j]) { a.distpred[j] = kDistInf; a.settled[j] = 0; }
        }
        for (int base = blockIdx.x * blockDim.x; base < n; base += nthreads) {
            const int i = base + threadIdx.x;
            bool is_free = false, is_carry = false;
            if (i < n) {
                a.claim[i] = INT_MAX;
                is_free = i < nr && a.mate_r[i] < 0;
                if (is_free) { a.drow[i] = 0; a.root[i] = i; }
                else if (carried && a.drow[i] == 0) is_carry = true;
                else a.drow[i] = kRowInf;
            }
            const unsigned ball = __ballot_sync(0xffffffffu, is_free);
            const unsigned ballc = __ballot_sync(0xffffffffu, is_carry);
            unsigned wb = 0, wc = 0;
            if (lane == 0 && ball) wb = atomicAdd(&ctrl->fcount[0], __popc(ball));
            if (lane == 0 && ballc) wc = atomicAdd(&ctrl->ncarry, __popc(ballc));
            wb = __shfl_sync(0xffffffffu, wb, 0);
            wc = __shfl_sync(0xffffffffu, wc, 0);
            if (is_free) {
                const unsigned slot_i = wb + __popc(ball & ((1u << lane) - 1));
                a.frontier[0][slot_i] = i;
                a.fbase[0][slot_i] = -a.u[i];
            }
            if (is_carry) {
                const unsigned slot_i = wc + __popc(ballc & ((1u << lane) - 1));
                a.carry[slot_i] = i;
                a.cbase[slot_i] = -a.u[i];
            }
        }
        grid.sync();
        tick(16);
        const unsigned nfree = ctrl->fcount[0];
        if (first_phase && tid == 0) ctrl->free_after_init = nfree;
        first_phase = false;
        if (nfree == 0) break;
        if (phase >= a.max_phases) { if (tid == 0) ctrl->status = TD_ERR_NOT_CONVERGED; break; }
        if (phase > 0) {
            // Level 0 without re-reading the free rows.  Every free row has been free since the start and has
            // received the same potential shift (sfree), and rows only LEAVE the free set, so the column minimum
            // over the free rows taken once (base0) stays valid until its arg-min row is matched; only those
            // columns are refreshed (a strided read of the column over the free-row list).
            for (int j = tid; j < n; j += nthreads)
                if (a.mate_r[dp_row(a.base0[j])] >= 0) a.stale[atomicAdd(&ctrl->nstale, 1u)] = j;
            grid.sync();
            tick(17);
            const unsigned ns_cols = ctrl->nstale;
            for (unsigned sidx = gwarp; sidx < ns_cols; sidx += nwarps) {
                const int j = a.stale[sidx];
                const long long vj0 = a.vinit[j];
                unsigned long long best = kDistInf;
                for (unsigned t = lane; t < nfree; t += 32) {
                    const int i = a.frontier[0][t];
                    const unsigned long long key = pack_dp((long long)__ldg(a.cost + size_t(i) * n + j) - a.uinit[i] - vj0, i);
                    best = key < best ? key : best;
                }
                best = warp_min_u64(best);
                if (lane == 0) a.base0[j] = best;
            }
            if (tid == 0) ctrl->stale_cells += (unsigned long long)ns_cols * nfree;
            grid.sync();
            tick(18);
            const long long sfree = ctrl->sfree;
            unsigned long long lmin = kDistInf;
            for (int j = tid; j < n; j += nthreads) {
                if (a.settled[j]) continue;   // column of a surviving tree
                const unsigned long long b = a.base0[j];
                const long long d0 = dp_dist(b) + a.vinit[j] - a.v[j] - sfree;
                atomicMin(&a.distpred[j], pack_dp(d0, dp_row(b)));   // the level-0 sweep of the carried rows may run already
                lmin = (unsigned long long)d0 < lmin ? (unsigned long long)d0 : lmin;
            }
            lmin = warp_min_u64(lmin);
            if (lane == 0 && lmin != kDistInf) atomicMin(&ctrl->gmin[0], lmin);
            if (tid == 0) ctrl->nstale = 0;
        }

        int cur = 0, nlevels = 0;
        long long dstar = 0, last_delta = 0;
        // a phase does not stop at the first sink: it keeps growing the forest (distances stay exact, every
        // settled node is included in the dual update, so all forest edges become tight) until this many trees
        // own a sink; each of them is augmented.  Fewer phases, and a phase never scans a row twice.
        unsigned want_done = unsigned((unsigned long long)nfree * unsigned(a.deep_permille) / 1000u);
        want_done = want_done < 1u ? 1u : want_done;
        // rectangular: stop at the first level that reaches a free column, so that every sink sits at distance D and
        // the columns that stay unmatched keep v = 0 (their dual constraint is  v <= 0, = 0 when slack)
        if (rect) want_done = 1u;
        tick(4);
        for (int level = 0;; ++level) {
            const int slot = level % 3;
            // ---- (a) relax: every frontier row against all unsettled columns ------------------
            // level 0 of a later phase: the free rows come from the cache, the rows of surviving trees are swept
            const bool from_carry = phase > 0 && level == 0;
            const unsigned fc = from_carry ? ctrl->ncarry : ctrl->fcount[cur];
            const int32_t *lrows = from_carry ? a.carry : a.frontier[cur];
            const long long *lbase = from_carry ? a.cbase : a.fbase[cur];
            unsigned long long bmin = kDistInf;
            // 32-bit guard: every (distance - u - v + c) of this level is below 4 cabs + 2 sfree + last_delta
            const bool narrow = kVec && !a.force_wide &&
                                4 * ctrl->cabs + 2 * (unsigned long long)ctrl->sfree + (unsigned long long)last_delta < (1ull << 30);
            if (narrow && kVec) {
                // 32-bit relaxation through the cp.async ring: one IADD3 + compare/select pair per cost cell instead of
                // the ~13 integer instructions of the 64-bit (distance, predecessor) keys of sweep_rows
                int nv[8], best[8];
                unsigned bsr[8];   // scrambled predecessor row: (distance, scrambled row) is minimised lexicographically,
                                   // so the result does not depend on the order of the frontier list or on the chunking
                bool act[8];
                const bool small_sweep = ring_chunk_rows(int(fc), (n + 255) >> 8, nwarps) <= 16 && fc > 0;
                ring_sweep(a.cost, n, lrows, lbase, int(fc), gwarp, nwarps, lane, ring, &ctrl->ticket[slot],
                           [&](int j0) {
#pragma unroll
                               for (int k = 0; k < 8; ++k) {
                                   const int col = slot_col(j0, k);
                                   act[k] = col < n && !a.settled[col < n ? col : 0];
                                   nv[k] = act[k] ? -int(a.v[col]) : 0;
                                   best[k] = INT_MAX;
                                   bsr[k] = kRowMask;
                               }
                           },
                           [&](int, int i, int base, const int (&c)[8]) {
                               const unsigned sr = scramble_row(i);
#pragma unroll
                               for (int k = 0; k < 8; ++k) {
                                   const int val = c[k] + base + nv[k];
                                   if (val < best[k] || (val == best[k] && sr < bsr[k])) { best[k] = val; bsr[k] = sr; }
                               }
                           },
                           [&](int j0) {
#pragma unroll
                               for (int k = 0; k < 8; ++k) {
                                   if (!act[k] || best[k] == INT_MAX) continue;
                                   const int col = slot_col(j0, k);
                                   const unsigned long long key = ((unsigned long long)(long long)best[k] << kRowBits) | bsr[k];
                                   // small (latency-bound) sweeps skip the pre-check load; a candidate that does not
                                   // improve its column cannot lower the level minimum below the true one either
                                   if (small_sweep || key < a.distpred[col]) {
                                       atomicMin(&a.distpred[col], key);
                                       bmin = key < bmin ? key : bmin;
                                   }
                               }
                           });
            }
            else sweep_rows<1, kVec>(a, lrows, int(fc), gwarp, nwarps, lane, bmin);
            if (prof && tid == 0 && narrow) ctrl->narrow_levels += 1;
            bmin = warp_min_u64(bmin);
            if (lane == 0) s_red[threadIdx.x >> 5] = bmin;
            __syncthreads();
            if (threadIdx.x < 32) {
                unsigned long long m = threadIdx.x < kAsgThreads / 32 ? s_red[threadIdx.x] : kDistInf;
                m = warp_min_u64(m);
                if (threadIdx.x == 0 && m != kDistInf) atomicMin(&ctrl->gmin[slot], m >> kRowBits);
            }
            if (tid == 0 && fc) atomicAdd(&ctrl->rows_scanned, (unsigned long long)fc);   // fire and forget
            if (prof && tid == 0) {   // diagnostics: levels and scan time by frontier size (<= 32, <= 256, <= 2048, larger)
                const int bkt = fc <= 32 ? 0 : (fc <= 256 ? 1 : (fc <= 2048 ? 2 : 3));
                unsigned long long t;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                ctrl->t_prof[8 + bkt] += t - t_last;
                ctrl->t_prof[12 + bkt] += 1;
            }
            tick(0);
            grid.sync();
            tick(1);
            // ---- (b) settle every column at the new minimum distance -------------------------
            const unsigned long long dl = ctrl->gmin[slot];
            if (dl == kDistInf) {
                // nothing left to settle: the forest is complete.  Fine when some tree already owns a sink.
                if (ctrl->ndone > 0) { dstar = last_delta; break; }
                if (tid == 0) ctrl->status = TD_ERR_NOT_CONVERGED;
                dstar = -1;
                break;
            }
            if (level > 2 * n + 16) { if (tid == 0) ctrl->status = TD_ERR_NOT_CONVERGED; dstar = -1; break; }   // cannot happen
            const long long delta = (long long)dl;
            last_delta = delta;
            unsigned long long carry = kDistInf;
            for (int base = blockIdx.x * blockDim.x; base < n; base += nthreads) {
                // all loads of a step are independent of each other: three round trips per level (state, tree data,
                // frontier slot) instead of one per dependent access
                const int j = base + threadIdx.x;
                const bool inb = j < n;
                const bool was_settled = inb ? a.settled[j] != 0 : true;
                const unsigned long long k = inb ? a.distpred[j] : kDistInf;
                const int mate = inb ? a.mate_c[j] : -1;
                if (phase == 0 && level == 0 && inb) a.base0[j] = k;   // sfree = 0, v = v_init here
                bool now = false;
                if (!was_settled && k != kDistInf) {
                    const long long d = dp_dist(k);
                    now = d == delta;
                    if (!now) carry = (unsigned long long)d < carry ? (unsigned long long)d : carry;
                }
                const bool push = now && mate >= 0, sink = now && mate < 0;
                int root_p = 0;
                long long u_mate = 0;
                if (now) root_p = a.root[dp_row(k)];
                if (push) u_mate = a.u[mate];
                // frontier slots: one global atomic per CTA and pass (up to 640 warps hit the same counter otherwise)
                const unsigned ball = __ballot_sync(0xffffffffu, push);
                if (lane == 0) s_push[threadIdx.x >> 5] = __popc(ball);
                __syncthreads();
                if (threadIdx.x == 0) {
                    unsigned run = 0;
#pragma unroll
                    for (int w2 = 0; w2 < kAsgThreads / 32; ++w2) { const unsigned c = s_push[w2]; s_push[w2] = run; run += c; }
                    s_push_base = run ? atomicAdd(&ctrl->fcount[cur ^ 1], run) : 0u;
                }
                __syncthreads();
                unsigned wb = s_push_base + s_push[threadIdx.x >> 5];
                if (now) a.settled[j] = 1;
                if (sink) {
                    a.sinks[atomicAdd(&ctrl->nsinks, 1u)] = j;
                    // one augmenting path per tree: the smallest sink column wins (order-independent)
                    if (atomicMin(&a.claim[root_p], j) == INT_MAX) atomicAdd(&ctrl->ndone, 1u);
                }
                if (push) { a.drow[mate] = delta; a.root[mate] = root_p; }
                __syncthreads();   // s_push is rewritten by the next pass of this loop
                if (push) {
                    const unsigned slot_i = wb + __popc(ball & ((1u << lane) - 1));
                    a.frontier[cur ^ 1][slot_i] = mate;
                    a.fbase[cur ^ 1][slot_i] = delta - u_mate;
                }
            }
            carry = warp_min_u64(carry);
            if (lane == 0 && carry != kDistInf) atomicMin(&ctrl->gmin[(level + 1) % 3], carry);
            if (tid == 0) { ctrl->gmin[(level + 2) % 3] = kDistInf; ctrl->ticket[(level + 2) % 3] = 0; atomicAdd(&ctrl->levels, 1u); }
            tick(2);
            grid.sync();
            tick(3);
            if (tid == 0) ctrl->fcount[cur] = 0;  // consumed; becomes the target two levels from now
            nlevels = level + 1;
            if (ctrl->ndone >= want_done) { dstar = delta; break; }
            cur ^= 1;
        }
        if (dstar < 0) break;

        // Surviving trees are kept for the next phase only when this phase was deep: re-discovering a deep forest costs
        // one latency-bound level per tight edge on the way, while shallow phases (easy instances) are better off with
        // freshly balanced trees.
        keep_forest = a.carry_forest != 0 && nlevels >= a.carry_min_levels;
        // ---- augment: one sink per tree, smallest column index wins ---------------------------
        const unsigned ns = ctrl->nsinks;
        for (unsigned s = tid; s < ns; s += nthreads) {
            int j = a.sinks[s];
            if (a.claim[a.root[dp_row(a.distpred[j])]] != j) continue;
            for (;;) {  // flip the tree path sink -> root
                const int i = dp_row(a.distpred[j]);
                const int nxt = a.mate_r[i];
                a.mate_r[i] = j;
                a.mate_c[j] = i;
                if (nxt < 0) break;
                j = nxt;
            }
            atomicAdd(&ctrl->augment, 1u);
        }
        // potentials: every forest edge becomes tight, feasibility is kept
        for (int i = tid; i < n; i += nthreads) {
            const long long d = a.drow[i];
            if (d != kRowInf) {
                a.u[i] += dstar - d;
                // rows of trees that found no sink stay in the forest (distance 0 after this update)
                a.drow[i] = (keep_forest && a.claim[a.root[i]] == INT_MAX) ? 0 : kRowInf;
            }
        }
        for (int j = tid; j < n; j += nthreads) {
            if (!a.settled[j]) continue;
            const unsigned long long k = a.distpred[j];
            a.v[j] -= dstar - dp_dist(k);
            // distpred of a column on an augmenting path is still being read by the flip above: only survivors are rewritten
            if (keep_forest && a.claim[a.root[dp_row(k)]] == INT_MAX) a.distpred[j] = pack_dp(0, dp_row(k));
            else a.settled[j] = 0;
        }
        if (tid == 0) {
            // nsinks / ndone are reset at the start of the next phase: slower CTAs may still be reading them here
            ctrl->fcount[0] = ctrl->fcount[1] = 0; ctrl->phases += 1; ctrl->sfree += dstar;
            ctrl->gmin[0] = ctrl->gmin[1] = ctrl->gmin[2] = kDistInf;
            ctrl->ticket[0] = ctrl->ticket[1] = ctrl->ticket[2] = 0; ctrl->ncarry = 0;
        }
        grid.sync();
        tick(5);
    }

    // ================= finish ===================================================================
    if (rect) {
        // padding rows take the columns no real row uses, in index order (any choice has the same cost)
        if (blockIdx.x == 0 && threadIdx.x < 32) {
            int next_row = nr;
            for (int base = 0; base < n; base += 32) {
                const int j = base + lane;
                const bool is_free = j < n && a.mate_c[j] < 0;
                const unsigned ball = __ballot_sync(0xffffffffu, is_free);
                if (is_free) {
                    const int r = next_row + __popc(ball & ((1u << lane) - 1));
                    if (r < n) { a.mate_r[r] = j; a.mate_c[j] = r; }
                }
                next_row += __popc(ball);
            }
        }
        grid.sync();
    }
    long long part = 0;
    for (int i = tid; i < n; i += nthreads) {
        const int j = a.mate_r[i];
        a.col_of_row_out[i] = j;
        if (j >= 0) {
            part += a.cost[size_t(i) * n + j];
            if (a.x_out) a.x_out[size_t(i) * n + j] = 1;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0 && part != 0) atomicAdd(reinterpret_cast<unsigned long long *>(&ctrl->objective), (unsigned long long)part);
    grid.sync();
    // A solve that gave up (phase / level guards; cannot happen on finite integer costs) must not look like a result when
    // the caller passed no stats: the matching is withdrawn (-1 everywhere) and the objective is INT64_MIN.
    const bool failed = *reinterpret_cast<volatile int *>(&ctrl->status) != TD_OK;
    if (failed)
        for (int i = tid; i < n; i += nthreads) a.col_of_row_out[i] = -1;
    if (tid == 0) *a.objective_out = failed ? LLONG_MIN : ctrl->objective;
}

// ---- small instances: one CTA, everything in shared memory ------------------------------------------------------------
// BASELINE config 1 (200 x 200, python.py:6-25) spends its time in grid barriers when it runs through assign_kernel
// (0.68 ms for a 160 KB matrix).  Up to kSmallN rows the whole matrix fits the shared memory of ONE SM: a single CTA runs
// the classic primal-dual shortest-augmenting-path method (Kuhn-Munkres with potentials; column j lives in thread j's
// registers: its minimum reduced cost, predecessor, potential and visited flag), so a path step costs three block
// barriers and one block-wide arg-min instead of two grid-wide barriers.  Start: row minima, column minima of the
// row-reduced costs, greedy matching on tight cells -- only the rows that stay free are augmented.
// Exact for any int32 costs (potentials and distances in int64); ties resolve to the smallest column, deterministic.
// Leaves the dual potentials in the workspace like assign_kernel does (td_assign_read_duals / td_assign_certify).
// The body is a device routine shared by the single-instance kernel and the batched one (one CTA per instance), so both
// return the same matching and the same potentials for the same matrix.  u_out / v_out may be NULL; the objective is
// written to *objective_out and returned on thread 0.
constexpr int kSmallN = TD_BATCH_MAX_N;   // 232^2 * 4 B = 210 KB of the 227 KB
constexpr int kSmallThreads = 256;
static_assert(kSmallN <= kSmallThreads, "column j lives in thread j");
__host__ __device__ constexpr size_t small_smem_bytes(int n) {
    return ((size_t(n) * n * 4 + 15) & ~size_t(15)) + size_t(n) * (8 + 4 + 4 + 4 + 4) + 64;
}
__device__ __forceinline__ long long
assign_small_solve(const int32_t *__restrict__ cost, int n, int32_t *col_of_row_out, long long *objective_out, uint8_t *x_out,
                   long long *u_out, long long *v_out) {
    extern __shared__ __align__(16) unsigned char ssm[];
    int32_t *c = reinterpret_cast<int32_t *>(ssm);                                   // [n][n]
    long long *u = reinterpret_cast<long long *>(ssm + ((size_t(n) * n * 4 + 15) & ~size_t(15)));   // [n]
    int *p = reinterpret_cast<int *>(u + n);        // p[j]: row matched to column j, -1: free       [n]
    int *way = p + n;                               // predecessor column on the alternating path, -1: the root   [n]
    int *mate = way + n;                            // mate[i]: column of row i, -1: free            [n]
    __shared__ long long s_rk[kSmallThreads / 32];
    __shared__ int s_rj[kSmallThreads / 32];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const long long kInf = LLONG_MAX / 4;
    for (int i = t; i < n * n; i += kSmallThreads) c[i] = __ldg(cost + i);
    __syncthreads();
    // row minima -> u; column minima of the row-reduced costs -> v (thread j owns column j)
    if (t < n) {
        int m = INT_MAX;
        for (int j = 0; j < n; ++j) { const int v0 = c[t * n + ((j + t) % n)]; m = v0 < m ? v0 : m; }   // rotated: spreads the banks
        u[t] = m;
        p[t] = -1; mate[t] = -1;
    }
    __syncthreads();
    long long v = 0;
    if (t < n) {
        long long m = kInf;
        for (int i = 0; i < n; ++i) { const long long r = (long long)c[i * n + t] - u[i]; m = r < m ? r : m; }
        v = m;
    }
    // greedy matching on tight cells: every free column asks for the lowest free row that is tight with it, every asked
    // row accepts the lowest such column
    __shared__ int s_progress;
    for (int round = 0; round < 4; ++round) {   // more rounds cost more than the few pairs they add (measured)
        __syncthreads();
        if (t == 0) s_progress = 0;
        int pick = -1;
        if (t < n && p[t] < 0)
            for (int i = 0; i < n && pick < 0; ++i)
                if (mate[i] < 0 && (long long)c[i * n + t] - u[i] - v == 0) pick = i;
        if (t < n) way[t] = pick;                // several columns may ask for the same row
        __syncthreads();
        if (t < n && mate[t] < 0) {
            int got = -1;
            for (int j = 0; j < n && got < 0; ++j)
                if (way[j] == t) got = j;
            if (got >= 0) { mate[t] = got; p[got] = t; s_progress = 1; }
        }
        __syncthreads();
        if (!s_progress) break;
    }
    __syncthreads();
    // ---- augment every row that is still free ---------------------------------------------------------------------
    // Dijkstra over the columns from row i, one DISTANCE LEVEL per step: every unvisited column at the current minimum
    // joins the tree together and the rows matched to them are relaxed in the same step (on the reference's degenerate
    // costs a level holds dozens of columns; one column per step took 2.6x longer than the cooperative kernel).
    int *rows_new = mate + n;                    // rows whose edges are relaxed in this step                     [n]
    __shared__ int s_nnew, s_jfree, s_wcnt[kSmallThreads / 32];
    for (int i = 0; i < n; ++i) {
        if (mate[i] >= 0) continue;              // uniform: mate[] is in shared memory, read after a barrier
        long long minv = kInf;                   // column t: best reduced distance so far
        bool used = false;                       // column t is in the tree
        if (t < n) way[t] = -1;
        if (t == 0) { rows_new[0] = i; s_nnew = 1; }
        __syncthreads();
        int jend;
        for (;;) {
            // relax the rows that joined in the previous step (list order = column order: deterministic predecessors)
            const int nnew = s_nnew;
            long long key = kInf;
            if (t < n && !used) {
                for (int k = 0; k < nnew; ++k) {
                    const int r = rows_new[k];
                    const long long cur = (long long)c[r * n + t] - u[r] - v;
                    if (cur < minv) { minv = cur; way[t] = r == i ? -1 : mate[r]; }
                }
                key = minv;
            }
            // block minimum of the distances of the unvisited columns
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { const long long ok = __shfl_xor_sync(0xffffffffu, key, o); key = ok < key ? ok : key; }
            if (lane == 0) s_rk[w] = key;
            __syncthreads();                     // (also: everybody has read s_nnew / rows_new)
            long long delta = s_rk[0];
#pragma unroll
            for (int k = 1; k < kSmallThreads / 32; ++k) delta = s_rk[k] < delta ? s_rk[k] : delta;
            // dual update: tree rows up, tree columns down, the other columns come closer
            const bool joins = t < n && !used && minv == delta;
            if (t < n) {
                if (used) { u[p[t]] += delta; v -= delta; }
                else minv -= delta;
            }
            if (t == 0) { u[i] += delta; s_jfree = INT_MAX; }
            // the columns at the minimum join the tree; their rows form the next list (positions by block prefix)
            const unsigned ball = __ballot_sync(0xffffffffu, joins && p[t] >= 0);
            if (lane == 0) s_wcnt[w] = __popc(ball);
            __syncthreads();                     // u[] settled, s_jfree reset, warp counts published
            if (joins) {
                used = true;
                if (p[t] < 0) atomicMin(&s_jfree, t);
                else {
                    int pos = __popc(ball & ((1u << lane) - 1));
                    for (int k = 0; k < w; ++k) pos += s_wcnt[k];
                    rows_new[pos] = p[t];
                }
            }
            if (t == 0) { int tot = 0; for (int k = 0; k < kSmallThreads / 32; ++k) tot += s_wcnt[k]; s_nnew = tot; }
            __syncthreads();
            if (s_jfree != INT_MAX) { jend = s_jfree; break; }   // a free column at this level: augment (smallest one)
        }
        // flip the alternating path (thread 0; a handful of steps)
        if (t == 0) {
            int j = jend;
            for (;;) {
                const int jp = way[j];
                const int r = jp < 0 ? i : p[jp];
                p[j] = r; mate[r] = j;
                if (jp < 0) break;
                j = jp;
            }
        }
        __syncthreads();
    }
    // ---- results ------------------------------------------------------------------------------------------------------
    long long part = 0;
    if (t < n) {
        const int j = mate[t];
        col_of_row_out[t] = j;
        part = c[t * n + j];
        if (x_out) x_out[size_t(t) * n + j] = 1;
        if (u_out) u_out[t] = u[t];
        if (v_out) v_out[t] = v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) s_rk[w] = part;
    __syncthreads();
    long long tot = 0;
    if (t == 0) {
        for (int k = 0; k < kSmallThreads / 32; ++k) tot += s_rk[k];
        *objective_out = tot;
    }
    return tot;
}

__global__ void __launch_bounds__(kSmallThreads)
assign_small_kernel(const int32_t *__restrict__ cost, int n, int32_t *col_of_row_out, long long *objective_out, uint8_t *x_out,
                    long long *u_out, long long *v_out, AsgCtrl *ctrl) {
    const long long tot = assign_small_solve(cost, n, col_of_row_out, objective_out, x_out, u_out, v_out);
    if (threadIdx.x == 0) { ctrl->objective = tot; ctrl->status = TD_OK; ctrl->phases = 1; }
}

// Batch: CTA b solves instance b (sizes[b] x sizes[b] at costs + offsets[b]) with the routine above.  Outputs have a stride
// of n_max; the slots past an instance's size hold col -1 and potentials 0.  An instance whose size or offset is out of
// range is withdrawn (objective INT64_MIN, every col -1) without touching its matrix.
__global__ void __launch_bounds__(kSmallThreads)
assign_batch_kernel(const int32_t *__restrict__ costs, const int32_t *__restrict__ sizes, const int64_t *__restrict__ offsets,
                    int n_max, int32_t *col_of_row_out, long long *objective_out, long long *u_out, long long *v_out) {
    const int b = blockIdx.x;
    const int n = sizes[b];
    const long long off = offsets[b];
    const size_t o = size_t(b) * n_max;
    const bool bad = n < 0 || n > n_max || off < 0 || (off & 3) != 0;
    const int keep = bad ? 0 : n;
    for (int t = keep + threadIdx.x; t < n_max; t += kSmallThreads) {
        col_of_row_out[o + t] = -1;
        if (u_out) u_out[o + t] = 0;
        if (v_out) v_out[o + t] = 0;
    }
    if (bad) {
        if (threadIdx.x == 0) objective_out[b] = LLONG_MIN;
        return;
    }
    assign_small_solve(costs + off, n, col_of_row_out + o, objective_out + b, nullptr, u_out ? u_out + o : nullptr,
                       v_out ? v_out + o : nullptr);
}

static AsgArgs carve_assign(void *ws, int n, size_t *bytes) {
    Carver c(ws);
    AsgArgs a;
    memset(&a, 0, sizeof a);
    const size_t nn = n > 0 ? n : 1;
    a.ctrl = c.take<AsgCtrl>(1);
    a.u = c.take<long long>(nn); a.v = c.take<long long>(nn); a.drow = c.take<long long>(nn);
    a.uinit = c.take<long long>(nn); a.vinit = c.take<long long>(nn);
    a.base0 = c.take<unsigned long long>(nn); a.stale = c.take<int32_t>(nn);
    a.distpred = c.take<unsigned long long>(nn);
    a.vmin = c.take<int32_t>(nn); a.mate_r = c.take<int32_t>(nn); a.mate_c = c.take<int32_t>(nn);
    a.root = c.take<int32_t>(nn); a.claim = c.take<int32_t>(nn); a.prop = c.take<int32_t>(nn); a.argcol = c.take<int32_t>(nn);
    a.frontier[0] = c.take<int32_t>(nn); a.frontier[1] = c.take<int32_t>(nn); a.sinks = c.take<int32_t>(nn);
    a.fbase[0] = c.take<long long>(nn); a.fbase[1] = c.take<long long>(nn);
    a.carry = c.take<int32_t>(nn); a.cbase = c.take<long long>(nn);
    a.settled = c.take<uint8_t>(nn);
    *bytes = c.used();
    return a;
}

}  // namespace td

extern "C" size_t td_assign_workspace_bytes(int n) {
    size_t b = 0;
    td::carve_assign(nullptr, n, &b);
    return b;
}

namespace td {

// 32 x 32 tiles through shared memory; used when the padding of a rectangular instance sits in the columns
__global__ void asg_transpose_kernel(const int32_t *__restrict__ in, int32_t *__restrict__ out, int n) {
    __shared__ int32_t tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = by + r, j = bx + threadIdx.x;
        if (i < n && j < n) tile[r][threadIdx.x] = in[size_t(i) * n + j];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = bx + r, j = by + threadIdx.x;
        if (i < n && j < n) out[size_t(i) * n + j] = tile[threadIdx.x][r];
    }
}

// row_of_col (the solution of the transposed instance) -> col_of_row and the reference's x vector
__global__ void asg_invert_kernel(const int32_t *__restrict__ row_of_col, int n, int32_t *__restrict__ col_of_row, uint8_t *x_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int i = row_of_col[j];
    if (i < 0 || i >= n) return;
    col_of_row[i] = j;
    if (x_out) x_out[size_t(i) * n + j] = 1;
}

static int assign_run(const int32_t *cost, int n, int nr, int32_t *col_of_row_out, int64_t *objective_out, uint8_t *x_out,
                      td_assign_stats *stats, void *workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace td

extern "C" int td_assign_exact(const int32_t *cost, int n, int32_t *col_of_row_out, int64_t *objective_out, uint8_t *x_out,
                               td_assign_stats *stats, void *workspace, size_t workspace_bytes, void *stream) {
    return td_assign_exact_rect(cost, n, n, n, col_of_row_out, objective_out, x_out, stats, workspace, workspace_bytes, stream);
}

extern "C" size_t td_assign_rect_workspace_bytes(int n, int n_real_rows, int n_real_cols) {
    size_t b = td_assign_workspace_bytes(n);
    if (n > 0 && n_real_cols < n && n_real_rows == n)   // transposed copy + the row-of-column result
        b += ((size_t(n) * n * 4 + 255) & ~size_t(255)) + ((size_t(n) * 4 + 255) & ~size_t(255));
    return b;
}

extern "C" int td_assign_exact_rect(const int32_t *cost, int n, int n_real_rows, int n_real_cols, int32_t *col_of_row_out,
                                    int64_t *objective_out, uint8_t *x_out, td_assign_stats *stats, void *workspace,
                                    size_t workspace_bytes, void *stream) {
    using namespace td;
    if (n < 0 || n >= (1 << kRowBits)) return TD_ERR_INVALID;
    if (n_real_rows < 0 || n_real_cols < 0 || n_real_rows > n || n_real_cols > n) return TD_ERR_INVALID;
    if (n > 0 && n_real_rows != n && n_real_cols != n) return TD_ERR_INVALID;   // n = max(real rows, real columns)
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n == 0 || n_real_cols == n)
        return assign_run(cost, n, n_real_rows, col_of_row_out, objective_out, x_out, stats, workspace, workspace_bytes, st);
    // padding columns: solve the transposed instance (its padding sits in the rows), then invert the matching
    if (stats) memset(stats, 0, sizeof *stats);
    if (!have_device()) return TD_ERR_NO_DEVICE;
    if (!cost || !col_of_row_out || !objective_out || !workspace) return TD_ERR_INVALID;
    if (workspace_bytes < td_assign_rect_workspace_bytes(n, n_real_rows, n_real_cols)) return TD_ERR_WORKSPACE;
    const size_t base_b = td_assign_workspace_bytes(n);
    char *wsp = static_cast<char *>(workspace);
    int32_t *cost_t = reinterpret_cast<int32_t *>(wsp + base_b);
    int32_t *row_of_col = reinterpret_cast<int32_t *>(wsp + base_b + ((size_t(n) * n * 4 + 255) & ~size_t(255)));
    asg_transpose_kernel<<<dim3((n + 31) / 32, (n + 31) / 32), dim3(32, 8), 0, st>>>(cost, cost_t, n);
    TD_LAUNCH_CHECK();
    const int rc = assign_run(cost_t, n, n_real_cols, row_of_col, objective_out, nullptr, stats, workspace, base_b, st);
    if (rc != TD_OK) return rc;
    if (x_out) TD_CUDA_TRY(cudaMemsetAsync(x_out, 0, size_t(n) * n, st));
    asg_invert_kernel<<<(n + 255) / 256, 256, 0, st>>>(row_of_col, n, col_of_row_out, x_out);
    TD_LAUNCH_CHECK();
    return TD_OK;
}

static int td::assign_run(const int32_t *cost, int n, int nr, int32_t *col_of_row_out, int64_t *objective_out, uint8_t *x_out,
                          td_assign_stats *stats, void *workspace, size_t workspace_bytes, cudaStream_t st) {
    using namespace td;
    if (n < 0 || n >= (1 << kRowBits)) return TD_ERR_INVALID;
    if (stats) memset(stats, 0, sizeof *stats);
    if (!have_device()) return TD_ERR_NO_DEVICE;
    if (n == 0) {
        if (objective_out) TD_CUDA_TRY(cudaMemsetAsync(objective_out, 0, sizeof(int64_t), st));
        return TD_OK;
    }
    if (!cost || !col_of_row_out || !objective_out || !workspace) return TD_ERR_INVALID;
    if (workspace_bytes < td_assign_workspace_bytes(n)) return TD_ERR_WORKSPACE;
    size_t bytes = 0;
    AsgArgs a = carve_assign(workspace, n, &bytes);
    a.cost = cost; a.n = n; a.col_of_row_out = col_of_row_out; a.objective_out = reinterpret_cast<long long *>(objective_out);
    a.x_out = x_out; a.max_phases = n + 8; a.nr = nr;
    a.deep_permille = 20;
    if (const char *e = getenv("TD_ASSIGN_DEEP")) a.deep_permille = atoi(e);
    if (const char *e = getenv("TD_ASSIGN_WIDE")) a.force_wide = atoi(e);
    a.prof = getenv("TD_ASSIGN_PROF") ? 1 : 0;
    a.greedy_rounds = kGreedyRounds;
    if (const char *e = getenv("TD_ASSIGN_GREEDY")) { const int v = atoi(e); if (v >= 1 && v <= 64) a.greedy_rounds = v; }
    a.carry_forest = 1;
    if (const char *e = getenv("TD_ASSIGN_CARRY")) a.carry_forest = atoi(e);
    a.carry_min_levels = 3;
    if (const char *e = getenv("TD_ASSIGN_CARRY_MIN")) a.carry_min_levels = atoi(e);
    TD_CUDA_TRY(cudaMemsetAsync(a.ctrl, 0, sizeof(AsgCtrl), st));
    if (x_out) TD_CUDA_TRY(cudaMemsetAsync(x_out, 0, size_t(n) * n, st));
    if (n <= kSmallN && nr == n && !getenv("TD_ASSIGN_NO_SMALL")) {   // balanced and small: one CTA in shared memory
        const size_t smem = small_smem_bytes(n);
        TD_CUDA_TRY(cudaFuncSetAttribute(assign_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        {
            ProfScope prof(TD_PROF_ASSIGN, st);
            assign_small_kernel<<<1, kSmallThreads, smem, st>>>(cost, n, col_of_row_out, a.objective_out, x_out, a.u, a.v, a.ctrl);
        }
        TD_LAUNCH_CHECK();
        if (stats) {
            AsgCtrl h;
            TD_CUDA_TRY(cudaMemcpyAsync(&h, a.ctrl, sizeof h, cudaMemcpyDeviceToHost, st));
            TD_CUDA_TRY(cudaStreamSynchronize(st));
            stats->objective = h.objective;
            stats->rows_scanned = n;          // the matrix is read from HBM once
            stats->phases = 1;
        }
        return TD_OK;
    }
    const bool vec = (n % 4 == 0) && ((reinterpret_cast<uintptr_t>(cost) & 15) == 0);
    void *kern = vec ? (void *)assign_kernel<true> : (void *)assign_kernel<false>;
    int per_sm = 0;
    const size_t dyn_smem = vec ? size_t(kAsgRingBytes) : 0;
    if (vec) {
        TD_CUDA_TRY(cudaFuncSetAttribute(assign_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(dyn_smem)));
        TD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, assign_kernel<true>, kAsgThreads, dyn_smem));
    } else {
        TD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, assign_kernel<false>, kAsgThreads, 0));
    }
    if (per_sm < 1) return TD_ERR_CUDA;
    per_sm = per_sm > 2 ? 2 : per_sm;
    int grid = device_sm_count() * per_sm;
    // small problems: fewer CTAs make grid.sync cheaper; keep at least one warp per 256-column tile and row
    const long long want_warps = (long long)((n + 255) / 256) * (n < 64 ? n : 64);
    const int need = int((want_warps * 32 + kAsgThreads - 1) / kAsgThreads);
    if (grid > need) grid = need < 1 ? 1 : need;
    void *args[] = {(void *)&a};
    {
        ProfScope prof(TD_PROF_ASSIGN, st);
        TD_CUDA_TRY(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(kAsgThreads), args, dyn_smem, st));
    }
    count_launch();
    if (stats) {
        AsgCtrl h;
        TD_CUDA_TRY(cudaMemcpyAsync(&h, a.ctrl, sizeof h, cudaMemcpyDeviceToHost, st));
        TD_CUDA_TRY(cudaStreamSynchronize(st));
        stats->objective = h.objective;
        // + the two init sweeps + the strided refreshes of cached level-0 minima (one cost cell each)
        stats->rows_scanned = int64_t(h.rows_scanned) + 2 * int64_t(n) + int64_t(h.stale_cells / (unsigned long long)n);
        stats->auction_rounds = a.greedy_rounds;
        stats->phases = int32_t(h.phases);
        stats->search_steps = int32_t(h.levels);
        stats->augmentations = int32_t(h.augment);
        stats->unassigned_after_auction = int32_t(h.free_after_init);
        if (getenv("TD_ASSIGN_PROF"))
            fprintf(stderr, "[td_assign] us: scan %.0f sync1 %.0f settle %.0f sync2 %.0f phase_start %.0f augment %.0f\n",
                    h.t_prof[0] / 1e3, h.t_prof[1] / 1e3, h.t_prof[2] / 1e3, h.t_prof[3] / 1e3, h.t_prof[4] / 1e3, h.t_prof[5] / 1e3);
        if (getenv("TD_ASSIGN_PROF"))
            fprintf(stderr, "[td_assign] phase start us: reset + lists %.0f, stale detection %.0f, stale refresh %.0f (%.1f M cells), cache -> distances %.0f\n",
                    h.t_prof[16] / 1e3, h.t_prof[17] / 1e3, h.t_prof[18] / 1e3, h.stale_cells / 1e6, h.t_prof[4] / 1e3);
        if (getenv("TD_ASSIGN_PROF"))
            fprintf(stderr, "[td_assign] max|c| %llu, 32-bit relaxation sweeps %llu of %u\n", h.cabs, h.narrow_levels, h.levels);
        if (getenv("TD_ASSIGN_PROF"))
            fprintf(stderr, "[td_assign] init us: column-min sweep %.0f, row-min sweep %.0f\n", h.t_prof[6] / 1e3, h.t_prof[7] / 1e3);
        if (getenv("TD_ASSIGN_PROF"))
            fprintf(stderr, "[td_assign] scan us by frontier size <=32: %.0f (%llu levels)  <=256: %.0f (%llu)  <=2048: %.0f (%llu)  >2048: %.0f (%llu)\n",
                    h.t_prof[8] / 1e3, h.t_prof[12], h.t_prof[9] / 1e3, h.t_prof[13], h.t_prof[10] / 1e3, h.t_prof[14],
                    h.t_prof[11] / 1e3, h.t_prof[15]);
        if (h.status != TD_OK) return h.status;
    }
    return TD_OK;
}

extern "C" int td_assign_exact_batch(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                                     int32_t *col_of_row_out, int64_t *objective_out, int64_t *u_out, int64_t *v_out,
                                     void *stream) {
    using namespace td;
    if (batch < 0 || n_max < 0 || n_max > TD_BATCH_MAX_N) return TD_ERR_INVALID;
    if (batch == 0) return TD_OK;
    if (!costs || !sizes || !offsets || !col_of_row_out || !objective_out) return TD_ERR_INVALID;
    if ((reinterpret_cast<uintptr_t>(costs) & 15) != 0) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t smem = small_smem_bytes(n_max);
    TD_CUDA_TRY(cudaFuncSetAttribute(assign_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    assign_batch_kernel<<<batch, kSmallThreads, smem, st>>>(costs, sizes, offsets, n_max, col_of_row_out,
                                                            reinterpret_cast<long long *>(objective_out),
                                                            reinterpret_cast<long long *>(u_out),
                                                            reinterpret_cast<long long *>(v_out));
    TD_LAUNCH_CHECK();
    return TD_OK;
}

// ---- optimality certificate -----------------------------------------------------------------------------------------
// The solver ends with dual potentials u (rows) and v (columns) that prove its matching optimal (complementary slackness):
//   c[i][j] - u[i] - v[j] >= 0 on the real block, == 0 on the matched real cells, and -- for an unbalanced instance --
//   the potentials of the side that has spare members are <= 0 and == 0 on the members no real partner uses.
// Then  sum u + sum v  is a lower bound of every assignment and equals the cost of this one.  td_assign_read_duals hands
// the potentials out of the workspace of the last solve; td_assign_certify checks the conditions with ONE sweep over the
// cost matrix (1.6 GB at n = 20 000) -- the replacement for re-solving with an independent exact solver (scipy needs
// minutes at that size).  Reference semantics being certified: solver.py:11-27 (min sum c x, row and column sums = 1).
namespace td {

__global__ void __launch_bounds__(256)
assign_certify_kernel(const int32_t *__restrict__ cost, int n, int nr, int nc, const int32_t *__restrict__ col_of_row,
                      const long long *__restrict__ u, const long long *__restrict__ v, td_assign_certificate *out) {
    const int lane = threadIdx.x & 31;
    const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    long long mn = LLONG_MAX, tight = 0, dual = 0, primal = 0;
    int bad = 0;
    for (int i = gwarp; i < nr; i += nwarps) {
        const long long ui = u[i];
        const int32_t *row = cost + size_t(i) * n;
        for (int j = lane; j < nc; j += 32) {
            const long long red = (long long)__ldg(row + j) - ui - v[j];
            mn = red < mn ? red : mn;
        }
        if (lane == 0) {
            dual += ui;
            const int j = col_of_row[i];
            if (j >= 0 && j < nc) {
                const long long red = (long long)row[j] - ui - v[j];
                const long long ab = red < 0 ? -red : red;
                tight = ab > tight ? ab : tight;
                primal += row[j];
            } else {
                bad += (ui != 0);             // a real row without a real column (spare rows): its potential must be 0
            }
            if (nc < n) bad += (ui > 0);      // spare rows exist: row potentials are <= 0
        }
    }
    // column side: potentials of the real columns, sign / zero conditions when there are spare columns
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nc; j += gridDim.x * blockDim.x) {
        dual += v[j];
        if (nr < n) bad += (v[j] > 0);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long m2 = __shfl_xor_sync(0xffffffffu, mn, o); mn = m2 < mn ? m2 : mn;
        const long long t2 = __shfl_xor_sync(0xffffffffu, tight, o); tight = t2 > tight ? t2 : tight;
        dual += __shfl_xor_sync(0xffffffffu, dual, o);
        primal += __shfl_xor_sync(0xffffffffu, primal, o);
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
    }
    if (lane == 0) {
        atomicMin(reinterpret_cast<long long *>(&out->min_reduced_cost), mn);
        atomicMax(reinterpret_cast<long long *>(&out->max_matched_slack), tight);
        atomicAdd(reinterpret_cast<unsigned long long *>(&out->dual_objective), (unsigned long long)dual);
        atomicAdd(reinterpret_cast<unsigned long long *>(&out->matched_real_cost), (unsigned long long)primal);
        if (bad) atomicAdd(&out->sign_violations, bad);
    }
}

// spare columns (nr < n): a real column no real row uses must have potential 0
__global__ void assign_certify_cols_kernel(int n, int nr, int nc, const int32_t *__restrict__ col_of_row,
                                           const long long *__restrict__ v, uint8_t *used, td_assign_certificate *out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < nr) { const int j = col_of_row[t]; if (j >= 0 && j < nc) used[j] = 1; }
}
__global__ void assign_certify_cols2_kernel(int nc, const long long *__restrict__ v, const uint8_t *used,
                                            td_assign_certificate *out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nc && !used[j] && v[j] != 0) atomicAdd(&out->sign_violations, 1);
}

__global__ void assign_cert_init_kernel(td_assign_certificate *out) {
    out->min_reduced_cost = LLONG_MAX; out->max_matched_slack = 0; out->dual_objective = 0; out->matched_real_cost = 0;
    out->sign_violations = 0; out->reserved = 0;
}

}  // namespace td

extern "C" int td_assign_read_duals(const void *workspace, int n, int n_real_rows, int n_real_cols, int64_t *u_out,
                                    int64_t *v_out, void *stream) {
    using namespace td;
    if (n < 0 || !workspace || !u_out || !v_out || n_real_rows > n || n_real_cols > n) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    if (n == 0) return TD_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    size_t bytes = 0;
    const AsgArgs a = carve_assign(const_cast<void *>(workspace), n, &bytes);
    // padding columns: the instance was solved transposed, its rows are the caller's columns
    const bool transposed = n_real_cols < n && n_real_rows == n;
    TD_CUDA_TRY(cudaMemcpyAsync(u_out, transposed ? a.v : a.u, size_t(n) * 8, cudaMemcpyDeviceToDevice, st));
    TD_CUDA_TRY(cudaMemcpyAsync(v_out, transposed ? a.u : a.v, size_t(n) * 8, cudaMemcpyDeviceToDevice, st));
    return TD_OK;
}

extern "C" size_t td_assign_certify_workspace_bytes(int n) { return size_t(n > 0 ? n : 1) + 256; }

extern "C" int td_assign_certify(const int32_t *cost, int n, int n_real_rows, int n_real_cols, const int32_t *col_of_row,
                                 const int64_t *u, const int64_t *v, td_assign_certificate *cert_out /* device */,
                                 void *workspace, size_t workspace_bytes, void *stream) {
    using namespace td;
    if (n < 0 || n_real_rows < 0 || n_real_cols < 0 || n_real_rows > n || n_real_cols > n || !cert_out) return TD_ERR_INVALID;
    if (!have_device()) return TD_ERR_NO_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    assign_cert_init_kernel<<<1, 1, 0, st>>>(cert_out);
    TD_LAUNCH_CHECK();
    if (n == 0 || n_real_rows == 0 || n_real_cols == 0) return TD_OK;
    if (!cost || !col_of_row || !u || !v || !workspace || workspace_bytes < td_assign_certify_workspace_bytes(n)) return TD_ERR_INVALID;
    const int grid = device_sm_count() * 8;
    assign_certify_kernel<<<grid, 256, 0, st>>>(cost, n, n_real_rows, n_real_cols, col_of_row,
                                                reinterpret_cast<const long long *>(u), reinterpret_cast<const long long *>(v), cert_out);
    TD_LAUNCH_CHECK();
    if (n_real_rows < n) {
        uint8_t *used = static_cast<uint8_t *>(workspace);
        TD_CUDA_TRY(cudaMemsetAsync(used, 0, size_t(n), st));
        assign_certify_cols_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, n_real_rows, n_real_cols, col_of_row,
                                                                    reinterpret_cast<const long long *>(v), used, cert_out);
        TD_LAUNCH_CHECK();
        assign_certify_cols2_kernel<<<(n + 255) / 256, 256, 0, st>>>(n_real_cols, reinterpret_cast<const long long *>(v), used, cert_out);
        TD_LAUNCH_CHECK();
    }
    return TD_OK;
}
