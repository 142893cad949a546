/*
 * taxidispatch.h -- C ABI of libtaxidispatch.so, the B200 (sm_100a) dispatch engine.
 *
 * The reference (boguszjelinski/taxidispatcher) has no FFI: its boundary for this path is the
 * Python-level function surface plus two file/CLI protocols (SURVEY.md section 8(b)).  Each
 * entry point below names the reference interface it replaces.  INTEGRATION.md shows the
 * bindings a reference maintainer would add (ctypes for the Python scripts, JNI for
 * Simulator.java, a pool_n-compatible CLI for findpool.c).
 *
 * Conventions
 *   - plain C: pointers and sizes only, no C++/torch types.
 *   - td_*  (device entry points): every data pointer is a DEVICE pointer into caller-owned
 *     memory; `stream` is a cudaStream_t passed as void* (NULL = default stream).  The call is
 *     asynchronous on `stream` unless a HOST out-parameter (marked "host") is non-NULL, in which
 *     case the stream is synchronised before returning.  Scratch memory is caller-provided and
 *     sized by the matching td_*_workspace_bytes() query; nothing is allocated behind the
 *     caller's back, there is no global mutable state and calls on different streams with
 *     different workspaces are independent.
 *   - tdh_* (host entry points): same operations on HOST buffers; they allocate device memory,
 *     copy in, run, copy out and free.  These are what a cgo/JNI/ctypes stub binds when the
 *     caller has no device memory of its own.
 *   - every function returns TD_OK (0) or a negative TD_ERR_* code; nothing ever calls exit()
 *     (the reference does: pool_n.c:36-39,68-71, findpool.c:166-169).
 *   - there is no CPU fallback: without a CUDA device every compute call returns
 *     TD_ERR_NO_DEVICE.
 */
#ifndef TAXIDISPATCH_H
#define TAXIDISPATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TD_OK 0
#define TD_ERR_INVALID (-1)    /* bad argument */
#define TD_ERR_CUDA (-2)       /* a CUDA call failed; see td_last_cuda_error() */
#define TD_ERR_WORKSPACE (-3)  /* workspace smaller than td_*_workspace_bytes() */
#define TD_ERR_CAPACITY (-4)   /* an output / intermediate capacity was exceeded; stats say by how much */
#define TD_ERR_NO_DEVICE (-5)  /* no usable CUDA device */
#define TD_ERR_NOT_CONVERGED (-6)

#define TD_BIG_COST 250000     /* split.py:5, simulate.py:13, Simulator.java:114 */
#define TD_POOL_REC_W 9        /* pool_n.c:26: 4 pickups + 4 drop-offs + cost at column 8 */
#define TD_POOL_MAX_IN_POOL 4  /* pool_n.c:12 */
#define TD_POOL_REF_SHARDS 8   /* pool_n.c:13 MAX_THREAD */
#define TD_POOL_MAX_CUSTOMERS 16384

const char *td_version(void);
const char *td_strerror(int code);
/* text of the last CUDA error seen by the calling thread ("" if none) */
const char *td_last_cuda_error(void);
/* number of visible CUDA devices, or TD_ERR_NO_DEVICE */
int td_device_count(void);
/* kernels launched by this library on the calling thread since the last td_launch_count_reset() */
int64_t td_launch_count(void);
void td_launch_count_reset(void);

/* Optional per-kernel device timing (CUDA events recorded on the launching stream around the
 * dominant kernel of each operation).  Off by default; used by bench.py for the roofline figure. */
#define TD_PROF_COST 0        /* cost_matrix_kernel */
#define TD_PROF_LCM 1         /* lcm_rounds_kernel */
#define TD_PROF_ASSIGN 2      /* assign_kernel */
#define TD_PROF_POOL_ENUM 3   /* pool_enum_kernel */
#define TD_PROF_POOL_SELECT 4 /* pool_select_kernel */
#define TD_PROF_KINDS 5
void td_prof_enable(int on);
void td_prof_reset(void);
/* waits for the recorded events; total_ms = sum of durations, count = launches */
int td_prof_read(int kind, double *total_ms, int64_t *count);

/* ------------------------------------------------------------------------------------------
 * K1  cost matrix            replaces calculate_cost(distances, demand, cabs)
 *     split.py:123-136 (= greedy_opt.py:86-99), cutoff variant simulate.py:17-33 and
 *     Simulator.java:493-520; fill n*n variant procedure.py:6-12.
 *
 * n = max(n_cabs, n_cust).  cost_out[i*n + j] = dist[cab_to[i]*n_stands + cust_from[j]] for
 * i < n_cabs, j < n_cust (and, when cutoff >= 0, only if that distance < cutoff); `fill`
 * everywhere else.  cab_to / cust_from are POSITIONAL (split.py:128-134).
 * ------------------------------------------------------------------------------------------ */
int td_cost_matrix(const int32_t *dist, int n_stands,
                   const int32_t *cab_to, int n_cabs,
                   const int32_t *cust_from, int n_cust,
                   int32_t fill, int32_t cutoff /* < 0: none */,
                   int32_t *cost_out /* n*n */, void *stream);

/* Rows [row_begin, row_begin + row_count) of the same matrix, written to a row_count x n buffer: the multi-GPU path
 * builds contiguous cab-row blocks per device (the loop of split.py:129-134 / Simulator.java:503-511 has no carried
 * state, so rows split trivially). */
int td_cost_matrix_rows(const int32_t *dist, int n_stands,
                        const int32_t *cab_to, int n_cabs,
                        const int32_t *cust_from, int n_cust,
                        int32_t fill, int32_t cutoff /* < 0: none */,
                        int row_begin, int row_count,
                        int32_t *cost_out /* row_count*n */, void *stream);

/* ------------------------------------------------------------------------------------------
 * K3  LCM greedy             replaces LCM(...) in heuristic.py:24-33, split.py:161-175,
 *     greedy_opt.py:61-82, simulate.py:76-97 and Simulator.LCM (Simulator.java:523-549).
 *
 * Repeats up to max_iters (<0: n) times: e = FIRST index of the minimum of the n*n working
 * array; stop rules are tested on that minimum; record (e / n, e % n); overwrite that row and
 * column with mask_value.  The mask is a value: masked cells still take part in the argmin
 * (SURVEY.md section 4 trap 4) -- results are bit-identical to the literal array algorithm.
 * A 0-row call runs no iteration: n_pairs 0, total 0 and last_min INT32_MAX.
 * ------------------------------------------------------------------------------------------ */
typedef struct td_lcm_params {
    int32_t mask_value;    /* heuristic.py:32 -> 100; split.py:173 / Simulator.java:541 -> big_cost */
    int32_t stop_above;    /* break before recording when min >  stop_above (greedy_opt.py:69);  INT32_MAX: never */
    int32_t stop_at_value; /* break before recording when min >= stop_at_value (Simulator.java:538); INT32_MAX: never */
    int32_t sum_below;     /* add min to the total only when min < sum_below (split.py:167);      INT32_MAX: always */
    int32_t residual_size; /* break after recording when n - picks == residual_size (Simulator.java:545); 0: never */
    int32_t max_iters;     /* < 0: n */
} td_lcm_params;

size_t td_lcm_workspace_bytes(int n);
int td_lcm(const int32_t *cost, int n, const td_lcm_params *params /* host */,
           int32_t *rows_out /* n */, int32_t *cols_out /* n */,
           int32_t *n_pairs_out /* 1 */, int64_t *total_out /* 1 */, int32_t *last_min_out /* 1, may be NULL */,
           void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * K2  exact balanced assignment     replaces the model build + cvxopt.glpk.ilp call of
 *     solver.py:11-27, python.py:6-25, procedure.py:14-29, split.py:139-155, heuristic.py:37.
 *
 * Minimises sum cost[i*n+j] over permutations.  col_of_row_out[i] = customer column of cab row
 * i; x_out (optional) is the reference solution vector, x[n*cab + cust] in {0,1}
 * (procedure.py:56, split.py:23, Simulator.java:380).  The objective is exact (int64).
 * ------------------------------------------------------------------------------------------ */
typedef struct td_assign_stats {
    int64_t objective;
    int64_t rows_scanned;   /* cost rows read by bidding / path-search sweeps (x 4n bytes each) */
    int32_t auction_rounds;
    int32_t phases;         /* augmentation phases of the exact finish */
    int32_t search_steps;   /* grid-wide frontier steps inside those phases */
    int32_t augmentations;
    int32_t unassigned_after_auction;
    int32_t reserved;
} td_assign_stats;

size_t td_assign_workspace_bytes(int n);
int td_assign_exact(const int32_t *cost, int n,
                    int32_t *col_of_row_out /* n */, int64_t *objective_out /* 1 */,
                    uint8_t *x_out /* n*n or NULL */, td_assign_stats *stats /* host, may be NULL */,
                    void *workspace, size_t workspace_bytes, void *stream);

/* Unbalanced-native variant (SURVEY.md 8(f)-4).  Every real call of the reference is unbalanced: the cost
 * matrix is padded to n = max(cabs, customers) with constant `big_cost` rows or columns (split.py:123-136,
 * Simulator.java:493-520; simulog_solv.txt: supply 600 vs demand 218-368).  cost is still that padded n x n
 * matrix and all outputs keep the padded layout, but only the real rows / columns are searched: rows
 * n_real_rows..n-1 (or columns n_real_cols..n-1) MUST be constant, they receive the leftover columns (rows) in
 * index order.  The objective equals td_assign_exact's.  One of n_real_rows, n_real_cols must be n. */
size_t td_assign_rect_workspace_bytes(int n, int n_real_rows, int n_real_cols);
int td_assign_exact_rect(const int32_t *cost, int n, int n_real_rows, int n_real_cols,
                         int32_t *col_of_row_out /* n */, int64_t *objective_out /* 1 */,
                         uint8_t *x_out /* n*n or NULL */, td_assign_stats *stats /* host, may be NULL */,
                         void *workspace, size_t workspace_bytes, void *stream);

/* Optimality certificate.  The solver ends with dual potentials u (per cab row) and v (per customer column) that
 * prove its matching optimal by complementary slackness: cost[i][j] - u[i] - v[j] >= 0 on the real block and == 0 on
 * the matched real cells; with spare (padding) rows or columns the potentials of the side that has spare members are
 * <= 0 and == 0 where no real partner is matched.  sum u + sum v is then a lower bound of every assignment and equals
 * the cost of this one.  td_assign_read_duals copies the potentials out of the workspace of the LAST solve (device
 * int64[n] each); td_assign_certify evaluates the conditions with one sweep over the matrix and fills a DEVICE struct.
 * This is what checks the exact optimum where an independent solver is too slow (scipy: minutes at n = 20 000).
 * Certified semantics: solver.py:11-27 (min sum c x, every row and column sum = 1); invariant heuristic.py:40. */
typedef struct td_assign_certificate {
    int64_t min_reduced_cost;   /* min over the real block of cost - u - v          (must be >= 0) */
    int64_t max_matched_slack;  /* max over matched real cells of |cost - u - v|    (must be == 0) */
    int64_t dual_objective;     /* sum of u over real rows + sum of v over real columns */
    int64_t matched_real_cost;  /* cost of the matched real cells                   (must equal dual_objective) */
    int32_t sign_violations;    /* potentials with the wrong sign / nonzero on unused spare members (must be 0) */
    int32_t reserved;
} td_assign_certificate;
int td_assign_read_duals(const void *workspace, int n, int n_real_rows, int n_real_cols,
                         int64_t *u_out /* n */, int64_t *v_out /* n */, void *stream);
size_t td_assign_certify_workspace_bytes(int n);
int td_assign_certify(const int32_t *cost, int n, int n_real_rows, int n_real_cols, const int32_t *col_of_row,
                      const int64_t *u, const int64_t *v, td_assign_certificate *cert_out /* device */,
                      void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * Batches of small independent instances     replace the per-instance loops of heuristic.py:20-40
 *     (1000 random 100 x 100 cases, each through LCM and the exact solver) and python.py:6-25.
 *
 * One launch per call, one CTA per instance; the instance sits in shared memory, so sizes are
 * limited to TD_BATCH_MAX_N.  Instance b is sizes[b] x sizes[b] row-major int32 at
 * costs + offsets[b] (elements, a multiple of 4); costs is 16-byte aligned; sizes / offsets are
 * DEVICE arrays; outputs use a stride of n_max per instance (slots past an instance's result hold
 * -1, potentials 0).  Always asynchronous, no workspace.  An instance with size < 0 or > n_max, or
 * an offset < 0 or not a multiple of 4, is withdrawn (objective / total INT64_MIN, n_pairs -1,
 * last_min INT32_MIN, every col / row -1); the other instances are unaffected.  A size-0 instance
 * has objective 0 and 0 pairs.
 *
 * td_assign_exact_batch runs the same routine as td_assign_exact does for a balanced n <= 232
 * matrix, so both return the identical col_of_row; u_out / v_out (optional) are the dual
 * potentials (see td_assign_certificate below).  td_lcm_batch runs the literal array algorithm
 * of td_lcm with the same params for every instance and returns the same trace.
 * ------------------------------------------------------------------------------------------ */
#define TD_BATCH_MAX_N 232     /* 232^2 x 4 B = 210 KB of the 227 KB of shared memory of one CTA */
int td_assign_exact_batch(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                          int32_t *col_of_row_out /* batch x n_max */, int64_t *objective_out /* batch */,
                          int64_t *u_out /* batch x n_max or NULL */, int64_t *v_out /* batch x n_max or NULL */,
                          void *stream);
int td_lcm_batch(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                 const td_lcm_params *params /* host, same for every instance */,
                 int32_t *rows_out /* batch x n_max */, int32_t *cols_out /* batch x n_max */,
                 int32_t *n_pairs_out /* batch */, int64_t *total_out /* batch */,
                 int32_t *last_min_out /* batch, may be NULL */, void *stream);

/* ------------------------------------------------------------------------------------------
 * Batches of mid-size instances (n <= TD_BATCH_CLUSTER_MAX_N)   the paper's 400 x 400 split /
 *     hybrid experiment (split.py:186-212, greedy_opt.py:129-163) and Simulator.java's
 *     MAX_NON_LCM = 600 solver limit, over many instances.
 *
 * Exactly the arguments, layout and semantics of td_assign_exact_batch / td_lcm_batch above
 * (packed instances, output stride n_max, -1 / 0 fill, withdrawal of an instance with a bad size or
 * offset, batch == 0 launches nothing), for n_max up to 640.  One launch per call; every instance
 * runs on one thread-block cluster of K CTAs (K = 1, 2, 4 or 8, the smallest whose share of the
 * matrix fits one CTA's shared memory; it depends on n_max only) that holds the instance in its
 * distributed shared memory.  Returns TD_ERR_CUDA when no such cluster fits the device.
 *
 * td_assign_exact_batch_cluster runs the algorithm of td_assign_exact_batch step for step: for
 * every n <= 232 it returns the identical col_of_row, u, v and objective, and for any n the result
 * does not depend on n_max or on the instance's position in the batch.  td_lcm_batch_cluster
 * returns the literal trace of td_lcm for every params.
 * ------------------------------------------------------------------------------------------ */
#define TD_BATCH_CLUSTER_MAX_N 640   /* 8 CTAs x (640/8) x 640 x 4 B = 8 x 200 KB of shared memory */
int td_assign_exact_batch_cluster(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                                  int32_t *col_of_row_out /* batch x n_max */, int64_t *objective_out /* batch */,
                                  int64_t *u_out /* batch x n_max or NULL */, int64_t *v_out /* batch x n_max or NULL */,
                                  void *stream);
int td_lcm_batch_cluster(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                         const td_lcm_params *params /* host, same for every instance */,
                         int32_t *rows_out /* batch x n_max */, int32_t *cols_out /* batch x n_max */,
                         int32_t *n_pairs_out /* batch */, int64_t *total_out /* batch */,
                         int32_t *last_min_out /* batch, may be NULL */, void *stream);

/* ------------------------------------------------------------------------------------------
 * Batches of large instances (n <= TD_BATCH_LARGE_MAX_N)   heuristic.py's 2000 x 2000 LCM-vs-
 *     optimum experiment, Simulator.java's 1300-row LCM model and perf.jl's 1000 x 1000 solve,
 *     over many instances.
 *
 * Exactly the arguments, layout and semantics of the *_batch_cluster pair above (packed
 * instances, output stride n_max, -1 / 0 fill, withdrawal of an instance with a bad size or
 * offset, batch == 0 launches nothing, no workspace, always asynchronous), for 0 <= n_max <= 2048,
 * small n_max included.  One launch per call; every instance runs on one thread-block cluster of
 * K CTAs (K = 4 up to n_max 1024, 8 above: at most 256 columns / rows per CTA, one per thread)
 * that keeps only the O(n) state in shared memory and reads the matrix from global memory.
 * Returns TD_ERR_CUDA when no such cluster fits the device.
 *
 * The same algorithms as the *_batch_cluster pair, step for step: td_assign_exact_batch_large
 * returns, for every instance of n <= 640, the identical col_of_row, u, v and objective as
 * td_assign_exact_batch_cluster (and for n <= 232 as td_assign_exact_batch), an exact optimum with
 * valid duals for every n, and results that do not depend on n_max or on the position in the
 * batch.  td_lcm_batch_large returns the literal trace of td_lcm for every params.
 * ------------------------------------------------------------------------------------------ */
#define TD_BATCH_LARGE_MAX_N 2048    /* 8 CTAs x 256 columns / rows: one per thread */
int td_assign_exact_batch_large(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                                int32_t *col_of_row_out /* batch x n_max */, int64_t *objective_out /* batch */,
                                int64_t *u_out /* batch x n_max or NULL */, int64_t *v_out /* batch x n_max or NULL */,
                                void *stream);
int td_lcm_batch_large(const int32_t *costs, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                       const td_lcm_params *params /* host, same for every instance */,
                       int32_t *rows_out /* batch x n_max */, int32_t *cols_out /* batch x n_max */,
                       int32_t *n_pairs_out /* batch */, int64_t *total_out /* batch */,
                       int32_t *last_min_out /* batch, may be NULL */, void *stream);

/* ------------------------------------------------------------------------------------------
 * K4  pool finder          replaces one `pool_n <pool-size> <thread> <file> <n> <out>` process
 *     (pool_n.c:209-238): findPool :153-177, drop_customers :101-151, removeDuplicates :187-207,
 *     shard rule :226-229.
 *
 * demand: n x 5 int32 rows (id, from, to, maxWait, maxLoss) as pool_n.c:20; dist: n_stands^2.
 * plans_out rows use the in-memory record of pool_n.c:123-134: [p0..p{k-1}, drop-off customers
 * in drop order, zero padding, cost at column 8]; values are ROW INDICES into `demand`.
 * Survivors are written in (cost, enumeration rank) order, i.e. the order of out<thread>.csv.
 * Limits: n <= TD_POOL_MAX_CUSTOMERS; with pool_size 4 every stand distance must be <= 2^22 (the 24 drop-off orders
 * are evaluated in a x32 fixed point) -- larger tables return TD_ERR_INVALID (asynchronous calls: count -1).
 * ------------------------------------------------------------------------------------------ */
typedef struct td_pool_stats {
    int64_t evaluated;  /* pool_n.c:103 count_all: leaf plans = (pickup tuple, drop-off permutation) */
    int64_t feasible;   /* pool_n.c:135 pool_count */
    int64_t kept;       /* pool_n.c:237 good_count */
    int32_t rounds;     /* dominance rounds of the parallel greedy selection */
    int32_t passes;     /* enumeration passes (1 unless the feasible list had to be chunked) */
} td_pool_stats;

size_t td_pool_workspace_bytes(int n, int n_stands, int pool_size, int64_t max_feasible);
int td_pool_find(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                 int shard, int n_shards /* reference: 8 */,
                 int32_t *plans_out /* cap x 9 */, int32_t cap, int32_t *n_plans_out /* 1 */,
                 td_pool_stats *stats /* host, may be NULL */,
                 void *workspace, size_t workspace_bytes, int64_t max_feasible, void *stream);

/* Several CONSECUTIVE logical shards [shard_begin, shard_begin + shard_count) in one call (shard_count <= 64):
 * one enumeration launch and one selection launch serve all of them (the shards stay independent --
 * each keeps its own dedup state, exactly like separate pool_n processes).  plans_out holds
 * shard_count blocks of `cap` rows, counts_out[s] the survivors of shard shard_begin + s (-1 if the
 * record list overflowed); stats is a HOST array of shard_count entries (may be NULL). */
size_t td_pool_shards_workspace_bytes(int n, int n_stands, int pool_size, int shard_count, int64_t max_feasible);
int td_pool_find_shards(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                        int shard_begin, int shard_count, int n_shards,
                        int32_t *plans_out /* shard_count x cap x 9 */, int32_t cap, int32_t *counts_out /* shard_count */,
                        td_pool_stats *stats /* host[shard_count], may be NULL */,
                        void *workspace, size_t workspace_bytes, int64_t max_feasible /* all shards together */,
                        void *stream);

/* ------------------------------------------------------------------------------------------
 * 2-passenger pool of the Simulator      replaces Simulator.findPool (Simulator.java:681-758; pool.c:64-131)
 *
 * Customers are given by their from / to stands (from[i] < 0 marks a removed row, Simulator.java:688).
 * Every ordered pair (A picked up first, then B) is a candidate; the cheaper of the two drop orders
 * is its plan (pairs_out plan column: 1 = B ends / CLNT_B_ENDS, 0 = A ends).  accept_all != 0 keeps
 * every pair -- the Simulator's actual behaviour (plan1 = plan2 = true at :691); accept_all == 0 applies
 * the loss tests as written (:701-707) with max_loss (1.01).  Stable sort by cost, greedy disjoint scan.
 * pairs_out rows: [custA, custB, plan, cost] in scan order.
 * ------------------------------------------------------------------------------------------ */
size_t td_pool_pairs_workspace_bytes(int n);
int td_pool_pairs(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                  int accept_all, double max_loss,
                  int32_t *pairs_out /* cap x 4 */, int32_t cap, int32_t *n_pairs_out /* 1 */,
                  void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * Exact 2-passenger pool, batched: minimum-cost maximum-cardinality pair matching
 * (the optimum pool_optimum.py / pool_opt_min.py ask for; greedy counterpart: td_pool_pairs)
 *
 * Instance b has sizes[b] customers at from[offsets[b]..], to[offsets[b]..] (from < 0: removed row); the stand
 * table dist (n_stands x n_stands, n_stands <= 128, every entry in [0, 2^22]) is shared by the whole batch.  The
 * pair {i, j} is an edge when td_pool_pairs would accept (i, j) or (j, i); its row [custA, custB, plan, cost] is the
 * accepted candidate smallest in (cost, A*n+B).  Among the matchings of maximum cardinality, one of minimum total
 * cost is returned: pairs_out[b] holds its rows in (cost, A*n+B) order (n_max/2 rows per instance, unused rows -1),
 * n_pairs_out[b] their count and cost_out[b] their total.  Which optimum comes back when several exist is not
 * specified, but it depends on nothing but the instance: not on its position, its neighbours or n_max.
 *
 * One CTA per instance, one launch.  An instance with sizes[b] < 0 or > n_max, offsets[b] < 0 or a live row whose
 * stand lies outside the table is withdrawn (n_pairs -1, cost INT64_MIN, rows -1); a table entry outside
 * [0, 2^22] withdraws every instance.  The arguments are checked before anything else: TD_ERR_INVALID for batch < 0,
 * n_max outside [0, TD_PAIRS_EXACT_MAX_N], a bad n_stands, a non-finite max_loss with accept_all == 0 or a NULL
 * pointer with batch > 0; TD_ERR_WORKSPACE for a workspace smaller than td_pool_pairs_exact_workspace_bytes.
 * ------------------------------------------------------------------------------------------ */
#define TD_PAIRS_EXACT_MAX_N 4096
size_t td_pool_pairs_exact_workspace_bytes(int batch, int n_max);
int td_pool_pairs_exact_batch(const int32_t *from, const int32_t *to, const int32_t *sizes, const int64_t *offsets,
                              int batch, int n_max, const int32_t *dist, int n_stands, int accept_all, double max_loss,
                              int32_t *pairs_out /* batch x (n_max/2) x 4 */, int32_t *n_pairs_out /* batch */,
                              int64_t *cost_out /* batch */, void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * Greedy 2-passenger pool, batched: td_pool_pairs over many instances in one launch
 *
 * Arguments, layout, argument checks, withdrawal and return codes are those of td_pool_pairs_exact_batch above, without
 * the workspace (one CTA per instance, everything in shared memory).  pairs_out[b] holds exactly the rows
 * [custA, custB, plan, cost] that td_pool_pairs returns for instance b with the same dist / accept_all / max_loss, in
 * its scan order; n_pairs_out[b] is their count and cost_out[b] their total; unused rows are -1.  The greedy under the
 * strict order (cost, A*n+B) has one answer, so it depends on nothing but the instance.  Unlike td_pool_pairs, an
 * instance holds at most TD_PAIRS_BATCH_MAX_N customers and every table entry must lie in [0, 2^22].
 * ------------------------------------------------------------------------------------------ */
#define TD_PAIRS_BATCH_MAX_N 4096
int td_pool_pairs_batch(const int32_t *from, const int32_t *to, const int32_t *sizes, const int64_t *offsets,
                        int batch, int n_max, const int32_t *dist, int n_stands, int accept_all, double max_loss,
                        int32_t *pairs_out /* batch x (n_max/2) x 4 */, int32_t *n_pairs_out /* batch */,
                        int64_t *cost_out /* batch */, void *stream);

/* ------------------------------------------------------------------------------------------
 * The whole findpool job, batched: td_pool_find_shards over every logical shard + td_pool_merge, for many small
 * demand sets in one launch
 *
 * Instance b is sizes[b] demand rows of 5 int32 (id, from, to, maxWait, maxLoss) starting at ROW offsets[b] of `demand`;
 * the stand table dist (n_stands x n_stands, n_stands <= 128, every entry in [0, 2^22]) serves the whole batch.
 * pool_size (2..4) and n_shards (1..64) hold for every instance.  Per instance the call does what tdh_pool_find_all does:
 * the n_shards logical shards of pool_n.c:226-229, each with its own greedy dedup, then the findpool.c:83-108 merge in
 * shard order with the td_pool_merge quirk (K = 4: scan in (cost, concatenation position) order; K < 4: concatenation
 * order).  Ties are broken exactly as the reference breaks them, so every result depends on the instance alone: not on
 * its position, its neighbours or n_max.
 *   plans_out[b]      n_max / pool_size + 1 rows x 9 in the pool_n.c:123-134 layout (row indices of the instance's own
 *                     demand rows), merged, in findpool order; unused rows -1
 *   n_plans_out[b]    merged count; -1: withdrawn; -2: a shard's record slice was too small (rows -1)
 *   evaluated_out / feasible_out / kept_out [b * n_shards + s]   per logical shard: pool_n.c count_all, pool_count and
 *                     the survivors of its dedup (kept -1 for a shard whose slice was too small; all 0 when withdrawn)
 *   needed_out[b]     the largest per-shard count of materialised records (one per pickup tuple with a feasible drop-off
 *                     order); always written, so a rerun with records_per_shard = needed_out fits
 * The workspace holds records_per_shard 8-byte records per (instance, shard): td_pool_batch_workspace_bytes(batch,
 * n_shards, records_per_shard).  A shard that fills its slice stops writing but keeps enumerating and counting; only
 * its own instance comes back -2.
 *
 * One CTA per (instance, shard), one launch, always asynchronous.  An instance with sizes[b] < 0 or > n_max, offsets[b]
 * < 0 or a stand outside the table is withdrawn without touching its neighbours; a table entry outside [0, 2^22]
 * withdraws every instance.  The arguments are checked before anything else: TD_ERR_INVALID for batch < 0, n_max outside
 * [0, TD_POOL_BATCH_MAX_N], pool_size outside 2..4, n_shards outside [1, 64], n_stands outside [1, 128],
 * records_per_shard outside [0, 2^31) or a NULL pointer with batch > 0; TD_ERR_WORKSPACE for a workspace smaller than
 * td_pool_batch_workspace_bytes.
 * ------------------------------------------------------------------------------------------ */
#define TD_POOL_BATCH_MAX_N 512   /* 9 bits per customer: (cost, pickup tuple) is one exact 64-bit key */
size_t td_pool_batch_workspace_bytes(int batch, int n_shards, int64_t records_per_shard);
int td_pool_find_all_batch(const int32_t *demand, const int32_t *sizes, const int64_t *offsets, int batch, int n_max,
                           const int32_t *dist, int n_stands, int pool_size, int n_shards,
                           int32_t *plans_out /* batch x (n_max/pool_size + 1) x 9 */, int32_t *n_plans_out /* batch */,
                           int64_t *evaluated_out /* batch x n_shards */, int64_t *feasible_out /* batch x n_shards */,
                           int32_t *kept_out /* batch x n_shards */, int64_t *needed_out /* batch */,
                           void *workspace, size_t workspace_bytes, int64_t records_per_shard, void *stream);

/* After an ASYNCHRONOUS td_pool_find / td_pool_find_shards call (stats == NULL) on `workspace`: waits for the
 * stream and reads the per-shard counters back (one small copy).  *overflow_out != 0: the record list was too
 * small for a single pass -- counts_out holds -1 and the call has to be repeated synchronously (stats != NULL),
 * which falls back to cost windows. */
int td_pool_read_stats(const void *workspace, int shard_count, td_pool_stats *stats /* host[shard_count] */,
                       int *overflow_out /* host, may be NULL */, void *stream);
/* bytes td_pool_read_stats copies device -> host (for callers that account their PCIe traffic) */
size_t td_pool_read_stats_bytes(void);

/* findpool.c:83-108: concatenated shard survivors (shard order) -> sort on column 8 -> greedy
 * disjoint scan.  Reference quirk kept: for pool_size < 4 findpool.c sorts on a column it never
 * filled (findpool.c:34-35,70), so the scan runs in concatenation order.
 * Every merge entry point below checks the first pool_size columns of every valid row: a customer outside [0, n)
 * makes *n_plans_out -1 and leaves plans_out untouched (the rows may come from the caller). */
size_t td_pool_merge_workspace_bytes(int total_plans, int n);
int td_pool_merge(const int32_t *shard_plans /* total x 9 */, int total_plans, int n, int pool_size,
                  int32_t *plans_out /* total x 9 */, int32_t *n_plans_out /* 1 */,
                  void *workspace, size_t workspace_bytes, void *stream);

/* Same merge on the fixed-capacity layout that travels through the gather: n_slots slots of `cap`
 * rows each, slot_counts[slot] valid rows per slot (device), slot_shard[slot] = logical shard of the
 * slot (device, NULL: slot index); concatenation order = shard order.  No host round trip. */
int td_pool_merge_padded(const int32_t *slot_plans, const int32_t *slot_counts, const int32_t *slot_shard,
                         int n_slots, int cap, int n, int pool_size,
                         int32_t *plans_out /* n_slots*cap x 9 */, int32_t *n_plans_out /* 1 */,
                         void *workspace, size_t workspace_bytes /* td_pool_merge_workspace_bytes(n_slots*cap, n) */,
                         void *stream);

/* Headed blocks: the layout that travels through ONE collective in the multi-GPU path (findpool.c:149-160 collects
 * out<i>.csv + out<i>.flg per shard; here a shard's survivors, their count and its counters are one block).
 * blocks_out holds shard_count blocks of (cap + 1) rows of 9 int32: row 0 = header {count (-1: the record list
 * overflowed), evaluated lo, evaluated hi, feasible lo, feasible hi, 0, 0, 0, 0}, rows 1.. = the plans.  Always
 * asynchronous (no host out-parameters).  td_pool_merge_headed merges n_slots such blocks (slot_shard as above). */
int td_pool_find_shards_headed(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                               int shard_begin, int shard_count, int n_shards,
                               int32_t *blocks_out /* shard_count x (cap + 1) x 9 */, int32_t cap,
                               void *workspace, size_t workspace_bytes, int64_t max_feasible, void *stream);
int td_pool_merge_headed(const int32_t *blocks, const int32_t *slot_shard, int n_slots, int cap, int n, int pool_size,
                         int32_t *plans_out /* n_slots*cap x 9 */, int32_t *n_plans_out /* 1 */,
                         void *workspace, size_t workspace_bytes /* td_pool_merge_workspace_bytes(n_slots*cap, n) */,
                         void *stream);

/* ------------------------------------------------------------------------------------------
 * Host-buffer twins (allocate, copy, run, copy back).  Same semantics as above.
 * ------------------------------------------------------------------------------------------ */
int tdh_cost_matrix(const int32_t *dist, int n_stands, const int32_t *cab_to, int n_cabs,
                    const int32_t *cust_from, int n_cust, int32_t fill, int32_t cutoff, int32_t *cost_out);
int tdh_lcm(const int32_t *cost, int n, const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out,
            int32_t *n_pairs_out, int64_t *total_out, int32_t *last_min_out);
int tdh_assign_exact(const int32_t *cost, int n, int32_t *col_of_row_out, int64_t *objective_out,
                     uint8_t *x_out, td_assign_stats *stats);
int tdh_assign_exact_rect(const int32_t *cost, int n, int n_real_rows, int n_real_cols, int32_t *col_of_row_out,
                          int64_t *objective_out, uint8_t *x_out, td_assign_stats *stats);
int tdh_pool_find(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                  int shard, int n_shards, int32_t *plans_out, int32_t cap, int32_t *n_plans_out,
                  td_pool_stats *stats);
/* one instance of td_pool_pairs_exact_batch (what a JNI binding of Simulator.findPool calls); pairs_out holds n/2
 * rows; a live row with a stand outside the table, or a table entry outside [0, 2^22], is TD_ERR_INVALID here */
int tdh_pool_pairs_exact(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                         int accept_all, double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out);
/* one instance of td_pool_pairs_batch: the Simulator's own greedy (Simulator.findPool) from host buffers, with the checks
 * of tdh_pool_pairs_exact; pairs_out holds n/2 rows */
int tdh_pool_pairs(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                   int accept_all, double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out);
/* all n_shards logical shards + merge, i.e. what `findpool` produces (findpool.c:122-176) */
int tdh_pool_find_all(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                      int n_shards, int32_t *plans_out, int32_t cap, int32_t *n_plans_out,
                      td_pool_stats *stats);

#ifdef __cplusplus
}
#endif
#endif /* TAXIDISPATCH_H */
