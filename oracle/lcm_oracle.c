/*
 * lcm_oracle.c -- CPU restatement of the reference's LCM ("lowest cost method") greedy.
 *
 * TEST INFRASTRUCTURE ONLY (checker for the CUDA path; see oracle/README.md).
 * Parity status: PINNED -- the reference LCM bodies are pure numpy and were run as they
 * stand (lifted out of scripts that import cvxopt on line 1) by oracle/lcm_ref.py; this C
 * version is checked against those restatements in tests/test_oracle_lcm.py and exists only
 * because the O(n * n^2) numpy loop needs ~10 s at n = 2000.
 *
 * One parametrised body covers every variant on the hot path (SURVEY.md section 8(a) a5/a6):
 *   heuristic.py:24-33      mask 100, n iterations, every value summed
 *   split.py:161-175        mask big_cost, n iterations, values >= big_cost not summed (:167)
 *   greedy_opt.py:61-82     + break when min > THRESHOLD (:69), returns rows/cols
 *   simulate.py:76-97       same with THRESHOLD 20
 *   Simulator.java:523-549  strict '<' scan from big_cost (:531-537) => break when min >= big_cost
 *                           (:538); break after a pick when the residual size == MAX_NON_LCM (:545)
 *
 * Semantics that matter (SURVEY.md section 4 trap 4): the mask is a VALUE.  Masked cells keep
 * taking part in the first-index argmin, so once every free cell is >= mask the argmin
 * re-selects an already masked cell.  This restatement keeps the literal array and literally
 * overwrites it, so that behaviour falls out by construction.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int32_t mask_value;    /* written over the chosen row and column */
    int32_t stop_above;    /* break (before recording) when min >  stop_above;   INT32_MAX = never */
    int32_t stop_at_value; /* break (before recording) when min >= stop_at_value; INT32_MAX = never */
    int32_t sum_below;     /* add min to the total only when min < sum_below;     INT32_MAX = always */
    int32_t residual_size; /* break (after recording) when n - picks == residual_size; 0 = never */
    int32_t max_iters;     /* number of iterations, normally n; <0 = n */
} lcm_oracle_params;

int lcm_oracle(const int32_t *cost, int n, const lcm_oracle_params *p, int32_t *rows_out, int32_t *cols_out,
               int32_t *n_pairs_out, int64_t *total_out, int32_t *last_min_out) {
    int64_t nn = (int64_t)n * n;
    int32_t *d = (int32_t *)malloc((size_t)(nn ? nn : 1) * sizeof(int32_t));
    if (!d) return -1;
    memcpy(d, cost, (size_t)nn * sizeof(int32_t));
    int64_t total = 0;
    int32_t pairs = 0, last_min = INT32_MAX;
    int iters = (p->max_iters < 0 || p->max_iters > n) ? n : p->max_iters;
    int size = n;
    for (int it = 0; it < iters; it++) {
        int64_t e = 0;
        int32_t v = d[0];
        for (int64_t i = 1; i < nn; i++) if (d[i] < v) { v = d[i]; e = i; } /* first index of the minimum */
        last_min = v;
        if (p->stop_above != INT32_MAX && v > p->stop_above) break;
        if (p->stop_at_value != INT32_MAX && v >= p->stop_at_value) break;
        int row = (int)(e / n), col = (int)(e - (int64_t)row * n);
        if (rows_out) rows_out[pairs] = row;
        if (cols_out) cols_out[pairs] = col;
        pairs++;
        if (p->sum_below == INT32_MAX || v < p->sum_below) total += v;
        for (int j = 0; j < n; j++) {
            d[(int64_t)n * row + j] = p->mask_value;
            d[(int64_t)j * n + col] = p->mask_value;
        }
        size--;
        if (p->residual_size > 0 && size == p->residual_size) break;
    }
    free(d);
    if (n_pairs_out) *n_pairs_out = pairs;
    if (total_out) *total_out = total;
    if (last_min_out) *last_min_out = last_min;
    return 0;
}

/*
 * lcm_sorted_walk -- the same algorithm without the array, for sizes where the literal scan
 * (O(iters * n^2)) is out of reach.  keys: every cell's (uint32(cost) ^ 0x80000000) << 32 | flat
 * index, sorted ascending (n <= 65535, so the index fits 32 bits); that is first-index argmin order.
 * A cell is masked once its row or its column has been picked, and then reads as mask_value.
 * The smallest masked cell in first-index order is (0, 0) once row 0 is picked, else (0, smallest
 * picked column), so each iteration's argmin is the smaller of that masked key and the first key
 * of the sorted list whose row and column are both free.  The cursor into the list only moves
 * forward (a masked cell never becomes free again): O(n^2) after the sort.
 */
static uint64_t walk_key(int32_t v, uint32_t idx) { return ((uint64_t)((uint32_t)v ^ 0x80000000u) << 32) | idx; }

int lcm_sorted_walk(const uint64_t *keys, int n, const lcm_oracle_params *p, int32_t *rows_out, int32_t *cols_out,
                    int32_t *n_pairs_out, int64_t *total_out, int32_t *last_min_out) {
    if (n < 0 || n > 65535) return -1;
    const uint64_t nn = (uint64_t)n * n;
    uint8_t *row_picked = (uint8_t *)calloc((size_t)(n ? n : 1), 1), *col_picked = (uint8_t *)calloc((size_t)(n ? n : 1), 1);
    if (!row_picked || !col_picked) { free(row_picked); free(col_picked); return -1; }
    int64_t total = 0;
    int32_t pairs = 0, last_min = INT32_MAX;
    int iters = (p->max_iters < 0 || p->max_iters > n) ? n : p->max_iters;
    int size = n, row0_picked = 0, minc = n;
    uint64_t q = 0;
    for (int it = 0; it < iters; it++) {
        while (q < nn) {
            const uint32_t idx = (uint32_t)keys[q];
            if (!row_picked[idx / (uint32_t)n] && !col_picked[idx % (uint32_t)n]) break;
            q++;
        }
        const uint64_t fk = q < nn ? keys[q] : UINT64_MAX;
        const uint64_t mk = it >= 1 ? walk_key(p->mask_value, row0_picked ? 0u : (uint32_t)minc) : UINT64_MAX;
        const uint64_t k = fk < mk ? fk : mk;
        const int32_t v = (int32_t)((uint32_t)(k >> 32) ^ 0x80000000u);
        last_min = v;
        if (p->stop_above != INT32_MAX && v > p->stop_above) break;
        if (p->stop_at_value != INT32_MAX && v >= p->stop_at_value) break;
        const uint32_t idx = (uint32_t)k;
        const int row = (int)(idx / (uint32_t)n), col = (int)(idx % (uint32_t)n);
        if (rows_out) rows_out[pairs] = row;
        if (cols_out) cols_out[pairs] = col;
        pairs++;
        if (p->sum_below == INT32_MAX || v < p->sum_below) total += v;
        row_picked[row] = 1;
        col_picked[col] = 1;
        if (row == 0) row0_picked = 1;
        if (col < minc) minc = col;
        size--;
        if (p->residual_size > 0 && size == p->residual_size) break;
    }
    free(row_picked);
    free(col_picked);
    if (n_pairs_out) *n_pairs_out = pairs;
    if (total_out) *total_out = total;
    if (last_min_out) *last_min_out = last_min;
    return 0;
}
