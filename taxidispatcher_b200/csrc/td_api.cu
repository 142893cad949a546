// td_api.cu -- library plumbing (version, errors, device probe, launch counter) and the
// host-buffer twins tdh_* of the device entry points.
#include "td_common.cuh"
#include <cmath>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

namespace td {

static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;

void set_cuda_error(cudaError_t e, const char *what) {
    snprintf(g_err, sizeof g_err, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    cudaGetLastError();  // clear the sticky-less error state
}
void count_launch(int n) { g_launches += n; }

bool have_device() {
    static int cached = -1;
    if (cached < 0) {
        int c = 0;
        cudaError_t e = cudaGetDeviceCount(&c);
        if (e != cudaSuccess) { set_cuda_error(e, "cudaGetDeviceCount"); c = 0; }
        cached = c > 0 ? 1 : 0;
    }
    return cached == 1;
}

int device_sm_count() {
    static thread_local int dev_cached = -1;
    static thread_local int sms = kNumSMsFallback;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return kNumSMsFallback;
    if (dev != dev_cached) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) sms = v;
        dev_cached = dev;
    }
    return sms;
}

// ---- optional per-kernel timing ------------------------------------------------------------------
struct ProfPair { cudaEvent_t a, b; };
static thread_local bool g_prof_on = false;
static thread_local std::vector<ProfPair> g_prof[TD_PROF_KINDS];
static thread_local std::vector<ProfPair> g_prof_pool;

ProfScope::ProfScope(int kind_, cudaStream_t st_) : kind(kind_), st(st_), slot(nullptr) {
    if (!g_prof_on || kind < 0 || kind >= TD_PROF_KINDS) return;
    ProfPair p;
    if (!g_prof_pool.empty()) { p = g_prof_pool.back(); g_prof_pool.pop_back(); }
    else if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) return;
    cudaEventRecord(p.a, st);
    g_prof[kind].push_back(p);
    slot = &g_prof[kind];
}
ProfScope::~ProfScope() {
    if (slot) cudaEventRecord(g_prof[kind].back().b, st);
}

// RAII device buffer for the tdh_* twins
struct DevBuf {
    void *p = nullptr;
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    ~DevBuf() { if (p) cudaFree(p); }
    template <typename T> T *as() { return static_cast<T *>(p); }
};

}  // namespace td

extern "C" const char *td_version(void) { return "taxidispatcher_b200 0.1 (sm_100a)"; }

extern "C" const char *td_strerror(int code) {
    switch (code) {
        case TD_OK: return "ok";
        case TD_ERR_INVALID: return "invalid argument";
        case TD_ERR_CUDA: return "CUDA error (see td_last_cuda_error)";
        case TD_ERR_WORKSPACE: return "workspace too small";
        case TD_ERR_CAPACITY: return "capacity exceeded";
        case TD_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
        case TD_ERR_NOT_CONVERGED: return "solver did not converge";
        default: return "unknown error";
    }
}
extern "C" const char *td_last_cuda_error(void) { return td::g_err; }
extern "C" int td_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess || c <= 0) { cudaGetLastError(); return TD_ERR_NO_DEVICE; }
    return c;
}
extern "C" void td_prof_enable(int on) { td::g_prof_on = on != 0; }
extern "C" void td_prof_reset(void) {
    for (int k = 0; k < TD_PROF_KINDS; ++k) {
        for (auto &p : td::g_prof[k]) td::g_prof_pool.push_back(p);
        td::g_prof[k].clear();
    }
}
extern "C" int td_prof_read(int kind, double *total_ms, int64_t *count) {
    if (kind < 0 || kind >= TD_PROF_KINDS || !total_ms || !count) return TD_ERR_INVALID;
    double tot = 0;
    for (auto &p : td::g_prof[kind]) {
        cudaError_t e = cudaEventSynchronize(p.b);
        if (e != cudaSuccess) { td::set_cuda_error(e, "cudaEventSynchronize"); return TD_ERR_CUDA; }
        float ms = 0;
        e = cudaEventElapsedTime(&ms, p.a, p.b);
        if (e != cudaSuccess) { td::set_cuda_error(e, "cudaEventElapsedTime"); return TD_ERR_CUDA; }
        tot += ms;
    }
    *total_ms = tot;
    *count = int64_t(td::g_prof[kind].size());
    return TD_OK;
}
extern "C" int64_t td_launch_count(void) { return td::g_launches; }
extern "C" void td_launch_count_reset(void) { td::g_launches = 0; }

#define TDH_TRY(expr)                                  \
    do {                                               \
        cudaError_t _e = (expr);                       \
        if (_e != cudaSuccess) {                       \
            td::set_cuda_error(_e, #expr);             \
            return TD_ERR_CUDA;                        \
        }                                              \
    } while (0)
#define TDH_RC(expr)            \
    do {                        \
        int _rc = (expr);       \
        if (_rc != TD_OK) return _rc; \
    } while (0)

extern "C" int tdh_cost_matrix(const int32_t *dist, int n_stands, const int32_t *cab_to, int n_cabs,
                               const int32_t *cust_from, int n_cust, int32_t fill, int32_t cutoff, int32_t *cost_out) {
    if (n_cabs < 0 || n_cust < 0 || n_stands < 0) return TD_ERR_INVALID;
    const int n = n_cabs > n_cust ? n_cabs : n_cust;
    if (n == 0) return TD_OK;
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    td::DevBuf d_dist, d_cab, d_cust, d_cost;
    const size_t ds = size_t(n_stands) * n_stands * 4;
    TDH_TRY(d_dist.alloc(ds)); TDH_TRY(d_cab.alloc(size_t(n_cabs) * 4)); TDH_TRY(d_cust.alloc(size_t(n_cust) * 4));
    TDH_TRY(d_cost.alloc(size_t(n) * n * 4));
    if (ds) TDH_TRY(cudaMemcpy(d_dist.p, dist, ds, cudaMemcpyHostToDevice));
    if (n_cabs) TDH_TRY(cudaMemcpy(d_cab.p, cab_to, size_t(n_cabs) * 4, cudaMemcpyHostToDevice));
    if (n_cust) TDH_TRY(cudaMemcpy(d_cust.p, cust_from, size_t(n_cust) * 4, cudaMemcpyHostToDevice));
    TDH_RC(td_cost_matrix(d_dist.as<int32_t>(), n_stands, d_cab.as<int32_t>(), n_cabs, d_cust.as<int32_t>(), n_cust,
                          fill, cutoff, d_cost.as<int32_t>(), nullptr));
    TDH_TRY(cudaMemcpy(cost_out, d_cost.p, size_t(n) * n * 4, cudaMemcpyDeviceToHost));
    return TD_OK;
}

extern "C" int tdh_lcm(const int32_t *cost, int n, const td_lcm_params *params, int32_t *rows_out, int32_t *cols_out,
                       int32_t *n_pairs_out, int64_t *total_out, int32_t *last_min_out) {
    if (n < 0 || !params || !n_pairs_out || !total_out) return TD_ERR_INVALID;
    if (n == 0) { *n_pairs_out = 0; *total_out = 0; if (last_min_out) *last_min_out = INT32_MAX; return TD_OK; }
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    td::DevBuf d_cost, d_rows, d_cols, d_scal, d_ws;
    const size_t wsb = td_lcm_workspace_bytes(n);
    TDH_TRY(d_cost.alloc(size_t(n) * n * 4)); TDH_TRY(d_rows.alloc(size_t(n) * 4)); TDH_TRY(d_cols.alloc(size_t(n) * 4));
    TDH_TRY(d_scal.alloc(32)); TDH_TRY(d_ws.alloc(wsb));
    TDH_TRY(cudaMemcpy(d_cost.p, cost, size_t(n) * n * 4, cudaMemcpyHostToDevice));
    char *sc = d_scal.as<char>();
    TDH_RC(td_lcm(d_cost.as<int32_t>(), n, params, d_rows.as<int32_t>(), d_cols.as<int32_t>(),
                  reinterpret_cast<int32_t *>(sc + 8), reinterpret_cast<int64_t *>(sc), reinterpret_cast<int32_t *>(sc + 12),
                  d_ws.p, wsb, nullptr));
    char host[16];
    TDH_TRY(cudaMemcpy(host, sc, 16, cudaMemcpyDeviceToHost));
    memcpy(total_out, host, 8); memcpy(n_pairs_out, host + 8, 4);
    if (last_min_out) memcpy(last_min_out, host + 12, 4);
    if (rows_out && *n_pairs_out > 0) TDH_TRY(cudaMemcpy(rows_out, d_rows.p, size_t(*n_pairs_out) * 4, cudaMemcpyDeviceToHost));
    if (cols_out && *n_pairs_out > 0) TDH_TRY(cudaMemcpy(cols_out, d_cols.p, size_t(*n_pairs_out) * 4, cudaMemcpyDeviceToHost));
    return TD_OK;
}

extern "C" int tdh_assign_exact_rect(const int32_t *cost, int n, int n_real_rows, int n_real_cols, int32_t *col_of_row_out,
                                     int64_t *objective_out, uint8_t *x_out, td_assign_stats *stats) {
    if (n < 0) return TD_ERR_INVALID;
    if (n == 0) { if (objective_out) *objective_out = 0; if (stats) memset(stats, 0, sizeof *stats); return TD_OK; }  // solver.py:12
    if (!cost) return TD_ERR_INVALID;
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    td::DevBuf d_cost, d_col, d_obj, d_x, d_ws;
    const size_t wsb = td_assign_rect_workspace_bytes(n, n_real_rows, n_real_cols);
    TDH_TRY(d_cost.alloc(size_t(n) * n * 4)); TDH_TRY(d_col.alloc(size_t(n) * 4)); TDH_TRY(d_obj.alloc(8));
    TDH_TRY(d_ws.alloc(wsb));
    if (x_out) TDH_TRY(d_x.alloc(size_t(n) * n));
    TDH_TRY(cudaMemcpy(d_cost.p, cost, size_t(n) * n * 4, cudaMemcpyHostToDevice));
    TDH_RC(td_assign_exact_rect(d_cost.as<int32_t>(), n, n_real_rows, n_real_cols, d_col.as<int32_t>(), d_obj.as<int64_t>(),
                                x_out ? d_x.as<uint8_t>() : nullptr, stats, d_ws.p, wsb, nullptr));
    TDH_TRY(cudaDeviceSynchronize());
    if (col_of_row_out) TDH_TRY(cudaMemcpy(col_of_row_out, d_col.p, size_t(n) * 4, cudaMemcpyDeviceToHost));
    if (objective_out) TDH_TRY(cudaMemcpy(objective_out, d_obj.p, 8, cudaMemcpyDeviceToHost));
    if (x_out) TDH_TRY(cudaMemcpy(x_out, d_x.p, size_t(n) * n, cudaMemcpyDeviceToHost));
    return TD_OK;
}

extern "C" int tdh_assign_exact(const int32_t *cost, int n, int32_t *col_of_row_out, int64_t *objective_out,
                                uint8_t *x_out, td_assign_stats *stats) {
    return tdh_assign_exact_rect(cost, n, n, n, col_of_row_out, objective_out, x_out, stats);
}

static int pool_find_retry(const int32_t *d_dem, int n, const int32_t *d_dist, int n_stands, int pool_size, int shard,
                           int n_shards, int32_t *d_plans, int32_t cap, int32_t *d_cnt, td_pool_stats *stats) {
    // the feasible list is materialised in the workspace; grow it when a shard overflows
    int64_t max_feasible = 1 << 20;
    for (int attempt = 0; attempt < 8; ++attempt) {
        td::DevBuf d_ws;
        const size_t wsb = td_pool_workspace_bytes(n, n_stands, pool_size, max_feasible);
        TDH_TRY(d_ws.alloc(wsb));
        td_pool_stats st;
        memset(&st, 0, sizeof st);
        int rc = td_pool_find(d_dem, n, d_dist, n_stands, pool_size, shard, n_shards, d_plans, cap, d_cnt, &st, d_ws.p, wsb,
                              max_feasible, nullptr);
        if (stats) *stats = st;
        if (rc != TD_ERR_CAPACITY || st.feasible <= max_feasible) return rc;
        max_feasible = st.feasible + 1024;
    }
    return TD_ERR_CAPACITY;
}

extern "C" int tdh_pool_find(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size, int shard,
                             int n_shards, int32_t *plans_out, int32_t cap, int32_t *n_plans_out, td_pool_stats *stats) {
    if (n < 0 || n_stands <= 0 || !n_plans_out || cap < 0) return TD_ERR_INVALID;
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    td::DevBuf d_dem, d_dist, d_plans, d_cnt;
    TDH_TRY(d_dem.alloc(size_t(n) * 5 * 4)); TDH_TRY(d_dist.alloc(size_t(n_stands) * n_stands * 4));
    TDH_TRY(d_plans.alloc(size_t(cap) * TD_POOL_REC_W * 4)); TDH_TRY(d_cnt.alloc(4));
    if (n) TDH_TRY(cudaMemcpy(d_dem.p, demand, size_t(n) * 5 * 4, cudaMemcpyHostToDevice));
    TDH_TRY(cudaMemcpy(d_dist.p, dist, size_t(n_stands) * n_stands * 4, cudaMemcpyHostToDevice));
    TDH_RC(pool_find_retry(d_dem.as<int32_t>(), n, d_dist.as<int32_t>(), n_stands, pool_size, shard, n_shards,
                           d_plans.as<int32_t>(), cap, d_cnt.as<int32_t>(), stats));
    TDH_TRY(cudaMemcpy(n_plans_out, d_cnt.p, 4, cudaMemcpyDeviceToHost));
    int m = *n_plans_out < cap ? *n_plans_out : cap;
    if (m > 0) TDH_TRY(cudaMemcpy(plans_out, d_plans.p, size_t(m) * TD_POOL_REC_W * 4, cudaMemcpyDeviceToHost));
    return *n_plans_out > cap ? TD_ERR_CAPACITY : TD_OK;
}

// one instance of td_pool_pairs_exact_batch (exact) or td_pool_pairs_batch (greedy) from host buffers
static int tdh_pool_pairs_one(bool exact, const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                              int accept_all, double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out) {
    if (n < 0 || n > TD_PAIRS_EXACT_MAX_N || n_stands < 1 || n_stands > 128 || !n_pairs_out || !cost_out) return TD_ERR_INVALID;
    if (!accept_all && !std::isfinite(max_loss)) return TD_ERR_INVALID;
    if (n > 0 && (!from || !to)) return TD_ERR_INVALID;
    if (!dist || (n >= 2 && !pairs_out)) return TD_ERR_INVALID;
    for (int k = 0; k < n_stands * n_stands; ++k) if (dist[k] < 0 || dist[k] > (1 << 22)) return TD_ERR_INVALID;
    for (int i = 0; i < n; ++i) if (from[i] >= 0 && (from[i] >= n_stands || to[i] < 0 || to[i] >= n_stands)) return TD_ERR_INVALID;
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    td::DevBuf d_in, d_out, d_ws;
    const size_t nn = size_t(n > 0 ? n : 1), words = 2 * nn + 2 + 2 + size_t(n_stands) * n_stands;   // from, to, size, offset, dist
    TDH_TRY(d_in.alloc(words * 4));
    std::vector<int32_t> h(words, 0);
    if (n) { memcpy(h.data(), from, size_t(n) * 4); memcpy(h.data() + nn, to, size_t(n) * 4); }
    h[2 * nn] = n;                                                     // size; the offset (int64 0) follows at an 8-byte boundary
    const size_t off_at = (2 * nn + 1 + 1) & ~size_t(1), dist_at = off_at + 2;
    memcpy(h.data() + dist_at, dist, size_t(n_stands) * n_stands * 4);
    TDH_TRY(cudaMemcpy(d_in.p, h.data(), words * 4, cudaMemcpyHostToDevice));
    const int rows = n / 2;
    const size_t out_bytes = 16 + size_t(rows > 0 ? rows : 1) * 16;   // cost (8), count (4), pad, rows
    TDH_TRY(d_out.alloc(out_bytes));
    int32_t *in = d_in.as<int32_t>();
    char *out = d_out.as<char>();
    const int64_t *offs = reinterpret_cast<const int64_t *>(in + off_at);
    int32_t *rows_d = reinterpret_cast<int32_t *>(out + 16), *count_d = reinterpret_cast<int32_t *>(out + 8);
    int64_t *cost_d = reinterpret_cast<int64_t *>(out);
    if (exact) {
        const size_t wsb = td_pool_pairs_exact_workspace_bytes(1, n);
        TDH_TRY(d_ws.alloc(wsb));
        TDH_RC(td_pool_pairs_exact_batch(in, in + nn, in + 2 * nn, offs, 1, n, in + dist_at, n_stands, accept_all, max_loss,
                                         rows_d, count_d, cost_d, d_ws.p, wsb, nullptr));
    } else {
        TDH_RC(td_pool_pairs_batch(in, in + nn, in + 2 * nn, offs, 1, n, in + dist_at, n_stands, accept_all, max_loss, rows_d,
                                   count_d, cost_d, nullptr));
    }
    std::vector<char> host(out_bytes);
    TDH_TRY(cudaMemcpy(host.data(), out, out_bytes, cudaMemcpyDeviceToHost));
    memcpy(cost_out, host.data(), 8); memcpy(n_pairs_out, host.data() + 8, 4);
    if (*n_pairs_out > 0) memcpy(pairs_out, host.data() + 16, size_t(*n_pairs_out) * 16);
    return TD_OK;
}

extern "C" int tdh_pool_pairs_exact(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                                    int accept_all, double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out) {
    return tdh_pool_pairs_one(true, from, to, n, dist, n_stands, accept_all, max_loss, pairs_out, n_pairs_out, cost_out);
}

extern "C" int tdh_pool_pairs(const int32_t *from, const int32_t *to, int n, const int32_t *dist, int n_stands,
                              int accept_all, double max_loss, int32_t *pairs_out, int32_t *n_pairs_out, int64_t *cost_out) {
    return tdh_pool_pairs_one(false, from, to, n, dist, n_stands, accept_all, max_loss, pairs_out, n_pairs_out, cost_out);
}

extern "C" int tdh_pool_find_all(const int32_t *demand, int n, const int32_t *dist, int n_stands, int pool_size,
                                 int n_shards, int32_t *plans_out, int32_t cap, int32_t *n_plans_out, td_pool_stats *stats) {
    if (n < 0 || n_stands <= 0 || n_shards < 1 || n_shards > 64 || !n_plans_out || cap < 0) return TD_ERR_INVALID;
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    const int per_shard_cap = n / 2 + 1;  // survivors are customer-disjoint: at most n / pool_size per shard
    td::DevBuf d_dem, d_dist, d_all, d_cnt, d_tot, d_out, d_ws;
    TDH_TRY(d_dem.alloc(size_t(n) * 5 * 4)); TDH_TRY(d_dist.alloc(size_t(n_stands) * n_stands * 4));
    TDH_TRY(d_all.alloc(size_t(per_shard_cap) * n_shards * TD_POOL_REC_W * 4)); TDH_TRY(d_cnt.alloc(size_t(n_shards) * 4));
    TDH_TRY(d_tot.alloc(4));
    if (n) TDH_TRY(cudaMemcpy(d_dem.p, demand, size_t(n) * 5 * 4, cudaMemcpyHostToDevice));
    TDH_TRY(cudaMemcpy(d_dist.p, dist, size_t(n_stands) * n_stands * 4, cudaMemcpyHostToDevice));
    std::vector<td_pool_stats> st(n_shards);
    int64_t max_feasible = int64_t(1) << 22;
    int rc = TD_ERR_CAPACITY;
    for (int attempt = 0; attempt < 8 && rc == TD_ERR_CAPACITY; ++attempt) {
        td::DevBuf ws;
        const size_t wsb = td_pool_shards_workspace_bytes(n, n_stands, pool_size, n_shards, max_feasible);
        TDH_TRY(ws.alloc(wsb));
        rc = td_pool_find_shards(d_dem.as<int32_t>(), n, d_dist.as<int32_t>(), n_stands, pool_size, 0, n_shards, n_shards,
                                 d_all.as<int32_t>(), per_shard_cap, d_cnt.as<int32_t>(), st.data(), ws.p, wsb, max_feasible, nullptr);
        int64_t need = 0;
        for (auto &q : st) need += q.feasible;
        if (rc == TD_ERR_CAPACITY && need <= max_feasible) break;
        max_feasible = need + 1024;
    }
    if (rc != TD_OK) return rc;
    td_pool_stats tot;
    memset(&tot, 0, sizeof tot);
    for (auto &q : st) { tot.evaluated += q.evaluated; tot.feasible += q.feasible; }
    tot.rounds = st[0].rounds; tot.passes = 1;
    const int total = per_shard_cap * n_shards;
    TDH_TRY(d_out.alloc(size_t(total) * TD_POOL_REC_W * 4));
    const size_t wsb = td_pool_merge_workspace_bytes(total, n);
    TDH_TRY(d_ws.alloc(wsb));
    TDH_RC(td_pool_merge_padded(d_all.as<int32_t>(), d_cnt.as<int32_t>(), nullptr, n_shards, per_shard_cap, n, pool_size,
                                d_out.as<int32_t>(), d_tot.as<int32_t>(), d_ws.p, wsb, nullptr));
    TDH_TRY(cudaMemcpy(n_plans_out, d_tot.p, 4, cudaMemcpyDeviceToHost));
    tot.kept = *n_plans_out;
    if (stats) *stats = tot;
    int m = *n_plans_out < cap ? *n_plans_out : cap;
    if (m > 0) TDH_TRY(cudaMemcpy(plans_out, d_out.p, size_t(m) * TD_POOL_REC_W * 4, cudaMemcpyDeviceToHost));
    return *n_plans_out > cap ? TD_ERR_CAPACITY : TD_OK;
}

extern "C" int tdh_assign_stands(const int32_t *dist, int n_stands, const int32_t *cab_to, int n_cabs, const int32_t *cust_from,
                                 int n_cust, int32_t fill, int32_t cutoff, int32_t *col_of_row_out, int32_t *cost_of_row_out,
                                 int64_t *objective_out, int64_t *u_out, int64_t *v_out, int32_t *stats_out) {
    if (n_cabs < 0 || n_cust < 0 || n_stands < 1 || n_stands > TD_STANDS_MAX_S || !dist || !objective_out) return TD_ERR_INVALID;
    const int n = n_cabs > n_cust ? n_cabs : n_cust;
    if ((n_cabs && !cab_to) || (n_cust && !cust_from) || (n && !col_of_row_out)) return TD_ERR_INVALID;
    for (int i = 0; i < n_cabs; ++i) if (cab_to[i] < 0 || cab_to[i] >= n_stands) return TD_ERR_INVALID;
    for (int j = 0; j < n_cust; ++j) if (cust_from[j] < 0 || cust_from[j] >= n_stands) return TD_ERR_INVALID;
    if (!td::have_device()) return TD_ERR_NO_DEVICE;
    // one upload: dist, cab_to, cust_from, then the sizes and (8-byte aligned) offsets of the single instance
    const size_t S2 = size_t(n_stands) * n_stands, at_cab = S2, at_cust = at_cab + n_cabs, at_size = at_cust + n_cust;
    const size_t at_off = (at_size + 2 + 1) & ~size_t(1), words = at_off + 4;
    std::vector<int32_t> h(words, 0);
    memcpy(h.data(), dist, S2 * 4);
    if (n_cabs) memcpy(h.data() + at_cab, cab_to, size_t(n_cabs) * 4);
    if (n_cust) memcpy(h.data() + at_cust, cust_from, size_t(n_cust) * 4);
    h[at_size] = n_cabs; h[at_size + 1] = n_cust;                 // cab_off = cust_off = 0 (int64 zeros)
    const size_t nn = size_t(n > 0 ? n : 1), S = size_t(n_stands);
    const size_t out_bytes = 8 + 8 + 2 * S * 8 + 2 * nn * 4;      // objective, stats, u, v, col, cost
    const size_t wsb = td_assign_stands_workspace_bytes(1, n_stands, n);
    td::DevBuf d_in, d_out, d_ws;
    TDH_TRY(d_in.alloc(words * 4)); TDH_TRY(d_out.alloc(out_bytes)); TDH_TRY(d_ws.alloc(wsb));
    TDH_TRY(cudaMemcpy(d_in.p, h.data(), words * 4, cudaMemcpyHostToDevice));
    int32_t *in = d_in.as<int32_t>();
    char *out = d_out.as<char>();
    const int64_t *offs = reinterpret_cast<const int64_t *>(in + at_off);
    int64_t *obj_d = reinterpret_cast<int64_t *>(out), *u_d = reinterpret_cast<int64_t *>(out + 16), *v_d = u_d + S;
    int32_t *stats_d = reinterpret_cast<int32_t *>(out + 8), *col_d = reinterpret_cast<int32_t *>(v_d + S), *cost_d = col_d + nn;
    TDH_RC(td_assign_stands_batch(in, n_stands, fill, cutoff, in + at_cab, offs, in + at_size, in + at_cust, offs + 1,
                                  in + at_size + 1, 1, n, col_d, cost_d, obj_d, u_d, v_d, stats_d, d_ws.p, wsb, nullptr));
    std::vector<char> host(out_bytes);
    TDH_TRY(cudaMemcpy(host.data(), out, out_bytes, cudaMemcpyDeviceToHost));
    memcpy(objective_out, host.data(), 8);
    if (stats_out) memcpy(stats_out, host.data() + 8, 8);
    if (u_out) memcpy(u_out, host.data() + 16, S * 8);
    if (v_out) memcpy(v_out, host.data() + 16 + S * 8, S * 8);
    if (n) memcpy(col_of_row_out, host.data() + 16 + 2 * S * 8, size_t(n) * 4);
    if (n && cost_of_row_out) memcpy(cost_of_row_out, host.data() + 16 + 2 * S * 8 + nn * 4, size_t(n) * 4);
    return TD_OK;
}
