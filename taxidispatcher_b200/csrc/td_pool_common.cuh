// td_pool_common.cuh -- device pieces of the 2..4-passenger pool finder shared by td_pool.cu (one instance, whole GPU)
// and td_pool_batch.cu (many small instances, one CTA per logical shard): the detour threshold, the stand-table limit and
// the evaluation of all drop-off orders of one pickup tuple.
#pragma once
#include "td_common.cuh"

namespace td {

constexpr int kPermBits = 5;

// Stand-table limit for every pool size: an entry above kDistLimit is refused (K = 4: the x32 fixed point of eval4s needs
// 7 legs x 32 < 2^31; K = 2, 3: the (cost << 5 | permutation) order key needs 5 legs < 2^26), never clamped.
constexpr int kDistLimit = 1 << 22;

// pool_n.c:115-116: ride > d * (1 + l/100.0), evaluated in fp64 with round-to-nearest, no contraction; for an integer ride
// that is exactly ride > floor(d * (1 + l/100.0)) (SURVEY.md section 4 trap 3)
__device__ __forceinline__ int pool_detour_thr(int d, int l) {
    const double lim = __dmul_rn(double(d), __dadd_rn(1.0, __ddiv_rn(double(l), 100.0)));
    double fl = floor(lim);
    int thr;
    if (fl >= 2147483647.0) thr = INT_MAX;
    else if (fl < -2147483647.0) thr = INT_MIN;
    else thr = int(fl);
    return thr;
}

// customer record {from, to, thr, wait} with the detour threshold in the fixed point of the evaluation:
// (clamped thr) * 2^SH + (2^SH - 1).  The clamp keeps every comparison exact because no ride exceeds 7 * kDistLimit.
__device__ __forceinline__ int4 scale_cust_rt(int4 c, int sh) {
    if (sh > 0) {
        const int lim = 1 << 25;
        const int z = c.z > lim ? lim : (c.z < -lim ? -lim : c.z);
        c.z = (z << sh) | ((1 << sh) - 1);
    }
    return c;
}

// K = 4, fixed point x32: every distance is pre-multiplied by kSh4 = 32 (the tables are staged that way), the slacks are
// 32 * slack + 31, and a leaf's key is  32 * (drop legs) + permutation index  -- ONE three-input add per leaf gives both the
// last partial sum and the (cost, permutation) order key, and  key <= sl  is exactly  legs <= slack  because the index is
// below 32.  e[i] = D(F3,T_i); t[i][j] = D(T_i,T_j); sl[i] from thr_i - (pickup legs from i to the last pickup).
constexpr int kSh4 = 5;
__device__ __forceinline__ void eval4s(const int e[4], const int t[4][4], const int sl[4], int &nfeas, int &best) {
    nfeas = 0; best = INT_MAX;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int d0 = e[i];
        const bool ok0 = d0 <= sl[i];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j == i) continue;
            const int d1 = d0 + t[i][j];
            const bool ok1 = ok0 && d1 <= sl[j];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (k == i || k == j) continue;
                const int l = 6 - i - j - k;
                const int d2 = d1 + t[j][k];
                // lexicographic permutation index (pool_n.c:137-150 order)
                const int rj = j - (j > i);
                const int rk = k - (k > i) - (k > j);
                const int perm = i * 6 + rj * 2 + rk;
                const int key = d2 + t[k][l] + perm;
                const bool ok = ok1 && d2 <= sl[k] && key <= sl[l];
                nfeas += ok;
                best = (ok && key < best) ? key : best;
            }
        }
    }
}
__device__ __forceinline__ void eval3(const int e[3], const int t[3][3], const int sl[3], int pick_sum, int &nfeas,
                                      int &best) {
    nfeas = 0; best = INT_MAX;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const int d0 = e[i];
        const bool ok0 = d0 <= sl[i];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            if (j == i) continue;
            const int k = 3 - i - j;
            const int d1 = d0 + t[i][j];
            const int d2 = d1 + t[j][k];
            const bool ok = ok0 && d1 <= sl[j] && d2 <= sl[k];
            const int perm = i * 2 + (j - (j > i));
            const int key = ((pick_sum + d2) << kPermBits) | perm;
            nfeas += ok;
            best = (ok && key < best) ? key : best;
        }
    }
}

}  // namespace td
