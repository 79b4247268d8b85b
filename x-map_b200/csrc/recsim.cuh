// Device helpers of the recommender kernels shared by recsim.cu (item-based) and usersim.cu (user-based, the
// same formulas on the transposed profile): the cosine of RecommenderSim, the prediction of
// RecommenderPrediction before bound_rating, and the running top-n of one warp.
#pragma once
#include "common.cuh"

namespace xmap {

__device__ __forceinline__ double rs_cosine(double dot, double nn) {           // recommenderSim.py:84-88
    return nn != 0.0 ? dot / nn : 0.0;                                        // a NaN product is truthy in Python
}

// The two leave-one-out similarities of one co-rating entry (ra, rb) of a pair (recommenderSim.py:98-116), as
// deviations from the pair's sim: d1 drops ra from the first norm, d2 drops rb from the second.  w = min(n - 1, N).
__device__ __forceinline__ void rs_deviations(double inner, double ra, double rb, double nx, double ny, double w, double N,
                                              double sim, double &d1, double &d2) {
    const double mi = __dsub_rn(inner, __dmul_rn(ra, rb));                 // no fused multiply-add: a single-entry pair must give 0
    const double nx2 = __dmul_rn(nx, nx), ny2 = __dmul_rn(ny, ny);
    const double m1 = sqrt(__dmul_rn(__dsub_rn(nx2, __dmul_rn(ra, ra)), ny2));
    const double m2 = sqrt(__dmul_rn(nx2, __dsub_rn(ny2, __dmul_rn(rb, rb))));
    d1 = fabs(1.0 * rs_cosine(mi, m1) * w / N - sim);
    d2 = fabs(1.0 * rs_cosine(mi, m2) * w / N - sim);
}

constexpr int PRED_CAP = 128;

// One user's records in profile list order (the test pairs of recsim_predict_kernel): the records on an item are
// found by a scan.  first(nid) / after(e, nid) walk them in list order and give hi at the end.
struct ListRecords {
    const int32_t *item; const double *rating; const int64_t *ts; int64_t lo, hi;
    __device__ __forceinline__ int64_t next(int64_t e, int nid) const {      // the first record on nid at or after e
        while (e < hi && item[e] != nid) ++e;
        return e;
    }
    __device__ __forceinline__ int64_t first(int nid) const { return next(lo, nid); }
    __device__ __forceinline__ int64_t after(int64_t e, int nid) const { return next(e + 1, nid); }
};

// One user's records sorted by (item, list position) (the top-N kernels): the records on an item are one run, found
// by a binary search, in list order -- the same records in the same order as ListRecords.
__device__ __forceinline__ int64_t rs_lower_bound(const int32_t *a, int64_t lo, int64_t hi, int32_t v) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

struct SortedRecords {
    const int32_t *item; const double *rating; const int64_t *ts; int64_t lo, hi;
    __device__ __forceinline__ int64_t first(int nid) const {
        const int64_t e = rs_lower_bound(item, lo, hi, nid);
        return e < hi && item[e] == nid ? e : hi;
    }
    __device__ __forceinline__ int64_t after(int64_t e, int nid) const { return e + 1 < hi && item[e + 1] == nid ? e + 1 : hi; }
    __device__ __forceinline__ bool has(int nid) const {
        const int64_t e = rs_lower_bound(item, lo, hi, nid);
        return e < hi && item[e] == nid;
    }
};

// The prediction of item `it` (nb_len[it] = L > 0) for the user whose records `recs` holds, before bound_rating:
// p0 without decay, p1 with decay.  Returns 0, or 4 when more than PRED_CAP records match (p0 / p1 are then
// meaningless).  The one implementation of the formula: recsim_predict_kernel and the top-N kernels call it.
template <class Records>
__device__ __forceinline__ int rs_predict_raw(const Records &recs, int it, int L, const double *__restrict__ info,
                                              const int32_t *__restrict__ nb_idx, const double *__restrict__ nb_sim,
                                              int K, double alpha, double &p0, double &p1) {
    double ea[PRED_CAP], eb[PRED_CAP];
    long long et[PRED_CAP];
    int n = 0;
    for (int r = 0; r < L; ++r) {
        const int nid = nb_idx[(size_t)it * K + r];
        const double ns = nb_sim[(size_t)it * K + r];
        const double avg_n = info[3 * (size_t)nid];
        for (int64_t e = recs.first(nid); e < recs.hi; e = recs.after(e, nid)) {
            if (n == PRED_CAP) { ++n; goto gathered; }               // n = PRED_CAP + 1 marks the overflow
            ea[n] = __dmul_rn(ns, __dsub_rn(recs.rating[e], avg_n)); eb[n] = fabs(ns); et[n] = recs.ts[e];
            ++n;
        }
    }
gathered:
    const int err = n > PRED_CAP ? 4 : 0;
    n = min(n, PRED_CAP);
    const double avg = info[3 * (size_t)it];
    p0 = avg; p1 = avg;
    if (n > 0) {
        double sa = 0.0, sb = 0.0;
        for (int k = 0; k < n; ++k) { sa = __dadd_rn(sa, ea[k]); sb = __dadd_rn(sb, eb[k]); }
        p0 = __dadd_rn(avg, __ddiv_rn(sa, sb));
        for (int k = 1; k < n; ++k) {                              // stable insertion sort by time
            const double a0 = ea[k], b0 = eb[k];
            const long long t0 = et[k];
            int m = k - 1;
            while (m >= 0 && et[m] > t0) { ea[m + 1] = ea[m]; eb[m + 1] = eb[m]; et[m + 1] = et[m]; --m; }
            ea[m + 1] = a0; eb[m + 1] = b0; et[m + 1] = t0;
        }
        int order = 0, top = 0;
        for (int k = 0; k < n; ++k) if (k == 0 || et[k] != et[k - 1]) ++top;
        const double cur = (double)(top + 1);
        sa = 0.0; sb = 0.0;
        for (int k = 0; k < n; ++k) {
            if (k == 0 || et[k] != et[k - 1]) ++order;
            const double f = exp(-alpha * (cur - (double)order));
            sa = __dadd_rn(sa, __dmul_rn(ea[k], f)); sb = __dadd_rn(sb, __dmul_rn(eb[k], f));
        }
        p1 = __dadd_rn(avg, __ddiv_rn(sa, sb));
    }
    return err;
}

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ bool rs_before(double sa, int ia, double sb, int ib) {
    return sa > sb || (sa == sb && ia < ib);
}

// The running top-n (n <= 64) of one warp: position p is held by lane p & 31 in slot p >> 5; (ts, ti) is the n-th
// entry once the list is full.  Every lane calls every member with the same arguments, except offer's own candidate.
struct WarpTopN {
    double s0, s1, ts;
    int i0, i1, ti, cnt, n;

    __device__ __forceinline__ void init(int n_) { s0 = s1 = ts = 0.0; i0 = i1 = ti = -1; cnt = 0; n = n_; }
    __device__ __forceinline__ bool admits(double s, int i) const { return cnt < n || rs_before(s, i, ts, ti); }

    __device__ __forceinline__ void insert(double s, int i, int lane) {
        const int pos = __popc(__ballot_sync(FULL, lane < cnt && rs_before(s0, i0, s, i))) +
                        __popc(__ballot_sync(FULL, lane + 32 < cnt && rs_before(s1, i1, s, i)));
        if (pos >= n) return;
        const double u0 = __shfl_up_sync(FULL, s0, 1), u1 = __shfl_up_sync(FULL, s1, 1), c = __shfl_sync(FULL, s0, 31);
        const int j0 = __shfl_up_sync(FULL, i0, 1), j1 = __shfl_up_sync(FULL, i1, 1), ci = __shfl_sync(FULL, i0, 31);
        if (lane > pos) { s0 = u0; i0 = j0; } else if (lane == pos) { s0 = s; i0 = i; }
        if (lane + 32 > pos) { s1 = lane ? u1 : c; i1 = lane ? j1 : ci; } else if (lane + 32 == pos) { s1 = s; i1 = i; }
        cnt = min(cnt + 1, n);
        if (cnt == n) {
            ts = __shfl_sync(FULL, n > 32 ? s1 : s0, (n - 1) & 31);
            ti = __shfl_sync(FULL, n > 32 ? i1 : i0, (n - 1) & 31);
        }
    }

    // each lane may hold one candidate (has); the admitted ones go in one at a time
    __device__ __forceinline__ void offer(bool has, double s, int i, int lane) {
        unsigned m = __ballot_sync(FULL, has && admits(s, i));
        while (m) {
            const int src = __ffs(m) - 1;
            m &= m - 1;
            insert(__shfl_sync(FULL, s, src), __shfl_sync(FULL, i, src), lane);
        }
    }

    __device__ __forceinline__ void store(int32_t *idx, double *score, int32_t *len, int lane) const {
        const double nan = __longlong_as_double(0x7FF8000000000000ll);
        if (lane < n) { idx[lane] = lane < cnt ? i0 : -1; score[lane] = lane < cnt ? s0 : nan; }
        if (lane + 32 < n) { idx[lane + 32] = lane + 32 < cnt ? i1 : -1; score[lane + 32] = lane + 32 < cnt ? s1 : nan; }
        if (lane == 0) *len = cnt;
    }
};

}  // namespace xmap
