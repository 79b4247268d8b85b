// RecommenderSim on the AlterEgo profile: item-item cosine similarity with significance weighting and the
// per-pair local sensitivity (recommenderSim.py:64-75 produce_pairwise, :90-132 cosine_sim, :186-195
// calculate_sim with method "cosine_item"; assist.py:153-175).
//
// What the reference computes (pinned by oracle/harness.run_recommender_sim, tests/golden/*_recsim.npz):
//   * the profile is a flat list of (user, item, rating) records; a (user, item) pair may occur twice (a real
//     target rating next to a synthetic one, generator.py:156-157), which yields self pairs (i, i) and double
//     co-rating entries -- nothing is deduplicated and nothing is filtered;
//   * every user with d >= 2 records emits, for every 2-combination (p < q) of its records in list order, the
//     entry (item_p, item_q) <- (r_p, r_q) and then (item_q, item_p) <- (r_q, r_p)        (:64-75);
//   * per directed pair, over its entries in arrival order: n = #entries, inner = sum r_a r_b,
//     sim = cosine(inner, norm_i norm_j) * min(n, N) / N with the norms over ALL records of the item (:118-122),
//     and the local sensitivity max |v - sim| over the 2 n leave-one-out similarities (:98-116), where
//     Python's max() lets a NaN win only if it is the first element.
//
// Device design: HBM-bound streaming in three steps, run on a contiguous block of item rows at a time (rows never
// share a directed pair, so a block is complete by itself).  (1) fill: one thread per co-rating entry whose first
// record lies on an item of the block computes its directed pair key and the positions of its two records (in the
// reference's emission order, so a STABLE sort by key leaves every pair's entries in arrival order); (2) the caller sorts the keys
// (CUB radix sort through torch: library plumbing); (3) pairs: one warp per pair walks its entries twice --
// the inner product, then the 2 n leave-one-out deviations, which need the finished inner product.
#include "common.cuh"

namespace xmap {

// (count, sum r, sum r^2) per item over records grouped by item: one warp per item, fixed fold order
__global__ void __launch_bounds__(256) recsim_item_info_kernel(const int64_t *__restrict__ item_ptr,
                                                               const double *__restrict__ rating_by_item, int32_t n_items,
                                                               double *__restrict__ info) {
    const int i = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= n_items) return;
    const int64_t lo = item_ptr[i], hi = item_ptr[i + 1];
    double s = 0.0, s2 = 0.0;
    for (int64_t e = lo + lane; e < hi; e += 32) { const double r = rating_by_item[e]; s += r; s2 = __dadd_rn(s2, __dmul_rn(r, r)); }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, off);
        s2 += __shfl_down_sync(0xffffffffu, s2, off);
    }
    if (lane == 0) {
        const double c = (double)(hi - lo);
        info[3 * (size_t)i + 0] = c > 0 ? s / c : 0.0;      // average          (recommenderSim.py:51-58)
        info[3 * (size_t)i + 1] = sqrt(s2);                 // norm2            (:41-49)
        info[3 * (size_t)i + 2] = c;                        // count
    }
}

// Entries of the item rows [i0, i1): entry (p -> q) of a user (records [lo, hi), p != q) belongs to the rows when
// item[p] lies in the range.  The reference emits a user's entries by combination (m, q), m < q, in lexicographic
// order, (m -> q) before (q -> m) (recommenderSim.py:64-75).  Thread t writes the t-th entry of the rows in that
// same order, so a STABLE sort by key leaves every pair's entries in arrival order, whatever the range.  Per record x
// (positions in the user-grouped arrays): in_before[x] = in-range records before x; ent_before[x] = the entries whose
// smaller position lies before x, i.e. the exclusive scan of [x in range] (hi - x - 1) + (in-range records after x in
// its user).  With the full range this is the d (d - 1) entries of every user in emission order.
__global__ void __launch_bounds__(256) recsim_fill_kernel(const int64_t *__restrict__ user_ptr, int32_t n_users,
                                                          const int64_t *__restrict__ in_before,
                                                          const int64_t *__restrict__ ent_before, int64_t n_rec,
                                                          const int32_t *__restrict__ item, int64_t n_items, int32_t i0,
                                                          int32_t i1, int64_t total, int64_t *__restrict__ key,
                                                          int64_t *__restrict__ src) {
    const int64_t t = blockIdx.x * (int64_t)256 + threadIdx.x;
    if (t >= total) return;
    int64_t m = 0, b = n_rec;                            // the smaller position: largest m with ent_before[m] <= t
    while (b - m > 1) {
        const int64_t mid = (m + b) >> 1;
        if (__ldg(ent_before + mid) <= t) m = mid; else b = mid;
    }
    int32_t ua = 0, ub = n_users;                        // its user: largest u with user_ptr[u] <= m
    while (ub - ua > 1) {
        const int32_t mid = (ua + ub) >> 1;
        if (__ldg(user_ptr + mid) <= m) ua = mid; else ub = mid;
    }
    const int64_t hi = user_ptr[ua + 1], e = t - ent_before[m], base = in_before[m + 1];
    const int32_t im = item[m];
    const int64_t fm = (im >= i0 && im < i1) ? 1 : 0;
    // partner q > m: the entries of (m, q') for q' < q number fm (q - m - 1) + in-range records in (m, q)
    int64_t q = m + 1, qb = hi;                          // largest q with that count <= e
    while (qb - q > 1) {
        const int64_t mid = (q + qb) >> 1;
        if (fm * (mid - m - 1) + __ldg(in_before + mid) - base <= e) q = mid; else qb = mid;
    }
    const bool fwd = fm && e == fm * (q - m - 1) + in_before[q] - base;     // (m -> q) comes before (q -> m)
    const int64_t pa = fwd ? m : q, pb = fwd ? q : m;
    key[t] = (int64_t)item[pa] * n_items + (int64_t)item[pb];
    src[t] = (pa << 32) | pb;
}

__device__ __forceinline__ double rs_cosine(double dot, double nn) {           // recommenderSim.py:84-88
    return nn != 0.0 ? dot / nn : 0.0;                                        // a NaN product is truthy in Python
}

// one warp per directed pair: entries [seg_ptr[g], seg_ptr[g + 1]) of the sorted arrays
__global__ void __launch_bounds__(256) recsim_pair_kernel(const int64_t *__restrict__ seg_ptr, const int64_t *__restrict__ seg_key,
                                                          const int64_t *__restrict__ src, const double *__restrict__ rating,
                                                          const double *__restrict__ info, int64_t n_items, int64_t n_pairs,
                                                          int32_t num_atleast, int32_t *__restrict__ out_i, int32_t *__restrict__ out_j,
                                                          int64_t *__restrict__ out_n, double *__restrict__ out_sim,
                                                          double *__restrict__ out_ls) {
    const int64_t g = (blockIdx.x * (int64_t)256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= n_pairs) return;
    const int64_t lo = seg_ptr[g], hi = seg_ptr[g + 1], n = hi - lo;
    const int64_t k = seg_key[g];
    const int i = (int)(k / n_items), j = (int)(k % n_items);
    const double nx = info[3 * (size_t)i + 1], ny = info[3 * (size_t)j + 1];
    const double N = (double)num_atleast;
    double inner = 0.0;
    for (int64_t e = lo + lane; e < hi; e += 32) {
        const int64_t s = src[e];
        inner = __dadd_rn(inner, __dmul_rn(rating[s >> 32], rating[s & 0xFFFFFFFFll]));      // products rounded like the reference's
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) inner += __shfl_xor_sync(0xffffffffu, inner, off);
    const double sim = 1.0 * rs_cosine(inner, nx * ny) * (double)min(n, (int64_t)num_atleast) / N;      // :77-82, :121-122
    // local sensitivity (:98-116): per entry the two leave-one-out similarities, v1 then v2
    const double w = (double)min(n - 1, (int64_t)num_atleast);
    double best = -1.0;                                   // max over the non-NaN deviations (all are >= 0)
    bool first_nan = false;
    for (int64_t e = lo + lane; e < hi; e += 32) {
        const int64_t s = src[e];
        const double ra = rating[s >> 32], rb = rating[s & 0xFFFFFFFFll];
        const double mi = __dsub_rn(inner, __dmul_rn(ra, rb));                 // no fused multiply-add: a single-entry pair must give 0
        const double nx2 = __dmul_rn(nx, nx), ny2 = __dmul_rn(ny, ny);
        const double m1 = sqrt(__dmul_rn(__dsub_rn(nx2, __dmul_rn(ra, ra)), ny2));
        const double m2 = sqrt(__dmul_rn(nx2, __dsub_rn(ny2, __dmul_rn(rb, rb))));
        const double d1 = fabs(1.0 * rs_cosine(mi, m1) * w / N - sim);
        const double d2 = fabs(1.0 * rs_cosine(mi, m2) * w / N - sim);
        if (e == lo && d1 != d1) first_nan = true;        // Python's max(): a NaN only wins when it comes first
        if (d1 == d1 && d1 > best) best = d1;
        if (d2 == d2 && d2 > best) best = d2;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, off));
    first_nan = __shfl_sync(0xffffffffu, first_nan ? 1 : 0, 0) != 0;
    if (lane == 0) {
        out_i[g] = i; out_j[g] = j; out_n[g] = n; out_sim[g] = sim;
        // every deviation NaN except possibly none: with a non-NaN first element the result is the max of the
        // non-NaN ones (best >= 0 always holds then, the first element itself being one of them)
        out_ls[g] = first_nan ? __longlong_as_double(0x7FF8000000000000ll) : best;
    }
}

// ---- non-private neighbour selection (recommenderPrivacy.py:141-178): per item the first K neighbours by |sim|
// descending, ties to the smaller neighbour index; the self pair is a neighbour like any other.  One warp per
// item over its run of the (i, j)-sorted pair list: K rounds of a warp arg-best, each taking the best
// candidate strictly after the previous winner.
__global__ void __launch_bounds__(256) recsim_neighbors_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ pj,
                                                               const double *__restrict__ psim, int32_t n_items, int32_t K,
                                                               int32_t *__restrict__ nb_idx, double *__restrict__ nb_sim,
                                                               int32_t *__restrict__ nb_len) {
    const int i = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= n_items) return;
    const int64_t lo = row_ptr[i], hi = row_ptr[i + 1];
    unsigned long long last_k = ~0ull;
    int last_t = -1, got = 0;
    for (int r = 0; r < K; ++r) {
        unsigned long long bk = 0ull; int bt = 0x7FFFFFFF, bp = -1;
        for (int64_t e = lo + lane; e < hi; e += 32) {
            const unsigned long long ak = abs_key(psim[e]);
            const int jj = pj[e];
            if (r > 0 && !better(last_k, last_t, ak, jj)) continue;
            if (bp < 0 || better(ak, jj, bk, bt)) { bk = ak; bt = jj; bp = (int)(e - lo); }
        }
        warp_argbest(bk, bt, bp);
        if (bp < 0) break;
        if (lane == 0) { nb_idx[(size_t)i * K + r] = bt; nb_sim[(size_t)i * K + r] = psim[lo + bp]; }
        last_k = bk; last_t = bt;
        got = r + 1;
    }
    if (lane == 0) nb_len[i] = got;
}

// ---- item-based prediction (recommenderPrediction.py:26-103): one thread per test (user, item) pair.
// Entries = (sim * (r - avg_n), |sim|, time) for every profile record of the user on a neighbour n of the item, in
// (neighbour, profile list) order; no-decay = avg + sum a / sum b; decay = the same with weights
// exp(-alpha (cur - rank)) after a stable sort by time (equal times share a rank, :36-49).
constexpr int PRED_CAP = 128;

__device__ __forceinline__ double rs_bound_rating(double x) {      // :19-24, int() truncates towards zero
    const int v = (int)(x + 0.5);
    return 1.0 * (double)max(0, min(v, 5));
}

__global__ void __launch_bounds__(128) recsim_predict_kernel(const int64_t *__restrict__ prof_ptr, const int32_t *__restrict__ prof_item,
                                                             const double *__restrict__ prof_rating, const int64_t *__restrict__ prof_ts,
                                                             const double *__restrict__ info, const int32_t *__restrict__ nb_idx,
                                                             const double *__restrict__ nb_sim, const int32_t *__restrict__ nb_len, int32_t K,
                                                             const int32_t *__restrict__ t_user, const int32_t *__restrict__ t_item,
                                                             int64_t n_test, double alpha, double *__restrict__ pred0,
                                                             double *__restrict__ pred1, int32_t *__restrict__ error_flag) {
    const int64_t q = blockIdx.x * (int64_t)128 + threadIdx.x;
    if (q >= n_test) return;
    const int u = t_user[q], it = t_item[q];
    const int L = nb_len[it];
    if (L == 0) { pred0[q] = -1.0; pred1[q] = -1.0; return; }        // `iid not in sim_bd.value.keys()` -> ()
    double ea[PRED_CAP], eb[PRED_CAP];
    long long et[PRED_CAP];
    int n = 0;
    const int64_t lo = prof_ptr[u], hi = prof_ptr[u + 1];
    for (int r = 0; r < L; ++r) {
        const int nid = nb_idx[(size_t)it * K + r];
        const double ns = nb_sim[(size_t)it * K + r];
        const double avg_n = info[3 * (size_t)nid];
        for (int64_t e = lo; e < hi; ++e) {
            if (prof_item[e] != nid) continue;
            if (n == PRED_CAP) { atomicExch(error_flag, 4); break; }
            ea[n] = __dmul_rn(ns, __dsub_rn(prof_rating[e], avg_n)); eb[n] = fabs(ns); et[n] = prof_ts[e];
            ++n;
        }
    }
    const double avg = info[3 * (size_t)it];
    double p0 = avg, p1 = avg;
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
    pred0[q] = rs_bound_rating(p0); pred1[q] = rs_bound_rating(p1);
}


// ---- private neighbour selection + noise perturbation (recommenderPrivacy.py:35-139, 152-171) -----------------------
// As the reference behaves under Python 3: np.count_nonzero(map(...)) (:81) counts the map object, so ONE neighbour is
// drawn per item, from the exponential-mechanism weights over all its neighbours in |sim|-descending order, and Laplace
// noise of scale |local sensitivity| / eps is added to its similarity.  One thread per item: every sum is formed in the
// reference's order (Python's sum(): sequential; np.cumsum: sequential; np.sum: numpy's pairwise scheme), so an injected
// uniform picks the same neighbour.

// Philox4x32-10 uniform in [0, 1) with 53 random bits (the generator of generate.cu; counter = (lo, hi), key = seed)
__device__ __forceinline__ double rs_philox_uniform(uint64_t seed, uint32_t c0, uint32_t c1) {
    uint32_t c[4] = {c0, c1, 0u, 0u};
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const unsigned long long bits = (((unsigned long long)c[0] << 32) | c[1]) >> 11;
    return (double)bits * (1.0 / 9007199254740992.0);
}

// numpy's pairwise summation of a contiguous double array (the algorithm behind np.sum): blocks of <= 128 elements with
// 8 running sums, longer arrays halved (the left half a multiple of 8) recursively
__device__ double np_block_sum(const double *a, long long n) {
    if (n < 8) {
        double r = 0.0;
        for (long long i = 0; i < n; ++i) r = __dadd_rn(r, a[i]);
        return r;
    }
    double r[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) r[q] = a[q];
    long long i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int q = 0; q < 8; ++q) r[q] = __dadd_rn(r[q], a[i + q]);
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                           __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, a[i]);
    return res;
}

__device__ double np_pairwise_sum(const double *a, long long n) {
    // explicit stack instead of recursion: (offset, length) of the pieces still to be summed, left to right;
    // results are combined in the order the recursion would: res(left) + res(right)
    struct Frame { long long off, len; int state; double left; };
    Frame st[48];
    int sp = 0;
    st[0].off = 0; st[0].len = n; st[0].state = 0; st[0].left = 0.0;
    double ret = 0.0;
    for (;;) {
        Frame &f = st[sp];
        if (f.len <= 128) {
            ret = np_block_sum(a + f.off, f.len);
            if (sp == 0) return ret;
            --sp;
            continue;
        }
        long long n2 = f.len / 2;
        n2 -= n2 % 8;
        if (f.state == 0) {                                // descend into the left half
            f.state = 1;
            st[sp + 1].off = f.off; st[sp + 1].len = n2; st[sp + 1].state = 0;
            ++sp;
        } else if (f.state == 1) {                         // left done: keep it, descend into the right half
            f.left = ret; f.state = 2;
            st[sp + 1].off = f.off + n2; st[sp + 1].len = f.len - n2; st[sp + 1].state = 0;
            ++sp;
        } else {                                           // both done
            ret = __dadd_rn(f.left, ret);
            if (sp == 0) return ret;
            --sp;
        }
    }
}

__global__ void __launch_bounds__(128) recsim_private_kernel(const int64_t *__restrict__ row_ptr, const int32_t *__restrict__ nbr,
                                                             const double *__restrict__ sim, const double *__restrict__ ls,
                                                             int n_items, int k, double eps, double rpo,
                                                             const double *__restrict__ u_pick, const double *__restrict__ u_noise,
                                                             uint64_t seed, double *__restrict__ scratch,
                                                             int32_t *__restrict__ out_nbr, double *__restrict__ out_sim,
                                                             int32_t *__restrict__ out_len) {
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= n_items) return;
    const long long a = row_ptr[it], b = row_ptr[it + 1], n = b - a;
    if (n <= 0) { out_len[it] = 0; return; }
    // the local sensitivity of largest magnitude, the first one among equals (:103-106)
    double max_rs = ls[a], m = fabs(ls[a]);
    for (long long q = a + 1; q < b; ++q) {
        const double v = fabs(ls[q]);
        if (v > m || (m != m && v == v)) { m = v; max_rs = ls[q]; }
    }
    const double k_sim = n >= k ? sim[a + k - 1] : sim[b - 1];                       // :43-46
    double w = k_sim;                                                               // :54-66
    if (n > k) {
        const double x = __dmul_rn(__ddiv_rn(__dmul_rn((double)(2 * k), max_rs), eps),
                                   log(__ddiv_rn((double)((long long)k * (n - k)), rpo)));
        if (x < k_sim) w = x;                                                       // Python's min(k_sim, x)
    }
    const double two_k = (double)(2 * k);
    double tot = 0.0;
    for (long long q = a; q < b; ++q) {
        const double s_ = sim[q], sw = __dsub_rn(s_, w);
        const double ms = sw > s_ ? sw : s_;                                        // :71-73 max(sim, sim - w)
        const double pr = exp(__ddiv_rn(__dmul_rn(eps, ms), __dmul_rn(two_k, ls[q])));   // :88-93
        scratch[q] = pr;
        tot = __dadd_rn(tot, pr);                                                   // Python sum(): sequential
    }
    for (long long q = a; q < b; ++q) scratch[q] = __ddiv_rn(scratch[q], tot);      // :97-99
    const double up = u_pick ? u_pick[it] : rs_philox_uniform(seed, (uint32_t)it, 0u);
    const double target = __dmul_rn(up, np_pairwise_sum(scratch + a, n));           // rand * np.sum(weights), :116-118
    long long idx = n - 1;
    double cum = 0.0;
    for (long long q = 0; q < n; ++q) {                                             // np.searchsorted(np.cumsum(w), target), side='left'
        cum = __dadd_rn(cum, scratch[a + q]);
        if (cum >= target) { idx = q; break; }
    }
    const double un = u_noise ? u_noise[it] : rs_philox_uniform(seed, (uint32_t)it, 1u);
    const double scale = __ddiv_rn(fabs(ls[a + idx]), eps);                         // :159-166, legacy RandomState.laplace
    const double noise = un >= 0.5 ? __dsub_rn(0.0, __dmul_rn(scale, log(__dsub_rn(__dsub_rn(2.0, un), un))))
                                   : __dadd_rn(0.0, __dmul_rn(scale, log(__dadd_rn(un, un))));
    out_nbr[it] = nbr[a + idx];
    out_sim[it] = __dadd_rn(sim[a + idx], noise);
    out_len[it] = 1;
}

}  // namespace xmap

using namespace xmap;

extern "C" int xmap_recsim_item_info(const int64_t *item_ptr, const double *rating_by_item, int32_t n_items, double *info,
                                     void *stream_) {
    if (n_items <= 0) return 0;
    recsim_item_info_kernel<<<(unsigned)((n_items + 7) / 8), 256, 0, (cudaStream_t)stream_>>>(item_ptr, rating_by_item, n_items, info);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_recsim_fill_rows(const int64_t *user_ptr, int32_t n_users, const int64_t *in_before,
                                     const int64_t *ent_before, int64_t n_rec, const int32_t *item, int64_t n_items,
                                     int32_t i0, int32_t i1, int64_t total, int64_t *key, int64_t *src, void *stream_) {
    if (total <= 0) return 0;
    if (i0 < 0 || i1 < i0 || i1 > n_items) return fail_msg("xmap_recsim_fill_rows: row range outside [0, n_items]");
    recsim_fill_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream_>>>(
        user_ptr, n_users, in_before, ent_before, n_rec, item, n_items, i0, i1, total, key, src);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_recsim_pairs(const int64_t *seg_ptr, const int64_t *seg_key, const int64_t *src, const double *rating,
                                 const double *info, int64_t n_items, int64_t n_pairs, int32_t num_atleast,
                                 int32_t *out_i, int32_t *out_j, int64_t *out_n, double *out_sim, double *out_ls, void *stream_) {
    if (n_pairs <= 0) return 0;
    if (num_atleast < 1) return fail_msg("xmap_recsim_pairs: num_atleast must be >= 1");
    recsim_pair_kernel<<<(unsigned)((n_pairs + 7) / 8), 256, 0, (cudaStream_t)stream_>>>(seg_ptr, seg_key, src, rating, info, n_items,
                                                                                        n_pairs, num_atleast, out_i, out_j, out_n,
                                                                                        out_sim, out_ls);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_recsim_neighbors(const int64_t *row_ptr, const int32_t *pair_j, const double *pair_sim, int32_t n_items,
                                     int32_t k, int32_t *nb_idx, double *nb_sim, int32_t *nb_len, void *stream_) {
    if (n_items <= 0) return 0;
    if (k < 1 || k > XMAP_KMAX) return fail_msg("xmap_recsim_neighbors: k out of range");
    recsim_neighbors_kernel<<<(unsigned)((n_items + 7) / 8), 256, 0, (cudaStream_t)stream_>>>(row_ptr, pair_j, pair_sim, n_items, k,
                                                                                          nb_idx, nb_sim, nb_len);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_recsim_predict(const int64_t *prof_ptr, const int32_t *prof_item, const double *prof_rating,
                                   const int64_t *prof_ts, const double *info, const int32_t *nb_idx, const double *nb_sim,
                                   const int32_t *nb_len, int32_t k, const int32_t *t_user, const int32_t *t_item, int64_t n_test,
                                   double alpha, double *pred_nodecay, double *pred_decay, int32_t *error_flag, void *stream_) {
    if (n_test <= 0) return 0;
    recsim_predict_kernel<<<(unsigned)((n_test + 127) / 128), 128, 0, (cudaStream_t)stream_>>>(
        prof_ptr, prof_item, prof_rating, prof_ts, info, nb_idx, nb_sim, nb_len, k, t_user, t_item, n_test, alpha,
        pred_nodecay, pred_decay, error_flag);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_recsim_private_neighbor(const int64_t *row_ptr, const int32_t *nbr, const double *sim, const double *ls,
                                            int32_t n_items, int32_t mapping_range, double eps, double rpo,
                                            const double *u_pick, const double *u_noise, uint64_t seed, double *scratch,
                                            int32_t *out_nbr, double *out_sim, int32_t *out_len, void *stream_) {
    if (n_items <= 0) return 0;
    if (mapping_range < 1) return fail_msg("xmap_recsim_private_neighbor: mapping_range must be >= 1");
    if (!(eps > 0.0) || !(rpo > 0.0)) return fail_msg("xmap_recsim_private_neighbor: eps and rpo must be positive");
    recsim_private_kernel<<<(unsigned)((n_items + 127) / 128), 128, 0, (cudaStream_t)stream_>>>(
        row_ptr, nbr, sim, ls, n_items, mapping_range, eps, rpo, u_pick, u_noise, seed, scratch, out_nbr, out_sim, out_len);
    XMAP_LAUNCH_CHECK();
    return 0;
}
