// User-based kNN on the AlterEgo profile: RecommenderSim "cosine_user" (the item-based stage with the roles of user and
// item exchanged; DESIGN.md section 3.9 states the definition as the project's own), its neighbour selection, and the
// user-based top-N.  The prediction needs no kernel of its own: it is xmap_recsim_predict on the transposed profile.
//
// Similarity rows.  A row (query user u) walks u's records, and for each record a on item i the raters of i (the
// records grouped by item, sorted by (item, user, list position)); every other record b on i gives the co-rating
// entry (a -> b) of the pair (u, user(b)).  The pairs of a row are accumulated on chip in a direct-indexed
// shared-memory table over one tile [v0, v0 + tile) of the user axis at a time: a binary search on each sorted rater
// list finds its part of the tile, and the next tile starts at the smallest neighbour past the current one, so a
// row costs at most min(ceil(n_users / tile), distinct neighbours) passes.  Within a pass the products of up to 32
// records are dealt to the lanes flattened (one lane per product, not per record), so skewed rater lists idle no lane.
//
// Exactness.  Per cell the entry count n and the inner product in 64-bit fixed point with resolution 2^-q,
// q = qbase - E_u - E_v, 2^(E-1) <= norm < 2^E, qbase = 62 - ceil(log2 m), m the largest record count of one
// (user, item).  By Cauchy-Schwarz over the entry multiset |inner| <= m norm_u norm_v < 2^(62 - q), so the sum fits;
// integer addition is associative, so every result is bit-identical for any launch shape, tile or world size.
//
// Two modes.  select: the running top-K of the row (|sim| descending, ties to the smaller user, the self pair
// counting) stays in registers across the passes; nothing per pair reaches HBM.  emit: a second walk of each pass
// forms the local sensitivities (the max over the 2n leave-one-out deviations, a NaN first deviation winning as in
// Python's max(); "first" = the entry of the smallest item, then list position), and (v, n, sim, ls) of every cell
// is written to the row's extent in user order.
#include "recsim.cuh"

namespace xmap {

constexpr int US_CTA_WARPS = 8;

struct UsArgs {
    const int64_t *item_ptr; const int32_t *t_user; const int32_t *t_item; const double *t_rating;
    const int64_t *u_ptr; const int64_t *u_rec; const double *info; const int32_t *uexp;
    int32_t n_users, qbase, num_atleast, k, tile;
    int32_t *nb_idx; double *nb_sim; int32_t *nb_len;
    const int64_t *emit_ptr; int32_t *e_v; int64_t *e_n; double *e_sim; double *e_ls; int64_t *e_len;
    unsigned long long *stats; int32_t *error_flag;
};

// dynamic shared memory of one row group
__host__ __device__ __forceinline__ size_t us_smem_bytes(int tile, int warps, bool emit) {
    return (size_t)tile * (emit ? 24 : 12) + (size_t)warps * 32 * 32 + 16;
}

template <int WARPS>
__device__ __forceinline__ void us_sync() {
    if (WARPS > 1) __syncthreads(); else __syncwarp();
}

// The pair's similarity from its cell (recommenderSim.py:77-82, 118-122): the formula of recsim_pair_kernel.
__device__ __forceinline__ double us_cell_sim(unsigned long long acc, int n, int q, double nx, double ny, int num_atleast,
                                              double &inner) {
    inner = (double)(long long)acc * pow2d(-q);
    return 1.0 * rs_cosine(inner, nx * ny) * (double)min((int64_t)n, (int64_t)num_atleast) / (double)num_atleast;
}

template <int WARPS, bool EMIT>
__global__ void __launch_bounds__(32 * WARPS, 1) usersim_rows_kernel(UsArgs a, const int32_t *__restrict__ rows, int n_rows) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int tile = a.tile;
    unsigned long long *acc = reinterpret_cast<unsigned long long *>(smem);
    unsigned long long *lsb = acc + tile;                                  // emit: bits of the running max deviation
    int64_t *s_lo = reinterpret_cast<int64_t *>(acc + (EMIT ? 2 : 1) * (size_t)tile);
    int64_t *s_a = s_lo + WARPS * 32;
    double *s_ra = reinterpret_cast<double *>(s_a + WARPS * 32);
    int *s_end = reinterpret_cast<int *>(s_ra + WARPS * 32);
    int *s_first = s_end + WARPS * 32;
    int *cnt = s_first + WARPS * 32;
    unsigned *fst = reinterpret_cast<unsigned *>(cnt + tile);              // emit: 2 item + [first deviation NaN]
    int *s_next = reinterpret_cast<int *>(EMIT ? (int *)(fst + tile) : (int *)(cnt + tile));

    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int q_row = blockIdx.x;
    if (q_row >= n_rows) return;
    const int u = rows[q_row];
    const int64_t ulo = a.u_ptr[u], uhi = a.u_ptr[u + 1];
    const double nx = a.info[3 * (size_t)u + 1];
    const int eu = a.uexp[u];
    const double N = (double)a.num_atleast;
    WarpTopN t;
    t.init(a.k);
    int64_t ecount = 0, ecap = 0, ebase = 0;
    if (EMIT) { ebase = a.emit_ptr[q_row]; ecap = a.emit_ptr[q_row + 1] - ebase; }
    unsigned long long products = 0, distinct = 0, passes = 0;

    int v_end = 0;                                        // users below v_end are done
    for (;;) {
        // the next tile starts at the smallest neighbour at or past v_end
        if (threadIdx.x == 0) *s_next = 0x7FFFFFFF;
        us_sync<WARPS>();
        int m = 0x7FFFFFFF;
        for (int64_t e = ulo + threadIdx.x; e < uhi; e += 32 * WARPS) {
            const int64_t r = a.u_rec[e];
            const int i = a.t_item[r];
            const int64_t hi = a.item_ptr[i + 1];
            int64_t p = rs_lower_bound(a.t_user, a.item_ptr[i], hi, v_end);
            if (p < hi && p == r) ++p;                    // the record itself is no partner
            if (p < hi) m = min(m, a.t_user[p]);
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m = min(m, __shfl_xor_sync(FULL, m, off));
        if (lane == 0) atomicMin(s_next, m);
        us_sync<WARPS>();
        const int v0 = *s_next;
        if (v0 == 0x7FFFFFFF) break;
        const int v1 = (int)min((int64_t)a.n_users, (int64_t)v0 + tile);
        const int width = v1 - v0;
        ++passes;
        for (int c = threadIdx.x; c < width; c += 32 * WARPS) {
            acc[c] = 0ull; cnt[c] = 0;
            if (EMIT) { lsb[c] = 0ull; fst[c] = 0xFFFFFFFFu; }
        }
        us_sync<WARPS>();
        // walk 0 accumulates (n, inner); walk 1 (emit) forms the deviations from the finished cells
        for (int walk = 0; walk < (EMIT ? 2 : 1); ++walk) {
            for (int64_t base = ulo + (int64_t)w * 32; base < uhi; base += 32 * WARPS) {
                const int64_t e = base + lane;
                int64_t lo = 0, hi = 0, r = -1;
                double ra = 0.0;
                int first = 0;
                if (e < uhi) {
                    r = a.u_rec[e];
                    const int i = a.t_item[r];
                    ra = a.t_rating[r];
                    first = (e == ulo || a.t_item[a.u_rec[e - 1]] != i) ? (2 * i + 1) : 0;
                    const int64_t ihi = a.item_ptr[i + 1];
                    lo = rs_lower_bound(a.t_user, a.item_ptr[i], ihi, v0);
                    hi = rs_lower_bound(a.t_user, lo, ihi, v1);
                }
                int end = (int)(hi - lo);
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const int x = __shfl_up_sync(FULL, end, off);
                    if (lane >= off) end += x;
                }
                const int total = __shfl_sync(FULL, end, 31);
                s_lo[w * 32 + lane] = lo; s_a[w * 32 + lane] = r; s_ra[w * 32 + lane] = ra;
                s_end[w * 32 + lane] = end; s_first[w * 32 + lane] = first;
                __syncwarp();
                for (int p = lane; p < total; p += 32) {
                    int s = 0;                            // owner: the first record whose inclusive end exceeds p
#pragma unroll
                    for (int step = 16; step > 0; step >>= 1)
                        if (s_end[w * 32 + s + step - 1] <= p) s += step;
                    const int before = s ? s_end[w * 32 + s - 1] : 0;
                    const int64_t b = s_lo[w * 32 + s] + (p - before);
                    if (b == s_a[w * 32 + s]) continue;
                    const int v = a.t_user[b];
                    const double rb = a.t_rating[b];
                    const int c = v - v0;
                    const int q = a.qbase - eu - a.uexp[v];
                    const double rau = s_ra[w * 32 + s];
                    if (walk == 0) {
                        const long long fx = __double2ll_rn(__dmul_rn(rau, rb) * pow2d(q));
                        atomicAdd(acc + c, (unsigned long long)fx);
                        atomicAdd(cnt + c, 1);
                        ++products;
                    } else {
                        const int n = cnt[c];
                        const double ny = a.info[3 * (size_t)v + 1];
                        double inner;
                        const double sim = us_cell_sim(acc[c], n, q, nx, ny, a.num_atleast, inner);
                        double d1, d2;
                        rs_deviations(inner, rau, rb, nx, ny, (double)min((int64_t)n - 1, (int64_t)a.num_atleast), N,
                                      sim, d1, d2);
                        double best = -1.0;
                        if (d1 == d1) best = d1;
                        if (d2 == d2 && d2 > best) best = d2;
                        if (best >= 0.0) atomicMax(lsb + c, (unsigned long long)__double_as_longlong(best));
                        const int f = s_first[w * 32 + s];
                        if (f) atomicMin(fst + c, (unsigned)(f - 1) | (d1 != d1 ? 1u : 0u));
                    }
                }
                __syncwarp();
            }
            us_sync<WARPS>();
        }
        // the cells of the tile, in user order
        if (!EMIT) {
            for (int c0 = w * 32; c0 < width; c0 += 32 * WARPS) {
                const int c = c0 + lane;
                const int n = c < width ? cnt[c] : 0;
                bool has = n > 0;
                double key = 0.0;
                int code = -1;
                if (has) {
                    const int v = v0 + c;
                    double inner;
                    const double sim = us_cell_sim(acc[c], n, a.qbase - eu - a.uexp[v], nx, a.info[3 * (size_t)v + 1],
                                                   a.num_atleast, inner);
                    key = fabs(sim);
                    code = 2 * v + (signbit(sim) ? 1 : 0);
                    ++distinct;
                }
                t.offer(has, key, code, lane);
            }
        } else if (w == 0) {
            for (int c0 = 0; c0 < width; c0 += 32) {
                const int c = c0 + lane;
                const int n = c < width ? cnt[c] : 0;
                const unsigned m = __ballot_sync(FULL, n > 0);
                if (n > 0) {
                    const int64_t pos = ecount + __popc(m & ((1u << lane) - 1u));
                    const int v = v0 + c;
                    double inner;
                    const double sim = us_cell_sim(acc[c], n, a.qbase - eu - a.uexp[v], nx, a.info[3 * (size_t)v + 1],
                                                   a.num_atleast, inner);
                    const double ls = (fst[c] & 1u) ? __longlong_as_double(0x7FF8000000000000ll)
                                                    : __longlong_as_double((long long)lsb[c]);
                    if (pos < ecap) { a.e_v[ebase + pos] = v; a.e_n[ebase + pos] = n; a.e_sim[ebase + pos] = sim; a.e_ls[ebase + pos] = ls; }
                    ++distinct;
                }
                ecount += __popc(m);
            }
        }
        us_sync<WARPS>();
        v_end = v1;
    }
    // statistics: products and distinct neighbours of the row, passes
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        products += __shfl_xor_sync(FULL, products, off);
        distinct += __shfl_xor_sync(FULL, distinct, off);
    }
    if (lane == 0) {
        atomicAdd(a.stats, products);
        atomicAdd(a.stats + 1, distinct);
        if (w == 0) atomicAdd(a.stats + 2, passes);
    }
    if (EMIT) {
        if (threadIdx.x == 0) {
            a.e_len[q_row] = ecount;
            if (ecount > ecap) atomicExch(a.error_flag, 2);
        }
        return;
    }
    if (WARPS > 1) {                                      // the warps' lists, merged by warp 0
        double *ms = reinterpret_cast<double *>(smem);
        int *mi = reinterpret_cast<int *>(ms + WARPS * 64), *mc = mi + WARPS * 64;
        ms[w * 64 + lane] = t.s0; ms[w * 64 + lane + 32] = t.s1;
        mi[w * 64 + lane] = t.i0; mi[w * 64 + lane + 32] = t.i1;
        if (lane == 0) mc[w] = t.cnt;
        __syncthreads();
        if (w != 0) return;
        for (int v = 1; v < WARPS; ++v)
            for (int p = lane; p < 64; p += 32) t.offer(p < mc[v], ms[v * 64 + p], mi[v * 64 + p], lane);
    }
    int32_t *idx = a.nb_idx + (size_t)u * a.k;
    double *sim = a.nb_sim + (size_t)u * a.k;
    if (lane < t.cnt) { idx[lane] = t.i0 >> 1; sim[lane] = (t.i0 & 1) ? -t.s0 : t.s0; }
    if (lane + 32 < t.cnt) { idx[lane + 32] = t.i1 >> 1; sim[lane + 32] = (t.i1 & 1) ? -t.s1 : t.s1; }
    if (lane == 0) a.nb_len[u] = t.cnt;
}

// ---- user-based top-N: the first n items of user u by p0 (or p1) before bound_rating, over the items u has no record
// on.  Only items some neighbour v in N(u) rated can score anything but avg_u; each is scored once, by rs_predict_raw
// on the item's records sorted by user (the transposed profile's SortedRecords), when first seen in a shared-memory
// bitmap over a tile of the item axis (the neighbours' records are sorted by item, so a tile's part is one binary
// search away).  The other items all score avg_u and follow in index order.  One warp per light user, one CTA per
// heavy one (bound: sum over N(u) of the neighbours' record counts).
struct UsTopNArgs {
    const int64_t *up_ptr; const int32_t *up_item;                      // records by (user, item, list position)
    const int64_t *item_ptr; const int32_t *t_user; const double *t_rating; const int64_t *t_ts;    // by (item, user, list)
    const double *info; const int32_t *nb_idx; const double *nb_sim; const int32_t *nb_len; int K, n_items;
    int n; double alpha; int decay; int tile;
    int32_t *out_idx; double *out_score; int32_t *out_len; unsigned long long *stats; int32_t *error_flag;
};

__device__ __forceinline__ bool us_rated(const UsTopNArgs &a, int u, int i) {
    const int64_t lo = a.up_ptr[u], hi = a.up_ptr[u + 1];
    const int64_t e = rs_lower_bound(a.up_item, lo, hi, i);
    return e < hi && a.up_item[e] == i;
}

template <int WARPS>
__global__ void __launch_bounds__(32 * WARPS) usersim_topn_kernel(UsTopNArgs a, const int32_t *__restrict__ users, int n_users) {
    extern __shared__ __align__(16) unsigned char smem_t[];
    unsigned *bm = reinterpret_cast<unsigned *>(smem_t);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if ((int)blockIdx.x >= n_users) return;
    const int u = users[blockIdx.x];
    const int L = a.nb_len[u];
    WarpTopN t;
    t.init(a.n);
    unsigned long long visits = 0, cands = 0;
    if (L > 0) {
        for (int t0 = 0; t0 < a.n_items; t0 += a.tile) {
            const int t1 = min(a.n_items, t0 + a.tile);
            for (int s = threadIdx.x; s < (t1 - t0 + 31) / 32; s += blockDim.x) bm[s] = 0u;
            us_sync<WARPS>();
            for (int r = w; r < L; r += WARPS) {
                const int v = a.nb_idx[(size_t)u * a.K + r];
                int64_t lo = a.up_ptr[v], hi = a.up_ptr[v + 1];
                if (a.tile < a.n_items) { lo = rs_lower_bound(a.up_item, lo, hi, t0); hi = rs_lower_bound(a.up_item, lo, hi, t1); }
                visits += hi - lo;
                for (int64_t base = lo; base < hi; base += 32) {
                    bool has = false;
                    double s = 0.0;
                    int i = -1;
                    if (base + lane < hi) {
                        i = a.up_item[base + lane];
                        const unsigned bit = 1u << ((i - t0) & 31);
                        if (!(atomicOr(bm + ((i - t0) >> 5), bit) & bit) && !us_rated(a, u, i)) {
                            const SortedRecords recs{a.t_user, a.t_rating, a.t_ts, a.item_ptr[i], a.item_ptr[i + 1]};
                            double p0, p1;
                            if (rs_predict_raw(recs, u, L, a.info, a.nb_idx, a.nb_sim, a.K, a.alpha, p0, p1))
                                atomicExch(a.error_flag, 4);
                            s = a.decay ? p1 : p0;
                            ++cands;
                            has = s == s;
                        }
                    }
                    t.offer(has, s, i, lane);
                }
            }
            us_sync<WARPS>();
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cands += __shfl_xor_sync(FULL, cands, off);
    if (lane == 0) { atomicAdd(a.stats, visits); atomicAdd(a.stats + 1, cands); }
    if (WARPS > 1) {
        double *ms = reinterpret_cast<double *>(smem_t);
        int *mi = reinterpret_cast<int *>(ms + WARPS * 64), *mc = mi + WARPS * 64;
        ms[w * 64 + lane] = t.s0; ms[w * 64 + lane + 32] = t.s1;
        mi[w * 64 + lane] = t.i0; mi[w * 64 + lane + 32] = t.i1;
        if (lane == 0) mc[w] = t.cnt;
        __syncthreads();
        if (w != 0) return;
        for (int v = 1; v < WARPS; ++v)
            for (int p = lane; p < 64; p += 32) t.offer(p < mc[v], ms[v * 64 + p], mi[v * 64 + p], lane);
    }
    // the items no neighbour rated score avg_u: the unrated ones in index order, until the list admits no more
    const double avg = a.info[3 * (size_t)u];
    if (L > 0 && avg == avg) {
        for (int base = 0; base < a.n_items; base += 32) {
            const int i = base + lane;
            const bool ok = i < a.n_items && t.admits(avg, i);
            const bool end = __ballot_sync(FULL, !ok) != 0u;
            bool has = ok && !us_rated(a, u, i);
            for (int r = 0; has && r < L; ++r) has = !us_rated(a, a.nb_idx[(size_t)u * a.K + r], i);
            t.offer(has, avg, i, lane);
            if (end) break;
        }
    }
    t.store(a.out_idx + (size_t)u * a.n, a.out_score + (size_t)u * a.n, a.out_len + u, lane);
}

}  // namespace xmap

using namespace xmap;

extern "C" size_t xmap_usersim_smem_bytes(int32_t tile, int32_t cta, int32_t emit) {
    return us_smem_bytes(tile, cta ? US_CTA_WARPS : 1, emit != 0);
}

extern "C" int xmap_usersim_rows(const int64_t *item_ptr, const int32_t *t_user, const int32_t *t_item,
                                 const double *t_rating, const int64_t *u_ptr, const int64_t *u_rec, const double *info,
                                 const int32_t *uexp, int32_t n_users, int32_t qbase, int32_t num_atleast, int32_t k,
                                 const int32_t *rows, int32_t n_rows, int32_t cta, int32_t tile, int32_t *nb_idx,
                                 double *nb_sim, int32_t *nb_len, const int64_t *emit_ptr, int32_t *e_v, int64_t *e_n,
                                 double *e_sim, double *e_ls, int64_t *e_len, unsigned long long *stats,
                                 int32_t *error_flag, void *stream_) {
    if (n_rows <= 0) return 0;
    if (num_atleast < 1) return fail_msg("xmap_usersim_rows: num_atleast must be >= 1");
    const bool emit = emit_ptr != nullptr;
    if (!emit && (k < 1 || k > XMAP_KMAX)) return fail_msg("xmap_usersim_rows: k out of [1, 64]");
    if (tile < 32 * US_CTA_WARPS) return fail_msg("xmap_usersim_rows: tile below 256 cells");
    const size_t smem = us_smem_bytes(tile, cta ? US_CTA_WARPS : 1, emit);
    if (smem > 227 * 1024) return fail_msg("xmap_usersim_rows: tile does not fit in shared memory");
    const UsArgs a{item_ptr, t_user, t_item, t_rating, u_ptr, u_rec, info, uexp, n_users, qbase, num_atleast, k, tile,
                   nb_idx, nb_sim, nb_len, emit_ptr, e_v, e_n, e_sim, e_ls, e_len, stats, error_flag};
    cudaStream_t st = (cudaStream_t)stream_;
#define XMAP_US_LAUNCH(W, E)                                                                                     \
    do {                                                                                                         \
        XMAP_CUDA(cudaFuncSetAttribute(usersim_rows_kernel<W, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                       (int)smem));                                                             \
        usersim_rows_kernel<W, E><<<(unsigned)n_rows, 32 * W, smem, st>>>(a, rows, n_rows);                      \
    } while (0)
    if (cta) { if (emit) XMAP_US_LAUNCH(US_CTA_WARPS, true); else XMAP_US_LAUNCH(US_CTA_WARPS, false); }
    else { if (emit) XMAP_US_LAUNCH(1, true); else XMAP_US_LAUNCH(1, false); }
#undef XMAP_US_LAUNCH
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_usersim_top_n(const int64_t *up_ptr, const int32_t *up_item, const int64_t *item_ptr,
                                  const int32_t *t_user, const double *t_rating, const int64_t *t_ts, const double *info,
                                  const int32_t *nb_idx, const double *nb_sim, const int32_t *nb_len, int32_t k,
                                  int32_t n_items, const int32_t *users, int32_t n_users, int32_t cta, int32_t tile_,
                                  int32_t n,
                                  double alpha, int32_t decay, int32_t *out_idx, double *out_score, int32_t *out_len,
                                  unsigned long long *stats, int32_t *error_flag, void *stream_) {
    if (n < 1 || n > XMAP_TOPN_MAX) return fail_msg("xmap_usersim_top_n: n out of [1, 64]");
    if (n_users <= 0 || n_items <= 0) return 0;
    const int warps = cta ? US_CTA_WARPS : 1;
    if (tile_ != 0 && tile_ < 32) return fail_msg("xmap_usersim_top_n: tile below 32 items");
    const int tile = min(n_items, tile_ ? tile_ : (cta ? XMAP_USERSIM_TOPN_CTA_TILE : XMAP_USERSIM_TOPN_WARP_TILE));
    const size_t merge = (size_t)warps * 64 * (sizeof(double) + sizeof(int)) + warps * sizeof(int);
    const size_t smem = max((size_t)(tile + 31) / 32 * sizeof(unsigned), merge);
    const UsTopNArgs a{up_ptr, up_item, item_ptr, t_user, t_rating, t_ts, info, nb_idx, nb_sim, nb_len, k, n_items,
                       n, alpha, decay, tile, out_idx, out_score, out_len, stats, error_flag};
    cudaStream_t st = (cudaStream_t)stream_;
    if (cta) {
        XMAP_CUDA(cudaFuncSetAttribute(usersim_topn_kernel<US_CTA_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        usersim_topn_kernel<US_CTA_WARPS><<<(unsigned)n_users, 32 * US_CTA_WARPS, smem, st>>>(a, users, n_users);
    } else {
        usersim_topn_kernel<1><<<(unsigned)n_users, 32, smem, st>>>(a, users, n_users);
    }
    XMAP_LAUNCH_CHECK();
    return 0;
}
