// Explicit-feedback ALS (ALS-WR, the form of MLlib's explicit ALS): factor init, the normal equations of every row in
// segments of XMAP_ALS_SEGMENT records, their fp64 Cholesky solve, scores and a streaming top-N (C ABI section 8).
// The definition, and why every bit of the factors is fixed by it, is in DESIGN.md section 3.8.  There is no tensor-core
// path: the definition fixes the order of every sum, which MMA does not.
#include <math.h>

#include "common.cuh"

namespace xmap {

namespace {

constexpr int ALS_WARPS = 4;             // warps per block of the normal-equation and solve kernels
constexpr int ALS_CHUNK = 32;            // records whose factor rows a warp stages in shared memory at once
constexpr int TOPN_USERS = 64;           // users per top-N block (8 per warp)
constexpr int TOPN_UPW = 8;              // users per warp
constexpr int TOPN_TILE = 128;           // candidate items per shared-memory tile (4 per lane)
constexpr int TOPN_THREADS = 256;

// packed lower triangle, column-major: column j holds rows j .. r-1; entry (i, j), i >= j, at col0(j) + i - j
__device__ __forceinline__ int col0(int j, int r) { return j * r - (j * (j - 1)) / 2; }

// tab[t] = i | j << 8 of packed entry t (t < T), (0, 0) for the padding up to n_tab
__device__ void fill_tab(uint16_t *tab, int n_tab, int r) {
    const int T = r * (r + 1) / 2;
    for (int t = threadIdx.x; t < n_tab; t += blockDim.x) {
        uint16_t v = 0;
        if (t < T) {
            int j = 0;
            while (col0(j + 1, r) <= t) ++j;
            v = (uint16_t)((t - col0(j, r) + j) | (j << 8));
        }
        tab[t] = v;
    }
}

// ---- normal equations: one warp per segment ------------------------------------------------------------------------
// partial[seg] = (A packed, b) of the segment's records, each entry summed over the records in list order from +0.0.
// y_i * y_j of two fp32 values is exact in fp64, so the fma rounds once, as (a + y_i * y_j) does; r * y is not exact,
// so b takes an explicit multiply and add.  Lane l owns the packed entries l + 32 e and the b entries l, l + 32.
template <int NE>
__global__ void __launch_bounds__(ALS_WARPS * 32) als_normal_kernel(const int32_t *__restrict__ col,
                                                                    const double *__restrict__ rating,
                                                                    const int64_t *__restrict__ seg_lo,
                                                                    const int32_t *__restrict__ seg_n, int64_t n_seg,
                                                                    const float *__restrict__ Y, int r,
                                                                    double *__restrict__ partial) {
    extern __shared__ __align__(16) unsigned char sm[];
    uint16_t *tab = reinterpret_cast<uint16_t *>(sm);
    const int warp = threadIdx.x >> 5, lane = lane_id();
    float *ybuf = reinterpret_cast<float *>(sm + NE * 32 * sizeof(uint16_t)) + warp * ALS_CHUNK * r;
    fill_tab(tab, NE * 32, r);
    __syncthreads();
    const int64_t seg = (int64_t)blockIdx.x * ALS_WARPS + warp;
    if (seg >= n_seg) return;
    const int T = r * (r + 1) / 2, P = T + r;
    double acc[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) acc[e] = 0.0;
    double b0 = 0.0, b1 = 0.0;
    const int64_t lo = seg_lo[seg];
    const int cnt = seg_n[seg];
    for (int base = 0; base < cnt; base += ALS_CHUNK) {
        const int m = min(ALS_CHUNK, cnt - base);
        int c = 0;
        double rt = 0.0;
        if (lane < m) { c = col[lo + base + lane]; rt = rating[lo + base + lane]; }
        for (int k = 0; k < m; ++k) {
            const int ck = __shfl_sync(0xffffffffu, c, k);
            const float *src = Y + (size_t)ck * r;
            if (lane < r) ybuf[k * r + lane] = __ldg(src + lane);
            if (lane + 32 < r) ybuf[k * r + lane + 32] = __ldg(src + lane + 32);
        }
        __syncwarp();
        for (int k = 0; k < m; ++k) {
            const float *y = ybuf + k * r;
            const double rr = __shfl_sync(0xffffffffu, rt, k);
#pragma unroll
            for (int e = 0; e < NE; ++e) {
                const int ij = tab[lane + 32 * e];
                acc[e] = fma((double)y[ij & 255], (double)y[ij >> 8], acc[e]);
            }
            if (lane < r) b0 = __dadd_rn(b0, __dmul_rn(rr, (double)y[lane]));
            if (lane + 32 < r) b1 = __dadd_rn(b1, __dmul_rn(rr, (double)y[lane + 32]));
        }
        __syncwarp();
    }
    double *out = partial + seg * P;
#pragma unroll
    for (int e = 0; e < NE; ++e)
        if (lane + 32 * e < T) out[lane + 32 * e] = acc[e];
    if (lane < r) out[T + lane] = b0;
    if (lane + 32 < r) out[T + lane + 32] = b1;
}

// ---- solve: one warp per row ---------------------------------------------------------------------------------------
// The row's segment partials are added in segment order, lam * n_u is added to the diagonal last, then the packed
// system is factored (right-looking column Cholesky: every entry still takes its updates k = 0, 1, ... in index order,
// so the bits are those of the left-looking form), and solved forward (k ascending) and backward (k descending).
__global__ void __launch_bounds__(ALS_WARPS * 32) als_solve_kernel(const int32_t *__restrict__ rows,
                                                                   const int64_t *__restrict__ row_seg,
                                                                   const int64_t *__restrict__ row_n, int32_t n_rows,
                                                                   const double *__restrict__ partial, int r, double lam,
                                                                   float *__restrict__ out, int8_t *__restrict__ status) {
    extern __shared__ __align__(16) unsigned char sm[];
    const int T = r * (r + 1) / 2, P = T + r;
    const int tab_bytes = (T * (int)sizeof(uint16_t) + 15) & ~15;
    uint16_t *tab = reinterpret_cast<uint16_t *>(sm);
    const int warp = threadIdx.x >> 5, lane = lane_id();
    double *A = reinterpret_cast<double *>(sm + tab_bytes) + warp * P;
    double *bb = A + T;
    fill_tab(tab, T, r);
    __syncthreads();
    const int q = blockIdx.x * ALS_WARPS + warp;
    if (q >= n_rows) return;
    const int64_t s0 = row_seg[q], s1 = row_seg[q + 1];
    for (int t = lane; t < P; t += 32) {
        double v = partial[s0 * P + t];
        for (int64_t s = s0 + 1; s < s1; ++s) v = __dadd_rn(v, partial[s * P + t]);
        A[t] = v;
    }
    __syncwarp();
    const double reg = __dmul_rn(lam, (double)row_n[q]);
    for (int p = lane; p < r; p += 32) A[col0(p, r)] = __dadd_rn(A[col0(p, r)], reg);
    bool ok = true;
    for (int k = 0; k < r; ++k) {
        __syncwarp();
        const int ck = col0(k, r);
        const double d = A[ck];
        if (!(d > 0.0)) { ok = false; break; }             // the same value in every lane: the warp leaves together
        const double dk = __dsqrt_rn(d);
        for (int i = k + 1 + lane; i < r; i += 32) A[ck + i - k] = __ddiv_rn(A[ck + i - k], dk);
        __syncwarp();
        if (lane == 0) A[ck] = dk;
        for (int t = col0(k + 1, r) + lane; t < T; t += 32) {
            const int ij = tab[t], i = ij & 255, j = ij >> 8;
            A[t] = __dsub_rn(A[t], __dmul_rn(A[ck + i - k], A[ck + j - k]));
        }
    }
    const int row = rows[q];
    if (!ok) {
        for (int p = lane; p < r; p += 32) out[(size_t)row * r + p] = 0.0f;
        if (lane == 0) status[row] = 1;
        return;
    }
    for (int k = 0; k < r; ++k) {                          // L z = b
        __syncwarp();
        const int ck = col0(k, r);
        const double zk = __ddiv_rn(bb[k], A[ck]);
        __syncwarp();
        for (int i = k + 1 + lane; i < r; i += 32) bb[i] = __dsub_rn(bb[i], __dmul_rn(A[ck + i - k], zk));
        if (lane == 0) bb[k] = zk;
    }
    for (int k = r - 1; k >= 0; --k) {                     // L^T x = z
        __syncwarp();
        const double xk = __ddiv_rn(bb[k], A[col0(k, r)]);
        __syncwarp();
        for (int i = lane; i < k; i += 32) bb[i] = __dsub_rn(bb[i], __dmul_rn(A[col0(i, r) + k - i], xk));
        if (lane == 0) bb[k] = xk;
    }
    __syncwarp();
    for (int p = lane; p < r; p += 32) out[(size_t)row * r + p] = __double2float_rn(bb[p]);
    if (lane == 0) status[row] = 0;
}

// ---- init: Philox4x32-10(seed, (row, block)) -> Box-Muller normals -> unit L2 norm ---------------------------------
__device__ __forceinline__ void als_normal_pair(uint64_t seed, uint32_t row, uint32_t blk, double &z0, double &z1) {
    uint32_t c[4] = {row, blk, 0u, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u1 = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6) + 1.0) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)(c[2] >> 5) * 67108864.0 + (double)(c[3] >> 6)) * (1.0 / 9007199254740992.0);
    const double rad = sqrt(-2.0 * log(u1));                // u1 in (0, 1]
    double s, co;
    sincospi(2.0 * u2, &s, &co);
    z0 = rad * co;
    z1 = rad * s;
}

__global__ void als_init_kernel(int32_t n_rows, int r, uint64_t seed, float *__restrict__ out) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    double ss = 0.0;
    for (int p = 0; p < r; p += 2) {
        double z0, z1;
        als_normal_pair(seed, (uint32_t)row, (uint32_t)(p >> 1), z0, z1);
        ss += z0 * z0;
        if (p + 1 < r) ss += z1 * z1;
    }
    const double nrm = sqrt(ss);
    for (int p = 0; p < r; p += 2) {
        double z0, z1;
        als_normal_pair(seed, (uint32_t)row, (uint32_t)(p >> 1), z0, z1);
        out[(size_t)row * r + p] = __double2float_rn(z0 / nrm);
        if (p + 1 < r) out[(size_t)row * r + p + 1] = __double2float_rn(z1 / nrm);
    }
}

// ---- score: sum_k x[k] * y[k] in fp64 from +0.0, component order (each product exact: fma rounds once) -------------
__global__ void als_predict_kernel(const float *__restrict__ X, const float *__restrict__ Y,
                                   const int64_t *__restrict__ x_n, const int64_t *__restrict__ y_n, int r,
                                   const int32_t *__restrict__ pu, const int32_t *__restrict__ pi, int64_t n_pairs,
                                   double *__restrict__ score) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs) return;
    const int u = pu[t], i = pi[t];
    if (x_n[u] == 0 || y_n[i] == 0) { score[t] = __longlong_as_double(0x7FF8000000000000ll); return; }
    const float *x = X + (size_t)u * r, *y = Y + (size_t)i * r;
    double s = 0.0;
    for (int k = 0; k < r; ++k) s = fma((double)x[k], (double)y[k], s);
    score[t] = s;
}

// ---- top-N: 64 users per block against the candidate factors, streamed in tiles of 128 items ----------------------
// Each warp scores its 8 users against the tile (lane: 4 items x 8 users, fp64 accumulators), then keeps each user's
// running list, best first, in shared memory: a candidate enters only if it beats the list's last entry when the
// list is full, so nothing per candidate leaves the chip.  Order: score descending, then the smaller item (== treats
// -0.0 as 0.0); NaN never enters.  The result is the first n of a total order over a set: no launch shape shows in it.
__device__ __forceinline__ bool rank_before(double sa, int ia, double sb, int ib) {
    return sa > sb || (sa == sb && ia < ib);
}

__device__ __forceinline__ bool rated(const int64_t *rated_ptr, const int32_t *rated_item, int u, int item) {
    int64_t lo = rated_ptr[u], hi = rated_ptr[u + 1];
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int v = rated_item[mid];
        if (v == item) return true;
        if (v < item) lo = mid + 1; else hi = mid;
    }
    return false;
}

__device__ void list_insert(double *ls, int *li, int *len, int n, double s, int it) {
    const int lane = lane_id();
    const int L = *len;
    const bool b0 = lane < L && rank_before(ls[lane], li[lane], s, it);
    const bool b1 = lane + 32 < L && rank_before(ls[lane + 32], li[lane + 32], s, it);
    const int pos = __popc(__ballot_sync(0xffffffffu, b0)) + __popc(__ballot_sync(0xffffffffu, b1));
    if (pos >= n) return;
    const int last = min(L, n - 1);                       // entries [pos, last) move down one slot
    double v0 = 0.0, v1 = 0.0;
    int j0 = 0, j1 = 0;
    const bool m0 = lane >= pos && lane < last, m1 = lane + 32 >= pos && lane + 32 < last;
    if (m0) { v0 = ls[lane]; j0 = li[lane]; }
    if (m1) { v1 = ls[lane + 32]; j1 = li[lane + 32]; }
    __syncwarp();
    if (m0) { ls[lane + 1] = v0; li[lane + 1] = j0; }
    if (m1) { ls[lane + 33] = v1; li[lane + 33] = j1; }
    if (lane == 0) { ls[pos] = s; li[pos] = it; *len = min(L + 1, n); }
    __syncwarp();
}

__global__ void __launch_bounds__(TOPN_THREADS) als_top_n_kernel(
        const float *__restrict__ X, const float *__restrict__ Y, int r, const int32_t *__restrict__ users,
        int32_t n_users, const int32_t *__restrict__ cand, int32_t n_cand, const int64_t *__restrict__ rated_ptr,
        const int32_t *__restrict__ rated_item, int n, int32_t *__restrict__ out_idx, double *__restrict__ out_score,
        int32_t *__restrict__ out_len) {
    extern __shared__ __align__(16) unsigned char sm[];
    double *xs = reinterpret_cast<double *>(sm);                               // [64][r]
    double *lsc = xs + TOPN_USERS * r;                                         // [64][n]
    int *lid = reinterpret_cast<int *>(lsc + TOPN_USERS * n);                  // [64][n]
    int *llen = lid + TOPN_USERS * n;                                          // [64]
    int *tid = llen + TOPN_USERS;                                              // [128] candidate items of the tile
    float *ys = reinterpret_cast<float *>(tid + TOPN_TILE);                    // [128][r + 1]
    const int warp = threadIdx.x >> 5, lane = lane_id();
    const int u0 = blockIdx.x * TOPN_USERS;
    const int nu = min(TOPN_USERS, n_users - u0);
    for (int e = threadIdx.x; e < TOPN_USERS * r; e += blockDim.x) {
        const int q = e / r;
        xs[e] = q < nu ? (double)X[(size_t)users[u0 + q] * r + e % r] : 0.0;
    }
    for (int q = threadIdx.x; q < TOPN_USERS; q += blockDim.x) llen[q] = 0;
    const int rs = r + 1;                                                       // odd stride: lanes hit distinct banks
    for (int c0 = 0; c0 < n_cand; c0 += TOPN_TILE) {
        const int nt = min(TOPN_TILE, n_cand - c0);
        __syncthreads();
        for (int c = threadIdx.x; c < TOPN_TILE; c += blockDim.x) tid[c] = c < nt ? cand[c0 + c] : -1;
        __syncthreads();
        for (int e = threadIdx.x; e < nt * r; e += blockDim.x) {
            const int c = e / r, k = e - c * r;
            ys[c * rs + k] = __ldg(Y + (size_t)tid[c] * r + k);
        }
        __syncthreads();
        double acc[4][TOPN_UPW];
#pragma unroll
        for (int m = 0; m < 4; ++m)
#pragma unroll
            for (int u = 0; u < TOPN_UPW; ++u) acc[m][u] = 0.0;
        const double *xw = xs + warp * TOPN_UPW * r;
        for (int k = 0; k < r; ++k) {
            double yv[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) yv[m] = (double)ys[(lane + 32 * m) * rs + k];
#pragma unroll
            for (int u = 0; u < TOPN_UPW; ++u) {
                const double xv = xw[u * r + k];
#pragma unroll
                for (int m = 0; m < 4; ++m) acc[m][u] = fma(xv, yv[m], acc[m][u]);
            }
        }
#pragma unroll
        for (int u = 0; u < TOPN_UPW; ++u) {
            const int q = warp * TOPN_UPW + u;
            if (q >= nu) break;                                                // the same in every lane
            const int uid = users[u0 + q];
            double *ls = lsc + q * n;
            int *li = lid + q * n;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const int c = lane + 32 * m;
                const double s = acc[m][u];
                const int it = c < nt ? tid[c] : -1;
                const int L = llen[q];
                bool pass = it >= 0 && s == s && (L < n || rank_before(s, it, ls[n - 1], li[n - 1]));
                if (pass && rated_ptr) pass = !rated(rated_ptr, rated_item, uid, it);
                unsigned mask = __ballot_sync(0xffffffffu, pass);
                while (mask) {
                    const int src = __ffs(mask) - 1;
                    mask &= mask - 1;
                    list_insert(ls, li, llen + q, n, __shfl_sync(0xffffffffu, s, src),
                                __shfl_sync(0xffffffffu, it, src));
                }
            }
        }
    }
    __syncthreads();
    for (int u = 0; u < TOPN_UPW; ++u) {
        const int q = warp * TOPN_UPW + u;
        if (q >= nu) break;
        const size_t row = (size_t)users[u0 + q];
        const int L = llen[q];
        for (int p = lane; p < L; p += 32) {
            out_idx[row * n + p] = lid[q * n + p];
            out_score[row * n + p] = lsc[q * n + p];
        }
        if (lane == 0) out_len[row] = L;
    }
}

template <int NE>
int launch_normal(const int32_t *col, const double *rating, const int64_t *seg_lo, const int32_t *seg_n, int64_t n_seg,
                  const float *Y, int r, double *partial, cudaStream_t st) {
    const size_t smem = NE * 32 * sizeof(uint16_t) + (size_t)ALS_WARPS * ALS_CHUNK * r * sizeof(float);
    const int64_t blocks = (n_seg + ALS_WARPS - 1) / ALS_WARPS;
    als_normal_kernel<NE><<<(unsigned)blocks, ALS_WARPS * 32, smem, st>>>(col, rating, seg_lo, seg_n, n_seg, Y, r,
                                                                         partial);
    XMAP_LAUNCH_CHECK();
    return 0;
}

inline int bad_rank(int r) { return r < 1 || r > XMAP_ALS_RANK_MAX; }

}  // namespace

}  // namespace xmap

using namespace xmap;

extern "C" int xmap_als_init(int32_t n_rows, int32_t rank, uint64_t seed, float *out, void *stream) {
    if (bad_rank(rank)) return fail_msg("xmap_als_init: rank outside [1, 64]");
    if (n_rows <= 0) return 0;
    als_init_kernel<<<(n_rows + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n_rows, rank, seed, out);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_als_normal(const int32_t *col, const double *rating, const int64_t *seg_lo, const int32_t *seg_n,
                               int64_t n_seg, const float *factors, int32_t rank, double *partial, void *stream) {
    if (bad_rank(rank)) return fail_msg("xmap_als_normal: rank outside [1, 64]");
    if (n_seg <= 0) return 0;
    if ((n_seg + ALS_WARPS - 1) / ALS_WARPS > 0x7FFFFFFFll) return fail_msg("xmap_als_normal: too many segments");
    cudaStream_t st = (cudaStream_t)stream;
    if (rank <= 8) return launch_normal<2>(col, rating, seg_lo, seg_n, n_seg, factors, rank, partial, st);
    if (rank <= 16) return launch_normal<5>(col, rating, seg_lo, seg_n, n_seg, factors, rank, partial, st);
    if (rank <= 32) return launch_normal<17>(col, rating, seg_lo, seg_n, n_seg, factors, rank, partial, st);
    return launch_normal<65>(col, rating, seg_lo, seg_n, n_seg, factors, rank, partial, st);
}

extern "C" size_t xmap_als_solve_smem_bytes(int32_t rank) {
    const int T = rank * (rank + 1) / 2;
    return (size_t)((T * 2 + 15) & ~15) + (size_t)ALS_WARPS * (T + rank) * sizeof(double);
}

extern "C" int xmap_als_solve(const int32_t *rows, const int64_t *row_seg, const int64_t *row_n, int32_t n_rows,
                              const double *partial, int32_t rank, double lam, float *out, int8_t *status, void *stream) {
    if (bad_rank(rank)) return fail_msg("xmap_als_solve: rank outside [1, 64]");
    if (!(lam >= 0.0)) return fail_msg("xmap_als_solve: lambda must be >= 0");
    if (n_rows <= 0) return 0;
    const size_t smem = xmap_als_solve_smem_bytes(rank);
    XMAP_CUDA(cudaFuncSetAttribute(als_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    als_solve_kernel<<<(n_rows + ALS_WARPS - 1) / ALS_WARPS, ALS_WARPS * 32, smem, (cudaStream_t)stream>>>(
        rows, row_seg, row_n, n_rows, partial, rank, lam, out, status);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_als_predict(const float *X, const float *Y, const int64_t *x_n, const int64_t *y_n, int32_t rank,
                                const int32_t *pu, const int32_t *pi, int64_t n_pairs, double *score, void *stream) {
    if (bad_rank(rank)) return fail_msg("xmap_als_predict: rank outside [1, 64]");
    if (n_pairs <= 0) return 0;
    als_predict_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(X, Y, x_n, y_n, rank, pu, pi,
                                                                                            n_pairs, score);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_als_top_n(const float *X, const float *Y, int32_t rank, const int32_t *users, int32_t n_users,
                              const int32_t *cand, int32_t n_cand, const int64_t *rated_ptr, const int32_t *rated_item,
                              int32_t n, int32_t *out_idx, double *out_score, int32_t *out_len, void *stream) {
    if (bad_rank(rank)) return fail_msg("xmap_als_top_n: rank outside [1, 64]");
    if (n < 1 || n > XMAP_TOPN_MAX) return fail_msg("xmap_als_top_n: n outside [1, 64]");
    if (n_users <= 0) return 0;
    const size_t smem = (size_t)TOPN_USERS * rank * 8 + (size_t)TOPN_USERS * n * 12 + TOPN_USERS * 4 + TOPN_TILE * 4 +
                        (size_t)TOPN_TILE * (rank + 1) * 4;
    XMAP_CUDA(cudaFuncSetAttribute(als_top_n_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    als_top_n_kernel<<<(n_users + TOPN_USERS - 1) / TOPN_USERS, TOPN_THREADS, smem, (cudaStream_t)stream>>>(
        X, Y, rank, users, n_users, cand, n_cand, rated_ptr, rated_item, n, out_idx, out_score, out_len);
    XMAP_LAUNCH_CHECK();
    return 0;
}
