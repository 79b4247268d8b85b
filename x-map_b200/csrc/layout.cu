// Ratings layout builder: CSR by user + CSC by item + the per-user / per-item
// statistics of BaselinerSim.get_universal_user_info / get_universal_item_info
// (reference baselinerSim.py:17-82).  HBM-bound: every pass is a coalesced
// stream over nnz-sized arrays plus one gather.  The two key sorts use CUB's
// device radix sort (library plumbing, not the hot path).
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace xmap {
thread_local char g_err[512] = "";

__global__ void make_keys_kernel(const int32_t *__restrict__ major, const int32_t *__restrict__ minor,
                                 int64_t nnz, uint64_t *__restrict__ keys, int32_t *__restrict__ vals) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < nnz) {
        keys[k] = ((uint64_t)(uint32_t)major[k] << 32) | (uint32_t)minor[k];
        vals[k] = (int32_t)k;
    }
}

// ptr[m] = first position whose major id >= m (keys sorted by major).
__global__ void boundaries_kernel(const uint64_t *__restrict__ keys, int64_t nnz, int32_t n_major,
                                  int32_t *__restrict__ ptr) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k > nnz) return;
    int32_t hi = (k == nnz) ? n_major : (int32_t)(keys[k] >> 32);
    int32_t lo = (k == 0) ? -1 : (int32_t)(keys[k - 1] >> 32);
    for (int32_t m = lo + 1; m <= hi; ++m) ptr[m] = (int32_t)k;
}

// One thread per user, sequential like the reference's Python sum() (baselinerSim.py:24-30).
__global__ void user_mean_kernel(const int32_t *__restrict__ csr_ptr, const int32_t *__restrict__ perm,
                                 const float *__restrict__ rating, int32_t n_users,
                                 double *__restrict__ mu) {
    int32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_users) return;
    int32_t a = csr_ptr[u], b = csr_ptr[u + 1];
    double s = 0.0;
    for (int32_t k = a; k < b; ++k) s += (double)rating[perm[k]];
    mu[u] = (b > a) ? s / (double)(b - a) : 0.0;
}

// One CTA per item: sum r, sum r^2, sum (r - mu_u)^2, count (baselinerSim.py:56-81).  Thread t takes
// raters t, t + 256, ...; the partial sums are folded lane-wise (xor tree) and then warp by warp in
// index order, so the result is a fixed function of the column (no atomics).
constexpr int IS_THREADS = 256;
__global__ void __launch_bounds__(IS_THREADS) item_stats_kernel(
    const int32_t *__restrict__ csc_ptr, const uint64_t *__restrict__ keys_i, const int32_t *__restrict__ perm,
    const float *__restrict__ rating, const double *__restrict__ mu, int32_t n_items, double *__restrict__ stats) {
    __shared__ double sh[3][IS_THREADS / 32];
    const int32_t i = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int32_t a = csc_ptr[i], b = csc_ptr[i + 1];
    if (warp > 0 && b - a <= 32 * warp) return;          // short columns: the surplus warps leave (no barrier needed)
    double s = 0.0, s2 = 0.0, a2 = 0.0;
    for (int32_t k = a + threadIdx.x; k < b; k += IS_THREADS) {
        double r = (double)rating[perm[k]];
        double c = r - mu[(uint32_t)(keys_i[k] & 0xFFFFFFFFu)];
        s += r;
        s2 = __dadd_rn(s2, __dmul_rn(r, r));
        a2 = __dadd_rn(a2, __dmul_rn(c, c));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, off);
        s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        a2 += __shfl_xor_sync(0xffffffffu, a2, off);
    }
    const int live = min(IS_THREADS / 32, (b - a + 31) / 32);        // warps that stayed (>= 1 unless empty)
    if (live > 1) {
        if (lane == 0) { sh[0][warp] = s; sh[1][warp] = s2; sh[2][warp] = a2; }
        // every staying warp reaches this barrier: bar.sync counts warps, and exited warps no longer count
        __syncthreads();
        if (warp == 0) {
            s = sh[0][0]; s2 = sh[1][0]; a2 = sh[2][0];
            for (int w = 1; w < live; ++w) { s += sh[0][w]; s2 = __dadd_rn(s2, sh[1][w]); a2 = __dadd_rn(a2, sh[2][w]); }
        }
    }
    if (threadIdx.x == 0) {
        double n = (double)(b - a);
        stats[4 * (int64_t)i + 0] = (b > a) ? s / n : 0.0;
        stats[4 * (int64_t)i + 1] = sqrt(s2);
        stats[4 * (int64_t)i + 2] = sqrt(a2);
        stats[4 * (int64_t)i + 3] = n;
    }
}

__global__ void pack_csr_kernel(const uint64_t *__restrict__ keys_u, const int32_t *__restrict__ perm,
                                const float *__restrict__ rating, const double *__restrict__ stats,
                                int64_t nnz, uint64_t *__restrict__ csr_ent, int32_t *__restrict__ csr_src) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    uint32_t item = (uint32_t)(keys_u[k] & 0xFFFFFFFFu);
    int32_t src = perm[k];
    float r = rating[src];
    double avg = stats[4 * (int64_t)item + 0];
    uint32_t ge = ((double)r >= avg) ? 1u : 0u;
    uint32_t w0 = item | (ge << GE_SHIFT);
    csr_ent[k] = ((uint64_t)__float_as_uint(r) << 32) | w0;
    csr_src[k] = src;
}

__global__ void pack_csc_kernel(const uint64_t *__restrict__ keys_i, const int32_t *__restrict__ perm,
                                const float *__restrict__ rating, const double *__restrict__ stats,
                                int64_t nnz, uint64_t *__restrict__ csc_ent) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    uint32_t item = (uint32_t)(keys_i[k] >> 32);
    uint32_t user = (uint32_t)(keys_i[k] & 0xFFFFFFFFu);
    float r = rating[perm[k]];
    uint32_t ge = ((double)r >= stats[4 * (int64_t)item + 0]) ? 1u : 0u;
    csc_ent[k] = ((uint64_t)__float_as_uint(r) << 32) | (user | (ge << 31));
}

// One thread per CSC entry; a warp whose 32 entries belong to one item folds them into one atomic.
__global__ void row_work_kernel(const int32_t *__restrict__ csr_ptr, const int32_t *__restrict__ csc_ptr,
                                const uint64_t *__restrict__ csc_ent, int32_t n_items, int64_t nnz,
                                unsigned long long *__restrict__ work) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int32_t item = -1;
    long long w = 0;
    if (e < nnz) {
        int32_t lo = 0, hi = n_items;                   // largest i with csc_ptr[i] <= e
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (__ldg(csc_ptr + mid) <= e) lo = mid; else hi = mid;
        }
        item = lo;
        const uint32_t u = (uint32_t)(csc_ent[e] & 0x7FFFFFFFu);
        w = csr_ptr[u + 1] - csr_ptr[u];
    }
    const int32_t item0 = __shfl_sync(0xffffffffu, item, 0);
    if (__all_sync(0xffffffffu, item == item0)) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) w += __shfl_xor_sync(0xffffffffu, w, off);
        if (lane == 0 && item0 >= 0) atomicAdd(work + item0, (unsigned long long)w);
    } else if (item >= 0) {
        atomicAdd(work + item, (unsigned long long)w);
    }
}

// ---- triangular layout (see include/xmap_b200.h) ---------------------------------------------
struct __align__(16) OStat {
    double den;
    uint32_t item;
    uint32_t prefix_exp;      // prefix << 8 | item exponent (tri_ostat_kernel)
};

// key = user << 32 | ord(item), value = the CSR entry with the item replaced by its ord, plus the item's exponent
__global__ void tri_keys_kernel(const int32_t *__restrict__ csr_ptr, const uint64_t *__restrict__ csr_ent,
                                const int32_t *__restrict__ ord, const OStat *__restrict__ ostat, int32_t n_users,
                                int64_t nnz, uint64_t *__restrict__ keys, uint64_t *__restrict__ vals) {
    int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    int32_t lo = 0, hi = n_users;                       // largest u with csr_ptr[u] <= k
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (__ldg(csr_ptr + mid) <= k) lo = mid; else hi = mid;
    }
    const uint64_t e = csr_ent[k];
    const uint32_t w0 = (uint32_t)e;
    const uint32_t o = (uint32_t)__ldg(ord + (w0 & ITEM_MASK));
    keys[k] = ((uint64_t)(uint32_t)lo << 32) | o;
    const uint32_t ex = ostat[o].prefix_exp & 0xFFu;
    vals[k] = (e & 0xFFFFFFFF00000000ull) | (uint64_t)((w0 & ~ITEM_MASK) | exp_bits(ex) | o);
}

// One thread per CSC entry (i, u): position of the entry in u's ord-sorted row, suffix length, and
// the row work of i (entries of one item are contiguous, so a warp usually folds its 32 lengths
// into one atomic).
__global__ void tri_aux_kernel(const int32_t *__restrict__ csr_ptr, const int32_t *__restrict__ csc_ptr,
                               const uint64_t *__restrict__ csc_ent, const uint64_t *__restrict__ tcsr_ent,
                               const double *__restrict__ user_mu, const int32_t *__restrict__ ord, int32_t n_items,
                               int64_t nnz, int32_t method, uint4 *__restrict__ csc_aux,
                               unsigned long long *__restrict__ tri_work) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int32_t item = -1;
    long long len = 0;
    if (e < nnz) {
        int32_t lo = 0, hi = n_items;                   // largest i with csc_ptr[i] <= e
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (__ldg(csc_ptr + mid) <= e) lo = mid; else hi = mid;
        }
        item = lo;
        const uint32_t oi = (uint32_t)__ldg(ord + item);
        const uint32_t u = (uint32_t)(csc_ent[e] & 0x7FFFFFFFu);
        int32_t plo = csr_ptr[u], phi = csr_ptr[u + 1];
        const int32_t end = phi;
        while (phi - plo > 1) {                         // largest pos with ord(pos) <= oi
            const int32_t mid = (plo + phi) >> 1;
            if (((uint32_t)__ldg(tcsr_ent + mid) & ITEM_MASK) <= oi) plo = mid; else phi = mid;
        }
        len = end - plo - 1;
        const double mu = (method == XMAP_METHOD_ADJUST_COSINE) ? user_mu[u] : 0.0;
        csc_aux[e] = make_uint4((uint32_t)plo, (uint32_t)len, (uint32_t)__double2loint(mu), (uint32_t)__double2hiint(mu));
    }
    const int32_t item0 = __shfl_sync(0xffffffffu, item, 0);
    if (__all_sync(0xffffffffu, item == item0)) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) len += __shfl_xor_sync(0xffffffffu, len, off);
        if (lane == 0 && item0 >= 0 && len) atomicAdd(tri_work + item0, (unsigned long long)len);
    } else if (item >= 0 && len) {
        atomicAdd(tri_work + item, (unsigned long long)len);
    }
}

// The item exponent: E with 2^(E-1) <= den < 2^E, stored as clamp(E - e_base, 0, EXP_MAX); 0 for den == 0
// (every product of such an item is 0).
__global__ void tri_ostat_kernel(const double *__restrict__ item_stats, const int32_t *__restrict__ prefix_code,
                                 const int32_t *__restrict__ ord, int32_t n_items, int32_t method, int32_t e_base,
                                 OStat *__restrict__ ostat) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const double *s = item_stats + 4 * (int64_t)i;
    OStat o;
    o.den = (method == XMAP_METHOD_COSINE) ? s[1] : s[2];
    o.item = (uint32_t)i;
    int ex = 0;
    if (o.den > 0.0) {
        frexp(o.den, &ex);
        ex = min(max(ex - e_base, 0), EXP_MAX);
    }
    o.prefix_exp = ((uint32_t)prefix_code[i] << 8) | (uint32_t)ex;
    ostat[ord[i]] = o;
}

static inline size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

struct LayoutWs {
    size_t keys_a, keys_b, vals_a, vals_b, keys_i, perm_i, cub, total, cub_bytes;
};

static int bits_for(int32_t n) {
    int b = 1;
    while (b < 31 && (1LL << b) < (long long)n) ++b;
    return b;
}

static LayoutWs layout_ws(int64_t nnz, int32_t n_users, int32_t n_items) {
    LayoutWs w{};
    size_t cub_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint64_t *)nullptr, (uint64_t *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, (int64_t)nnz, 0, 64);
    size_t off = 0;
    w.keys_a = off; off += align_up(nnz * 8);
    w.keys_b = off; off += align_up(nnz * 8);
    w.vals_a = off; off += align_up(nnz * 4);
    w.vals_b = off; off += align_up(nnz * 4);
    w.keys_i = off; off += align_up(nnz * 8);
    w.perm_i = off; off += align_up(nnz * 4);
    w.cub = off; off += align_up(cub_bytes);
    w.cub_bytes = cub_bytes;
    w.total = off + 256;
    (void)n_users; (void)n_items;
    return w;
}

}  // namespace xmap

using namespace xmap;

extern "C" int xmap_abi_version(void) { return XMAP_B200_ABI_VERSION; }
extern "C" const char *xmap_last_error(void) { return xmap::g_err; }

extern "C" size_t xmap_layout_workspace_bytes(int64_t nnz, int32_t n_users, int32_t n_items) {
    return layout_ws(nnz, n_users, n_items).total;
}

extern "C" int xmap_build_layout(const int32_t *user, const int32_t *item, const float *rating,
                                 int64_t nnz, int32_t n_users, int32_t n_items,
                                 int32_t *csr_ptr, uint64_t *csr_ent, int32_t *csr_src,
                                 int32_t *csc_ptr, uint64_t *csc_ent,
                                 double *user_mu, double *item_stats,
                                 void *workspace, size_t workspace_bytes, void *stream_) {
    cudaStream_t st = (cudaStream_t)stream_;
    if (n_items > (1 << 24)) return fail_msg("xmap_build_layout: n_items exceeds 2^24");
    if (nnz >= (1LL << 31)) return fail_msg("xmap_build_layout: nnz exceeds 2^31-1");
    LayoutWs w = layout_ws(nnz, n_users, n_items);
    if (workspace_bytes < w.total) return fail_msg("xmap_build_layout: workspace too small");
    char *base = (char *)workspace;
    uint64_t *keys_a = (uint64_t *)(base + w.keys_a), *keys_u = (uint64_t *)(base + w.keys_b);
    int32_t *vals_a = (int32_t *)(base + w.vals_a), *perm_u = (int32_t *)(base + w.vals_b);
    uint64_t *keys_i = (uint64_t *)(base + w.keys_i);
    int32_t *perm_i = (int32_t *)(base + w.perm_i);
    void *cub_ws = base + w.cub;
    size_t cub_bytes = w.cub_bytes;
    const int T = 256;
    const unsigned gN = (unsigned)((nnz + T - 1) / T), gN1 = (unsigned)((nnz + 1 + T - 1) / T);
    if (nnz == 0) {
        XMAP_CUDA(cudaMemsetAsync(csr_ptr, 0, sizeof(int32_t) * (n_users + 1), st));
        XMAP_CUDA(cudaMemsetAsync(csc_ptr, 0, sizeof(int32_t) * (n_items + 1), st));
        XMAP_CUDA(cudaMemsetAsync(user_mu, 0, sizeof(double) * n_users, st));
        XMAP_CUDA(cudaMemsetAsync(item_stats, 0, sizeof(double) * 4 * n_items, st));
        return 0;
    }
    // --- CSR order: sort by (user, item)
    make_keys_kernel<<<gN, T, 0, st>>>(user, item, nnz, keys_a, vals_a);
    XMAP_LAUNCH_CHECK();
    XMAP_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_bytes, keys_a, keys_u, vals_a, perm_u, nnz, 0,
                                              32 + bits_for(n_users), st));
    boundaries_kernel<<<gN1, T, 0, st>>>(keys_u, nnz, n_users, csr_ptr);
    XMAP_LAUNCH_CHECK();
    user_mean_kernel<<<(n_users + T - 1) / T, T, 0, st>>>(csr_ptr, perm_u, rating, n_users, user_mu);
    XMAP_LAUNCH_CHECK();
    // --- CSC order: sort by (item, user)
    make_keys_kernel<<<gN, T, 0, st>>>(item, user, nnz, keys_a, vals_a);
    XMAP_LAUNCH_CHECK();
    XMAP_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_bytes, keys_a, keys_i, vals_a, perm_i, nnz, 0,
                                              32 + bits_for(n_items), st));
    boundaries_kernel<<<gN1, T, 0, st>>>(keys_i, nnz, n_items, csc_ptr);
    XMAP_LAUNCH_CHECK();
    item_stats_kernel<<<(unsigned)n_items, IS_THREADS, 0, st>>>(csc_ptr, keys_i, perm_i, rating, user_mu, n_items,
                                                                item_stats);
    XMAP_LAUNCH_CHECK();
    pack_csr_kernel<<<gN, T, 0, st>>>(keys_u, perm_u, rating, item_stats, nnz, csr_ent, csr_src);
    XMAP_LAUNCH_CHECK();
    pack_csc_kernel<<<gN, T, 0, st>>>(keys_i, perm_i, rating, item_stats, nnz, csc_ent);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_row_work(const int32_t *csr_ptr, const int32_t *csc_ptr, const uint64_t *csc_ent,
                             int32_t n_items, int64_t *row_work, void *stream_) {
    cudaStream_t st = (cudaStream_t)stream_;
    const int T = 256;
    if (n_items == 0) return 0;
    XMAP_CUDA(cudaMemsetAsync(row_work, 0, sizeof(int64_t) * (size_t)n_items, st));
    int32_t nnz32 = 0;
    XMAP_CUDA(cudaMemcpyAsync(&nnz32, csc_ptr + n_items, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    XMAP_CUDA(cudaStreamSynchronize(st));
    if (nnz32 <= 0) return 0;
    row_work_kernel<<<(unsigned)(((int64_t)nnz32 + T - 1) / T), T, 0, st>>>(
        csr_ptr, csc_ptr, csc_ent, n_items, (int64_t)nnz32, reinterpret_cast<unsigned long long *>(row_work));
    XMAP_LAUNCH_CHECK();
    return 0;
}

static size_t tri_ws(int64_t nnz, size_t *cub_bytes_out) {
    size_t cub_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint64_t *)nullptr, (uint64_t *)nullptr,
                                    (const uint64_t *)nullptr, (uint64_t *)nullptr, (int64_t)nnz, 0, 64);
    if (cub_bytes_out) *cub_bytes_out = cub_bytes;
    return 3 * align_up((size_t)nnz * 8) + align_up(cub_bytes) + 256;
}

extern "C" size_t xmap_tri_workspace_bytes(int64_t nnz) { return tri_ws(nnz, nullptr); }

extern "C" int xmap_build_tri_layout(const int32_t *csr_ptr, const uint64_t *csr_ent,
                                     const int32_t *csc_ptr, const uint64_t *csc_ent,
                                     const double *user_mu, const double *item_stats, const int32_t *prefix_code,
                                     const int32_t *ord, int32_t n_users, int32_t n_items, int64_t nnz, int32_t method,
                                     int32_t e_base, uint64_t *tcsr_ent, void *csc_aux, void *ostat, int64_t *tri_work,
                                     void *workspace, size_t workspace_bytes, void *stream_) {
    cudaStream_t st = (cudaStream_t)stream_;
    const int T = 256;
    if (n_items > 0) {
        tri_ostat_kernel<<<(n_items + T - 1) / T, T, 0, st>>>(item_stats, prefix_code, ord, n_items, method, e_base,
                                                              reinterpret_cast<OStat *>(ostat));
        XMAP_LAUNCH_CHECK();
        XMAP_CUDA(cudaMemsetAsync(tri_work, 0, sizeof(int64_t) * (size_t)n_items, st));
    }
    if (nnz == 0) return 0;
    size_t cub_bytes = 0;
    if (workspace_bytes < tri_ws(nnz, &cub_bytes)) return fail_msg("xmap_build_tri_layout: workspace too small");
    char *base = (char *)workspace;
    const size_t seg = align_up((size_t)nnz * 8);
    uint64_t *keys_a = (uint64_t *)base, *keys_b = (uint64_t *)(base + seg), *vals_a = (uint64_t *)(base + 2 * seg);
    void *cub_ws = base + 3 * seg;
    const unsigned gN = (unsigned)((nnz + T - 1) / T);
    tri_keys_kernel<<<gN, T, 0, st>>>(csr_ptr, csr_ent, ord, reinterpret_cast<const OStat *>(ostat), n_users, nnz,
                                      keys_a, vals_a);
    XMAP_LAUNCH_CHECK();
    XMAP_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cub_bytes, keys_a, keys_b, vals_a, tcsr_ent, nnz, 0,
                                              32 + bits_for(n_users), st));
    tri_aux_kernel<<<gN, T, 0, st>>>(csr_ptr, csc_ptr, csc_ent, tcsr_ent, user_mu, ord, n_items, nnz, method,
                                     reinterpret_cast<uint4 *>(csc_aux),
                                     reinterpret_cast<unsigned long long *>(tri_work));
    XMAP_LAUNCH_CHECK();
    return 0;
}
