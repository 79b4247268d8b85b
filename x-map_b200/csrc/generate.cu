// AlterEgo generation: per-target-item replacement choice (argmax / exponential
// mechanism / non-private uniform), inversion to a source->target map, and the
// per-user profile rewrite with mean-merge of duplicates.
// Reference: generator.py:27-157, assist.py:210-215.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "common.cuh"

namespace xmap {

__device__ __forceinline__ double philox_uniform(uint64_t seed, uint32_t row) {
    uint32_t c[4] = {row, 0u, 0u, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    // 53-bit uniform in [0, 1)
    return ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0);
}

__global__ void choose_kernel(const int32_t *__restrict__ top_end, const double *__restrict__ top_xsim,
                              const int32_t *__restrict__ top_len, int n_rows, int top_m, int mode, int n_cand,
                              double epsilon, int mapping_range, int gs, const double *__restrict__ uniforms,
                              uint64_t seed, int32_t *__restrict__ chosen) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const int m = min(min(top_len[row], n_cand), 16);
    if (m <= 0) { chosen[row] = -1; return; }
    const int32_t *e = top_end + (size_t)row * top_m;
    const double *xs = top_xsim + (size_t)row * top_m;
    int idx = 0;
    if (mode != 0) {
        const double u = uniforms ? uniforms[row] : philox_uniform(seed, (uint32_t)row);
        if (mode == 1) {
            // generator.py:46-48: exp(eps * xsim / (2 * mapping_range * GS)), then normalise (:54-56)
            double w[16];
            double sum = 0.0;
            const double denom = (double)(2 * mapping_range * gs);
            for (int i = 0; i < m; ++i) { w[i] = exp(__ddiv_rn(__dmul_rn(epsilon, xs[i]), denom)); sum = __dadd_rn(sum, w[i]); }
            for (int i = 0; i < m; ++i) w[i] = __ddiv_rn(w[i], sum);
            // s = np.sum(weights): pairwise with 8 accumulators once m >= 8 (numpy), sequential below
            double s;
            if (m < 8) {
                s = 0.0;
                for (int i = 0; i < m; ++i) s = __dadd_rn(s, w[i]);
            } else {
                s = __dadd_rn(__dadd_rn(__dadd_rn(w[0], w[1]), __dadd_rn(w[2], w[3])),
                              __dadd_rn(__dadd_rn(w[4], w[5]), __dadd_rn(w[6], w[7])));
                for (int i = 8; i < m; ++i) s = __dadd_rn(s, w[i]);
            }
            const double target = __dmul_rn(u, s);
            double cum = 0.0;
            idx = m - 1;
            for (int i = 0; i < m; ++i) {          // np.searchsorted(cumsum, target), side='left' (:68-70)
                cum = __dadd_rn(cum, w[i]);
                if (cum >= target) { idx = i; break; }
            }
        } else {
            // generator.py:109-110: randint(0, len-1) over the first min(m, topn) candidates
            if (m == 1) idx = 0;   // the reference raises here; deliberate, documented divergence
            else idx = min((int)floor(u * (double)(m - 1)), m - 2);
        }
    }
    chosen[row] = e[idx];
}

__global__ void invert_kernel(const int32_t *__restrict__ start_item, const int32_t *__restrict__ chosen,
                              int n_rows, int32_t *__restrict__ map) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const int s = chosen[row];
    if (s >= 0) atomicMax(&map[s], start_item[row]);     // later (= larger target index) wins, assist.py:215
}

// flag[k] = rating k (CSR order) maps to a target item
__global__ void flag_mapped_kernel(const uint64_t *__restrict__ csr_ent, const int32_t *__restrict__ map,
                                   int64_t nnz, uint8_t *__restrict__ flag) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nnz) return;
    flag[k] = map[(uint32_t)(csr_ent[k] & ITEM_MASK)] >= 0;
}

__global__ void mapped_keys_kernel(const int32_t *__restrict__ csr_ptr, const uint64_t *__restrict__ csr_ent,
                                   const int32_t *__restrict__ map, const int32_t *__restrict__ pos,
                                   int64_t n_sel, int n_users, uint64_t *__restrict__ keys) {
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_sel) return;
    const int32_t k = pos[q];
    int lo = 0, hi = n_users;                 // largest u with csr_ptr[u] <= k
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (csr_ptr[mid] <= k) lo = mid; else hi = mid;
    }
    const uint32_t t = (uint32_t)map[(uint32_t)(csr_ent[k] & ITEM_MASK)];
    keys[q] = ((uint64_t)(uint32_t)lo << 32) | t;
}

__global__ void heads_kernel(const uint64_t *__restrict__ keys, int64_t n_sel, int32_t *__restrict__ head) {
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_sel) return;
    head[q] = (q == 0 || keys[q] != keys[q - 1]) ? 1 : 0;
}

// one thread per group head: mean of the group's ratings (np.mean, generator.py:132),
// time of the first member = smallest source item (stable order).
__global__ void merge_kernel(const uint64_t *__restrict__ keys, const int32_t *__restrict__ pos_sorted,
                             const int32_t *__restrict__ head, const int32_t *__restrict__ rank,
                             int64_t n_sel, const uint64_t *__restrict__ csr_ent,
                             const int32_t *__restrict__ csr_src, const int64_t *__restrict__ ts,
                             int32_t *__restrict__ out_user, int32_t *__restrict__ out_item,
                             double *__restrict__ out_rating, int64_t *__restrict__ out_ts) {
    const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (q >= n_sel || !head[q]) return;
    const uint64_t key = keys[q];
    double s = 0.0;
    int c = 0;
    for (int64_t p = q; p < n_sel && keys[p] == key; ++p) {
        s = __dadd_rn(s, (double)__uint_as_float((uint32_t)(csr_ent[pos_sorted[p]] >> 32)));
        ++c;
    }
    const int o = rank[q];
    out_user[o] = (int32_t)(key >> 32);
    out_item[o] = (int32_t)(key & 0xFFFFFFFFu);
    out_rating[o] = __ddiv_rn(s, (double)c);
    out_ts[o] = ts[csr_src[pos_sorted[q]]];
}

static inline size_t au(size_t x) { return (x + 255) & ~(size_t)255; }

struct AeWs {
    size_t flag, pos, nsel, keys_a, keys_b, pos_b, head, rank, cub, cub_bytes, total;
};

static AeWs ae_ws(int64_t nnz) {
    AeWs w{};
    size_t b1 = 0, b2 = 0, b3 = 0;
    cub::DeviceSelect::Flagged(nullptr, b1, thrust::counting_iterator<int32_t>(0), (const uint8_t *)nullptr,
                               (int32_t *)nullptr, (int64_t *)nullptr, (int)nnz);
    cub::DeviceRadixSort::SortPairs(nullptr, b2, (const uint64_t *)nullptr, (uint64_t *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, (int64_t)nnz, 0, 64);
    cub::DeviceScan::ExclusiveSum(nullptr, b3, (const int32_t *)nullptr, (int32_t *)nullptr, (int)nnz);
    size_t cb = b1 > b2 ? b1 : b2;
    if (b3 > cb) cb = b3;
    size_t off = 0;
    w.flag = off; off += au(nnz);
    w.pos = off; off += au(nnz * 4);
    w.nsel = off; off += 256;
    w.keys_a = off; off += au(nnz * 8);
    w.keys_b = off; off += au(nnz * 8);
    w.pos_b = off; off += au(nnz * 4);
    w.head = off; off += au(nnz * 4);
    w.rank = off; off += au(nnz * 4 + 4);
    w.cub = off; off += au(cb);
    w.cub_bytes = cb;
    w.total = off + 256;
    return w;
}

}  // namespace xmap

using namespace xmap;

extern "C" int xmap_choose_mapping(const int32_t *top_end, const double *top_xsim, const int32_t *top_len,
                                   int32_t n_rows, int32_t top_m, int32_t mode, int32_t n_cand, double epsilon,
                                   int32_t mapping_range, int32_t global_sensitivity, const double *uniforms,
                                   uint64_t seed, int32_t *chosen, void *stream_) {
    if (n_rows <= 0) return 0;
    if (mode < 0 || mode > 2) return fail_msg("xmap_choose_mapping: bad mode");
    if (n_cand < 1 || n_cand > 16 || n_cand > top_m) return fail_msg("xmap_choose_mapping: n_cand out of range");
    if (mode == 1 && (mapping_range < 1 || global_sensitivity < 1))
        return fail_msg("xmap_choose_mapping: mapping_range and global sensitivity must be >= 1");
    cudaStream_t st = (cudaStream_t)stream_;
    choose_kernel<<<(n_rows + 255) / 256, 256, 0, st>>>(top_end, top_xsim, top_len, n_rows, top_m, mode, n_cand,
                                                        epsilon, mapping_range, global_sensitivity, uniforms,
                                                        seed, chosen);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_invert_mapping(const int32_t *start_item, const int32_t *chosen, int32_t n_rows,
                                   int32_t *map, void *stream_) {
    if (n_rows <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream_;
    invert_kernel<<<(n_rows + 255) / 256, 256, 0, st>>>(start_item, chosen, n_rows, map);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" size_t xmap_alterego_workspace_bytes(int64_t nnz) { return ae_ws(nnz).total; }

extern "C" int xmap_build_alterego(const int32_t *csr_ptr, const uint64_t *csr_ent, const int32_t *csr_src,
                                   const int64_t *ts, int32_t n_users, int64_t nnz, const int32_t *map,
                                   int32_t *out_user, int32_t *out_item, double *out_rating, int64_t *out_ts,
                                   int64_t *n_out_h, void *workspace, size_t workspace_bytes, void *stream_) {
    cudaStream_t st = (cudaStream_t)stream_;
    *n_out_h = 0;
    if (nnz == 0) return 0;
    AeWs w = ae_ws(nnz);
    if (workspace_bytes < w.total) return fail_msg("xmap_build_alterego: workspace too small");
    char *base = (char *)workspace;
    uint8_t *flag = (uint8_t *)(base + w.flag);
    int32_t *pos = (int32_t *)(base + w.pos), *pos_sorted = (int32_t *)(base + w.pos_b);
    int64_t *nsel_d = (int64_t *)(base + w.nsel);
    uint64_t *keys_a = (uint64_t *)(base + w.keys_a), *keys_b = (uint64_t *)(base + w.keys_b);
    int32_t *head = (int32_t *)(base + w.head), *rank = (int32_t *)(base + w.rank);
    void *cub_ws = base + w.cub;
    size_t cb = w.cub_bytes;
    const int T = 256;
    flag_mapped_kernel<<<(unsigned)((nnz + T - 1) / T), T, 0, st>>>(csr_ent, map, nnz, flag);
    XMAP_LAUNCH_CHECK();
    XMAP_CUDA(cub::DeviceSelect::Flagged(cub_ws, cb, thrust::counting_iterator<int32_t>(0), flag, pos, nsel_d,
                                         (int)nnz, st));
    int64_t n_sel = 0;
    XMAP_CUDA(cudaMemcpyAsync(&n_sel, nsel_d, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    XMAP_CUDA(cudaStreamSynchronize(st));
    if (n_sel == 0) return 0;
    const unsigned gS = (unsigned)((n_sel + T - 1) / T);
    mapped_keys_kernel<<<gS, T, 0, st>>>(csr_ptr, csr_ent, map, pos, n_sel, n_users, keys_a);
    XMAP_LAUNCH_CHECK();
    cb = w.cub_bytes;
    XMAP_CUDA(cub::DeviceRadixSort::SortPairs(cub_ws, cb, keys_a, keys_b, pos, pos_sorted, n_sel, 0, 64, st));
    heads_kernel<<<gS, T, 0, st>>>(keys_b, n_sel, head);
    XMAP_LAUNCH_CHECK();
    cb = w.cub_bytes;
    XMAP_CUDA(cub::DeviceScan::ExclusiveSum(cub_ws, cb, head, rank, (int)n_sel, st));
    merge_kernel<<<gS, T, 0, st>>>(keys_b, pos_sorted, head, rank, n_sel, csr_ent, csr_src, ts, out_user, out_item,
                                   out_rating, out_ts);
    XMAP_LAUNCH_CHECK();
    int32_t last_rank = 0, last_head = 0;
    XMAP_CUDA(cudaMemcpyAsync(&last_rank, rank + (n_sel - 1), 4, cudaMemcpyDeviceToHost, st));
    XMAP_CUDA(cudaMemcpyAsync(&last_head, head + (n_sel - 1), 4, cudaMemcpyDeviceToHost, st));
    XMAP_CUDA(cudaStreamSynchronize(st));
    *n_out_h = (int64_t)last_rank + last_head;
    return 0;
}
