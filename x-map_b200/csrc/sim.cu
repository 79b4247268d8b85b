// Item-item co-rating similarity: triangular sparse R^T R with a fused epilogue
// (adjusted-cosine / cosine, significance weighting, mutuality, exact-zero
// filter, cross-domain label) into per-row neighbour-record lists, then per-row
// top-k selection over the lists.
//
// Reference semantics: baselinerSim.py:84-216 (pairs, similarity, mutuality,
// filter, label), :218-233 (adjacency), assist.py:82-87 (BB set) and
// extender.py:16-44 (find_knn_items).
//
// Work decomposition.  sim(i, j) == sim(j, i), so every unordered pair is
// evaluated once, by the row of the LESS popular item (ord = rank by ascending
// rating count).  Row i walks its raters (CSC); for rater u it streams only the
// suffix of u's ord-sorted ratings that lies on more popular items (csc_aux
// gives the suffix extent directly).  That halves the products (W/2), moves
// almost all of them into rows with few raters (small tables), and leaves the
// popular rows with very few candidate columns (direct-indexed tables).  The
// result is appended to the neighbour-record lists of BOTH rows.
//
// Numerics.  Per pair three exact integer accumulators: n_ij, the mutuality
// count, and the inner product in 64-bit fixed point with 2^-q resolution,
// q = 62 - E_i - E_j, where 2^(E-1) <= den < 2^E for the item's norm den
// (entries and ostat carry E - e_base in 7 bits; r2_bits = 2 e_base).  By
// Cauchy-Schwarz every product and every partial co-rater sum is at most
// den_i den_j < 2^(E_i + E_j), so the final sum is below 2^62 + n and fits
// (the lo/hi words may wrap on the way; only the final sum matters), and the
// rounding error of the cosine is at most n 2^-61 whatever the rating scale.
// Because integer addition is associative the result does not depend on the
// order products arrive in: any split of a row over lanes, warps or GPUs gives
// bit-identical output.  The 64-bit sum is kept as two 32-bit shared-memory
// words (native 32-bit atomics; the carry out of the low word is recovered from
// the value the atomic returns).
//
// Memory.  The hot loop streams 8-byte entries of the ord-sorted CSR
// (coalesced within a suffix, read-only path); algorithmic bytes = 8 per product.
#include "common.cuh"

namespace xmap {

constexpr int KMAX = XMAP_KMAX;

struct __align__(16) OStat {
    double den;
    uint32_t item;
    uint32_t prefix_exp;      // prefix << 8 | item exponent
};

// 16-byte accumulator cell.
//   hash   : key = ord(j) + 1 (0 = empty), cnt = n << 16 | mutu
//   direct : key = #agreeing co-raters (= mutu), cnt = #disagreeing  (n = key + cnt)
//   lo/hi  : the two halves of the 64-bit fixed-point inner product
struct __align__(16) Cell {
    unsigned key, cnt, lo, hi;
};

// 16-byte neighbour record: bits of sim, other_item | mutu << 32; the co-rating count n of the record at
// position p lives in the parallel array rec_n[p] (only the winners of the selection ever read it), so the item
// index and both counts are full 32-bit values.
struct __align__(16) Rec {
    unsigned long long sim;
    unsigned long long pack;
};
__device__ __forceinline__ unsigned long long rec_pack(unsigned item, unsigned mutu) {
    return (unsigned long long)item | ((unsigned long long)mutu << 32);
}
__device__ __forceinline__ int rec_item(unsigned long long p) { return int((unsigned)p); }
__device__ __forceinline__ int rec_mutu(unsigned long long p) { return int((unsigned)(p >> 32)); }

// Everything a row's group needs before it can start, gathered once at planning time into one
// 48-byte record per launch slot (one load instead of a chain of dependent gathers).
struct __align__(16) RowHdr {
    int row, oi, lo, hi;          // item, its ord, its rater range (CSC positions; a segment of it for split rows)
    long long work;               // tri_work[row]
    double den;                   // ostat[oi].den
    long long rec_base;           // rec_ptr[row]
    unsigned prefix_exp;          // ostat[oi].prefix_exp
    int rec_cap;                  // rec_ptr[row + 1] - rec_ptr[row]
};
static_assert(sizeof(RowHdr) == 48, "RowHdr layout");

__device__ __forceinline__ RowHdr load_hdr(const RowHdr *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    const uint4 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    RowHdr h;
    h.row = (int)a.x; h.oi = (int)a.y; h.lo = (int)a.z; h.hi = (int)a.w;
    h.work = (long long)(((unsigned long long)b.y << 32) | b.x);
    h.den = __hiloint2double((int)b.w, (int)b.z);
    h.rec_base = (long long)(((unsigned long long)c.y << 32) | c.x);
    h.prefix_exp = c.z; h.rec_cap = (int)c.w;
    return h;
}

__global__ void row_headers_kernel(xmap_sim_args a, const int32_t *__restrict__ rows, int n_rows,
                                   const int32_t *__restrict__ seg_lo, const int32_t *__restrict__ seg_hi,
                                   RowHdr *__restrict__ out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int row = rows[r];
    const OStat *ostat = reinterpret_cast<const OStat *>(a.ostat);
    RowHdr h;
    h.row = row; h.oi = a.ord[row];
    h.lo = seg_lo ? seg_lo[r] : a.csc_ptr[row];
    h.hi = seg_hi ? seg_hi[r] : a.csc_ptr[row + 1];
    h.work = a.tri_work[row];
    const OStat si = ostat[h.oi];
    h.den = si.den; h.prefix_exp = si.prefix_exp;
    h.rec_base = a.rec_ptr[row];
    h.rec_cap = (int)(a.rec_ptr[row + 1] - a.rec_ptr[row]);
    out[r] = h;
}

__host__ __device__ __forceinline__ long long hash_cells_for(long long work) {
    long long c = (work * 4 + 2) / 3;
    return c < 32 ? 32 : c;
}

// --------------------------------------------------------------------------
// Accumulate + epilogue of one row by a group of threads (one warp, or a whole CTA).
// --------------------------------------------------------------------------
template <bool CTA_ROW>
__device__ __forceinline__ void group_sync() {
    if (CTA_ROW) __syncthreads(); else __syncwarp();
}

// rater descriptor of one lane: suffix start | ge_i << 31, suffix length, centred rating, user mean
struct RaterDesc {
    unsigned start;
    int len;
    double ci, mu;
};

__device__ __forceinline__ RaterDesc load_rater(const xmap_sim_args &a, int e, int hi) {
    RaterDesc d{0u, 0, 0.0, 0.0};
    if (e < hi) {
        const uint2 ce = ld_ent(a.csc_ent + e);
        const uint4 ax = __ldg(reinterpret_cast<const uint4 *>(a.csc_aux) + e);      // {pos, len, mean of the rater}
        d.mu = __hiloint2double((int)ax.w, (int)ax.z);
        d.ci = (double)__uint_as_float(ce.y) - d.mu;
        d.start = (ax.x + 1u) | (ce.x & 0x80000000u);      // bit 31 = (rating of i >= average of i)
        d.len = (int)ax.y;
    }
    return d;
}

// Accumulate + epilogue of one row by a group of threads (one warp, or a whole CTA).
//   T    : cells_cap accumulator cells;  occ : cells_cap slot indices (IDX = uint16 in shared memory)
//   s_cnt: one int of group-shared scratch (CTA mode)
// A row with very many raters can be cut into segments of its rater list, one CTA each: every
// segment accumulates into its own shared-memory table, adds it into the row's table in global
// memory (exact integer adds, so the split never changes a bit), and the CTA that arrives last
// reloads the sum, clears the global table for the next use and runs the epilogue.
struct SplitCtx {
    uint4 *gtab;        // the row's direct-indexed table in global memory, zero outside a stage
    int *done;          // arrival counter of the row's segments, zero outside a stage
    int nseg;
};

template <bool CTA_ROW, class IDX>
__device__ void tri_row(const xmap_sim_args &a, Cell *__restrict__ T, IDX *__restrict__ occ_list, int *s_cnt,
                        int cells_cap, const RowHdr *hdr_p, const SplitCtx *sp = nullptr) {
    const int lane = threadIdx.x & 31;
    const int gwarps = CTA_ROW ? (blockDim.x >> 5) : 1;
    const int gw = CTA_ROW ? (threadIdx.x >> 5) : 0;
    const int gthreads = gwarps * 32, gtid = gw * 32 + lane;
    const unsigned lt_mask = (1u << lane) - 1u;
    const OStat *__restrict__ ostat = reinterpret_cast<const OStat *>(a.ostat);

    const RowHdr hd = load_hdr(hdr_p);
    const int row = hd.row, oi = hd.oi;
    const int e_i = int(hd.prefix_exp & 0xFFu);
    const unsigned prefix_i = hd.prefix_exp >> 8;
    const int lo = hd.lo, hi = hd.hi;
    const long long work = hd.work;
    const int rtop = a.n_items - 1 - oi;                   // items more popular than `row`
    const long long hcells = hash_cells_for(work);
    const bool direct = (long long)rtop <= hcells;
    const long long ncell_ll = direct ? (long long)rtop : hcells;
    if (ncell_ll > cells_cap || (!direct && min((long long)(hi - lo), work) >= 65536)) {
        if (gtid == 0) atomicExch(a.error_flag, ncell_ll > cells_cap ? 1 : 3);
        return;
    }
    const int ncell = (int)ncell_ll;
    uint4 *T4 = reinterpret_cast<uint4 *>(T);
    for (int s = gtid; s < ncell; s += gthreads) T4[s] = make_uint4(0u, 0u, 0u, 0u);
    if (CTA_ROW && gtid == 0) *s_cnt = 0;
    group_sync<CTA_ROW>();

    // ---- accumulate: batches of 32 raters per warp, products flattened over the lanes ----------
    const int qbase = 62 - a.r2_bits;                      // 62 - 2 e_base
    const int top_ord = a.n_items - 1;
    // Many raters: one batch per warp.  Few raters (fewer batches than warps): every warp walks every
    // batch and takes every gwarps-th chunk of 32 products, so the whole group stays busy.
    const bool coop = CTA_ROW && ((hi - lo + 31) >> 5) < gwarps;
    const int bfirst = coop ? 0 : gw, bstride = coop ? 1 : gwarps;
    const int cfirst = coop ? gw : 0, cstride = coop ? gwarps : 1;
    constexpr int UC = 2;                                  // chunks in flight per warp
    RaterDesc nxt = load_rater(a, lo + bfirst * 32 + lane, hi);
    for (int b0 = lo + bfirst * 32; b0 < hi; b0 += bstride * 32) {
        const RaterDesc cur = nxt;
        nxt = load_rater(a, b0 + bstride * 32 + lane, hi);  // prefetch the next batch of this warp
        int incl = cur.len;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += t;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        const int excl = incl - cur.len;
        for (int t0 = cfirst * 32; t0 < total; t0 += cstride * 32 * UC) {
            uint2 en[UC];
            unsigned st_l[UC];
            double ci_l[UC], mu_l[UC];
            bool valid[UC];
#pragma unroll
            for (int u = 0; u < UC; ++u) {
                const int t = t0 + u * cstride * 32 + lane;
                int l = 0;                                 // smallest lane with incl > t
#pragma unroll
                for (int step = 16; step >= 1; step >>= 1) {
                    const int v = __shfl_sync(0xffffffffu, incl, l + step - 1);
                    if (v <= t) l += step;
                }
                st_l[u] = __shfl_sync(0xffffffffu, cur.start, l);
                const int ex_l = __shfl_sync(0xffffffffu, excl, l);
                ci_l[u] = __shfl_sync(0xffffffffu, cur.ci, l);
                mu_l[u] = __shfl_sync(0xffffffffu, cur.mu, l);
                valid[u] = t < total;
                if (valid[u]) en[u] = ld_ent(a.tcsr_ent + ((st_l[u] & 0x7FFFFFFFu) + (unsigned)(t - ex_l)));
            }
#pragma unroll
            for (int u = 0; u < UC; ++u) {
                if (!valid[u]) continue;
                const int oj = ent_item(en[u].x);
                const double cj = (double)__uint_as_float(en[u].y) - mu_l[u];
                const double p = __dmul_rn(ci_l[u], cj);
                const int q = qbase - (e_i + ent_exp(en[u].x));
                const long long fx = __double2ll_rn(p * pow2d(q));
                const unsigned agree = ((unsigned)ent_ge(en[u].x) == (st_l[u] >> 31)) ? 1u : 0u;
                int slot;
                bool ok = true;
                if (direct) {
                    slot = top_ord - oj;                   // in [0, rtop)
                    atomicAdd(agree ? &T[slot].key : &T[slot].cnt, 1u);
                } else {
                    const unsigned key = (unsigned)oj + 1u;
                    slot = (int)__umulhi((unsigned)oj * 2654435761u, (unsigned)ncell);
                    ok = false;
                    for (int probe = 0; probe < ncell; ++probe) {
                        unsigned c = *(volatile unsigned *)&T[slot].key;
                        if (c != key) {
                            if (c == 0u) c = atomicCAS(&T[slot].key, 0u, key);
                            if (c != 0u && c != key) { slot = (slot + 1 == ncell) ? 0 : slot + 1; continue; }
                        }
                        ok = true;
                        break;
                    }
                    if (ok) atomicAdd(&T[slot].cnt, (1u << 16) | agree);
                    else atomicExch(a.error_flag, 1);
                }
                if (ok) {
                    if (sizeof(IDX) == 4) {
                        // table in global memory: one native 64-bit reduction, nothing to wait for
                        atomicAdd(reinterpret_cast<unsigned long long *>(&T[slot].lo), (unsigned long long)fx);
                    } else {
                        const unsigned flo = (unsigned)(unsigned long long)fx;
                        unsigned fhi = (unsigned)((unsigned long long)fx >> 32);
                        if (flo) {
                            const unsigned old = atomicAdd(&T[slot].lo, flo);
                            fhi += ((unsigned)(old + flo) < old) ? 1u : 0u;
                        }
                        if (fhi) atomicAdd(&T[slot].hi, fhi);
                    }
                }
            }
        }
    }
    group_sync<CTA_ROW>();

    if (CTA_ROW && sp) {
        if (!direct) {                                     // only direct-indexed rows can be merged cell by cell
            if (gtid == 0) atomicExch(a.error_flag, 1);
            return;
        }
        for (int s = gtid; s < ncell; s += gthreads) {
            const uint4 v = T4[s];
            if (v.x) atomicAdd(&sp->gtab[s].x, v.x);
            if (v.y) atomicAdd(&sp->gtab[s].y, v.y);
            const unsigned long long fx = ((unsigned long long)v.w << 32) | v.z;
            if (fx) atomicAdd(reinterpret_cast<unsigned long long *>(&sp->gtab[s].z), fx);
        }
        __threadfence();
        __syncthreads();
        if (gtid == 0) *s_cnt = (atomicAdd(sp->done, 1) == sp->nseg - 1) ? 1 : 0;
        __syncthreads();
        const bool last = *s_cnt != 0;
        __syncthreads();
        if (!last) return;
        __threadfence();
        for (int s = gtid; s < ncell; s += gthreads) {
            T4[s] = __ldcg(sp->gtab + s);
            sp->gtab[s] = make_uint4(0u, 0u, 0u, 0u);
        }
        if (gtid == 0) { *sp->done = 0; *s_cnt = 0; }
        __syncthreads();
    }

    // ---- index list of the occupied cells (order irrelevant) ---------------------------------------
    int n_ent = 0;
    for (int s0 = gw * 32; s0 < ncell; s0 += gthreads) {
        const int s = s0 + lane;
        bool occ = false;
        if (s < ncell) {
            const uint2 kc = *reinterpret_cast<const uint2 *>(&T[s]);
            occ = direct ? (kc.x | kc.y) != 0u : kc.x != 0u;
        }
        const unsigned m = __ballot_sync(0xffffffffu, occ);
        if (m) {
            int base = n_ent;
            if (CTA_ROW) {
                if (lane == 0) base = atomicAdd(s_cnt, __popc(m));
                base = __shfl_sync(0xffffffffu, base, 0);
            }
            if (occ) occ_list[base + __popc(m & lt_mask)] = (IDX)s;
            n_ent += __popc(m);
        }
    }
    group_sync<CTA_ROW>();
    if (CTA_ROW) n_ent = *s_cnt;
    if (gtid == 0 && n_ent) a.row_npairs[row] += n_ent;     // this row's group is the only writer

    // ---- epilogue pass 1: similarity, filter, label of every occupied cell, in place ---------------
    // baselinerSim.py:163-173 / :125-141, :89, :95, :191, :207.  A kept cell becomes
    //   hash row   : {other item, n << 16 | mutu, sim bits}     (n < 2^16: checked at entry)
    //   direct row : {mutu, n, sim bits}                        (the other item follows from the slot)
    // and a dropped one becomes zero.
    constexpr int EU = 2;
    int nkept = 0;
    for (int i0 = gtid; i0 < n_ent; i0 += gthreads * EU) {
        uint4 cv[EU];
        int sidx[EU];
        unsigned n[EU], mutu[EU];
        OStat sj[EU];
#pragma unroll
        for (int u = 0; u < EU; ++u) {
            const int i = i0 + u * gthreads;
            sidx[u] = -1;
            if (i < n_ent) {
                sidx[u] = (int)occ_list[i];
                cv[u] = T4[sidx[u]];
                int oj;
                if (direct) { n[u] = cv[u].x + cv[u].y; mutu[u] = cv[u].x; oj = top_ord - sidx[u]; }
                else { oj = (int)cv[u].x - 1; n[u] = cv[u].y >> 16; mutu[u] = cv[u].y & 0xFFFFu; }
                sj[u] = ostat[oj];
            }
        }
#pragma unroll
        for (int u = 0; u < EU; ++u) {
            if (sidx[u] < 0) continue;
            uint4 out = make_uint4(0u, 0u, 0u, 0u);
            const int q = qbase - (e_i + int(sj[u].prefix_exp & 0xFFu));
            const long long fx = (long long)(((unsigned long long)cv[u].w << 32) | (unsigned long long)cv[u].z);
            if (fx == 0 || mutu[u] == 0u) { T4[sidx[u]] = out; continue; }     // sim == 0 or mutu == 0: filtered
            const double inner = (double)fx * pow2d(-q);
            const double dd = __dmul_rn(hd.den, sj[u].den);
            const double cosv = (dd != 0.0) ? __ddiv_rn(inner, dd) : 0.0;
            const int mn = min((int)n[u], a.num_atleast);
            const double sim = __ddiv_rn(__dmul_rn(cosv, (double)mn), (double)a.num_atleast);
            if (sim != 0.0 && mutu[u] != 0u) {
                ++nkept;
                const unsigned long long sb = (unsigned long long)__double_as_longlong(sim);
                out = direct ? make_uint4(mutu[u], n[u], (unsigned)sb, (unsigned)(sb >> 32))
                             : make_uint4(sj[u].item, (n[u] << 16) | mutu[u], (unsigned)sb, (unsigned)(sb >> 32));
                if ((sj[u].prefix_exp >> 8) != prefix_i) { a.bb[row] = 1; a.bb[sj[u].item] = 1; }
            }
            T4[sidx[u]] = out;
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) nkept += __shfl_xor_sync(0xffffffffu, nkept, off);
    if (nkept == 0) return;                                // warp-uniform; no barrier follows

    // ---- epilogue pass 2: one reservation per warp in the row's own list, then append the records
    // to the own list (compacted) and to each neighbour's list (one cursor bump per record) --------
    Rec *__restrict__ rec = reinterpret_cast<Rec *>(a.rec);
    const long long base_i = hd.rec_base;
    const int cap_i = hd.rec_cap;
    int wbase = 0;
    if (lane == 0) wbase = atomicAdd(a.rec_cnt + row, nkept);
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    if (a.count_only) {                                    // sizing pass: only the list lengths are wanted
        for (int i = gw * 32 + lane; i < n_ent; i += gthreads) {
            const int sl = (int)occ_list[i];
            const uint4 cv = T4[sl];
            if ((cv.z | cv.w) != 0u) atomicAdd(a.rec_cnt + (direct ? __ldg(a.ord_item + (top_ord - sl)) : (int)cv.x), 1);
        }
        return;
    }
    if (wbase + nkept > cap_i) {
        if (lane == 0) atomicExch(a.error_flag, 2);
        return;
    }
    for (int i0 = gw * 32; i0 < n_ent; i0 += gthreads * EU) {
        uint4 cv[EU];
        bool keep[EU];
        long long base_j[EU];
        int cap_j[EU], p2[EU], jit[EU];
        unsigned nn[EU], mu[EU];
#pragma unroll
        for (int u = 0; u < EU; ++u) {
            const int i = i0 + u * gthreads + lane;
            int sl = 0;
            cv[u] = make_uint4(0u, 0u, 0u, 0u);
            if (i < n_ent) { sl = (int)occ_list[i]; cv[u] = T4[sl]; }
            keep[u] = (cv[u].z | cv[u].w) != 0u;
            jit[u] = 0; nn[u] = mu[u] = 0u;
            if (keep[u]) {
                if (direct) { jit[u] = __ldg(a.ord_item + (top_ord - sl)); mu[u] = cv[u].x; nn[u] = cv[u].y; }
                else { jit[u] = (int)cv[u].x; nn[u] = cv[u].y >> 16; mu[u] = cv[u].y & 0xFFFFu; }
            }
        }
#pragma unroll
        for (int u = 0; u < EU; ++u) {
            if (keep[u]) {
                base_j[u] = a.rec_ptr[jit[u]];
                cap_j[u] = (int)(a.rec_ptr[jit[u] + 1] - base_j[u]);
                p2[u] = atomicAdd(a.rec_cnt + jit[u], 1);
            }
        }
#pragma unroll
        for (int u = 0; u < EU; ++u) {
            const unsigned m = __ballot_sync(0xffffffffu, keep[u]);
            if (keep[u]) {
                const unsigned long long sb = ((unsigned long long)cv[u].w << 32) | cv[u].z;
                const long long own = base_i + wbase + __popc(m & lt_mask);
                rec[own] = Rec{sb, rec_pack((unsigned)jit[u], mu[u])};
                a.rec_n[own] = (int)nn[u];
                if (p2[u] < cap_j[u]) {
                    rec[base_j[u] + p2[u]] = Rec{sb, rec_pack((unsigned)row, mu[u])};
                    a.rec_n[base_j[u] + p2[u]] = (int)nn[u];
                } else atomicExch(a.error_flag, 2);
            }
            wbase += __popc(m);
        }
    }
}

// shared memory per row: cells_cap cells + cells_cap 16-bit slot indices
__host__ __device__ constexpr size_t row_smem_bytes(int cells_cap) { return (size_t)cells_cap * (sizeof(Cell) + 2); }

// one warp per row, tables in shared memory, rows sorted by descending work
__global__ void __launch_bounds__(128) tri_warp_kernel(xmap_sim_args a, const RowHdr *__restrict__ hdr, int n_rows,
                                                       int cells_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const int r = blockIdx.x * (blockDim.x >> 5) + warp;
    if (r >= n_rows) return;
    Cell *T = reinterpret_cast<Cell *>(smem_raw) + (size_t)warp * cells_cap;
    unsigned short *occ = reinterpret_cast<unsigned short *>(smem_raw + (size_t)(blockDim.x >> 5) * cells_cap * sizeof(Cell)) +
                          (size_t)warp * cells_cap;
    tri_row<false, unsigned short>(a, T, occ, nullptr, cells_cap, hdr + r);
}

// one CTA per row, table in shared memory
__global__ void __launch_bounds__(512) tri_cta_kernel(xmap_sim_args a, const RowHdr *__restrict__ hdr, int n_rows,
                                                       int cells_cap) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_cnt;
    tri_row<true, unsigned short>(a, reinterpret_cast<Cell *>(smem_raw),
                                  reinterpret_cast<unsigned short *>(smem_raw + (size_t)cells_cap * sizeof(Cell)),
                                  &s_cnt, cells_cap, hdr + blockIdx.x);
}

// one CTA per segment of a split row (see SplitCtx)
__global__ void __launch_bounds__(512) tri_split_kernel(xmap_sim_args a, const RowHdr *__restrict__ hdr,
                                                         const int32_t *__restrict__ seg_slot,
                                                         const int32_t *__restrict__ slot_nseg, int cells_cap,
                                                         uint4 *__restrict__ gtab, int *__restrict__ done) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_cnt;
    const int g = blockIdx.x, slot = seg_slot[g];
    SplitCtx sp{gtab + (size_t)slot * cells_cap, done + slot, slot_nseg[slot]};
    tri_row<true, unsigned short>(a, reinterpret_cast<Cell *>(smem_raw),
                                  reinterpret_cast<unsigned short *>(smem_raw + (size_t)cells_cap * sizeof(Cell)),
                                  &s_cnt, cells_cap, hdr + g, &sp);
}

// persistent CTAs, tables in global memory (rows whose table exceeds shared memory):
// per CTA cells_cap cells followed by cells_cap 32-bit slot indices
__global__ void __launch_bounds__(512) tri_gmem_kernel(xmap_sim_args a, const RowHdr *__restrict__ hdr, int n_rows,
                                                        int cells_cap, unsigned char *__restrict__ gtab) {
    __shared__ int s_cnt;
    unsigned char *mine = gtab + (size_t)blockIdx.x * (((size_t)cells_cap * (sizeof(Cell) + 4) + 15) & ~(size_t)15);
    Cell *T = reinterpret_cast<Cell *>(mine);
    unsigned *occ = reinterpret_cast<unsigned *>(mine + (size_t)cells_cap * sizeof(Cell));
    for (int r = blockIdx.x; r < n_rows; r += gridDim.x) {
        tri_row<true, unsigned>(a, T, occ, &s_cnt, cells_cap, hdr + r);
        __syncthreads();
    }
}

// --------------------------------------------------------------------------
// Selection (extender.py:16-44).
// --------------------------------------------------------------------------
constexpr int SEL_BUF = 192;                      // survivors per list
constexpr int SEL_WARP_BYTES = 2 * SEL_BUF * 16;  // two survivor buffers; aliases the 2 x 256-bin histogram (sim_bin)

// list membership of neighbour j for row i: bit 0 = list 0, bit 1 = list 1
//   BB row: list 0 = other-domain neighbours, list 1 = same-domain (extender.py:30-35)
//   NB row: list 0 = BB neighbours, list 1 = every neighbour (extender.py:37-43, bug :41-42)
__device__ __forceinline__ unsigned list_bits(const xmap_sim_args &a, bool bb_i, int dom_i, int j) {
    if (bb_i) return ((__ldg(a.contains + j) >> dom_i) & 1) ? 2u : 1u;
    return 2u | (a.bb[j] ? 1u : 0u);
}

struct __align__(16) Surv {
    unsigned long long key;
    int q, j;
};

constexpr int SU = 4;                             // records per lane per step of the streaming passes
constexpr int SEL_DIRECT = 64;                    // lists up to this long skip the histogram

__global__ void __launch_bounds__(128) select_warp_kernel(xmap_sim_args a, const int32_t *__restrict__ rows,
                                                          int n_rows) {
    __shared__ __align__(16) unsigned char s_sel[4][SEL_WARP_BYTES];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r = blockIdx.x * 4 + warp;
    if (r >= n_rows) return;
    const int row = rows ? rows[r] : r;
    const int m = a.rec_cnt[row];
    if (m > XMAP_SELECT_LONG) return;
    const int K = a.k;
    if (m == 0) {
        if (lane < 2) a.tab_len[(size_t)row * 2 + lane] = 0;
        return;
    }
    const Rec *__restrict__ R = reinterpret_cast<const Rec *>(a.rec) + a.rec_ptr[row];
    const int32_t *__restrict__ RN = a.rec_n + a.rec_ptr[row];
    const bool bb_i = a.bb[row] != 0;
    const int dom_i = a.dom_code[row];
    const unsigned lt_mask = (1u << lane) - 1u;

    if (m <= 32) {
        // the whole list sits in one register per lane: rank by counting
        unsigned long long key = 0ull, sbits = 0ull, pack = 0ull;
        unsigned lb = 0u;
        int j = 0x7FFFFFFF;
        if (lane < m) {
            const Rec v = R[lane];
            sbits = v.sim; pack = v.pack;
            key = sbits & 0x7FFFFFFFFFFFFFFFull;
            j = rec_item(pack);
            lb = list_bits(a, bb_i, dom_i, j);
        }
        int rank0 = 0, rank1 = 0, n0 = 0, n1 = 0;
        for (int t = 0; t < m; ++t) {
            const unsigned long long k2 = __shfl_sync(0xffffffffu, key, t);
            const int j2 = __shfl_sync(0xffffffffu, j, t);
            const unsigned lb2 = __shfl_sync(0xffffffffu, lb, t);
            const bool before = better(k2, j2, key, j);
            if (lb2 & 1u) { ++n0; if (before) ++rank0; }
            if (lb2 & 2u) { ++n1; if (before) ++rank1; }
        }
        if ((lb & 1u) && rank0 < K) {
            const size_t o = ((size_t)row * 2 + 0) * K + rank0;
            a.tab_idx[o] = j; a.tab_sim[o] = __longlong_as_double((long long)sbits);
            a.tab_mutu[o] = rec_mutu(pack); a.tab_n[o] = RN[lane];
        }
        if ((lb & 2u) && rank1 < K) {
            const size_t o = ((size_t)row * 2 + 1) * K + rank1;
            a.tab_idx[o] = j; a.tab_sim[o] = __longlong_as_double((long long)sbits);
            a.tab_mutu[o] = rec_mutu(pack); a.tab_n[o] = RN[lane];
        }
        if (lane == 0) {
            a.tab_len[(size_t)row * 2 + 0] = min(n0, K);
            a.tab_len[(size_t)row * 2 + 1] = min(n1, K);
        }
        return;
    }

    unsigned *hist = reinterpret_cast<unsigned *>(s_sel[warp]);      // [2][SIM_BINS]
    Surv *buf[2] = {reinterpret_cast<Surv *>(s_sel[warp]), reinterpret_cast<Surv *>(s_sel[warp]) + SEL_BUF};
    int nb[2] = {0, 0}, want[2] = {0, 0}, bstar[2] = {0, 0};
    bool overflow[2] = {false, false};
    if (m > SEL_DIRECT) {
        // ---- pass A: per-list histogram of |sim| -------------------------------------------------
        for (int b = lane; b < 2 * SIM_BINS; b += 32) hist[b] = 0u;
        __syncwarp();
        // long lists: the histogram is built from every 4th block of 128 records.  The threshold bin of
        // the sample has at least min(K, sample members) entries at or above it, so the full list has
        // too, and pass B (which sees every record) keeps a superset of the true top-K.
        const int stride = (m > 1024) ? 4 : 1;
        int n0 = 0, n1 = 0;
        for (int q0 = 0; q0 < m; q0 += 32 * SU * stride) {
            Rec v[SU];
            unsigned lb[SU];
#pragma unroll
            for (int u = 0; u < SU; ++u) {
                const int q = q0 + u * 32 + lane;
                v[u] = (q < m) ? R[q] : Rec{0ull, 0ull};
            }
#pragma unroll
            for (int u = 0; u < SU; ++u)
                lb[u] = (q0 + u * 32 + lane < m) ? list_bits(a, bb_i, dom_i, rec_item(v[u].pack)) : 0u;
#pragma unroll
            for (int u = 0; u < SU; ++u) {
                const int bin = sim_bin(v[u].sim);
                if (lb[u] & 1u) { atomicAdd(&hist[bin], 1u); ++n0; }
                if (lb[u] & 2u) { atomicAdd(&hist[SIM_BINS + bin], 1u); ++n1; }
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            n0 += __shfl_xor_sync(0xffffffffu, n0, off);
            n1 += __shfl_xor_sync(0xffffffffu, n1, off);
        }
        __syncwarp();
        for (int list = 0; list < 2; ++list) {
            want[list] = min(K, list == 0 ? n0 : n1);       // of the sample; the final value comes from pass B
            if (want[list] < K) continue;                    // fewer than K sampled members: keep everything (b* = 0)
            // largest bin b* such that #(bin >= b*) >= want: scan the histogram from the top
            int run = 0;
            bool found = false;
            for (int hb = SIM_BINS - 32; hb >= 0 && !found; hb -= 32) {
                unsigned suf = hist[list * SIM_BINS + hb + lane];      // suffix sums, highest lane = highest bin
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const unsigned t = __shfl_down_sync(0xffffffffu, suf, off);
                    if (lane + off < 32) suf += t;
                }
                const unsigned hit = __ballot_sync(0xffffffffu, run + (int)suf >= want[list]);
                if (hit) { bstar[list] = hb + (31 - __clz(hit)); found = true; }
                else run += (int)__shfl_sync(0xffffffffu, suf, 0);
            }
        }
        __syncwarp();                                      // the histogram is dead; its memory becomes the survivor buffers
    }
    // ---- pass B: the survivors of both lists (everything when the list fits the buffer) ------------
    int nl0 = 0, nl1 = 0;                                  // members of each list, counted over every record
    for (int q0 = 0; q0 < m; q0 += 32 * SU) {
        Rec v[SU];
        unsigned lb[SU];
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const int q = q0 + u * 32 + lane;
            v[u] = (q < m) ? R[q] : Rec{0ull, 0ull};
        }
#pragma unroll
        for (int u = 0; u < SU; ++u)
            lb[u] = (q0 + u * 32 + lane < m) ? list_bits(a, bb_i, dom_i, rec_item(v[u].pack)) : 0u;
#pragma unroll
        for (int u = 0; u < SU; ++u) {
            const unsigned long long key = v[u].sim & 0x7FFFFFFFFFFFFFFFull;
            const int bin = sim_bin(key);
            nl0 += int(lb[u] & 1u); nl1 += int((lb[u] >> 1) & 1u);
#pragma unroll
            for (int list = 0; list < 2; ++list) {
                const bool take = ((lb[u] >> list) & 1u) && bin >= bstar[list];
                const unsigned mk = __ballot_sync(0xffffffffu, take);
                if (overflow[list] || nb[list] + __popc(mk) > SEL_BUF) { overflow[list] = true; continue; }
                if (take) buf[list][nb[list] + __popc(mk & lt_mask)] = Surv{key, q0 + u * 32 + lane, rec_item(v[u].pack)};
                nb[list] += __popc(mk);
            }
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        nl0 += __shfl_xor_sync(0xffffffffu, nl0, off);
        nl1 += __shfl_xor_sync(0xffffffffu, nl1, off);
    }
    want[0] = min(K, nl0); want[1] = min(K, nl1);
    __syncwarp();
    // ---- K arg-best rounds per list --------------------------------------------------------------
    for (int list = 0; list < 2; ++list) {
        int got = 0;
        const size_t o = ((size_t)row * 2 + list) * K;
        unsigned long long last_k = ~0ull; int last_t = -1;
        if (!overflow[list] && nb[list] <= 64) {
            // at most two survivors per lane: rank by counting, every winner writes its own table entry
            const int n = nb[list];
            Surv m0{0ull, -1, 0x7FFFFFFF}, m1{0ull, -1, 0x7FFFFFFF};
            if (lane < n) m0 = buf[list][lane];
            if (lane + 32 < n) m1 = buf[list][lane + 32];
            int r0 = 0, r1 = 0;
            for (int t = 0; t < n; ++t) {
                const Surv o2 = buf[list][t];               // same address in every lane: a broadcast read
                r0 += better(o2.key, o2.j, m0.key, m0.j) ? 1 : 0;
                r1 += better(o2.key, o2.j, m1.key, m1.j) ? 1 : 0;
            }
            if (lane < n && r0 < want[list]) {
                const Rec v = R[m0.q];
                a.tab_idx[o + r0] = m0.j;
                a.tab_sim[o + r0] = __longlong_as_double((long long)v.sim);
                a.tab_mutu[o + r0] = rec_mutu(v.pack); a.tab_n[o + r0] = RN[m0.q];
            }
            if (lane + 32 < n && r1 < want[list]) {
                const Rec v = R[m1.q];
                a.tab_idx[o + r1] = m1.j;
                a.tab_sim[o + r1] = __longlong_as_double((long long)v.sim);
                a.tab_mutu[o + r1] = rec_mutu(v.pack); a.tab_n[o + r1] = RN[m1.q];
            }
            if (lane == 0) a.tab_len[(size_t)row * 2 + list] = want[list];
            continue;
        }
        for (int rr = 0; rr < want[list]; ++rr) {
            unsigned long long bk = 0; int bt = 0x7FFFFFFF, bp = -1;
            if (!overflow[list]) {
                for (int q = lane; q < nb[list]; q += 32) {
                    const Surv sv = buf[list][q];
                    if (rr > 0 && !better(last_k, last_t, sv.key, sv.j)) continue;
                    if (bp < 0 || better(sv.key, sv.j, bk, bt)) { bk = sv.key; bt = sv.j; bp = sv.q; }
                }
            } else {   // many equal similarities in the threshold bin: rounds over all records
                for (int q = lane; q < m; q += 32) {
                    const Rec v = R[q];
                    const int tt = rec_item(v.pack);
                    if (!((list_bits(a, bb_i, dom_i, tt) >> list) & 1u)) continue;
                    const unsigned long long kk = v.sim & 0x7FFFFFFFFFFFFFFFull;
                    if (rr > 0 && !better(last_k, last_t, kk, tt)) continue;
                    if (bp < 0 || better(kk, tt, bk, bt)) { bk = kk; bt = tt; bp = q; }
                }
            }
            warp_argbest(bk, bt, bp);
            if (bp < 0) break;
            if (lane == 0) {
                const Rec v = R[bp];
                a.tab_idx[o + rr] = bt;
                a.tab_sim[o + rr] = __longlong_as_double((long long)v.sim);
                a.tab_mutu[o + rr] = rec_mutu(v.pack); a.tab_n[o + rr] = RN[bp];
            }
            last_k = bk; last_t = bt;
            got = rr + 1;
        }
        if (lane == 0) a.tab_len[(size_t)row * 2 + list] = got;
    }
}

// ---- long rows: one CTA per row, streaming with a running threshold + register tournament ----
// Candidate buffer: a candidate belongs to exactly one list (an NB row's BB neighbour is pushed
// twice); 128-bit sortable record:
//   skey = (list 0 ? 1<<63 : 0) | bits(|sim|)        (0 = empty pad)
//   spay = sign(sim)<<63 | item<<16 | position        (position indexes c_mutu / c_n)
template <int THREADS, int CAP_>
struct Scratch {
    static constexpr int CAP = CAP_;
    unsigned long long skey[CAP];
    unsigned long long spay[CAP];
    double t_sim[2][KMAX];
    unsigned long long thr[2];
    int c_mutu[CAP], c_n[CAP];
    int t_j[2][KMAX], t_mutu[2][KMAX], t_n[2][KMAX];
    int t_len[2];
    int fin_len[2][THREADS / 32];
    int ncand;
};

constexpr unsigned long long LIST0_BIT = 1ull << 63;
constexpr unsigned long long ABS_MASK = ~LIST0_BIT;

__device__ __forceinline__ int pay_item(unsigned long long pay) { return int((pay & ABS_MASK) >> 16); }

// Two-stage tournament over the candidate buffer (plus the running tops):
//   stage 1  every warp takes a contiguous slice of the buffer, holds it in registers and extracts
//            its own best K per list with K rounds of a register-local max + a warp arg-best;
//   stage 2  warp 0 (list 0) and warp 1 (list 1) pick the best K among the <= nwarps*K finalists.
template <int THREADS, int CAP>
__device__ void select_lists(Scratch<THREADS, CAP> &S, int K) {
    constexpr int NW = THREADS / 32;
    constexpr int PER_LANE = CAP / THREADS;               // slice = PER_LANE * 32 records per warp
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n0t = S.t_len[0], n1t = S.t_len[1];
    const int nc = S.ncand;
    // running tops re-enter as candidates of their own list
    if (tid < n0t) {
        const int p = nc + tid;
        const double v = S.t_sim[0][tid];
        S.skey[p] = LIST0_BIT | abs_key(v);
        S.spay[p] = (v < 0.0 ? LIST0_BIT : 0ull) | ((unsigned long long)S.t_j[0][tid] << 16) | (unsigned)p;
        S.c_mutu[p] = S.t_mutu[0][tid]; S.c_n[p] = S.t_n[0][tid];
    } else if (tid >= KMAX && tid < KMAX + n1t) {
        const int q = tid - KMAX, p = nc + n0t + q;
        const double v = S.t_sim[1][q];
        S.skey[p] = abs_key(v);
        S.spay[p] = (v < 0.0 ? LIST0_BIT : 0ull) | ((unsigned long long)S.t_j[1][q] << 16) | (unsigned)p;
        S.c_mutu[p] = S.t_mutu[1][q]; S.c_n[p] = S.t_n[1][q];
    }
    __syncthreads();
    const int total = nc + n0t + n1t;
    unsigned long long rk[PER_LANE], rp[PER_LANE];
    const int base = warp * (PER_LANE * 32);
#pragma unroll
    for (int r = 0; r < PER_LANE; ++r) {
        const int p = base + r * 32 + lane;
        rk[r] = (p < total) ? S.skey[p] : 0ull;
        rp[r] = (p < total) ? S.spay[p] : 0ull;
    }
    __syncthreads();                                        // everybody has its slice; reuse skey/spay
    // finalists of warp w, list l live at skey[(l * NW + w) * K + r]   (needs 2*NW*K <= CAP)
    for (int list = 0; list < 2; ++list) {
        const unsigned long long want = (list == 0) ? LIST0_BIT : 0ull;
        int got = 0;
        for (int rr = 0; rr < K; ++rr) {
            unsigned long long bk = 0ull, bpay = 0ull;
            int bt = 0x7FFFFFFF, bp = -1;
#pragma unroll
            for (int r = 0; r < PER_LANE; ++r) {
                const unsigned long long key = rk[r];
                if (key == 0ull || (key & LIST0_BIT) != want) continue;
                const int tt = pay_item(rp[r]);
                if (bp < 0 || better(key, tt, bk, bt)) { bk = key; bt = tt; bp = r * 32 + lane; bpay = rp[r]; }
            }
            unsigned long long k2 = bk; int t2 = bt, p2 = bp;
            warp_argbest(k2, t2, p2);
            if (p2 < 0) break;
            const int owner = p2 & 31, slot = p2 >> 5;
            const unsigned long long wpay = __shfl_sync(0xffffffffu, bpay, owner);
            if (lane == owner) {
#pragma unroll
                for (int r = 0; r < PER_LANE; ++r) if (r == slot) rk[r] = 0ull;   // taken
            }
            if (lane == 0) {
                const int f = (list * NW + warp) * K + rr;
                S.skey[f] = k2; S.spay[f] = wpay;
            }
            got = rr + 1;
        }
        if (lane == 0) S.fin_len[list][warp] = got;
    }
    __syncthreads();
    if (warp < 2) {
        const int list = warp;
        int got = 0;
        unsigned long long last_k = ~0ull; int last_t = -1;
        for (int rr = 0; rr < K; ++rr) {
            unsigned long long bk = 0ull; int bt = 0x7FFFFFFF, bp = -1;
            for (int w = 0; w < NW; ++w) {
                const int fl = S.fin_len[list][w];
                for (int r = lane; r < fl; r += 32) {
                    const int f = (list * NW + w) * K + r;
                    const unsigned long long key = S.skey[f];
                    const int tt = pay_item(S.spay[f]);
                    if (rr > 0 && !better(last_k, last_t, key, tt)) continue;   // already taken
                    if (bp < 0 || better(key, tt, bk, bt)) { bk = key; bt = tt; bp = f; }
                }
            }
            warp_argbest(bk, bt, bp);
            if (bp < 0) break;
            if (lane == 0) {
                const unsigned long long pay = S.spay[bp];
                const double mag = __longlong_as_double((long long)(bk & ABS_MASK));
                const int pos = int(pay & 0xFFFFull);
                S.t_sim[list][rr] = (pay & LIST0_BIT) ? -mag : mag;
                S.t_j[list][rr] = bt; S.t_mutu[list][rr] = S.c_mutu[pos]; S.t_n[list][rr] = S.c_n[pos];
            }
            last_k = bk; last_t = bt;
            got = rr + 1;
        }
        if (lane == 0) {
            S.t_len[list] = got;
            S.thr[list] = (got == K) ? (last_k & ABS_MASK) : 0ull;
        }
    }
    __syncthreads();
    if (tid == 0) S.ncand = 0;
    __syncthreads();
}

constexpr int FIN_THREADS = 256;
constexpr int SEL_UNROLL = 4;                 // records per thread per step
constexpr int SEL_CAP = 12 * FIN_THREADS;     // candidate buffer (a record can enter both lists)

__global__ void __launch_bounds__(FIN_THREADS) select_cta_kernel(xmap_sim_args a, const int32_t *__restrict__ rows,
                                                                 int n_rows) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using ScratchT = Scratch<FIN_THREADS, SEL_CAP>;
    ScratchT &S = *reinterpret_cast<ScratchT *>(smem_raw);
    const int tid = threadIdx.x;
    const int row = rows ? rows[blockIdx.x] : blockIdx.x;
    const int m = a.rec_cnt[row];
    if (m <= XMAP_SELECT_LONG) return;
    const Rec *__restrict__ R = reinterpret_cast<const Rec *>(a.rec) + a.rec_ptr[row];
    const int32_t *__restrict__ RN = a.rec_n + a.rec_ptr[row];
    const bool bb_i = a.bb[row] != 0;
    const int dom_i = a.dom_code[row];
    const int K = a.k;
    if (tid == 0) {
        S.ncand = 0;
        S.t_len[0] = S.t_len[1] = 0; S.thr[0] = S.thr[1] = 0ull;
    }
    __syncthreads();
    for (int base = 0; base < m; base += FIN_THREADS * SEL_UNROLL) {
        if (S.ncand + 2 * FIN_THREADS * SEL_UNROLL + 2 * KMAX > SEL_CAP) select_lists<FIN_THREADS, SEL_CAP>(S, K);
        const unsigned long long f0 = S.thr[0], f1 = S.thr[1];
        const unsigned long long floor_key = (f0 < f1) ? f0 : f1;     // the weakest threshold still open
        Rec v[SEL_UNROLL];
#pragma unroll
        for (int u = 0; u < SEL_UNROLL; ++u) {
            const int e = base + u * FIN_THREADS + tid;
            v[u] = (e < m) ? R[e] : Rec{0ull, 0ull};
        }
#pragma unroll
        for (int u = 0; u < SEL_UNROLL; ++u) {
            if (v[u].sim == 0ull) continue;
            const unsigned long long key = v[u].sim & ABS_MASK;
            if (key < floor_key) continue;
            const int j = rec_item(v[u].pack);
            const unsigned lb = list_bits(a, bb_i, dom_i, j);
#pragma unroll
            for (int lst = 0; lst < 2; ++lst) {
                if (!((lb >> lst) & 1u)) continue;
                const unsigned long long th = lst == 0 ? f0 : f1;
                if (th && key < th) continue;
                const int p = atomicAdd(&S.ncand, 1);
                S.skey[p] = (lst == 0 ? LIST0_BIT : 0ull) | key;
                S.spay[p] = (v[u].sim & LIST0_BIT) | ((unsigned long long)j << 16) | (unsigned)p;
                S.c_mutu[p] = rec_mutu(v[u].pack); S.c_n[p] = RN[base + u * FIN_THREADS + tid];
            }
        }
        __syncthreads();
    }
    select_lists<FIN_THREADS, SEL_CAP>(S, K);
    for (int slot = 0; slot < 2; ++slot) {
        const int len = S.t_len[slot];
        const size_t o = ((size_t)row * 2 + slot) * K;
        if (tid < len) {
            a.tab_idx[o + tid] = S.t_j[slot][tid]; a.tab_sim[o + tid] = S.t_sim[slot][tid];
            a.tab_mutu[o + tid] = S.t_mutu[slot][tid]; a.tab_n[o + tid] = S.t_n[slot][tid];
        }
        if (tid == 0) a.tab_len[(size_t)row * 2 + slot] = len;
    }
}

static int check_args(const xmap_sim_args &a) {
    if (a.k < 1 || a.k > KMAX) return fail_msg("xmap_sim: k out of range [1, XMAP_KMAX]");
    if (a.method != XMAP_METHOD_ADJUST_COSINE && a.method != XMAP_METHOD_COSINE)
        return fail_msg("xmap_sim: bad method");
    if (a.num_atleast < 1) return fail_msg("xmap_sim: num_atleast must be >= 1");
    return 0;
}

}  // namespace xmap

using namespace xmap;

extern "C" int64_t xmap_sim_row_cells(int64_t tri_work, int32_t n_more_popular) {
    const long long h = hash_cells_for(tri_work);
    return (long long)n_more_popular <= h ? (long long)n_more_popular : h;
}

extern "C" int xmap_sim_row_headers(const xmap_sim_args *args_h, const int32_t *rows, int32_t n_rows,
                                    const int32_t *seg_lo, const int32_t *seg_hi, void *hdr_out, void *stream_) {
    if (n_rows <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream_;
    row_headers_kernel<<<(n_rows + 255) / 256, 256, 0, st>>>(*args_h, rows, n_rows, seg_lo, seg_hi,
                                                             reinterpret_cast<RowHdr *>(hdr_out));
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_sim_accumulate(const xmap_sim_args *args_h, const void *hdr_, int32_t n_rows,
                                   int32_t cells_cap, int32_t threads_per_row,
                                   void *gtab, int32_t gtab_ctas, void *stream_) {
    const RowHdr *rows = reinterpret_cast<const RowHdr *>(hdr_);
    if (int rc = check_args(*args_h)) return rc;
    if (n_rows <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream_;
    if (threads_per_row < 32 || threads_per_row > 512 || (threads_per_row & 31))
        return fail_msg("xmap_sim_accumulate: threads_per_row must be a multiple of 32 in [32, 512]");
    if (cells_cap < 1) return fail_msg("xmap_sim_accumulate: cells_cap must be positive");
    if (gtab) {
        if (gtab_ctas < 1) return fail_msg("xmap_sim_accumulate: gtab_ctas must be positive");
        const int grid = n_rows < gtab_ctas ? n_rows : gtab_ctas;
        tri_gmem_kernel<<<grid, threads_per_row < 64 ? 64 : threads_per_row, 0, st>>>(
            *args_h, rows, n_rows, cells_cap, reinterpret_cast<unsigned char *>(gtab));
        XMAP_LAUNCH_CHECK();
        return 0;
    }
    if (cells_cap > XMAP_SIM_MAX_SMEM_CELLS) return fail_msg("xmap_sim_accumulate: cells_cap exceeds shared memory");
    if (threads_per_row == 32) {
        const size_t smem = 4 * row_smem_bytes(cells_cap);
        if (smem > 227 * 1024) return fail_msg("xmap_sim_accumulate: warp-row tables exceed shared memory");
        XMAP_CUDA(cudaFuncSetAttribute(tri_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tri_warp_kernel<<<(n_rows + 3) / 4, 128, smem, st>>>(*args_h, rows, n_rows, cells_cap);
    } else {
        const size_t smem = row_smem_bytes(cells_cap);
        XMAP_CUDA(cudaFuncSetAttribute(tri_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        tri_cta_kernel<<<n_rows, threads_per_row, smem, st>>>(*args_h, rows, n_rows, cells_cap);
    }
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_sim_accumulate_split(const xmap_sim_args *args_h, const void *hdr_, const int32_t *seg_slot,
                                         const int32_t *slot_nseg, int32_t n_segs, int32_t cells_cap, void *gtab,
                                         int32_t *done, void *stream_) {
    if (int rc = check_args(*args_h)) return rc;
    if (n_segs <= 0) return 0;
    if (cells_cap < 1 || cells_cap > XMAP_SIM_MAX_SMEM_CELLS)
        return fail_msg("xmap_sim_accumulate_split: cells_cap out of range");
    cudaStream_t st = (cudaStream_t)stream_;
    const size_t smem = row_smem_bytes(cells_cap);
    XMAP_CUDA(cudaFuncSetAttribute(tri_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tri_split_kernel<<<n_segs, 512, smem, st>>>(*args_h, reinterpret_cast<const RowHdr *>(hdr_), seg_slot, slot_nseg,
                                                cells_cap, reinterpret_cast<uint4 *>(gtab), done);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_sim_select(const xmap_sim_args *args_h, const int32_t *rows, int32_t n_rows,
                               int32_t long_rows, void *stream_) {
    if (int rc = check_args(*args_h)) return rc;
    if (n_rows <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream_;
    if (!long_rows) {
        select_warp_kernel<<<(n_rows + 3) / 4, 128, 0, st>>>(*args_h, rows, n_rows);
    } else {
        const size_t sel_smem = sizeof(Scratch<FIN_THREADS, SEL_CAP>);
        XMAP_CUDA(cudaFuncSetAttribute(select_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
        select_cta_kernel<<<n_rows, FIN_THREADS, sel_smem, st>>>(*args_h, rows, n_rows);
    }
    XMAP_LAUNCH_CHECK();
    return 0;
}
