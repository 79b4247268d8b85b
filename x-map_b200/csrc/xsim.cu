// X-SIM bridge extension: every (left segment, bridge pair, right segment)
// combination is one path of the reference's enumeration (extender.py:124-169);
// its similarity s_p = sum(sim*mutu)/sum(mutu) and certainty c_p = prod(frac)
// (extender.py:83-89) are accumulated per (start, end) into
// xsim = sum(s_p c_p) / sum(c_p) (extender.py:198-201) without ever storing a path.
//
// Design: the accumulator of a start never leaves the SM, and no two warps ever share a cell.
// One WARP owns one unit = (start item, a run of passes) at a time and a private hash table in shared
// memory; a pass covers a range of the hashed end axis pi(y) = y * 0x9E3779B1 (every right-segment list
// is stored sorted by pi, and a per-source pointer table gives the sub-range of a pass without a search),
// chosen so that the distinct ends of the pass fit the table.  Inside a pass the warp walks the
// (leg, partner) pairs of its start 32 at a time: each lane loads one pair descriptor {list, folded (N, D, C)
// of leg + bridge edge} and resolves the list's sub-range of the pass, a shuffle scan numbers the products
// of the batch and they are dealt to the lanes in chunks of 32 whatever the sub-range lengths.  A lane
// loads one 28-byte right segment (the next chunk's loads are issued before the current chunk is
// processed) and evaluates the path.  Lanes that hit the same end: adjacent ones (the lists are ordered
// by pi(end), so a run of equal ends is the rule in a fused list) are summed by a segmented shuffle scan,
// the heads of the runs are grouped (MATCH.ANY) and the group's lowest lane adds the run totals in lane
// (= path) order to the cell: plain shared-memory loads and stores, no atomics on values, no block
// barrier.  The summation order of a (start, end) cell is a function of the path structure and the pass
// plan only, so results are bit-identical from run to run and for any number of GPUs (every rank builds
// the same plan).
//
// A pass whose table overflows is split in two on the device (the tile range halves) and redone; the top-m
// of a unit is kept in shared memory across its passes and a small kernel merges the units of a start.
// Units are fetched from a global counter in descending-work order (results do not depend on which warp
// runs a unit).
//
// Bound: issue rate of the per-path instruction stream and the 28 B right-segment read per path from
// L2/HBM; accumulator traffic is shared memory only.
//
// CTA-cooperative variant (xsim_cta_kernel, for the hot units): one CTA of 8 warps owns one unit and ONE
// shared-memory hash table of 2^cells_lg cells (8x the per-warp table, so a start needs 8x fewer passes:
// longer sub-ranges per (leg, partner) pair, fewer pair look-ups, fewer duplicates per step).  Two CTAs are
// resident per SM, so one runs while the other waits at its barrier.
//
//   prep      256 (leg, partner) pairs at a time: each thread resolves one pair to a descriptor; a block
//             scan numbers the products of the macro-batch and compacts the non-empty descriptors;
//   produce   the products are dealt to the 8 warps in chunks of 32 (chunk c -> warp c mod 8): a lane finds
//             its descriptor, loads one 28-byte right segment (the next chunk's loads are issued first),
//             evaluates the path; lanes of the chunk that hit the same end are summed in lane (= path)
//             order by the lowest one, which leaves (end, num, den) in its payload slot; per
//             (owner, producer) lane masks say which slots belong to which owner warp (3 bits of a hash);
//   consume   after ONE block barrier, warp o walks the slots addressed to it in (producer, lane) order,
//             combines slots of the same end in that order and updates its private region of the table
//             with plain loads and stores (the key is claimed with a CAS): no atomics on values.
//
// The two kernels share the path step, the table probe, the pass schedule, the top-m ranking and the
// publication of a unit (the helpers below); they differ in where descriptors live, who owns a cell and
// how run totals reach it.
#include "common.cuh"

namespace xmap {

constexpr unsigned XGOLD2 = 0x85EBCA6Bu;      // second multiplicative hash of the end: owner warp and home cell
                                              // (the first one, pi(y) = y * 0x9E3779B1, orders the lists: host side)
// warp kernel
constexpr int XT_MAX = 640;                   // threads per CTA (a multiple of 32, chosen at launch)
constexpr int XSTACK_WARP = 16;               // pending halves of split passes (depth <= gb + 1)
constexpr int XSV = 64;                       // candidates of a top-m merge: survivors (<= 32) + running best (<= 32)
// CTA kernel
constexpr int XT = 256;                       // threads per CTA
constexpr int XW = XT / 32;                   // warps = owners
constexpr int XMB = 256;                      // (leg, partner) pairs per macro-batch
constexpr int XOB = 3;                        // log2(XW): owner bits
constexpr int XSTACK_CTA = 24;
constexpr int XSURV = 256;

// ---- shared by both kernels ---------------------------------------------------------------------------

// pending halves of split passes: tile ranges [g0, g1), the top one runs next
template <int DEPTH>
struct SplitStack {
    int g0[DEPTH], g1[DEPTH];
};

// the next pass of a unit: the top split half if one is pending, else the unit's next own pass (its tile
// range [ug0, ug1) cut into unpass equal passes); false once the unit is done
template <int DEPTH>
__device__ __forceinline__ bool take_pass(const SplitStack<DEPTH> &st, int &n, int &next, int ug0, int ug1, int unpass,
                                          int &g0, int &g1) {
    if (n > 0) { --n; g0 = st.g0[n]; g1 = st.g1[n]; return true; }
    if (next >= unpass) return false;
    const long long w = ug1 - ug0;
    g0 = ug0 + (int)(w * next / unpass);
    g1 = ug0 + (int)(w * (next + 1) / unpass);
    ++next;
    return true;
}

// the pass [g0, g1) does not fit its table: push both halves of its tile range, the lower one on top; false
// when it cannot be split (one tile, or the stack is full)
template <int DEPTH>
__device__ __forceinline__ bool split_pass(SplitStack<DEPTH> &st, int &n, int g0, int g1) {
    if (g1 - g0 < 2 || n + 2 > DEPTH) return false;
    const int mid = (g0 + g1) >> 1;
    st.g0[n] = mid; st.g1[n] = g1;
    st.g0[n + 1] = g0; st.g1[n + 1] = mid;
    n += 2;
    return true;
}

struct PairDesc {
    double N, D, C;
    long long base;
    int len;
};

// pair q of the unit: its descriptor {list, folded (N, D, C)} (one coalesced load per thread) and the sub-range of
// the list that falls into the pass (empty for a q past the unit's pairs)
__device__ __forceinline__ PairDesc load_pair(const xmap_xsim_args &a, long long q, bool in_unit, bool whole,
                                              int g0, int g1, int G1) {
    PairDesc d;
    d.N = d.D = d.C = 0.0; d.base = 0; d.len = 0;
    if (in_unit) {
        const int s = __ldg(a.pd_s + q);
        d.N = __ldg(a.pd_n + q); d.D = __ldg(a.pd_d + q); d.C = __ldg(a.pd_c + q);
        const long long rb = __ldg(a.rs_ptr + s);
        if (whole) { d.base = rb; d.len = (int)(__ldg(a.rs_ptr + s + 1) - rb); }
        else {
            const int32_t *tp = a.tile_ptr + (size_t)s * G1;
            const int b0 = __ldg(tp + g0), b1 = __ldg(tp + g1);
            d.base = rb + b0; d.len = b1 - b0;
        }
    }
    return d;
}

// one product of a chunk: the pair's folded (N, D, C) and the right segment's end and (N, D, C)
struct Fetched {
    double N, D, C, rn, rd, rc;
    int y;
    bool valid;
};

// the 28-byte right segment r
__device__ __forceinline__ void load_rseg(const xmap_xsim_args &a, long long r, Fetched &f) {
    f.y = __ldg(a.rs_end + r);
    f.rn = __ldg(a.rs_n + r); f.rd = __ldg(a.rs_d + r); f.rc = __ldg(a.rs_c + r);
}

// The lane's path: num = s_p c_p, den = c_p (extender.py:88-89; zero without a product, whose end y is then
// -1 - lane).  The lists are ordered by pi(end), so equal ends sit in ADJACENT lanes (a fused list holds an end
// once per way of reaching it): a run of equal ends is summed into its head by a segmented suffix scan over the
// lanes (a fixed tree).  Returns whether the lane heads a run; heads with equal ends (a chunk that spans several
// lists) are the caller's to group.
__device__ __forceinline__ bool eval_runs(const Fetched &f, int lane, int &y, double &num, double &den) {
    num = 0.0; den = 0.0;
    if (f.valid) {
        const double Nn = __dadd_rn(f.N, f.rn);
        const double Dd = __dadd_rn(f.D, f.rd);
        den = __dmul_rn(f.C, f.rc);
        const double sp = (Dd != 0.0) ? __ddiv_rn(Nn, Dd) : 0.0;
        num = __dmul_rn(sp, den);
    }
    y = f.valid ? f.y : (-1 - lane);
    const int y_prev = __shfl_up_sync(0xffffffffu, y, 1);
    const bool head = lane == 0 || y != y_prev;
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (heads != 0xffffffffu) {
        const unsigned later = lane == 31 ? 0u : (heads >> (lane + 1));
        const int run_end = later ? lane + __ffs(later) - 1 : 31;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const double vn = __shfl_down_sync(0xffffffffu, num, off);
            const double vd = __shfl_down_sync(0xffffffffu, den, off);
            if (lane + off <= run_end) { num = __dadd_rn(num, vn); den = __dadd_rn(den, vd); }
        }
    }
    return head;
}

// Find-or-insert of key (end + 1) in a table region of 2^lg cells, probing linearly from the home cell.  Only
// one warp touches the region; the CAS settles lanes racing for one empty cell.  Returns the cell within the
// region (-1: the region is full) and whether the key is new.
__device__ __forceinline__ int find_or_insert(int *keys, int lg, int pos, int key, bool &isnew) {
    isnew = false;
    for (int probes = 0; probes < (1 << lg); ++probes) {
        const int kcur = *(volatile int *)(keys + pos);
        if (kcur == key) return pos;
        if (kcur == 0) {
            const int old = atomicCAS(keys + pos, 0, key);
            if (old == 0) { isnew = true; return pos; }
            if (old == key) return pos;
        }
        pos = (pos + 1) & ((1 << lg) - 1);
    }
    return -1;
}

// a top-m list in shared memory: |xsim| key, xsim and end of every entry
struct TopList {
    unsigned long long *key;
    double *x;
    int *end;
};

// candidate q of n takes position `rank` (the number of better candidates) of the new list if rank < len
__device__ __forceinline__ void rank_candidate(const TopList &cand, int n, int q, const TopList &out, int len) {
    const unsigned long long mk = cand.key[q]; const int me = cand.end[q];
    int rank = 0;
    for (int t = 0; t < n; ++t) rank += better(cand.key[t], cand.end[t], mk, me) ? 1 : 0;
    if (rank < len) { out.key[rank] = mk; out.x[rank] = cand.x[q]; out.end[rank] = me; }
}

// Slow path of the top-m selection (top_m > 32, or one value repeated very often): newlen rounds of an arg-best
// over every cell of the table (C cells) and the running best (positions C ..), thread t of a stride nt; each
// round takes the best candidate strictly after the last.  reduce(key, tie, pos) hands the winner to every
// thread, and thread 0 writes it to position r of `out` (positions < r are final).
template <class Reduce>
__device__ __forceinline__ void topm_rounds(const int *keys, const double2 *vals, int C, const TopList &best, int nbest,
                                            const TopList &out, int newlen, int t, int nt, Reduce reduce) {
    unsigned long long last_k = ~0ull; int last_t = -1;
    for (int r = 0; r < newlen; ++r) {
        unsigned long long bk = 0ull; int bt = 0x7FFFFFFF, bp = -1;
        for (int c = t; c < C + nbest; c += nt) {
            unsigned long long ak; int ee;
            if (c < C) { const int kk = keys[c]; if (kk == 0) continue; ak = abs_key(vals[c].x); ee = kk - 1; }
            else { ak = best.key[c - C]; ee = best.end[c - C]; }
            if (r > 0 && !better(last_k, last_t, ak, ee)) continue;
            if (bp < 0 || better(ak, ee, bk, bt)) { bk = ak; bt = ee; bp = c; }
        }
        reduce(bk, bt, bp);
        if (t == 0 && bp >= 0) {
            out.key[r] = bk; out.end[r] = bt;
            out.x[r] = bp < C ? vals[bp].x : best.x[bp - C];
        }
        last_k = bk; last_t = bt;
    }
}

// the unit's distinct ends, paths, top-m list and error (thread t of NT; the loop over the list is unrolled)
template <int NT>
__device__ __forceinline__ void publish_unit(const xmap_xsim_args &a, int u, int t, int count, long long combos,
                                             const TopList &best, int len, int status) {
    if (t == 0) {
        a.unit_count[u] = count;
        a.unit_combos[u] = combos;
        a.unit_top_len[u] = len;
        if (status) atomicExch(a.error_flag, 2);
    }
#pragma unroll
    for (int q = t; q < XMAP_KMAX; q += NT) {
        if (q < len) {
            a.unit_top_end[(size_t)u * a.top_m + q] = best.end[q];
            a.unit_top_xsim[(size_t)u * a.top_m + q] = best.x[q];
        }
    }
}

// ---- warp kernel ----------------------------------------------------------------------------------------

// Per-warp staging (shared memory).  `sv` doubles as the chunk staging of the in-order combine
// (accumulate phase) and as the survivor list of the top-m selection (finalize phase).
struct __align__(16) WarpScratch {
    union {
        struct { double c_num[32], c_den[32]; } acc;
        struct { unsigned long long key[XSV]; double x[XSV]; int end[XSV]; } sv;
    } u;
    unsigned long long best_key[XMAP_KMAX];    // running top-m of the unit over its finished passes
    double best_x[XMAP_KMAX];
    int best_end[XMAP_KMAX];
    SplitStack<XSTACK_WARP> stack;
};

// products [32 c, 32 c + 32) of the batch: the lane's descriptor by a shuffle search over the inclusive
// product counts (empty descriptors are skipped by construction), then the right-segment loads
__device__ __forceinline__ Fetched fetch_chunk(const xmap_xsim_args &a, int c, int total, int incl, int len,
                                               long long base, double dN, double dD, double dC, int lane) {
    Fetched f;
    const int p = (c << 5) + lane;
    int l = 0;                                              // smallest lane with incl > p
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int v = __shfl_sync(0xffffffffu, incl, l + step - 1);
        if (v <= p) l += step;
    }
    const int excl = __shfl_sync(0xffffffffu, incl - len, l);
    const long long b = __shfl_sync(0xffffffffu, base, l);
    f.N = __shfl_sync(0xffffffffu, dN, l);
    f.D = __shfl_sync(0xffffffffu, dD, l);
    f.C = __shfl_sync(0xffffffffu, dC, l);
    f.valid = p < total;
    f.y = 0; f.rn = f.rd = f.rc = 0.0;
    if (f.valid) load_rseg(a, b + (long long)(p - excl), f);
    return f;
}

// One warp = one unit at a time (fetched from a global counter in descending-work order); the warps of a
// CTA are independent: no block barrier anywhere.
template <int MAXT>
__global__ void __launch_bounds__(MAXT, 1) xsim_warp_kernel(xmap_xsim_args a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int nw = blockDim.x >> 5;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int CS = 1 << a.cells_lg;                        // cells of a warp's shared-memory table
    WarpScratch &W = reinterpret_cast<WarpScratch *>(smem_raw)[warp];
    const TopList sv{W.u.sv.key, W.u.sv.x, W.u.sv.end}, best{W.best_key, W.best_x, W.best_end};
    double2 *s_vals = reinterpret_cast<double2 *>(smem_raw + (size_t)nw * sizeof(WarpScratch)) + (size_t)warp * CS;
    int *s_keys = reinterpret_cast<int *>(smem_raw + (size_t)nw * sizeof(WarpScratch) + (size_t)nw * CS * sizeof(double2)) +
                  (size_t)warp * CS;
    // units whose ends do not fit the shared-memory table use this warp's slot of the global workspace
    // (L2-resident while the unit runs): 2^gcells_lg cells, vals first
    unsigned char *gslot = a.gws ? reinterpret_cast<unsigned char *>(a.gws) +
                                       ((size_t)blockIdx.x * nw + warp) * ((size_t)20 << a.gcells_lg) : nullptr;
    const int G = 1 << a.gb, G1 = G + 1;
    const int M = a.top_m;
    const unsigned lt_mask = (1u << lane) - 1u;

    for (;;) {
        int uq = 0;
        if (lane == 0) uq = atomicAdd(a.unit_counter, 1);
        uq = __shfl_sync(0xffffffffu, uq, 0);
        if (uq >= a.n_units) break;
        const int u = a.unit_order ? __ldg(a.unit_order + uq) : uq;
        const long long t_unit = a.unit_cycles ? clock64() : 0ll;
        const long long leg_lo = a.unit_leg_lo[u], leg_hi = a.unit_leg_hi[u];
        const long long q_lo = a.lp_ptr[leg_lo], q_hi = a.lp_ptr[leg_hi];
        const int ug0 = a.unit_g0[u], ug1 = a.unit_g1[u], unpass = a.unit_npass[u];
        long long combos = 0;
        int unit_count = 0, best_len = 0, stack_n = 0, next_pass = 0, status = 0, emitted = 0;
        const int clg = a.unit_clg ? min(a.unit_clg[u], gslot ? a.gcells_lg : a.cells_lg) : a.cells_lg;
        const bool in_smem = clg <= a.cells_lg;
        const int C = 1 << clg;
        double2 *vals = in_smem ? s_vals : reinterpret_cast<double2 *>(gslot);
        int *keys = in_smem ? s_keys : reinterpret_cast<int *>(gslot + ((size_t)16 << a.gcells_lg));

        for (;;) {
            int g0, g1;                                    // warp-uniform
            if (!take_pass(W.stack, stack_n, next_pass, ug0, ug1, unpass, g0, g1)) break;
            const bool whole = g0 == 0 && g1 == G;
            for (int c = lane; c < C; c += 32) keys[c] = 0;
            __syncwarp();

            // =================== accumulate ======================================================
            long long q0 = q_lo, pass_combos = 0;
            bool ovf = false;
            int n_ins = 0;                                 // occupied cells of the table
            PairDesc nxd = load_pair(a, q0 + lane, q0 + lane < q_hi, whole, g0, g1, G1);
            while (q0 < q_hi && !ovf) {
                const int nq = (int)min(32ll, q_hi - q0);
                const PairDesc pd = nxd;
                q0 += nq;
                nxd = load_pair(a, q0 + lane, q0 + lane < q_hi, whole, g0, g1, G1);   // the next 32 pairs resolve while these are walked
                const int len = pd.len;
                const long long base = pd.base;
                const double dN = pd.N, dD = pd.D, dC = pd.C;
                int incl = len;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, off);
                    if (lane >= off) incl += t;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                pass_combos += total;

                const int nchunk = (total + 31) >> 5;
                Fetched nxt = fetch_chunk(a, 0, total, incl, len, base, dN, dD, dC, lane);
                for (int c = 0; c < nchunk; ++c) {
                    const Fetched cur = nxt;
                    nxt = fetch_chunk(a, c + 1, total, incl, len, base, dN, dD, dC, lane);
                    int y;
                    double num, den;
                    const bool head = eval_runs(cur, lane, y, num, den);
                    W.u.acc.c_num[lane] = num; W.u.acc.c_den[lane] = den;
                    const unsigned grp = __match_any_sync(0xffffffffu, head ? y : (-1 - lane));
                    __syncwarp();
                    bool lane_ovf = false, inserted = false;
                    if (cur.valid && head && (__ffs(grp) - 1) == lane) {
                        bool isnew;
                        const int slot = find_or_insert(keys, clg, (int)(((unsigned)y * XGOLD2) >> (32 - clg)), y + 1, isnew);
                        inserted = isnew;
                        if (slot < 0) lane_ovf = true;
                        else {
                            // the runs of this end, one by one in lane (= path) order
                            double an = 0.0, ad = 0.0;
                            if (!isnew) { const double2 v = vals[slot]; an = v.x; ad = v.y; }
                            unsigned rem = grp;
                            while (rem) {
                                const int b = __ffs(rem) - 1;
                                an = __dadd_rn(an, W.u.acc.c_num[b]); ad = __dadd_rn(ad, W.u.acc.c_den[b]);
                                rem &= rem - 1u;
                            }
                            vals[slot] = make_double2(an, ad);
                        }
                    }
                    __syncwarp();                                  // staging reads done before the next chunk's writes
                    n_ins += __popc(__ballot_sync(0xffffffffu, inserted));
                    ovf = __any_sync(0xffffffffu, lane_ovf) || n_ins > C - (C >> 3);   // linear probing degrades past 7/8
                    if (ovf) break;
                }
            }
            if (ovf) {
                // the pass does not fit: redo both halves of it (nothing of it was published)
                if (!split_pass(W.stack, stack_n, g0, g1)) status = 1;
                __syncwarp();
                continue;
            }
            combos += pass_combos;

            // =================== finalize the pass ==============================================
            // xsim of every cell (kept in vals[c].x), count, lane-local best, optional emit
            int mycnt = 0;
            unsigned long long lk = 0ull; int le = 0x7FFFFFFF;
            for (int c0 = 0; c0 < C; c0 += 32) {
                const int c = c0 + lane;
                const int kk = keys[c];
                const bool occ = kk != 0;
                double x = 0.0;
                if (occ) {
                    const double2 v = vals[c];
                    x = __ddiv_rn(v.x, v.y);                   // extender.py:198-201
                    vals[c].x = x;
                    ++mycnt;
                    const unsigned long long ak = abs_key(x);
                    if (mycnt == 1 || better(ak, kk - 1, lk, le)) { lk = ak; le = kk - 1; }
                }
                if (a.emit_ptr) {
                    const unsigned mo = __ballot_sync(0xffffffffu, occ);
                    if (occ) {
                        const long long o = a.emit_ptr[u] + emitted + __popc(mo & lt_mask);
                        a.emit_end[o] = kk - 1; a.emit_xsim[o] = x;
                    }
                    emitted += __popc(mo);
                }
            }
            const unsigned have = __ballot_sync(0xffffffffu, mycnt > 0);
            int cnt_pass = mycnt;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) cnt_pass += __shfl_xor_sync(0xffffffffu, cnt_pass, off);
            unit_count += cnt_pass;
            const int newlen = min(M, cnt_pass + best_len);
            __syncwarp();
            // threshold (tk, te): a candidate worse than it cannot enter the list
            unsigned long long tk = 0ull; int te = 0x7FFFFFFF;
            bool fast = M <= 32;
            if (fast && cnt_pass > XSV / 2 && __popc(have) >= M) {
                // the M-th best of the lane-local maxima bounds the M-th best cell from below
                const int want = M;
                int rank = 0;
                for (int t = 0; t < 32; ++t) {
                    const unsigned long long k2 = __shfl_sync(0xffffffffu, lk, t);
                    const int e2 = __shfl_sync(0xffffffffu, le, t);
                    if (((have >> t) & 1u) && better(k2, e2, lk, le)) ++rank;
                }
                const unsigned sel = __ballot_sync(0xffffffffu, mycnt > 0 && rank == want - 1);
                const int sl = __ffs(sel) - 1;
                tk = __shfl_sync(0xffffffffu, lk, sl); te = __shfl_sync(0xffffffffu, le, sl);
            }
            if (best_len == M) {
                const unsigned long long bk = W.best_key[M - 1]; const int be = W.best_end[M - 1];
                if (better(bk, be, tk, te)) { tk = bk; te = be; }
            }
            // survivors: cells not worse than the threshold
            int nsurv = 0;
            for (int c0 = 0; c0 < C && fast; c0 += 32) {
                const int c = c0 + lane;
                const int kk = keys[c];
                bool take = false;
                unsigned long long ak = 0ull; double x = 0.0;
                if (kk != 0) { x = vals[c].x; ak = abs_key(x); take = !better(tk, te, ak, kk - 1); }
                const unsigned mt = __ballot_sync(0xffffffffu, take);
                if (nsurv + __popc(mt) > XSV / 2) { fast = false; break; }
                if (take) { const int q = nsurv + __popc(mt & lt_mask); W.u.sv.key[q] = ak; W.u.sv.x[q] = x; W.u.sv.end[q] = kk - 1; }
                nsurv += __popc(mt);
            }
            if (fast) {
                // candidates = survivors + the running best; rank by counting, winners rewrite the list
                if (lane < best_len) { W.u.sv.key[nsurv + lane] = W.best_key[lane]; W.u.sv.x[nsurv + lane] = W.best_x[lane]; W.u.sv.end[nsurv + lane] = W.best_end[lane]; }
                __syncwarp();
                const int ncand = nsurv + best_len;                 // <= XSV
                for (int q = lane; q < ncand; q += 32) rank_candidate(sv, ncand, q, best, newlen);
            } else {
                // the new list grows in the candidate arrays
                __syncwarp();
                topm_rounds(keys, vals, C, best, best_len, sv, newlen, lane, 32,
                            [](unsigned long long &bk, int &bt, int &bp) { warp_argbest(bk, bt, bp); });
                __syncwarp();
                for (int q = lane; q < newlen; q += 32) { W.best_key[q] = W.u.sv.key[q]; W.best_x[q] = W.u.sv.x[q]; W.best_end[q] = W.u.sv.end[q]; }
            }
            best_len = newlen;
            __syncwarp();
        }

        if (lane == 0 && a.unit_cycles) a.unit_cycles[u] = clock64() - t_unit;
        publish_unit<32>(a, u, lane, unit_count, combos, best, best_len, status);
        __syncwarp();
    }
}

// ---- CTA kernel -----------------------------------------------------------------------------------------

struct CShared {
    // fixed part (the table follows, sized at launch)
    double d_N[XMB], d_D[XMB], d_C[XMB];      // descriptors of the macro-batch (compacted, non-empty)
    long long d_base[XMB];
    double p_num[2][XW][32], p_den[2][XW][32];   // payload slots, double-buffered; finalize scratch aliases them
    int d_cum[XMB + 4];                        // exclusive product prefix, d_cum[n_desc] = total
    int p_y[2][XW][32];
    unsigned p_mask[2][XW][XW];                // [owner][producer]
    int c_loc[XW][32];                         // consumer: payload slot (producer << 5 | lane) of the 32 items in flight
    unsigned long long s_wsum[XW];
    unsigned long long best_key[XMAP_KMAX];    // running top-m of the unit over its finished passes
    double best_x[XMAP_KMAX];
    int best_end[XMAP_KMAX];
    int best_len;
    SplitStack<XSTACK_CTA> stack;
    int stack_n, next_pass, cur_g0, cur_g1;
    int s_nd, s_total, s_overflow;
    int s_ins[XW];                             // occupied cells per owner region
    int s_cnt, s_nsurv, s_bstar, s_emit;
    int status;
    unsigned long long r_key[XW]; int r_tie[XW], r_pos[XW];   // block arg-best exchange (fallback path)
};

// products [32 c, 32 c + 32) of the macro-batch: descriptor lookup + the right-segment loads
__device__ __forceinline__ Fetched fetch_chunk_cta(const xmap_xsim_args &a, const CShared &S, int c, int nd, int total,
                                                   int lane) {
    Fetched f;
    f.valid = false; f.y = 0; f.N = f.D = f.C = f.rn = f.rd = f.rc = 0.0;
    const int base_p = c << 5;
    if (base_p >= total) return f;
    // descriptor holding product base_p: largest d with d_cum[d] <= base_p (a 32-way and an 8-way step)
    constexpr int GS = XMB / 32;                          // descriptors per coarse group
    const int i1 = lane * GS;
    const unsigned m1 = __ballot_sync(0xffffffffu, i1 < nd && S.d_cum[i1] <= base_p);
    const int coarse = (__popc(m1) - 1) * GS;
    const int i2 = coarse + (lane % GS);
    const unsigned m2 = __ballot_sync(0xffffffffu, lane < GS && i2 < nd && S.d_cum[i2] <= base_p);
    const int d0 = coarse + __popc(m2) - 1;
    // inclusive product ends of the 32 descriptors from d0 on (every descriptor holds >= 1 product)
    const int e = S.d_cum[min(d0 + 1 + lane, nd)];
    const int p = base_p + lane;
    int l = 0;
#pragma unroll
    for (int step = 16; step >= 1; step >>= 1) {
        const int v = __shfl_sync(0xffffffffu, e, l + step - 1);
        if (v <= p) l += step;
    }
    const int eprev = __shfl_sync(0xffffffffu, e, (l + 31) & 31);
    const int d0cum = S.d_cum[d0];
    if (p < total) {
        const int di = d0 + l;
        const int excl = l == 0 ? d0cum : eprev;
        f.valid = true;
        f.N = S.d_N[di]; f.D = S.d_D[di]; f.C = S.d_C[di];
        load_rseg(a, S.d_base[di] + (long long)(p - excl), f);
    }
    return f;
}

__global__ void __launch_bounds__(XT, 2) xsim_cta_kernel(xmap_xsim_args a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CShared &S = *reinterpret_cast<CShared *>(smem_raw);
    const TopList best{S.best_key, S.best_x, S.best_end};
    const int C = 1 << a.cells_lg;
    const int RB = a.cells_lg - XOB;                       // log2 of an owner's region
    double2 *vals = reinterpret_cast<double2 *>(smem_raw + ((sizeof(CShared) + 15) & ~(size_t)15));
    int *keys = reinterpret_cast<int *>(vals + C);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int u = a.unit_order ? a.unit_order[blockIdx.x] : (int)blockIdx.x;
    const long long leg_lo = a.unit_leg_lo[u], leg_hi = a.unit_leg_hi[u];
    const long long q_lo = a.lp_ptr[leg_lo], q_hi = a.lp_ptr[leg_hi];
    const int G = 1 << a.gb, G1 = G + 1;
    const int ug0 = a.unit_g0[u], ug1 = a.unit_g1[u], unpass = a.unit_npass[u];
    const int M = a.top_m;
    long long combos = 0;                                  // identical in every thread
    int unit_count = 0;
    unsigned ss = 0;                                       // superstep counter (payload buffer parity)
    if (tid == 0) {
        S.best_len = 0; S.stack_n = 0; S.next_pass = 0; S.status = 0; S.s_emit = 0;
    }
    __syncthreads();

    for (;;) {
        if (tid == 0) {
            if (!take_pass(S.stack, S.stack_n, S.next_pass, ug0, ug1, unpass, S.cur_g0, S.cur_g1)) S.cur_g0 = -1;
            S.s_overflow = 0; S.s_cnt = 0; S.s_nsurv = 0;
        }
        if (tid < XW) S.s_ins[tid] = 0;
        for (int c = tid; c < C; c += XT) keys[c] = 0;
        __syncthreads();
        const int g0 = S.cur_g0, g1 = S.cur_g1;
        if (g0 < 0) break;
        const bool whole = g0 == 0 && g1 == G;

        // =================== accumulate ======================================================
        long long q0 = q_lo;
        long long pass_combos = 0;
        while (q0 < q_hi) {
            const int nq = (int)min((long long)XMB, q_hi - q0);
            __syncthreads();
            if (S.s_overflow) break;                       // uniform: nobody writes the flag before the next barrier
            const PairDesc pd = load_pair(a, q0 + tid, tid < nq, whole, g0, g1, G1);
            // block scan of (non-empty flag, len)
            const unsigned long long mine = (pd.len > 0 ? (1ull << 40) : 0ull) | (unsigned long long)pd.len;
            unsigned long long incl = mine;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off) incl += t;
            }
            if (lane == 31) S.s_wsum[warp] = incl;
            __syncthreads();
            unsigned long long ws = lane < XW ? S.s_wsum[lane] : 0ull, wi = ws;
#pragma unroll
            for (int off = 1; off < XW; off <<= 1) {
                const unsigned long long t = __shfl_up_sync(0xffffffffu, wi, off);
                if (lane >= off) wi += t;
            }
            const unsigned long long tot = __shfl_sync(0xffffffffu, wi, XW - 1);
            const unsigned long long woff = __shfl_sync(0xffffffffu, wi - ws, warp);
            const unsigned long long excl = woff + incl - mine;
            if (pd.len > 0) {
                const int c = (int)(excl >> 40);
                S.d_cum[c] = (int)(excl & ((1ull << 40) - 1ull));
                S.d_base[c] = pd.base; S.d_N[c] = pd.N; S.d_D[c] = pd.D; S.d_C[c] = pd.C;
            }
            const int nd = (int)(tot >> 40), total = (int)(tot & ((1ull << 40) - 1ull));
            if (tid == 0) S.d_cum[nd] = total;
            __syncthreads();
            q0 += nq;
            pass_combos += total;

            // ---- supersteps: 16 chunks of 32 products, one per warp -------------------------------
            const int nchunk = (total + 31) >> 5;
            Fetched nxt = fetch_chunk_cta(a, S, warp, nd, total, lane);
            for (int k = 0; k * XW < nchunk; ++k) {
                const Fetched cur = nxt;
                nxt = fetch_chunk_cta(a, S, (k + 1) * XW + warp, nd, total, lane);
                const int buf = ss & 1u; ++ss;
                // produce: evaluate, then sum the lanes of this chunk that hit the same end (lane = path order)
                int y;
                double num, den;
                const bool head = eval_runs(cur, lane, y, num, den);
                if (cur.valid) {
                    S.p_num[buf][warp][lane] = num;
                    S.p_den[buf][warp][lane] = den;
                    S.p_y[buf][warp][lane] = cur.y;
                }
                if (lane < XW) S.p_mask[buf][lane][warp] = 0u;
                const unsigned gy = __match_any_sync(0xffffffffu, head ? y : (-1 - lane));
                __syncwarp();
                const bool lead = cur.valid && head && (__ffs(gy) - 1) == lane;
                if (lead && (gy & (gy - 1u))) {
                    double an = num, ad = den;
                    unsigned rem = gy & ~(1u << lane);
                    while (rem) {
                        const int b = __ffs(rem) - 1;
                        an = __dadd_rn(an, S.p_num[buf][warp][b]); ad = __dadd_rn(ad, S.p_den[buf][warp][b]);
                        rem &= rem - 1u;
                    }
                    S.p_num[buf][warp][lane] = an; S.p_den[buf][warp][lane] = ad;
                }
                const int owner = lead ? (int)(((unsigned)y * XGOLD2) >> (32 - XOB)) : XW;
                const unsigned grp = __match_any_sync(0xffffffffu, owner);
                if (lead && (__ffs(grp) - 1) == lane) S.p_mask[buf][owner][warp] = grp;
                __syncthreads();
                // consume: the slots addressed to owner `warp`, in (producer, lane) order
                const unsigned pm = lane < XW ? S.p_mask[buf][warp][lane] : 0u;
                const int cntl = __popc(pm);
                int incl_i = cntl;
#pragma unroll
                for (int off = 1; off < XW; off <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl_i, off);
                    if (lane >= off) incl_i += t;
                }
                const int tot_o = __shfl_sync(0xffffffffu, incl_i, XW - 1);
                const int region = warp << RB;
                for (int i0 = 0; i0 < tot_o; i0 += 32) {
                    const int i = i0 + lane;
                    const bool valid = i < tot_o;
                    int pr = 0;                            // smallest producer with incl > i
#pragma unroll
                    for (int step = XW / 2; step >= 1; step >>= 1) {
                        const int v = __shfl_sync(0xffffffffu, incl_i, pr + step - 1);
                        if (v <= i) pr += step;
                    }
                    pr = min(pr, XW - 1);
                    const int before = __shfl_sync(0xffffffffu, incl_i - cntl, pr);
                    const unsigned mk = __shfl_sync(0xffffffffu, pm, pr);
                    int yy = -1 - lane, loc = 0;
                    if (valid) {
                        loc = (pr << 5) | __fns(mk, 0, i - before + 1);
                        yy = (&S.p_y[buf][0][0])[loc];
                    }
                    S.c_loc[warp][lane] = loc;
                    const unsigned g2 = __match_any_sync(0xffffffffu, yy);
                    __syncwarp();
                    if (valid && (__ffs(g2) - 1) == lane) {
                        // the owner's region, then the slots of this end one by one in (producer, lane) order
                        bool isnew;
                        const int home = (int)((((unsigned)yy * XGOLD2) << XOB) >> (32 - RB));
                        const int slot = find_or_insert(keys + region, RB, home, yy + 1, isnew);
                        if (slot < 0) *(volatile int *)&S.s_overflow = 1;
                        else {
                            double2 *cell = vals + region + slot;
                            double an = 0.0, ad = 0.0;
                            if (!isnew) { const double2 v = *cell; an = v.x; ad = v.y; }
                            unsigned rem = g2;
                            while (rem) {
                                const int l2 = S.c_loc[warp][__ffs(rem) - 1];
                                an = __dadd_rn(an, (&S.p_num[buf][0][0])[l2]); ad = __dadd_rn(ad, (&S.p_den[buf][0][0])[l2]);
                                rem &= rem - 1u;
                            }
                            *cell = make_double2(an, ad);
                            if (isnew) atomicAdd(&S.s_ins[warp], 1);
                        }
                    }
                    __syncwarp();
                }
                if (lane == 0 && S.s_ins[warp] > (1 << RB) - (1 << (RB - 3))) *(volatile int *)&S.s_overflow = 1;   // region past 7/8
            }
        }
        __syncthreads();
        if (S.s_overflow) {
            // the pass does not fit: redo both halves of it (nothing of it was published)
            if (tid == 0 && !split_pass(S.stack, S.stack_n, g0, g1)) S.status = 1;
            __syncthreads();
            continue;
        }
        combos += pass_combos;

        // =================== finalize the pass ==============================================
        unsigned *hist = reinterpret_cast<unsigned *>(&S.p_num[0][0][0]);                       // 1 KB
        unsigned long long *sv_key = reinterpret_cast<unsigned long long *>(&S.p_den[0][0][0]); // 4 KB
        double *sv_x = reinterpret_cast<double *>(&S.p_den[1][0][0]);                           // 4 KB
        int *sv_end = reinterpret_cast<int *>(&S.p_num[1][0][0]);                               // 2 KB
        const TopList sv{sv_key, sv_x, sv_end};
        for (int bq = tid; bq < SIM_BINS; bq += XT) hist[bq] = 0u;
        __syncthreads();
        int mycnt = 0;
        for (int c0 = warp * 32; c0 < C; c0 += XT) {
            const int c = c0 + lane;
            const int kk = keys[c];
            const bool occ = kk != 0;
            double x = 0.0;
            if (occ) {
                const double2 v = vals[c];
                x = __ddiv_rn(v.x, v.y);                   // extender.py:198-201
                vals[c].x = x;
                atomicAdd(&hist[sim_bin(abs_key(x))], 1u);
                ++mycnt;
            }
            if (a.emit_ptr) {
                const unsigned mo = __ballot_sync(0xffffffffu, occ);
                int base = 0;
                if (lane == 0 && mo) base = atomicAdd(&S.s_emit, __popc(mo));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (occ) {
                    const long long o = a.emit_ptr[u] + base + __popc(mo & ((1u << lane) - 1u));
                    a.emit_end[o] = kk - 1; a.emit_xsim[o] = x;
                }
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) mycnt += __shfl_xor_sync(0xffffffffu, mycnt, off);
        if (lane == 0 && mycnt) atomicAdd(&S.s_cnt, mycnt);
        __syncthreads();
        const int cnt_pass = S.s_cnt;
        unit_count += cnt_pass;
        const int want = min(M, cnt_pass);
        if (warp == 0) {
            // largest bin b* such that #(bin >= b*) >= want
            int bstar = 0, run = 0;
            bool found = false;
            for (int hb = SIM_BINS - 32; hb >= 0 && !found && want > 0; hb -= 32) {
                unsigned suf = hist[hb + lane];
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const unsigned t = __shfl_down_sync(0xffffffffu, suf, off);
                    if (lane + off < 32) suf += t;
                }
                const unsigned hit = __ballot_sync(0xffffffffu, run + (int)suf >= want);
                if (hit) { bstar = hb + (31 - __clz(hit)); found = true; }
                else run += (int)__shfl_sync(0xffffffffu, suf, 0);
            }
            if (lane == 0) S.s_bstar = bstar;
        }
        __syncthreads();
        const int bstar = S.s_bstar;
        // survivors: cells at or above the threshold bin, plus the running best of the earlier passes
        for (int c = tid; c < C && want > 0; c += XT) {
            const int kk = keys[c];
            if (kk == 0) continue;
            const double x = vals[c].x;
            const unsigned long long ak = abs_key(x);
            if (sim_bin(ak) < bstar) continue;
            const int pos = atomicAdd(&S.s_nsurv, 1);
            if (pos < XSURV) { sv_key[pos] = ak; sv_x[pos] = x; sv_end[pos] = kk - 1; }
        }
        const int nbest = S.best_len;
        __syncthreads();
        int nsurv = S.s_nsurv;
        const int newlen = min(M, cnt_pass + nbest);
        if (nsurv + nbest <= XSURV) {
            if (tid < nbest) { sv_key[nsurv + tid] = S.best_key[tid]; sv_x[nsurv + tid] = S.best_x[tid]; sv_end[nsurv + tid] = S.best_end[tid]; }
            __syncthreads();
            nsurv += nbest;
            if (tid < nsurv) rank_candidate(sv, nsurv, tid, best, newlen);
            if (tid == 0) S.best_len = newlen;
        } else {
            // one bin holds too many equal values: the new list grows in sv_*, the winner of a round goes through
            // a cross-warp exchange
            __syncthreads();
            topm_rounds(keys, vals, C, best, nbest, sv, newlen, tid, XT, [&](unsigned long long &bk, int &bt, int &bp) {
                warp_argbest(bk, bt, bp);
                if (lane == 0) { S.r_key[warp] = bk; S.r_tie[warp] = bt; S.r_pos[warp] = bp; }
                __syncthreads();
                bk = lane < XW ? S.r_key[lane] : 0ull; bt = lane < XW ? S.r_tie[lane] : 0x7FFFFFFF; bp = lane < XW ? S.r_pos[lane] : -1;
                warp_argbest(bk, bt, bp);
                __syncthreads();                               // the exchange is read before the next round writes it
            });
            __syncthreads();
            if (tid < newlen) { S.best_key[tid] = sv_key[tid]; S.best_x[tid] = sv_x[tid]; S.best_end[tid] = sv_end[tid]; }
            if (tid == 0) S.best_len = newlen;
        }
        __syncthreads();
    }

    publish_unit<XT>(a, u, tid, unit_count, combos, best, S.best_len, S.status);
}

// ---- merge ----------------------------------------------------------------------------------------------

// One warp per start: distinct ends and paths are the sums over its units, its top-m the best m of the units' lists
// (the units of a start cover disjoint ends).
__global__ void __launch_bounds__(256) xsim_merge_kernel(xmap_xsim_args a) {
    const int x = (blockIdx.x * 256 + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (x >= a.n_starts) return;
    const int u0 = a.start_unit_ptr[x], u1 = a.start_unit_ptr[x + 1];
    const int M = a.top_m;
    int cnt = 0; long long comb = 0;
    for (int u = u0 + lane; u < u1; u += 32) { cnt += a.unit_count[u]; comb += a.unit_combos[u]; }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
        comb += __shfl_xor_sync(0xffffffffu, comb, off);
    }
    if (lane == 0) { a.out_count[x] = cnt; a.out_combos[x] = comb; }
    unsigned long long last_k = ~0ull;
    int last_t = -1, got = 0;
    const int ncand = (u1 - u0) * M;
    for (int r = 0; r < M; ++r) {
        unsigned long long bk = 0ull; int bt = 0x7FFFFFFF, bp = -1;
        for (int q = lane; q < ncand; q += 32) {
            const int u = u0 + q / M, p = q % M;
            if (p >= a.unit_top_len[u]) continue;
            const size_t o = (size_t)u * M + p;
            const unsigned long long ak = abs_key(a.unit_top_xsim[o]);
            const int ee = a.unit_top_end[o];
            if (r > 0 && !better(last_k, last_t, ak, ee)) continue;
            if (bp < 0 || better(ak, ee, bk, bt)) { bk = ak; bt = ee; bp = (int)(o - (size_t)u0 * M); }
        }
        warp_argbest(bk, bt, bp);
        if (bp < 0) break;
        if (lane == 0) {
            a.top_end[(size_t)x * M + r] = bt;
            a.top_xsim[(size_t)x * M + r] = a.unit_top_xsim[(size_t)u0 * M + bp];
        }
        last_k = bk; last_t = bt;
        got = r + 1;
    }
    if (lane == 0) a.top_len[x] = got;
}

// the arguments both unit kernels read; the CTA kernel needs cells_lg >= 9 (8 owner regions of >= 64 cells)
static int check_unit_args(const xmap_xsim_args &a, const char *fn, int min_cells_lg) {
    const char *bad = nullptr;
    if (a.top_m < 1 || a.top_m > XMAP_KMAX) bad = "top_m";
    else if (a.cells_lg < min_cells_lg || a.cells_lg > XMAP_XSIM_MAX_CELLS_LG) bad = "cells_lg";
    else if (a.gb < 0 || a.gb > 16) bad = "gb";
    if (!bad) return 0;
    snprintf(g_err, sizeof(g_err), "%s: %s out of range", fn, bad);
    return 2;
}

}  // namespace xmap

using namespace xmap;

extern "C" int64_t xmap_xsim_smem_bytes(int32_t cells_lg, int32_t warps) {
    return (int64_t)warps * ((int64_t)sizeof(WarpScratch) + ((int64_t)20 << cells_lg));
}

extern "C" int64_t xmap_xsim_cta_smem_bytes(int32_t cells_lg) {
    return (int64_t)((sizeof(CShared) + 15) & ~(size_t)15) + ((int64_t)20 << cells_lg);
}

extern "C" int xmap_xsim_extend(const xmap_xsim_args *args_h, void *stream_) {
    const xmap_xsim_args &a = *args_h;
    if (a.n_starts <= 0 || a.n_units <= 0) return 0;
    if (int rc = check_unit_args(a, "xmap_xsim_extend", 6)) return rc;
    if (a.gws && (a.gcells_lg < a.cells_lg || a.gcells_lg > 24)) return fail_msg("xmap_xsim_extend: gcells_lg out of range");
    if (a.warps < 1 || a.warps * 32 > XT_MAX) return fail_msg("xmap_xsim_extend: warps per CTA out of range");
    if (!a.unit_counter) return fail_msg("xmap_xsim_extend: unit_counter is required");
    cudaStream_t st = (cudaStream_t)stream_;
    const size_t smem = (size_t)xmap_xsim_smem_bytes(a.cells_lg, a.warps);
    if (smem > 227 * 1024) return fail_msg("xmap_xsim_extend: warps x table exceed shared memory");
    // two register budgets: up to 16 warps per CTA get 128 registers per thread, up to 20 get 96
    auto kern = a.warps * 32 <= 512 ? xsim_warp_kernel<512> : xsim_warp_kernel<XT_MAX>;
    XMAP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    XMAP_CUDA(cudaMemsetAsync(a.unit_counter, 0, sizeof(int32_t), st));
    int dev = 0, sms = 148;
    XMAP_CUDA(cudaGetDevice(&dev));
    XMAP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const long long ctas = min((long long)sms, ((long long)a.n_units + a.warps - 1) / a.warps);
    kern<<<(unsigned)ctas, a.warps * 32, smem, st>>>(a);
    XMAP_LAUNCH_CHECK();
    return 0;
}

// one CTA per unit: blockIdx b runs unit_order[b]; the unit results are merged by xmap_xsim_merge
extern "C" int xmap_xsim_extend_cta(const xmap_xsim_args *args_h, void *stream_) {
    const xmap_xsim_args &a = *args_h;
    if (a.n_starts <= 0 || a.n_units <= 0) return 0;
    if (int rc = check_unit_args(a, "xmap_xsim_extend_cta", 9)) return rc;
    const size_t smem = (size_t)xmap_xsim_cta_smem_bytes(a.cells_lg);
    if (smem > 227 * 1024) return fail_msg("xmap_xsim_extend_cta: table exceeds shared memory");
    XMAP_CUDA(cudaFuncSetAttribute(xsim_cta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    xsim_cta_kernel<<<(unsigned)a.n_units, XT, smem, (cudaStream_t)stream_>>>(a);
    XMAP_LAUNCH_CHECK();
    return 0;
}

extern "C" int xmap_xsim_merge(const xmap_xsim_args *args_h, void *stream_) {
    const xmap_xsim_args &a = *args_h;
    if (a.n_starts <= 0) return 0;
    if (a.top_m < 1 || a.top_m > XMAP_KMAX) return fail_msg("xmap_xsim_merge: top_m out of range");
    xsim_merge_kernel<<<(unsigned)((a.n_starts + 7) / 8), 256, 0, (cudaStream_t)stream_>>>(a);
    XMAP_LAUNCH_CHECK();
    return 0;
}
