/*
 * xmap_b200 -- C ABI of the B200 (sm_100a) implementation of X-MAP's AlterEgo
 * construction hot path: item-item co-rating similarity, per-item top-k
 * neighbour selection, X-SIM bridge extension, AlterEgo generation.
 *
 * The reference (LPD-EPFL-ML/X-MAP) is pure Python on PySpark RDDs and has no
 * FFI; its boundary for this path is five pipeline functions
 * (code/xmap/utils/assist.py:9-150).  The Python facade in x-map_b200/ keeps
 * those names and signatures and calls the entry points below through ctypes,
 * one call per stage.  Each entry point cites the reference code it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _h;
 *   - buffers are caller-owned (the facade allocates them with torch);
 *   - `stream` is a cudaStream_t passed as void*; calls are stream-ordered and
 *     return without synchronising unless stated;
 *   - return value 0 = ok, otherwise an error whose text xmap_last_error()
 *     returns (thread-local);
 *   - items and users are dense int32 indices; item index < 2^24 (the 8-byte rating entries carry 24-bit items).
 */
#ifndef XMAP_B200_H
#define XMAP_B200_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XMAP_B200_ABI_VERSION 10
#define XMAP_KMAX 64                 /* largest supported top-k (extend_among_topk) */
#define XMAP_METHOD_ADJUST_COSINE 0  /* baselinerSim.py:144-174 */
#define XMAP_METHOD_COSINE 1         /* baselinerSim.py:115-142 */

int xmap_abi_version(void);
const char *xmap_last_error(void);

/* ---------------------------------------------------------------------------
 * (1) Ratings layout + per-user / per-item statistics.
 * Replaces: the (uid, [(iid, rating, time)]) record grouping the RDDs carry,
 * BaselinerSim.get_universal_user_info (baselinerSim.py:17-38) and
 * get_universal_item_info (baselinerSim.py:40-82), and the two
 * collectAsMap+broadcast round trips at assist.py:68-73.
 *
 * In : nnz deduplicated (user, item, rating) triples in any order.
 * Out: CSR by user (entries ascending by item) and CSC by item (entries
 *      ascending by user).  Entry formats (8 bytes each):
 *        csr_ent[k] = { item | ge_avg<<29 , float bits of rating }
 *        csc_ent[k] = { user | ge_avg<<31 , float bits of rating }
 *      ge_avg = (rating >= item average),
 *      the comparison retrieve_path_info makes (baselinerSim.py:106-111).
 *      csr_src[k] = index of the input triple stored at CSR position k.
 *      user_mu[u] = mean rating of u (baselinerSim.py:30).
 *      item_stats[4*i..] = (average, norm2, adjusted norm2, count) exactly the
 *      tuple of baselinerSim.py:56-63.
 * ------------------------------------------------------------------------- */
size_t xmap_layout_workspace_bytes(int64_t nnz, int32_t n_users, int32_t n_items);

int xmap_build_layout(const int32_t *user, const int32_t *item, const float *rating,
                      int64_t nnz, int32_t n_users, int32_t n_items,
                      int32_t *csr_ptr, uint64_t *csr_ent, int32_t *csr_src,
                      int32_t *csc_ptr, uint64_t *csc_ent,
                      double *user_mu, double *item_stats,
                      void *workspace, size_t workspace_bytes, void *stream);

/* Per output row i of R^T R: w[i] = sum over raters u of i of degree(u), the
 * number of co-rating products the full row would cost (SURVEY.md 8: W + nnz in
 * total).  Bounds the length of a row's neighbour-record list.  Synchronises the
 * stream once (it reads nnz = csc_ptr[n_items]). */
int xmap_row_work(const int32_t *csr_ptr, const int32_t *csc_ptr, const uint64_t *csc_ent,
                  int32_t n_items, int64_t *row_work, void *stream);

/* Triangular layout of the similarity stage.  Items are ranked by ascending
 * popularity, ord[i] = rank of (count(i), i) (computed by the caller: one sort of
 * n_items keys).  Every unordered pair {i, j} is evaluated ONCE, by the row of
 * the less popular item, so row i only needs, for each of its raters u, the part
 * of u's ratings that lies on more popular items.  With the user's ratings
 * sorted by ord that part is a suffix:
 *   tcsr_ent[k]  = { ord(item) | (x & 31)<<24 | ge_avg<<29 | (x >> 5)<<30 , float bits of rating }
 *                  same extents as csr_ptr, entries ascending by ord; x = x(item) below;
 *   csc_aux[e]   = 16 bytes { uint32 pos, uint32 len, double mu }: CSC entry e = (i, u) sits at
 *                  tcsr position pos, the len entries after it are u's ratings of items more
 *                  popular than i, and mu = user_mu[u] (0 for the cosine method);
 *   tri_work[i]  = sum of len over the raters of i = products row i evaluates
 *                  (sum over i = W / 2);
 *   ostat[o]     = 16 bytes per ord o: { double den; uint32 item; uint32 prefix<<8 | x }
 *                  den = norm2 (cosine) or adjusted norm2 (adjust_cosine) of the item,
 *                  baselinerSim.py:131-132,164-165;
 *                  x = clamp(E - e_base, 0, 127) with 2^(E-1) <= den < 2^E, 0 when den == 0:
 *                  the item's exponent, which scales the fixed-point inner products of its pairs.
 *                  e_base = max E - 127 over the items with den > 0 keeps every x in the field.
 * workspace >= xmap_tri_workspace_bytes(nnz). */
size_t xmap_tri_workspace_bytes(int64_t nnz);
int xmap_build_tri_layout(const int32_t *csr_ptr, const uint64_t *csr_ent,
                          const int32_t *csc_ptr, const uint64_t *csc_ent,
                          const double *user_mu, const double *item_stats, const int32_t *prefix_code,
                          const int32_t *ord, int32_t n_users, int32_t n_items, int64_t nnz, int32_t method,
                          int32_t e_base, uint64_t *tcsr_ent, void *csc_aux, void *ostat, int64_t *tri_work,
                          void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------
 * (2) Similarity (triangular sparse R^T R) + fused epilogue, then per-row
 * top-k selection.
 * Replaces: produce_pairwise_items + reduceByKey + calculate_*_sim +
 * retrieve_path_info + filter + detect_domain (baselinerSim.py:84-216),
 * get_item_sim (:218-233), the BB-item SQL (assist.py:82-87) and
 * ExtendSim.find_knn_items (extender.py:16-44).
 *
 * xmap_sim_accumulate: for every requested row i and every more popular item j
 * co-rated with i, accumulates over the common raters n_ij, the mutuality count
 * and the inner product (64-bit fixed point, order-independent), computes
 * sim / mutu, applies the reference's filter (sim != 0 and mutu != 0) and
 * appends one neighbour record to the list of row i AND to the list of
 * row j (sim(i,j) == sim(j,i) bitwise, so the pair is never evaluated twice):
 *   rec[rec_ptr[r] + p]   = { bits of sim (f64) , other_item | mutu<<32 }   (16 bytes)
 *   rec_n[rec_ptr[r] + p] = n  (co-rating count; a parallel int32 array that only the winners of the
 *                               selection read, so item index, n and mutu are full 32-bit values)
 *   p = atomic cursor rec_cnt[r]; order within a list is unspecified.
 * The lists are the materialised return value of baseliner_calculate_sim_pipeline
 * (assist.py:66-77).  bb[r] is set to 1 for both ends of a kept cross-domain pair
 * (label by 2-character prefix, baselinerSim.py:191; the BB set of assist.py:84-86).
 * row_npairs[i] += co-rated columns row i evaluated (pre-filter).
 * rec_cnt, bb, row_npairs must be zero on entry of the first call of a stage.
 * List extents: rec_ptr may come from the upper bound min(n_items - 1, row_work - count) per row, or,
 * when that does not fit in memory, from a sizing pass (count_only = 1) that leaves the exact list
 * lengths in rec_cnt (the caller scans them into rec_ptr, clears the counters and runs the real pass).
 *
 * A row's accumulator lives in shared memory: a direct-indexed table when the
 * row has few more-popular columns (the popular rows), otherwise an open-
 * addressing hash of ceil(4/3 * tri_work) cells; 32-bit shared-memory atomics.
 *   threads_per_row = 32  : one warp per row, 4 rows per CTA (no CTA barrier)
 *   threads_per_row > 32  : one CTA of that many threads per row
 *   cells_cap             : table capacity (16-byte cells) of every row in `rows`
 *   gtab != NULL          : tables in global memory instead (rows too large for shared
 *                           memory); gtab holds gtab_ctas * cells_cap * 20 bytes.
 * ------------------------------------------------------------------------- */
typedef struct xmap_sim_args {
    /* layout */
    const int32_t *csc_ptr; const uint64_t *csc_ent; const void *csc_aux;
    const uint64_t *tcsr_ent;
    const void *ostat; const int32_t *ord; const int64_t *tri_work;
    const int32_t *ord_item;       /* [n_items] inverse of ord: the item ranked o-th by popularity */
    /* per-item codes (host-computed from the id strings) */
    const uint8_t *dom_code;       /* iid[-2:] -- extender.py:29     */
    const uint8_t *contains;       /* bit d: label d is a substring of iid -- extender.py:32,34 */
    int32_t n_items; int32_t method; int32_t num_atleast; int32_t k;
    int32_t r2_bits;               /* 2 * e_base of xmap_build_tri_layout: the inner product of items i, j is
                                      summed in units of 2^-(62 - r2_bits - x_i - x_j) */
    int32_t count_only;            /* 1: sizing pass -- bump the list cursors, write no record (rec_ptr unused) */
    /* neighbour-record lists */
    const int64_t *rec_ptr;        /* [n_items + 1] list extents (capacity) */
    int32_t *rec_cnt;              /* [n_items] cursors = list lengths */
    void *rec;                     /* 16-byte records {f64 sim, u32 other item | u32 mutu << 32} */
    int32_t *rec_n;                /* co-rating count n of every record (same extents as rec) */
    uint8_t *bb;                   /* [n_items] bridge-item flags */
    int32_t *row_npairs;           /* [n_items] */
    /* selection output: tables [n_items][2][k] */
    int32_t *tab_idx; double *tab_sim; int32_t *tab_mutu; int32_t *tab_n; int32_t *tab_len;
    int32_t *error_flag;           /* device int: 1 table overflow, 2 list capacity, 3 count range */
} xmap_sim_args;

/* Row headers: everything a row's thread group needs before it can start (item, ord, rater range, work,
 * norm, prefix / class, list extent) gathered into one 48-byte record per launch slot, so a group begins
 * with one load instead of a chain of dependent gathers.  Built once per plan (and again when rec_ptr
 * changes).  seg_lo / seg_hi (both NULL or both given) replace the rater range for split rows. */
#define XMAP_SIM_ROW_HDR_BYTES 48
int xmap_sim_row_headers(const xmap_sim_args *args_h, const int32_t *rows, int32_t n_rows,
                         const int32_t *seg_lo, const int32_t *seg_hi, void *hdr_out, void *stream);

#define XMAP_SIM_MAX_SMEM_CELLS 12288     /* 12288 x (16-byte cell + 2-byte slot index) = 216 KB */
/* cells a row needs: min(#more popular items, ceil(4/3 * tri_work)), at least 32 */
int64_t xmap_sim_row_cells(int64_t tri_work, int32_t n_more_popular);
int xmap_sim_accumulate(const xmap_sim_args *args_h, const void *row_hdr, int32_t n_rows,
                        int32_t cells_cap, int32_t threads_per_row,
                        void *gtab, int32_t gtab_ctas, void *stream);

/* Rows with very many raters (the most popular items: long rater lists, few products per rater)
 * are bound by the walk over their raters, so their rater list is cut into segments, one CTA each.
 * Segment g (header seg_hdr[g], built with its rater range [seg_lo[g], seg_hi[g])) belongs to the seg_slot[g]-th
 * split row; slot_nseg[slot] = number of segments of that row.  Only direct-indexed rows (at most
 * cells_cap more popular items) may be split.  gtab: [n_slots][cells_cap] 16-byte cells and
 * done: [n_slots] ints, both zero on entry and zero again on exit.  Results are bit-identical to
 * the unsplit row (the partial tables are combined with exact integer adds). */
int xmap_sim_accumulate_split(const xmap_sim_args *args_h, const void *seg_hdr, const int32_t *seg_slot,
                              const int32_t *slot_nseg, int32_t n_segs, int32_t cells_cap, void *gtab,
                              int32_t *done, void *stream);

/* Per-row top-k selection over the neighbour-record lists (extender.py:16-44), after
 * every rank's records are in place and bb holds the flags of ALL items:
 *   BB row : table slot 0 = BB_BB (top-k other-domain), slot 1 = BB_NB (top-k same-domain)
 *   NB row : table slot 0 = NB_BB (top-k neighbours that are BB), slot 1 = NB_NN (top-k of all)
 * Ordering = |sim| descending, ties to the smaller item index (SURVEY.md App. A.6 rule 3).
 * long_rows = 0: one warp per row, rows with more than XMAP_SELECT_LONG records are skipped;
 * long_rows = 1: one CTA per row, only rows with more than XMAP_SELECT_LONG records are done.
 * rows == NULL means all rows 0 .. n_rows-1. */
#define XMAP_SELECT_LONG 8192
int xmap_sim_select(const xmap_sim_args *args_h, const int32_t *rows, int32_t n_rows,
                    int32_t long_rows, void *stream);

/* Segmented copy of 16-byte records: record k of segment g goes from src[src_pos[g] + k] to
 * dst[dst_pos[g] + k]; seg_off = exclusive scan of the segment lengths, total = their sum.
 * Packs the neighbour-record lists addressed to another rank's rows into a contiguous send buffer
 * and appends received records to the owned lists, around the NCCL all-to-all that replaces the
 * reduceByKey shuffle of baselinerSim.py:210-211, 232-233. */
int xmap_segmented_copy16(const void *src, const int64_t *src_pos, void *dst, const int64_t *dst_pos,
                          const int64_t *seg_off, int32_t n_seg, int64_t total, void *stream);
/* the same for 4-byte elements (the rec_n array travels with the records) */
int xmap_segmented_copy4(const void *src, const int64_t *src_pos, void *dst, const int64_t *dst_pos,
                         const int64_t *seg_off, int32_t n_seg, int64_t total, void *stream);

/* ---------------------------------------------------------------------------
 * (3) X-SIM extension: masked path composition with fused aggregation and top-m.
 * Replaces: ExtendSim.sim_extend + get_final_extension (extender.py:46-217).
 * The facade turns the top-k tables into three index structures (all CSR-like):
 *   legs      per start item x: the left segments x -> t   (extender.py:160-168)
 *   partners  per bridge target t: the bridge pairs (t, s) (extender.py:61-81,178)
 *   rsegs     per bridge source s: the right segments s -> y (extender.py:134-138)
 * and this entry point evaluates every (leg, partner, rseg) combination = one
 * reference path: s_p = sum(sim*mutu)/sum(mutu), c_p = prod(frac)
 * (extender.py:83-89), accumulating xsim[x,y] = sum(s_p c_p)/sum(c_p)
 * (extender.py:198-201) in a SHARED-MEMORY hash table, never materialising paths and never touching a
 * global accumulator cell.
 *
 * Work unit = (start, a run of passes), run by ONE WARP with a private table of 2^cells_lg cells in
 * shared memory.  The end axis is hashed, pi(y) = (uint32)(y * 0x9E3779B1), and cut into 2^gb tiles by the
 * top gb bits of pi; a pass covers a range of tiles chosen so that its distinct ends fit the table.  Every
 * rseg list is stored sorted by pi and tile_ptr[s * (2^gb + 1) + g] = number of entries of list s in
 * tiles < g gives the sub-range of a pass without a search.  A pass that overflows its table is split in
 * two on the device and redone, down to one tile (then error 2).  Lanes that hit the same end in one
 * 32-path step are combined in lane (= path) order by the lowest lane, which updates the cell with plain
 * loads and stores: no atomics on values, no block barrier, and the summation order of every (start, end)
 * is a function of the path structure and the pass plan only, hence bit-identical for any number of GPUs.
 * ------------------------------------------------------------------------- */
#define XMAP_XSIM_MAX_CELLS_LG 13             /* per-warp table: warps x (2^cells_lg x 20 B + 2.9 KB) <= 227 KB */
typedef struct xmap_xsim_args {
    int32_t n_starts;                         /* start items covered by the units */
    int32_t n_units;                          /* units of this launch */
    const int32_t *unit_order;                /* [n_units] the q-th unit fetched is unit_order[q] (NULL: q); ids index the unit arrays */
    int32_t *unit_counter;                    /* device int: the fetch counter (zeroed by the call) */
    int32_t warps;                            /* warps per CTA, warps * 32 <= 640 */
    const int64_t *unit_leg_lo, *unit_leg_hi; /* leg range of the unit's start */
    const int32_t *unit_g0, *unit_g1;         /* the unit's range of hash tiles, 0 <= g0 < g1 <= 2^gb ... */
    const int32_t *unit_npass;                /* ... which it covers in npass equal passes (<= g1 - g0) */
    const int32_t *start_unit_ptr;            /* [n_starts + 1] unit id range of every start (merge) */
    /* (leg, partner) pairs in (start, leg, partner) order: lp_ptr = exclusive scan of the partners per leg over ALL
     * legs (lp_ptr[n_legs] = number of pairs; the kernels read it only at the unit's leg range); per pair the list it
     * walks and the left segment + bridge edge folded in path order: N = sum sim*mutu, D = sum mutu, C = prod frac */
    const int64_t *lp_ptr;
    const int32_t *pd_s;                      /* index into the right-segment / fused lists */
    const double *pd_n, *pd_d, *pd_c;
    const int64_t *rs_ptr;                    /* [n_s + 1] */
    const int32_t *rs_end;                    /* per right segment: end item, sorted by pi within a list */
    const double *rs_n, *rs_d, *rs_c;         /* sum sim*mutu, sum mutu, prod frac of its edges */
    const int32_t *tile_ptr; int32_t gb;
    int32_t cells_lg;                         /* log2 of a warp's shared-memory table size, 6 .. XMAP_XSIM_MAX_CELLS_LG */
    const int32_t *unit_clg;                  /* [n_units] log2 of the table a unit wants (NULL: cells_lg); a unit wanting more
                                               * than cells_lg runs with its table in the warp's slot of the global workspace */
    void *gws; int32_t gcells_lg;             /* workspace: (SMs x warps) slots of 20 B << gcells_lg (NULL: shared memory only) */
    int32_t top_m;                            /* <= XMAP_KMAX */
    /* per unit: distinct ends, paths, top-m by |xsim| (ties to the smaller end) */
    int32_t *unit_count; int64_t *unit_combos;
    int32_t *unit_top_end; double *unit_top_xsim; int32_t *unit_top_len;
    /* per start (merge) */
    int32_t *out_count; int64_t *out_combos;
    int32_t *top_end; double *top_xsim; int32_t *top_len;   /* [n_starts][top_m] */
    /* optional: every (end, xsim) of unit u written at emit_ptr[u] + 0 .. unit_count[u]-1 (order unspecified) */
    const int64_t *emit_ptr; int32_t *emit_end; double *emit_xsim;
    int32_t *error_flag;                      /* 2: a pass overflowed at the finest split */
    int64_t *unit_cycles;                     /* optional (NULL: off): SM clock cycles every unit took (xmap_xsim_extend only; tools/) */
} xmap_xsim_args;

int64_t xmap_xsim_smem_bytes(int32_t cells_lg, int32_t warps);
/* Both unit launchers write the per-unit results only; xmap_xsim_merge turns them into the per-start ones. */
int xmap_xsim_extend(const xmap_xsim_args *args_h, void *stream);
/* CTA-cooperative variant: one CTA of 8 warps per unit (blockIdx b runs unit_order[b]) with ONE table of
 * 2^cells_lg cells (two CTAs per SM, cells_lg >= 9); products are routed through shared memory to the warp that
 * owns the end's table region.  Same unit arrays, outputs and determinism contract; unit_counter / warps /
 * unit_clg / gws are not used. */
int64_t xmap_xsim_cta_smem_bytes(int32_t cells_lg);
int xmap_xsim_extend_cta(const xmap_xsim_args *args_h, void *stream);
/* only the per-start merge (multi-GPU: after the unit results of all ranks have been summed) */
int xmap_xsim_merge(const xmap_xsim_args *args_h, void *stream);

/* ---------------------------------------------------------------------------
 * (4) AlterEgo generation.
 * Replaces: Generator.cross_private_mapping / cross_nonprivate_mapping
 * (generator.py:27-111), assist.map_to_dict (assist.py:210-215) and
 * Generator.build_alterEgo (generator.py:113-157).
 * choose modes: 0 argmax (the shipped py3 behaviour of the private path),
 *               1 exponential mechanism, w_i = exp(eps*xsim_i/(2*range*GS)),
 *                 index = searchsorted_left(cumsum(w/sum w), u)  (generator.py:42-70),
 *               2 non-private: index floor(u*(m-1)) over the first min(m,4)
 *                 candidates (generator.py:109-110); m == 1 -> index 0.
 * uniforms: injected u[row] in [0,1) or NULL -> Philox4x32-10(seed, row).
 * ------------------------------------------------------------------------- */
int xmap_choose_mapping(const int32_t *top_end, const double *top_xsim, const int32_t *top_len,
                        int32_t n_rows, int32_t top_m, int32_t mode, int32_t n_cand,
                        double epsilon, int32_t mapping_range, int32_t global_sensitivity,
                        const double *uniforms, uint64_t seed,
                        int32_t *chosen, void *stream);

/* map[s] = max over rows with chosen == s of start_item[row]; map pre-filled with -1. */
int xmap_invert_mapping(const int32_t *start_item, const int32_t *chosen, int32_t n_rows,
                        int32_t *map, void *stream);

/* Rewrite every rating whose item has map >= 0 (CSR order), merge duplicates
 * of (user, target) by mean with the time of the smallest source item.
 * Returns the number of merged synthetic records through *n_out_h
 * (synchronises the stream). Output arrays sized >= nnz. */
size_t xmap_alterego_workspace_bytes(int64_t nnz);
int xmap_build_alterego(const int32_t *csr_ptr, const uint64_t *csr_ent, const int32_t *csr_src,
                        const int64_t *ts, int32_t n_users, int64_t nnz, const int32_t *map,
                        int32_t *out_user, int32_t *out_item, double *out_rating, int64_t *out_ts,
                        int64_t *n_out_h, void *workspace, size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------
 * (5) RecommenderSim on the AlterEgo profile (SURVEY.md 8(f) #1): item-item cosine with significance
 * weighting + per-pair local sensitivity.
 * Replaces: RecommenderSim.get_info / produce_pairwise / cosine_sim / calculate_sim with method
 * "cosine_item" (recommenderSim.py:29-62, 64-75, 90-132, 186-195; assist.py:153-175).
 * The profile is a flat record list (a (user, item) pair may occur twice; nothing is deduplicated or
 * filtered; self pairs (i, i) exist).
 *   xmap_recsim_item_info : info[3*i..] = (average, norm2, count) over the records of item i, the records
 *                           grouped by item (item_ptr [n_items + 1], rating_by_item).
 *   xmap_recsim_fill_rows : the entries of the item rows [i0, i1), i.e. those whose first record lies on an item
 *                           in the range (rows never share a directed pair, so a block of rows is filled, sorted and
 *                           reduced by itself).  Records grouped by user in list order (user_ptr [n_users + 1],
 *                           n_rec records); in_before [n_rec + 1] = exclusive scan of [item in range] over the
 *                           records; ent_before [n_rec + 1] = exclusive scan of [record in range] (user end - x - 1)
 *                           + (in-range records after x in its user), total = ent_before[n_rec].
 *                           key[t] = item_a * n_items + item_b, src[t] = pos_a << 32 | pos_b, t in the reference's
 *                           emission order restricted to the rows, so a STABLE sort by key keeps arrival order.
 *                           With [0, n_items) these are all d(d-1) entries of every user.
 *   xmap_recsim_pairs     : per run of equal keys [seg_ptr[g], seg_ptr[g+1]) of the sorted entries:
 *                           (i, j, n, sim, local sensitivity); NaN rule of Python's max() reproduced.
 * ------------------------------------------------------------------------- */
int xmap_recsim_item_info(const int64_t *item_ptr, const double *rating_by_item, int32_t n_items, double *info,
                          void *stream);
int xmap_recsim_fill_rows(const int64_t *user_ptr, int32_t n_users, const int64_t *in_before, const int64_t *ent_before,
                          int64_t n_rec, const int32_t *item, int64_t n_items, int32_t i0, int32_t i1, int64_t total,
                          int64_t *key, int64_t *src, void *stream);
int xmap_recsim_pairs(const int64_t *seg_ptr, const int64_t *seg_key, const int64_t *src, const double *rating,
                      const double *info, int64_t n_items, int64_t n_pairs, int32_t num_atleast,
                      int32_t *out_i, int32_t *out_j, int64_t *out_n, double *out_sim, double *out_ls, void *stream);

/* (5b) Non-private neighbour selection on the RecommenderSim output (SURVEY.md 8(f) #2;
 * RecommenderPrivacy.nonprivate_neighbor_selection + nonnoise_perturbation, recommenderPrivacy.py:141-189):
 * per item the first k neighbours by |sim| descending, ties to the smaller index; row_ptr [n_items + 1]
 * indexes the (i, j)-sorted pair arrays.  Tables [n_items][k]. */
int xmap_recsim_neighbors(const int64_t *row_ptr, const int32_t *pair_j, const double *pair_sim, int32_t n_items,
                          int32_t k, int32_t *nb_idx, double *nb_sim, int32_t *nb_len, void *stream);
/* (5c) Item-based prediction of test (user, item) pairs on the AlterEgo profile (SURVEY.md 8(f) #3;
 * RecommenderPrediction.item_based_prediction, recommenderPrediction.py:26-103): profile records grouped by user
 * in list order (prof_ptr [n_users + 1]); pred_* = bounded rating without / with temporal decay, -1 where the
 * item has no neighbour list.  error_flag 4: more than 128 matching profile records for one prediction. */
int xmap_recsim_predict(const int64_t *prof_ptr, const int32_t *prof_item, const double *prof_rating,
                        const int64_t *prof_ts, const double *info, const int32_t *nb_idx, const double *nb_sim,
                        const int32_t *nb_len, int32_t k, const int32_t *t_user, const int32_t *t_item, int64_t n_test,
                        double alpha, double *pred_nodecay, double *pred_decay, int32_t *error_flag, void *stream);

/* (5c) PRIVATE neighbour selection + noise perturbation (RecommenderPrivacy.private_neighbor_selection +
 * noise_perturbation, recommenderPrivacy.py:35-139, 152-171) as the reference behaves under Python 3 (one neighbour per
 * item: np.count_nonzero(map(...)), :81, counts the map object): drawn from exp(eps * max(sim, sim - w) / (2 k RS_j))
 * over the item's neighbours in |sim|-descending order; its similarity + Laplace(|RS| / eps).
 *   row_ptr [n_items + 1], nbr / sim / ls: per item its neighbours in |sim|-descending STABLE order (the caller sorts)
 *   eps = privacy_epsilon / 2 (recommenderPrivacy.py:18); u_pick / u_noise [n_items]: injected uniforms or NULL ->
 *   Philox4x32-10(seed, item, 0 / 1); scratch: one double per neighbour; out_len[i] = 0 for an item without neighbours */
int xmap_recsim_private_neighbor(const int64_t *row_ptr, const int32_t *nbr, const double *sim, const double *ls,
                                 int32_t n_items, int32_t mapping_range, double eps, double rpo,
                                 const double *u_pick, const double *u_noise, uint64_t seed, double *scratch,
                                 int32_t *out_nbr, double *out_sim, int32_t *out_len, void *stream);

/* ---------------------------------------------------------------------------
 * (6) Clean stage on encoded records (SURVEY.md 8(f) #4).
 * Replaces the data-parallel part of BaselinerClean: the period test of parse_data (baselinerClean.py:47-52, given as
 * the two instants [t_lo, t_hi) the local-time years [date_from, date_to] span), filter_data (:62-92: per (user, item)
 * the strictly latest rating, the first seen winning ties) and clean_data (:94-97: users with fewer than num_atleast
 * items are dropped).  Splitting the text lines and the id dictionaries stay on the host.
 *   order      : [n] record indices sorted, stable, by (out-of-period last, user, item)
 *   keep       : [n] out, 1 for the records that survive
 *   user_items : [n_users] out, distinct in-period items per user (before the num_atleast test)
 * ------------------------------------------------------------------------- */
int xmap_clean_records(const int32_t *user, const int32_t *item, const double *ts, const int64_t *order,
                       int64_t n, int32_t n_users, double t_lo, double t_hi, int32_t num_atleast,
                       uint8_t *keep, int32_t *user_items, void *stream);

/* ---------------------------------------------------------------------------
 * (7) Text ingest of the rating files: the 4-column reader and the per-record work of clean / split.
 * Replaces LocalContext.textFile (text mode), the per-line work of BaselinerClean.parse_data
 * (baselinerClean.py:38-56) and the record placement of BaselinerSplit.split_data (baselinerSplit.py:60-106).
 * The facade is x-map_b200/ingest.py; the per-user steps of the split (randomSplit, random.sample) stay on the host.
 *
 * Byte pass: xmap_ingest_line_masks reads the file bytes (16-byte aligned, padded to 16 bytes) with 16-byte loads and
 * writes one 16-bit mask per 16-byte chunk, bit b = byte 16c+b ends a line (\n, or \r not followed by \n);
 * block_cnt[blockIdx] = terminators of each 4 096-byte block.  The caller scans block_cnt into block_off (exclusive,
 * int64) and xmap_ingest_line_offsets writes offs[k] = byte position of the k-th terminator.  Line k is
 * [offs[k-1] + 1, offs[k]) (offs[-1] = -1); a file that does not end in a terminator gets one appended by the caller.
 *
 * xmap_ingest_parse: per line, status (below), rating and timestamp as float64 (NaN unless OK), and the two ids as
 * big-endian 64-bit words, zero padded, column-major: uid_words[w * ld + line], iid_words the same with the domain
 * label (<= 16 bytes) appended to the raw item id.  Only the words an id covers are written: the caller zeroes the
 * word arrays.  Whitespace = Python's ASCII str.split() set; fields after the fourth are ignored.  Numbers:
 * [+-]?(d+(.d*)?|.d+)([eE][+-]?d+)? with at most 15 significant digits and a decimal exponent within +-22 (one
 * correctly rounded operation: bit-equal to Python's float()); timestamps within [ts_min, ts_max].
 *
 * xmap_ingest_rank_flags / _scatter: over ids sorted by an LSD sequence of stable sorts of their words (perm),
 * flag[p] = (id at p != id at p-1); the caller scans flag into csum (inclusive, int64); rank[perm[p]] = csum[p] - 1 and
 * rep[rank] = a line holding that id.
 * xmap_ingest_first: records in clean order (xmap_clean_records' `order`): first_user[u] = min in-period line of u
 * (initialised to INT32_MAX by the caller), pair_first[r] = first in-period line of the (user, item) of kept record r.
 * xmap_ingest_item_suffix: present[key of iid[-2:]] = 1 (65 536 bytes, zeroed by the caller; key = byte[-2] << 8 |
 * byte[-1], a 1-byte id: byte << 8).  xmap_ingest_item_codes: the codes of encode.item_codes for items in ascending
 * id order, rep[i] = a line holding item i; labels = the sorted present keys (<= 8); prefix_new[i] = iid[:2] differs
 * from item i-1's (scanned by the caller into the prefix rank).
 * xmap_ingest_train_keys: key[r] = group << 58 | upos[user] << 26 | sub, -1 for a test record; grp[u] 0 non-overlap
 * source, 1 non-overlap target, 2 both, 3 rest, 4 test user; a test user's record without "S:" is drawn into training
 * if srank[r] >= 0 (sub = 1 + srank, the order of random.sample), else it is a test record.
 * ------------------------------------------------------------------------- */
#define XMAP_INGEST_ID_MAX 48          /* longest uid, and longest raw iid + label, in bytes */
#define XMAP_INGEST_OK 0
#define XMAP_INGEST_BLANK 1            /* whitespace only: skipped */
#define XMAP_INGEST_FEW_FIELDS 2
#define XMAP_INGEST_NON_ASCII 3
#define XMAP_INGEST_NUL 4
#define XMAP_INGEST_BAD_TIME 5
#define XMAP_INGEST_TIME_RANGE 6
#define XMAP_INGEST_BAD_RATING 7
#define XMAP_INGEST_UID_LONG 8
#define XMAP_INGEST_IID_LONG 9
int xmap_ingest_line_masks(const void *buf, int64_t size, uint16_t *masks, int32_t *block_cnt, void *stream);
int xmap_ingest_line_offsets(const uint16_t *masks, int64_t size, const int64_t *block_off, int64_t *offs, void *stream);
int xmap_ingest_parse(const uint8_t *buf, const int64_t *offs, int64_t n_lines, const char *label_h, int32_t label_len,
                      double ts_min, double ts_max, int64_t ld, uint8_t *status, double *rating, double *ts,
                      uint64_t *uid_words, uint8_t *uid_len, uint64_t *iid_words, uint8_t *iid_len, void *stream);
int xmap_ingest_rank_flags(const uint64_t *words, int64_t ld, int32_t n_words, const int64_t *perm, int64_t n,
                           int32_t *flag, void *stream);
int xmap_ingest_rank_scatter(const int64_t *perm, const int32_t *flag, const int64_t *csum, int64_t n, int32_t *rank,
                             int64_t *rep, void *stream);
int xmap_ingest_first(const int32_t *user, const int32_t *item, const double *ts, const int64_t *order,
                      const uint8_t *keep, int64_t n, double t_lo, double t_hi, int32_t *first_user, int32_t *pair_first,
                      void *stream);
int xmap_ingest_item_suffix(const uint64_t *iid_words, int64_t ld, const uint8_t *iid_len, const int64_t *rep,
                            int32_t n_items, uint8_t *present, void *stream);
int xmap_ingest_item_codes(const uint64_t *iid_words, int64_t ld, const uint8_t *iid_len, const int64_t *rep,
                           int32_t n_items, const int32_t *labels, int32_t n_labels, int32_t *prefix_new,
                           uint8_t *dom_code, uint8_t *contains, bool *has_S, bool *has_T, void *stream);
int xmap_ingest_train_keys(const int32_t *user, const int32_t *item, const int8_t *grp, const int32_t *upos,
                           const bool *has_S, const int32_t *srank, int64_t n, int64_t *key, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* XMAP_B200_H */
