"""Array-level driver of the CUDA hot path (one process = one GPU).

Everything here works on integer-encoded tensors resident in HBM and calls the
C ABI (include/xmap_b200.h) through ctypes; torch supplies device memory,
streams and a few index-building primitives (sort / cumsum / repeat_interleave)
around the kernels.  The reference-shaped facades in core/ and utils/assist.py
sit on top of this module.  No CPU fallback exists: without a GPU and the built
extension these functions raise.
"""
import os
from dataclasses import dataclass, field

import torch

from . import _native as N



def _stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def _dev(t, dtype, device):
    return torch.as_tensor(t, dtype=dtype).to(device, non_blocking=True).contiguous()


@dataclass
class ItemMeta:
    """Per-item codes the reference derives from id strings (see encode.py)."""
    prefix_code: torch.Tensor     # int32  iid[:2]
    dom_code: torch.Tensor        # uint8  iid[-2:]
    contains: torch.Tensor        # uint8  bit d: label d in iid
    has_S: torch.Tensor           # bool   "S:" in iid
    has_T: torch.Tensor           # bool   "T:" in iid


def to_device_meta(meta, device="cuda"):
    """dict of host arrays (encode.item_codes order: prefix_code, dom_code, contains, has_S, has_T) -> ItemMeta."""
    T = lambda key, dt: torch.as_tensor(meta[key], dtype=dt, device=device)
    return ItemMeta(prefix_code=T("prefix_code", torch.int32), dom_code=T("dom_code", torch.uint8),
                    contains=T("contains", torch.uint8), has_S=T("has_S", torch.bool), has_T=T("has_T", torch.bool))


@dataclass
class Layout:
    n_users: int
    n_items: int
    nnz: int
    csr_ptr: torch.Tensor
    csr_ent: torch.Tensor
    csr_src: torch.Tensor
    csc_ptr: torch.Tensor
    csc_ent: torch.Tensor
    user_mu: torch.Tensor
    item_stats: torch.Tensor      # [n_items, 4] = (avg, norm2, adj_norm2, count)
    row_work: torch.Tensor        # int64 [n_items]


def build_layout(user, item, rating, n_users, n_items, device="cuda"):
    """CSR/CSC + user/item statistics (xmap_build_layout, xmap_row_work)."""
    L = N.lib()
    user = _dev(user, torch.int32, device)
    item = _dev(item, torch.int32, device)
    rating = _dev(rating, torch.float32, device)
    nnz = int(user.numel())
    i32 = dict(dtype=torch.int32, device=device)
    f64 = dict(dtype=torch.float64, device=device)
    csr_ptr = torch.empty(n_users + 1, **i32)
    csc_ptr = torch.empty(n_items + 1, **i32)
    csr_ent = torch.empty(nnz, dtype=torch.int64, device=device)
    csc_ent = torch.empty(nnz, dtype=torch.int64, device=device)
    csr_src = torch.empty(nnz, **i32)
    user_mu = torch.empty(n_users, **f64)
    item_stats = torch.empty(n_items, 4, **f64)
    ws_bytes = L.xmap_layout_workspace_bytes(nnz, n_users, n_items)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)
    N.check(L.xmap_build_layout(N.ptr(user), N.ptr(item), N.ptr(rating), nnz, n_users, n_items,
                                N.ptr(csr_ptr), N.ptr(csr_ent), N.ptr(csr_src),
                                N.ptr(csc_ptr), N.ptr(csc_ent), N.ptr(user_mu), N.ptr(item_stats),
                                N.ptr(ws), ws_bytes, _stream_ptr()), "xmap_build_layout")
    row_work = torch.empty(n_items, dtype=torch.int64, device=device)
    N.check(L.xmap_row_work(N.ptr(csr_ptr), N.ptr(csc_ptr), N.ptr(csc_ent), n_items,
                            N.ptr(row_work), _stream_ptr()), "xmap_row_work")
    del ws
    return Layout(n_users, n_items, nnz, csr_ptr, csr_ent, csr_src, csc_ptr, csc_ent,
                  user_mu, item_stats, row_work)


EXP_FIELD_MAX = 127           # largest item exponent the 7-bit field of the triangular entries holds
EXP_CLAMP_MAX = 16            # octaves an item exponent may be raised to fit the field before the input is refused


def exponent_base(method, item_stats):
    """e_base of the item exponents (xmap_build_tri_layout): with 2^(E-1) <= den < 2^E for the norm den of
    every item with den > 0, e_base = max E - 127, and the kernels scale the inner product of items i, j by
    2^(62 - E_i - E_j).  An item whose E lies below e_base is raised to it, which costs its pairs that many
    bits; more than EXP_CLAMP_MAX of them raises ValueError."""
    den = item_stats[:, 1 if method == "cosine" else 2]
    den = den[den > 0]
    if den.numel() == 0:
        return 0
    e = torch.frexp(den).exponent
    lo, hi = int(e.min()), int(e.max())
    if hi - lo > EXP_FIELD_MAX + EXP_CLAMP_MAX:
        raise ValueError("item norms span 2^%d (from 2^%d to 2^%d): more than the similarity stage's fixed-point "
                         "inner product resolves (2^%d)" % (hi - lo, lo - 1, hi, EXP_FIELD_MAX + EXP_CLAMP_MAX))
    return hi - EXP_FIELD_MAX


@dataclass
class SimTables:
    """Output of the similarity + selection stage."""
    k: int
    n_items: int
    row_flags: torch.Tensor       # uint8 [I]  1: bridge (BB) item
    row_npairs: torch.Tensor      # int32 [I]  co-rated pairs (pre-filter) row i evaluated: the pairs (i, j)
                                  #            with j more popular than i; 2 * sum = directed co-rated pairs
    row_nkept: torch.Tensor       # int32 [I]  neighbours surviving the filter (= length of the record list)
    tab_idx: torch.Tensor         # int32 [I,2,k]
    tab_sim: torch.Tensor         # f64   [I,2,k]
    tab_mutu: torch.Tensor        # int32 [I,2,k]
    tab_n: torch.Tensor           # int32 [I,2,k]
    tab_len: torch.Tensor         # int32 [I,2]
    launches: int = 0
    stats: dict = field(default_factory=dict)

    @property
    def n_pairs_total(self):
        """Directed co-rated item pairs evaluated (SURVEY.md 8d: P)."""
        return 2 * int(self.row_npairs.sum().item())


CELL_CLASSES = tuple(int(c) for c in os.environ.get("XMAP_CELL_CLASSES", "256,512,1024,1536,2048,3072,4096,6144,8192,12288").split(","))   # table capacities (16-byte cells) of the launches


def _threads_for_cells(c):
    """Threads per row a table capacity gets at least: 8 cells per thread (measured best of 4 / 8 / 16 / 32)."""
    return max(32, min(512, (c // 8 + 31) // 32 * 32))

REC_BYTES = 20                                              # 16-byte record + its int32 co-rating count
SPLIT_RATERS = int(os.environ.get("XMAP_SPLIT_RATERS", "16384"))   # rows with at least this many raters are split ...
SPLIT_SEG = 4096                                            # ... into segments of this many raters
_PINNED = {}                                                # pinned host buffers of tables_to_host


_REC_POOL = {}                                              # device -> record buffers of finished engines


def _rec_words(n_records):
    """int64 words of the storage of n records: [n, 2] record words followed by the int32 counts."""
    n = max(int(n_records), 1)
    return 2 * n + (n + 1) // 2


def _rec_buffer(n_records, device):
    """Record-list storage (one flat int64 buffer, see _rec_views).  The buffer is by far the largest
    allocation of the stage (15 GB at cfg2); engines hand it back when they die and the next one takes it
    over, so a sequence of runs does not depend on how the caching allocator happens to split and re-grow
    a block of that size."""
    need = _rec_words(n_records)
    pool = _REC_POOL.setdefault(str(device), [])
    fit = [q for q, t in enumerate(pool) if t.numel() >= need]
    if fit:
        return pool.pop(min(fit, key=lambda q: pool[q].numel()))      # by position: `in` / remove would compare tensors
    pool.clear()                                          # too small for this problem: let the allocator have them
    return torch.empty(need, dtype=torch.int64, device=device)


def _rec_views(raw, n_records):
    """(rec [n, 2] int64 = {sim bits, other item | mutu << 32}, rec_n [n] int32) inside a raw buffer."""
    n = max(int(n_records), 1)
    return raw[:2 * n].view(n, 2), raw[2 * n:2 * n + (n + 1) // 2].view(torch.int32)[:n]


def popularity_order(count):
    """ord[i] = rank of (count(i), i) ascending; the most popular item gets the largest ord."""
    I = int(count.numel())
    key = count.long() * (1 << 24) + torch.arange(I, device=count.device)
    perm = torch.argsort(key)
    ord_ = torch.empty(I, dtype=torch.int32, device=count.device)
    ord_[perm] = torch.arange(I, dtype=torch.int32, device=count.device)
    return ord_


class SimEngine:
    """Similarity + top-k selection over a Layout (C ABI section 2)."""

    def __init__(self, layout, meta, method="adjust_cosine", num_atleast=50, k=10,
                 max_smem_cells=CELL_CLASSES[-1], rec_budget=None):
        if method not in N.METHODS:
            raise ValueError("unknown similarity method %r" % (method,))
        if not (1 <= k <= N.KMAX):
            raise ValueError("top_k must be in [1, %d]" % N.KMAX)
        self.lay, self.meta = layout, meta
        self.method, self.num_atleast, self.k = method, int(num_atleast), int(k)
        self.device = layout.csr_ptr.device
        self.e_base = exponent_base(method, layout.item_stats)
        self.max_smem_cells = int(max_smem_cells)
        self.launches = 0
        I = layout.n_items
        dev = self.device
        L = N.lib()
        # ---- triangular layout -------------------------------------------------------------------
        count = layout.item_stats[:, 3]
        self.ord = popularity_order(count)
        self.ord_item = torch.empty(I, dtype=torch.int32, device=dev)
        self.ord_item[self.ord.long()] = torch.arange(I, dtype=torch.int32, device=dev)
        self.tcsr_ent = torch.empty(layout.nnz, dtype=torch.int64, device=dev)
        self.csc_aux = torch.empty((layout.nnz, 2), dtype=torch.int64, device=dev)
        self.ostat = torch.empty(max(I, 1) * 16, dtype=torch.uint8, device=dev)
        self.tri_work = torch.zeros(I, dtype=torch.int64, device=dev)
        ws_bytes = L.xmap_tri_workspace_bytes(layout.nnz)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        N.check(L.xmap_build_tri_layout(
            N.ptr(layout.csr_ptr), N.ptr(layout.csr_ent), N.ptr(layout.csc_ptr), N.ptr(layout.csc_ent),
            N.ptr(layout.user_mu), N.ptr(layout.item_stats), N.ptr(meta.prefix_code), N.ptr(self.ord),
            layout.n_users, I, layout.nnz, N.METHODS[method], self.e_base,
            N.ptr(self.tcsr_ent), N.ptr(self.csc_aux), N.ptr(self.ostat), N.ptr(self.tri_work),
            N.ptr(ws), ws_bytes, _stream_ptr()), "xmap_build_tri_layout")
        del ws
        # ---- neighbour-record lists: capacity = co-rating products of the full row, at most I - 1;
        # when that bound does not fit (rec_budget), the first run does an exact sizing pass instead
        cap = torch.clamp(layout.row_work - count.long(), min=0, max=max(I - 1, 0))
        self.rec_ptr = torch.zeros(I + 1, dtype=torch.int64, device=dev)
        self.rec_ptr[1:] = torch.cumsum(cap, 0)
        self.rec_cap = cap
        self.rec_cap_bound = cap       # rank-invariant upper bound (rec_cap becomes rank-specific after exact sizing)
        total = int(self.rec_ptr[-1].item()) if I else 0
        if rec_budget is None:
            free, _ = torch.cuda.mem_get_info(dev)
            pooled = max((t.numel() * 8 for t in _REC_POOL.get(str(dev), [])), default=0)
            rec_budget = max(free // 2, pooled)
        self.exact_sizing = total * REC_BYTES > rec_budget
        self._rec_raw = None
        self.rec = self.rec_n = None
        if not self.exact_sizing:
            self._set_rec(_rec_buffer(total, dev), total)
        self.rec_cnt = torch.zeros(I, dtype=torch.int32, device=dev)
        self.bb = torch.zeros(I, dtype=torch.uint8, device=dev)
        self.row_npairs = torch.zeros(I, dtype=torch.int32, device=dev)
        self.error_flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self.tab_idx = torch.full((I, 2, k), -1, dtype=torch.int32, device=dev)
        self.tab_sim = torch.zeros((I, 2, k), dtype=torch.float64, device=dev)
        self.tab_mutu = torch.zeros((I, 2, k), dtype=torch.int32, device=dev)
        self.tab_n = torch.zeros((I, 2, k), dtype=torch.int32, device=dev)
        self.tab_len = torch.zeros((I, 2), dtype=torch.int32, device=dev)
        self._gtab = None
        self._side = None
        self._plans = {}
        self.profile = None        # dict kind -> [(start_event, end_event)] when enabled

    def _set_rec(self, raw, n_records):
        self._rec_raw = raw
        self.rec, self.rec_n = _rec_views(raw, n_records)

    def _give_back(self):
        raw = getattr(self, "_rec_raw", None)
        self._rec_raw = self.rec = self.rec_n = None
        if raw is not None and raw.numel() > (1 << 21) and _REC_POOL is not None:
            pool = _REC_POOL.setdefault(str(raw.device), [])
            if len(pool) < 2:
                pool.append(raw)

    def __del__(self):
        try:
            self._give_back()
        except Exception:            # interpreter shutdown: module globals may be gone
            pass

    def release_lists(self):
        """Drop the record storage so that the next stage sizes the lists exactly (multi-GPU: decided collectively)."""
        self._give_back()
        self.exact_sizing = True

    # -- argument block ----------------------------------------------------
    def _args(self):
        lay, m = self.lay, self.meta
        a = N.SimArgs()
        a.csc_ptr, a.csc_ent, a.csc_aux = N.ptr(lay.csc_ptr), N.ptr(lay.csc_ent), N.ptr(self.csc_aux)
        a.tcsr_ent = N.ptr(self.tcsr_ent)
        a.ostat, a.ord, a.tri_work = N.ptr(self.ostat), N.ptr(self.ord), N.ptr(self.tri_work)
        a.ord_item = N.ptr(self.ord_item)
        a.dom_code, a.contains = N.ptr(m.dom_code), N.ptr(m.contains)
        a.n_items, a.method = lay.n_items, N.METHODS[self.method]
        a.num_atleast, a.k, a.r2_bits = self.num_atleast, self.k, 2 * self.e_base
        a.rec_ptr, a.rec_cnt, a.rec, a.rec_n = N.ptr(self.rec_ptr), N.ptr(self.rec_cnt), N.ptr(self.rec), N.ptr(self.rec_n)
        a.count_only = 1 if self.rec is None else 0
        a.bb, a.row_npairs = N.ptr(self.bb), N.ptr(self.row_npairs)
        a.tab_idx, a.tab_sim = N.ptr(self.tab_idx), N.ptr(self.tab_sim)
        a.tab_mutu, a.tab_n, a.tab_len = N.ptr(self.tab_mutu), N.ptr(self.tab_n), N.ptr(self.tab_len)
        a.error_flag = N.ptr(self.error_flag)
        return a

    # -- planning ----------------------------------------------------------
    def plan(self, rows=None):
        """Group the rows by table capacity and threads per row (cached per row set).
        Returns (launches, long_candidates, split): launches = [(rows sorted by descending work,
        cells_cap, threads_per_row, in_global_memory, row headers)], long_candidates = rows whose record
        list can exceed XMAP_SELECT_LONG, split = segment arrays of the rows whose rater list is
        cut over several CTAs (or None)."""
        key = None
        if rows is not None:
            n = int(rows.numel())
            lo = int(rows[0]) if n else -1
            contiguous = n == 0 or (int(rows[-1]) == lo + n - 1 and bool((rows[1:] - rows[:-1] == 1).all()))
            key = (lo, n) if contiguous else ("set", hash(tuple(rows.cpu().tolist())))
        if key in self._plans:
            return self._plans[key]
        dev, I = self.device, self.lay.n_items
        if rows is None:
            rows = torch.arange(I, dtype=torch.int32, device=dev)
        else:
            rows = rows.to(dev, dtype=torch.int32)
        rl = rows.long()
        work = self.tri_work[rl]
        rtop = (I - 1 - self.ord[rl]).long()
        h = torch.clamp((work * 4 + 2) // 3, min=32)
        cells = torch.where(rtop <= h, rtop, h)
        classes = [c for c in CELL_CLASSES if c <= self.max_smem_cells] or [self.max_smem_cells]
        if classes[-1] < self.max_smem_cells:
            classes.append(self.max_smem_cells)
        bounds = torch.tensor(classes, dtype=torch.int64, device=dev)
        cls = torch.bucketize(cells, bounds)                       # len(classes) = global-memory fallback
        t_cells = torch.tensor([_threads_for_cells(c) for c in classes] + [512], dtype=torch.int64, device=dev)[cls]
        t_work = torch.full_like(work, 32)
        t_work[work > 3072] = 128
        t_work[work > 8192] = 256
        t_work[work > 32768] = 512
        threads = torch.maximum(t_cells, t_work)
        live = work > 0
        # rows with very long rater lists (popular items) are cut into segments, one CTA each
        craters = (self.lay.csc_ptr[rl + 1] - self.lay.csc_ptr[rl]).long()
        is_split = live & (rtop <= h) & (craters >= SPLIT_RATERS) & (cells <= self.max_smem_cells)
        split = None
        if bool(is_split.any()):
            srows, sr_c = rows[is_split], craters[is_split]
            o = torch.argsort(sr_c, descending=True, stable=True)
            srows, sr_c = srows[o], sr_c[o]
            nseg = (sr_c + SPLIT_SEG - 1) // SPLIT_SEG
            slot = torch.repeat_interleave(torch.arange(srows.numel(), device=dev), nseg)
            q = torch.arange(int(nseg.sum().item()), device=dev) - (torch.cumsum(nseg, 0) - nseg)[slot]
            base = self.lay.csc_ptr[srows.long()].long()[slot]
            seg_lo = base + q * SPLIT_SEG
            seg_hi = torch.minimum(seg_lo + SPLIT_SEG, base + sr_c[slot])
            cap = max(32, int(cells[is_split].max().item()))
            i32 = lambda t: t.to(torch.int32).contiguous()
            split = dict(hdr=self._headers(i32(srows[slot]), i32(seg_lo), i32(seg_hi)), seg_slot=i32(slot),
                         slot_nseg=i32(nseg), n_segs=int(slot.numel()), cells_cap=cap, rows=srows,
                         gtab=torch.zeros((srows.numel() * cap, 2), dtype=torch.int64, device=dev),
                         done=torch.zeros(srows.numel(), dtype=torch.int32, device=dev))
            live = live & ~is_split
        # one sort by (launch group, descending work) yields every launch's row list as a slice
        code = (cls * 2048 + threads)[live]
        rows_l, work_l, cells_l = rows[live], work[live], cells[live]
        order = torch.argsort(code * (1 << 40) + ((1 << 40) - 1 - work_l.clamp(max=(1 << 40) - 1)))
        rows_s = rows_l[order].contiguous()
        codes, counts = torch.unique_consecutive(code[order], return_counts=True)
        gmax = torch.zeros(int(cls.max().item()) * 2048 + 2048 if cls.numel() else 1, dtype=torch.int64, device=dev)
        gmax.scatter_reduce_(0, code, cells_l, "amax")
        launches, at = [], 0
        for c, n, mx in zip(codes.tolist(), counts.tolist(), gmax[codes].tolist()):
            r = rows_s[at:at + n]
            at += n
            q, th = c // 2048, c % 2048
            if q < len(classes):
                launches.append((r, classes[q], th, False, self._headers(r)))
            else:
                launches.append((r, int(mx), 512, True, self._headers(r)))
        launches.sort(key=lambda t: (-t[2], -t[1]))                # big CTAs first
        long_cand = rows[self.rec_cap[rl] > N.SELECT_LONG].contiguous()
        out = (launches, long_cand, split)
        self._plans[key] = out
        return out

    def _headers(self, rows, seg_lo=None, seg_hi=None):
        """48-byte row headers of a launch (xmap_sim_row_headers)."""
        n = int(rows.numel())
        hdr = torch.empty(max(n, 1) * N.ROW_HDR_BYTES, dtype=torch.uint8, device=self.device)
        N.check(N.lib().xmap_sim_row_headers(self._args(), N.ptr(rows), n, N.ptr(seg_lo), N.ptr(seg_hi), N.ptr(hdr),
                                             _stream_ptr()), "xmap_sim_row_headers")
        return hdr

    def enable_profile(self):
        """Record a CUDA event pair around every kernel group (read with profile_ms())."""
        self.profile = {}

    def _timed(self, kind, fn):
        if self.profile is None:
            return fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        self.profile.setdefault(kind, []).append((a, b))
        return r

    def profile_ms(self):
        """{kind: (launch groups, total ms)}; synchronises."""
        torch.cuda.synchronize()
        out = {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in (self.profile or {}).items()}
        self.profile = {}
        return out

    def _check_error(self):
        e = int(self.error_flag.item())
        if e != 0:
            raise N.NativeError("similarity kernel error %d (1: table overflow, 2: record-list capacity, "
                                "3: co-rating count out of range)" % e)

    # -- stages ------------------------------------------------------------
    def reset(self):
        self.rec_cnt.zero_()
        self.bb.zero_()
        self.row_npairs.zero_()

    def _size_lists(self, rows=None):
        """Exact sizing pass (only when the upper bound does not fit): the accumulate kernels run once
        with count_only = 1, the list lengths become the extents.  In a multi-GPU run the lengths are
        this rank's own records; the exchange appends the others', so the caller must add them (see
        multi.similarity_step)."""
        self._give_back()
        self.reset()
        self._accumulate(rows)
        self._check_error()
        return self.rec_cnt.long().clone()

    def _alloc_lists(self, lengths):
        I, dev = self.lay.n_items, self.device
        self.rec_ptr = torch.zeros(I + 1, dtype=torch.int64, device=dev)
        self.rec_ptr[1:] = torch.cumsum(lengths, 0)
        self.rec_cap = lengths
        total = int(self.rec_ptr[-1].item()) if I else 0
        self._set_rec(_rec_buffer(total, dev), total)
        self._plans = {}
        self.reset()

    def accumulate(self, rows=None):
        if self.rec is None:
            self._alloc_lists(self._size_lists(rows))
        return self._accumulate(rows)

    def _accumulate(self, rows=None):
        """Triangular similarity rows -> neighbour records of both ends, BB flags (xmap_sim_accumulate).
        The launches (one per table capacity / group width) are dealt round-robin to a few streams so
        that the tail of one overlaps the next and the long-running popular rows do not hold the GPU;
        with per-kernel timing enabled everything is serialised on the current stream."""
        L = N.lib()
        args = self._args()
        launches, _, split = self.plan(rows)
        main = torch.cuda.current_stream()
        n_streams = int(os.environ.get("XMAP_SIM_STREAMS", "3"))
        use_side = self.profile is None and len(launches) > 1 and n_streams > 1
        if use_side and self._side is None:
            self._side = [torch.cuda.Stream(device=self.device) for _ in range(n_streams - 1)]
        if use_side:
            for sd in self._side:
                sd.wait_stream(main)
        stats = []
        if split is not None:
            sp = split
            self._timed("accumulate_split", lambda: N.check(L.xmap_sim_accumulate_split(
                args, N.ptr(sp["hdr"]), N.ptr(sp["seg_slot"]), N.ptr(sp["slot_nseg"]), sp["n_segs"], sp["cells_cap"],
                N.ptr(sp["gtab"]), N.ptr(sp["done"]), main.cuda_stream), "xmap_sim_accumulate_split"))
            self.launches += 1
            stats.append(("accumulate_split", int(sp["rows"].numel())))
        for q, (r, cells_cap, threads, in_gmem, hdr) in enumerate(launches):
            gtab, ctas = None, 0
            if in_gmem:
                ctas = min(int(r.numel()), 296)
                need = ctas * ((cells_cap * 20 + 15) // 16 * 16)
                if self._gtab is None or self._gtab.numel() < need:
                    self._gtab = None
                    self._gtab = torch.empty(need, dtype=torch.uint8, device=self.device)
                gtab = self._gtab
            kind = "accumulate_%s%d_t%d" % ("g" if in_gmem else "c", cells_cap, threads)
            stream = main
            if use_side and not in_gmem and q % n_streams:
                stream = self._side[q % n_streams - 1]
            st = stream.cuda_stream
            self._timed(kind, lambda: N.check(L.xmap_sim_accumulate(
                args, N.ptr(hdr), r.numel(), cells_cap, threads, N.ptr(gtab), ctas, st), "xmap_sim_accumulate"))
            self.launches += 1
            stats.append((kind, int(r.numel())))
        if use_side:
            for sd in self._side:
                main.wait_stream(sd)
        return stats

    def select(self, rows=None):
        """Per-row top-k lists from the neighbour records (xmap_sim_select); needs every item's BB flag."""
        L = N.lib()
        st = _stream_ptr()
        args = self._args()
        _, long_cand, _ = self.plan(rows)
        n = self.lay.n_items if rows is None else int(rows.numel())
        rp = None if rows is None else N.ptr(rows.to(self.device, dtype=torch.int32).contiguous())
        self._timed("select_warp", lambda: N.check(L.xmap_sim_select(args, rp, n, 0, st), "xmap_sim_select"))
        self.launches += 1
        if long_cand.numel():
            self._timed("select_cta", lambda: N.check(
                L.xmap_sim_select(args, N.ptr(long_cand), long_cand.numel(), 1, st), "xmap_sim_select(long)"))
            self.launches += 1

    def run(self, rows=None):
        """Single-GPU convenience: reset, accumulate, select, error check."""
        self.reset()
        stats = self.accumulate(rows)
        self.select(rows)
        self._check_error()
        return self.tables(dict(accumulate=stats))

    def tables(self, stats=None, row_nkept=None):
        return SimTables(self.k, self.lay.n_items, self.bb, self.row_npairs,
                         self.rec_cnt if row_nkept is None else row_nkept,
                         self.tab_idx, self.tab_sim, self.tab_mutu, self.tab_n, self.tab_len,
                         self.launches, stats or {})

    def tables_to_host(self, tabs=None, reuse=False):
        """Neighbour tables + BB flags in pinned host memory (reuse=True: module-level buffers that the next
        call overwrites; default: buffers owned by the caller):
        the device -> host read of the stage's result (the reference's collectAsMap, assist.py:121-129)."""
        tabs = tabs or self.tables()
        src = dict(row_flags=tabs.row_flags, tab_len=tabs.tab_len, tab_idx=tabs.tab_idx, tab_sim=tabs.tab_sim,
                   tab_mutu=tabs.tab_mutu, tab_n=tabs.tab_n)
        key = tuple((k, tuple(v.shape), v.dtype) for k, v in src.items())
        if reuse:
            # benchmark fast path: one module-level set of pinned buffers (page-locking is slow), shared by
            # every engine of the same shapes -- the previous result is overwritten
            if key not in _PINNED:
                _PINNED.clear()
                _PINNED[key] = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in src.items()}
            host = _PINNED[key]
        else:
            host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in src.items()}
        for k, v in src.items():
            host[k].copy_(v, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return host

    def emit_pairs(self, rows=None):
        """Every kept directed pair (the return value of baseliner_calculate_sim_pipeline,
        assist.py:66-77), sorted by (i, j): the neighbour-record lists themselves."""
        dev = self.device
        I = self.lay.n_items
        cnt = self.rec_cnt.long()
        if rows is not None:
            keep = torch.zeros(I, dtype=torch.bool, device=dev)
            keep[rows.long()] = True
            cnt = torch.where(keep, cnt, torch.zeros_like(cnt))
        i = torch.repeat_interleave(torch.arange(I, device=dev), cnt)
        first = torch.cumsum(cnt, 0) - cnt
        src = self.rec_ptr[:-1][i] + (torch.arange(i.numel(), device=dev) - first[i])
        r = self.rec[src]
        pack = r[:, 1]
        j = pack & 0xFFFFFFFF
        n = self.rec_n[src]
        mutu = ((pack >> 32) & 0xFFFFFFFF).to(torch.int32)
        sim = r[:, 0].contiguous().view(torch.float64)
        order = torch.argsort(i * I + j)
        i, j, sim, mutu, n = i[order], j[order], sim[order], mutu[order], n[order]
        cnt_i = self.lay.item_stats[:, 3]
        frac = mutu.double() / (cnt_i[i] + cnt_i[j] - n.double())
        label = (self.meta.prefix_code[i] != self.meta.prefix_code[j]).to(torch.int32)
        return dict(i=i, j=j, sim=sim, mutu=mutu, n=n, frac=frac, label=label)
