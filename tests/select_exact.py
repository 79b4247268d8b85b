"""Exact reference of the similarity stage's top-k selection (xmap_sim_select, include/xmap_b200.h) computed from
the neighbour records themselves, a classifier of the path every (row, list) takes through the two select kernels of
x-map_b200/csrc/sim.cu, and record lists designed to drive those paths.

Order: the bits of |sim| descending, then the smaller neighbour index -- the kernels' better() on integer keys, so no
float comparison can blur a tie.  The reference refuses NaN and +-0.0 similarities (the accumulate filter never emits
them) and repeated (row, neighbour) records.  It does not depend on the order of the records within a row.

Lists (list_bits() of sim.cu):
  BB row: slot 0 = neighbours j with ((contains[j] >> dom_code[i]) & 1) == 0, slot 1 = the others;
  NB row: slot 0 = neighbours with bb[j], slot 1 = every neighbour.
"""
import numpy as np

SELECT_LONG = 8192        # XMAP_SELECT_LONG: longer lists go to select_cta_kernel
SEL_DIRECT = 64           # select_warp_kernel: lists up to this long skip the histogram
SEL_BUF = 192             # survivor buffer of select_warp_kernel, per list
SIM_BINS = 256
SAMPLE_FROM = 1024        # longer lists build the histogram from every 4th block of 128 records only
CTA_STEP = 256 * 4        # records per step of select_cta_kernel (FIN_THREADS * SEL_UNROLL)
CTA_FLUSH = 12 * 256 - 2 * CTA_STEP - 2 * 64     # the candidate buffer is flushed when it holds more than this
ABS_MASK = np.uint64(0x7FFF_FFFF_FFFF_FFFF)
PATHS = ("empty", "count32", "direct64", "hist_rank", "hist_rounds", "overflow", "cta")
MIN_PER_PATH = 100        # (row, list) cases of every path but "empty" at every k of KS in designed_cases()
FILL = dict(idx=-1, sim_bits=0, mutu=0, n=0)   # SimEngine's initial table contents


def abs_key(sim):
    return np.ascontiguousarray(sim, dtype=np.float64).view(np.uint64) & ABS_MASK


def list_bits(i, j, bb, dom_code, contains):
    """Per record: bit 0 set if it belongs to list 0 of its row, bit 1 if to list 1."""
    i, j = np.asarray(i, np.int64), np.asarray(j, np.int64)
    bb = np.asarray(bb).astype(bool)
    same = ((np.asarray(contains)[j].astype(np.int64) >> np.asarray(dom_code)[i].astype(np.int64)) & 1) == 1
    return np.where(bb[i], np.where(same, 2, 1), 2 | bb[j].astype(np.int64)).astype(np.uint8)


class Ranked:
    """Every record's rank within each list of its row; tables(k) cuts them at any k."""

    def __init__(self, i, j, sim, mutu, n, bb, dom_code, contains, n_rows=None):
        i, j = np.asarray(i, np.int64), np.asarray(j, np.int64)
        sim = np.ascontiguousarray(sim, dtype=np.float64)
        assert not np.isnan(sim).any(), "NaN similarity"
        key = abs_key(sim)
        assert (key != 0).all(), "+-0.0 similarity"
        self.n_rows = len(bb) if n_rows is None else int(n_rows)
        assert len(i) == 0 or (i.min() >= 0 and i.max() < self.n_rows)
        order = np.lexsort((j, ABS_MASK - key, i))
        io, jo = i[order], j[order]
        assert not ((io[1:] == io[:-1]) & (jo[1:] == jo[:-1])).any(), "repeated (row, neighbour) record"
        lb = list_bits(i, j, bb, dom_code, contains)[order]
        self.j, self.sim, self.mutu, self.n = j, sim, np.asarray(mutu), np.asarray(n)
        self.lists = []
        self.count = np.zeros((self.n_rows, 2), np.int64)
        for lst in range(2):
            sel = order[((lb >> lst) & 1) == 1]
            rows = i[sel]
            rank = np.arange(len(sel)) - np.searchsorted(rows, rows, side="left")
            self.lists.append((sel, rows, rank))
            self.count[:, lst] = np.bincount(rows, minlength=self.n_rows)

    def tables(self, k, fill=FILL):
        R = self.n_rows
        idx = np.full((R, 2, k), fill["idx"], np.int32)
        sim_bits = np.full((R, 2, k), fill["sim_bits"], np.int64)
        mutu = np.full((R, 2, k), fill["mutu"], np.int32)
        n = np.full((R, 2, k), fill["n"], np.int32)
        length = np.minimum(self.count, k).astype(np.int32)
        for lst, (sel, rows, rank) in enumerate(self.lists):
            m = rank < k
            s, r, p = sel[m], rows[m], rank[m]
            idx[r, lst, p] = self.j[s]
            sim_bits[r, lst, p] = self.sim[s].view(np.int64)
            mutu[r, lst, p] = self.mutu[s]
            n[r, lst, p] = self.n[s]
        return dict(tab_len=length, tab_idx=idx, tab_sim=sim_bits.view(np.float64), tab_mutu=mutu, tab_n=n)


def select_exact(i, j, sim, mutu, n, bb, dom_code, contains, k, n_rows=None):
    """The tables xmap_sim_select must produce from these records: tab_len [R, 2], tab_idx / tab_sim / tab_mutu /
    tab_n [R, 2, k] (R = len(bb) unless n_rows is given); entries past tab_len hold SimEngine's initial values."""
    return Ranked(i, j, sim, mutu, n, bb, dom_code, contains, n_rows).tables(k)


def from_engine(eng, meta, rows=None, pairs=None):
    """select_exact over the records of a finished SimEngine (eng.emit_pairs(rows), or `pairs` when the caller
    already has them) with the device BB flags; meta holds the host per-item codes."""
    p = eng.emit_pairs(rows) if pairs is None else pairs
    host = lambda t: t.cpu().numpy()
    return select_exact(host(p["i"]), host(p["j"]), host(p["sim"]), host(p["mutu"]), host(p["n"]), host(eng.bb),
                        np.asarray(meta["dom_code"]), np.asarray(meta["contains"]), eng.k, n_rows=eng.lay.n_items)


def engine_records(eng, rows):
    """(i, j, sim) of the records of `rows` in the order the select kernels read them (emit_pairs sorts them)."""
    import torch
    rows = torch.as_tensor(rows, device=eng.device).long()
    cnt = eng.rec_cnt.long()[rows]
    i = torch.repeat_interleave(rows, cnt)
    src = torch.repeat_interleave(eng.rec_ptr[rows], cnt) + torch.arange(i.numel(), device=eng.device) - \
        torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    r = eng.rec[src]
    return i.cpu().numpy(), (r[:, 1] & 0xFFFFFFFF).cpu().numpy(), r[:, 0].contiguous().view(torch.float64).cpu().numpy()


def table_mismatches(ref, got, rows=None):
    """Rows (of `rows`, default all) whose tab_len or any entry below tab_len differs from ref, bit for bit."""
    rows = np.arange(len(ref["tab_len"])) if rows is None else np.asarray(rows, np.int64)
    L = ref["tab_len"][rows]
    bad = (np.asarray(got["tab_len"])[rows] != L).any(axis=1)
    k = ref["tab_idx"].shape[2]
    valid = np.arange(k)[None, None, :] < L[:, :, None]
    for name in ("tab_idx", "tab_sim", "tab_mutu", "tab_n"):
        a, b = ref[name][rows], np.asarray(got[name])[rows]
        if name == "tab_sim":
            a, b = a.view(np.int64), b.view(np.int64)
        bad |= ((a != b) & valid).any(axis=(1, 2))
    return rows[bad]


def assert_engine_selection(eng, meta, rows=None, pairs=None):
    """The engine's tables of `rows` (default every row) equal select_exact over the engine's own records."""
    ref = from_engine(eng, meta, rows, pairs)
    got = {name: getattr(eng, name).cpu().numpy() for name in ("tab_len", "tab_idx", "tab_sim", "tab_mutu", "tab_n")}
    rows = None if rows is None else np.asarray(rows.cpu() if hasattr(rows, "cpu") else rows, np.int64)
    bad = table_mismatches(ref, got, rows)
    if len(bad):
        r = int(bad[0])
        raise AssertionError("%d rows' neighbour tables differ from the exact selection of their records; row %d: "
                             "len %s vs %s, idx %s vs %s" % (len(bad), r, got["tab_len"][r].tolist(),
                                                            ref["tab_len"][r].tolist(), got["tab_idx"][r].tolist(),
                                                            ref["tab_idx"][r].tolist()))
    return len(ref["tab_len"]) if rows is None else len(rows)


# --------------------------------------------------------------------------
# Which path each (row, list) takes
# --------------------------------------------------------------------------
def sim_bin(key):
    """sim_bin() of common.cuh: 16 bins per octave from 2^-16; smaller keys share bin 0, keys >= 1 the top bin."""
    return np.clip((key >> np.uint64(48)).astype(np.int64) - ((1023 - 16) << 4), 0, SIM_BINS - 1)


def _warp_path(key, member, k):
    """select_warp_kernel's path for one list of a row with 64 < m <= SELECT_LONG records (key, member in list order)."""
    m = len(key)
    pos = np.arange(m)
    sampled = (pos // 128) % 4 == 0 if m > SAMPLE_FROM else np.ones(m, bool)
    bins = sim_bin(key)
    s = member & sampled
    bstar = 0
    if s.sum() >= k:          # fewer sampled members than k keep everything
        suffix = np.cumsum(np.bincount(bins[s], minlength=SIM_BINS)[::-1])[::-1]
        bstar = int(np.nonzero(suffix >= k)[0].max())
    surv = int((member & (bins >= bstar)).sum())
    return "hist_rank" if surv <= 64 else "hist_rounds" if surv <= SEL_BUF else "overflow"


def _cta_flushes(key, lb, k):
    """How many times select_cta_kernel runs its tournament on one row (the flushes of the candidate buffer and the
    final one): the running thresholds are the k-th best key of each list over the records before the flush."""
    thr = [np.uint64(0), np.uint64(0)]
    tops = [np.zeros(0, np.uint64), np.zeros(0, np.uint64)]
    since = [[], []]
    ncand = flushes = 0
    for base in range(0, len(key), CTA_STEP):
        if ncand > CTA_FLUSH:
            flushes += 1
            ncand = 0
            for lst in range(2):
                tops[lst] = np.sort(np.concatenate([tops[lst]] + since[lst]))[-k:]
                since[lst] = []
                thr[lst] = tops[lst][0] if len(tops[lst]) == k else np.uint64(0)
        kk, bits = key[base:base + CTA_STEP], lb[base:base + CTA_STEP]
        floor = min(thr)
        for lst in range(2):
            take = (((bits >> lst) & 1) == 1) & (kk >= floor) & ((thr[lst] == 0) | (kk >= thr[lst]))
            ncand += int(take.sum())
            since[lst].append(kk[take])
    return flushes + 1


def classify(i, j, sim, bb, dom_code, contains, k, n_rows=None):
    """Path of every (row, list) when the rows' records are stored in the given order: labels [R, 2] (indices into
    PATHS) and, for the rows of the CTA kernel, the number of tournaments it runs ({row: count})."""
    i = np.asarray(i, np.int64)
    R = len(bb) if n_rows is None else int(n_rows)
    key = abs_key(sim)
    lb = list_bits(i, j, bb, dom_code, contains)
    o = np.argsort(i, kind="stable")
    ptr = np.searchsorted(i[o], np.arange(R + 1))
    labels = np.zeros((R, 2), np.int64)
    flushes = {}
    for r in range(R):
        seg = o[ptr[r]:ptr[r + 1]]
        m = len(seg)
        if m == 0:
            path = ("empty", "empty")
        elif m <= 32:
            path = ("count32", "count32")
        elif m <= SEL_DIRECT:
            path = ("direct64", "direct64")
        elif m > SELECT_LONG:
            path = ("cta", "cta")
            flushes[r] = _cta_flushes(key[seg], lb[seg], k)
        else:
            path = tuple(_warp_path(key[seg], ((lb[seg] >> lst) & 1) == 1, k) for lst in range(2))
        labels[r] = [PATHS.index(p) for p in path]
    return labels, flushes


def path_counts(labels):
    return {p: int((labels == q).sum()) for q, p in enumerate(PATHS)}


# --------------------------------------------------------------------------
# Designed record lists
# --------------------------------------------------------------------------
ITEM_BITS = 24                        # the record layout's item limit: indices below 2^24
N_ITEMS = 1 << ITEM_BITS
ROW_SPACE = 1 << 16                   # rows are items [0, R); neighbours are drawn from [ROW_SPACE, N_ITEMS)
BIG = (1 << 31) - 1
LENGTHS = (0, 1, 2, 31, 32, 33, 63, 64, 65, 191, 192, 193, 1023, 1024, 1025, 8191, 8192, 8193)
KS = (1, 2, 10, 31, 32, 33, 63, 64)
# row kind -> (row is BB, share of its records in list 0); list 0 of a BB row = other-domain neighbours,
# of an NB row = BB neighbours (so an NB row with share 0 has no BB neighbour)
KINDS = dict(bb=(True, 0.5), bb_same=(True, 0.0), nb_some=(False, 0.3), nb_all=(False, 1.0), nb_none=(False, 0.0))


def item_codes():
    """Per-item codes of the designed cases, a function of the index's low bits: contains = bits 0-2 (several
    labels per item), bb = bit 3.  Rows override bb and dom_code."""
    x = np.arange(N_ITEMS, dtype=np.int64)
    return (x & 7).astype(np.uint8), ((x >> 3) & 1).astype(np.uint8), np.zeros(N_ITEMS, np.uint8)


def _in_list0(x, row_bb, dom):
    return ((x & 7) >> dom) & 1 == 0 if row_bb else (x >> 3) & 1 == 1


def _draw(rng, in0, row_bb, dom):
    """Distinct neighbour indices whose list-0 membership is in0 (bool per record)."""
    m = len(in0)
    props = np.arange(16)
    ok0 = props[_in_list0(props, row_bb, dom)]
    ok1 = props[~_in_list0(props, row_bb, dom)]
    x = np.zeros(m, np.int64)
    need = np.ones(m, bool)
    while need.any():
        q = int(need.sum())
        hi = rng.integers(ROW_SPACE >> 4, (N_ITEMS >> 4), q)
        p = np.where(in0[need], rng.choice(ok0, q), rng.choice(ok1, q))
        x[need] = (hi << 4) | p
        _, first = np.unique(x, return_index=True)
        need = np.ones(m, bool)
        need[first] = False
    return x


def _with_low_bits(v, rng, bits):
    b = np.asarray(v, np.float64).view(np.uint64)
    return ((b & ~np.uint64((1 << bits) - 1)) | rng.integers(0, 1 << bits, len(b)).astype(np.uint64)).view(np.float64)


EDGE_VALUES = np.array([2.0 ** -16, np.nextafter(2.0 ** -16, 0), np.nextafter(2.0 ** -16, 1), 2.0 ** -17,
                        5e-324, 1e-310, np.nextafter(2.2250738585072014e-308, 0), 2.2250738585072014e-308,
                        1.0, np.nextafter(1.0, 2), np.nextafter(1.0, 0), 2.0, 3.5, 1e10, 0.5, 0.5 + 2 ** -53])


def magnitudes(kind, m, rng, k=None):
    """|sim| of a list of m records in list order (all > 0)."""
    if kind == "distinct":
        return 1.0 - rng.random(m)
    if kind == "equal":
        return np.full(m, 1.0 / 7)
    if kind == "cut_ties":        # k - 1 distinct large values, then the rest tied at the k-th value
        return np.concatenate([0.9 + 0.09 * rng.random(min(m, k - 1)), np.full(max(0, m - k + 1), 0.5)])
    if kind == "sign_pairs":      # +s and -s on two neighbours (signs are set by the caller)
        return np.repeat(1.0 - rng.random((m + 1) // 2), 2)[:m]
    if kind == "one_bin":         # one 1/16-octave bin, keys differing in the low 16 mantissa bits only
        return _with_low_bits(np.full(m, 0.7), rng, 16)
    if kind == "edges":
        return rng.choice(EDGE_VALUES, m)
    if kind == "tiny":            # the whole list below 2^-16: one histogram bin
        return np.exp2(-16.0 - 1000 * (1.0 - rng.random(m))).clip(5e-324)
    if kind == "ascending":
        return np.sort(1.0 - rng.random(m))
    if kind == "descending":
        return np.sort(1.0 - rng.random(m))[::-1].copy()
    if kind == "level_ties":      # ascending levels of 700 tied records: ties at the running threshold of every flush
        return 1e-3 * (1 + np.arange(m) // 700)
    raise ValueError(kind)


class Design:
    """Rows of designed lists; each list is stored three times: as built, reversed and randomly permuted."""

    def __init__(self, seed=7):
        self.rng = np.random.default_rng(seed)
        self.contains, self.bb, self.dom_code = item_codes()
        self.parts = []
        self.names = []           # per row: (kind, magnitudes, length, order)

    def add(self, kind, mags, m, k=None, in0=None, signs=None, vals=None):
        rng = self.rng
        row_bb, share = KINDS[kind]
        dom = int(rng.integers(0, 3))
        v = magnitudes(mags, m, rng, k) if vals is None else vals
        if in0 is None:
            in0 = rng.random(m) < share
        if signs is None:
            signs = np.where(np.arange(m) % 2 == 1, -1.0, 1.0) if mags == "sign_pairs" else rng.choice([-1.0, 1.0], m)
        j = _draw(rng, in0, row_bb, dom)
        mutu = rng.integers(1, BIG, m, endpoint=True)
        n = rng.integers(1, BIG, m, endpoint=True)
        if m and mags == "distinct":
            # carried fields at their limits on the best record: the largest index the layout allows where it
            # has the list-0 membership of that record, and mutu = n = 2^31 - 1
            b = int(np.argmax(v))
            if bool(_in_list0(N_ITEMS - 1, row_bb, dom)) == bool(in0[b]) and (j != N_ITEMS - 1).all():
                j[b] = N_ITEMS - 1
            mutu[b] = n[b] = BIG
        sim = signs * v
        perm = rng.permutation(m)
        for order, o in (("built", np.arange(m)), ("reversed", np.arange(m)[::-1]), ("permuted", perm)):
            r = len(self.names)
            self.bb[r] = 1 if row_bb else 0
            self.dom_code[r] = dom
            self.parts.append((np.full(m, r), j[o], sim[o], mutu[o], n[o]))
            self.names.append((kind, mags, m, order))

    def records(self):
        cat = lambda q, dt: np.concatenate([p[q] for p in self.parts]).astype(dt)
        return dict(i=cat(0, np.int64), j=cat(1, np.int64), sim=cat(2, np.float64), mutu=cat(3, np.int64),
                    n=cat(4, np.int64), bb=self.bb, dom_code=self.dom_code, contains=self.contains,
                    n_rows=len(self.names), names=self.names)


def sampled_mask(m):
    return (np.arange(m) // 128) % 4 == 0


def designed_cases(seed=7, long_rows=True):
    """Every length x row kind x magnitude pattern, the k-dependent tie cuts, the sampling and CTA adversaries,
    and (long_rows) lists of 50 000 and 200 000 records."""
    D = Design(seed)
    base = ("distinct", "equal", "sign_pairs", "one_bin", "edges", "tiny")
    for m in LENGTHS:
        for kind in KINDS:
            for mags in base:
                D.add(kind, mags, m)
        for k in KS:
            for kind in ("bb", "nb_some"):
                if m >= k:
                    D.add(kind, "cut_ties", m, k)
    rng = D.rng
    for m in (1025, 1500, 4097, 8191, 8192):
        s = sampled_mask(m)
        for kind in ("bb", "nb_some"):
            # the true top-64 only in blocks the histogram does not sample
            v = 0.05 * (1.0 - rng.random(m))
            v[rng.choice(np.nonzero(~s)[0], 64, replace=False)] = 0.5 + 0.4 * rng.random(64)
            D.add(kind, "unsampled_top", m, vals=v)
            # list 0: three records in the sample (the best ones), 150 outside it
            in0 = np.zeros(m, bool)
            top3 = rng.choice(np.nonzero(s)[0], 3, replace=False)
            in0[top3] = True
            in0[rng.choice(np.nonzero(~s)[0], 150, replace=False)] = True
            v = 0.8 * (1.0 - rng.random(m))
            v[top3] = 0.95 + 0.04 * rng.random(3)
            D.add(kind, "list0_unsampled", m, in0=in0, vals=v)
            # list 0 entirely outside the sample
            in0 = np.zeros(m, bool)
            in0[rng.choice(np.nonzero(~s)[0], 120, replace=False)] = True
            D.add(kind, "list0_unsampled", m, in0=in0, vals=1.0 - rng.random(m))
    for m in (8193, 12000):
        for kind in ("bb", "nb_some", "nb_all"):
            for mags in ("ascending", "descending", "level_ties"):
                D.add(kind, mags, m)
    if long_rows:
        for kind in ("bb", "nb_some"):
            for mags in ("ascending", "descending", "level_ties", "distinct"):
                D.add(kind, mags, 50000)
            for k in (10, 64):
                D.add(kind, "cut_ties", 50000, k)
        D.add("nb_some", "distinct", 200000)
    return D.records()
