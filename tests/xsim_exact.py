"""X-SIM reference with a derived error bound, and neighbour tables whose path structure is built on purpose.

Reference.  `exact_rows(plan, starts)` enumerates every path of the given starts from the UNFOLDED edge terms of an
extend.XsimPlan (leg_vals e1, m1, f1, e2, m2, f2; par_vals e, m, f; rs_vals e1, m1, f1, e2, m2, f2) and evaluates
them in extended precision (numpy longdouble, a 64-bit significand: unit roundoff v = 2^-64 on x86-64):

    N_p = sum of the <= 5 edge terms sim*mutu    D_p = sum of their mutu (integers: exact)    c_p = prod of the fracs
    s_p = N_p / D_p  (0 when D_p = 0, extender.py:85-88)      xsim = sum_p s_p c_p / sum_p c_p  (extender.py:198-201)

and per cell n (paths) and A = sum_p (sum_e |e_e|) / D_p * c_p.  The edge terms are taken as given: the sim*mutu
products and the fracs are rounded once in build_plan, and the kernel reads the same fp64 numbers.

Bound.  What the kernel does to a cell of n paths, with u = 2^-53 and gamma_k = k u / (1 - k u):
  * N_p: <= 5 terms, <= 4 additions in any association (the leg, the bridge edge and the right segment are folded
    in different orders by the pair descriptors and the fused lists, DESIGN.md 6.5): |N^ - N| <= gamma_4 sum|e|.
    D_p: a sum of integers below 2^53: exact.  s^ = fl(N^ / D): |s^ - s| <= gamma_5 alpha_p, alpha_p = sum|e| / D_p.
  * c_p: <= 4 products of exact inputs: c^ = c (1 + t), |t| <= gamma_4.
  * num_p = fl(s^ c^): |num_p - s_p c_p| <= (2 gamma_5 + gamma_5^2) a_p <= gamma_10 a_p, a_p = alpha_p c_p
    (|s_p| <= alpha_p).  den_p = c^: |den_p - c_p| <= gamma_4 c_p.
  * the n terms of the numerator and of the denominator are summed with n - 1 additions each, in an order set by
    the runs, chunks and table (any summation tree): the numerator's error is <= gamma_10 A + gamma_(n-1) (1 +
    gamma_10) A <= gamma_(n+9) A, the denominator's relative error rho <= gamma_(n+3) (positive terms).
  * one final division (1 + d), |d| <= u.  With X = SN / SD, SD = sum c_p:
        got - X = (SN (d - rho) + E_N (1 + d)) / (SD (1 + rho))
        |got - X| <= (gamma_(n+10) A / SD + gamma_(n+4) |X|) / (1 - gamma_(n+3))        =: bound
    i.e. (n + 10) u A / sum c + (n + 4) u |X| to first order.  The |X| term grows with n because the denominator
    is itself a sum of n terms; since |X| <= A / sum c, the whole bound is at most (2 n + 14) u A / sum c.
The reference's own error follows from the same derivation with u replaced by v = 2^-64 (every operation above is
one rounding of the extended format; D_p is exact there too): it is at most 2^-11 of the bound, so a kernel value is
accepted when |got - ref| <= bound (1 + 2^-11).
"""
import numpy as np

U = 2.0 ** -53
LD = np.longdouble
REF_SHARE = 2.0 ** -11                          # reference error / bound
assert np.finfo(LD).nmant >= 63, "the X-SIM reference needs an extended long double (64-bit significand)"


def _gamma(k):
    k = np.asarray(k, dtype=np.float64)
    return k * U / (1.0 - k * U)


def cell_bound(n, A, sum_c, x):
    """The bound of the module docstring for cells of n paths (arrays)."""
    return (_gamma(n + 10) * A / sum_c + _gamma(n + 4) * np.abs(x)) / (1.0 - _gamma(n + 3))


def _plan_arrays(plan):
    g = lambda t: t.cpu().numpy()
    p = plan
    return dict(leg_ptr=g(p.leg_ptr), leg_t=g(p.leg_t), leg_jo=g(p.leg_joint_only).astype(bool),
                lv=[g(v) for v in p.leg_vals], par_ptr=g(p.par_ptr), par_s=g(p.par_s),
                par_j=g(p.par_joint).astype(bool), pv=[g(v) for v in p.par_vals], rs_ptr=g(p.rs_ptr),
                rs_end=g(p.rs_end), rv=[g(v) for v in p.rs_vals], start_item=g(p.start_item), ub=g(p.ub))


def enumerate_paths(P, x):
    """Every path of plan start x: (end [n], e [5, n], m [5, n], f [5, n]) in the plan's path order."""
    legs, pars = [], []
    for lg in range(P["leg_ptr"][x], P["leg_ptr"][x + 1]):
        t = P["leg_t"][lg]
        pp = np.arange(P["par_ptr"][t], P["par_ptr"][t + 1])
        if P["leg_jo"][lg]:
            pp = pp[P["par_j"][pp]]
        legs.append(np.full(len(pp), lg)); pars.append(pp)
    lg = np.concatenate(legs) if legs else np.zeros(0, np.int64)
    pp = np.concatenate(pars) if pars else np.zeros(0, np.int64)
    s = P["par_s"][pp]
    a, b = P["rs_ptr"][s], P["rs_ptr"][s + 1]
    ln = b - a
    pair = np.repeat(np.arange(len(pp)), ln)
    r = np.repeat(a, ln) + (np.arange(int(ln.sum())) - np.repeat(np.cumsum(ln) - ln, ln))
    L, Q = lg[pair], pp[pair]
    lv, pv, rv = P["lv"], P["pv"], P["rv"]
    e = np.stack([lv[0][L], lv[3][L], pv[0][Q], rv[0][r], rv[3][r]])
    m = np.stack([lv[1][L], lv[4][L], pv[1][Q], rv[1][r], rv[4][r]])
    f = np.stack([lv[2][L], lv[5][L], pv[2][Q], rv[2][r], rv[5][r]])
    return P["rs_end"][r].astype(np.int64), e, m, f


def cells_of_paths(y, e, m, f):
    """Per distinct end (sorted): reference xsim (fp64 nearest of the extended value, plus its extended value),
    path count n, A, sum c and the bound."""
    D = m.sum(0)
    assert np.all(m == np.round(m)) and np.all(np.abs(D) < 2.0 ** 53)     # mutu sums are exact
    N = e.astype(LD).sum(0)
    c = f.astype(LD).prod(0)
    Dl = D.astype(LD)
    nz = D != 0
    s = np.zeros(len(D), dtype=LD)
    s[nz] = N[nz] / Dl[nz]
    alpha = np.zeros(len(D))
    alpha[nz] = np.abs(e[:, nz]).sum(0) / D[nz]
    o = np.argsort(y, kind="stable")
    uy, first, n = np.unique(y[o], return_index=True, return_counts=True)
    SN = np.add.reduceat((s * c)[o], first) if len(o) else np.zeros(0, LD)
    SD = np.add.reduceat(c[o], first) if len(o) else np.zeros(0, LD)
    X = SN / SD
    cd = c.astype(np.float64)
    A = np.add.reduceat((alpha * cd)[o], first) if len(o) else np.zeros(0)
    sc = SD.astype(np.float64)
    x64 = X.astype(np.float64)
    return dict(end=uy, x=x64, x_ld=X, n=n, A=A, sum_c=sc, bound=cell_bound(n, A, sc, x64))


def exact_rows(plan, starts):
    """{plan start index: cells_of_paths(...) of its paths, plus 'paths'}"""
    P = _plan_arrays(plan)
    out = {}
    for x in starts:
        y, e, m, f = enumerate_paths(P, int(x))
        row = cells_of_paths(y, e, m, f)
        row["paths"] = len(y)
        out[int(x)] = row
    return out


def err_ratio(got, row):
    """|got - reference| / bound per cell (the reference's own error is <= REF_SHARE of the bound)."""
    d = np.abs((np.asarray(got, dtype=LD) - row["x_ld"]).astype(np.float64))
    return np.where(row["bound"] > 0, d / np.where(row["bound"] > 0, row["bound"], 1.0), np.where(d == 0, 0.0, np.inf))


def ref_top(row, m):
    """The reference's top-m of a row: |xsim| desc, then the smaller end (indices into the row)."""
    return np.lexsort((row["end"], -np.abs(row["x"])))[:m]


def check_top(te, tx, tl, row, m):
    """A kernel top-m row (te, tx, tl) against the reference: same length, and where a position names another end
    than the reference's, the two exact values lie within the sum of their bounds (a near-tie in exact arithmetic);
    every listed value is within its own bound.  Returns the number of positions that differ."""
    want = ref_top(row, m)
    assert tl == len(want), (tl, len(want))
    pos = np.searchsorted(row["end"], te[:tl])
    assert np.all(row["end"][pos] == te[:tl])
    assert np.all(err_ratio(tx[:tl], {k: row[k][pos] for k in ("x_ld", "bound")}) <= 1.0 + REF_SHARE)
    diff = np.flatnonzero(te[:tl] != row["end"][want])
    gap = np.abs(np.abs(row["x"][pos[diff]]) - np.abs(row["x"][want[diff]]))
    assert np.all(gap <= (row["bound"][pos[diff]] + row["bound"][want[diff]]) * (1.0 + REF_SHARE)), \
        "top-%d position(s) %s name another end than the reference outside the rounding bound" % (m, diff.tolist())
    return len(diff)


# ------------------------------------------------------------------------------------------------------------
# neighbour tables built on purpose
# ------------------------------------------------------------------------------------------------------------
class Tables:
    """The fields extend.build_plan reads, plus the item counts and domain flags it takes."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


PI_MULT, XGOLD2 = 0x9E3779B1, 0x85EBCA6B


def pi_tile(y, gb):
    """Hash tile of end y among 2^gb (extend.PI_MULT)."""
    return ((np.asarray(y, dtype=np.int64) * PI_MULT) & 0xFFFFFFFF) >> (32 - gb)


def cta_owner(y):
    """Owner warp (= table region) of end y in the CTA kernel (csrc/xsim.cu XGOLD2, 3 owner bits)."""
    return ((np.asarray(y, dtype=np.int64) * XGOLD2) & 0xFFFFFFFF) >> 29


class Graph:
    """Neighbour lists written item by item.  An edge's (sim, mutu, n) is a function of the unordered pair, so the
    tables are symmetric in value (sim(a, b) == sim(b, a) bit for bit) as the engine's are, whichever rows list it.
      BB item:  slot 0 = BB_BB (bridge items of the other domain), slot 1 = BB_NB
      NB item:  slot 0 = NB_BB (what it attaches to), slot 1 = NB_NN
    Default edge values: sim uniform in [-1, 1] (mixed signs, so N_p cancels), mutu in [1, 30], n in [mutu, 35],
    every item counted 40 times (frac = mutu / (80 - n) in (0, 1])."""

    def __init__(self, seed, count=40, sim=None, mutu=None):
        self.rng = np.random.default_rng(seed)
        self.dom, self.bb, self.rows, self.edges = [], [], [], {}
        self.count, self.sim, self.mutu = count, sim, mutu

    def items(self, n, dom, bb=False):
        i0 = len(self.dom)
        self.dom += [dom] * n; self.bb += [bb] * n; self.rows += [([], []) for _ in range(n)]
        return list(range(i0, i0 + n))

    def item(self, dom, bb=False):
        return self.items(1, dom, bb)[0]

    def items_where(self, n, dom, pred):
        """n new NB items (ends) whose index satisfies pred; the items skipped on the way are created too."""
        got = []
        while len(got) < n:
            i = self.item(dom)
            if pred(i):
                got.append(i)
        return got

    def lst(self, i, slot, nbrs):
        self.rows[i][slot].extend(int(j) for j in nbrs)

    def set_edge(self, a, b, sim, mutu=None, n=None):
        key = (min(a, b), max(a, b))
        mutu = self.mutu if mutu is None else mutu
        self.edges[key] = (float(sim), int(mutu), int(mutu if n is None else n))

    def edge(self, a, b):
        key = (min(a, b), max(a, b))
        if key not in self.edges:
            if self.sim is not None:
                self.edges[key] = (float(self.sim), int(self.mutu), int(self.mutu))
            else:
                mu = int(self.rng.integers(1, 31))
                self.edges[key] = (float(self.rng.uniform(-1, 1)), mu, int(self.rng.integers(mu, 36)))
        return self.edges[key]

    def tables(self, device="cpu"):
        import torch
        I = len(self.dom)
        k = max(1, max(len(l) for r in self.rows for l in r))
        idx = np.full((I, 2, k), -1, np.int32); sim = np.zeros((I, 2, k)); mutu = np.zeros((I, 2, k), np.int32)
        nn = np.zeros((I, 2, k), np.int32); ln = np.zeros((I, 2), np.int32)
        for i, r in enumerate(self.rows):
            for slot in range(2):
                assert len(set(r[slot])) == len(r[slot]) and i not in r[slot], (i, slot)
                for q, j in enumerate(r[slot]):
                    s_, m_, n_ = self.edge(i, j)
                    idx[i, slot, q] = j; sim[i, slot, q] = s_; mutu[i, slot, q] = m_; nn[i, slot, q] = n_
                ln[i, slot] = len(r[slot])
        T = lambda a, dt: torch.as_tensor(a, dtype=dt, device=device)
        dom = np.array(self.dom)
        return Tables(n_items=I, k=k, row_flags=T(np.array(self.bb, np.uint8), torch.uint8),
                      tab_idx=T(idx, torch.int32), tab_sim=T(sim, torch.float64), tab_mutu=T(mutu, torch.int32),
                      tab_n=T(nn, torch.int32), tab_len=T(ln, torch.int32),
                      item_count=T(np.full(I, self.count), torch.int32), has_S=T(dom == "S", torch.bool),
                      has_T=T(dom == "T", torch.bool))

    # ---- building blocks ------------------------------------------------------------------------------
    def source(self, ends_of_attach):
        """A bridge source s (BB, domain S) with one attach item n per entry; n lists s (NB_BB) and the given ends
        (NB_NN), so right(s) = [s] + per n: [n] + its ends."""
        s = self.item("S", bb=True)
        for ends in ends_of_attach:
            n = self.item("S")
            self.lst(n, 0, [s]); self.lst(n, 1, ends)
        return s

    def bridge(self, t, sources, joint=False):
        """Bridge pairs (t, s): every s lists t (BB_BB); joint: t lists s too, and t gets an attach item if it has
        none, so its attach items start joint-only legs."""
        for s in sources:
            self.lst(s, 0, [t])
        if joint:
            self.lst(t, 0, sources)


def build_plan(tabs):
    from xmap_b200 import extend as X
    return X.build_plan(tabs, tabs.item_count, tabs.has_S, tabs.has_T)


# ---- the cases -------------------------------------------------------------------------------------------------
PARTNER_COUNTS = (31, 32, 33, 255, 256, 257)      # (leg, partner) pairs of a start: warp batch 32, CTA macro-batch 256
LIST_LENGTHS = (2, 3, 31, 32, 33, 64, 65)         # right-segment lists: chunk size 32
RUN_LENGTHS = (1, 31, 32, 33, 100)                # equal ends in a row in a fused bridge list


def case_batches(seed=11):
    """Bridge targets with 31, 32, 33, 255, 256 and 257 partners (each its own start: the type-0 leg walks every
    partner), over 300 sources whose right-segment lists are 2, 3, 31, 32, 33, 64 and 65 entries long."""
    G = Graph(seed)
    ends = G.items(400, "S")
    srcs = [G.source([G.rng.choice(ends, L - 2, replace=False)]) for L in np.resize(LIST_LENGTHS, 300)]
    for P in PARTNER_COUNTS:
        t = G.item("T", bb=True)
        G.bridge(t, sorted(G.rng.choice(srcs, P, replace=False).tolist()))
    return G


def case_runs(seed=12):
    """One bridge target t with 100 joint partners whose right segments share ends: in the fused list B(t) one end
    repeats 100 times, others 33, 32, 31 and 1 times, the rest a few times.  t's attach item a starts a joint-only
    leg of type 1, a's neighbours x1, x2 legs of type 2; t itself walks the unfused pair lists."""
    G = Graph(seed)
    t = G.item("T", bb=True)
    a = G.item("T")
    xs = G.items(2, "T")
    G.lst(a, 0, [t]); G.lst(a, 1, xs)
    shared = dict((r, G.item("S")) for r in RUN_LENGTHS)
    filler = G.items(150, "S")
    srcs = []
    for i in range(100):
        ends = [y for r, y in shared.items() if i < r] + G.rng.choice(filler, 3, replace=False).tolist()
        srcs.append(G.source([ends]))
    G.bridge(t, srcs, joint=True)
    return G


def _one_partner_start(G, ends_fn):
    """A start t whose only partner s has one attach n: right(s) = [s, n] + ends_fn(s, n)."""
    t = G.item("T", bb=True)
    s = G.item("S", bb=True)
    n = G.item("S")
    G.lst(n, 0, [s]); G.lst(n, 1, ends_fn(s, n))
    G.bridge(t, [s])
    return t


WARP_FILL = (55, 56, 57)           # distinct ends of one pass around 7/8 of a 64-cell warp table (56)
SPLIT_TILES = (6, 7)               # sibling tiles at gb = 4 holding 50 and 10 ends


def case_pressure(seed=13):
    """Starts with 55, 56 and 57 distinct ends (7/8 of the 64-cell warp table is 56); starts with 55, 56 and 57 ends
    in CTA owner region 0 (7/8 of a 64-cell region at cells_lg = 9) and 5 in region 1; a start with 50 ends in hash
    tile 6 and 10 in tile 7 (of 16), so that a 64-cell table fits only after the splits reach single tiles."""
    G = Graph(seed)
    for k in WARP_FILL:
        _one_partner_start(G, lambda s, n, k=k: G.items(k - 2, "S"))
    for k in WARP_FILL:
        def ends(s, n, k=k):
            c0 = int(cta_owner(s) == 0) + int(cta_owner(n) == 0)
            c1 = int(cta_owner(s) == 1) + int(cta_owner(n) == 1)
            return (G.items_where(k - c0, "S", lambda i: cta_owner(i) == 0) +
                    G.items_where(5 - c1, "S", lambda i: cta_owner(i) == 1))
        _one_partner_start(G, ends)

    def tiles(s, n):
        ca = sum(int(pi_tile(i, 4) == SPLIT_TILES[0]) for i in (s, n))
        cb = sum(int(pi_tile(i, 4) == SPLIT_TILES[1]) for i in (s, n))
        return (G.items_where(50 - ca, "S", lambda i: pi_tile(i, 4) == SPLIT_TILES[0]) +
                G.items_where(10 - cb, "S", lambda i: pi_tile(i, 4) == SPLIT_TILES[1]))
    _one_partner_start(G, tiles)
    return G


def case_overflow(seed=14):
    """One start with 118 ends in hash tile 3 (of 16) besides s and n: more than 7/8 of a 128-cell table."""
    G = Graph(seed)
    _one_partner_start(G, lambda s, n: G.items_where(118, "S", lambda i: pi_tile(i, 4) == 3))
    return G


def case_signs(seed=15):
    """Exact zeros: start t0 reaches each of 5 ends z by two paths whose edges are v and -v with equal mutu and
    frac, so xsim(z) = 0.  Besides, bridge targets over random mixed-sign edges (N_p cancels)."""
    G = Graph(seed)
    t0 = G.item("T", bb=True)
    sp, sm = G.item("S", bb=True), G.item("S", bb=True)
    npl, nmi = G.item("S"), G.item("S")
    Z = G.items(5, "S")
    G.lst(npl, 0, [sp]); G.lst(npl, 1, Z); G.lst(nmi, 0, [sm]); G.lst(nmi, 1, Z)
    G.bridge(t0, [sp, sm])
    G.set_edge(t0, sp, 0.3, 7, 9); G.set_edge(t0, sm, -0.3, 7, 9)
    G.set_edge(sp, npl, 0.55, 4, 6); G.set_edge(sm, nmi, -0.55, 4, 6)
    for z in Z:
        v, mu = float(G.rng.uniform(-1, 1)), int(G.rng.integers(1, 31))
        G.set_edge(npl, z, v, mu, mu + 2); G.set_edge(nmi, z, -v, mu, mu + 2)
    ends = G.items(60, "S")
    srcs = [G.source([G.rng.choice(ends, int(L), replace=False) for L in G.rng.integers(0, 12, size=2)])
            for _ in range(20)]
    for _ in range(6):
        t = G.item("T", bb=True)
        G.bridge(t, sorted(G.rng.choice(srcs, int(G.rng.integers(1, 15)), replace=False).tolist()))
    return G


TIE_ENDS = (42, 300, 300, 600)      # distinct ends of the tie starts (the second 300 at -0.5)


def case_ties(seed=16):
    """Every edge 0.5 (one component -0.5), mutu = n = item count = 7, so frac = 1 and every cell is exactly
    +-0.5: the top-m is decided by the end alone.  Starts with 42, 300, 300 and 600 distinct ends."""
    G = Graph(seed, count=7, sim=0.5, mutu=7)
    for q, E in enumerate(TIE_ENDS):
        t = G.item("T", bb=True)
        nsrc = max(2, E // 30)
        srcs = []
        for i in range(nsrc):
            ln = E // nsrc - 2 + (E % nsrc if i == 0 else 0)
            s = G.item("S", bb=True)
            n = G.item("S")
            ys = G.items(ln, "S")
            G.lst(n, 0, [s]); G.lst(n, 1, ys)
            srcs.append(s)
            if q == 2:
                G.set_edge(t, s, -0.5); G.set_edge(s, n, -0.5)
                for y in ys:
                    G.set_edge(n, y, -0.5)
        G.bridge(t, srcs)
    return G


DESIGNED = dict(batches=case_batches, runs=case_runs, pressure=case_pressure, signs=case_signs, ties=case_ties)
