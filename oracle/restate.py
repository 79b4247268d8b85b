"""Array-level CPU restatement of the reference hot path -- the scalable oracle.

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module; the product
package never does and has no CPU fallback.

oracle/harness.py executes the reference itself but is only feasible up to
~1e5 ratings (and a few thousand items for the extender, SURVEY.md App. B.4).
This module restates the same arithmetic over integer-encoded arrays with
numpy/scipy so that it (a) can be pinned against the harness on small inputs
(tests/test_oracle.py does that on every golden case) and (b) finishes in
seconds on inputs large enough to exercise the CUDA kernels.  It needs nothing
from /root/reference at run time, so it travels to the GPU box.

Encoding convention shared with the product: users and items are numbered by
the rank of their id string in sorted order ("canonical index", SURVEY.md
App. A.6), so "ties resolve to the smaller index" means the same thing on both
sides.  Per item the caller supplies
  prefix_code[i]   dictionary code of iid[:2]      (baselinerSim.py:189-191)
  dom_code[i]      dictionary code of iid[-2:]     (extender.py:29)
  contains[i]      bit d set iff label d is a substring of iid (extender.py:32,34)
  has_S[i], has_T[i]  "S:" in iid / "T:" in iid    (extender.py:68,79,174-175)
"""
import numpy as np
import scipy.sparse as sp


# --------------------------------------------------------------------------
# Similarity  (baselinerSim.py:17-216, SURVEY.md App. A.2)
# --------------------------------------------------------------------------
def user_item_stats(user, item, rating, n_users, n_items):
    """baselinerSim.py:17-38 and :40-82.  Inputs must be sorted user-major so
    the per-item sums run in ascending user order like the reference's
    combineByKey over the flatMap of user records."""
    r = rating.astype(np.float64)
    d_u = np.bincount(user, minlength=n_users).astype(np.float64)
    s_u = np.bincount(user, weights=r, minlength=n_users)
    with np.errstate(invalid="ignore", divide="ignore"):
        mu = s_u / d_u                                   # :30
    c_i = np.bincount(item, minlength=n_items).astype(np.float64)
    s_i = np.bincount(item, weights=r, minlength=n_items)
    s2_i = np.bincount(item, weights=r * r, minlength=n_items)
    cen = r - mu[user]
    a2_i = np.bincount(item, weights=cen * cen, minlength=n_items)   # :70,75
    with np.errstate(invalid="ignore", divide="ignore"):
        avg_i = 1.0 * s_i / c_i                          # :60
    return dict(mu=mu, d_u=d_u, avg=avg_i, norm2=np.sqrt(s2_i),
                adj_norm2=np.sqrt(a2_i), count=c_i, sum_r=s_i)


def sim_pairs(user, item, rating, n_users, n_items, prefix_code,
              method="adjust_cosine", num_atleast=50):
    """All kept directed pairs, sorted by (i, j).

    baselinerSim.py:144-174 (adjust_cosine) / :115-142 (cosine), :97-113
    (mutuality), :198-199,207-208 (filter), :189-191 (label).
    """
    order = np.lexsort((item, user))
    user, item, rating = user[order], item[order], rating[order]
    st = user_item_stats(user, item, rating, n_users, n_items)
    r = rating.astype(np.float64)
    shape = (n_users, n_items)
    M = sp.csr_matrix((np.ones(len(user)), (user, item)), shape=shape)
    if method == "adjust_cosine":
        val = r - st["mu"][user]
        den = st["adj_norm2"]
    elif method == "cosine":
        val = r
        den = st["norm2"]
    else:
        raise ValueError(method)
    # explicit zeros must survive (a centred rating of exactly 0 still co-rates)
    C = sp.csr_matrix((val, (user, item)), shape=shape)
    a = (r >= st["avg"][item]).astype(np.float64)        # :106-107
    A = sp.csr_matrix((a, (user, item)), shape=shape)
    B = sp.csr_matrix((1.0 - a, (user, item)), shape=shape)

    N = (M.T @ M).tocoo()                                 # co-rating counts
    keep = N.row != N.col
    i = N.row[keep].astype(np.int64)
    j = N.col[keep].astype(np.int64)
    n = np.rint(N.data[keep])
    o = np.lexsort((j, i))
    i, j, n = i[o], j[o], n[o]

    Ct = C.T.tocsr()
    # scipy's csr_matmat accumulates each output row in traversal order, i.e.
    # ascending user index: the same order as the reference's np.sum for n<8.
    inner_m = _matmul_keep_zeros(Ct, C)
    inner = np.asarray(inner_m[i, j]).ravel()
    agree = (A.T @ A + B.T @ B).tocsr()
    mutu = np.rint(np.asarray(agree[i, j]).ravel())

    dd = den[i] * den[j]
    with np.errstate(invalid="ignore", divide="ignore"):
        cosv = np.where(dd != 0, 1.0 * inner / dd, 0.0)   # :95
    sim = 1.0 * cosv * np.minimum(n, num_atleast) / num_atleast   # :89
    frac = 1.0 * mutu / (st["count"][i] + st["count"][j] - n)     # :139-141
    kept = (sim != 0.0) & (mutu != 0.0) & (frac != 0.0)
    label = (prefix_code[i] != prefix_code[j]).astype(np.int32)
    return dict(i=i[kept], j=j[kept], sim=sim[kept], mutu=mutu[kept],
                n=n[kept], frac=frac[kept], label=label[kept],
                n_pairs_total=int(len(i)), inner_all=inner, n_all=n,
                i_all=i, j_all=j, stats=st)


def sim_rows(user, item, rating, n_users, n_items, prefix_code, rows,
             method="adjust_cosine", num_atleast=50):
    """sim_pairs restricted to the directed pairs (i, j) with i in `rows` (a 1-D array of item indices), so
    that a full-size input (BASELINE.json configs[1]) can be checked on a sample of item rows.  One row at a
    time: the ratings of the row's raters are gathered (ascending user, like the reference's arrival order
    under the canonical rules) and reduced per column with np.bincount, which adds in array order.  Returns
    the kept pairs sorted by (i, j) and, per sampled row, the number of co-rated columns (pre-filter)."""
    rows = np.unique(np.asarray(rows, dtype=np.int64))
    order = np.lexsort((item, user))
    user, item, rating = user[order], item[order], rating[order]
    st = user_item_stats(user, item, rating, n_users, n_items)
    r = rating.astype(np.float64)
    if method == "adjust_cosine":
        val, den = r - st["mu"][user], st["adj_norm2"]
    elif method == "cosine":
        val, den = r, st["norm2"]
    else:
        raise ValueError(method)
    ge = (r >= st["avg"][item])                                   # baselinerSim.py:106-107
    uptr = np.zeros(n_users + 1, dtype=np.int64); uptr[1:] = np.cumsum(np.bincount(user, minlength=n_users))
    o2 = np.argsort(item, kind="stable")                          # CSC: ascending user inside a column
    iptr = np.zeros(n_items + 1, dtype=np.int64); iptr[1:] = np.cumsum(np.bincount(item, minlength=n_items))
    c_user, c_val, c_ge = user[o2], val[o2], ge[o2]
    out = {k: [] for k in ("i", "j", "sim", "mutu", "n", "frac", "label")}
    n_cols = np.zeros(len(rows), dtype=np.int64)
    for q, i in enumerate(rows):
        ru = c_user[iptr[i]:iptr[i + 1]]
        lens = uptr[ru + 1] - uptr[ru]
        tot = int(lens.sum())
        if tot == 0:
            continue
        rep = np.repeat(np.arange(len(ru)), lens)
        pos = uptr[ru][rep] + (np.arange(tot) - (np.cumsum(lens) - lens)[rep])
        cols = item[pos]
        keep = cols != i
        cols, rep, pos = cols[keep], rep[keep], pos[keep]
        n = np.bincount(cols, minlength=n_items)
        inner = np.bincount(cols, weights=c_val[iptr[i]:iptr[i + 1]][rep] * val[pos], minlength=n_items)
        mutu = np.bincount(cols, weights=(c_ge[iptr[i]:iptr[i + 1]][rep] == ge[pos]).astype(np.float64), minlength=n_items)
        j = np.flatnonzero(n)
        n_cols[q] = len(j)
        nj, inj, mj = n[j].astype(np.float64), inner[j], np.rint(mutu[j])
        dd = den[i] * den[j]
        with np.errstate(invalid="ignore", divide="ignore"):
            cosv = np.where(dd != 0, 1.0 * inj / dd, 0.0)
        sim = 1.0 * cosv * np.minimum(nj, num_atleast) / num_atleast
        frac = 1.0 * mj / (st["count"][i] + st["count"][j] - nj)
        kept = (sim != 0.0) & (mj != 0.0) & (frac != 0.0)
        out["i"].append(np.full(int(kept.sum()), i, dtype=np.int64)); out["j"].append(j[kept])
        out["sim"].append(sim[kept]); out["mutu"].append(mj[kept]); out["n"].append(nj[kept]); out["frac"].append(frac[kept])
        out["label"].append((prefix_code[i] != prefix_code[j[kept]]).astype(np.int32))
    cat = lambda k, dt: np.concatenate(out[k]) if out[k] else np.zeros(0, dtype=dt)
    return dict(rows=rows, i=cat("i", np.int64), j=cat("j", np.int64), sim=cat("sim", np.float64),
                mutu=cat("mutu", np.float64), n=cat("n", np.float64), frac=cat("frac", np.float64),
                label=cat("label", np.int32), n_cols=n_cols, stats=st)


def _matmul_keep_zeros(At, B):
    """At @ B where stored zeros in the operands do not change the pattern of
    interest; returns a CSR matrix that can be fancy-indexed."""
    out = (At @ B).tocsr()
    return out


# --------------------------------------------------------------------------
# Selection  (extender.py:16-44, SURVEY.md App. A.3)
# --------------------------------------------------------------------------
def select_knn(pairs, n_items, k, dom_code, contains):
    """Returns dict with bb (bool[I]), valid_nb (bool[I]) and four ragged
    neighbour tables keyed 'BB_BB','BB_NB','NB_BB','NB_NN': each a list of
    int arrays of positions into `pairs` (so every per-edge value is reachable).
    """
    i, j, sim, label = pairs["i"], pairs["j"], pairs["sim"], pairs["label"]
    bb = np.zeros(n_items, dtype=bool)
    bb[i[label == 1]] = True                               # assist.py:84-86
    # stable sort by |sim| desc with ties to the smaller neighbour index
    order = np.lexsort((j, -np.abs(sim), i))
    ptr = np.searchsorted(i[order], np.arange(n_items + 1))
    out = {name: [np.zeros(0, np.int64)] * n_items
           for name in ("BB_BB", "BB_NB", "NB_BB", "NB_NN")}
    valid_nb = np.zeros(n_items, dtype=bool)
    for it in range(n_items):
        pos = order[ptr[it]:ptr[it + 1]]
        if len(pos) == 0:
            continue
        nb = j[pos]
        if bb[it]:
            same = ((contains[nb] >> dom_code[it]) & 1).astype(bool)
            out["BB_BB"][it] = pos[~same][:k]              # extender.py:31-32
            out["BB_NB"][it] = pos[same][:k]               # :33-34
        else:
            isbb = bb[nb]
            if isbb.any():
                valid_nb[it] = True
                out["NB_BB"][it] = pos[isbb][:k]           # :37-40
                out["NB_NN"][it] = pos[:k]                 # :41-42 (the `not in NB` test is always true)
    out["bb"] = bb
    out["valid_nb"] = valid_nb
    return out


# --------------------------------------------------------------------------
# Extension  (extender.py:46-217, SURVEY.md App. A.4)
# --------------------------------------------------------------------------
def xsim_extend(pairs, knn, n_items, has_S, has_T):
    """Returns X-SIM as (start, end, xsim) arrays sorted by (start, end), plus
    the number of (left, right) combos == reference paths enumerated."""
    j, sim, mutu, frac = pairs["j"], pairs["sim"], pairs["mutu"], pairs["frac"]
    bb = knn["bb"]

    def edges(pos):
        return j[pos], sim[pos] * mutu[pos], mutu[pos], frac[pos]

    # attach(b) = [(n, pos of edge (n,b), NB_NN(n))]  in ascending n   (extender.py:53-59,171-173)
    attach = {}
    for nidx in np.nonzero(knn["valid_nb"])[0]:
        for p in knn["NB_BB"][nidx]:
            attach.setdefault(int(j[p]), []).append((int(nidx), int(p)))

    def right_of(s):
        """(end, N-terms[2], D-terms[2], c-terms[2], n_edges) for every right segment of s."""
        ends, e1, m1, f1, e2, m2, f2, ne = [s], [0.0], [0.0], [1.0], [0.0], [0.0], [1.0], [0]
        for (nidx, p) in attach.get(s, ()):
            en, em, ef = sim[p] * mutu[p], mutu[p], frac[p]
            ends.append(nidx); e1.append(en); m1.append(em); f1.append(ef)
            e2.append(0.0); m2.append(0.0); f2.append(1.0); ne.append(1)
            for q in knn["NB_NN"][nidx]:
                ends.append(int(j[q])); e1.append(en); m1.append(em); f1.append(ef)
                e2.append(sim[q] * mutu[q]); m2.append(mutu[q]); f2.append(frac[q]); ne.append(2)
        return tuple(np.asarray(v) for v in (ends, e1, m1, f1, e2, m2, f2, ne))

    def left_of(t):
        """Left segments of t: start, edges in path order (x,n) then (n,t)."""
        st, e1, m1, f1, e2, m2, f2, ne = [], [], [], [], [], [], [], []
        for (nidx, p) in attach.get(t, ()):
            en, em, ef = sim[p] * mutu[p], mutu[p], frac[p]
            st.append(nidx); e1.append(en); m1.append(em); f1.append(ef)
            e2.append(0.0); m2.append(0.0); f2.append(1.0); ne.append(1)
            for q in knn["NB_NN"][nidx]:
                # path (x, n, t): first edge (x,n) then (n,t)
                st.append(int(j[q])); e1.append(sim[q] * mutu[q]); m1.append(mutu[q]); f1.append(frac[q])
                e2.append(en); m2.append(em); f2.append(ef); ne.append(2)
        return tuple(np.asarray(v) for v in (st, e1, m1, f1, e2, m2, f2, ne))

    # knn_BB[b] keys -> position of the edge (b, key)      (assist.py:121-124)
    def knn_bb_entries(b):
        return np.concatenate([knn["BB_BB"][b], knn["BB_NB"][b]])

    src = {}
    for s in attach:
        if bb[s] and has_S[s]:
            for p in knn_bb_entries(s):
                t = int(j[p])
                if has_T[t]:
                    src[(t, s)] = int(p)                    # extender.py:61-70
    tgt = set()
    for t in attach:
        if bb[t] and has_T[t]:
            for p in knn_bb_entries(t):
                s = int(j[p])
                if has_S[s]:
                    tgt.add((t, s))                         # :72-81

    S_, E_, NUM, DEN = [], [], [], []
    combos = 0
    rcache, lcache = {}, {}
    for (t, s), p in sorted(src.items()):
        if s not in rcache:
            rcache[s] = right_of(s)
        ry, re1, rm1, rf1, re2, rm2, rf2, rne = rcache[s]
        em, mm, fm = sim[p] * mutu[p], mutu[p], frac[p]
        # left list: the bare (t) start always (nonjoint, extender.py:180), plus
        # left(t) when the pair is also target-side (joint, :178-179)
        lx = np.array([t]); le1 = np.zeros(1); lm1 = np.zeros(1); lf1 = np.ones(1)
        le2 = np.zeros(1); lm2 = np.zeros(1); lf2 = np.ones(1); lne = np.zeros(1, int)
        if (t, s) in tgt:
            if t not in lcache:
                lcache[t] = left_of(t)
            L = lcache[t]
            lx = np.concatenate([lx, L[0]]); le1 = np.concatenate([le1, L[1]])
            lm1 = np.concatenate([lm1, L[2]]); lf1 = np.concatenate([lf1, L[3]])
            le2 = np.concatenate([le2, L[4]]); lm2 = np.concatenate([lm2, L[5]])
            lf2 = np.concatenate([lf2, L[6]]); lne = np.concatenate([lne, L[7]])
        # sequential sums in path order (extender.py:85-88): absent edges add an
        # exact 0.0 / multiply by an exact 1.0, which leaves fp64 results unchanged
        Nn = ((((le1[:, None] + le2[:, None]) + em) + re1[None, :]) + re2[None, :])
        Dd = ((((lm1[:, None] + lm2[:, None]) + mm) + rm1[None, :]) + rm2[None, :])
        cp = ((((lf1[:, None] * lf2[:, None]) * fm) * rf1[None, :]) * rf2[None, :])
        with np.errstate(invalid="ignore", divide="ignore"):
            spv = np.where(Dd != 0, 1.0 * Nn / Dd, 0.0)
        combos += Nn.size
        S_.append(np.repeat(lx, len(ry))); E_.append(np.tile(ry, len(lx)))
        NUM.append((spv * cp).ravel()); DEN.append(cp.ravel())
    if not S_:
        z = np.zeros(0)
        return dict(start=z.astype(np.int64), end=z.astype(np.int64), xsim=z, combos=0,
                    n_src=0, n_joint=0)
    S_ = np.concatenate(S_); E_ = np.concatenate(E_)
    NUM = np.concatenate(NUM); DEN = np.concatenate(DEN)
    key = S_.astype(np.int64) * n_items + E_
    o = np.argsort(key, kind="stable")
    key, NUM, DEN = key[o], NUM[o], DEN[o]
    uk, first = np.unique(key, return_index=True)
    num = np.add.reduceat(NUM, first)
    den = np.add.reduceat(DEN, first)
    return dict(start=uk // n_items, end=uk % n_items, xsim=1.0 * num / den,
                combos=int(combos), n_src=len(src),
                n_joint=sum(1 for k_ in src if k_ in tgt))


# --------------------------------------------------------------------------
# Generation  (generator.py:27-157, assist.py:210-215, SURVEY.md App. A.5)
# --------------------------------------------------------------------------
def candidates(start, end, xsim, top):
    """Per start row: first `top` ends by |xsim| desc, ties to smaller end."""
    o = np.lexsort((end, -np.abs(xsim), start))
    s, e, x = start[o], end[o], xsim[o]
    rows, ptr = np.unique(s, return_index=True)
    ptr = np.append(ptr, len(s))
    return rows, [(e[ptr[r]:ptr[r + 1]][:top], x[ptr[r]:ptr[r + 1]][:top])
                  for r in range(len(rows))]


def choose(rows, cands, mode, uniforms=None, epsilon=0.6, mapping_range=1, gs=2):
    """mode: 'argmax' (generator.py as shipped on py3: weighted_pick returns 0),
    'exp_mech' (generator.py:42-75 as intended: searchsorted_left(cumsum(w), u*sum w)),
    'nonprivate' (generator.py:109-110: index floor(u*(m-1)); m==1 -> index 0, flagged)."""
    out = np.zeros(len(rows), dtype=np.int64)
    single = 0
    for r, (e, x) in enumerate(cands):
        m = len(e)
        if mode == "argmax":
            idx = 0
        elif mode == "exp_mech":
            w = np.exp(epsilon * x / (2 * mapping_range * gs))     # :46-48
            w = w / w.sum()                                       # :54-56
            idx = int(np.searchsorted(np.cumsum(w), uniforms[r] * np.sum(w)))   # :68-70
            idx = min(idx, m - 1)
        elif mode == "nonprivate":
            if m == 1:
                idx = 0
                single += 1
            else:
                idx = min(int(np.floor(uniforms[r] * (m - 1))), m - 2)
        else:
            raise ValueError(mode)
        out[r] = e[idx]
    return out, single


def invert_mapping(rows, chosen, n_items):
    """assist.py:215 with rows consumed in ascending target index: largest wins.  A row without a
    candidate (chosen = -1, the device's marker) maps nothing."""
    mp = np.full(n_items, -1, dtype=np.int64)
    for t, s in zip(rows, chosen):
        if s >= 0:
            mp[s] = t
    return mp


def build_alterego(user, item, rating, ts, mapping, has_T):
    """generator.py:140-157.  Returns (user, item, rating, ts, synthetic_flag)
    with the untouched "T:" ratings first (in input order), then the mapped,
    mean-merged records sorted by (user, target)."""
    keep_t = has_T[item]
    mt = mapping[item]
    m = mt >= 0
    u2, t2, r2, ts2, src = user[m], mt[m], rating[m].astype(np.float64), ts[m], item[m]
    o = np.lexsort((src, t2, u2))
    u2, t2, r2, ts2 = u2[o], t2[o], r2[o], ts2[o]
    key = u2.astype(np.int64) * (mapping.shape[0] + 1) + t2
    uk, first, cnt = np.unique(key, return_index=True, return_counts=True)
    mean = np.array([np.mean(r2[f:f + c]) for f, c in zip(first, cnt)]) if len(uk) else np.zeros(0)
    return dict(user=np.concatenate([user[keep_t], u2[first]]),
                item=np.concatenate([item[keep_t], t2[first]]),
                rating=np.concatenate([rating[keep_t].astype(np.float64), mean]),
                ts=np.concatenate([ts[keep_t], ts2[first]]),
                synthetic=np.concatenate([np.zeros(int(keep_t.sum()), bool),
                                          np.ones(len(uk), bool)]))


# --------------------------------------------------------------------------
# Next row of the scope table (SURVEY.md 8(f) #1): RecommenderSim on the AlterEgo profile
# (recommenderSim.py:29-62 get_info, :64-75 produce_pairwise, :90-132 cosine_sim + local
# sensitivity, :186-195 calculate_sim with method "cosine_item").  No product kernel consumes
# this yet; it pins the semantics (duplicate (user, item) records, self pairs, no filter).
# --------------------------------------------------------------------------
def recommender_cosine_item(user, item, rating, n_items, num_atleast=50):
    """Flat profile records (user, item, rating), in the order the reference receives them
    (sorted by user; a (user, item) pair may occur twice: a real target rating next to a
    synthetic one, generator.py:156-157).  Returns every directed item pair with at least one
    co-rating entry, sorted by (i, j): dict(i, j, n, sim, ls, norm2)."""
    user = np.asarray(user, dtype=np.int64)
    item = np.asarray(item, dtype=np.int64)
    r = np.asarray(rating, dtype=np.float64)
    norm2 = np.sqrt(np.bincount(item, weights=r * r, minlength=n_items))          # :41-49 over ALL records of the item
    # co-rating entries: both orders of every 2-combination of a user's records (:64-75)
    order = np.argsort(user, kind="stable")
    us, it, rr = user[order], item[order], r[order]
    starts = np.flatnonzero(np.r_[True, us[1:] != us[:-1]])
    ends = np.r_[starts[1:], len(us)]
    ki, kj, ra, rb = [], [], [], []
    for a, b in zip(starts, ends):
        d = b - a
        if d < 2:
            continue
        p, q = np.triu_indices(d, 1)
        # combinations() order: (p, q) then its reverse, interleaved
        ki.append(np.stack([it[a + p], it[a + q]], 1).ravel()); kj.append(np.stack([it[a + q], it[a + p]], 1).ravel())
        ra.append(np.stack([rr[a + p], rr[a + q]], 1).ravel()); rb.append(np.stack([rr[a + q], rr[a + p]], 1).ravel())
    if not ki:
        z = np.zeros(0)
        return dict(i=z.astype(np.int64), j=z.astype(np.int64), n=z.astype(np.int64), sim=z, ls=z, norm2=norm2)
    ki, kj, ra, rb = (np.concatenate(x) for x in (ki, kj, ra, rb))
    key = ki * n_items + kj
    o = np.argsort(key, kind="stable")                      # entries of a pair stay in arrival (user) order
    key, ki, kj, ra, rb = key[o], ki[o], kj[o], ra[o], rb[o]
    first = np.flatnonzero(np.r_[True, key[1:] != key[:-1]])
    n = np.diff(np.r_[first, len(key)])
    seg = np.repeat(np.arange(len(first)), n)
    prod = ra * rb
    inner = np.add.reduceat(prod, first)                    # :118
    pi, pj = ki[first], kj[first]
    nx, ny = norm2[pi], norm2[pj]
    N = float(num_atleast)

    def cosine(dot, nn):                                    # :84-88 (a NaN norm product is truthy)
        with np.errstate(invalid="ignore", divide="ignore"):
            return np.where(nn != 0, 1.0 * dot / nn, 0.0)

    sim = 1.0 * cosine(inner, nx * ny) * np.minimum(n, num_atleast) / N            # :77-82, :121-122
    # local sensitivity (:98-116): two leave-one-out similarities per co-rating entry
    m_inner = inner[seg] - prod
    with np.errstate(invalid="ignore"):
        m1 = np.sqrt((nx[seg] ** 2 - ra ** 2) * (ny[seg] ** 2))
        m2 = np.sqrt((nx[seg] ** 2) * (ny[seg] ** 2 - rb ** 2))
    w = np.minimum(n[seg] - 1, num_atleast)
    v1 = 1.0 * cosine(m_inner, m1) * w / N
    v2 = 1.0 * cosine(m_inner, m2) * w / N
    dev = np.abs(np.stack([v1, v2], 1) - sim[seg][:, None]).ravel()                # result order: v1, v2 per entry
    first2, seg2 = 2 * first, np.repeat(np.arange(len(first)), 2 * n)
    ls = np.fmax.reduceat(dev, first2)                       # NaN-free pairs
    for g in np.unique(seg2[np.isnan(dev)]):                 # Python's max(): a NaN only wins if it comes first
        vals = dev[first2[g]:first2[g] + 2 * n[g]]
        res = vals[0]
        for x in vals[1:]:
            if x > res:
                res = x
        ls[g] = res
    return dict(i=pi, j=pj, n=n, sim=sim, ls=ls, norm2=norm2)


# --------------------------------------------------------------------------
# SURVEY.md 8(f) #2-#3: non-private neighbour selection (recommenderPrivacy.py:141-178) and item-based
# prediction + MAE (recommenderPrediction.py:26-139) on the AlterEgo profile.
# --------------------------------------------------------------------------
def recommender_neighbors(pairs, n_items, mapping_range=10):
    """pairs: output of recommender_cosine_item (sorted by (i, j)).  Per item the first `mapping_range`
    neighbours by |sim| descending, ties to the smaller neighbour index (stable sort of the canonical order);
    the self pair (i, i) is a neighbour like any other.  Returns (ptr [n_items + 1], idx, sim)."""
    i, j, sim = pairs["i"], pairs["j"], pairs["sim"]
    o = np.lexsort((j, -np.abs(sim), i))
    ptr_all = np.searchsorted(i[o], np.arange(n_items + 1))
    idx, val, ptr = [], [], np.zeros(n_items + 1, dtype=np.int64)
    for it in range(n_items):
        sel = o[ptr_all[it]:ptr_all[it + 1]][:mapping_range]
        idx.append(j[sel]); val.append(sim[sel])
        ptr[it + 1] = ptr[it] + len(sel)
    return ptr, (np.concatenate(idx) if idx else np.zeros(0, np.int64)), (np.concatenate(val) if val else np.zeros(0))


def bound_rating(x):
    """recommenderPrediction.py:19-24: int() truncates towards zero."""
    return 1.0 * max(0, min(int(x + 0.5), 5))


def recommender_predict(p_user, p_item, p_rating, p_ts, nb_ptr, nb_idx, nb_sim, item_avg,
                        t_user, t_item, t_rating, alpha=0.03, raw=False):
    """Item-based prediction of every test (user, item) pair: (no-decay, decay) predictions (-1 where the item
    has no neighbour list) and the two MAEs (recommenderPrediction.py:26-139).  Profile records in list order.
    raw=True also returns the no-decay and decay values before bound_rating (NaN where the item has no
    neighbour list), so a caller can tell a value at a rounding boundary from a real mismatch."""
    by_ui = {}
    for q, (u, i) in enumerate(zip(p_user, p_item)):
        by_ui.setdefault((int(u), int(i)), []).append(q)          # profile order within (user, item)
    out0, out1 = np.full(len(t_user), -1.0), np.full(len(t_user), -1.0)
    raw0, raw1 = np.full(len(t_user), np.nan), np.full(len(t_user), np.nan)
    for q, (u, it) in enumerate(zip(t_user, t_item)):
        a, b = nb_ptr[it], nb_ptr[it + 1]
        if b == a:
            continue                                              # `iid not in sim_bd.value.keys()` -> ()
        ent = []                                                  # (sim * (r - avg_n), |sim|, time)
        for nid, ns in zip(nb_idx[a:b], nb_sim[a:b]):
            for r in by_ui.get((int(u), int(nid)), ()):
                ent.append((ns * (p_rating[r] - item_avg[nid]), abs(ns), p_ts[r]))
        avg = item_avg[it]
        if ent:
            nd = avg + sum(e[0] for e in ent) / sum(e[1] for e in ent)
            srt = sorted(ent, key=lambda e: e[2])                 # sort_by_time: equal times share a rank
            order, ranks = 0, []
            for k, e in enumerate(srt):
                if not (k != 0 and e[2] == srt[k - 1][2]):
                    order += 1
                ranks.append(order)
            cur = max(ranks) + 1
            f = [np.exp(-alpha * (cur - t)) for t in ranks]
            dc = avg + sum(e[0] * w for e, w in zip(srt, f)) / sum(e[1] * w for e, w in zip(srt, f))
        else:
            nd = dc = avg
        out0[q], out1[q] = bound_rating(nd), bound_rating(dc)
        raw0[q], raw1[q] = nd, dc
    ok = out0 >= 0
    mae0 = float(np.abs(t_rating[ok] - out0[ok]).sum() / ok.sum()) if ok.any() else float("nan")
    mae1 = float(np.abs(t_rating[ok] - out1[ok]).sum() / ok.sum()) if ok.any() else float("nan")
    if raw:
        return out0, out1, mae0, mae1, raw0, raw1
    return out0, out1, mae0, mae1


def laplace_from_uniform(u, scale):
    """numpy's legacy RandomState.laplace(0, scale) as a function of the one double it consumes."""
    u = np.asarray(u, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(u >= 0.5, 0.0 - scale * np.log(2.0 - u - u), 0.0 + scale * np.log(u + u))


def recommender_private_neighbors(pairs, n_items, mapping_range, epsilon, rpo, u_pick, u_noise):
    """The private branch of the neighbour selection AS IT BEHAVES UNDER PYTHON 3 (recommenderPrivacy.py:35-139, 152-171):
    per item with at least one pair, ONE neighbour is drawn (`np.count_nonzero(map(...))`, :81, counts the map object, so
    num_selection is 1 for any mapping_range) from the exponential-mechanism weights over ALL its neighbours in
    |sim|-descending order (stable: ties keep the (i, j) order), and Laplace noise of scale |local sensitivity| / eps is
    added to its similarity.  eps = privacy_epsilon / 2 (:18).  u_pick / u_noise: one uniform per such item, in item order.

    pairs: output of recommender_cosine_item (sorted by (i, j)).  Returns (items, chosen neighbour, noisy sim)."""
    i, j, sim, ls = pairs["i"], pairs["j"], pairs["sim"], pairs["ls"]
    eps, k = epsilon / 2.0, int(mapping_range)
    ptr = np.searchsorted(i, np.arange(n_items + 1))
    items, chosen, out = [], [], []
    q = 0
    for it in range(n_items):
        a, b = ptr[it], ptr[it + 1]
        if b == a:
            continue
        o = a + np.argsort(-np.abs(sim[a:b]), kind="stable")           # :123
        s_, r_, n = sim[o], ls[o], b - a
        max_rs = r_[np.argsort(-np.abs(r_), kind="stable")[0]]         # :103-106
        k_sim = s_[k - 1] if n >= k else s_[-1]                        # :43-46
        if n > k:                                                      # :54-66
            with np.errstate(divide="ignore", invalid="ignore"):
                w = min(k_sim, (2 * k * max_rs / eps) * np.log(k * (n - k) / rpo))
        else:
            w = k_sim
        msim = np.maximum(s_, s_ - w)                                  # :71-73
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            prob = np.exp(eps * msim / (2 * k * r_))                   # :88-93
            tot = 0.0
            for v in prob:                                             # Python sum(): sequential
                tot = tot + v
            p = prob / tot                                             # :97-99
        t = np.cumsum(p)                                               # :115
        idx = int(np.searchsorted(t, u_pick[q] * np.sum(p)))           # :116-118
        idx = min(idx, n - 1)
        items.append(it); chosen.append(j[o[idx]])
        out.append(s_[idx] + laplace_from_uniform(u_noise[q], abs(r_[idx]) / eps))      # :159-166
        q += 1
    return np.array(items, dtype=np.int64), np.array(chosen, dtype=np.int64), np.array(out, dtype=np.float64)
