"""Shared helpers of the parity tests: run the CUDA path through the public
engine / C ABI and compare with the oracle (oracle/restate.py, golden files).

oracle/ is imported here only as the checker.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
GOLDEN_CASES = ("adj_low_overlap", "cos_half_ratings", "adj_all_bridge")
SIM_RTOL = 1e-5          # BASELINE.json north_star: similarities within 1e-5 relative


def load_golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    g = {k: g[k] for k in g.files}
    return expand_pairs(g) if "pair_ptr" in g else g


def expand_pairs(g):
    """A compact sim-only golden (oracle/make_golden.compact_sim_only: the pairs i < j, similarity and frac on a
    sample of them) -> every directed pair sorted by (i, j), as the other goldens hold them; sim_val and sim_frac
    are NaN where the sample has no value."""
    n_items = len(g["iids"])
    i = np.repeat(np.arange(n_items), np.diff(g["pair_ptr"]))
    j = g["pair_j"].astype(np.int64)
    val = np.full(len(j), np.nan)
    val[g["sample"]] = g["sample_sim"]
    frac = np.full(len(j), np.nan, dtype=np.float32)
    frac[g["sample"]] = g["sample_frac"]
    ii, jj = np.concatenate([i, j]), np.concatenate([j, i])
    o = np.argsort(ii * n_items + jj)
    idt = g["pair_j"].dtype
    return dict(g, sim_i=ii[o].astype(idt), sim_j=jj[o].astype(idt), sim_val=np.concatenate([val, val])[o],
                sim_mutu=np.concatenate([g["pair_mutu"]] * 2)[o], sim_label=np.concatenate([g["pair_label"]] * 2)[o],
                sim_frac=np.concatenate([frac, frac])[o])


def golden_meta(g):
    from xmap_b200.encode import item_codes
    pc, dc, ct, hs, ht = item_codes(g["iids"])
    return dict(prefix_code=pc, dom_code=dc, contains=ct, has_S=hs, has_T=ht)


def to_device_meta(meta, device="cuda"):
    from xmap_b200.engine import to_device_meta as f
    return f(meta, device)


def _case_from_ratings(sr, keep=None, half=False):
    """Compact the (optionally masked) synthetic ratings to the users / items that occur, numbered in
    sorted id order, with the per-item codes (ids built like the reference's)."""
    from xmap_b200 import synth
    from xmap_b200.encode import item_codes
    user, item, rating_i, ts = sr.user, sr.item, sr.rating, sr.ts
    if keep is not None:
        user, item, rating_i, ts = user[keep], item[keep], rating_i[keep], ts[keep]
    present = np.unique(item)
    iid_all = np.array([synth.item_id(int(g), sr.n_items_per_domain, sr.labels) for g in present])
    order = np.argsort(iid_all)
    present, iids = present[order], iid_all[order]
    imap = np.full(int(item.max()) + 1, -1, dtype=np.int64)
    imap[present] = np.arange(len(present))
    uu = np.unique(user)              # user ids are zero-padded -> numeric order == string order
    umap = np.full(int(user.max()) + 1, -1, dtype=np.int64)
    umap[uu] = np.arange(len(uu))
    rating = rating_i.astype(np.float64)
    if half:
        rating = rating - 0.5 * ((user + item) & 1)
    pc, dc, ct, hs, ht = item_codes(iids)
    return dict(user=umap[user], item=imap[item], rating=rating, ts=ts,
                n_users=len(uu), n_items=len(iids), iids=iids,
                meta=dict(prefix_code=pc, dom_code=dc, contains=ct, has_S=hs, has_T=ht))


def synth_case(n_users, n_items, n_draws, overlap, seed, half=False):
    """Synthetic two-domain arrays + per-item codes."""
    from xmap_b200 import synth
    return _case_from_ratings(synth.make_ratings(n_users, n_items, n_draws, overlap=overlap, seed=seed), half=half)


def multi_domain_cases(n_users, n_items, n_draws, overlap, seed, n_domains=3):
    """The multi-domain shape (labels "S:1:", "S:2:", ..., "T:"): the reference runs one independent
    two-domain pipeline per source domain and unions the results (multidomain_demo.py:101-128), so
    this yields one two-domain case per source domain, cut from ONE multi-domain rating set."""
    from xmap_b200 import synth
    sr = synth.make_ratings(n_users, n_items, n_draws, n_domains=n_domains, overlap=overlap, seed=seed)
    tgt = n_domains - 1
    return [(sr.labels[d], _case_from_ratings(sr, (sr.domain == d) | (sr.domain == tgt)))
            for d in range(n_domains - 1)]


def run_gpu_sim(user, item, rating, n_users, n_items, meta, method, num_atleast, k, emit=True, **engine_kw):
    """engine_kw: SimEngine options (max_smem_cells, rec_budget)."""
    import torch
    from xmap_b200 import engine as E
    lay = E.build_layout(user, item, rating, n_users, n_items)
    eng = E.SimEngine(lay, to_device_meta(meta), method, num_atleast, k, **engine_kw)
    tabs = eng.run()
    pairs = eng.emit_pairs() if emit else None
    torch.cuda.synchronize()
    return lay, eng, tabs, pairs


def compare_layout(lay, st):
    """user means / item stats vs oracle (restate.user_item_stats or golden item_info)."""
    mu = lay.user_mu.cpu().numpy()
    its = lay.item_stats.cpu().numpy()
    assert np.array_equal(mu, st["mu"]), "user means differ"
    assert np.array_equal(its[:, 3], st["count"]), "item counts differ"
    assert np.array_equal(its[:, 0], st["avg"]), "item averages differ"
    np.testing.assert_allclose(its[:, 1], st["norm2"], rtol=1e-14)
    np.testing.assert_allclose(its[:, 2], st["adj_norm2"], rtol=1e-13)


FRAGILE_SIM = 1e-13      # |sim| below this is a pure rounding residue of a cancelling inner product


def compare_pairs(pairs, ref_i, ref_j, ref_sim, ref_mutu, ref_frac, ref_label, n_items, rtol=SIM_RTOL):
    """Kept-pair set, mutuality, frac, label bit-exact; sim within rtol.

    The one tolerated divergence: "fragile zeros" -- pairs whose inner product
    cancels exactly in exact arithmetic.  The reference's fp64 sum leaves a
    ~1e-17 residue (so it keeps the pair with |sim| ~ 1e-18, and under a real
    Spark shuffle whether it does depends on arrival order); the order-free
    fixed-point accumulator returns exactly 0 and the filter drops it.
    Returns (max rel err, set of fragile keys i*n_items+j)."""
    gi, gj = pairs["i"].cpu().numpy(), pairs["j"].cpu().numpy()
    gkey = gi.astype(np.int64) * n_items + gj
    rkey = ref_i.astype(np.int64) * n_items + ref_j
    only_ref = np.setdiff1d(rkey, gkey, assume_unique=True)
    only_gpu = np.setdiff1d(gkey, rkey, assume_unique=True)
    gs = pairs["sim"].cpu().numpy()
    if len(only_ref):
        m = np.isin(rkey, only_ref)
        assert (np.abs(ref_sim[m]) < FRAGILE_SIM).all(), "GPU dropped %d non-fragile pairs" % m.sum()
        assert len(only_ref) <= 1e-4 * len(rkey) + 1, "too many fragile zeros: %d" % len(only_ref)
    if len(only_gpu):
        m = np.isin(gkey, only_gpu)
        assert (np.abs(gs[m]) < FRAGILE_SIM).all(), "GPU kept %d pairs the reference filtered" % m.sum()
    gm = np.isin(gkey, rkey, assume_unique=True)
    rm = np.isin(rkey, gkey, assume_unique=True)
    assert np.array_equal(gkey[gm], rkey[rm])
    assert np.array_equal(pairs["mutu"].cpu().numpy()[gm], ref_mutu[rm].astype(np.int64)), "mutuality differs"
    assert np.array_equal(pairs["label"].cpu().numpy()[gm], ref_label[rm].astype(np.int64)), "labels differ"
    assert np.array_equal(pairs["frac"].cpu().numpy()[gm], ref_frac[rm]), "frac_mutu differs"
    rs = ref_sim[rm]
    solid = np.abs(rs) >= FRAGILE_SIM
    rel = np.abs(gs[gm][solid] - rs[solid]) / np.abs(rs[solid])
    assert rel.size == 0 or rel.max() <= rtol, "sim max rel err %g" % rel.max()
    fragile = set(only_ref.tolist()) | set(only_gpu.tolist()) | set(rkey[rm][~solid].tolist())
    return (float(rel.max()) if rel.size else 0.0), fragile


def gpu_lists(tabs):
    """(flags, len[I,2], idx[I,2,k]) as numpy."""
    return (tabs.row_flags.cpu().numpy(), tabs.tab_len.cpu().numpy(), tabs.tab_idx.cpu().numpy(),
            tabs.tab_sim.cpu().numpy(), tabs.tab_mutu.cpu().numpy(), tabs.tab_n.cpu().numpy())


NEAR_TIE_RTOL = 1e-9     # |sim| values closer than this are a tie up to fp64 rounding noise


def compare_knn(tabs, bb, valid_nb, lists, fragile=frozenset(), ref_pairs=None, ref_sim=None):
    """lists: dict name -> (ptr, nbr) ragged arrays in canonical order.
    Neighbour lists must be identical, order included, with two tolerated divergences:
      * neighbours that are fragile zeros (see compare_pairs) may be missing / extra;
      * neighbours whose |sim| agree to NEAR_TIE_RTOL may be permuted or swapped at the cut:
        mathematically tied similarities are ordered by ulp-level rounding noise in the fp64
        reference and by item index in the order-free fixed-point kernels (ref_sim: callable
        (item, neighbour) -> reference sim, needed to recognise them).
    Returns the number of lists that differed only by near-ties."""
    flags, tl, ti, ts, _, _ = gpu_lists(tabs)
    n_items = len(bb)
    gbb = flags.astype(bool)
    if not np.array_equal(gbb, bb):
        assert fragile and ref_pairs is not None, "BB flags differ"
        # an item may lose BB status only if every cross-domain kept pair of it is fragile
        ri, rj, rl = ref_pairs
        for it in np.nonzero(gbb != bb)[0]:
            js = rj[(ri == it) & (rl == 1)]
            assert all((int(it) * n_items + int(j)) in fragile for j in js), "BB flag of item %d differs" % it
    bad, near, examples = 0, 0, []
    for it in range(n_items):
        if gbb[it] != bb[it]:
            continue
        if bb[it]:
            names = ("BB_BB", "BB_NB")
        elif valid_nb[it]:
            names = ("NB_BB", "NB_NN")
        else:
            if tl[it, 0] != 0:
                bad += 1
            continue
        for slot, nm in enumerate(names):
            ptr, nbr = lists[nm]
            want = nbr[ptr[it]:ptr[it + 1]]
            got = ti[it, slot, :tl[it, slot]]
            if np.array_equal(got, want):
                continue
            if fragile:
                w2 = [int(j) for j in want if (it * n_items + int(j)) not in fragile]
                g2 = [int(j) for j in got if (it * n_items + int(j)) not in fragile]
                if g2[:len(w2)] == w2:
                    continue
            if ref_sim is not None and len(got) == len(want):
                rs = np.abs(np.array([ref_sim(it, int(j)) for j in want]))
                gs = np.abs(ts[it, slot, :tl[it, slot]])
                if np.allclose(gs, rs, rtol=NEAR_TIE_RTOL, atol=0):
                    near += 1
                    continue
                examples.append((it, nm, got.tolist(), want.tolist(), gs.tolist(), rs.tolist()))
            bad += 1
    assert bad == 0, "%d neighbour lists differ, e.g. %r" % (bad, examples[:2])
    return near


def restate_lists(knn, pairs):
    """oracle/restate.select_knn output -> the (ptr, nbr) form compare_knn takes."""
    out = {}
    for nm in ("BB_BB", "BB_NB", "NB_BB", "NB_NN"):
        ptr = np.zeros(len(knn[nm]) + 1, dtype=np.int64)
        ptr[1:] = np.cumsum([len(p) for p in knn[nm]])
        nbr = np.concatenate([pairs["j"][p] for p in knn[nm]]) if ptr[-1] else np.zeros(0, np.int64)
        out[nm] = (ptr, nbr)
    return out


def check_sim_against_restatement(case, method, num_atleast, k, **engine_kw):
    from oracle import restate as RS
    lay, eng, tabs, pairs = run_gpu_sim(case["user"], case["item"], case["rating"], case["n_users"],
                                        case["n_items"], case["meta"], method, num_atleast, k, **engine_kw)
    P = RS.sim_pairs(case["user"], case["item"], case["rating"], case["n_users"], case["n_items"],
                     case["meta"]["prefix_code"], method, num_atleast)
    compare_layout(lay, P["stats"])
    rel, fragile = compare_pairs(pairs, P["i"], P["j"], P["sim"], P["mutu"], P["frac"], P["label"],
                                 case["n_items"])
    assert tabs.n_pairs_total == P["n_pairs_total"], "co-rated pair count differs"
    knn = RS.select_knn(P, case["n_items"], k, case["meta"]["dom_code"], case["meta"]["contains"])
    n_items = case["n_items"]
    pkey = P["i"].astype(np.int64) * n_items + P["j"]          # sorted by construction

    def ref_sim(it, j):
        q = np.searchsorted(pkey, it * n_items + j)
        return P["sim"][q] if q < len(pkey) and pkey[q] == it * n_items + j else 0.0
    near = compare_knn(tabs, knn["bb"], knn["valid_nb"], restate_lists(knn, P), fragile,
                       (P["i"], P["j"], P["label"]), ref_sim)
    n_lists = 2 * int(knn["bb"].sum() + knn["valid_nb"].sum())
    assert near <= 0.005 * n_lists + 1, "%d of %d lists differ by near-ties" % (near, n_lists)
    return dict(lay=lay, eng=eng, tabs=tabs, pairs=pairs, P=P, knn=knn, rel=rel, fragile=fragile, near_ties=near)


def run_smoke():
    """One small hot-path invocation on cuda:0, checked against the oracle."""
    import torch
    assert torch.cuda.is_available(), "smoke() needs a GPU"
    case = synth_case(400, 150, 6000, 0.05, seed=3)
    out = check_sim_against_restatement(case, "adjust_cosine", 50, 4)
    print("smoke: %d kept pairs, sim max rel err %.3g, launches %d" % (
        len(out["P"]["i"]), out["rel"], out["eng"].launches))
    # the rest of the path on the same case: X-SIM extension (both kernels) and the argmax mapping vs the oracle
    from oracle import restate as RS
    X = RS.xsim_extend(out["P"], out["knn"], case["n_items"], case["meta"]["has_S"], case["meta"]["has_T"])
    for mode in ("hybrid", "warp", "cta"):
        plan, xe, res, (s, e, v) = run_gpu_extend(out["tabs"], out["lay"], case["meta"], mode=mode)
        rel = compare_xsim(s, e, v, X["start"], X["end"], X["xsim"])
        assert int(res.combos.sum()) == X["combos"]
        print("smoke: X-SIM (%s kernel) %d pairs from %d paths, max rel err %.3g" % (mode, len(v), X["combos"], rel))


# --------------------------------------------------------------------------
# X-SIM extension + generation
# --------------------------------------------------------------------------
def tables_from_restatement(P, knn, n_items, k, device="cpu"):
    """oracle/restate.select_knn output -> engine.SimTables (host tensors): lets the
    host-side plan builder be checked without a GPU."""
    import torch
    from xmap_b200.engine import SimTables
    idx = np.full((n_items, 2, k), -1, np.int32); sim = np.zeros((n_items, 2, k))
    mutu = np.zeros((n_items, 2, k), np.int32); nn = np.zeros((n_items, 2, k), np.int32)
    ln = np.zeros((n_items, 2), np.int32)
    for it in range(n_items):
        names = ("BB_BB", "BB_NB") if knn["bb"][it] else ("NB_BB", "NB_NN")
        for slot, nm in enumerate(names):
            pos = knn[nm][it]
            L = len(pos)
            ln[it, slot] = L
            idx[it, slot, :L] = P["j"][pos]; sim[it, slot, :L] = P["sim"][pos]
            mutu[it, slot, :L] = P["mutu"][pos]; nn[it, slot, :L] = P["n"][pos]
    T = lambda a, dt: torch.as_tensor(a, dtype=dt, device=device)
    nk = np.bincount(P["i"], minlength=n_items)
    return SimTables(k, n_items, T(knn["bb"].astype(np.uint8), torch.uint8), T(nk, torch.int32),
                     T(nk, torch.int32), T(idx, torch.int32), T(sim, torch.float64),
                     T(mutu, torch.int32), T(nn, torch.int32), T(ln, torch.int32))


def eval_plan_numpy(plan):
    """Reference evaluation of an extend.XsimPlan in plain Python (small cases only):
    mirrors what the CUDA kernel computes."""
    p = plan
    g = lambda t: t.cpu().numpy()
    leg_ptr, leg_t, leg_jo = g(p.leg_ptr), g(p.leg_t), g(p.leg_joint_only)
    lv = [g(v) for v in p.leg_vals]
    par_ptr, par_s, par_j = g(p.par_ptr), g(p.par_s), g(p.par_joint)
    pv = [g(v) for v in p.par_vals]
    rs_ptr, rs_end = g(p.rs_ptr), g(p.rs_end)
    rv = [g(v) for v in p.rs_vals]
    start_item = g(p.start_item)
    S, E, X = [], [], []
    combos = 0
    for x in range(len(start_item)):
        acc = {}
        for lg in range(leg_ptr[x], leg_ptr[x + 1]):
            t = leg_t[lg]
            Nl = lv[0][lg] + lv[3][lg]; Dl = lv[1][lg] + lv[4][lg]; Cl = lv[2][lg] * lv[5][lg]
            for pp in range(par_ptr[t], par_ptr[t + 1]):
                if leg_jo[lg] and not par_j[pp]:
                    continue
                s = par_s[pp]
                Nm = Nl + pv[0][pp]; Dm = Dl + pv[1][pp]; Cm = Cl * pv[2][pp]
                a, b = rs_ptr[s], rs_ptr[s + 1]
                Nn = Nm + (rv[0][a:b] + rv[3][a:b])
                Dd = Dm + (rv[1][a:b] + rv[4][a:b])
                cp = Cm * (rv[2][a:b] * rv[5][a:b])
                with np.errstate(invalid="ignore", divide="ignore"):
                    sp = np.where(Dd != 0, Nn / Dd, 0.0)
                combos += b - a
                for y, n_, d_ in zip(rs_end[a:b], sp * cp, cp):
                    c = acc.setdefault(int(y), [0.0, 0.0])
                    c[0] += n_; c[1] += d_
        for y in sorted(acc):
            S.append(int(start_item[x])); E.append(y); X.append(acc[y][0] / acc[y][1])
    o = np.lexsort((E, S))
    return np.array(S)[o], np.array(E)[o], np.array(X)[o], combos


def eval_engine_numpy(xe, g_ranges=None):
    """Evaluates the arrays an extend.XsimEngine hands to the kernel (legs, partner lists incl. the virtual
    partners of the fused bridge lists, pi-ordered right-segment / fused lists, tile pointers) the way the kernel
    does, in numpy: pins the engine's host-side index building (small cases only).  g_ranges: tile ranges to walk
    (default one pass over every tile); the union must cover [0, 2^gb)."""
    g = lambda t: t.cpu().numpy()
    p = xe.plan
    leg_ptr, start_item = g(p.leg_ptr), g(p.start_item)
    lp_ptr = g(xe.lp_ptr)
    pd_s, pd_n, pd_d, pd_c = g(xe.pd_s), g(xe.pd_n), g(xe.pd_d), g(xe.pd_c)
    # the pair descriptors restate (leg, partner): list of the partner, leg and bridge edge folded in path order
    lp_base, lp_n = g(xe.leg_par_base), g(xe.leg_npar)
    lN, lD, lC = g(xe.leg_n), g(xe.leg_d), g(xe.leg_c)
    ps, pe, pm, pf = g(xe.par_s), g(xe.par_e), g(xe.par_m), g(xe.par_f)
    assert np.array_equal(np.diff(lp_ptr), lp_n) and len(pd_s) == lp_ptr[-1]
    for lg in range(len(lp_n)):
        for k in range(lp_n[lg]):
            q, pp = lp_ptr[lg] + k, lp_base[lg] + k
            assert pd_s[q] == ps[pp] and pd_n[q] == lN[lg] + pe[pp] and pd_d[q] == lD[lg] + pm[pp] and pd_c[q] == lC[lg] * pf[pp]
    rs_ptr, rs_end = g(xe.rs_ptr), g(xe.rs_end)
    rN, rD, rC = (g(v) for v in xe.rs_ndc)
    tp = g(xe.tile_ptr)
    G = 1 << xe.gb
    assert np.array_equal(tp[:, G], rs_ptr[1:] - rs_ptr[:-1]) and (tp[:, 0] == 0).all() and (np.diff(tp, axis=1) >= 0).all()
    pi = (rs_end.astype(np.int64) * 0x9E3779B1) & 0xFFFFFFFF
    tile = pi >> (32 - xe.gb)
    for s_ in range(len(rs_ptr) - 1):                     # every list is ordered by pi and cut by tile_ptr
        a, b = rs_ptr[s_], rs_ptr[s_ + 1]
        assert (np.diff(pi[a:b]) >= 0).all()
        assert np.array_equal(np.searchsorted(tile[a:b], np.arange(G + 1), side="left"), tp[s_])
    g_ranges = g_ranges or [(0, G)]
    S, E, X = [], [], []
    combos = 0
    for x in range(len(start_item)):
        acc = {}
        for g0, g1 in g_ranges:
            for q in range(lp_ptr[leg_ptr[x]], lp_ptr[leg_ptr[x + 1]]):
                if True:
                    s_ = pd_s[q]
                    Nm, Dm, Cm = pd_n[q], pd_d[q], pd_c[q]
                    a, b = rs_ptr[s_] + tp[s_, g0], rs_ptr[s_] + tp[s_, g1]
                    Nn = Nm + rN[a:b]; Dd = Dm + rD[a:b]; cp = Cm * rC[a:b]
                    with np.errstate(invalid="ignore", divide="ignore"):
                        sp = np.where(Dd != 0, Nn / Dd, 0.0)
                    combos += b - a
                    for y, n_, d_ in zip(rs_end[a:b], sp * cp, cp):
                        c = acc.setdefault(int(y), [0.0, 0.0])
                        c[0] += n_; c[1] += d_
        for y in sorted(acc):
            S.append(int(start_item[x])); E.append(y); X.append(acc[y][0] / acc[y][1])
    o = np.lexsort((E, S))
    return np.array(S)[o], np.array(E)[o], np.array(X)[o], combos


def eval_plan_starts(plan, starts):
    """X-SIM rows of a few starts (plan indices) evaluated in numpy straight from the plan arrays, one start
    at a time with the terms of a cell in path order: {start index: (ends sorted, xsim, n_paths)}.  Checks
    the kernel at sizes where the whole extension cannot be evaluated on the host."""
    p = plan
    g = lambda t: t.cpu().numpy()
    leg_ptr, leg_t, leg_jo = g(p.leg_ptr), g(p.leg_t), g(p.leg_joint_only)
    lv = [g(v) for v in p.leg_vals]
    par_ptr, par_s, par_j = g(p.par_ptr), g(p.par_s), g(p.par_joint)
    pv = [g(v) for v in p.par_vals]
    rs_ptr, rs_end = g(p.rs_ptr), g(p.rs_end)
    rv = [g(v) for v in p.rs_vals]
    rN, rD, rC = rv[0] + rv[3], rv[1] + rv[4], rv[2] * rv[5]
    out = {}
    for x in starts:
        Y, NUM, DEN = [], [], []
        for lg in range(leg_ptr[x], leg_ptr[x + 1]):
            t = leg_t[lg]
            Nl = lv[0][lg] + lv[3][lg]; Dl = lv[1][lg] + lv[4][lg]; Cl = lv[2][lg] * lv[5][lg]
            for pp in range(par_ptr[t], par_ptr[t + 1]):
                if leg_jo[lg] and not par_j[pp]:
                    continue
                s = par_s[pp]
                a, b = rs_ptr[s], rs_ptr[s + 1]
                Nn = (Nl + pv[0][pp]) + rN[a:b]
                Dd = (Dl + pv[1][pp]) + rD[a:b]
                cp = (Cl * pv[2][pp]) * rC[a:b]
                with np.errstate(invalid="ignore", divide="ignore"):
                    sp = np.where(Dd != 0, Nn / Dd, 0.0)
                Y.append(rs_end[a:b]); NUM.append(sp * cp); DEN.append(cp)
        Y = np.concatenate(Y); NUM = np.concatenate(NUM); DEN = np.concatenate(DEN)
        o = np.argsort(Y, kind="stable")
        uy, first = np.unique(Y[o], return_index=True)
        out[int(x)] = (uy, np.add.reduceat(NUM[o], first) / np.add.reduceat(DEN[o], first), len(Y))
    return out


def compare_xsim(start, end, val, ref_start, ref_end, ref_val, rtol=SIM_RTOL):
    """(start, end) key set identical; values within rtol."""
    assert len(start) == len(ref_start), "X-SIM pair count %d != %d" % (len(start), len(ref_start))
    assert np.array_equal(start, ref_start) and np.array_equal(end, ref_end), "X-SIM key sets differ"
    rel = np.abs(val - ref_val) / np.maximum(np.abs(ref_val), 1e-300)
    assert rel.size == 0 or rel.max() <= rtol, "xsim max rel err %g" % rel.max()
    return float(rel.max()) if rel.size else 0.0


def run_gpu_extend(tabs, lay, meta, top_m=10, **engine_kw):
    import torch
    from xmap_b200 import extend as X
    dm = to_device_meta(meta)
    plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), dm.has_S, dm.has_T)
    xe = X.XsimEngine(plan, top_m, **engine_kw)
    res = xe.run()
    s, e, v = xe.emit(res)
    torch.cuda.synchronize()
    return plan, xe, res, (s.cpu().numpy(), e.cpu().numpy(), v.cpu().numpy())


def philox_uniforms(seed, n):
    """numpy port of the kernel's Philox4x32-10 uniform (counter = row, key = seed)."""
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    c = [np.arange(n, dtype=np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.uint64)]
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64((seed >> 32) & 0xFFFFFFFF)
    mask = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(M0) * c[0]; p1 = np.uint64(M1) * c[2]
        n0 = ((p1 >> np.uint64(32)) ^ c[1] ^ k0) & mask
        n1 = p1 & mask
        n2 = ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & mask
        n3 = p0 & mask
        c = [n0, n1, n2, n3]
        k0 = (k0 + np.uint64(W0)) & mask; k1 = (k1 + np.uint64(W1)) & mask
    hi = (c[0] >> np.uint64(5)).astype(np.float64); lo = (c[1] >> np.uint64(6)).astype(np.float64)
    return (hi * 67108864.0 + lo) / 9007199254740992.0


# --------------------------------------------------------------------------
# clean stage (SURVEY.md 8(f) #4)
# --------------------------------------------------------------------------
def clean_encoded_numpy(user, item, ts, n_users, t_lo, t_hi, num_atleast):
    """numpy restatement of what xmap_clean_records decides (baselinerClean.py:47-52, 62-97): a record survives if it is
    in the period, is the STRICTLY latest of its (user, item) pair -- the first seen winning ties -- and its user keeps
    at least num_atleast items.  Returns (keep uint8 [n], items per user int32 [n_users])."""
    user, item, ts = np.asarray(user), np.asarray(item), np.asarray(ts, dtype=np.float64)
    n = len(user)
    inp = (ts >= t_lo) & (ts < t_hi)
    keep = np.zeros(n, np.uint8)
    best = {}
    for r in np.flatnonzero(inp):
        k = (int(user[r]), int(item[r]))
        if k not in best or ts[r] > ts[best[k]]:
            best[k] = r
    per_user = np.zeros(max(n_users, 1), np.int32)
    for (u, _), r in best.items():
        per_user[u] += 1
    for (u, _), r in best.items():
        if per_user[u] >= num_atleast:
            keep[r] = 1
    return keep, per_user[:n_users]
