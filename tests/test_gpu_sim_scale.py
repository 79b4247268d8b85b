"""GPU: the similarity stage on rating scales other than 1-5 stars.

The encoder accepts any rating that is exact in binary32, so the fixed-point inner product of the
accumulate kernels has to hold its accuracy for outliers, play counts, negative scales and user
populations many octaves apart.  Every case is checked against oracle/restate.py (kept pairs, n, mutu,
frac and labels exact, sim within SIM_RTOL, neighbour lists) and, on a sample of pairs that includes
every neighbour-list pair, against an exact rational inner product with the error bound of DESIGN.md
section 3.2."""
import math

import numpy as np
import pytest

from tests import parity as PT

pytestmark = pytest.mark.gpu

METHODS = ("adjust_cosine", "cosine")
N_ATLEAST, K = 50, 10
E_FIELD_MAX = 127                        # largest per-item exponent the 7-bit entry field holds


# --------------------------------------------------------------------------
# case builders
# --------------------------------------------------------------------------
def _meta(n_items):
    """Two domains (S: / T:), half of the items each, ids built like the synthetic workloads'."""
    from xmap_b200 import synth
    from xmap_b200.encode import item_codes
    half = (n_items + 1) // 2
    pc, dc, ct, hs, ht = item_codes([synth.item_id(g, half, ("S:", "T:")) for g in range(n_items)])
    return dict(prefix_code=pc, dom_code=dc, contains=ct, has_S=hs, has_T=ht)


def _pairs(rng, n_users, n_items, n_draws, items=None):
    """Deduplicated (user, item) draws, items Zipf-popular (1/rank) over `items` (default all)."""
    items = np.arange(n_items) if items is None else np.asarray(items)
    p = 1.0 / np.arange(1, len(items) + 1)
    user = rng.integers(0, n_users, n_draws)
    item = items[rng.choice(len(items), n_draws, p=p / p.sum())]
    return user, item


def _case(user, item, rating, n_users, n_items):
    key = np.unique(np.asarray(user, np.int64) * n_items + np.asarray(item, np.int64), return_index=True)[1]
    user, item = np.asarray(user, np.int64)[key], np.asarray(item, np.int64)[key]
    rating = np.asarray(rating, np.float64)[key]
    assert np.array_equal(rating.astype(np.float32).astype(np.float64), rating)     # exact in binary32
    return dict(user=user, item=item, rating=rating, n_users=n_users, n_items=n_items, meta=_meta(n_items))


def _half_stars(rng, n):
    return rng.integers(2, 11, n) * 0.5


def half_star_case(seed=1, scale=1.0, outlier=None, outlier_user=False):
    """1 500 users, 200 items, half-star ratings times `scale`; `outlier` replaces one rating, or with
    outlier_user every rating of the most active user."""
    rng = np.random.default_rng(seed)
    u, i = _pairs(rng, 1500, 200, 20000)
    case = _case(u, i, _half_stars(rng, len(u)), 1500, 200)
    case["rating"] = case["rating"] * scale
    if outlier is not None:
        if outlier_user:
            top = np.bincount(case["user"]).argmax()
            case["rating"][case["user"] == top] = outlier
        else:
            case["rating"][0] = outlier
    return case


def play_count_case(seed=2):
    """Integer play counts, log-normal in [1, 2^20]; three items with more than 2^16 raters."""
    rng = np.random.default_rng(seed)
    n_users, n_items = 70000, 300
    u, i = _pairs(rng, n_users, n_items, 200000, items=np.arange(3, n_items))
    pop = rng.random((n_users, 3)) < 0.96
    pu, pi = np.nonzero(pop)
    u, i = np.concatenate([u, pu]), np.concatenate([i, pi])
    r = np.clip(np.rint(rng.lognormal(2.0, 2.2, len(u))), 1, 2 ** 20)
    return _case(u, i, r, n_users, n_items)


def quarter_step_case(seed=3):
    """Ratings on -10 ... 10 in quarter steps (zero and negative values included)."""
    rng = np.random.default_rng(seed)
    u, i = _pairs(rng, 1500, 200, 20000)
    return _case(u, i, rng.integers(-40, 41, len(u)) * 0.25, 1500, 200)


def two_population_case(lo_exp, hi_exp, seed=4):
    """Two user populations on disjoint items of both domains: the first rates the even items with half
    stars times 2^lo_exp, the second the odd items with half stars times 2^hi_exp.  (A pair of items from
    different populations would have a cosine near 2^(lo_exp - hi_exp): nothing to resolve.)"""
    rng = np.random.default_rng(seed)
    nu = 1500
    ua, ia = _pairs(rng, nu // 2, 200, 10000, items=np.arange(0, 200, 2))
    ub, ib = _pairs(rng, nu // 2, 200, 10000, items=np.arange(1, 200, 2))
    u = np.concatenate([ua, ub + nu // 2])
    i = np.concatenate([ia, ib])
    scale = np.where(u < nu // 2, 2.0 ** lo_exp, 2.0 ** hi_exp)
    return _case(u, i, _half_stars(rng, len(u)) * scale, nu, 200)


# --------------------------------------------------------------------------
# exact reference
# --------------------------------------------------------------------------
def _exponents(den):
    """E with 2^(E-1) <= den < 2^E for den > 0 (frexp); None for den == 0."""
    return [math.frexp(float(d))[1] if d > 0 else None for d in den]


def _clamp_bits(den):
    """Bits by which each item's exponent is raised to fit the 7-bit field (0 for most items)."""
    E = _exponents(den)
    live = [e for e in E if e is not None]
    base = max(live) - E_FIELD_MAX if live else 0
    return np.array([max(base - e, 0) if e is not None else 0 for e in E], np.int64)


def _exact_inner(a, b):
    """sum(a * b) of two float64 arrays, exactly, as (integer, power-of-two exponent)."""
    if len(a) == 0:
        return 0, 0
    ma, ea = np.frexp(a)
    mb, eb = np.frexp(b)
    ia = (ma * 2.0 ** 53).astype(np.int64)
    ib = (mb * 2.0 ** 53).astype(np.int64)
    e = ea.astype(np.int64) + eb.astype(np.int64) - 106
    e0 = int(e.min())
    return sum(int(x) * int(y) << int(s) for x, y, s in zip(ia.tolist(), ib.tolist(), (e - e0).tolist())), e0


def check_exact(case, method, out, n_sample=2000, seed=0):
    """|sim_gpu - sim_exact| <= 1e-12 |sim_exact| + (2^-52 + n 2^-61 2^(d_i + d_j)) min(n, N) / N on a sample
    of the kept pairs of either side plus every pair of a neighbour list; sim_exact divides the exact
    inner product of the fp64 centred values by the den of restate.user_item_stats; d = clamp bits."""
    from fractions import Fraction
    from oracle import restate as RS
    nI, P = case["n_items"], out["P"]
    o = np.lexsort((case["item"], case["user"]))
    user, item, r = case["user"][o], case["item"][o], case["rating"][o]
    st = RS.user_item_stats(user, item, r, case["n_users"], nI)
    val = r - st["mu"][user] if method == "adjust_cosine" else r
    den = st["adj_norm2"] if method == "adjust_cosine" else st["norm2"]
    gpu_den = out["lay"].item_stats[:, 2 if method == "adjust_cosine" else 1].cpu().numpy()
    d = _clamp_bits(gpu_den)
    oc = np.lexsort((user, item))                                   # by item, then user
    c_user, c_val = user[oc], val[oc]
    ptr = np.searchsorted(item[oc], np.arange(nI + 1))

    g = out["pairs"]
    gi, gj, gs = (g[k].cpu().numpy() for k in ("i", "j", "sim"))
    gsim = dict(zip((gi * nI + gj).tolist(), gs.tolist()))
    cand = np.union1d((gi * nI + gj)[gi < gj], (P["i"] * nI + P["j"])[P["i"] < P["j"]])
    rng = np.random.default_rng(seed)
    keys = set(rng.choice(cand, min(n_sample, len(cand)), replace=False).tolist()) if len(cand) else set()
    tl, ti = out["tabs"].tab_len.cpu().numpy(), out["tabs"].tab_idx.cpu().numpy()
    for it in range(nI):
        for slot in range(2):
            for j in ti[it, slot, :tl[it, slot]].tolist():
                keys.add(min(it, j) * nI + max(it, j))
    for key in sorted(keys):
        a, b = divmod(key, nI)
        ua, ub = c_user[ptr[a]:ptr[a + 1]], c_user[ptr[b]:ptr[b + 1]]
        _, pa, pb = np.intersect1d(ua, ub, assume_unique=True, return_indices=True)
        n = len(pa)
        m, e = _exact_inner(c_val[ptr[a]:ptr[a + 1]][pa], c_val[ptr[b]:ptr[b + 1]][pb])
        dd = Fraction(float(den[a])) * Fraction(float(den[b]))
        exact = 0.0
        if dd != 0 and m != 0:
            exact = float(Fraction(m) * Fraction(2) ** e / dd * min(n, N_ATLEAST) / N_ATLEAST)
        bound = 1e-12 * abs(exact) + (2.0 ** -52 + n * 2.0 ** (-61 + int(d[a] + d[b]))) * min(n, N_ATLEAST) / N_ATLEAST
        got = gsim.get(key, 0.0)
        assert gsim.get(b * nI + a, 0.0) == got
        err = abs(got - exact)
        assert err <= bound, "pair (%d, %d) n=%d: gpu %.17g exact %.17g (err %.3g > bound %.3g)" % (
            a, b, n, got, exact, err, bound)


def check_case(case, method, **engine_kw):
    out = PT.check_sim_against_restatement(case, method, N_ATLEAST, K, **engine_kw)
    check_exact(case, method, out)
    return out


def _same(a, b):
    for k in ("i", "j", "sim", "mutu", "n", "frac"):
        assert np.array_equal(a["pairs"][k].cpu().numpy(), b["pairs"][k].cpu().numpy()), k
    for t in ("tab_idx", "tab_sim", "tab_len", "tab_mutu", "tab_n", "row_flags", "row_npairs"):
        assert np.array_equal(getattr(a["tabs"], t).cpu().numpy(), getattr(b["tabs"], t).cpu().numpy()), t


def _kinds(out):
    return [k for k, _ in out["tabs"].stats["accumulate"]]


# --------------------------------------------------------------------------
# tests
# --------------------------------------------------------------------------
@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("outlier,whole_user", [(1000.0, False), (65536.0, False), (2.0 ** 24, False),
                                                (65536.0, True)])
def test_one_outlier_rating(method, outlier, whole_user):
    """Half stars plus one extreme rating (or one user who gives only that rating): the outlier must not
    coarsen the inner products of the pairs whose ratings are all 1-5 stars."""
    check_case(half_star_case(outlier=outlier, outlier_user=whole_user), method)


@pytest.mark.parametrize("method", METHODS)
def test_play_counts_with_popular_items(method):
    """Heavy-tailed play counts; the three items with more than 2^16 raters are direct-indexed rows
    (hashed rows refuse that many) whose class is 17, where wide products meet long sums."""
    from xmap_b200 import engine as E
    case = play_count_case()
    out = check_case(case, method)
    eng = out["eng"]
    cnt = out["lay"].item_stats[:, 3]
    big = cnt > 65536
    assert int(big.sum()) == 3
    rtop = (case["n_items"] - 1 - eng.ord).long()
    h = ((eng.tri_work * 4 + 2) // 3).clamp(min=32)
    assert bool((rtop[big] <= h[big]).all())
    assert "accumulate_split" in _kinds(out) and E.SPLIT_RATERS <= 65536


@pytest.mark.parametrize("method", METHODS)
def test_quarter_steps_with_negative_ratings(method):
    check_case(quarter_step_case(), method)


@pytest.mark.parametrize("method", METHODS)
def test_populations_2_to_the_plus_minus_40(method):
    """Two populations 80 octaves apart: the small one's pairs must keep their own resolution."""
    check_case(two_population_case(-40, 40), method)


@pytest.mark.parametrize("method", METHODS)
def test_exponent_spread_just_past_the_field_is_clamped(method):
    """Item norms spread over a few more than 127 octaves: the smallest items are clamped up by a few
    bits and the bar still holds."""
    case = two_population_case(-62, 64)
    out = check_case(case, method)
    den = out["lay"].item_stats[:, 2 if method == "adjust_cosine" else 1].cpu().numpy()
    E = [e for e in _exponents(den) if e is not None]
    assert E_FIELD_MAX < max(E) - min(E) <= E_FIELD_MAX + 16, max(E) - min(E)
    assert _clamp_bits(den).max() > 0


@pytest.mark.parametrize("method", METHODS)
def test_exponent_spread_far_past_the_field_raises(method):
    from xmap_b200 import engine as E
    case = two_population_case(-100, 100)
    lay = E.build_layout(case["user"], case["item"], case["rating"], case["n_users"], case["n_items"])
    with pytest.raises(ValueError):
        E.SimEngine(lay, PT.to_device_meta(case["meta"]), method, N_ATLEAST, K)


@pytest.mark.parametrize("method", METHODS)
def test_power_of_two_scaling_is_bit_identical(method):
    """Scaling every rating by 2^s moves each item's exponent by s and the pair's scale with it, so the
    tables, pairs, n, mutu and sim do not change by a bit."""
    ref = check_case(half_star_case(), method)
    for s in (-60, -20, 20, 60):
        case = half_star_case(scale=2.0 ** s)
        _same(ref, dict(zip(("lay", "eng", "tabs", "pairs"),
                            PT.run_gpu_sim(case["user"], case["item"], case["rating"], case["n_users"],
                                           case["n_items"], case["meta"], method, N_ATLEAST, K))))


@pytest.mark.parametrize("method", METHODS)
def test_every_accumulate_path_is_bit_identical(method, monkeypatch):
    """The 65 536 outlier case through warp rows, CTA rows, split rows, global-memory tables and exact
    list sizing: the split and global paths add raw 64-bit words, so they see the same scale."""
    from xmap_b200 import engine as E
    case = half_star_case(outlier=65536.0)
    warp = check_case(case, method)
    assert all(k.endswith("_t32") for k in _kinds(warp)), _kinds(warp)
    gmem = check_case(case, method, max_smem_cells=64)
    assert any("accumulate_g" in k for k in _kinds(gmem))
    exact = check_case(case, method, rec_budget=0)
    assert exact["eng"].exact_sizing
    with monkeypatch.context() as mp:
        mp.setattr(E, "_threads_for_cells", lambda c: 256)
        cta = check_case(case, method)
    assert not any(k.endswith("_t32") for k in _kinds(cta)), _kinds(cta)
    with monkeypatch.context() as mp:
        mp.setattr(E, "SPLIT_RATERS", 64)
        mp.setattr(E, "SPLIT_SEG", 96)
        split = check_case(case, method)
    assert dict(split["tabs"].stats["accumulate"]).get("accumulate_split", 0) > 5
    for other in (gmem, exact, cta, split):
        _same(warp, other)
