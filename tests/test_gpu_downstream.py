"""GPU parity of the stages after X-SIM at the shapes the reference goldens do not reach: AlterEgo mean-merge over
groups of many sources, the source -> target inversion under collisions, non-private neighbour selection with long
rows, |sim| ties and K up to XMAP_KMAX, and item-based prediction with tied times, missing neighbour lists and the
128-entry cap.  Every check is against oracle/restate.py (bit for bit where the operation order is the same)."""
from datetime import datetime, timedelta

import numpy as np
import pytest

from oracle import restate as RS

pytestmark = pytest.mark.gpu

DAY = 86400
T0 = 1356998400          # 2013-01-01 00:00:00 UTC


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.int64)


# ---------------------------------------------------------------------------------------------------------------
# AlterEgo generation (generate.cu: invert_kernel, mapped_keys_kernel, merge_kernel)
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ae_case():
    """Ratings with merge groups of every size: a band of 200 popular sources maps onto 3 targets (150 / 40 / 10
    sources each), the other sources map one-to-one or not at all.  Ratings are arbitrary float32 values, times are
    day-granular (ties), for a third of the users they decrease with the item index, and a quarter of the users
    rate nothing (user 0, the last user and many in between)."""
    rng = np.random.default_rng(3)
    nU, nI = 4000, 4000
    active = np.sort(rng.choice(np.arange(1, nU - 1), 3000, replace=False))
    w = np.ones(nI); w[100:300] = 40.0; w /= w.sum()
    d = rng.integers(1, 40, len(active)); d[rng.choice(len(active), 25, replace=False)] = rng.integers(300, 700, 25)
    users, items, times = [], [], []
    for u, n in zip(active, d):
        it = np.sort(rng.choice(nI, size=n, replace=False, p=w))
        t = T0 + rng.integers(0, 60, n) * DAY
        if u % 3 == 0:
            t = np.sort(t)[::-1]                   # later items rated earlier: earliest time != smallest source's
        users.append(np.full(n, u)); items.append(it); times.append(t)
    user, item, ts = (np.concatenate(x) for x in (users, items, times))
    o = rng.permutation(len(user))                 # input order is not the CSR order
    user, item, ts = user[o].astype(np.int32), item[o].astype(np.int32), ts[o].astype(np.int64)
    rating = rng.uniform(0.5, 5.0, len(user)).astype(np.float32)
    mp = np.full(nI, -1, dtype=np.int64)
    mp[100:250], mp[250:290], mp[290:300] = 0, nI - 1, 2500
    rest = np.arange(300, 2000)
    keep = rest[rng.random(len(rest)) < 0.8]
    pool = np.setdiff1d(np.arange(2001, nI - 1), [2500])
    mp[keep] = rng.choice(pool, len(keep), replace=False)
    return dict(user=user, item=item, rating=rating, ts=ts, n_users=nU, n_items=nI, mapping=mp)


def _gpu_alterego(case, mapping, lay=None):
    import torch
    from xmap_b200 import engine as E, generate as G
    if lay is None:
        lay = E.build_layout(case["user"], case["item"], case["rating"], case["n_users"], case["n_items"])
    out = G.build_alterego(lay, case["ts"], torch.as_tensor(mapping, dtype=torch.int32, device="cuda"))
    return lay, [t.cpu().numpy() for t in out]


def _check_alterego(case, mapping, got):
    ref = RS.build_alterego(case["user"], case["item"], case["rating"], case["ts"], mapping,
                            np.zeros(case["n_items"], dtype=bool))
    ou, oi, orr, ot = got
    assert np.array_equal(ou, ref["user"]) and np.array_equal(oi, ref["item"])
    assert np.array_equal(_bits(orr), _bits(ref["rating"])), "merged means differ"
    assert np.array_equal(ot, ref["ts"]), "merged times differ"
    return ref


def test_alterego_merge_groups_vs_restatement(ae_case):
    """Means over groups of 1 to ~150 sources match bit for bit (a double sum of float32 values in [0.5, 5] is exact
    at these sizes, a float32 mean is not), and every group takes the time of its smallest source item."""
    c = ae_case
    lay, got = _gpu_alterego(c, c["mapping"])
    ref = _check_alterego(c, c["mapping"], got)
    # the data reach what the test is about
    m = c["mapping"][c["item"]] >= 0
    key = c["user"][m].astype(np.int64) * c["n_items"] + c["mapping"][c["item"][m]]
    _, first, size = np.unique(key, return_index=True, return_counts=True)
    assert size.max() >= 100 and (size == 1).sum() > 1000 and len(np.unique(size)) > 30
    ks = np.argsort(key, kind="stable")
    t_min = np.minimum.reduceat(c["ts"][m][ks], np.r_[0, np.cumsum(size)[:-1]])
    t_max = np.maximum.reduceat(c["ts"][m][ks], np.r_[0, np.cumsum(size)[:-1]])
    assert int((ref["ts"] != t_min).sum()) > 100 and int((t_min != t_max).sum()) > 1000
    assert {0, c["n_items"] - 1} <= set(np.unique(got[1]).tolist())
    ptr = lay.csr_ptr.cpu().numpy()
    empty = np.flatnonzero(np.diff(ptr) == 0)
    assert empty[0] == 0 and empty[-1] == c["n_users"] - 1 and len(empty) > 900
    print("alterego records", len(got[0]), "largest group", int(size.max()))


def test_alterego_edge_mappings(ae_case):
    """The all -1 mapping selects nothing (four empty tensors); a mapping of every item (targets included) merges
    across the whole profile."""
    c = ae_case
    lay, got = _gpu_alterego(c, np.full(c["n_items"], -1))
    assert all(len(t) == 0 for t in got)
    rng = np.random.default_rng(9)
    every = rng.integers(0, 60, c["n_items"])
    every[:5] = c["n_items"] - 1
    _, got = _gpu_alterego(c, every, lay)
    _check_alterego(c, every, got)
    assert len(got[0]) > 10000


def test_alterego_at_the_24_bit_item_limit():
    """n_items = 2^24, the largest layout build_layout accepts: sources and targets at 2^24 - 2 and 2^24 - 1 survive
    the 24-bit item field of the CSR entries and the (user, target) key."""
    top = 1 << 24
    user = np.array([0, 0, 0, 0, 2, 2, 2], dtype=np.int32)
    item = np.array([top - 1, 5, top - 2, 0, top - 2, 7, 5], dtype=np.int32)
    rating = np.array([1.5, 2.25, 4.75, 3.0, 0.5, 5.0, 1.0], dtype=np.float32)
    ts = np.array([10, 20, 30, 40, 50, 60, 70], dtype=np.int64)
    mp = np.full(top, -1, dtype=np.int64)
    mp[top - 2], mp[5], mp[top - 1], mp[7] = top - 1, top - 1, top - 2, 0
    case = dict(user=user, item=item, rating=rating, ts=ts, n_users=3, n_items=top)
    _, got = _gpu_alterego(case, mp)
    ref = _check_alterego(case, mp, got)
    assert ref["item"].tolist() == [top - 2, top - 1, 0, top - 1]
    # user 2's merge onto 2^24 - 1 takes the time of source 5 (70), not the earlier one of source 2^24 - 2 (50)
    assert ref["rating"].tolist() == [1.5, 3.5, 5.0, 0.75] and ref["ts"].tolist() == [10, 20, 60, 70]


def test_invert_mapping_collisions():
    """Many target rows choose the same source, some choose nothing (-1): the largest target wins (assist.py:215)."""
    import torch
    from xmap_b200 import generate as G
    rng = np.random.default_rng(12)
    nI = 20000
    rows = np.sort(rng.choice(nI, 6000, replace=False))
    chosen = rng.choice(np.r_[np.arange(40), nI - 1], len(rows))
    chosen[rng.random(len(rows)) < 0.1] = -1
    chosen[-1] = -1                                  # the largest row maps nothing
    dev = torch.device("cuda")
    mp = G.invert_mapping(torch.as_tensor(rows, dtype=torch.int32, device=dev),
                          torch.as_tensor(chosen, dtype=torch.int32, device=dev), nI).cpu().numpy()
    ref = RS.invert_mapping(rows, chosen, nI)
    assert np.array_equal(mp, ref)
    assert int((ref >= 0).sum()) == 41 and ref[nI - 1] >= 0


def test_generator_build_alterego_facade_merges():
    """Generator.build_alterEgo with string ids, datetimes and a mapping dict on a merge-heavy profile: the kept
    "T:" ratings then the merged records, equal to the restatement mapped back to strings."""
    from xmap_b200.core import Generator
    from xmap_b200.rdd import LocalRDD
    rng = np.random.default_rng(21)
    nS, nT, nU = 400, 100, 300
    iids = ["bk%04dS:" % s for s in range(nS)] + ["mv%04dT:" % t for t in range(nT)]      # sorted: canonical order
    uids = ["u%04d" % u for u in range(nU)]
    w = np.ones(nS + nT); w[:60] = 25.0; w /= w.sum()
    recs, user, item, rating, times = [], [], [], [], []
    for u in range(nU):
        # the last user rates every item, so that the canonical index of an id is its position in iids
        its = np.arange(nS + nT) if u == nU - 1 else np.sort(rng.choice(nS + nT, rng.integers(1, 80), replace=False, p=w))
        lst = []
        for i in its:
            r = float(np.float32(rng.uniform(0.5, 5.0)))
            t = datetime(2013, 1, 1) + timedelta(days=int(rng.integers(0, 20)))
            lst.append((iids[i], r, t))
            user.append(u); item.append(i); rating.append(r); times.append(t)
        recs.append((uids[u], lst))
    mp = np.full(nS + nT, -1, dtype=np.int64)
    mp[:60] = nS + rng.integers(0, 3, 60)            # 60 popular sources onto the first 3 targets
    one = np.arange(60, nS)[rng.random(nS - 60) < 0.7]
    mp[one] = nS + 3 + rng.choice(nT - 3, len(one))    # the rest: mostly distinct targets, some shared
    mapping_dict = {iids[s]: iids[t] for s, t in enumerate(mp) if t >= 0}
    got = Generator(1, 0.6, "adjust_cosine", 0.1).build_alterEgo(LocalRDD(recs), mapping_dict).collect()
    user, item = np.array(user), np.array(item)
    has_T = np.array(["T:" in s for s in iids])
    ref = RS.build_alterego(user, item, np.array(rating, dtype=np.float32), np.arange(len(user)), mp, has_T)
    want = [(uids[u], iids[i], float(r), times[t]) for u, i, r, t in zip(ref["user"], ref["item"], ref["rating"], ref["ts"])]
    assert [(a, b, float(c), d) for a, b, c, d in got] == want
    m = mp[item] >= 0
    _, size = np.unique(user[m] * 1000 + mp[item[m]], return_counts=True)
    assert size.max() >= 10 and int((size > 1).sum()) > 100 and int((~ref["synthetic"]).sum()) > 100


# ---------------------------------------------------------------------------------------------------------------
# Non-private neighbour selection (recsim.cu: recsim_neighbors_kernel)
# ---------------------------------------------------------------------------------------------------------------
def _recsim_of(i, j, sim, n_items):
    import torch
    from xmap_b200 import recsim
    dev = torch.device("cuda")
    return recsim.RecSim(torch.as_tensor(i, dtype=torch.int32, device=dev), torch.as_tensor(j, dtype=torch.int32, device=dev),
                         torch.ones(len(i), dtype=torch.int64, device=dev), torch.as_tensor(sim, dtype=torch.float64, device=dev),
                         torch.zeros(len(i), dtype=torch.float64, device=dev),
                         torch.zeros((n_items, 3), dtype=torch.float64, device=dev), len(i))


def _check_neighbors(nb, P, n_items, K):
    ptr, idx, val = RS.recommender_neighbors(P, n_items, K)
    ln, ni, ns = nb.len.cpu().numpy(), nb.idx.cpu().numpy(), nb.sim.cpu().numpy()
    assert ni.shape == (n_items, K)
    assert np.array_equal(ln, np.diff(ptr)), "list lengths differ (K=%d)" % K
    live = np.arange(K)[None, :] < ln[:, None]
    assert np.array_equal(ni[live], idx), "neighbour indices differ (K=%d)" % K
    assert np.array_equal(_bits(ns[live]), _bits(val)), "neighbour similarities differ (K=%d)" % K
    assert (ni[~live] == -1).all() and (_bits(ns[~live]) == 0).all()


def test_neighbors_long_rows_and_sign_ties_vs_restatement():
    """Rows of 0 .. 5000 pairs (one, a few and several warp strides), sims on a coarse grid with random signs (so
    |sim| ties across signs, +0.0 and -0.0 are common), a self pair in every row; K from 1 to XMAP_KMAX."""
    from xmap_b200 import _native as N, recsim
    rng = np.random.default_rng(5)
    nI = 5200
    lens = np.zeros(nI, dtype=np.int64)
    special = [0, 1, 2, 31, 32, 33, 63, 64, 65, 128, 1000, 5000]
    at = rng.choice(nI, 300, replace=False)
    lens[at[:12]] = special
    lens[at[12:]] = rng.integers(0, 100, 288)
    lens[nI - 1] = 70
    i = np.repeat(np.arange(nI), lens)
    j = np.concatenate([np.sort(np.r_[it, rng.choice(np.delete(np.arange(nI), it), n - 1, replace=False)])
                        for it, n in enumerate(lens) if n > 0])
    sim = rng.integers(0, 6, len(i)) / 8.0 * rng.choice([-1.0, 1.0], len(i))
    assert ((sim == 0) & np.signbit(sim)).any() and ((sim == 0) & ~np.signbit(sim)).any()
    P = dict(i=i, j=j, sim=sim)
    R = _recsim_of(i, j, sim, nI)
    for K in (1, 10, 32, 33, 64):
        _check_neighbors(recsim.neighbors(R, nI, K), P, nI, K)
    for K in (0, N.KMAX + 1):
        with pytest.raises(N.NativeError, match="k out of range"):
            recsim.neighbors(R, nI, K)


# ---------------------------------------------------------------------------------------------------------------
# RecommenderSim + prediction on an AlterEgo-like profile (recsim.cu: fill / pair / neighbors / predict kernels)
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def profile():
    """~3 000 users on 600 items (the last 8 never rated): half-star ratings, synthetic merged means next to real
    ratings of the same (user, item) with equal or different times, day-granular times in a 30-day window, a block
    of users whose records all share one time, users without records, and power users with 1 000 and 3 000 records
    (repeated items)."""
    rng = np.random.default_rng(11)
    nU, nI = 3000, 600
    pop = 1.0 / np.arange(1, nI + 1) ** 0.8
    pop[nI - 8:] = 0.0
    pop /= pop.sum()
    d = rng.integers(0, 25, nU)
    d[[17, 1501]], d[2222] = 1000, 3000
    users, items, ratings, times = [], [], [], []
    for u in range(nU):
        n = int(d[u])
        if n == 0:
            continue
        it = rng.choice(nI, n, replace=n > 100, p=pop)
        r = rng.integers(1, 11, n) * 0.5
        t = T0 + rng.integers(0, 30, n) * DAY
        if 400 <= u < 500:
            t[:] = T0 + 7 * DAY                      # every record of these users at one time
        dup = np.flatnonzero(rng.random(n) < 0.2)    # a synthetic (merged) record next to the real one
        r_syn = np.array([rng.integers(1, 11, rng.integers(2, 5)).mean() * 0.5 for _ in dup])
        t_syn = np.where(rng.random(len(dup)) < 0.5, t[dup], T0 + rng.integers(0, 30, len(dup)) * DAY)
        o = rng.permutation(n + len(dup))
        users.append(np.full(n + len(dup), u)); items.append(np.r_[it, it[dup]][o])
        ratings.append(np.r_[r, r_syn][o]); times.append(np.r_[t, t_syn][o])
    user, item, rating, ts = (np.concatenate(x) for x in (users, items, ratings, times))
    return dict(user=user, item=item.astype(np.int64), rating=rating, ts=ts.astype(np.int64), n_users=nU, n_items=nI)


@pytest.fixture(scope="module")
def profile_sim(profile):
    from xmap_b200 import recsim
    p = profile
    return recsim.cosine_item(p["user"], p["item"], p["rating"], p["n_items"], 50)


def test_cosine_item_power_users_vs_restatement(profile, profile_sim):
    """Users with 1 000 and 3 000 records (up to 9e6 co-rating entries from one user: the combination unranking of
    recsim_fill_kernel far from small d), duplicates and self pairs: n exact, sim and local sensitivity to 1e-5."""
    p, R = profile, profile_sim
    P = RS.recommender_cosine_item(p["user"], p["item"], p["rating"], p["n_items"], 50)
    assert np.array_equal(R.i.cpu().numpy(), P["i"]) and np.array_equal(R.j.cpu().numpy(), P["j"])
    assert np.array_equal(R.n.cpu().numpy(), P["n"])
    np.testing.assert_allclose(R.sim.cpu().numpy(), P["sim"], rtol=1e-5, atol=0)
    ls, ok = R.ls.cpu().numpy(), ~np.isnan(P["ls"])
    assert np.array_equal(np.isnan(ls), ~ok)
    np.testing.assert_allclose(ls[ok], P["ls"][ok], rtol=1e-5, atol=1e-12)
    assert R.n_entries > 9_000_000 and int((P["i"] == P["j"]).sum()) > 100


def test_neighbors_of_cosine_item_at_kmax(profile, profile_sim):
    """The device's own RecSim at K = 64: the tables equal the restatement's selection from the same similarities."""
    from xmap_b200 import recsim
    R, nI = profile_sim, profile["n_items"]
    P = dict(i=R.i.cpu().numpy(), j=R.j.cpu().numpy(), sim=R.sim.cpu().numpy())
    nb = recsim.neighbors(R, nI, 64)
    _check_neighbors(nb, P, nI, 64)
    assert int((nb.len.cpu() == 64).sum()) > 300


def _tables(nb):
    ln, idx, sim = nb.len.cpu().numpy(), nb.idx.cpu().numpy(), nb.sim.cpu().numpy()
    live = np.arange(idx.shape[1])[None, :] < ln[:, None]
    return np.r_[0, np.cumsum(ln)], idx[live], sim[live], idx, ln


def _boundary(x):
    """x + 0.5 within 1e-9 of an integer: int(x + 0.5) may go either way once exp differs in the last bit."""
    y = x + 0.5
    return np.abs(y - np.round(y)) <= 1e-9


def _check_predict(p, R, nb, tu, ti, alpha, max_boundary):
    from xmap_b200 import recsim
    p0, p1, _, _ = recsim.predict(p["user"], p["item"], p["rating"], p["ts"], p["n_users"], R, nb, tu, ti, alpha=alpha)
    p0, p1 = p0.cpu().numpy(), p1.cpu().numpy()
    ptr, idx, sim, _, _ = _tables(nb)
    o0, o1, _, _, r0, r1 = RS.recommender_predict(p["user"], p["item"], p["rating"], p["ts"], ptr, idx, sim,
                                                  R.info[:, 0].cpu().numpy(), tu, ti, np.zeros(len(tu)), alpha, raw=True)
    assert np.array_equal(p0, o0), "no-decay predictions differ (alpha=%g)" % alpha
    edge = _boundary(r1)
    assert np.array_equal(p1[~edge], o1[~edge]), "decay predictions differ (alpha=%g)" % alpha
    assert (np.abs(p1[edge] - o1[edge]) <= 1.0).all()
    n_edge = int(edge.sum())
    print("alpha", alpha, "K", nb.idx.shape[1], "pairs", len(tu), "half-integer boundary cases", n_edge)
    assert n_edge <= max_boundary
    return p0, p1, o0, r0, r1


def test_predict_vs_restatement(profile, profile_sim):
    """~20 000 test pairs at K = 10 and 64, alpha = 0, 0.03 and 1: no-decay predictions identical everywhere (same
    operation order), decay predictions identical except where the unbounded value sits on a half-integer boundary.
    Covers items without a neighbour list (-1), users without a matching record (the bounded item average), tied
    times (shared ranks) and users whose records all share one time."""
    from xmap_b200 import recsim
    p, R = profile, profile_sim
    rng = np.random.default_rng(23)
    nU, nI = p["n_users"], p["n_items"]
    tu = rng.integers(0, nU, 20000)
    ti = rng.integers(0, nI, 20000)
    tu[:500] = rng.integers(400, 500, 500)           # the one-time block
    C = np.zeros((nU, nI), dtype=np.int64)
    np.add.at(C, (p["user"], p["item"]), 1)
    for K in (10, 64):
        nb = recsim.neighbors(R, nI, K)
        _, _, _, idx, ln = _tables(nb)
        live = np.arange(K)[None, :] < ln[ti][:, None]
        ent = (C[tu[:, None], np.maximum(idx[ti], 0)] * live).sum(1)
        ok = ent <= 128                              # more than 128 matching records is the kernel's error 4
        assert ok.mean() > 0.99
        u, it, ent = tu[ok], ti[ok], ent[ok]
        assert int((ln[it] == 0).sum()) > 50 and int(((ln[it] > 0) & (ent == 0)).sum()) > 1000
        assert int((ent >= 2).sum()) > 1000
        for alpha in (0.0, 0.03, 1.0):
            p0, p1, o0, r0, r1 = _check_predict(p, R, nb, u, it, alpha, max_boundary=20)
            assert (p0[ln[it] == 0] == -1).all()
            if alpha == 1.0:
                assert int((p0 != p1).sum()) > 20 and int(((r0 != r1) & ~np.isnan(r0)).sum()) > 1000


@pytest.fixture
def cap_case():
    """One user with two records on each of the 64 neighbours of test item 0: exactly 128 entries."""
    import torch
    from xmap_b200 import recsim
    dev = torch.device("cuda")
    nI, K = 70, 64
    rng = np.random.default_rng(31)
    nb_idx = np.full((nI, K), -1, dtype=np.int32); nb_idx[0] = np.arange(1, K + 1)
    nb_sim = np.zeros((nI, K)); nb_sim[0] = rng.integers(1, 9, K) / 8.0 * rng.choice([-1.0, 1.0], K)
    nb_len = np.zeros(nI, dtype=np.int32); nb_len[0] = K
    nb = recsim.Neighbors(torch.as_tensor(nb_idx, device=dev), torch.as_tensor(nb_sim, device=dev),
                          torch.as_tensor(nb_len, device=dev))
    info = np.zeros((nI, 3)); info[:, 0] = rng.integers(2, 9, nI) * 0.5 + 0.25      # never on a rounding boundary
    R = _recsim_of(np.zeros(1), np.zeros(1), np.zeros(1), nI)
    R.info = torch.as_tensor(info, device=dev)
    item = np.r_[np.arange(1, K + 1), np.arange(1, K + 1), 69]
    user = np.zeros(len(item), dtype=np.int64); user[-1] = 1
    rating = rng.integers(1, 11, len(item)) * 0.5
    ts = T0 + rng.integers(0, 10, len(item)) * DAY
    return dict(user=user, item=item, rating=rating, ts=ts, n_users=2, n_items=nI), R, nb


def test_predict_cap_at_128_entries(cap_case):
    """128 matching records succeed and match the restatement; a 129th raises NativeError (error 4, a flag the host
    turns into an exception); the next call on fresh inputs succeeds again."""
    from xmap_b200 import _native as N, recsim
    p, R, nb = cap_case
    tu, ti = np.array([0, 1, 0]), np.array([0, 0, 5])
    for alpha in (0.03, 1.0):
        p0, p1, o0, _, _ = _check_predict(p, R, nb, tu, ti, alpha, max_boundary=1)
        assert p0[2] == -1 and p0[0] >= 0
    over = dict(p, user=np.r_[p["user"], 0], item=np.r_[p["item"], 5], rating=np.r_[p["rating"], 4.0],
                ts=np.r_[p["ts"], T0])
    with pytest.raises(N.NativeError, match="error 4"):
        recsim.predict(over["user"], over["item"], over["rating"], over["ts"], 2, R, nb, tu, ti)
    _check_predict(p, R, nb, tu, ti, 0.03, max_boundary=1)


def test_predict_rejects_out_of_range_test_pairs(cap_case):
    """test_user outside [0, n_users) or test_item outside the neighbour tables raise ValueError before a launch."""
    from xmap_b200 import recsim
    p, R, nb = cap_case
    args = (p["user"], p["item"], p["rating"], p["ts"], 2, R, nb)
    for tu, ti in (([0, 2], [0, 0]), ([-1], [0]), ([0], [70]), ([1, 0], [0, -1]), ([2 ** 32], [0]), ([0], [0, 1])):
        with pytest.raises(ValueError):
            recsim.predict(*args, tu, ti)
    recsim.predict(*args, [1, 0], [69, 0])
