"""GPU: recsim.top_n against a brute force over every (user, item) pair built on restate.recommender_predict(raw=True),
with the order the top-N contract fixes: score descending, then the smaller item index, NaN scores left out, rated
items left out.  No-decay scores are bit-equal; decay scores agree within 1e-13 relative (CUDA's exp may differ from
libm's by an ulp), and lists may differ only where two scores lie within that tolerance."""
import numpy as np
import pytest
import torch

from oracle import restate as RE
from tests import parity as PT
from tests.test_gpu_recsim_passes import _dup_profile, _zipf_profile

pytestmark = pytest.mark.gpu

N_EMPTY = 3          # user indices past the last profile user, with no records
REL = 1e-13


def _dup():
    """The duplicate-record profile, plus a user who rated every item and one who rated all but items 0, 1, 2."""
    p = _dup_profile()
    nU, nI = p["n_users"], p["n_items"]
    extra_u = np.r_[np.full(nI, nU), np.full(nI - 3, nU + 1)]
    extra_i = np.r_[np.arange(nI), np.arange(3, nI)]
    p["user"], p["item"] = np.r_[p["user"], extra_u], np.r_[p["item"], extra_i]
    p["rating"] = np.r_[p["rating"], np.full(len(extra_u), 3.5)]
    p["ts"] = np.arange(len(p["user"]))
    p["n_users"] = nU + 2
    return p


def _zipf():
    """The Zipf profile with its power users, each user's records on one item cut to the first 12 in list order, so
    that no candidate gathers more than 128 entries from tables of 10 neighbours (the unthinned power users exceed
    the prediction's cap; test_errors covers that)."""
    p = _zipf_profile()
    key = p["user"].astype(np.int64) * p["n_items"] + p["item"]
    o = np.argsort(key, kind="stable")
    first = np.r_[True, key[o][1:] != key[o][:-1]]
    start = np.maximum.accumulate(np.where(first, np.arange(len(o)), 0))
    keep = np.zeros(len(o), bool)
    keep[o] = (np.arange(len(o)) - start) < 12
    for f in ("user", "item", "rating", "ts"):
        p[f] = p[f][keep]
    return p


PROFILES = {"dup": _dup, "zipf": _zipf}


def _tables(p, k):
    from xmap_b200 import recsim
    args = (p["user"], p["item"], p["rating"], p["n_items"], 50)
    return recsim.item_knn(*args, k=k) if k > 1 else recsim.item_knn(*args, k=1, private=dict(seed=3))


def _flat(nb):
    ln, idx, sim = (x.cpu().numpy() for x in (nb.len, nb.idx, nb.sim))
    ptr = np.zeros(len(ln) + 1, np.int64)
    ptr[1:] = np.cumsum(ln)
    m = np.arange(idx.shape[1])[None, :] < ln[:, None]
    return ptr, idx[m], sim[m], ln


def _brute(p, knn, users, alpha=0.03):
    """user -> (items with a neighbour list, raw no-decay scores, raw decay scores, the user's rated items)."""
    ptr, fidx, fsim, ln = _flat(knn.nb)
    has = np.flatnonzero(ln)
    avg = knn.info[:, 0].cpu().numpy()
    users = np.asarray(users)
    tu, ti = np.repeat(users, len(has)), np.tile(has, len(users))
    rounded = RE.bound_rating                 # the raw values are wanted; a NaN one cannot be rounded
    RE.bound_rating = lambda x: -2.0 if x != x else rounded(x)
    try:
        out = RE.recommender_predict(p["user"], p["item"], p["rating"], p["ts"], ptr, fidx, fsim, avg, tu, ti,
                                     np.zeros(len(tu)), alpha, raw=True)
    finally:
        RE.bound_rating = rounded
    r0, r1 = out[4].reshape(len(users), -1), out[5].reshape(len(users), -1)
    rated = {}
    for u, i in zip(p["user"], p["item"]):
        rated.setdefault(int(u), set()).add(int(i))
    return {int(u): (has, r0[q], r1[q], rated.get(int(u), set())) for q, u in enumerate(users)}


def _rank(items, scores, rated, n):
    ok = ~np.isin(items, np.fromiter(rated, np.int64, len(rated))) & ~np.isnan(scores)
    it, sc = items[ok], scores[ok]
    o = np.lexsort((it, -sc))
    return it[o][:n], sc[o][:n]


def _bounds(p, nb):
    from xmap_b200 import recsim
    rev_ptr, _ = recsim.reverse_index(nb)
    cnt = (rev_ptr[1:] - rev_ptr[:-1]).cpu().numpy()
    return np.bincount(p["user"], weights=cnt[p["item"]], minlength=p["n_users"] + N_EMPTY)


def _check(res, bf, n, decay):
    """Compare the lists of the brute-forced users; returns the count of near-ties that reorder a list."""
    idx, score, ln = res.idx.cpu().numpy(), res.score.cpu().numpy(), res.len.cpu().numpy()
    near = 0
    for u, (items, r0, r1, rated) in bf.items():
        want_i, want_s = _rank(items, r1 if decay else r0, rated, n)
        L = len(want_i)
        assert ln[u] == L, (u, ln[u], L)
        assert (idx[u, L:] == -1).all() and np.isnan(score[u, L:]).all()
        if not decay:
            assert np.array_equal(idx[u, :L], want_i), u
            assert np.array_equal(score[u, :L].view(np.int64), want_s.view(np.int64)), u
            continue
        got_i, got_s = idx[u, :L], score[u, :L]
        np.testing.assert_allclose(got_s, want_s, rtol=REL, atol=0)
        for q in np.flatnonzero(got_i != want_i):       # a swap is only allowed between scores within the tolerance
            near += 1
            assert abs(want_s[q] - got_s[q]) <= REL * abs(want_s[q]) + 1e-300, (u, q)
    return near


@pytest.fixture(scope="module", params=sorted(PROFILES))
def case(request):
    p = PROFILES[request.param]()
    p["name"] = request.param
    rng = np.random.default_rng(11)
    out = {}
    for k in (10, 1):
        knn = _tables(p, k)
        b = _bounds(p, knn.nb)
        from xmap_b200 import _native as N
        heavy = np.flatnonzero(b > N.TOPN_WARP_BOUND)
        present = np.unique(p["user"])
        sample = np.unique(np.r_[heavy, rng.choice(present, 300, replace=False), present[-2:],
                                 np.arange(p["n_users"], p["n_users"] + N_EMPTY)])
        out[k] = (knn, _brute(p, knn, sample), heavy)
    p["tables"] = out
    return p


@pytest.mark.parametrize("decay", [False, True])
@pytest.mark.parametrize("k", [10, 1])
def test_top_n_matches_brute_force(case, k, decay):
    from xmap_b200 import recsim
    p = case
    knn, bf, heavy = p["tables"][k]
    near = 0
    for n in (1, 10, 64):
        res = recsim.top_n(p["user"], p["item"], p["rating"], p["ts"], p["n_users"] + N_EMPTY, knn, knn.nb, n, decay=decay)
        near += _check(res, bf, n, decay)
        assert res.cta_users == len(heavy)
        if k == 10:
            assert res.warp_users > 0 and res.cta_users > 0          # both launch shapes run
        assert res.candidates <= res.visits
    print("%s k=%d decay=%s: %d users checked, %d near-ties" % (p["name"], k, decay, len(bf), near))
    assert near <= 3


def test_special_users(case):
    """Users without records get the top of the average order; a user who rated every item with neighbours gets an
    empty list, one who rated all but three items at most three."""
    from xmap_b200 import recsim
    p = case
    knn = p["tables"][10][0]
    nU = p["n_users"]
    res = recsim.top_n(p["user"], p["item"], p["rating"], p["ts"], nU + N_EMPTY, knn, knn.nb, 64)
    ln = knn.nb.len.cpu().numpy()
    avg = knn.info[:, 0].cpu().numpy()
    has = np.flatnonzero((ln > 0) & ~np.isnan(avg))
    want = has[np.lexsort((has, -avg[has]))][:64]
    for u in range(nU, nU + N_EMPTY):
        assert np.array_equal(res.idx[u, :res.len[u]].cpu().numpy(), want)
    if p["name"] == "dup":
        assert int(res.len[nU - 2]) == 0 and int(res.len[nU - 1]) <= 3


def test_tiled_item_axis():
    """The dup profile with its items spread over 1.2 M indices (more than one bitmap tile): the same lists, mapped."""
    from xmap_b200 import recsim
    p = _dup()
    stride = 2400
    sparse = p["item"] * stride + 7
    nI = p["n_items"] * stride
    knn = recsim.item_knn(p["user"], p["item"], p["rating"], p["n_items"], 50, k=10)
    knn_s = recsim.item_knn(p["user"], sparse, p["rating"], nI, 50, k=10)
    for decay in (False, True):
        a = recsim.top_n(p["user"], p["item"], p["rating"], p["ts"], p["n_users"], knn, knn.nb, 64, decay=decay)
        b = recsim.top_n(p["user"], sparse, p["rating"], p["ts"], p["n_users"], knn_s, knn_s.nb, 64, decay=decay)
        assert b.cta_users > 0
        assert torch.equal(a.len, b.len)
        assert torch.equal(torch.where(a.idx >= 0, a.idx * stride + 7, a.idx), b.idx)
        assert torch.equal(a.score.view(torch.int64), b.score.view(torch.int64))
        assert (a.visits, a.candidates) == (b.visits, b.candidates)


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_golden_profiles(name):
    """The AlterEgo profiles of the reference's prediction goldens, every user, both variants."""
    from xmap_b200 import recsim
    g = PT.load_golden(name + "_recpred")
    nI = int(max(g["ae_item"].max(), g["test_item"].max(), g["nb_idx"].max())) + 1
    nU = int(max(g["ae_user"].max(), g["test_user"].max())) + 1
    p = dict(user=g["ae_user"], item=g["ae_item"], rating=g["ae_rating"], ts=g["ae_ts"], n_users=nU, n_items=nI)
    knn = recsim.item_knn(p["user"], p["item"], p["rating"], nI, int(g["num_atleast"]), k=int(g["mapping_range"]))
    bf = _brute(p, knn, np.arange(nU))
    for decay in (False, True):
        for n in (1, 10, 64):
            res = recsim.top_n(p["user"], p["item"], p["rating"], p["ts"], nU, knn, knn.nb, n, decay=decay)
            assert _check(res, bf, n, decay) <= 1


def test_errors():
    from xmap_b200 import recsim, _native as N
    p = _dup()
    knn = _tables(p, 10)
    args = (p["user"], p["item"], p["rating"], p["ts"])
    for n in (0, 65, 2.5):
        with pytest.raises(ValueError):
            recsim.top_n(*args, p["n_users"], knn, knn.nb, n)
    with pytest.raises(ValueError):
        recsim.top_n(*args, p["n_users"] - 1, knn, knn.nb, 10)        # a user index past n_users
    bad = p["item"].copy()
    bad[0] = p["n_items"]
    with pytest.raises(ValueError):
        recsim.top_n(p["user"], bad, p["rating"], p["ts"], p["n_users"], knn, knn.nb, 10)
    # a user with 130 records on item 0: every candidate listing item 0 gathers more than 128 entries
    rev_ptr, _ = recsim.reverse_index(knn.nb)
    assert int(rev_ptr[1] - rev_ptr[0]) > 0
    u = np.r_[p["user"], np.full(130, p["n_users"])]
    i = np.r_[p["item"], np.zeros(130, np.int64)]
    r = np.r_[p["rating"], np.full(130, 4.0)]
    t = np.r_[p["ts"], np.arange(130)]
    with pytest.raises(N.NativeError, match="error 4"):
        recsim.top_n(u, i, r, t, p["n_users"] + 1, knn, knn.nb, 10)


def test_recommend_top_n_facade():
    """recommend_top_n on a profile passed through the pipeline functions: top_n's lists, as id strings."""
    from datetime import datetime
    from xmap_b200 import recsim
    from xmap_b200.rdd import LocalRDD
    from xmap_b200.core import (RecommenderSim, RecommenderPrivacy, recommender_calculate_sim_pipeline,
                                recommender_privacy_pipeline, recommend_top_n)
    g = PT.load_golden("adj_low_overlap_recpred")
    profile = LocalRDD([("u%d" % u, "i%d" % i, float(r), datetime.utcfromtimestamp(int(t)))
                        for u, i, r, t in zip(g["ae_user"], g["ae_item"], g["ae_rating"], g["ae_ts"])])
    out = recommender_calculate_sim_pipeline(None, RecommenderSim("cosine_item", int(g["num_atleast"])), profile)
    simpair = recommender_privacy_pipeline(RecommenderPrivacy(int(g["mapping_range"]), 0.6, 0.1), out[6], False).collectAsMap()
    st = simpair.handle
    for decay in (False, True):
        got = recommend_top_n(simpair, 10, decay=decay).collect()
        res = recsim.top_n(st.user, st.item, st.rating, st.ts, len(st.uids), st.knn, st.nb, 10, decay=decay)
        idx, score, ln = res.idx.cpu().numpy(), res.score.cpu().numpy(), res.len.cpu().numpy()
        assert [uid for uid, _ in got] == [str(s) for s in st.uids] == sorted(str(s) for s in st.uids)
        for u, (uid, lst) in enumerate(got):
            assert lst == [(str(st.iids[idx[u, q]]), float(score[u, q])) for q in range(ln[u])]
        assert sum(len(lst) for _, lst in got) > 0
    with pytest.raises(TypeError):
        recommend_top_n({}, 10)
