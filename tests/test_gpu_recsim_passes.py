"""GPU: RecommenderSim in blocks of item rows (recsim.pair_passes / cosine_item / item_knn).  Every pass plan gives
the bit pattern of the one-pass result: pairs, counts, similarities, local sensitivities (NaNs included), entry
counts, neighbour tables (non-private and private) and predictions."""
import numpy as np
import pytest
import torch

from tests import parity as PT

pytestmark = pytest.mark.gpu


def _dup_profile():
    """The profile of test_gpu_recsim.test_recsim_vs_restatement_with_duplicates."""
    rng = np.random.default_rng(17)
    nU, nI, n = 3000, 500, 60000
    p_item = 1.0 / np.arange(1, nI + 1); p_item /= p_item.sum()
    user = rng.integers(0, nU, n); item = rng.choice(nI, n, p=p_item)
    rating = rng.integers(1, 11, n) * 0.5
    dup = rng.choice(n, n // 20, replace=False)
    user = np.concatenate([user, user[dup]]); item = np.concatenate([item, item[dup]])
    rating = np.concatenate([rating, rng.integers(1, 11, len(dup)) * 0.5 + 0.25])
    o = np.argsort(user, kind="stable")
    return dict(user=user[o], item=item[o], rating=rating[o], ts=np.arange(len(o)), n_users=nU, n_items=nI)


def _zipf_profile():
    """Zipf items, power users of 1 200 and 2 500 records (repeated items: self pairs, double entries), synthetic
    records next to real ones, users listed out of order, three items with a single record (one of them from a user
    with no other record), an item whose one rating overflows its squared norm (the pairs of a single-record item
    with it have a NaN first leave-one-out deviation: a NaN local sensitivity) and an item nobody rated."""
    rng = np.random.default_rng(5)
    nU, nI = 2000, 400
    pop = 1.0 / np.arange(1, nI + 1) ** 0.9
    pop[nI - 5:] = 0.0
    pop /= pop.sum()
    d = rng.integers(0, 20, nU)
    d[[3, 1200]] = [1200, 2500]
    d[7] = 1
    users, items, ratings = [], [], []
    for u in range(nU):
        if d[u] == 0:
            continue
        it = rng.choice(nI, d[u], replace=True, p=pop)
        r = rng.integers(1, 11, d[u]) * 0.5
        dup = np.flatnonzero(rng.random(d[u]) < 0.15)
        it, r = np.r_[it, it[dup]], np.r_[r, rng.integers(2, 9, len(dup)) * 0.5 + 0.25]
        if u in (10, 11):                                   # items nI - 5, nI - 4: a single record each
            it, r = np.r_[it, nI - 5 + u - 10], np.r_[r, 3.0]
        if u == 10:                                         # item nI - 2: norm2 = inf
            it, r = np.r_[it, nI - 2], np.r_[r, 1e160]
        if u == 7:                                          # item nI - 3: the only record of its user
            it = np.array([nI - 3])
        o = rng.permutation(len(it))
        users.append(np.full(len(it), u)); items.append(it[o]); ratings.append(r[o])
    user, item, rating = (np.concatenate(x) for x in (users, items, ratings))
    o = rng.permutation(len(user))
    o = o[np.argsort(user[o] % 7, kind="stable")]           # the list is not sorted by user; each user's order is kept
    user, item, rating = user[o], item[o], rating[o]
    return dict(user=user, item=item, rating=rating, ts=(rng.integers(0, 30, len(user)) * 86400).astype(np.int64),
                n_users=nU, n_items=nI)


PROFILES = {"dup": _dup_profile, "zipf": _zipf_profile}


@pytest.fixture(scope="module", params=sorted(PROFILES))
def case(request):
    from xmap_b200 import recsim
    p = PROFILES[request.param]()
    p["name"] = request.param
    p["row_ent"] = recsim.row_entries(p["user"], p["item"], p["n_items"])
    p["one"] = recsim.cosine_item(p["user"], p["item"], p["rating"], p["n_items"], 50, budget=2 ** 62)
    return p


def _budget_for(row_ent, passes):
    """The smallest budget whose plan has at most `passes` blocks."""
    from xmap_b200 import recsim
    lo, hi = int(row_ent.max()) * recsim.ENTRY_BYTES, int(row_ent.sum()) * recsim.ENTRY_BYTES
    while lo < hi:
        mid = (lo + hi) // 2
        if len(recsim.pass_plan(row_ent, mid)) - 1 <= passes:
            hi = mid
        else:
            lo = mid + 1
    assert len(recsim.pass_plan(row_ent, lo)) - 1 == passes
    return lo


def _bits(t):
    return t.contiguous().view(torch.int64) if t.dtype == torch.float64 else t


def _same(a, b, fields):
    for f in fields:
        x, y = getattr(a, f), getattr(b, f)
        assert torch.equal(_bits(x), _bits(y)), f


def _same_recsim(a, b):
    _same(a, b, ("i", "j", "n", "sim", "ls", "info"))
    assert a.n_entries == b.n_entries


def test_one_pass_profile(case):
    R = case["one"]
    assert R.n_entries == int(case["row_ent"].sum()) == int(R.n.sum())
    assert int((R.i == R.j).sum()) > 100
    if case["name"] == "zipf":
        assert bool(torch.isnan(R.ls).any()) and not bool(torch.isnan(R.sim).any())


@pytest.mark.parametrize("passes", [1, 2, 7])
def test_cosine_item_any_budget(case, passes):
    from xmap_b200 import recsim
    p = case
    R = recsim.cosine_item(p["user"], p["item"], p["rating"], p["n_items"], 50, budget=_budget_for(p["row_ent"], passes))
    _same_recsim(R, p["one"])


def test_cosine_item_one_row_per_pass(case):
    from xmap_b200 import recsim
    p = case
    prof = recsim._Profile(p["user"], p["item"], p["rating"], p["n_items"], "cuda")
    parts = [prof.pairs(i, i + 1, 50) for i in range(p["n_items"])]
    R = recsim.RecSim(*(torch.cat([getattr(x, f) for x in parts]) for f in ("i", "j", "n", "sim", "ls")), prof.info,
                      sum(x.n_entries for x in parts))
    _same_recsim(R, p["one"])
    assert [x.n_entries for x in parts] == p["row_ent"].tolist()


def test_item_knn_matches_one_pass(case):
    from xmap_b200 import recsim
    p = case
    R, nI = p["one"], p["n_items"]
    args = (p["user"], p["item"], p["rating"], nI, 50)
    budget = _budget_for(p["row_ent"], 7)
    rng = np.random.default_rng(3)
    n_have = int((p["row_ent"] > 0).sum())
    up, un = rng.random(n_have), rng.random(n_have)
    # test users with at most 100 records: a prediction gathers at most 128 matching profile records, and a power
    # user's records on 10 neighbours can exceed that (the kernel then reports error 4 on both paths alike)
    d = np.bincount(p["user"], minlength=p["n_users"])
    light = np.flatnonzero((d > 0) & (d <= 100))
    tu = torch.as_tensor(light[rng.integers(0, len(light), 20000)], dtype=torch.int32)
    ti = torch.as_tensor(rng.integers(0, nI, 20000), dtype=torch.int32)
    for k in (1, 10, 64):
        knn = recsim.item_knn(*args, k=k, budget=budget)
        assert knn.passes == 7 and knn.n_entries == R.n_entries and knn.max_row_entries == int(p["row_ent"].max())
        _same(knn.nb, recsim.neighbors(R, nI, k), ("idx", "sim", "len"))
        assert torch.equal(_bits(knn.info), _bits(R.info))
        if k == 10:
            want = recsim.predict(p["user"], p["item"], p["rating"], p["ts"], p["n_users"], R, recsim.neighbors(R, nI, k), tu, ti)
            got = recsim.predict(p["user"], p["item"], p["rating"], p["ts"], p["n_users"], knn, knn.nb, tu, ti)
            assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])
    for priv in (dict(u_pick=up, u_noise=un), dict(seed=11), dict(privacy_epsilon=1.3, rpo=0.2, seed=12)):
        knn = recsim.item_knn(*args, k=10, private=priv, budget=budget)
        kw = dict(priv)
        u_pick, u_noise = kw.pop("u_pick", None), kw.pop("u_noise", None)
        want = recsim.private_neighbors(R, nI, 10, u_pick=u_pick, u_noise=u_noise, **kw)
        _same(knn.nb, want, ("idx", "sim", "len"))
        assert int(knn.nb.len.sum()) == n_have
    with pytest.raises(ValueError):
        recsim.item_knn(*args, k=10, private=dict(u_pick=up[1:], u_noise=un), budget=budget)


def test_row_over_budget_raises(case):
    from xmap_b200 import recsim
    p = case
    big = int(torch.argmax(p["row_ent"]))
    budget = int(p["row_ent"][big]) * recsim.ENTRY_BYTES - 1
    for fn in (recsim.cosine_item, recsim.item_knn):
        with pytest.raises(ValueError, match="item row %d has %d co-rating entries" % (big, int(p["row_ent"][big]))):
            fn(p["user"], p["item"], p["rating"], p["n_items"], 50, budget=budget)


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_goldens_through_item_knn(name):
    """The reference's neighbour tables and predictions (tests/golden/*_recpred.npz) and, where minted, its private
    draws (*_recpriv.npz) through item_knn under a budget of several passes."""
    from xmap_b200 import recsim
    g = PT.load_golden(name + "_recpred")
    nI = int(max(g["ae_item"].max(), g["test_item"].max(), g["nb_idx"].max())) + 1
    nU = int(max(g["ae_user"].max(), g["test_user"].max())) + 1
    K = int(g["mapping_range"])
    args = (g["ae_user"], g["ae_item"], g["ae_rating"], nI, int(g["num_atleast"]))
    row_ent = recsim.row_entries(g["ae_user"], g["ae_item"], nI)
    budget = _budget_for(row_ent, 3)
    R = recsim.cosine_item(*args)
    knn = recsim.item_knn(*args, k=K, budget=budget)
    assert knn.passes == 3
    _same(knn.nb, recsim.neighbors(R, nI, K), ("idx", "sim", "len"))
    ln, idx = knn.nb.len.cpu().numpy(), knn.nb.idx.cpu().numpy()
    has = np.flatnonzero(ln)
    assert np.array_equal(has, g["nb_item"]) and np.array_equal(ln[has], np.diff(g["nb_ptr"]))
    same = [np.array_equal(idx[it, :ln[it]], g["nb_idx"][g["nb_ptr"][q]:g["nb_ptr"][q + 1]]) for q, it in enumerate(g["nb_item"])]
    assert sum(not s for s in same) <= 1                   # as test_gpu_recsim: at most one near-tie reorders a list
    p0, p1, _, _ = recsim.predict(g["ae_user"], g["ae_item"], g["ae_rating"], g["ae_ts"], nU, knn, knn.nb,
                                  g["test_user"], g["test_item"])
    near = 0 if all(same) else 1
    assert int((p0.cpu().numpy() != g["pred_nodecay"]).sum()) <= near
    assert int((p1.cpu().numpy() != g["pred_decay"]).sum()) <= near
    if name in ("adj_low_overlap", "cos_half_ratings"):                # the cases with private draws minted
        gp, g0 = PT.load_golden(name + "_recpriv"), PT.load_golden(name)
        nI = len(g0["iids"])
        knn = recsim.item_knn(gp["ae_user"], gp["ae_item"], gp["ae_rating"], nI, int(gp["num_atleast"]),
                              k=int(gp["mapping_range"]), budget=_budget_for(recsim.row_entries(gp["ae_user"], gp["ae_item"], nI), 3),
                              private=dict(privacy_epsilon=float(gp["epsilon"]), rpo=float(gp["rpo"]),
                                           u_pick=gp["u_pick"], u_noise=gp["u_noise"]))
        ln, idx, sim = knn.nb.len.cpu().numpy(), knn.nb.idx.cpu().numpy()[:, 0], knn.nb.sim.cpu().numpy()[:, 0]
        has = np.flatnonzero(ln)
        assert np.array_equal(has, gp["item"]) and np.array_equal(idx[has], gp["chosen"])
        np.testing.assert_allclose(sim[has], gp["noisy_sim"], rtol=1e-9, atol=1e-12)


def test_pipeline_never_materialises_the_pairs():
    """recommender_calculate_sim_pipeline -> recommender_privacy_pipeline computes no pair record unless the
    similarity RDD is collected, and the records it gives when collected are cosine_item's."""
    from datetime import datetime
    from xmap_b200 import recsim
    from xmap_b200.rdd import LocalRDD
    from xmap_b200.core import (RecommenderSim, RecommenderPrivacy, recommender_calculate_sim_pipeline,
                                recommender_privacy_pipeline)
    g = PT.load_golden("adj_low_overlap_recpred")
    profile = LocalRDD([("u%d" % u, "i%d" % i, float(r), datetime.utcfromtimestamp(int(t)))
                        for u, i, r, t in zip(g["ae_user"], g["ae_item"], g["ae_rating"], g["ae_ts"])])
    out = recommender_calculate_sim_pipeline(None, RecommenderSim("cosine_item", int(g["num_atleast"])), profile)
    sims = out[6]
    recommender_privacy_pipeline(RecommenderPrivacy(int(g["mapping_range"]), 0.6, 0.1), sims, False).collectAsMap()
    assert sims._records is None
    state = sims.handle
    R = recsim.cosine_item(state.user, state.item, state.rating, len(state.iids), int(g["num_atleast"]))
    got = sims.collect()
    assert len(got) == int(R.i.numel())
    i, j, s = R.i.cpu().numpy(), R.j.cpu().numpy(), R.sim.cpu().numpy()
    assert all(k == (str(state.iids[i[q]]), str(state.iids[j[q]])) and v[0] == s[q] for q, (k, v) in enumerate(got))
