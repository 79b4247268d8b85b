"""User-based kNN (usersim.py, csrc/usersim.cu) against its definition: the item-based stage run on the transposed
profile (recsim.item_knn / predict with the user and item arrays exchanged), bit for bit on integer and half-star
profiles, where both inner products are exact; schedule invariance; edges; the top-N against a numpy host path."""
import numpy as np
import pytest
import torch

from tests import parity as PT

pytestmark = pytest.mark.gpu


def _profile(seed, nU=400, nI=300, n=6000, half=True, dup=0.05):
    rng = np.random.default_rng(seed)
    p = 1.0 / np.arange(1, nI + 1)
    item = rng.choice(nI, n, p=p / p.sum())
    user = rng.integers(0, nU, n)
    rating = rng.integers(1, 11 if half else 6, n) * (0.5 if half else 1.0)
    d = rng.choice(n, int(n * dup), replace=False)        # a synthetic record next to a real one
    user, item = np.concatenate([user, user[d]]), np.concatenate([item, item[d]])
    rating = np.concatenate([rating, rng.integers(1, 6, len(d)).astype(np.float64)])
    ts = rng.integers(0, 50, len(user))
    return user, item, rating, ts, nU, nI


def _tables_equal(a, b):
    return torch.equal(a.idx, b.idx) and torch.equal(a.sim, b.sim) and torch.equal(a.len, b.len)


@pytest.mark.parametrize("k", [1, 2, 10, 31, 32, 33, 64])
@pytest.mark.parametrize("half", [False, True])
def test_select_equals_item_knn_transposed(k, half):
    from xmap_b200 import recsim, usersim
    user, item, rating, _, nU, nI = _profile(3 + k, half=half)
    ref = recsim.item_knn(item, user, rating, nU, 50, k)
    got = usersim.user_knn(user, item, rating, nU, nI, 50, k)
    assert torch.equal(got.info, ref.info)
    assert _tables_equal(got.nb, ref.nb)
    assert got.products == ref.n_entries
    # schedules: every row as a warp, as a CTA, tiny tiles (many passes per row)
    for kw in (dict(shape="warp"), dict(shape="cta"), dict(shape="warp", tile=256), dict(shape="cta", tile=256)):
        assert _tables_equal(usersim.user_knn(user, item, rating, nU, nI, 50, k, **kw).nb, ref.nb), kw


@pytest.mark.parametrize("num_atleast", [3, 4, 5])
def test_significance_threshold_and_self_pairs(num_atleast):
    """n at N - 1, N, N + 1 (pairs of 4 co-ratings), duplicates giving self pairs, a one-record user, a one-rater item."""
    from xmap_b200 import recsim, usersim
    user = np.array([0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 5, 5])
    item = np.array([0, 1, 2, 3, 0, 1, 2, 3, 0, 0, 1, 4, 1, 5, 2])
    rating = np.array([1, 2, 3, 4, 5, 4, 3, 2, 3, 4, 1, 5, 2, 3, 4], dtype=np.float64)
    ref = recsim.item_knn(item, user, rating, 6, num_atleast, 6)
    got = usersim.user_knn(user, item, rating, 6, 6, num_atleast, 6)
    assert _tables_equal(got.nb, ref.nb)
    assert 2 in got.nb.idx[2, :got.nb.len[2]].tolist()          # user 2's two records on item 0: the self pair
    rs = recsim.cosine_item(item, user, rating, 6, num_atleast)
    pr = dict(privacy_epsilon=0.6, rpo=0.1, seed=5)
    a = usersim.user_knn(user, item, rating, 6, 6, num_atleast, 3, private=pr)
    b = recsim.item_knn(item, user, rating, 6, num_atleast, 3, private=pr)
    assert _tables_equal(a.nb, b.nb)
    assert int(rs.n.max()) >= 4


def test_private_equals_item_knn_transposed_and_blocks():
    from xmap_b200 import recsim, usersim
    user, item, rating, _, nU, nI = _profile(11)
    pr = dict(privacy_epsilon=0.8, rpo=0.1, seed=99)
    ref = recsim.item_knn(item, user, rating, nU, 50, 10, private=pr)
    got = usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=pr)
    assert _tables_equal(got.nb, ref.nb)
    small = usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=pr, budget=64 * 2000, tile=256)
    assert small.blocks > 5 and _tables_equal(small.nb, ref.nb)
    for shape in ("warp", "cta"):
        assert _tables_equal(usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=pr, shape=shape).nb, ref.nb)
    # injected uniforms, one per user with a pair
    have = int((torch.as_tensor(recsim.row_entries(item, user, nU)) > 0).sum())
    rng = np.random.default_rng(1)
    u = dict(privacy_epsilon=0.8, rpo=0.1, u_pick=rng.random(have), u_noise=rng.random(have))
    assert _tables_equal(usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=u).nb,
                         recsim.item_knn(item, user, rating, nU, 50, 10, private=u).nb)


def test_overflow_is_an_error():
    from xmap_b200 import _native, usersim
    user, item, rating, _, nU, nI = _profile(5)
    with pytest.raises(_native.NativeError, match="error 2"):
        usersim.user_knn(user, item, rating, nU, nI, 50, 10, private=dict(seed=1), emit_cap=2)


def test_users_subset_equals_full_run():
    from xmap_b200 import usersim
    user, item, rating, _, nU, nI = _profile(21)
    full = usersim.user_knn(user, item, rating, nU, nI, 50, 10)
    sel = torch.randperm(nU, generator=torch.Generator().manual_seed(0))[:77]
    part = usersim.user_knn(user, item, rating, nU, nI, 50, 10, users=sel)
    s = sel.cuda()
    assert torch.equal(part.nb.idx[s], full.nb.idx[s]) and torch.equal(part.nb.sim[s], full.nb.sim[s])
    rest = torch.ones(nU, dtype=torch.bool, device="cuda")
    rest[s] = False
    assert int(part.nb.len[rest].abs().sum()) == 0


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_golden_profiles_near_item_knn_transposed(name):
    """Synthetic-mean ratings: the fixed-point inner product is exact, the item path's fp64 sum is not; sim agrees to
    1e-12 relative and lists are equal except near-ties."""
    from xmap_b200 import recsim, usersim
    g = PT.load_golden(name + "_recsim")
    u, i, r = g["ae_user"], g["ae_item"], g["ae_rating"]
    nU, nI = int(u.max()) + 1, int(i.max()) + 1
    ref = recsim.item_knn(i, u, r, nU, int(g["num_atleast"]), 10)
    got = usersim.user_knn(u, i, r, nU, nI, int(g["num_atleast"]), 10)
    assert torch.equal(got.nb.len, ref.nb.len)
    diff = (got.nb.idx != ref.nb.idx).any(1)
    assert int(diff.sum()) <= max(1, nU // 100)
    same = ~diff
    a, b = got.nb.sim[same], ref.nb.sim[same]
    assert bool(((a - b).abs() <= 1e-12 * b.abs() + 1e-300).all())


def _host_top_n(user, item, rating, ts, nU, nI, nb, info, n, decay, alpha=0.03):
    """Every unrated item scored with the prediction formula, sorted by (score desc, index asc)."""
    out = []
    ln, idx, sim = nb.len.cpu().numpy(), nb.idx.cpu().numpy(), nb.sim.cpu().numpy()
    avg = info.cpu().numpy()[:, 0]
    recs = {}
    for q in range(len(user)):
        recs.setdefault((int(user[q]), int(item[q])), []).append(q)
    order = np.argsort(user, kind="stable")
    for u in range(nU):
        rated = {int(item[q]) for q in np.flatnonzero(user == u)}
        if ln[u] == 0:
            out.append([])
            continue
        sc = []
        for it in range(nI):
            if it in rated:
                continue
            ea, eb, et = [], [], []
            for r in range(ln[u]):
                v = int(idx[u, r])
                for q in order[np.flatnonzero(user[order] == v)]:
                    if int(item[q]) == it:
                        ea.append(sim[u, r] * (rating[q] - avg[v])); eb.append(abs(sim[u, r])); et.append(int(ts[q]))
            s = avg[u]
            if ea:
                if not decay:
                    sa = 0.0; sb = 0.0
                    for x, y in zip(ea, eb):
                        sa += x; sb += y
                    s = avg[u] + sa / sb
                else:
                    o = sorted(range(len(et)), key=lambda z: et[z])
                    e2 = [(ea[z], eb[z], et[z]) for z in o]
                    ranks, cur = [], 0
                    for z in range(len(e2)):
                        if z == 0 or e2[z][2] != e2[z - 1][2]:
                            cur += 1
                        ranks.append(cur)
                    top = cur + 1
                    sa = 0.0; sb = 0.0
                    for (x, y, _), rk in zip(e2, ranks):
                        f = float(torch.exp(torch.tensor(-alpha * (top - rk), dtype=torch.float64)))
                        sa += x * f; sb += y * f
                    s = avg[u] + sa / sb
            if s == s:
                sc.append((-s + 0.0, it, s))
        sc.sort()
        out.append([(it, s) for _, it, s in sc[:n]])
    return out


@pytest.mark.parametrize("decay", [False, True])
def test_top_n_equals_host_scoring(decay):
    from xmap_b200 import usersim
    user, item, rating, ts, nU, nI = _profile(31, nU=60, nI=40, n=700)
    knn = usersim.user_knn(user, item, rating, nU, nI, 50, 5)
    ref = _host_top_n(user, item, rating, ts, nU, nI, knn.nb, knn.info, 12, decay)
    for shape in (None, "warp", "cta"):
        top = usersim.top_n(user, item, rating, ts, nU, nI, knn, knn.nb, 12, decay=decay, shape=shape)
        ln, idx, sc = top.len.cpu().numpy(), top.idx.cpu().numpy(), top.score.cpu().numpy()
        for u in range(nU):
            assert [int(x) for x in idx[u, :ln[u]]] == [it for it, _ in ref[u]], (shape, u)
            if decay:       # device exp against torch's host exp: last-bit differences allowed
                np.testing.assert_allclose(sc[u, :ln[u]], [s for _, s in ref[u]], rtol=1e-13)
            else:
                assert np.array_equal(sc[u, :ln[u]], np.array([s for _, s in ref[u]]))


def test_prediction_equals_item_predict_transposed():
    from xmap_b200 import recsim, usersim
    user, item, rating, ts, nU, nI = _profile(41)
    ref = recsim.item_knn(item, user, rating, nU, 50, 10)
    got = usersim.user_knn(user, item, rating, nU, nI, 50, 10)
    rng = np.random.default_rng(0)
    tu, ti = rng.integers(0, nU, 3000), rng.integers(0, nI, 3000)
    a = usersim.predict(user, item, rating, ts, nI, got, got.nb, tu, ti)
    b = recsim.predict(item, user, rating, ts, nI, ref, ref.nb, ti, tu)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_facade_user_based_chain():
    """RecommenderSim("cosine_user") through the facades: similarity RDD, selection, prediction, top-N."""
    from datetime import datetime, timezone
    from xmap_b200.core import recommender as R
    from xmap_b200.rdd import LocalRDD
    user, item, rating, ts, nU, nI = _profile(51, nU=50, nI=30, n=500, dup=0.0)
    recs = [("u%03d" % u, "i%03d" % i, float(r), datetime.fromtimestamp(int(t), timezone.utc).replace(tzinfo=None))
            for u, i, r, t in zip(user, item, rating, ts)]
    tool = R.RecommenderSim("cosine_user", 50)
    ub, ib, ubd, ibd, uinfo, iinfo, sims = R.recommender_calculate_sim_pipeline(None, tool, recs)
    pairs = sims.collect()
    assert len(pairs) > 0 and all(len(k) == 2 for k, _ in pairs)
    nbd = R.recommender_privacy_pipeline(R.RecommenderPrivacy(5, 0.6, 0.1, seed=3), sims, False).collectAsMap()
    test = LocalRDD([("u000", [("i001", 4.0, recs[0][3]), ("i002", 3.0, recs[0][3])])])
    rec = R.RecommenderPrediction(0.03, "cosine_user")
    out = rec.user_based_recommendation(test, ubd, nbd, uinfo).collect()
    assert len(out) == 1 and len(out[0][1]) == 2
    mae = R.recommender_prediction_pipeline(rec, tool, test, nbd, ubd, ibd, uinfo, iinfo)
    assert ";" in mae
    top = R.recommend_top_n(nbd, 5).collect()
    assert len(top) == len({r[0] for r in recs})
    # the values are the user-based ones, not the item path's
    from xmap_b200 import usersim
    st = nbd.handle
    nU, nI = len(st.uids), len(st.iids)
    ref = usersim.user_knn(st.user, st.item, st.rating, nU, nI, 50, 5)
    assert _tables_equal(st.nb, ref.nb)
    p0, p1, _, _ = usersim.predict(st.user, st.item, st.rating, st.ts, nI, ref, ref.nb, [st.upos["u000"]] * 2,
                                   [st.ipos["i001"], st.ipos["i002"]])
    got = [e for e in out[0][1]]
    for q in range(2):
        assert (got[q] == () and p0[q] == -1) or (got[q][2] == p0[q] and got[q][3] == p1[q])
    t = usersim.top_n(st.user, st.item, st.rating, st.ts, nU, nI, ref, ref.nb, 5)
    for u, lst in top:
        r = st.upos[u]
        assert [(str(st.iids[t.idx[r, p]]), float(t.score[r, p])) for p in range(int(t.len[r]))] == lst


def _pairs_user(prof, cta, tile):
    from xmap_b200 import usersim
    rows = torch.arange(prof.n_users, dtype=torch.int64, device=prof.dev)
    stats = torch.zeros(3, dtype=torch.int64, device=prof.dev)
    err = torch.zeros(1, dtype=torch.int32, device=prof.dev)
    parts = [blk[1:] for blk in usersim._emit_blocks(prof, [(rows, cta)], 50, 1 << 30, tile, None, stats, err)]
    return [torch.cat([p[f] for p in parts]) for f in range(5)]


@pytest.mark.parametrize("crafted", [False, True])
def test_emitted_block_pairs_and_nan_first_rule(crafted):
    """Every emitted (u, v, n, sim, ls) equals recsim's pair kernel on the transposed profile, NaN pattern included.
    With finite ratings and true norms no deviation is NaN (norm_u >= |r| for each of u's records), so the crafted case
    sets each user's norm just below its largest |rating|: the records at that rating then give a NaN first deviation,
    and whether a pair's sensitivity is NaN depends on which entry is first (smallest item, then list position)."""
    from xmap_b200 import recsim, usersim
    user, item, rating, _, nU, nI = _profile(61, nU=200, nI=120, n=3000)
    ref = recsim._Profile(item, user, rating, nU, "cuda")
    prof = usersim.UserProfile(user, item, rating, nU, nI)
    if crafted:
        mx = torch.zeros(nU, dtype=torch.float64).index_reduce_(0, torch.as_tensor(user), torch.as_tensor(rating),
                                                                "amax", include_self=False).cuda()
        norm = torch.where(mx > 0, mx * 0.999, prof.info[:, 1])
        ref.info[:, 1] = norm
        prof.info[:, 1] = norm              # the fixed-point scale keeps the true norms' exponents: a bound suffices
    want = ref.pairs(0, nU, 50)
    for cta, tile in ((False, None), (True, None), (False, 256), (True, 256)):
        u, v, n, sim, ls = _pairs_user(prof, cta, tile)
        assert torch.equal(u.int(), want.i) and torch.equal(v, want.j) and torch.equal(n, want.n), (cta, tile)
        assert torch.equal(sim, want.sim), (cta, tile)
        assert torch.equal(torch.isnan(ls), torch.isnan(want.ls)), (cta, tile)
        ok = ~torch.isnan(ls)
        assert torch.equal(ls[ok], want.ls[ok]), (cta, tile)
    nan = int(torch.isnan(want.ls).sum())
    if crafted:         # both outcomes occur among pairs whose u has a record at its largest rating
        assert 0 < nan < int(want.ls.numel())
    else:
        assert nan == 0


def test_exact_ties_across_tiles():
    """300 users with the same records as user 0 tie exactly in |sim| with it; they are spread over the user axis, so
    with 256-user tiles the ties straddle tiles and the first k must be the smallest indices."""
    from xmap_b200 import recsim, usersim
    rng = np.random.default_rng(5)
    nU, nI = 2000, 50
    base_items, base_r = np.arange(6), np.array([1.0, 3.0, 2.0, 5.0, 4.0, 2.5])
    twins = np.sort(rng.choice(np.arange(1, nU), 300, replace=False))
    others = np.setdiff1d(np.arange(1, nU), twins)
    u = [np.zeros(6, np.int64)] + [np.full(6, t) for t in twins]
    i = [base_items] * (1 + len(twins))
    r = [base_r] * (1 + len(twins))
    ou = rng.choice(others, 3000)
    user = np.concatenate(u + [ou])
    item = np.concatenate(i + [rng.integers(6, nI, 3000)])          # the others never touch user 0's items
    rating = np.concatenate(r + [rng.integers(1, 6, 3000).astype(np.float64)])
    for k in (1, 10, 64):
        ref = recsim.item_knn(item, user, rating, nU, 50, k)
        for kw in (dict(shape="warp", tile=256), dict(shape="cta", tile=256), dict()):
            got = usersim.user_knn(user, item, rating, nU, nI, 50, k, **kw)
            assert _tables_equal(got.nb, ref.nb), ("tables", k, kw)
        row = got.nb.idx[0, :int(got.nb.len[0])].cpu().numpy()
        assert np.array_equal(row, twins[:k]), (k, row[:5])          # the twins tie at |sim| = 6 / 50


def test_top_n_tiled_item_axis_and_heavy_users():
    """A catalogue of 180 000 items (most without records) walked in tiles of 64 / 4 096 items, both shapes: the lists
    equal the untiled ones; users whose neighbours hold more than 2 048 records take the CTA shape by default."""
    from xmap_b200 import usersim
    rng = np.random.default_rng(71)
    nU, nI, d = 300, 200, 60                     # each user rates 60 distinct items (Zipf): no more than 128 matches
    p = 1.0 / np.arange(1, nI + 1)
    user = np.repeat(np.arange(nU), d)
    item = np.concatenate([rng.choice(nI, d, replace=False, p=p / p.sum()) for _ in range(nU)])
    rating = rng.integers(1, 11, nU * d) * 0.5
    ts = rng.integers(0, 50, nU * d)
    stride = 900
    item, nI = item * stride, nI * stride
    knn = usersim.user_knn(user, item, rating, nU, nI, 50, 40)      # 40 x up to 3 records of one (user, item) <= 128
    base = usersim.top_n(user, item, rating, ts, nU, nI, knn, knn.nb, 64)
    assert base.cta_users > 0 and base.warp_users >= 0
    for decay in (False, True):
        one = usersim.top_n(user, item, rating, ts, nU, nI, knn, knn.nb, 64, decay=decay)
        for kw in (dict(shape="warp", tile=64), dict(shape="cta", tile=64), dict(shape="cta", tile=4096),
                   dict(shape="warp")):
            got = usersim.top_n(user, item, rating, ts, nU, nI, knn, knn.nb, 64, decay=decay, **kw)
            assert torch.equal(got.idx, one.idx) and torch.equal(got.len, one.len), kw
            assert torch.equal(got.score.view(torch.int64), one.score.view(torch.int64)), kw
    # the unrated items nobody near rated follow at avg_u, in index order, after the scored ones that beat it
    with pytest.raises(ValueError):
        usersim.top_n(user, item, rating, None, nU, nI, knn, knn.nb, 10)


def test_evaluate_user_based_equals_facade(tmp_path):
    """evaluate with RecommenderSim("cosine_user") against the facade chain it mirrors (TZ=UTC), both selections."""
    from tests import test_gpu_evaluate as TE
    from oracle.make_golden_cleansplit import utc
    from xmap_b200 import evaluate
    from xmap_b200.core import (BaselinerSim, ExtendSim, Generator, RecommenderPrediction, RecommenderPrivacy,
                                RecommenderSim, baseliner_calculate_sim_pipeline, extender_pipeline,
                                generator_pipeline, recommend_top_n, recommender_calculate_sim_pipeline,
                                recommender_prediction_pipeline, recommender_privacy_pipeline)
    from xmap_b200 import ingest
    with utc():
        paths = TE._synth_files(str(tmp_path), 11)

    def tools():
        return (BaselinerSim("adjust_cosine", 5), ExtendSim(10),
                Generator(1, 0.6, "adjust_cosine", 0.1, private_mode="exp_mech", seed=20261022),
                RecommenderSim("cosine_user", 5), RecommenderPrivacy(10, 0.6, 0.1, seed=77))
    for private in (False, True):
        with utc():
            cs, ct, sp = TE._tools(TE._cfg(**dict(TE.CFG, num_left=2)))
            tr, te = ingest.clean_split_pipeline(None, cs, ct, sp, paths[0], paths[1], False)
            sim, ext, gen, rsim, priv = tools()
            xs = extender_pipeline(None, None, sim, ext, baseliner_calculate_sim_pipeline(None, sim, tr))
            out = recommender_calculate_sim_pipeline(None, rsim, generator_pipeline(gen, tr, xs, private))
            simpair = recommender_privacy_pipeline(priv, out[6], private).collectAsMap()
            rp = RecommenderPrediction(0.03, "cosine_user")
            pred = rp.user_based_recommendation(te, out[2], simpair, out[4]).collect()
            mae = recommender_prediction_pipeline(rp, rsim, te, simpair, out[2], out[3], out[4], out[5])
            tops = dict(recommend_top_n(simpair, 10).collect())
            A = TE._arrays(paths, 2)
            sim, ext, gen, rsim, priv = tools()
            ev = evaluate.evaluate(A, sim, ext, gen, private, rsim, priv, private)
        p0, p1 = ev.pred_nodecay.cpu().numpy(), ev.pred_decay.cpu().numpy()
        flat = [e for _, lst in pred for e in lst]
        assert len(flat) == len(p0)
        for q, e in enumerate(flat):
            if e == ():
                assert p0[q] == -1.0 and p1[q] == -1.0, q
            else:
                assert e[2] == p0[q] and e[3] == p1[q], q
        assert ev.counts["predicted"] == sum(e != () for e in flat) > 0
        assert str(ev.mae_nodecay) + "; " + str(ev.mae_decay) == mae
        mine = TE._lists(A, ev)
        compared = 0
        for uid, lst in mine.items():
            if uid in tops:
                assert lst == tops[uid], uid
                compared += 1
        assert compared > 0
