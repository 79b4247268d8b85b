"""GPU: explicit ALS (als.py, csrc/als.cu) against the numpy restatement of tests/als_exact.py, bit for bit: the
factors after every half-step, scores and top-N lists; the Philox init; the failing pivot; evaluate.evaluate_als and
the MLlib-shaped facade against the array calls."""
import math

import numpy as np
import pytest
import torch

from tests import als_exact as AX

pytestmark = pytest.mark.gpu
S = AX.S


def _case(seed, n_users=260, n_items=180, n_rand=3000):
    """Records with duplicate (user, item) pairs, fractional and zero / negative ratings, users and items with one
    record, items with S - 1, S, S + 1 and 3S + 1 records, a user with 2S + 3 records, and rows without any."""
    rng = np.random.default_rng(seed)
    u = rng.integers(0, n_users - 40, n_rand)
    i = rng.integers(0, n_items - 40, n_rand)
    u = np.r_[u, u[:200]]                                            # duplicates: the same (user, item) twice
    i = np.r_[i, i[:200]]
    parts_u, parts_i = [u], [i]
    for item, cnt in ((n_items - 40, S - 1), (n_items - 39, S), (n_items - 38, S + 1), (n_items - 37, 3 * S + 1)):
        parts_u.append(rng.integers(0, n_users - 40, cnt))
        parts_i.append(np.full(cnt, item))
    parts_u.append(np.full(2 * S + 3, n_users - 40))               # a heavy user (items repeat)
    parts_i.append(rng.integers(0, n_items - 40, 2 * S + 3))
    parts_u.append(np.arange(n_users - 39, n_users - 30))          # users with one record
    parts_i.append(rng.integers(0, n_items - 40, 9))
    parts_u.append(rng.integers(0, n_users - 40, 7))               # items with one record
    parts_i.append(np.arange(n_items - 36, n_items - 29))
    user = np.concatenate(parts_u).astype(np.int64)
    item = np.concatenate(parts_i).astype(np.int64)
    perm = rng.permutation(len(user))
    user, item = user[perm], item[perm]
    rating = rng.integers(-3, 16, len(user)) / 3.0                  # means such as 10/3, and 0.0
    return user, item, rating, n_users, n_items


def _init(seed, n_users, rank):
    """Injected initial factors with exact zeros of both signs (-0.0 products)."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n_users, rank)).astype(np.float32)
    X[::7, 0] = -0.0
    X[::5, rank - 1] = 0.0
    return X


def _eq(t, a):
    return torch.equal(t.cpu().view(torch.int32), torch.from_numpy(np.ascontiguousarray(a)).view(torch.int32))


CASES = [(r, lam) for r in (1, 2, 10, 31, 32, 33, 64) for lam in (0.01, 1.0)]


@pytest.mark.parametrize("rank,lam", CASES)
def test_train_equals_restatement(rank, lam):
    from xmap_b200 import als
    user, item, rating, nU, nI = _case(rank)
    X0 = _init(rank + 1, nU, rank)
    iters = 5 if rank <= 10 else 2
    want = AX.train(user, item, rating, nU, nI, X0, iters, lam)
    for it in range(1, iters + 1):
        m = als.train(torch.from_numpy(user), torch.from_numpy(item), torch.from_numpy(rating), nU, nI, rank, it, lam,
                      init=torch.from_numpy(X0))
        Y, X = want[it - 1]
        assert _eq(m.item_factors, Y), (rank, lam, it, "item")
        assert _eq(m.user_factors, X), (rank, lam, it, "user")
    cnt_u, cnt_i = np.bincount(user, minlength=nU), np.bincount(item, minlength=nI)
    assert np.array_equal(m.user_count.cpu().numpy(), cnt_u) and np.array_equal(m.item_count.cpu().numpy(), cnt_i)
    assert (cnt_i == 0).any() and (cnt_u == 0).any() and (cnt_i == 3 * S + 1).any()
    assert (m.item_factors[torch.from_numpy(cnt_i == 0).cuda()] == 0).all()


@pytest.mark.parametrize("rank", [3, 64])
def test_launch_split_same_bits(monkeypatch, rank):
    """The rows of a half-step cut into many normal / solve launches (down to one row each) give the same bits."""
    from xmap_b200 import als
    user, item, rating, nU, nI = _case(7)
    X0 = torch.from_numpy(_init(8, nU, rank))
    args = (torch.from_numpy(user), torch.from_numpy(item), torch.from_numpy(rating), nU, nI, rank, 2, 0.1)
    ref = als.train(*args, init=X0)
    P = rank * (rank + 1) // 2 + rank
    for per in (1, 3, 50):
        monkeypatch.setattr(als, "SCRATCH_BYTES", per * P * 8)
        got = als.train(*args, init=X0)
        assert torch.equal(got.user_factors, ref.user_factors) and torch.equal(got.item_factors, ref.item_factors)


def test_philox_init():
    from xmap_b200 import als
    for rank in (1, 10, 33, 64):
        a = als.init_factors(5000, rank, seed=12345)
        assert (a.double().norm(dim=1) - 1).abs().max().item() < 1e-6
        assert torch.equal(a, als.init_factors(5000, rank, seed=12345))
        assert not torch.equal(a, als.init_factors(5000, rank, seed=12346))
    assert torch.equal(als.init_factors(100, 4), als.init_factors(100, 4, seed=0))
    # the seed plays no part when init is injected
    user, item, rating, nU, nI = _case(2)
    X0 = torch.from_numpy(_init(3, nU, 6))
    args = (torch.from_numpy(user), torch.from_numpy(item), torch.from_numpy(rating), nU, nI, 6, 1, 0.1)
    a, b = als.train(*args, init=X0, seed=1), als.train(*args, init=X0, seed=2)
    assert torch.equal(a.user_factors, b.user_factors) and torch.equal(a.item_factors, b.item_factors)
    c, d = als.train(*args, seed=1), als.train(*args, seed=2)
    assert not torch.equal(c.user_factors, d.user_factors)


def test_zero_lambda_singular_row_raises():
    from xmap_b200 import als, _native
    rng = np.random.default_rng(4)
    nU, nI, rank = 60, 12, 3
    user = rng.integers(1, nU, 600)
    item = rng.integers(0, nI, 600)
    item[item == 5] = 6
    user, item = np.r_[user, 0], np.r_[item, 5]                       # item 5: one record, from user 0
    X0 = rng.standard_normal((nU, rank)).astype(np.float32)
    X0[0] = [1.0, 0.0, 0.0]                                            # A_5 = e0 e0^T: the second pivot is 0
    args = (torch.from_numpy(user), torch.from_numpy(item), torch.ones(len(user), dtype=torch.float64), nU, nI, rank, 1)
    with pytest.raises(_native.NativeError, match="item row 5 "):
        als.train(*args, 0.0, init=torch.from_numpy(X0))
    als.train(*args, 0.01, init=torch.from_numpy(X0))                  # lambda > 0: solvable


def test_predict_equals_restatement():
    from xmap_b200 import als
    user, item, rating, nU, nI = _case(11)
    m = als.train(torch.from_numpy(user), torch.from_numpy(item), torch.from_numpy(rating), nU, nI, 10, 2, 0.05,
                  seed=99)
    rng = np.random.default_rng(0)
    pu, pi = rng.integers(0, nU, 5000), rng.integers(0, nI, 5000)
    got = als.predict(m, torch.from_numpy(pu), torch.from_numpy(pi)).cpu().numpy()
    X, Y = m.user_factors.cpu().numpy(), m.item_factors.cpu().numpy()
    xn, yn = m.user_count.cpu().numpy(), m.item_count.cpu().numpy()
    want = AX.score(X, Y, xn, yn, pu, pi)
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
    nan = (xn[pu] == 0) | (yn[pi] == 0)
    assert nan.any() and np.isnan(got[nan]).all() and not np.isnan(got[~nan]).any()


def _model(seed, nU=150, nI=700, rank=10):
    """A hand-made model: random factors, rows without records, item rows duplicated (exact ties), zero item rows."""
    from xmap_b200 import als
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((nU, rank)).astype(np.float32)
    Y = rng.standard_normal((nI, rank)).astype(np.float32)
    Y[300:340] = Y[100:140]                                            # 40 exact ties, ordered by index
    Y[600:620] = 0.0
    Y[650:660] = -0.0
    xn, yn = rng.integers(1, 5, nU), rng.integers(1, 5, nI)
    xn[::17], yn[::23] = 0, 0
    X[xn == 0], Y[yn == 0] = 0.0, 0.0
    user = rng.integers(0, nU, 4000)
    item = rng.integers(0, nI, 4000)
    dev = torch.device("cuda")
    m = als.AlsModel(torch.from_numpy(X).to(dev), torch.from_numpy(Y).to(dev), torch.from_numpy(xn).to(dev),
                     torch.from_numpy(yn).to(dev), rank, 0.0, 0, None)
    return m, X, Y, xn, yn, user, item


def _check_lists(top, want, users, n):
    idx, score, ln = top.idx.cpu().numpy(), top.score.cpu().numpy(), top.len.cpu().numpy()
    for u in users:
        w = want[int(u)]
        assert ln[u] == len(w), u
        assert idx[u, :ln[u]].tolist() == [i for i, _ in w], u
        assert np.array_equal(score[u, :ln[u]].view(np.int64), np.array([s for _, s in w]).view(np.int64)), u
        assert (idx[u, ln[u]:] == -1).all() and np.isnan(score[u, ln[u]:]).all()


@pytest.mark.parametrize("n", [1, 10, 64])
@pytest.mark.parametrize("exclude", [True, False])
def test_top_n_equals_brute_force(n, exclude):
    from xmap_b200 import als
    m, X, Y, xn, yn, user, item = _model(n)
    nU, nI = X.shape[0], Y.shape[0]
    rated = {}
    for a, b in zip(user, item):
        rated.setdefault(int(a), set()).add(int(b))
    rated = {k: np.array(sorted(v)) for k, v in rated.items()} if exclude else None
    top = als.top_n(m, n, torch.from_numpy(user), torch.from_numpy(item), exclude_rated=exclude)
    want = AX.top_n(X, Y, xn, yn, n, range(nU), np.arange(nI), rated)
    _check_lists(top, want, range(nU), n)
    assert (top.len.cpu().numpy()[xn == 0] == 0).all()
    # ties: some user lists both copies of a duplicated item, the smaller index first
    if n == 64 and not exclude:
        assert any(set(i for i, _ in w) & set(range(300, 340)) for w in want.values())


def test_top_n_subsets():
    from xmap_b200 import als
    m, X, Y, xn, yn, user, item = _model(5)
    nU, nI = X.shape[0], Y.shape[0]
    rng = np.random.default_rng(1)
    rated = {}
    for a, b in zip(user, item):
        rated.setdefault(int(a), set()).add(int(b))
    rated = {k: np.array(sorted(v)) for k, v in rated.items()}
    for cand, sel, n in ((np.sort(rng.choice(nI, 5, replace=False)), None, 10),       # fewer candidates than n
                         (np.sort(rng.choice(nI, 333, replace=False)), rng.permutation(nU)[:70], 64),
                         (np.arange(0, nI, 3), np.arange(nU)[::-4].copy(), 7)):
        users = np.arange(nU) if sel is None else sel
        top = als.top_n(m, n, torch.from_numpy(user), torch.from_numpy(item), candidates=torch.from_numpy(cand),
                        users=None if sel is None else torch.from_numpy(sel))
        _check_lists(top, AX.top_n(X, Y, xn, yn, n, users, cand, rated), users, n)
        other = np.setdiff1d(np.arange(nU), users)
        assert (top.len.cpu().numpy()[other] == 0).all()
    for bad in (dict(n=0), dict(n=65), dict(candidates=torch.tensor([3, 2])), dict(candidates=torch.tensor([nI])),
                dict(users=torch.tensor([1, 1])), dict(users=torch.tensor([nU]))):
        kw = dict(n=10, user=torch.from_numpy(user), item=torch.from_numpy(item))
        kw.update(bad)
        with pytest.raises(ValueError):
            als.top_n(m, **kw)


# ---- evaluate_als and the facade ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def files(tmp_path_factory):
    from oracle import make_golden_cleansplit as CS
    from tests.test_gpu_ingest import _synth_files
    with CS.utc():
        return _synth_files(str(tmp_path_factory.mktemp("als")), 11)


def _arrays(paths):
    from oracle import make_golden_cleansplit as CS
    from tests.test_gpu_ingest import _cfg, _tools
    from xmap_b200 import ingest
    cs, ct, sp = _tools(_cfg(atleast=3, num_left=2, ratio_split=0.3, ratio_both=0.4))
    with CS.utc():
        return ingest.ingest_arrays(cs, ct, sp, paths[0], paths[1], False)


def _alterego_tools():
    from xmap_b200.core import BaselinerSim, ExtendSim, Generator
    return (BaselinerSim("adjust_cosine", 5), ExtendSim(10),
            Generator(1, 0.6, "adjust_cosine", 0.1, private_mode="exp_mech", seed=20261022), False)


@pytest.mark.parametrize("arm", ["baseline", "alterego"])
def test_evaluate_als_equals_array_calls(files, arm):
    from tests.test_gpu_evaluate import restate_metrics, _check_metrics
    from xmap_b200 import als, evaluate, recsim
    A = _arrays(files)
    ev = evaluate.evaluate_als(A, rank=6, iterations=3, lambda_=0.05, seed=5,
                               alterego=None if arm == "baseline" else _alterego_tools())
    # the training records the arm names
    if arm == "baseline":
        pu, pi, pr = A.user.long(), A.item.long(), A.rating
        n_items = len(A.iids)
        item_of = torch.arange(n_items, device=pu.device)
    else:
        pu, pi, pr = ev.train_user, ev.train_item, ev.train_rating
        n_items = int(ev.profile_items.numel())
        item_of = ev.profile_items
    m = als.train(pu, pi, pr, len(A.uids), n_items, 6, 3, 0.05, seed=5)
    assert torch.equal(m.user_factors, ev.model.user_factors) and torch.equal(m.item_factors, ev.model.item_factors)
    # predictions: every held-out pair, skipped ones NaN
    tu = A.train_user_of[A.test_user.long()].long()
    ti = A.train_item_of[A.test_item.long()].long()
    prof_of = torch.full((len(A.iids),), -1, dtype=torch.int64, device=tu.device)
    prof_of[item_of] = torch.arange(n_items, device=tu.device)
    tpi = torch.where(ti >= 0, prof_of[ti.clamp(min=0)], -1)
    ok = (tu >= 0) & (tpi >= 0)
    ok &= (m.user_count[tu.clamp(min=0)] > 0) & (m.item_count[tpi.clamp(min=0)] > 0)
    p = als.predict(m, tu[ok], tpi[ok])
    assert torch.equal(ev.pred[ok].view(torch.int64), p.view(torch.int64)) and torch.isnan(ev.pred[~ok]).all()
    c = ev.counts
    assert c["predicted"] == int(ok.sum()) > 0
    assert c["predicted"] + c["skipped_untrained"] + c["skipped_no_profile"] + c["skipped_no_factors"] == c["test_pairs"]
    tr = A.test_rating[ok]
    assert ev.mae == math.fsum((tr - p).abs().cpu().tolist()) / int(ok.sum())
    bounded = torch.clamp(torch.floor(p + 0.5), 0, 5)
    assert ev.mae_bounded == math.fsum((tr - bounded).abs().cpu().tolist()) / int(ok.sum())
    # the lists: top-n over target items with factors, training records excluded
    run = A.train_user_of[ev.users].long()
    has_T = A.meta.has_T[item_of.long()]
    cand = torch.nonzero(has_T & (m.item_count > 0)).flatten()
    top = als.top_n(m, 10, pu, pi, candidates=cand, users=run)
    assert torch.equal(top.idx[run], ev.top.idx[run]) and torch.equal(top.len[run], ev.top.len[run])
    assert c["catalogue_items"] == int(cand.numel())
    # the metrics against the restatement, over ids
    idx, ln = ev.top.idx.cpu().numpy(), ev.top.len.cpu().numpy()
    pit = item_of.cpu().numpy()
    rel = {}
    tu_all, ti_all = A.test_user.cpu().numpy(), A.test_item.cpu().numpy()
    for q in range(len(tu_all)):
        rel.setdefault(int(tu_all[q]), set()).add(str(A.all_iids[ti_all[q]]))
    lists = [[str(A.iids[pit[idx[r, s]]]) for s in range(ln[r])] for r in run.cpu().numpy()]
    want = restate_metrics(lists, [rel[int(u)] for u in ev.users.cpu().numpy()], 10, recsim.DISCOUNT)
    _check_metrics(ev.metrics, want)
    print(arm, c)


@pytest.mark.parametrize("ids", ["str", "int"])
def test_facade_equals_array_api(ids):
    from xmap_b200 import als
    from xmap_b200.core import ALS
    user, item, rating, nU, nI = _case(21, n_users=90, n_items=70, n_rand=800)
    if ids == "str":
        uk = np.array(["u%03d" % v for v in range(nU)], dtype=object)
        ik = np.array(["T:i%03d" % v for v in range(nI)], dtype=object)
    else:
        uk, ik = np.arange(nU) * 7 + 3, np.arange(nI) * 5 + 1
    recs = [(uk[a], ik[b], float(r), 1234) for a, b, r in zip(user, item, rating)]
    model = ALS.train(recs, 8, iterations=3, lambda_=0.1, seed=17, blocks=4)
    # the facade numbers ids by np.unique; here the id order is the index order, and unused ids are absent
    uu, inv_u = np.unique(user, return_inverse=True)
    ii, inv_i = np.unique(item, return_inverse=True)
    m = als.train(torch.from_numpy(inv_u), torch.from_numpy(inv_i), torch.from_numpy(rating), len(uu), len(ii), 8, 3,
                  0.1, seed=17)
    X, Y = m.user_factors.cpu().numpy(), m.item_factors.cpu().numpy()
    uf, pf = dict(model.userFeatures().collect()), dict(model.productFeatures().collect())
    assert len(uf) == len(uu) and len(pf) == len(ii)
    for q, u in enumerate(uu):
        assert np.array_equal(np.array(uf[uk[u]], np.float32), X[q])
    for q, i in enumerate(ii):
        assert np.array_equal(np.array(pf[ik[i]], np.float32), Y[q])
    s = als.predict(m, torch.arange(len(uu)).repeat_interleave(len(ii)), torch.arange(len(ii)).repeat(len(uu)))
    s = s.cpu().numpy().reshape(len(uu), len(ii))
    assert model.predict(uk[uu[2]], ik[ii[3]]) == s[2, 3]
    pairs = [(uk[uu[a]], ik[ii[b]]) for a, b in ((0, 0), (1, 5), (4, 2))]
    got = {(a, b): r for a, b, r in model.predictAll(pairs).collect()}
    assert got == {(uk[uu[a]], ik[ii[b]]): s[a, b] for a, b in ((0, 0), (1, 5), (4, 2))}
    top = als.top_n(m, 5, exclude_rated=False)
    lst = model.recommendProducts(uk[uu[7]], 5)
    assert [(r[0], r[1]) for r in lst] == [(uk[uu[7]], ik[ii[j]]) for j in top.idx[7, :5].tolist()]
    assert [r[2] for r in lst] == top.score[7, :5].tolist()
    allr = dict(model.recommendProductsForUsers(5).collect())
    assert len(allr) == len(uu) and [r[1] for r in allr[uk[uu[7]]]] == [r[1] for r in lst]
    with pytest.raises(ValueError):
        ALS.train(recs, 8, nonnegative=True)
    with pytest.raises(ValueError):
        model.recommendProducts(uk[uu[0]], 65)
