"""GPU: evaluate.evaluate (held-out MAE and top-N accuracy on the device) against the facade chain it mirrors,
recsim.rank_metrics against a plain Python restatement of its definitions, top_n(users=...) against the full run,
and the train index maps of ingest_arrays."""
import types

import numpy as np
import pytest
import torch

from oracle import make_golden_cleansplit as CS
from tests.test_gpu_ingest import _cfg, _synth_files, _tools

pytestmark = pytest.mark.gpu

CFG = dict(atleast=3, num_left=2, ratio_split=0.3, ratio_both=0.4)


# ---- the Python restatement of the ranking metrics (DESIGN.md section 3.6) ----------------------------------------
def restate_metrics(lists, relevant, n, disc):
    """lists[q]: user q's recommended items, best first; relevant[q]: its relevant items.  Sums in slot order."""
    out = []
    for lst, R in zip(lists, relevant):
        R = set(R)
        h, dcg, ap = 0, 0.0, 0.0
        for p, it in enumerate(lst[:n]):
            if it in R:
                h += 1
                dcg += disc[p]
                ap += h / (p + 1)
        m = min(n, len(R))
        idcg = 0.0
        for p in range(m):
            idcg += disc[p]
        out.append((h, h / n, h / len(R), dcg / idcg, ap / m))
    return out


def _check_metrics(res, want):
    got = [res.hits.cpu().numpy()] + [t.cpu().numpy() for t in (res.precision, res.recall, res.ndcg, res.ap)]
    assert np.array_equal(got[0], np.array([w[0] for w in want], np.int32))
    for f in range(1, 5):
        a = np.array([w[f] for w in want], np.float64)
        assert np.array_equal(got[f].view(np.int64), a.view(np.int64)), f
    import math
    for f, k in enumerate(("precision", "recall", "ndcg", "map"), 1):
        assert res.mean[k] == math.fsum(w[f] for w in want) / len(want)


# ---- 1. rank_metrics ---------------------------------------------------------------------------------------------
def _rank_case(seed, width=64, n_rows=300, n_items=5000):
    """Top-N rows of random lengths (0 .. width, distinct items) and, per evaluated row, a relevant set built to hit
    the edges: |R| below, equal to and above n, |R| > 1024, every slot a hit, no slot a hit, unreachable items."""
    rng = np.random.default_rng(seed)
    idx = np.full((n_rows, width), -1, np.int32)
    ln = rng.integers(0, width + 1, n_rows).astype(np.int32)
    ln[:5] = [0, 1, 3, width, width]
    for r in range(n_rows):
        idx[r, :ln[r]] = rng.choice(n_items, ln[r], replace=False)
    users = rng.permutation(n_rows)[:200]
    rel = []
    for q, u in enumerate(users):
        lst = idx[u, :ln[u]]
        kind = q % 8
        if kind == 0:                                    # every slot a hit (plus more)
            R = set(lst.tolist()) | set(rng.integers(0, n_items, 3).tolist())
        elif kind == 1:                                  # no hit, only unreachable items
            R = set((n_items + rng.integers(0, 10 ** 6, 5)).tolist())
        elif kind == 2:                                  # a long list, well over 1 024 items
            R = set(rng.choice(n_items, 1500 + q, replace=False).tolist())
        elif kind == 3:                                  # exactly one
            R = {int(lst[len(lst) // 2])} if len(lst) else {n_items + 1}
        else:                                            # |R| around n: some of the list, some other, some unreachable
            k = int(rng.integers(1, 80))
            R = set(rng.choice(lst, min(len(lst), k // 2), replace=False).tolist()) if len(lst) else set()
            R |= set(rng.integers(0, n_items, k - len(R)).tolist()) | {n_items + 7}
        rel.append(np.array(sorted(R), np.int64))
    ptr = np.zeros(len(users) + 1, np.int64)
    ptr[1:] = np.cumsum([len(r) for r in rel])
    top = types.SimpleNamespace(idx=torch.from_numpy(idx).cuda(), len=torch.from_numpy(ln).cuda())
    return top, users, ptr, np.concatenate(rel), rel, idx, ln


@pytest.mark.parametrize("n", [1, 10, 64])
def test_rank_metrics_match_restatement(n):
    from xmap_b200 import recsim
    top, users, ptr, flat, rel, idx, ln = _rank_case(n)
    res = recsim.rank_metrics(top, torch.from_numpy(users), ptr, flat, n, catalogue=5000)
    lists = [idx[u, :min(ln[u], n)].tolist() for u in users]
    _check_metrics(res, restate_metrics(lists, [r.tolist() for r in rel], n, recsim.DISCOUNT))
    assert max(len(r) for r in rel) > 1024
    h = res.hits.cpu().numpy()
    assert (h == 0).any() and (h == np.minimum(ln[users], n)).any()
    want_cov = len(set(v for u in users for v in idx[u, :min(ln[u], n)].tolist())) / 5000
    assert res.coverage == want_cov


def test_rank_metrics_errors():
    from xmap_b200 import recsim
    top, users, ptr, flat, rel, idx, ln = _rank_case(3)
    u = torch.from_numpy(users)
    for n in (0, 65, 2.5):
        with pytest.raises(ValueError):
            recsim.rank_metrics(top, u, ptr, flat, n)
    bad_u = users.copy()
    bad_u[0] = len(ln)
    with pytest.raises(ValueError):
        recsim.rank_metrics(top, torch.from_numpy(bad_u), ptr, flat, 10)
    with pytest.raises(ValueError):
        recsim.rank_metrics(top, u, ptr[:-1], flat, 10)                      # one extent short
    empty = np.r_[ptr[:2], ptr[1:]]                                         # a user without relevant items
    with pytest.raises(ValueError):
        recsim.rank_metrics(top, torch.from_numpy(np.r_[users[:1], users]), empty, flat, 10)
    unsorted = flat.copy()
    unsorted[ptr[2]], unsorted[ptr[2] + 1] = flat[ptr[2] + 1], flat[ptr[2]]
    with pytest.raises(ValueError):
        recsim.rank_metrics(top, u, ptr, unsorted, 10)
    neg = flat.copy()
    neg[0] = -1
    with pytest.raises(ValueError):
        recsim.rank_metrics(top, u, ptr, neg, 10)


# ---- 2. top_n(users=...) -----------------------------------------------------------------------------------------
def test_top_n_users_subset():
    from xmap_b200 import recsim
    from tests.test_gpu_topn import _dup, _tables
    p = _dup()
    knn = _tables(p, 10)
    args = (p["user"], p["item"], p["rating"], p["ts"], p["n_users"] + 2, knn, knn.nb, 10)
    full = recsim.top_n(*args)
    rng = np.random.default_rng(5)
    for sel in (rng.permutation(p["n_users"] + 2)[:40], np.arange(p["n_users"] + 2)[::-7].copy(), np.zeros(0, np.int64)):
        res = recsim.top_n(*args, users=torch.from_numpy(sel))
        other = np.setdiff1d(np.arange(p["n_users"] + 2), sel)
        s = torch.from_numpy(sel).cuda()
        assert torch.equal(res.idx[s], full.idx[s]) and torch.equal(res.len[s], full.len[s])
        assert torch.equal(res.score[s].view(torch.int64), full.score[s].view(torch.int64))
        o = torch.from_numpy(other).cuda()
        assert (res.idx[o] == -1).all() and torch.isnan(res.score[o]).all() and (res.len[o] == 0).all()
        assert res.warp_users + res.cta_users == len(sel) and res.candidates <= res.visits
        if len(sel) == 0:
            assert (res.visits, res.candidates) == (0, 0)
    for bad in (np.array([0, p["n_users"] + 2]), np.array([-1]), np.array([3, 4, 3]), np.zeros((2, 2), np.int64),
                np.array([0.5])):
        with pytest.raises(ValueError):
            recsim.top_n(*args, users=torch.from_numpy(bad))


# ---- 3. the train index maps ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def files(tmp_path_factory):
    with CS.utc():
        return [_synth_files(str(tmp_path_factory.mktemp("ev%d" % s)), s) for s in (11, 12)]


def _arrays(paths, num_left):
    from xmap_b200 import ingest
    cs, ct, sp = _tools(_cfg(**dict(CFG, num_left=num_left)))
    return ingest.ingest_arrays(cs, ct, sp, paths[0], paths[1], False)


def test_train_index_maps(files):
    A = _arrays(files[0], 2)
    for of, ids, all_ids in ((A.train_user_of, A.uids, A.all_uids), (A.train_item_of, A.iids, A.all_iids)):
        of = of.cpu().numpy()
        assert of.dtype == np.int32 and len(of) == len(all_ids)
        have = np.flatnonzero(of >= 0)
        assert np.array_equal(ids[of[have]], all_ids[have])
        assert np.array_equal(np.sort(of[have]), np.arange(len(ids)))          # every training id exactly once


# ---- 4. the array chain against the facade chain -------------------------------------------------------------------
def _chain_tools():
    from xmap_b200.core import BaselinerSim, ExtendSim, Generator, RecommenderSim, RecommenderPrivacy
    return (BaselinerSim("adjust_cosine", 5), ExtendSim(10),
            Generator(1, 0.6, "adjust_cosine", 0.1, private_mode="exp_mech", seed=20261022),
            RecommenderSim("cosine_item", 5), RecommenderPrivacy(10, 0.6, 0.1, seed=77))


def _facade(paths, num_left, private):
    from xmap_b200 import ingest
    from xmap_b200.core import (RecommenderPrediction, baseliner_calculate_sim_pipeline, extender_pipeline,
                                generator_pipeline, recommend_top_n, recommender_calculate_sim_pipeline,
                                recommender_prediction_pipeline, recommender_privacy_pipeline)
    cs, ct, sp = _tools(_cfg(**dict(CFG, num_left=num_left)))
    tr, te = ingest.clean_split_pipeline(None, cs, ct, sp, paths[0], paths[1], False)
    sim, ext, gen, rsim, priv = _chain_tools()
    simRDD = baseliner_calculate_sim_pipeline(None, sim, tr)
    xs = extender_pipeline(None, None, sim, ext, simRDD)
    alter = generator_pipeline(gen, tr, xs, private)
    out = recommender_calculate_sim_pipeline(None, rsim, alter)
    simpair = recommender_privacy_pipeline(priv, out[6], private).collectAsMap()
    rp = RecommenderPrediction(0.03, "cosine_item")
    pred = rp.item_based_recommendation(te, out[3], simpair, out[5]).collect()
    mae = recommender_prediction_pipeline(rp, rsim, te, simpair, out[2], out[3], out[4], out[5])
    return pred, mae, dict(recommend_top_n(simpair, 10).collect()), simpair.handle


def _evaluate(paths, num_left, private, **kw):
    from xmap_b200 import evaluate
    A = _arrays(paths, num_left)
    sim, ext, gen, rsim, priv = _chain_tools()
    return A, evaluate.evaluate(A, sim, ext, gen, private, rsim, priv, private, **kw)


def _lists(A, ev):
    """{uid: [(iid, score)]} of the evaluated users, and their relevant held-out item ids."""
    idx, score, ln = ev.top.idx.cpu().numpy(), ev.top.score.cpu().numpy(), ev.top.len.cpu().numpy()
    pit = ev.profile_items.cpu().numpy()
    uof = A.train_user_of.cpu().numpy()
    out = {}
    for u in ev.users.cpu().numpy():
        r = uof[u]
        out[str(A.all_uids[u])] = [(str(A.iids[pit[idx[r, p]]]), float(score[r, p])) for p in range(ln[r])]
    return out


@pytest.mark.parametrize("private", [False, True])
@pytest.mark.parametrize("pair,num_left", [(0, 2), (1, 0)])
def test_array_chain_equals_facade(files, pair, num_left, private):
    from xmap_b200 import recsim
    with CS.utc():
        pred, mae, tops, state = _facade(files[pair], num_left, private)
        A, ev = _evaluate(files[pair], num_left, private)
    # the profile numbering is the facade's
    assert np.array_equal(state.iids, A.iids[ev.profile_items.cpu().numpy()])
    # every held-out pair, in test order
    p0, p1 = ev.pred_nodecay.cpu().numpy(), ev.pred_decay.cpu().numpy()
    ti = A.test_item.cpu().numpy()
    flat = [e for _, lst in pred for e in lst]
    assert len(flat) == len(p0)
    for q, e in enumerate(flat):
        if e == ():
            assert p0[q] == -1.0 and p1[q] == -1.0, q
        else:
            assert e[0] == str(A.all_iids[ti[q]])
            assert np.float64(e[2]).view(np.int64) == p0[q].view(np.int64), q
            assert np.float64(e[3]).view(np.int64) == p1[q].view(np.int64), q
    c = ev.counts
    assert c["predicted"] == sum(e != () for e in flat) > 0
    assert c["predicted"] + c["skipped_untrained"] + c["skipped_no_profile"] + c["skipped_no_neighbours"] == len(flat)
    assert str(ev.mae_nodecay) + "; " + str(ev.mae_decay) == mae
    # the test users' lists, ids and scores bit for bit
    mine = _lists(A, ev)
    compared = 0
    for uid, lst in mine.items():
        if uid in tops:
            assert lst == tops[uid], uid
            compared += 1
    assert compared > 0 and compared + ev.counts["eval_users_without_profile"] == len(mine)
    # the metrics against the restatement, over ids (a relevant item outside the profile is in R but never listed)
    rel = {}
    tu = A.test_user.cpu().numpy()
    for q in range(len(tu)):
        rel.setdefault(str(A.all_uids[tu[q]]), set()).add(str(A.all_iids[ti[q]]))
    uids = [str(A.all_uids[u]) for u in ev.users.cpu().numpy()]
    want = restate_metrics([[i for i, _ in mine[u]] for u in uids], [rel[u] for u in uids], 10, recsim.DISCOUNT)
    _check_metrics(ev.metrics, want)
    print("pair %d private=%s: %s" % (pair, private, ev.counts))


def test_threshold_drops_users(files):
    with CS.utc():
        A, ev_all = _evaluate(files[0], 2, False)
        _, ev4 = _evaluate(files[0], 2, False, threshold=4.0, n=5)
    tu, tr = A.test_user.cpu().numpy(), A.test_rating.cpu().numpy()
    want = np.unique(tu[tr >= 4.0])
    assert np.array_equal(ev4.users.cpu().numpy(), want)
    assert 0 < len(want) < len(ev_all.users)
    assert ev4.counts["test_users_without_relevant"] == len(A.test_users) - len(want)
    assert np.array_equal(ev4.pred_nodecay.cpu().numpy(), ev_all.pred_nodecay.cpu().numpy())
    relevant = sum(len(set(A.test_item.cpu().numpy()[(tu == u) & (tr >= 4.0)])) for u in want)
    assert ev4.counts["relevant_items"] == relevant
