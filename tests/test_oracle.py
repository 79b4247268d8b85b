"""CPU: the oracle restatement (oracle/restate.py) is pinned against the golden vectors that
the UNMODIFIED reference produced (oracle/make_golden.py), stage by stage."""
import numpy as np
import pytest

from oracle import harness as H
from oracle import restate as RS
from tests import parity as PT


def _case(name):
    g = PT.load_golden(name)
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    P = RS.sim_pairs(g["user"].astype(np.int64), g["item"].astype(np.int64), g["rating"], nU, nI,
                     meta["prefix_code"], str(g["method"]), int(g["num_atleast"]))
    return g, meta, nU, nI, P


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_restatement_similarity_vs_reference(name):
    g, meta, nU, nI, P = _case(name)
    assert np.array_equal(P["i"], g["sim_i"]) and np.array_equal(P["j"], g["sim_j"])
    assert np.array_equal(P["mutu"], g["sim_mutu"]) and np.array_equal(P["frac"], g["sim_frac"])
    assert np.array_equal(P["label"], g["sim_label"])
    # bit-equal wherever numpy sums sequentially (n < 8), 1e-12 elsewhere
    small = P["n"] < 8
    assert np.array_equal(P["sim"][small], g["sim_val"][small])
    np.testing.assert_allclose(P["sim"], g["sim_val"], rtol=1e-10)
    st = P["stats"]
    assert np.array_equal(st["mu"], g["user_avg"])
    assert np.array_equal(np.stack([st["avg"], st["norm2"], st["adj_norm2"], st["count"]], 1), g["item_info"])


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_restatement_selection_extension_generation_vs_reference(name):
    g, meta, nU, nI, P = _case(name)
    k = int(g["k"])
    knn = RS.select_knn(P, nI, k, meta["dom_code"], meta["contains"])
    assert np.array_equal(knn["bb"], g["bb"]) and np.array_equal(knn["valid_nb"], g["valid_nb"])
    lists = PT.restate_lists(knn, P)
    for nm in ("BB_BB", "BB_NB", "NB_BB", "NB_NN"):
        assert np.array_equal(lists[nm][0], g[nm + "_ptr"]) and np.array_equal(lists[nm][1], g[nm + "_nbr"])
    X = RS.xsim_extend(P, knn, nI, meta["has_S"], meta["has_T"])
    PT.compare_xsim(X["start"], X["end"], X["xsim"], g["xs_start"], g["xs_end"], g["xs_val"], rtol=1e-9)
    if "priv_rows" not in g:
        return
    rows, cands = RS.candidates(X["start"], X["end"], X["xsim"], 10)
    ch, _ = RS.choose(rows, cands, "argmax")
    assert np.array_equal(rows, g["priv_rows"]) and np.array_equal(ch, g["priv_chosen"])
    mp = RS.invert_mapping(rows, ch, nI)
    ae = RS.build_alterego(g["user"], g["item"], g["rating"], g["ts"], mp, meta["has_T"])
    o = np.lexsort((ae["ts"], ae["rating"], ae["item"], ae["user"]))
    assert np.array_equal(ae["user"][o], g["priv_ae_user"]) and np.array_equal(ae["item"][o], g["priv_ae_item"])
    assert np.array_equal(ae["rating"][o], g["priv_ae_rating"]) and np.array_equal(ae["ts"][o], g["priv_ae_ts"])
    rows4, cands4 = RS.candidates(X["start"], X["end"], X["xsim"], 4)
    ok = np.array([len(c[0]) >= 2 for c in cands4])
    u = np.zeros(len(rows4)); u[ok] = g["nonpriv_uniforms"]
    chn, single = RS.choose(rows4, cands4, "nonprivate", uniforms=u)
    assert np.array_equal(rows4[ok], g["nonpriv_rows"]) and np.array_equal(chn[ok], g["nonpriv_chosen"])


@pytest.mark.skipif(not H.reference_available(), reason="needs the original X-MAP source (XMAP_REFERENCE_CODE)")
def test_harness_runs_the_reference_and_agrees_with_golden():
    """Where the original X-MAP source is available, re-run the reference itself on the smallest case."""
    import subprocess, sys
    code = ("import numpy as np;from oracle import make_golden as M;"
            "o=M.build_case('adj_all_bridge');g=np.load('tests/golden/adj_all_bridge.npz');"
            "assert all(np.array_equal(o[k],g[k]) for k in g.files if k!='ref_seconds');print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=PT.ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_restatement_recommender_sim_vs_reference(name):
    """Next row of the scope table (SURVEY.md 8(f) #1): RecommenderSim `cosine_item` + local sensitivity on the
    AlterEgo profile -- the restatement against what the unmodified reference produced
    (oracle/make_golden_recsim.py).  Pins duplicate (user, item) records, self pairs and the absence of a filter."""
    g = PT.load_golden(name + "_recsim")
    nI = int(max(g["ae_item"].max(), g["rs_i"].max(), g["rs_j"].max())) + 1
    P = RS.recommender_cosine_item(g["ae_user"], g["ae_item"], g["ae_rating"], nI, int(g["num_atleast"]))
    assert np.array_equal(P["i"], g["rs_i"]) and np.array_equal(P["j"], g["rs_j"])
    assert int((P["i"] == P["j"]).sum()) > 0                       # a real next to a synthetic rating of one item
    np.testing.assert_allclose(P["sim"], g["rs_sim"], rtol=1e-12, atol=0)
    np.testing.assert_allclose(P["ls"], g["rs_ls"], rtol=1e-9, atol=1e-13, equal_nan=True)
    np.testing.assert_allclose(P["norm2"][g["info_item"]], g["info_norm2"], rtol=1e-14)
    cnt = np.bincount(g["ae_item"], minlength=nI)
    assert np.array_equal(cnt[g["info_item"]], g["info_count"])


def test_sim_rows_restriction_equals_sim_pairs():
    """restate.sim_rows (the sampled-row oracle of the full-size GPU test) is bit-equal to sim_pairs on its rows."""
    from tests import parity as PT
    case = PT.synth_case(1500, 400, 20000, 0.05, seed=5)
    args = (case["user"], case["item"], case["rating"], case["n_users"], case["n_items"], case["meta"]["prefix_code"])
    for method in ("adjust_cosine", "cosine"):
        P = RS.sim_pairs(*args, method, 50)
        rows = np.array([0, 3, 17, 100, 250, 398, 399, 399])
        Q = RS.sim_rows(*args, rows, method, 50)
        m = np.isin(P["i"], rows)
        assert m.sum() > 100
        for key in ("i", "j", "sim", "mutu", "n", "frac", "label"):
            assert np.array_equal(P[key][m], Q[key]), key


def test_restatement_vs_reference_mid_size():
    """The mid-size golden (90 K ratings, 366 K kept pairs; the reference took 17 s for the similarity stage):
    similarity, mutuality, labels, BB set and all four neighbour tables of the restatement against the
    unmodified reference.  Lists of ~1e3 neighbours and rows with thousands of co-rating products."""
    g, meta, nU, nI, P = _case("adj_mid")
    assert len(g["user"]) > 85000 and len(g["sim_i"]) > 300000
    assert np.array_equal(P["i"], g["sim_i"]) and np.array_equal(P["j"], g["sim_j"])
    assert np.array_equal(P["mutu"], g["sim_mutu"]) and np.array_equal(P["label"], g["sim_label"])
    known = np.isfinite(g["sim_val"])          # similarity and frac are stored for a fixed sample of the pairs
    assert known.sum() > 70000
    assert np.array_equal(P["frac"][known].astype(np.float32), g["sim_frac"][known])      # stored as its float32 image
    np.testing.assert_allclose(P["sim"][known], g["sim_val"][known], rtol=1e-10)
    assert np.array_equal(P["stats"]["mu"], g["user_avg"])
    knn = RS.select_knn(P, nI, int(g["k"]), meta["dom_code"], meta["contains"])
    assert np.array_equal(knn["bb"], g["bb"]) and np.array_equal(knn["valid_nb"], g["valid_nb"])
    lists = PT.restate_lists(knn, P)
    n_diff = 0
    for nm in ("BB_BB", "BB_NB", "NB_BB", "NB_NN"):
        assert np.array_equal(lists[nm][0], g[nm + "_ptr"])
        n_diff += int((lists[nm][1] != g[nm + "_nbr"]).sum())
    assert n_diff == 0, "%d neighbour entries differ from the reference" % n_diff


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_restatement_neighbors_and_prediction_vs_reference(name):
    """SURVEY.md 8(f) #2-#3: non-private neighbour selection and item-based prediction + MAE on the AlterEgo
    profile -- the restatement against the unmodified reference (oracle/make_golden_recpred.py)."""
    g = PT.load_golden(name + "_recpred")
    nI = int(max(g["ae_item"].max(), g["test_item"].max(), g["nb_idx"].max())) + 1
    P = RS.recommender_cosine_item(g["ae_user"], g["ae_item"], g["ae_rating"], nI, int(g["num_atleast"]))
    ptr, idx, val = RS.recommender_neighbors(P, nI, int(g["mapping_range"]))
    has = np.flatnonzero(np.diff(ptr))
    assert np.array_equal(has, g["nb_item"])
    assert np.array_equal(np.diff(ptr)[has], np.diff(g["nb_ptr"]))
    assert np.array_equal(idx, g["nb_idx"])
    np.testing.assert_allclose(val, g["nb_sim"], rtol=1e-12)
    cnt = np.bincount(g["ae_item"], minlength=nI)
    avg = np.bincount(g["ae_item"], weights=g["ae_rating"], minlength=nI) / np.maximum(cnt, 1)
    p0, p1, m0, m1 = RS.recommender_predict(g["ae_user"], g["ae_item"], g["ae_rating"], g["ae_ts"], ptr, idx, val, avg,
                                            g["test_user"], g["test_item"], g["test_rating"], float(g["alpha"]))
    assert np.array_equal(p0, g["pred_nodecay"]) and np.array_equal(p1, g["pred_decay"])
    assert abs(m0 - float(g["mae_nodecay"])) < 1e-12 and abs(m1 - float(g["mae_decay"])) < 1e-12


@pytest.mark.parametrize("name", ["adj_low_overlap", "cos_half_ratings"])
def test_restatement_private_neighbors_vs_reference(name):
    """The PRIVATE branch of SURVEY.md 8(f) #2: private_neighbor_selection + noise_perturbation run by the unmodified
    reference with its np.random draws logged (tests/golden/*_recpriv.npz, oracle/make_golden_recpriv.py); the restatement
    fed the same uniforms picks the same neighbour for every item and returns the same noisy similarity."""
    g0, g = PT.load_golden(name), PT.load_golden(name + "_recpriv")
    nI = len(g0["iids"])
    P = RS.recommender_cosine_item(g["ae_user"], g["ae_item"], g["ae_rating"], nI, int(g["num_atleast"]))
    it, ch, out = RS.recommender_private_neighbors(P, nI, int(g["mapping_range"]), float(g["epsilon"]), float(g["rpo"]),
                                                   g["u_pick"], g["u_noise"])
    assert len(it) > 100 and np.array_equal(it, g["item"]) and np.array_equal(ch, g["chosen"])
    np.testing.assert_allclose(out, g["noisy_sim"], rtol=1e-13, atol=0)
    # the draw is not the arg-max: the mechanism really samples
    nb = RS.recommender_neighbors(P, nI, 1)
    assert 0 < int((ch != nb[1]).sum())


def test_restatement_alterego_merge_rule_hand_computed():
    """generator.py:140-157 on a merge (SURVEY.md:394, :577; DESIGN.md 3.4): the ratings a user gave to several
    sources mapped onto one target become ONE record with their mean and the time of the smallest source item --
    not the earliest time, and not the first record in input order.  A real "T:" rating of the same (user, target)
    is kept next to it.  Expected values written out by hand."""
    #        user  item  rating  ts      items: 1 = s1, 2 = s2 (both -> 3), 3 = T (a "T:" item)
    recs = [(0, 2, 2.5, 100),
            (0, 1, 1.25, 300),
            (0, 3, 4.0, 50),
            (1, 2, 3.5, 70)]
    user, item, rating, ts = (np.array(c) for c in zip(*recs))
    mapping = np.array([-1, 3, 3, -1])
    has_T = np.array([False, False, False, True])
    ae = RS.build_alterego(user, item, rating.astype(np.float32), ts, mapping, has_T)
    assert ae["user"].tolist() == [0, 0, 1]
    assert ae["item"].tolist() == [3, 3, 3]
    assert ae["rating"].tolist() == [4.0, 1.875, 3.5]
    assert ae["ts"].tolist() == [50, 300, 70]
    assert ae["synthetic"].tolist() == [False, True, True]


def test_restatement_invert_mapping_largest_target_wins_and_skips_empty_rows():
    """assist.py:215: rows in ascending target order, so the largest target choosing a source wins; a row
    without a candidate (chosen = -1) maps nothing."""
    mp = RS.invert_mapping(np.array([2, 5, 7, 9]), np.array([1, 1, -1, 1]), 10)
    assert mp.tolist() == [-1, 9, -1, -1, -1, -1, -1, -1, -1, -1]
    mp = RS.invert_mapping(np.array([2, 5, 7]), np.array([4, 1, -1]), 6)
    assert mp.tolist() == [-1, 5, -1, -1, 2, -1]


def test_restatement_prediction_tied_times_share_a_rank():
    """recommenderPrediction.py:36-49: entry times [5, 5, 9] rank [1, 1, 2], cur = 3, so the decay weights are
    e^{-2 alpha}, e^{-2 alpha}, e^{-alpha}.  Also: no neighbour list -> -1, no matching record -> the item
    average, and raw=True returns the values before bounding while leaving the default output as it was."""
    import math
    a = 0.5
    # profile of user 0 in list order: item 3 at t = 9, item 1 at t = 5, item 2 at t = 5; user 1 rates item 4 only
    p_user, p_item = np.array([0, 0, 0, 1]), np.array([3, 1, 2, 4])
    p_rating, p_ts = np.array([3.0, 4.0, 2.0, 1.0]), np.array([9, 5, 5, 7])
    nb_ptr = np.array([0, 3, 3, 3, 3, 3])                  # item 0: neighbours 1, 2, 3; no other item has a list
    nb_idx, nb_sim = np.array([1, 2, 3]), np.array([0.5, -0.25, 1.0])
    avg = np.array([3.0, 3.5, 2.5, 2.0, 1.0])
    t_user, t_item, t_rating = np.array([0, 1, 0]), np.array([0, 0, 2]), np.array([4.0, 3.0, 2.0])
    # entries (sim * (r - avg_n), |sim|): (0.25, 0.5) t=5, (0.125, 0.25) t=5, (1.0, 1.0) t=9
    nd = 3.0 + (0.25 + 0.125 + 1.0) / (0.5 + 0.25 + 1.0)
    w5, w9 = math.exp(-2 * a), math.exp(-a)
    dc = 3.0 + (0.25 * w5 + 0.125 * w5 + 1.0 * w9) / (0.5 * w5 + 0.25 * w5 + 1.0 * w9)
    assert abs(dc - 3.8436667) < 1e-7                      # distinct ranks 1, 2, 3 would give 3.8743713
    args = (p_user, p_item, p_rating, p_ts, nb_ptr, nb_idx, nb_sim, avg, t_user, t_item, t_rating, a)
    p0, p1, m0, m1, r0, r1 = RS.recommender_predict(*args, raw=True)
    assert r0[0] == nd and abs(r1[0] - dc) <= 1e-15 * dc
    assert r0[1] == r1[1] == 3.0 and np.isnan(r0[2]) and np.isnan(r1[2])
    assert p0.tolist() == [4.0, 3.0, -1.0] and p1.tolist() == [4.0, 3.0, -1.0]
    assert m0 == m1 == 0.0
    q0, q1, n0, n1 = RS.recommender_predict(*args)
    assert np.array_equal(q0, p0) and np.array_equal(q1, p1) and (n0, n1) == (m0, m1)
