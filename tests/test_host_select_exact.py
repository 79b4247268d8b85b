"""CPU: the exact selection of tests/select_exact.py -- it equals oracle/restate.select_knn on real pairs, its
designed cases reach every path of both select kernels, and those cases are sharp enough that small selection
errors (a tie rule, a sign, a threshold, a list rule, a sampling shortcut) change the tables of some row."""
import numpy as np
import pytest

from oracle import restate as RS
from tests import parity as PT
from tests import select_exact as SE


def _check_against_restatement(P, n_items, meta, k):
    knn = RS.select_knn(P, n_items, k, meta["dom_code"], meta["contains"])
    T = SE.select_exact(P["i"], P["j"], P["sim"], P["mutu"], P["n"], knn["bb"], meta["dom_code"], meta["contains"], k)
    lists = 0
    for it in range(n_items):
        if knn["bb"][it]:
            names = ("BB_BB", "BB_NB")
        elif knn["valid_nb"][it]:
            names = ("NB_BB", "NB_NN")
        else:                                  # an NB row without a BB neighbour: slot 0 is empty
            assert T["tab_len"][it, 0] == 0
            continue
        for slot, nm in enumerate(names):
            pos = knn[nm][it]
            L = len(pos)
            assert T["tab_len"][it, slot] == L
            assert np.array_equal(T["tab_idx"][it, slot, :L], P["j"][pos])
            assert np.array_equal(T["tab_sim"][it, slot, :L].view(np.int64), P["sim"][pos].view(np.int64))
            assert np.array_equal(T["tab_mutu"][it, slot, :L], P["mutu"][pos])
            assert np.array_equal(T["tab_n"][it, slot, :L], P["n"][pos])
            lists += 1
    return lists


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_reference_equals_restatement_on_goldens(name):
    g = PT.load_golden(name)
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    P = RS.sim_pairs(g["user"].astype(np.int64), g["item"].astype(np.int64), g["rating"], nU, nI,
                     meta["prefix_code"], str(g["method"]), int(g["num_atleast"]))
    for k in (1, int(g["k"]), 64):
        assert _check_against_restatement(P, nI, meta, k) > 0


@pytest.mark.parametrize("seed,half", [(3, False), (8, True)])
def test_reference_equals_restatement_on_synthetic_pairs(seed, half):
    case = PT.synth_case(400, 150, 6000, 0.05, seed=seed, half=half)
    P = RS.sim_pairs(case["user"], case["item"], case["rating"], case["n_users"], case["n_items"],
                     case["meta"]["prefix_code"], "adjust_cosine", 50)
    for k in (2, 10, 33):
        assert _check_against_restatement(P, case["n_items"], case["meta"], k) > 0


def test_reference_refuses_what_the_kernels_never_see():
    bb, dom, con = np.zeros(3, np.uint8), np.zeros(3, np.uint8), np.zeros(3, np.uint8)
    one = lambda *a: np.array(a)
    for i, j, s in ((one(0), one(1), one(np.nan)), (one(0), one(1), one(0.0)), (one(0), one(1), one(-0.0)),
                    (one(0, 0), one(1, 1), one(0.5, 0.25))):
        with pytest.raises(AssertionError):
            SE.select_exact(i, j, s, np.ones(len(i)), np.ones(len(i)), bb, dom, con, 2)


@pytest.fixture(scope="module")
def designed():
    return SE.designed_cases()


def test_designed_cases_reach_every_path(designed):
    c = designed
    for k in SE.KS:
        labels, flushes = SE.classify(c["i"], c["j"], c["sim"], c["bb"], c["dom_code"], c["contains"], k, c["n_rows"])
        counts = SE.path_counts(labels)
        print("k %2d: %s" % (k, counts))
        for p in SE.PATHS[1:]:
            assert counts[p] >= SE.MIN_PER_PATH, "k %d: path %s reached %d times" % (k, p, counts[p])
        assert max(flushes.values()) >= 40          # |sim| ascending: a tournament at nearly every step
    # the carried fields at their limits reach the tables of warp and CTA rows
    T = SE.Ranked(c["i"], c["j"], c["sim"], c["mutu"], c["n"], c["bb"], c["dom_code"], c["contains"],
                  c["n_rows"]).tables(64)
    cnt = np.bincount(c["i"], minlength=c["n_rows"])
    for rows in (cnt <= SE.SELECT_LONG, cnt > SE.SELECT_LONG):
        assert (T["tab_idx"][rows] == SE.N_ITEMS - 1).any()
        assert (T["tab_mutu"][rows] == SE.BIG).any() and (T["tab_n"][rows] == SE.BIG).any()


# ---- mutant selections, one (row, list) at a time ------------------------------------------------------------
def _exact(key, j, sim, k, pos):
    return j[np.lexsort((j, SE.ABS_MASK - key))[:k]]


def _ties_to_larger_j(key, j, sim, k, pos):
    return j[np.lexsort((-j, SE.ABS_MASK - key))[:k]]


def _signed(key, j, sim, k, pos):
    return j[np.lexsort((j, -sim))[:k]]


def _streaming(strict):
    """A running threshold over steps of CTA_STEP records: the k-th best key so far; strict drops records equal
    to it (`key <= th`), the kernel keeps them."""
    def sel(key, j, sim, k, pos):
        tk, tj = np.zeros(0, np.uint64), np.zeros(0, np.int64)
        for b in range(0, len(key), SE.CTA_STEP):
            kk, jj = key[b:b + SE.CTA_STEP], j[b:b + SE.CTA_STEP]
            if len(tk) == k:
                keep = kk > tk[-1] if strict else kk >= tk[-1]
                kk, jj = kk[keep], jj[keep]
            ak, aj = np.concatenate([tk, kk]), np.concatenate([tj, jj])
            o = np.lexsort((aj, SE.ABS_MASK - ak))[:k]
            tk, tj = ak[o], aj[o]
        return tj
    return sel


def _sampled_only(key, j, sim, k, pos):
    """Pass B over the sampled blocks only."""
    m = pos.max(initial=0) + 1
    s = SE.sampled_mask(m)[pos] if m > SE.SAMPLE_FROM else np.ones(len(pos), bool)
    return _exact(key[s], j[s], sim[s], k, pos[s])


def _sample_threshold_always(key, j, sim, k, pos):
    """The histogram threshold taken from the sample even when it holds fewer than k members of the list."""
    m = pos.max(initial=0) + 1
    s = SE.sampled_mask(m)[pos] if m > SE.SAMPLE_FROM else np.ones(len(pos), bool)
    want = min(k, int(s.sum()))
    bins = SE.sim_bin(key)
    suffix = np.cumsum(np.bincount(bins[s], minlength=SE.SIM_BINS)[::-1])[::-1]
    bstar = int(np.nonzero(suffix >= want)[0].max())
    t = bins >= bstar
    return _exact(key[t], j[t], sim[t], k, pos[t])


def _row_lists(c, bits):
    """Per row with records: (positions in the row, list bits), records in stored order."""
    o = np.argsort(c["i"], kind="stable")
    ptr = np.searchsorted(c["i"][o], np.arange(c["n_rows"] + 1))
    for r in range(c["n_rows"]):
        seg = o[ptr[r]:ptr[r + 1]]
        if len(seg):
            yield r, seg, bits[seg]


@pytest.mark.parametrize("mutant", ["ties_to_larger_j", "signed_sim", "threshold_excludes_kth_key",
                                    "nb_slot1_without_bb", "pass_b_sampled_blocks_only",
                                    "sample_threshold_below_k"])
def test_mutant_selections_are_caught(designed, mutant):
    c = designed
    k = 10
    key = SE.abs_key(c["sim"])
    bits = SE.list_bits(c["i"], c["j"], c["bb"], c["dom_code"], c["contains"])
    sel = dict(ties_to_larger_j=_ties_to_larger_j, signed_sim=_signed, threshold_excludes_kth_key=_streaming(True),
               pass_b_sampled_blocks_only=_sampled_only,
               sample_threshold_below_k=_sample_threshold_always).get(mutant, _exact)
    if mutant == "nb_slot1_without_bb":
        nb_row = ~c["bb"].astype(bool)[c["i"]]
        bits = np.where(nb_row & (bits & 1 == 1), 1, bits).astype(np.uint8)
    caught = 0
    for r, seg, lb in _row_lists(c, bits):
        pos = np.arange(len(seg))
        for lst in range(2):
            m = ((lb >> lst) & 1) == 1
            args = (key[seg][m], c["j"][seg][m], c["sim"][seg][m], k, pos[m])
            exact = _exact(*args) if mutant != "nb_slot1_without_bb" else None
            if exact is None:        # list rule mutant: compare with the exact list of the true membership
                tm = ((SE.list_bits(c["i"][seg], c["j"][seg], c["bb"], c["dom_code"], c["contains"]) >> lst) & 1) == 1
                exact = _exact(key[seg][tm], c["j"][seg][tm], c["sim"][seg][tm], k, pos[tm])
            if not np.array_equal(sel(*args), exact):
                caught += 1
    print("%s: %d (row, list) cases differ" % (mutant, caught))
    assert caught > 0


def test_streaming_with_the_kernels_threshold_is_exact(designed):
    """The non-strict running threshold (select_cta_kernel's rule) loses nothing on the designed CTA rows."""
    c = designed
    key = SE.abs_key(c["sim"])
    bits = SE.list_bits(c["i"], c["j"], c["bb"], c["dom_code"], c["contains"])
    sel = _streaming(False)
    n = 0
    for r, seg, lb in _row_lists(c, bits):
        if len(seg) <= SE.SELECT_LONG or len(seg) > 20000:
            continue
        for lst in range(2):
            m = ((lb >> lst) & 1) == 1
            args = (key[seg][m], c["j"][seg][m], c["sim"][seg][m], 64, None)
            assert np.array_equal(sel(*args), _exact(*args))
            n += 1
    assert n > 50
