"""CPU: the X-SIM reference of tests/xsim_exact.py -- its bound holds for fp64 sums in other orders, it agrees
with rational arithmetic, it is tight enough to see one path lost or counted twice -- and the designed cases hold
the path structures they are built for."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import restate as RS
from tests import parity as PT
from tests import xsim_exact as XE


def _golden_plan(name):
    import torch
    from xmap_b200 import extend as X
    g = PT.load_golden(name)
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    P = RS.sim_pairs(g["user"].astype(np.int64), g["item"].astype(np.int64), g["rating"], nU, nI,
                     meta["prefix_code"], str(g["method"]), int(g["num_atleast"]))
    knn = RS.select_knn(P, nI, int(g["k"]), meta["dom_code"], meta["contains"])
    tabs = PT.tables_from_restatement(P, knn, nI, int(g["k"]))
    plan = X.build_plan(tabs, torch.as_tensor(P["stats"]["count"]), torch.as_tensor(meta["has_S"]),
                        torch.as_tensor(meta["has_T"]))
    return g, P, knn, meta, plan


def _flat(plan, ref):
    st = plan.start_item.numpy()
    keys = np.concatenate([st[x] * plan.n_items + ref[x]["end"] for x in sorted(ref)])
    cat = lambda f: np.concatenate([ref[x][f] for x in sorted(ref)])
    return keys, dict(x_ld=cat("x_ld"), bound=cat("bound"), n=cat("n"), x=cat("x"))


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_golden_and_restatement_sums_lie_within_the_bound(name):
    """The reference's own fp64 X-SIM (golden xs_val) and oracle/restate.xsim_extend sum the same paths in other
    orders: both must fall inside the bound of every cell, and the key sets must be the reference's."""
    g, P, knn, meta, plan = _golden_plan(name)
    ref = XE.exact_rows(plan, range(plan.start_item.numel()))
    keys, flat = _flat(plan, ref)
    nI = plan.n_items
    Xr = RS.xsim_extend(P, knn, nI, meta["has_S"], meta["has_T"])
    for s, e, v in ((g["xs_start"], g["xs_end"], g["xs_val"]), (Xr["start"], Xr["end"], Xr["xsim"])):
        assert np.array_equal(s.astype(np.int64) * nI + e, keys)
        r = XE.err_ratio(v, flat)
        assert r.max() <= 1.0 + XE.REF_SHARE, r.max()
    assert sum(ref[x]["paths"] for x in ref) == Xr["combos"]


def test_reference_agrees_with_rational_arithmetic():
    """On the cells of adj_all_bridge the extended-precision reference is within its own stated error (REF_SHARE of
    the bound) of the value evaluated in fractions.Fraction, exactly."""
    _, _, _, _, plan = _golden_plan("adj_all_bridge")
    P = XE._plan_arrays(plan)
    checked = 0
    for x in range(plan.start_item.numel()):
        y, e, m, f = XE.enumerate_paths(P, x)
        row = XE.cells_of_paths(y, e, m, f)
        num, den = {}, {}
        for p in range(len(y)):
            D = int(m[:, p].sum())
            s = sum(Fraction(float(v)) for v in e[:, p]) / D if D else Fraction(0)
            c = Fraction(1)
            for v in f[:, p]:
                c *= Fraction(float(v))
            num[int(y[p])] = num.get(int(y[p]), 0) + s * c
            den[int(y[p])] = den.get(int(y[p]), 0) + c
        for q, end in enumerate(row["end"]):
            exact = num[int(end)] / den[int(end)]
            d = abs(Fraction(*row["x_ld"][q].as_integer_ratio()) - exact)
            assert d <= Fraction(XE.REF_SHARE) * Fraction(float(row["bound"][q])), (x, end)
            checked += 1
    assert checked > 400


def _sensitivity(plan, starts, heaviest):
    """Per cell among the `heaviest` (most paths, n >= 2): does dropping the path of largest c_p, or counting it
    twice, move the exact value by more than 10 bounds?"""
    P = XE._plan_arrays(plan)
    cells = []
    for x in starts:
        y, e, m, f = XE.enumerate_paths(P, x)
        row = XE.cells_of_paths(y, e, m, f)
        D = m.sum(0)
        c = f.astype(XE.LD).prod(0)
        s = np.where(D != 0, e.astype(XE.LD).sum(0) / np.where(D != 0, D, 1), 0)
        for q in np.flatnonzero(row["n"] >= 2):
            idx = np.flatnonzero(y == row["end"][q])
            j = idx[np.argmax(c[idx])]
            SN, SD = (s[idx] * c[idx]).sum(), c[idx].sum()
            X = SN / SD
            moved = [abs(float((SN - s[j] * c[j]) / (SD - c[j]) - X)), abs(float((SN + s[j] * c[j]) / (SD + c[j]) - X))]
            cells.append((row["n"][q], min(moved) > 10 * row["bound"][q]))
    cells.sort(key=lambda t: -t[0])
    return [ok for _, ok in cells[:heaviest]]


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_a_lost_or_doubled_path_exceeds_the_bound(name):
    """The bound is tight enough to see a kernel drop one path of a cell or count it twice: on the 200 heaviest
    cells, the largest-weight path moves the exact value by more than 10x the bound on >= 90 % of them."""
    _, _, _, _, plan = _golden_plan(name)
    ok = _sensitivity(plan, range(plan.start_item.numel()), 200)
    assert len(ok) >= 20 and np.mean(ok) >= 0.9, (len(ok), np.mean(ok))


@pytest.mark.parametrize("name", ["batches", "runs", "signs"])
def test_a_lost_or_doubled_path_exceeds_the_bound_designed(name):
    plan = XE.build_plan(XE.DESIGNED[name]().tables())
    ok = _sensitivity(plan, range(plan.start_item.numel()), 200)
    assert len(ok) >= 20 and np.mean(ok) >= 0.9, (len(ok), np.mean(ok))


def test_designed_cases_hold_their_structures(native_built):
    """What the GPU tests rely on: the pair counts and list lengths of `batches`, the runs of equal ends in the fused
    list of `runs`, the fill of `pressure` (total, per CTA owner region, per hash tile), the exact zeros of `signs`,
    the tie values and end counts of `ties`."""
    from xmap_b200 import extend as X
    plan = XE.build_plan(XE.case_batches().tables())
    xe = X.XsimEngine(plan, 10, mode="warp", fuse=False)
    pairs = np.diff(xe.lp_ptr.numpy()[plan.leg_ptr.numpy()])
    assert set(XE.PARTNER_COUNTS) <= set(pairs.tolist())
    assert set(XE.LIST_LENGTHS) <= set(np.diff(plan.rs_ptr.numpy()).tolist())

    plan = XE.build_plan(XE.case_runs().tables())
    xe = X.XsimEngine(plan, 10, mode="warp")
    assert xe.fused_entries > 0
    n_s = len(plan.rs_ptr) - 1                          # the fused lists follow the right-segment lists
    fe = xe.rs_end.numpy()[int(xe.rs_ptr[n_s]):]
    cut = np.flatnonzero(np.diff(fe)) + 1
    runs = np.diff(np.concatenate([[0], cut, [len(fe)]]))
    assert set(XE.RUN_LENGTHS) <= set(runs.tolist())
    assert sorted(np.diff(plan.leg_ptr.numpy()).tolist()) == [1, 1, 1, 1]    # t (type 0), a (type 1), x1, x2 (type 2)

    plan = XE.build_plan(XE.case_pressure().tables())
    ref = XE.exact_rows(plan, range(plan.start_item.numel()))
    ends = [ref[x]["end"] for x in sorted(ref)]
    assert [len(e) for e in ends[:3]] == list(XE.WARP_FILL)
    assert [int((XE.cta_owner(e) == 0).sum()) for e in ends[3:6]] == list(XE.WARP_FILL)
    assert all(int((XE.cta_owner(e) == 1).sum()) == 5 for e in ends[3:6])
    tiles = XE.pi_tile(ends[6], 4)
    assert [int((tiles == g).sum()) for g in XE.SPLIT_TILES] == [50, 10] and len(tiles) <= 62      # + s and n

    plan = XE.build_plan(XE.case_overflow().tables())
    e = XE.exact_rows(plan, [0])[0]["end"]
    assert np.bincount(XE.pi_tile(e, 4)).max() >= 118

    plan = XE.build_plan(XE.case_signs().tables())
    r0 = XE.exact_rows(plan, [0])[0]
    assert int((r0["x"] == 0).sum()) == 5 and int((r0["n"] == 2).sum()) == 5

    plan = XE.build_plan(XE.case_ties().tables())
    ref = XE.exact_rows(plan, range(plan.start_item.numel()))
    assert sorted(len(ref[x]["end"]) for x in ref) == sorted(XE.TIE_ENDS)
    assert all(np.all(np.abs(ref[x]["x"]) == 0.5) for x in ref)
