"""GPU: the X-SIM kernels against the extended-precision reference of tests/xsim_exact.py, cell by cell within the
derived rounding bound, on cases whose path structure is built to reach the kernels' edges, over every schedule the
engine has, and at top_m 1, 2, 31, 32, 33, 63 and 64.

For every case and plan: the (start, end) key set is the reference's; every value is within its cell's bound; per
start the distinct-end count is the reference's and the path count is plan.ub and the paths enumerated; every top-m
row is, bit for bit, the first top_m of the kernel's own emitted row (|xsim| desc, then the smaller end), and where it
names another end than the exact top-m the two exact values lie within the sum of their bounds; a second run of the
same plan gives identical bits.

What no engine attribute shows, and why the shapes force it:
  * device-side splits: `device_splits` and `cta_splits` give every start one pass (rho = 1e9, asserted: T == 1),
    so `pressure`'s start with 57 distinct ends cannot fit 7/8 of a 64-cell warp table (56 cells), its starts with
    57 ends in one CTA owner region cannot fit 7/8 of a 64-cell region, and its start with 50 + 10 ends in sibling
    tiles 6 and 7 (gb = 4, asserted) fits only once the halving reaches single tiles.  The starts with 55 and 56 ends
    sit just below and at the threshold.
  * the warp kernel's slow top-m path (topm_rounds) runs on every pass at top_m 33, 63 and 64 (the fast path needs
    top_m <= 32).  At top_m 31 and 32 it runs when more than 32 cells are not worse than the top_m-th best of the 32
    lanes' maxima: on a pass of `ties` with 300 or 600 ends every lane holds several cells of value 0.5, the threshold
    is nearly the weakest lane maximum, and far more than 32 cells pass it.
  * the CTA kernel's XSURV fallback: every cell of `ties` falls into one histogram bin, so all the ends of a pass
    survive the bin threshold; the CTA plans run the 300- and 600-end starts in one pass (cells_lg 12: asserted
    T == 1), and 300 > 256 = XSURV.
  * a split plan on a start whose ends crowd one hash tile past the table (`batches`: 61 to 63 ends of a tile against
    the 56 of a 64-cell warp table) must fail with the kernel's error 2; that plan is then checked one table size up.
  * xsim_merge_kernel with M > 32 over several units: `many_units` cuts starts into several units (asserted), among
    them starts with at least 64 ends (asserted), and runs top_m 33, 63 and 64."""
import time

import numpy as np
import pytest

from tests import parity as PT
from tests import xsim_exact as XE

pytestmark = pytest.mark.gpu

TOPMS = (1, 2, 31, 32, 33, 63, 64)
REPORT = {}


def plans(ub):
    W = dict(mode="warp")
    return dict(warp=dict(W), cta=dict(mode="cta"),
                hybrid_some_hot=dict(mode="hybrid", cells_lg=6, unit_work=max(8, int(ub.max()) // 4)),
                hybrid_all_hot=dict(mode="hybrid", hot_paths=0.0),
                device_splits=dict(W, cells_lg=6, rho=1e9, max_passes=10 ** 9),
                cta_splits=dict(mode="cta", cells_lg=9, rho=1e9),
                global_tables=dict(W, cells_lg=6, max_passes=1),
                many_units=dict(W, cells_lg=6, unit_work=max(8, int(ub.max()) // 8)),
                unfused=dict(W, fuse=False))


def some_hot(plan, kw):
    """A hot-unit threshold that puts some units of the plan on the CTA kernel and the others on the warp kernel."""
    from xmap_b200 import extend as X
    est = np.sort(X.XsimEngine(plan, 1, **kw).unit_est_paths.cpu().numpy())
    return float(est[(len(est) - 1) // 2])


def one_tile_overflow(name, cells_lg, ends_of):
    """Whether a one-pass split plan (gb = 4) must fail with error 2: some start holds, in one hash tile, more ends
    than 7/8 of the warp table (device_splits) or of one CTA owner region (cta_splits, 2^(cells_lg - 3) cells)."""
    if name == "device_splits":
        cap = (1 << cells_lg) - (1 << (cells_lg - 3))
        return any(np.bincount(XE.pi_tile(e, 4)).max(initial=0) > cap for e in ends_of)
    rb = cells_lg - 3
    cap = (1 << rb) - (1 << (rb - 3))
    return any(np.bincount(XE.pi_tile(e, 4) * 8 + XE.cta_owner(e)).max(initial=0) > cap for e in ends_of)


def _assert_schedule(name, xe, plan, res):
    n = plan.start_item.numel()
    if name in ("warp", "device_splits", "global_tables", "many_units", "unfused"):
        assert xe.hot_order.numel() == 0 and xe.cold_order.numel() == xe.n_units
    if name in ("cta", "cta_splits", "hybrid_all_hot"):
        assert xe.cold_order.numel() == 0 and xe.hot_order.numel() == xe.n_units
    if name == "hybrid_some_hot":
        assert xe.hot_order.numel() > 0 and xe.cold_order.numel() > 0
    if name in ("device_splits", "cta_splits"):
        assert int(xe.T.max()) == 1 and xe.gb == 4
    if name == "global_tables":
        assert xe.gws is not None and int(xe.unit_clg.max()) > xe.cells_lg
    if name == "many_units":
        multi = np.diff(xe.start_unit_ptr.cpu().numpy()) > 1
        cnt = res.count.cpu().numpy()
        assert xe.n_units > n and ((cnt[multi] >= 64).any() or (cnt < 64).all())
    if name == "unfused":
        assert xe.fused_entries == 0


def _kernel_rows(xe, res, s, e, v):
    """The kernel's own emitted rows, |xsim| desc then the smaller end, padded to 64: (ends, values, lengths)."""
    st = xe.plan.start_item.cpu().numpy()
    n = len(st)
    si = np.searchsorted(st, s)
    o = np.lexsort((e, -np.abs(v), si))
    si, e, v = si[o], e[o], v[o]
    ptr = np.searchsorted(si, np.arange(n + 1))
    rank = np.arange(len(si)) - ptr[si]
    keep = rank < 64
    KE = np.full((n, 64), -1, np.int64); KX = np.zeros((n, 64))
    KE[si[keep], rank[keep]] = e[keep]; KX[si[keep], rank[keep]] = v[keep]
    return KE, KX, np.minimum(np.diff(ptr), 64), np.diff(ptr)


def run_case(case, tabs, plan, ref, extra=None, topms=TOPMS):
    """Every plan of `plans` and every top_m on one case; ref: {start index: reference row} (every start, or a
    sample).  extra(name, xe): case-specific assertions on the schedule."""
    from xmap_b200 import _native as N
    from xmap_b200 import extend as X
    ub = plan.ub.cpu().numpy()
    st = plan.start_item.cpu().numpy()
    rs = sorted(ref)
    assert all(ref[x]["paths"] == ub[x] for x in rs)
    worst, cells, near = 0.0, 0, 0
    ends_of = None                                         # every start's ends, from the first plan's emission
    for name, kw in plans(ub).items():
        if name == "hybrid_some_hot":
            kw = dict(kw, hot_paths=some_hot(plan, kw))
        if name in ("device_splits", "cta_splits") and one_tile_overflow(name, kw["cells_lg"], ends_of):
            # the kernel must report that a single hash tile overflows its table; then the same schedule, one size up
            with pytest.raises(N.NativeError, match="kernel error 2"):
                X.XsimEngine(plan, 64, **kw).run()
            kw = dict(kw, cells_lg=kw["cells_lg"] + 1)
            REPORT.setdefault("error_2", []).append((case, name))
        xe = X.XsimEngine(plan, 64, **kw)
        res = xe.run()
        s, e, v = (t.cpu().numpy() for t in xe.emit(res))
        if ends_of is None:
            si0 = np.searchsorted(st, s)
            ends_of = np.split(e, np.searchsorted(si0, np.arange(1, len(st))))
        _assert_schedule(name, xe, plan, res)
        if extra:
            extra(name, xe)
        cnt, comb = res.count.cpu().numpy(), res.combos.cpu().numpy()
        assert np.array_equal(comb, ub), name
        KE, KX, KL, kcnt = _kernel_rows(xe, res, s, e, v)
        assert np.array_equal(kcnt, cnt), name
        si = np.searchsorted(st, s)
        ptr = np.searchsorted(si, np.arange(len(st) + 1))
        for x in rs:
            row = ref[x]
            assert cnt[x] == len(row["end"]), (name, x)
            assert np.array_equal(e[ptr[x]:ptr[x + 1]], row["end"]), (name, x)
            r = XE.err_ratio(v[ptr[x]:ptr[x + 1]], row)
            assert r.max(initial=0.0) <= 1.0 + XE.REF_SHARE, (name, x, r.max())
            worst = max(worst, float(r.max(initial=0.0)))
            cells += len(row["end"])
        # the same plan again: identical bits
        res2 = xe.run()
        s2, e2, v2 = (t.cpu().numpy() for t in xe.emit(res2))
        assert np.array_equal(e, e2) and np.array_equal(v.view(np.int64), v2.view(np.int64)), name
        for f in ("count", "combos", "top_end", "top_len"):
            assert np.array_equal(getattr(res, f).cpu().numpy(), getattr(res2, f).cpu().numpy()), (name, f)
        assert np.array_equal(res.top_xsim.cpu().numpy().view(np.int64), res2.top_xsim.cpu().numpy().view(np.int64))
        for m in topms:
            rm = res if m == 64 else X.XsimEngine(plan, m, **kw).run()
            te, tx, tl = rm.top_end.cpu().numpy(), rm.top_xsim.cpu().numpy(), rm.top_len.cpu().numpy()
            assert np.array_equal(tl, np.minimum(cnt, m)), (name, m)
            valid = np.arange(m)[None, :] < tl[:, None]
            assert np.array_equal(np.where(valid, te, -1), np.where(valid, KE[:, :m], -1)), (name, m)
            assert np.array_equal(np.where(valid, tx, 0.0).view(np.int64), np.where(valid, KX[:, :m], 0.0).view(np.int64)), (name, m)
            for x in rs:
                near += XE.check_top(te[x], tx[x], tl[x], ref[x], m)
    REPORT[case] = dict(cells_checked=cells, plans=len(plans(ub)), max_err_over_bound=worst, near_tie_positions=near)
    print("X-SIM exact [%s]: %d cells checked over %d plans, max |err| / bound %.3g, %d near-tie top-m positions"
          % (case, cells, len(plans(ub)), worst, near))
    return REPORT[case]


def _designed(name):
    tabs = XE.DESIGNED[name]().tables("cuda")
    plan = XE.build_plan(tabs)
    return tabs, plan, XE.exact_rows(plan, range(plan.start_item.numel()))


def test_batches_and_list_lengths():
    """31/32/33 and 255/256/257 (leg, partner) pairs per start (the warp kernel's 32-pair batch, the CTA kernel's
    256-pair macro-batch) over right-segment lists of 2 .. 65 entries."""
    tabs, plan, ref = _designed("batches")
    run_case("batches", tabs, plan, ref)


def test_runs_of_equal_ends_in_fused_lists():
    """Runs of 1, 31, 32, 33 and 100 equal ends in a fused bridge list, walked by joint-only legs of type 1 and 2,
    across the 32-path chunks of the segmented scan and the MATCH.ANY grouping; unfused in `unfused`."""
    tabs, plan, ref = _designed("runs")

    def fused(name, xe):
        assert (xe.fused_entries > 0) == (name != "unfused")
    run_case("runs", tabs, plan, ref, fused)


def test_table_pressure_and_single_tile_splits():
    tabs, plan, ref = _designed("pressure")
    run_case("pressure", tabs, plan, ref)


def test_signs_and_exact_zeros():
    tabs, plan, ref = _designed("signs")
    zero = ref[0]["x"] == 0
    assert zero.sum() == 5
    from xmap_b200 import extend as X
    for kw in plans(plan.ub.cpu().numpy()).values():
        xe = X.XsimEngine(plan, 64, **kw)
        s, e, v = (t.cpu().numpy() for t in xe.emit(xe.run()))
        assert np.all(v[(s == int(plan.start_item[0])) & np.isin(e, ref[0]["end"][zero])] == 0.0)
    run_case("signs", tabs, plan, ref)


def test_exact_ties_top_m_is_the_smallest_ends():
    """Every cell exactly +-0.5: the top-m of every plan is the m smallest ends with the exact values, bit for bit
    (the slow top-m paths of both kernels; see the module docstring)."""
    from xmap_b200 import extend as X
    tabs, plan, ref = _designed("ties")

    def one_pass(name, xe):
        if name in ("cta", "hybrid_all_hot"):
            assert int(xe.unit_npass.max()) == 1 and xe.n_units == plan.start_item.numel()
    run_case("ties", tabs, plan, ref, one_pass)
    for kw in plans(plan.ub.cpu().numpy()).values():
        for m in TOPMS:
            r = X.XsimEngine(plan, m, **kw).run()
            te, tx = r.top_end.cpu().numpy(), r.top_xsim.cpu().numpy()
            for x in ref:
                want = ref[x]["end"][:m]
                assert np.array_equal(te[x][:len(want)], want) and np.all(tx[x][:len(want)] == ref[x]["x"][:m]), (kw, m, x)


def test_overflow_at_one_tile_raises_error_2():
    """118 ends in one hash tile exceed 7/8 of the unit's 128-cell global-memory table; the pass cannot be split
    further, so the run raises the kernel's error 2 and returns nothing; the error flag is cleared, so a good plan
    runs afterwards."""
    from xmap_b200 import _native as N
    from xmap_b200 import extend as X
    plan = XE.build_plan(XE.case_overflow().tables("cuda"))
    xe = X.XsimEngine(plan, 10, mode="warp", cells_lg=6, rho=2.0, max_passes=1)
    assert xe.gws is not None and int(xe.unit_clg[0]) == 7 and xe.gb == 4
    with pytest.raises(N.NativeError, match="kernel error 2"):
        xe.run()
    assert int(xe.error_flag.item()) == 0
    _, plan2, _ = _designed("pressure")
    res = X.XsimEngine(plan2, 10, mode="warp").run()
    assert int(res.combos.sum()) == int(plan2.ub.sum())


def _sim_case(case, n_sample=300, seed=0):
    from xmap_b200 import extend as X
    lay, _, tabs, _ = PT.run_gpu_sim(case["user"], case["item"], case["rating"], case["n_users"], case["n_items"],
                                     case["meta"], "adjust_cosine", 50, 5, emit=False)
    dm = PT.to_device_meta(case["meta"])
    plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), dm.has_S, dm.has_T)
    ub = plan.ub.cpu().numpy()
    rng = np.random.default_rng(seed)
    heavy = np.argsort(-ub)[:20]
    rest = np.setdiff1d(np.arange(len(ub)), heavy)
    starts = np.concatenate([heavy, rng.choice(rest, min(n_sample - 20, len(rest)), replace=False)])
    return tabs, plan, XE.exact_rows(plan, starts)


def test_sim_derived_synth_case():
    """The case test_gpu_extend uses: every cell of 300 sampled starts, the 20 heaviest among them."""
    t0 = time.time()
    tabs, plan, ref = _sim_case(PT.synth_case(4000, 900, 60000, 0.04, seed=21))
    assert len(ref) >= 300
    run_case("synth", tabs, plan, ref)
    print("synth case %.1f s" % (time.time() - t0))


def test_sim_derived_multi_domain_cases():
    for lab, case in PT.multi_domain_cases(4500, 500, 60000, 0.08, seed=31):
        tabs, plan, ref = _sim_case(case)
        assert len(ref) >= min(300, plan.start_item.numel())
        run_case("multi " + lab, tabs, plan, ref)
