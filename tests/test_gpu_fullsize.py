"""GPU, BASELINE.json's full size (cfg2: 1 M users, 2 x 200 K items, 20 M draws): size-independent
properties of the similarity stage, the selection and the X-SIM extension -- the oracle cannot run
at this size, so the checks are internal consistency (mirror symmetry of the record lists, the
tables against an independent torch selection from the records, BB flags against the records,
sortedness, domain of X-SIM starts / ends, the exact path count of the plan)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cfg2():
    import torch
    import bench
    from xmap_b200.engine import to_device_meta
    from xmap_b200 import engine as E
    wl = bench.make_workload("cfg2")
    dev = torch.device("cuda")
    meta = to_device_meta(wl["meta"], dev)
    lay = E.build_layout(wl["user"], wl["item"], wl["rating"], wl["n_users"], wl["n_items"], device=dev)
    eng = E.SimEngine(lay, meta, "adjust_cosine", 50, wl["k"])
    tabs = eng.run()
    return dict(wl=wl, dev=dev, meta=meta, lay=lay, eng=eng, tabs=tabs)


def test_cfg2_sampled_rows_vs_oracle(cfg2):
    """The benchmarked size against the oracle port on a sample of item rows (R^T R restricted to the sampled
    rows fits in host memory): 1 000 random rows, the 40 longest neighbour lists, rows of every launch shape
    (warp rows, CTA rows of every table class, split rows).  Kept-pair sets, n, mutuality, frac, labels bit-exact,
    similarities to 1e-5 relative, BB flags of the sampled rows, and their top-k lists (order included; a list may
    differ only by similarities that are equal to 1e-9, i.e. ties decided by fp64 rounding noise in the reference)."""
    import torch
    from oracle import restate as RS
    from tests import parity as PT
    wl, eng, tabs, lay, meta = cfg2["wl"], cfg2["eng"], cfg2["tabs"], cfg2["lay"], cfg2["meta"]
    I, k = wl["n_items"], wl["k"]
    rng = np.random.default_rng(11)
    cnt = eng.rec_cnt.cpu().numpy()
    craters = (lay.csc_ptr[1:] - lay.csc_ptr[:-1]).cpu().numpy()
    work = eng.tri_work.cpu().numpy()
    picks = [rng.integers(0, I, 1000), np.argsort(-cnt)[:40], np.argsort(-craters)[:8]]
    launches, _, split = eng.plan(None)
    for r, cells_cap, threads, in_gmem, _hdr in launches:         # the heaviest and random rows of every launch group
        rr = r.cpu().numpy()
        picks.append(rr[:1]); picks.append(rng.choice(rr, size=min(3, len(rr)), replace=False))
    if split is not None:
        picks.append(split["rows"].cpu().numpy()[:4])
    rows = np.unique(np.concatenate(picks).astype(np.int64))
    Q = RS.sim_rows(wl["user"].astype(np.int64), wl["item"].astype(np.int64), wl["rating"].astype(np.float64),
                    wl["n_users"], I, wl["meta"]["prefix_code"], rows, "adjust_cosine", 50)
    PT.compare_layout(lay, Q["stats"])
    pairs = eng.emit_pairs(torch.as_tensor(rows, device=cfg2["dev"]))
    rel, fragile = PT.compare_pairs(pairs, Q["i"], Q["j"], Q["sim"], Q["mutu"], Q["frac"], Q["label"], I)
    assert np.array_equal(pairs["n"].cpu().numpy()[np.isin(pairs["i"].cpu().numpy() * I + pairs["j"].cpu().numpy(),
                                                           Q["i"] * I + Q["j"])],
                          Q["n"][np.isin(Q["i"] * I + Q["j"], pairs["i"].cpu().numpy() * I + pairs["j"].cpu().numpy())].astype(np.int64))
    assert len(fragile) <= 80, "fragile zeros among the sampled rows: %d (52 observed: regression ceiling)" % len(fragile)
    # BB flags of the sampled rows (assist.py:84-86) and their neighbour lists (extender.py:16-44); the BB
    # status of a NEIGHBOUR comes from the device flags (its own row is not in the sample)
    flags, tl, ti, ts, _, _ = PT.gpu_lists(tabs)
    bb_dev = flags.astype(bool)
    dom, contains = wl["meta"]["dom_code"], wl["meta"]["contains"]
    ptr = np.searchsorted(Q["i"], np.append(rows, I))
    near = bad = n_lists = 0
    for q, it in enumerate(rows):
        a, b = ptr[q], ptr[q + 1]
        jj, ss, lab = Q["j"][a:b], Q["sim"][a:b], Q["label"][a:b]
        bb_ref = bool((lab == 1).any())
        if bb_ref != bb_dev[it]:
            assert fragile, "BB flag of row %d differs" % it
            continue
        o = np.lexsort((jj, -np.abs(ss)))
        jj, ss = jj[o], ss[o]
        if bb_ref:
            same = ((contains[jj] >> dom[it]) & 1).astype(bool)
            want = (jj[~same][:k], jj[same][:k]); wsim = (ss[~same][:k], ss[same][:k])
        elif bb_dev[jj].any():
            isbb = bb_dev[jj]
            want = (jj[isbb][:k], jj[:k]); wsim = (ss[isbb][:k], ss[:k])
        else:
            assert tl[it, 0] == 0
            continue
        for slot in range(2):
            n_lists += 1
            got = ti[it, slot, :tl[it, slot]]
            if np.array_equal(got, want[slot]):
                assert np.allclose(ts[it, slot, :tl[it, slot]], wsim[slot], rtol=PT.SIM_RTOL, atol=0)
                continue
            if len(got) == len(want[slot]) and np.allclose(np.abs(ts[it, slot, :len(got)]), np.abs(wsim[slot]),
                                                           rtol=PT.NEAR_TIE_RTOL, atol=0):
                near += 1
                continue
            bad += 1
    assert bad == 0, "%d of %d sampled neighbour lists differ" % (bad, n_lists)
    assert near <= 12, "%d of %d sampled lists differ by near-ties (regression ceiling)" % (near, n_lists)
    print("cfg2 sampled parity: %d rows, %d kept pairs, sim max rel err %.3g, %d fragile, %d/%d near-tie lists"
          % (len(rows), len(Q["i"]), rel, len(fragile), near, n_lists))
    # the selection itself is exact on its own records: the sampled rows and every row of the CTA kernel
    from tests import select_exact as SE
    long_rows = np.nonzero(cnt > SE.SELECT_LONG)[0]
    sel_rows = torch.as_tensor(np.union1d(rows, long_rows), device=cfg2["dev"])
    n = SE.assert_engine_selection(eng, wl["meta"], sel_rows)
    ri, rj, rs = SE.engine_records(eng, sel_rows)
    labels, _ = SE.classify(ri, rj, rs, flags, dom, contains, k, I)
    print("cfg2 exact re-selection: %d rows, %d of them with more than %d records; paths %s"
          % (n, len(long_rows), SE.SELECT_LONG, SE.path_counts(labels[sel_rows.cpu().numpy()])))


def test_cfg2_xsim_sampled_starts_vs_plan_evaluation(cfg2):
    """X-SIM at the benchmarked size: the rows of sampled starts (light, median, multi-pass and the heaviest below
    2e6 paths) recomputed in numpy from the plan arrays; distinct ends, path counts, top-10 (ends and values).  The
    same starts against the extended-precision reference of tests/xsim_exact.py: every top-10 value within the
    derived rounding bound of its cell, and a top-10 position may name another end only where the two exact values
    lie within the sum of their bounds."""
    import torch
    from tests import parity as PT
    from xmap_b200 import extend as X
    tabs, lay, meta = cfg2["tabs"], cfg2["lay"], cfg2["meta"]
    plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T)
    xe = X.XsimEngine(plan, 10)
    res = xe.run()
    ub = plan.ub.cpu().numpy()
    rng = np.random.default_rng(3)
    order = np.argsort(ub)
    light = order[: len(order) // 2]
    mid = order[(ub[order] > 3e4) & (ub[order] < 3e5)]
    heavy = order[(ub[order] > 5e5) & (ub[order] < 2e6)]
    starts = np.concatenate([rng.choice(light, 12, replace=False), rng.choice(mid, 8, replace=False),
                             rng.choice(heavy, min(3, len(heavy)), replace=False)])
    ref = PT.eval_plan_starts(plan, starts)
    te, tx, tl = res.top_end.cpu().numpy(), res.top_xsim.cpu().numpy(), res.top_len.cpu().numpy()
    cnt, comb = res.count.cpu().numpy(), res.combos.cpu().numpy()
    for x in starts:
        ends, xs, n_paths = ref[int(x)]
        assert cnt[x] == len(ends) and comb[x] == n_paths == ub[x]
        o = np.lexsort((ends, -np.abs(xs)))[:10]
        L = tl[x]
        assert L == len(o)
        if not np.array_equal(te[x, :L], ends[o]):                      # only a near-tie may reorder the row
            assert np.allclose(np.abs(tx[x, :L]), np.abs(xs[o]), rtol=1e-9, atol=0), "top-10 of start %d differs" % x
        else:
            assert np.allclose(tx[x, :L], xs[o], rtol=1e-9, atol=0)
    from tests import xsim_exact as XE
    exact = XE.exact_rows(plan, starts)
    for x in starts:
        row = exact[int(x)]
        assert row["paths"] == ub[x] and cnt[x] == len(row["end"])
        XE.check_top(te[x], tx[x], tl[x], row, 10)
    assert int(xe.T.max()) > 8 and xe.n_units > plan.start_item.numel()   # multi-pass and multi-unit starts exist


def test_cfg2_properties(cfg2):
    import torch
    from xmap_b200 import extend as X
    wl, dev, meta, lay, eng, tabs = (cfg2[k] for k in ("wl", "dev", "meta", "lay", "eng", "tabs"))
    I, k = wl["n_items"], wl["k"]
    cnt = eng.rec_cnt.long()
    total = int(cnt.sum())
    assert tabs.n_pairs_total == 2 * int(eng.row_npairs.sum()) and total % 2 == 0 and total > 2e8

    # ---- record lists: every (i -> j) has a mirror (j -> i) with identical sim bits, n and mutu ----------
    i = torch.repeat_interleave(torch.arange(I, device=dev), cnt)
    src = eng.rec_ptr[:-1][i] + (torch.arange(total, device=dev) - (torch.cumsum(cnt, 0) - cnt)[i])
    sim_bits = eng.rec[src, 0]
    pack = eng.rec[src, 1]
    j = pack & 0xFFFFFFFF
    fwd = torch.argsort(i * I + j)
    rev = torch.argsort(j * I + i)
    assert torch.equal((i * I + j)[fwd], (j * I + i)[rev])              # same key multiset, no duplicates ...
    assert bool(((i * I + j)[fwd][1:] > (i * I + j)[fwd][:-1]).all())
    assert torch.equal(sim_bits[fwd], sim_bits[rev])                    # ... and bitwise equal payloads
    assert torch.equal(pack[fwd] >> 32, pack[rev] >> 32)
    n, mutu = eng.rec_n[src].long(), (pack >> 32) & 0xFFFFFFFF
    assert torch.equal(n[fwd], n[rev])
    sim = sim_bits.view(torch.float64)
    assert bool((mutu >= 1).all()) and bool((mutu <= n).all()) and bool((sim != 0).all())
    assert float(sim.abs().max()) <= 1.0 + 1e-12
    c = lay.item_stats[:, 3].long()
    assert bool((n <= torch.minimum(c[i], c[j])).all())
    del fwd, rev, src

    # ---- BB flags = "has a kept cross-domain pair" (assist.py:84-86) --------------------------------------
    cross = meta.prefix_code[i] != meta.prefix_code[j]
    bb_ref = torch.zeros(I, dtype=torch.bool, device=dev)
    bb_ref[i[cross]] = True
    assert torch.equal(bb_ref, tabs.row_flags.bool())

    # ---- tables vs an independent selection from the records, on a sample of rows incl. the longest lists --
    g = torch.Generator(device="cpu").manual_seed(5)
    sample = torch.cat([torch.randint(0, I, (1500,), generator=g), torch.argsort(cnt.cpu(), descending=True)[:40]]).unique()
    ptr = (torch.cumsum(cnt, 0) - cnt).cpu()
    bad = 0
    contains, dom = meta.contains.long(), meta.dom_code.long()
    tl, ti, ts = tabs.tab_len.cpu(), tabs.tab_idx.cpu(), tabs.tab_sim.cpu()
    for r in sample.tolist():
        a, b = int(ptr[r]), int(ptr[r]) + int(cnt[r])
        jr, sr = j[a:b], sim[a:b]
        if bool(bb_ref[r]):
            same = ((contains[jr] >> dom[r]) & 1).bool()
            lists = (~same, same)
        else:
            lists = (bb_ref[jr], torch.ones_like(jr, dtype=torch.bool))
        for slot, m in enumerate(lists):
            jj, ss = jr[m], sr[m]
            o = torch.argsort(jj)                                       # ties to the smaller index: stable sort
            jj, ss = jj[o], ss[o]
            o = torch.argsort(-ss.abs(), stable=True)[:k]
            want_j, want_s = jj[o].cpu(), ss[o].cpu()
            L = int(tl[r, slot])
            if L != len(want_j) or not torch.equal(ti[r, slot, :L].long(), want_j) or not torch.equal(ts[r, slot, :L], want_s):
                bad += 1
    assert bad == 0, "%d of %d sampled lists differ from the torch selection" % (bad, 2 * len(sample))
    del i, j, sim, sim_bits, pack, n, mutu, cross

    # ---- X-SIM: starts in T, ends in S, rows sorted, path count = the plan's exact bound ---------------------
    plan = X.build_plan(tabs, lay.item_stats[:, 3].contiguous(), meta.has_S, meta.has_T)
    res = X.XsimEngine(plan, 10).run()
    assert int(res.combos.sum()) == int(plan.ub.sum())
    assert bool(meta.has_T[res.start_item.long()].all())
    valid = torch.arange(10, device=dev)[None, :] < res.top_len[:, None]
    assert bool(meta.has_S[res.top_end.long().clamp(min=0)][valid].all())
    assert bool((res.top_len.long() == torch.clamp(res.count.long(), max=10)).all())
    ax = res.top_xsim.abs()
    ok = (ax[:, :-1] > ax[:, 1:]) | ((ax[:, :-1] == ax[:, 1:]) & (res.top_end[:, :-1] < res.top_end[:, 1:]))
    assert bool(ok[valid[:, 1:]].all())
    assert float(ax[valid].max()) <= 1.0 + 1e-9
