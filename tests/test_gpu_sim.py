"""GPU parity: similarity + selection through the C ABI vs the oracle."""
import numpy as np
import pytest

from tests import parity as PT

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_sim_matches_reference_golden(name):
    """Kept pairs / mutu / frac / label bit-exact, sim <= 1e-5 rel, neighbour lists
    identical to what the UNMODIFIED reference produced (tests/golden)."""
    g = PT.load_golden(name)
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    lay, eng, tabs, pairs = PT.run_gpu_sim(g["user"], g["item"], g["rating"], nU, nI, meta,
                                           str(g["method"]), int(g["num_atleast"]), int(g["k"]))
    # reference item_info = (avg, norm2, adj_norm2, count); user_avg
    its = lay.item_stats.cpu().numpy()
    assert np.array_equal(lay.user_mu.cpu().numpy(), g["user_avg"])
    assert np.array_equal(its[:, 0], g["item_info"][:, 0])
    assert np.array_equal(its[:, 3], g["item_info"][:, 3])
    np.testing.assert_allclose(its[:, 1:3], g["item_info"][:, 1:3], rtol=1e-13)
    rel, fragile = PT.compare_pairs(pairs, g["sim_i"], g["sim_j"], g["sim_val"], g["sim_mutu"],
                                    g["sim_frac"], g["sim_label"], nI)
    assert not fragile          # the golden cases contain no cancelling inner products
    lists = {n: (g[n + "_ptr"], g[n + "_nbr"]) for n in ("BB_BB", "BB_NB", "NB_BB", "NB_NN")}
    PT.compare_knn(tabs, g["bb"], g["valid_nb"], lists)


def test_sim_matches_reference_mid_size_golden():
    """The CTA launch shapes and the histogram path of the selection against the UNMODIFIED reference: the
    mid-size golden (90 K ratings, 366 K kept pairs, rows of up to 3 900 co-rating products, lists of ~1e3 neighbours)."""
    g = PT.load_golden("adj_mid")
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    lay, eng, tabs, pairs = PT.run_gpu_sim(g["user"], g["item"], g["rating"], nU, nI, meta,
                                           str(g["method"]), int(g["num_atleast"]), int(g["k"]))
    kinds = _kinds(dict(tabs=tabs))
    assert any(k.endswith("_t32") for k in kinds) and sum(1 for k in kinds if not k.endswith("_t32")) >= 3, kinds
    assert np.array_equal(lay.user_mu.cpu().numpy(), g["user_avg"])
    its = lay.item_stats.cpu().numpy()
    assert np.array_equal(its[:, 0], g["item_info"][:, 0]) and np.array_equal(its[:, 3], g["item_info"][:, 3])
    gi, gj = pairs["i"].cpu().numpy(), pairs["j"].cpu().numpy()
    assert np.array_equal(gi, g["sim_i"]) and np.array_equal(gj, g["sim_j"]), "kept-pair sets differ"
    assert np.array_equal(pairs["mutu"].cpu().numpy(), g["sim_mutu"]) and np.array_equal(pairs["label"].cpu().numpy(), g["sim_label"])
    known = np.isfinite(g["sim_val"])          # similarity and frac are stored for a fixed sample of the pairs
    assert known.sum() > 70000
    assert np.array_equal(pairs["frac"].cpu().numpy()[known].astype(np.float32), g["sim_frac"][known])
    rel = np.zeros(len(known))
    rel[known] = np.abs(pairs["sim"].cpu().numpy()[known] - g["sim_val"][known]) / np.abs(g["sim_val"][known])
    # |sim| < 1e-13 is the rounding residue of an inner product that cancels exactly (here one pair of two co-raters,
    # 1.1e-19 in the reference, 1.5e-19 here): not comparable digit by digit, see DESIGN.md 6.1
    rel[known & (np.abs(g["sim_val"]) < PT.FRAGILE_SIM)] = 0.0
    assert int((np.abs(g["sim_val"][known]) < PT.FRAGILE_SIM).sum()) <= 2
    if rel.max() > PT.SIM_RTOL:
        bad = np.flatnonzero(rel > PT.SIM_RTOL)
        cnt = its[:, 3]
        od = eng.ord.cpu().numpy(); tw = eng.tri_work.cpu().numpy()
        msg = ["%d of %d pairs off" % (len(bad), len(rel))]
        for q in bad[:12]:
            a, b = int(gi[q]), int(gj[q])
            lo = a if od[a] < od[b] else b
            msg.append("(%d,%d) n=%d gpu=%.6g ref=%.6g ratio=%.6f cnt=(%d,%d) row=%d ord=%d work=%d rtop=%d" % (
                a, b, int(pairs["n"][q]), float(pairs["sim"][q]), g["sim_val"][q], float(pairs["sim"][q]) / g["sim_val"][q],
                cnt[a], cnt[b], lo, od[lo], tw[lo], nI - 1 - od[lo]))
        raise AssertionError("; ".join(msg))
    lists = {n: (g[n + "_ptr"], g[n + "_nbr"]) for n in ("BB_BB", "BB_NB", "NB_BB", "NB_NN")}
    key = g["sim_i"].astype(np.int64) * nI + g["sim_j"]

    def ref_sim(it, j):
        q = np.searchsorted(key, it * nI + j)
        return g["sim_val"][q] if q < len(key) and key[q] == it * nI + j else 0.0
    near = PT.compare_knn(tabs, g["bb"], g["valid_nb"], lists, ref_sim=ref_sim)
    assert near <= 2, "%d lists differ from the reference by near-ties (regression ceiling)" % near


def _kinds(out):
    return [k for k, _ in out["tabs"].stats["accumulate"]]


@pytest.mark.parametrize("method", ["adjust_cosine", "cosine"])
def test_sim_all_tiers_vs_restatement(method):
    """Large enough that warp-per-row and CTA-per-row launches of several table sizes run, with both
    hashed and direct-indexed tables, and that the long-list selection kernel is exercised."""
    case = PT.synth_case(20000, 3000, 400000, 0.05, seed=11, half=(method == "cosine"))
    out = PT.check_sim_against_restatement(case, method, 50, 10)
    kinds = _kinds(out)
    assert any(k.endswith("_t32") for k in kinds) and any(not k.endswith("_t32") for k in kinds), kinds
    assert len(kinds) >= 4, kinds
    eng = out["eng"]
    I = case["n_items"]
    rtop = (I - 1 - eng.ord).long()
    h = ((eng.tri_work * 4 + 2) // 3).clamp(min=32)
    live = eng.tri_work > 0
    assert int(((rtop <= h) & live).sum()) > 0 and int(((rtop > h) & live).sum()) > 0   # direct and hashed rows


def test_wide_catalogue():
    """A wider catalogue (more hashed rows, bigger tables), against the restatement."""
    case = PT.synth_case(30000, 12000, 500000, 0.05, seed=13)
    out = PT.check_sim_against_restatement(case, "adjust_cosine", 50, 10)
    assert out["tabs"].n_pairs_total == out["P"]["n_pairs_total"]
    assert int((out["eng"].rec_cnt > 8192).sum()) > 0     # long rows: select_cta_kernel


def test_global_memory_tables_give_identical_results():
    """Tiny shared-memory table limit -> most rows run with their table in global memory (the
    fallback for rows that exceed shared memory); results must not change."""
    case = PT.synth_case(6000, 1200, 120000, 0.1, seed=5)
    a = PT.check_sim_against_restatement(case, "adjust_cosine", 50, 7)
    b = PT.check_sim_against_restatement(case, "adjust_cosine", 50, 7, max_smem_cells=64)
    assert any("accumulate_g" in k for k in _kinds(b)) and not any("accumulate_g" in k for k in _kinds(a))
    for k in ("i", "j", "sim", "mutu", "n"):
        assert np.array_equal(a["pairs"][k].cpu().numpy(), b["pairs"][k].cpu().numpy()), k
    for t in ("tab_idx", "tab_sim", "tab_len", "row_flags"):
        assert np.array_equal(getattr(a["tabs"], t).cpu().numpy(), getattr(b["tabs"], t).cpu().numpy()), t


def test_split_rows_give_identical_results(monkeypatch):
    """Rows with long rater lists cut into segments over several CTAs (merged through a global table
    with exact integer adds): forcing the split on a small case must not change a bit."""
    from xmap_b200 import engine as E
    case = PT.synth_case(6000, 1200, 120000, 0.1, seed=5)
    a = PT.check_sim_against_restatement(case, "adjust_cosine", 50, 7)
    assert not any(k == "accumulate_split" for k in _kinds(a))
    monkeypatch.setattr(E, "SPLIT_RATERS", 64)
    monkeypatch.setattr(E, "SPLIT_SEG", 96)
    b = PT.check_sim_against_restatement(case, "adjust_cosine", 50, 7)
    assert dict(b["tabs"].stats["accumulate"])["accumulate_split"] > 10
    for k in ("i", "j", "sim", "mutu", "n"):
        assert np.array_equal(a["pairs"][k].cpu().numpy(), b["pairs"][k].cpu().numpy()), k
    for t in ("tab_idx", "tab_sim", "tab_len", "row_flags"):
        assert np.array_equal(getattr(a["tabs"], t).cpu().numpy(), getattr(b["tabs"], t).cpu().numpy()), t
    tabs2 = b["eng"].run()                                # the global tables and counters were left clean
    assert np.array_equal(tabs2.tab_idx.cpu().numpy(), a["tabs"].tab_idx.cpu().numpy())


def test_exact_list_sizing_gives_identical_results():
    """When the upper bound on the record lists does not fit in memory the engine sizes them with a
    counting pass first; forced here with a zero budget."""
    import torch
    from xmap_b200 import engine as E
    case = PT.synth_case(6000, 1200, 120000, 0.1, seed=5)
    a = PT.check_sim_against_restatement(case, "adjust_cosine", 50, 7)
    lay = a["lay"]
    eng = E.SimEngine(lay, PT.to_device_meta(case["meta"]), "adjust_cosine", 50, 7, rec_budget=0)
    assert eng.exact_sizing and eng.rec is None
    tabs = eng.run()
    assert int(eng.rec_ptr[-1]) == int(tabs.row_nkept.sum())          # extents are exact
    pairs = eng.emit_pairs()
    for k in ("i", "j", "sim", "mutu", "n"):
        assert np.array_equal(a["pairs"][k].cpu().numpy(), pairs[k].cpu().numpy()), k
    for t in ("tab_idx", "tab_sim", "tab_len", "row_flags", "row_npairs"):
        assert np.array_equal(getattr(a["tabs"], t).cpu().numpy(), getattr(tabs, t).cpu().numpy()), t
    tabs = eng.run()                                                      # second run reuses the exact extents
    assert np.array_equal(a["tabs"].tab_idx.cpu().numpy(), tabs.tab_idx.cpu().numpy())


def test_segmented_copy_matches_torch():
    """The pack / append kernel of the multi-GPU record exchange against plain indexing."""
    import torch
    from xmap_b200 import multi as MG
    g = torch.Generator().manual_seed(12)
    n_seg = 5000
    seg_len = (torch.rand(n_seg, generator=g) ** 6 * 3000).long()
    seg_len[::7] = 0
    seg_len[123] = 200000                                  # one very long list
    seg_len = seg_len.cuda()
    total = int(seg_len.sum())
    src = torch.randint(-2**62, 2**62, (total + 1000, 2), generator=g, dtype=torch.int64).cuda()
    gaps = torch.randint(0, 5, (n_seg,), generator=g).cuda()
    dst_pos = torch.cumsum(seg_len + gaps, 0) - seg_len - gaps + 3
    src_pos = torch.cumsum(seg_len, 0) - seg_len + 1000
    dst = torch.zeros((int((seg_len + gaps).sum()) + 8, 2), dtype=torch.int64, device="cuda")
    MG._segmented_copy(src, src_pos, dst, dst_pos, seg_len)
    seg = torch.repeat_interleave(torch.arange(n_seg, device="cuda"), seg_len)
    k = torch.arange(total, device="cuda") - (torch.cumsum(seg_len, 0) - seg_len)[seg]
    want = torch.zeros_like(dst)
    want[dst_pos[seg] + k] = src[src_pos[seg] + k]
    assert torch.equal(dst, want)


def test_rerun_is_idempotent():
    """Running the stage twice on the same engine gives the same tables (cursors / flags reset)."""
    case = PT.synth_case(3000, 500, 40000, 0.2, seed=9)
    lay, eng, tabs, pairs = PT.run_gpu_sim(case["user"], case["item"], case["rating"], case["n_users"],
                                           case["n_items"], case["meta"], "adjust_cosine", 50, 10)
    first = {t: getattr(tabs, t).clone() for t in ("tab_idx", "tab_sim", "tab_len", "row_flags", "row_nkept")}
    tabs2 = eng.run()
    for t, v in first.items():
        assert bool((getattr(tabs2, t) == v).all()), t


@pytest.mark.parametrize("k", [1, 50, 64])
def test_topk_sizes(k):
    """k = 50 is BASELINE.json's large-scale configuration; 64 is the library maximum."""
    case = PT.synth_case(5000, 800, 80000, 0.1, seed=17)
    PT.check_sim_against_restatement(case, "cosine", 20, k)


def test_rejects_bad_arguments():
    import torch
    from xmap_b200 import engine as E
    case = PT.synth_case(300, 60, 2000, 0.2, seed=2)
    lay = E.build_layout(case["user"], case["item"], case["rating"], case["n_users"], case["n_items"])
    meta = PT.to_device_meta(case["meta"])
    with pytest.raises(ValueError):
        E.SimEngine(lay, meta, "pearson", 50, 10)
    with pytest.raises(ValueError):
        E.SimEngine(lay, meta, "cosine", 50, 65)
    with pytest.raises(ValueError):
        from xmap_b200.encode import check_ratings_f32
        check_ratings_f32([3.1400000001])


def test_symmetry_and_properties():
    case = PT.synth_case(3000, 500, 40000, 0.2, seed=8)
    lay, eng, tabs, pairs = PT.run_gpu_sim(case["user"], case["item"], case["rating"], case["n_users"],
                                           case["n_items"], case["meta"], "adjust_cosine", 50, 10)
    i, j = pairs["i"].cpu().numpy(), pairs["j"].cpu().numpy()
    sim, mutu, n = (pairs[k].cpu().numpy() for k in ("sim", "mutu", "n"))
    fwd = {(a, b): (s, m, c) for a, b, s, m, c in zip(i, j, sim, mutu, n)}
    for (a, b), v in fwd.items():
        assert fwd[(b, a)] == v            # sim(i,j) == sim(j,i) bitwise
    assert (np.abs(sim) <= 1 + 1e-12).all() and (mutu <= n).all() and (mutu > 0).all()
    frac = pairs["frac"].cpu().numpy()
    assert ((frac > 0) & (frac <= 1)).all()


def test_degenerate_inputs():
    """Empty input; single-rating users (no pairs); identical ratings (all centred values 0)."""
    import torch
    from xmap_b200 import engine as E
    meta = dict(prefix_code=np.zeros(3, np.int32), dom_code=np.zeros(3, np.uint8),
                contains=np.ones(3, np.uint8), has_S=np.ones(3, bool), has_T=np.zeros(3, bool))
    z = np.zeros(0, np.int32)
    lay, eng, tabs, pairs = PT.run_gpu_sim(z, z, np.zeros(0), 2, 3, meta, "adjust_cosine", 50, 5)
    assert len(pairs["i"]) == 0 and int(tabs.tab_len.sum()) == 0
    # users with one rating each: no co-rated pair at all
    lay, eng, tabs, pairs = PT.run_gpu_sim(np.array([0, 1, 2]), np.array([0, 1, 2]), np.array([5., 3., 1.]),
                                           3, 3, meta, "cosine", 50, 5)
    assert len(pairs["i"]) == 0 and tabs.n_pairs_total == 0
    # everybody gives 4 stars: adjusted cosine inner products are exactly 0 -> all filtered
    u = np.repeat(np.arange(4), 3); it = np.tile(np.arange(3), 4)
    lay, eng, tabs, pairs = PT.run_gpu_sim(u, it, np.full(12, 4.0), 4, 3, meta, "adjust_cosine", 50, 5)
    assert tabs.n_pairs_total == 6 and len(pairs["i"]) == 0
    lay, eng, tabs, pairs = PT.run_gpu_sim(u, it, np.full(12, 4.0), 4, 3, meta, "cosine", 50, 5)
    assert len(pairs["i"]) == 6
    torch.cuda.synchronize()
