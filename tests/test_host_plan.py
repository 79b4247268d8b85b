"""CPU: host-side logic -- the X-SIM plan builder (extend.build_plan) evaluated in plain Python
reproduces the oracle's X-SIM, and the C-ABI library exports every declared symbol."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import restate as RS
from tests import parity as PT


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
def test_plan_builder_reproduces_reference_xsim(name):
    import torch
    from xmap_b200 import extend as X
    g = PT.load_golden(name)
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    P = RS.sim_pairs(g["user"].astype(np.int64), g["item"].astype(np.int64), g["rating"], nU, nI,
                     meta["prefix_code"], str(g["method"]), int(g["num_atleast"]))
    k = int(g["k"])
    knn = RS.select_knn(P, nI, k, meta["dom_code"], meta["contains"])
    tabs = PT.tables_from_restatement(P, knn, nI, k)
    plan = X.build_plan(tabs, torch.as_tensor(P["stats"]["count"]), torch.as_tensor(meta["has_S"]),
                        torch.as_tensor(meta["has_T"]))
    s, e, v, combos = PT.eval_plan_numpy(plan)
    PT.compare_xsim(s, e, v, g["xs_start"], g["xs_end"], g["xs_val"], rtol=1e-9)
    Xr = RS.xsim_extend(P, knn, nI, meta["has_S"], meta["has_T"])
    assert combos == Xr["combos"] and plan.n_src == Xr["n_src"] and plan.n_joint == Xr["n_joint"]
    assert int(plan.ub.sum()) == combos            # the per-start bound is exact in total


@pytest.mark.parametrize("name", PT.GOLDEN_CASES)
@pytest.mark.parametrize("fuse", [False, True])
def test_engine_arrays_reproduce_the_plan(name, fuse, native_built):
    """The arrays XsimEngine hands to the kernel -- with and without the fused bridge lists B(t) -- evaluated in
    numpy give the plan's X-SIM: same keys, same path count, values within the reassociation bound."""
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
    xe = X.XsimEngine(plan, 10, fuse=fuse)
    assert (xe.fused_entries > 0) == (fuse and plan.n_joint > 0)     # adj_all_bridge has no joint pair
    if fuse:                                              # every joint-only leg walks exactly one list
        jo = plan.leg_joint_only.bool()
        assert bool((xe.leg_npar[jo] == 1).all())
    G = 1 << xe.gb
    s, e, v, combos = PT.eval_engine_numpy(xe, [(0, G // 3), (G // 3, G)])
    s0, e0, v0, combos0 = PT.eval_plan_numpy(plan)
    assert combos == combos0 == int(plan.ub.sum())
    PT.compare_xsim(s, e, v, s0, e0, v0, rtol=1e-12)
    PT.compare_xsim(s, e, v, g["xs_start"], g["xs_end"], g["xs_val"], rtol=1e-9)


@pytest.mark.parametrize("balance", ["heat", "uniform"])
def test_units_partition_the_tile_axis(balance, native_built):
    """Every start's units cut [0, 2^gb) into consecutive, non-empty tile ranges (equal heat or equal width); the hot /
    cold classes of the hybrid schedule partition the units; the heat estimate adds up to the plan's paths."""
    import torch
    from xmap_b200 import extend as X
    g = PT.load_golden("adj_low_overlap")
    meta = PT.golden_meta(g)
    nU, nI = len(g["uids"]), len(g["iids"])
    P = RS.sim_pairs(g["user"].astype(np.int64), g["item"].astype(np.int64), g["rating"], nU, nI,
                     meta["prefix_code"], str(g["method"]), int(g["num_atleast"]))
    knn = RS.select_knn(P, nI, int(g["k"]), meta["dom_code"], meta["contains"])
    tabs = PT.tables_from_restatement(P, knn, nI, int(g["k"]))
    plan = X.build_plan(tabs, torch.as_tensor(P["stats"]["count"]), torch.as_tensor(meta["has_S"]),
                        torch.as_tensor(meta["has_T"]))
    xe = X.XsimEngine(plan, 10, cells_lg=6, unit_work=200, balance=balance, hot_paths=1500.0)
    G = 1 << xe.gb
    g0, g1, sp = xe.unit_g0.numpy(), xe.unit_g1.numpy(), xe.start_unit_ptr.numpy()
    assert (np.diff(sp) > 1).sum() > 50                                  # many starts are cut into several units
    for x in range(len(sp) - 1):
        a, b = sp[x], sp[x + 1]
        assert g0[a] == 0 and g1[b - 1] == G and (g1[a:b] > g0[a:b]).all() and (g0[a + 1:b] == g1[a:b - 1]).all()
    npass = xe.unit_npass.numpy()
    assert (npass >= 1).all() and (npass <= g1 - g0).all()
    hot, cold = xe.hot_order.numpy(), xe.cold_order.numpy()
    assert len(hot) > 0 and len(cold) > 0 and np.array_equal(np.sort(np.concatenate([hot, cold])), np.arange(xe.n_units))
    est = xe.unit_est_paths.numpy()
    assert (est[hot] > 1500.0).all() and (est[cold] <= 1500.0).all()
    per_start = np.add.reduceat(est, sp[:-1])
    np.testing.assert_allclose(per_start, plan.ub.numpy().astype(np.float64), rtol=1e-9)


def test_library_exports_every_declared_symbol(native_built):
    from xmap_b200 import _native
    hdr = open(os.path.join(PT.ROOT, "include", "xmap_b200.h")).read()
    declared = set(re.findall(r"\b(xmap_[a-z_0-9]+)\s*\(", hdr))
    assert declared == set(_native.EXPORTED_SYMBOLS), declared ^ set(_native.EXPORTED_SYMBOLS)
    L = ctypes.CDLL(_native.LIB_PATH)
    for s in declared:
        assert hasattr(L, s), s
    L.xmap_abi_version.restype = ctypes.c_int
    assert L.xmap_abi_version() == _native.ABI_VERSION


def test_no_cpu_fallback_without_gpu():
    """The product path must fail loudly, not fall back, when CUDA is unavailable."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from xmap_b200 import engine as E
    with pytest.raises(Exception):
        E.build_layout(np.zeros(1, np.int32), np.zeros(1, np.int32), np.ones(1), 1, 1)


def test_engine_host_helpers():
    """Device-agnostic helpers of the engine: popularity rank, threads per table and the hand-over pool of
    record buffers."""
    import torch
    from xmap_b200 import engine as E
    cnt = torch.tensor([3., 1., 3., 7., 1.], dtype=torch.float64)
    assert E.popularity_order(cnt).tolist() == [2, 0, 3, 4, 1]          # ascending count, ties by index
    assert [E._threads_for_cells(c) for c in (32, 256, 512, 1024, 1536, 4096, 12288)] == [32, 32, 64, 128, 192, 512, 512]
    E._REC_POOL.pop("cpu", None)
    a = torch.empty(E._rec_words(100), dtype=torch.int64); b = torch.empty(E._rec_words(1000), dtype=torch.int64)
    E._REC_POOL["cpu"] = [b, a]
    assert E._rec_buffer(50, "cpu") is a and E._rec_buffer(500, "cpu") is b and E._REC_POOL["cpu"] == []
    E._REC_POOL["cpu"] = [a]
    t = E._rec_buffer(5000, "cpu")
    assert t.numel() == E._rec_words(5000) and E._REC_POOL["cpu"] == []     # too small: dropped, a fresh one allocated
    rec, rec_n = E._rec_views(t, 5000)                                       # [n, 2] records + their int32 counts, disjoint
    assert tuple(rec.shape) == (5000, 2) and tuple(rec_n.shape) == (5000,) and rec_n.dtype == torch.int32
    rec.fill_(-1); rec_n.fill_(7)
    assert int((rec != -1).sum()) == 0 and int((rec_n != 7).sum()) == 0


def test_predict_rejects_out_of_range_test_pairs_on_the_host():
    """recsim.predict checks test_user against [0, n_users) and test_item against the neighbour tables before it
    launches anything (the kernel indexes the profile and the tables without a bound check).  Every call here
    raises, so the CPU tensors never reach the kernel."""
    import torch
    from xmap_b200 import recsim
    nI, K = 5, 3
    R = recsim.RecSim(torch.zeros(1, dtype=torch.int32), torch.zeros(1, dtype=torch.int32), torch.ones(1, dtype=torch.int64),
                      torch.zeros(1, dtype=torch.float64), torch.zeros(1, dtype=torch.float64),
                      torch.zeros((nI, 3), dtype=torch.float64), 0)
    nb = recsim.Neighbors(torch.full((nI, K), -1, dtype=torch.int32), torch.zeros((nI, K), dtype=torch.float64),
                          torch.zeros(nI, dtype=torch.int32))
    prof = ([0, 1], [2, 3], [4.0, 3.5], [10, 20], 2, R, nb)
    for tu, ti in (([0, 2], [0, 0]), ([-1], [0]), ([0], [nI]), ([1, 0], [0, -1]), ([2 ** 32], [0]), ([0], [0, 1])):
        with pytest.raises(ValueError):
            recsim.predict(*prof, tu, ti)


def test_exponent_base():
    """e_base of the fixed-point scale: max E - 127 over the items with a non-zero norm (2^(E-1) <= den < 2^E),
    from the norm the method divides by; up to 16 octaves below the field are clamped, more raise."""
    import torch
    from xmap_b200 import engine as E

    def stats(norm2, adj):                                        # item_stats columns: avg, norm2, adj_norm2, count
        n = len(norm2)
        return torch.tensor([[1.0] * n, norm2, adj, [2.0] * n], dtype=torch.float64).T.contiguous()

    st = stats([5.0, 0.75, 0.0], [0.0, 4.0, 0.0])
    assert E.exponent_base("cosine", st) == 3 - 127                # frexp(5) = 0.625 * 2^3
    assert E.exponent_base("adjust_cosine", st) == 3 - 127          # 4 = 0.5 * 2^3; zero norms are ignored
    assert E.exponent_base("adjust_cosine", stats([5.0, 1.0], [0.0, 0.0])) == 0      # every norm zero
    assert E.exponent_base("cosine", stats([1.0, 0.5], [2.0 ** 40, 1.0])) == 1 - 127
    assert E.exponent_base("adjust_cosine", stats([1.0, 0.5], [2.0 ** 40, 1.0])) == 41 - 127
    assert E.exponent_base("cosine", stats([2.0 ** 100, 2.0 ** -27], [1.0, 1.0])) == 101 - 127    # spread 127: fits
    assert E.exponent_base("cosine", stats([2.0 ** 100, 2.0 ** -43], [1.0, 1.0])) == 101 - 127    # clamped by 16
    with pytest.raises(ValueError):
        E.exponent_base("cosine", stats([2.0 ** 100, 2.0 ** -44], [1.0, 1.0]))
    with pytest.raises(ValueError):
        E.exponent_base("adjust_cosine", stats([1.0, 1.0], [2.0 ** -60, 2.0 ** 100]))
