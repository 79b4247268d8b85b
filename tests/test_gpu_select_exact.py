"""GPU: select_warp_kernel and select_cta_kernel (x-map_b200/csrc/sim.cu) alone, against the exact selection of
tests/select_exact.py, bit for bit, on the designed record lists of select_exact.designed_cases.

The lists are laid out as the accumulate stage leaves them (int64 records {sim bits, j | mutu << 32}, int32 n,
rec_ptr / rec_cnt) and xmap_sim_select is launched as SimEngine.select launches it: the warp kernel over the rows,
then the CTA kernel over the rows with more than XMAP_SELECT_LONG records.  Only what selection reads is set; every
other pointer of the argument block is NULL.  At every k of select_exact.KS, once with rows = NULL for both launches
and once with a shuffled half of the rows: tab_len, tab_idx, tab_sim (as bits), tab_mutu and tab_n must equal the
reference, entries past tab_len and rows not passed must still hold the sentinels, and the three stored orders of
each list (as built, reversed, permuted) must give identical tables.  The classifier of select_exact names the path
of every (row, list, k); each path must run at least select_exact.MIN_PER_PATH times at every k."""
import numpy as np
import pytest

from tests import select_exact as SE

pytestmark = pytest.mark.gpu

SENTINEL = dict(idx=-7, sim_bits=0x7FF8_0000_DEAD_BEEF, mutu=-5, n=-9, len=-3)
NAMES = ("tab_len", "tab_idx", "tab_sim", "tab_mutu", "tab_n")


@pytest.fixture(scope="module")
def designed(native_built):
    import torch
    c = SE.designed_cases()
    rank = SE.Ranked(c["i"], c["j"], c["sim"], c["mutu"], c["n"], c["bb"], c["dom_code"], c["contains"], c["n_rows"])
    R = c["n_rows"]
    cnt = np.bincount(c["i"], minlength=R)
    dev = torch.device("cuda")
    rec = np.stack([c["sim"].view(np.int64), c["j"] | (c["mutu"] << 32)], axis=1)
    D = dict(rec=torch.as_tensor(rec, device=dev), rec_n=torch.as_tensor(c["n"].astype(np.int32), device=dev),
             rec_cnt=torch.as_tensor(cnt.astype(np.int32), device=dev),
             rec_ptr=torch.as_tensor(np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64), device=dev),
             bb=torch.as_tensor(c["bb"], device=dev), dom_code=torch.as_tensor(c["dom_code"], device=dev),
             contains=torch.as_tensor(c["contains"], device=dev))
    return dict(c=c, rank=rank, R=R, cnt=cnt, D=D, dev=dev)


def run_select(d, k, rows):
    """Both launches of SimEngine.select into sentinel-filled tables; rows = None passes NULL to both kernels."""
    import torch
    from xmap_b200 import _native as N
    R, D, dev = d["R"], d["D"], d["dev"]
    T = dict(tab_len=torch.full((R, 2), SENTINEL["len"], dtype=torch.int32, device=dev),
             tab_idx=torch.full((R, 2, k), SENTINEL["idx"], dtype=torch.int32, device=dev),
             tab_sim=torch.full((R, 2, k), SENTINEL["sim_bits"], dtype=torch.int64, device=dev).view(torch.float64),
             tab_mutu=torch.full((R, 2, k), SENTINEL["mutu"], dtype=torch.int32, device=dev),
             tab_n=torch.full((R, 2, k), SENTINEL["n"], dtype=torch.int32, device=dev))
    a = N.SimArgs()
    a.n_items, a.method, a.num_atleast, a.k = SE.N_ITEMS, N.METHODS["adjust_cosine"], 1, k
    a.dom_code, a.contains, a.bb = N.ptr(D["dom_code"]), N.ptr(D["contains"]), N.ptr(D["bb"])
    a.rec_ptr, a.rec_cnt, a.rec, a.rec_n = N.ptr(D["rec_ptr"]), N.ptr(D["rec_cnt"]), N.ptr(D["rec"]), N.ptr(D["rec_n"])
    a.tab_idx, a.tab_sim, a.tab_mutu = N.ptr(T["tab_idx"]), N.ptr(T["tab_sim"]), N.ptr(T["tab_mutu"])
    a.tab_n, a.tab_len = N.ptr(T["tab_n"]), N.ptr(T["tab_len"])
    L = N.lib()
    st = torch.cuda.current_stream().cuda_stream
    if rows is None:
        N.check(L.xmap_sim_select(a, None, R, 0, st), "xmap_sim_select")
        N.check(L.xmap_sim_select(a, None, R, 1, st), "xmap_sim_select(long)")
    else:
        rt = torch.as_tensor(rows.astype(np.int32), device=dev)
        lt = torch.as_tensor(rows[d["cnt"][rows] > SE.SELECT_LONG].astype(np.int32), device=dev)
        N.check(L.xmap_sim_select(a, N.ptr(rt), len(rows), 0, st), "xmap_sim_select")
        if lt.numel():
            N.check(L.xmap_sim_select(a, N.ptr(lt), lt.numel(), 1, st), "xmap_sim_select(long)")
    torch.cuda.synchronize()
    return {name: t.cpu().numpy() for name, t in T.items()}


def expected(d, k, rows):
    ref = d["rank"].tables(k, SENTINEL)
    if rows is not None:
        out = np.ones(d["R"], bool)
        out[rows] = False
        ref["tab_len"][out] = SENTINEL["len"]
        for name, v in (("tab_idx", "idx"), ("tab_mutu", "mutu"), ("tab_n", "n")):
            ref[name][out] = SENTINEL[v]
        ref["tab_sim"].view(np.int64)[out] = SENTINEL["sim_bits"]
    return ref


def differing_rows(ref, got):
    bad = np.zeros(len(ref["tab_len"]), bool)
    for name in NAMES:
        a, b = ref[name], got[name]
        if name == "tab_sim":
            a, b = a.view(np.int64), b.view(np.int64)
        bad |= (a != b).reshape(len(bad), -1).any(axis=1)
    return np.nonzero(bad)[0]


def test_select_kernels_equal_exact_selection(designed):
    d = designed
    c, R = d["c"], d["R"]
    rng = np.random.default_rng(5)
    totals = dict.fromkeys(SE.PATHS, 0)
    for k in SE.KS:
        labels, flushes = SE.classify(c["i"], c["j"], c["sim"], c["bb"], c["dom_code"], c["contains"], k, R)
        counts = SE.path_counts(labels)
        for p in SE.PATHS:
            totals[p] += counts[p]
        for mode, rows in (("NULL", None), ("subset", rng.permutation(R)[: R // 2])):
            got = run_select(d, k, rows)
            bad = differing_rows(expected(d, k, rows), got)
            if len(bad):
                r = int(bad[0])
                pytest.fail("k %d rows %s: %d rows differ from the exact selection; row %d %s (paths %s / %s): "
                            "len %s, idx %s" % (k, mode, len(bad), r, c["names"][r], SE.PATHS[labels[r, 0]],
                                                SE.PATHS[labels[r, 1]], got["tab_len"][r].tolist(),
                                                got["tab_idx"][r].tolist()))
            if rows is None:      # as built, reversed, permuted: identical tables
                for name in NAMES:
                    t = got[name].view(np.int64) if name == "tab_sim" else got[name]
                    assert np.array_equal(t[0::3], t[1::3]) and np.array_equal(t[0::3], t[2::3]), name
        print("k %2d: %s; CTA tournaments per row %d..%d" % (k, counts, min(flushes.values()), max(flushes.values())))
        for p in SE.PATHS[1:]:
            assert counts[p] >= SE.MIN_PER_PATH, "k %d: path %s ran %d times" % (k, p, counts[p])
        assert max(flushes.values()) >= 40
    print("(row, list, k) cases per path over k in %s: %s" % (SE.KS, totals))
