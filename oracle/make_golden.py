"""Freeze outputs of the UNMODIFIED reference into tests/golden/*.npz.

TEST INFRASTRUCTURE ONLY.  Run in the build container, where /root/reference
exists:   python -m oracle.make_golden
The GPU box has no /root/reference, so GPU-side parity tests read these files.

Every array below comes from executing the reference's own classes through
oracle/harness.py (not from oracle/restate.py), with ids replaced by their
canonical index (rank of the id string in sorted order).
"""
import calendar
import importlib.util
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import harness as H          # noqa: E402
from oracle import encode as EN          # noqa: E402

_spec = importlib.util.spec_from_file_location(
    "_xmap_synth", os.path.join(ROOT, "x-map_b200", "synth.py"))
synth = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(synth)

CASES = {
    # name: (users, items/domain, draws, overlap, seed, method, num_atleast, k, half_ratings)
    "adj_low_overlap": (500, 180, 8000, 0.04, 5, "adjust_cosine", 50, 4, False),
    "cos_half_ratings": (360, 110, 4400, 0.06, 7, "cosine", 50, 3, True),
    "adj_all_bridge": (200, 70, 3600, 0.5, 9, "adjust_cosine", 5, 10, False),
}
# mid-size case: similarity + classification only (the reference's extender is infeasible at this size,
# SURVEY.md App. B.4).  Rows with up to ~2e4 co-rating products and lists of ~1e3 neighbours: the CTA launch
# shapes of the accumulate kernels and the histogram path of the selection meet the real reference here.
SIM_ONLY_CASES = {
    "adj_mid": (5000, 600, 120000, 0.05, 13, "adjust_cosine", 50, 10, False),
}
CASES_ALL = dict(CASES, **SIM_ONLY_CASES)


def _ragged(lists):
    ptr = np.zeros(len(lists) + 1, dtype=np.int32)
    for k, l in enumerate(lists):
        ptr[k + 1] = ptr[k] + len(l)
    flat = np.array([x for l in lists for x in l], dtype=np.int32)
    return ptr, flat


def build_case(name):
    nu, ni, nd, ov, seed, method, na, k, half = CASES_ALL[name]
    sim_only = name in SIM_ONLY_CASES
    sr = synth.make_ratings(nu, ni, nd, overlap=ov, seed=seed)
    recs = synth.to_train_records(sr)
    if half:   # half-star ratings 0.5 .. 5.0 to exercise non-integer values
        recs = [(u, [(i, r - 0.5 * ((hash_det(u, i)) & 1), t) for i, r, t in lst])
                for u, lst in recs]
    user, item, rating, ts, meta = EN.encode_train(recs)
    iids, uids = meta["iids"], meta["uids"]
    ipos = {s: n for n, s in enumerate(iids)}
    upos = {s: n for n, s in enumerate(uids)}
    out = dict(uids=np.array(uids), iids=np.array(iids), user=user.astype(np.int32),
               item=item.astype(np.int32), rating=rating, ts=ts,
               method=np.array(method), num_atleast=np.int64(na), k=np.int64(k))

    tool, trainRDD, simRDD, dt_sim = H.run_sim(recs, method, na)
    ref = simRDD.collect()
    idt = np.int16 if (sim_only and len(iids) < 32000) else np.int32
    out.update(sim_i=np.array([ipos[a] for (a, b), _ in ref], dtype=idt),
               sim_j=np.array([ipos[b] for (a, b), _ in ref], dtype=idt),
               sim_val=np.array([float(v[0]) for _, v in ref]),
               sim_mutu=np.array([int(v[1]) for _, v in ref], dtype=idt),
               sim_frac=np.array([float(v[2]) for _, v in ref]),
               sim_label=np.array([v[3] for _, v in ref], dtype=np.int8))
    if sim_only:
        # keep the file small: frac is a function of (mutu, counts, n) and is checked bit-exactly against the
        # restatement, which test_oracle pins on this case; store its float32 image as a cross-check only
        out["sim_frac"] = out["sim_frac"].astype(np.float32)
    # item / user info straight from the reference (baselinerSim.py:17-82)
    R = H.load_reference()
    ui = tool.get_universal_user_info(trainRDD).collectAsMap()
    ii = tool.get_universal_item_info(trainRDD, R["sc"].broadcast(ui)).collectAsMap()
    out["user_avg"] = np.array([ui[u][0] for u in uids])
    out["item_info"] = np.array([ii[i] for i in iids])

    bb, classified = H.run_classify(tool, simRDD, k)
    bbm = np.zeros(len(iids), dtype=bool)
    bbm[[ipos[b] for b in bb]] = True
    out["bb"] = bbm
    lists = {n: [[] for _ in iids] for n in ("BB_BB", "BB_NB", "NB_BB", "NB_NN")}
    valid_nb = np.zeros(len(iids), dtype=bool)
    for iid, B, N in classified:
        it = ipos[iid]
        if B is not None:
            lists["BB_BB"][it] = [ipos[x[0]] for x in B[0]]
            lists["BB_NB"][it] = [ipos[x[0]] for x in B[1]]
        else:
            valid_nb[it] = True
            lists["NB_BB"][it] = [ipos[x[0]] for x in N[0]]
            lists["NB_NN"][it] = [ipos[x[0]] for x in N[1]]
    out["valid_nb"] = valid_nb
    for n, l in lists.items():
        out[n + "_ptr"], out[n + "_nbr"] = _ragged(l)

    if sim_only:
        out["ref_seconds"] = np.array([dt_sim, 0.0, 0.0])
        return compact_sim_only(out)
    xs, dt_ext = H.run_extend(tool, simRDD, k)
    xrows = xs.collect()
    out.update(xs_start=np.array([ipos[t] for t, lst in xrows for _ in lst], dtype=np.int32),
               xs_end=np.array([ipos[e] for t, lst in xrows for e, _ in lst], dtype=np.int32),
               xs_val=np.array([float(v) for t, lst in xrows for _, v in lst]))

    def enc_alter(alter):
        a = sorted((upos[u], ipos[i], float(r), calendar.timegm(t.timetuple()))
                   for u, i, r, t in alter)
        return (np.array([x[0] for x in a], dtype=np.int32), np.array([x[1] for x in a], dtype=np.int32),
                np.array([x[2] for x in a]), np.array([x[3] for x in a], dtype=np.int64))

    if xrows:
        pairs, _, alter, dt_gen = H.run_generate(trainRDD, xs, True, method)
        out["priv_rows"] = np.array([ipos[t] for t, _ in pairs], dtype=np.int32)
        out["priv_chosen"] = np.array([ipos[s] for _, s in pairs], dtype=np.int32)
        (out["priv_ae_user"], out["priv_ae_item"], out["priv_ae_rating"],
         out["priv_ae_ts"]) = enc_alter(alter)
        # non-private: rows with one candidate make the reference raise
        # (generator.py:110, randint(0, 0)); they are left out of ITS input.
        seed_np = 11
        xs2 = R["sc"].parallelize([r for r in xrows if len(r[1]) >= 2])
        pairsN, _, alterN, _ = H.run_generate(trainRDD, xs2, False, method, np_seed=seed_np)
        out["nonpriv_rows"] = np.array([ipos[t] for t, _ in pairsN], dtype=np.int32)
        out["nonpriv_chosen"] = np.array([ipos[s] for _, s in pairsN], dtype=np.int32)
        # replay the reference's np.random stream as uniforms u with floor(u*(m-1)) == its draw
        np.random.seed(seed_np)
        us = []
        for _, lst in xs2.collect():
            m = min(len(lst), 4)
            us.append((np.random.randint(0, m - 1) + 0.5) / (m - 1))
        out["nonpriv_uniforms"] = np.array(us)
        (out["nonpriv_ae_user"], out["nonpriv_ae_item"], out["nonpriv_ae_rating"],
         out["nonpriv_ae_ts"]) = enc_alter(alterN)
    else:
        dt_gen = 0.0
    out["ref_seconds"] = np.array([dt_sim, dt_ext, dt_gen])
    return out


MID_SAMPLE_RATE = 0.1      # share of the remaining pairs whose similarity a sim-only golden keeps


def compact_sim_only(out, seed=13):
    """Shrinks a sim-only case to well under 1 MB.  The reference's similarity records are symmetric (checked here),
    so the keys, mutualities and labels of the pairs i < j are stored whole and the tests mirror them.  Similarity and
    frac are kept for a fixed sample of those pairs: every pair in a neighbour list (the near-tie checks look their
    similarity up), every pair with |sim| < 1e-9 (the rounding residues of cancelling inner products) and a seeded
    MID_SAMPLE_RATE of the rest.  The rating times are dropped: the similarity stage does not read them."""
    n_items = len(out["iids"])
    si, sj = out["sim_i"].astype(np.int64), out["sim_j"].astype(np.int64)
    key, mirror = si * n_items + sj, sj * n_items + si
    o = np.argsort(mirror)
    assert np.array_equal(key, mirror[o]), "similarity records are not symmetric"
    for name in ("sim_val", "sim_mutu", "sim_frac", "sim_label"):
        assert np.array_equal(out[name], out[name][o]), name
    up = si < sj
    listed = np.zeros(n_items * n_items, dtype=bool)
    for name in ("BB_BB", "BB_NB", "NB_BB", "NB_NN"):
        ptr, nbr = out[name + "_ptr"], out[name + "_nbr"].astype(np.int64)
        rows = np.repeat(np.arange(n_items), np.diff(ptr))
        listed[rows * n_items + nbr] = listed[nbr * n_items + rows] = True
    val = out["sim_val"][up]
    keep = listed[key[up]] | (np.abs(val) < 1e-9) | (np.random.default_rng(seed).random(len(val)) < MID_SAMPLE_RATE)
    sample = np.flatnonzero(keep).astype(np.int32)
    small = {k: v for k, v in out.items() if k != "ts" and not k.startswith("sim_")}
    return dict(small, pair_ptr=np.searchsorted(si[up], np.arange(n_items + 1)).astype(np.int32),
                pair_j=out["sim_j"][up], pair_mutu=out["sim_mutu"][up], pair_label=out["sim_label"][up],
                sample=sample, sample_sim=val[sample], sample_frac=out["sim_frac"][up][sample])


def hash_det(u, i):
    """Deterministic (process-independent) parity bit for the half-rating case."""
    return sum(ord(c) for c in u) + sum(ord(c) for c in i)


def main():
    gdir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(gdir, exist_ok=True)
    for name in (sys.argv[1:] or list(CASES_ALL)):
        t0 = time.time()
        out = build_case(name)
        path = os.path.join(gdir, name + ".npz")
        np.savez_compressed(path, **out)
        print("%-18s pairs=%d bb=%d xsim=%d  ref s=%s  (%.1fs) -> %s (%d KB)" % (
            name, len(out["sim_i"]) if "sim_i" in out else 2 * len(out["pair_j"]), int(out["bb"].sum()), len(out.get("xs_val", ())),
            np.round(out["ref_seconds"], 2), time.time() - t0, path,
            os.path.getsize(path) // 1024))


if __name__ == "__main__":
    main()
