"""Downstream recommender stages on the AlterEgo profile, with the reference's class and method names
(xmap/core/recommenderSim.py:9-195, recommenderPrivacy.py:9-189, recommenderPrediction.py:6-139).

Offered: item-based `cosine_item` similarity with local sensitivity, NON-private neighbour selection, item-based
prediction with and without temporal decay, MAE.  `adjust_cosine_item` is accepted and, as in the reference (whose
dispatch tests the substring "cosine_item" first, recommenderSim.py:188), runs the same cosine_item path.  Not offered
(ValueError): the user-based variants (absent from the reference's own source tree, SURVEY.md 2.1).  The private neighbour
selection (recommenderPrivacy.py:70-139, 152-171) is offered as it behaves under Python 3, with injectable uniforms.  The work happens in csrc/recsim.cu; these classes
encode the flat (uid, iid, rating, time) records once and keep the device state on the objects they return.
"""
import calendar
from datetime import datetime

import numpy as np
import torch

from .. import recsim as RS
from ..rdd import Broadcast, LazyRDD, LocalRDD, records_of


def _ts(t):
    return calendar.timegm(t.timetuple()) if isinstance(t, datetime) else int(t)


class ProfileState(object):
    """The AlterEgo profile encoded for the device (list order kept: it fixes arrival order and tie-breaks)."""

    def __init__(self, records):
        recs = records_of(records)
        self.records = recs
        self.uids, user = np.unique(np.array([str(r[0]) for r in recs]), return_inverse=True)
        self.iids, item = np.unique(np.array([str(r[1]) for r in recs]), return_inverse=True)
        self.user, self.item = user.astype(np.int64), item.astype(np.int32)
        self.rating = np.array([float(r[2]) for r in recs], dtype=np.float64)
        self.ts = np.array([_ts(r[3]) for r in recs], dtype=np.int64)
        self.upos = {s: n for n, s in enumerate(self.uids)}
        self.ipos = {s: n for n, s in enumerate(self.iids)}
        self.num_atleast = None  # set by RecommenderSim.calculate_sim
        self.knn = None          # recsim.ItemKnn: item info and the neighbour tables
        self.nb = None           # recsim.Neighbors


class HandleDict(dict):
    """A plain dict for callers, plus the device state for the next pipeline stage."""
    handle = None


class RecommenderSim(object):
    def __init__(self, method, num_atleast):
        self.method = method
        self.num_atleast = num_atleast

    def build_sthbased_profile(self, rdd, profile):
        """recommenderSim.py:15-27."""
        pos = 0 if "user" in profile else 1
        rows = {}
        for l in records_of(rdd):
            rows.setdefault(l[pos], []).append((l[1 - pos], l[2], l[3]))
        out = LocalRDD(rows.items())
        out.handle = getattr(rdd, "handle", None)
        return out

    def calculate_sim(self, state):
        """((iid1, iid2), [sim, local sensitivity])* -- recommenderSim.py:186-195.  The reference dispatches on
        `"cosine_item" in self.method` FIRST (:188), and "adjust_cosine_item" contains that substring, so both method
        names run cosine_sim there (adjusted_cosine_sim, :135-184, is unreachable); both are accepted here and mean
        the same.  Anything else (the user-based names) returns None in the reference and raises here."""
        if "cosine_item" not in self.method:
            raise ValueError("only the item-based similarities are offered (got %r)" % (self.method,))
        state.num_atleast = self.num_atleast

        def build():
            # only when the records are collected, one block of item rows at a time; the neighbour selection
            # (recommender_privacy_pipeline) runs from the profile and never needs them
            for s in RS.pair_passes(state.user, state.item, state.rating, len(state.iids), self.num_atleast):
                i, j = s.i.cpu().numpy(), s.j.cpu().numpy()
                sim, ls = s.sim.cpu().numpy(), s.ls.cpu().numpy()
                for q in range(len(i)):
                    yield (str(state.iids[i[q]]), str(state.iids[j[q]])), [sim[q], ls[q]]
        return LazyRDD(build, handle=state)


class RecommenderPrivacy(object):
    def __init__(self, mapping_range, privacy_epsilon, rpo, uniforms=None, seed=None):
        """uniforms: optional (u_pick, u_noise), one injected uniform per item that has neighbours, in item order (the
        reference's np.random draws replayed); seed: Philox seed of the private branch (None: fresh entropy per object)."""
        self.mapping_range = mapping_range
        self.privacy_epsilon = privacy_epsilon / 2          # recommenderPrivacy.py:18
        self.rpo = rpo
        self.uniforms = uniforms
        if seed is None:
            import secrets
            seed = secrets.randbits(64)
        self.seed, self._calls = int(seed), 0

    def _neighbour_rdd(self, state):
        def build():
            ln, idx, sim = state.nb.len.cpu().numpy(), state.nb.idx.cpu().numpy(), state.nb.sim.cpu().numpy()
            for it in np.flatnonzero(ln):
                yield str(state.iids[it]), [(str(state.iids[idx[it, r]]), sim[it, r]) for r in range(ln[it])]
        out = LazyRDD(build, handle=state)
        out.collectAsMap = lambda: _handle_dict(out.collect(), state)
        return out

    def nonprivate_neighbor_selection(self, rdd):
        """(iid, [(neighbour, [sim, ls])*]) -- recommenderPrivacy.py:141-150; here the sensitivity is already dropped
        (nonnoise_perturbation, :180-189), which is all the non-private pipeline keeps."""
        state = rdd.handle
        state.knn = RS.item_knn(state.user, state.item, state.rating, len(state.iids), state.num_atleast,
                                int(self.mapping_range))
        state.nb = state.knn.nb
        return self._neighbour_rdd(state)

    def nonnoise_perturbation(self, rdd):
        return rdd

    def private_neighbor_selection(self, rdd):
        """recommenderPrivacy.py:70-139 as it behaves under Python 3 -- one neighbour per item, drawn by the exponential
        mechanism over all its neighbours (`np.count_nonzero(map(...))`, :81, counts the map object) -- fused with
        noise_perturbation (:152-171): the rows already carry sim + Laplace(|local sensitivity| / eps)."""
        state = rdd.handle
        up, un = self.uniforms if self.uniforms is not None else (None, None)
        seed = (self.seed + 0x9E3779B97F4A7C15 * self._calls) & (2 ** 64 - 1)
        self._calls += 1
        state.knn = RS.item_knn(state.user, state.item, state.rating, len(state.iids), state.num_atleast,
                                int(self.mapping_range), private=dict(privacy_epsilon=2 * self.privacy_epsilon, rpo=self.rpo,
                                                                      u_pick=up, u_noise=un, seed=seed))
        state.nb = state.knn.nb
        return self._neighbour_rdd(state)

    def noise_perturbation(self, rdd):
        return rdd


def _handle_dict(pairs, state):
    d = HandleDict(pairs)
    d.handle = state
    return d


class RecommenderPrediction(object):
    def __init__(self, alpha, method):
        self.alpha = alpha
        self.method = method

    def item_based_recommendation(self, test_dataRDD, item_based_dict_bd, itembased_sim_pair_dict_bd, item_info_bd):
        """(uid, [(iid, real rating, prediction, prediction with decay)*])* -- recommenderPrediction.py:105-114."""
        state = getattr(getattr(itembased_sim_pair_dict_bd, "value", itembased_sim_pair_dict_bd), "handle", None)
        if state is None or state.nb is None or state.knn is None:
            raise TypeError("expected the neighbour dictionary returned by recommender_privacy_pipeline "
                            "(it carries the device-resident tables)")
        test = records_of(test_dataRDD)
        tu, ti, tr, where = [], [], [], []
        for a, (uid, lst) in enumerate(test):
            for b, (iid, r, _t) in enumerate(lst):
                if str(iid) in state.ipos and str(uid) in state.upos:
                    tu.append(state.upos[str(uid)]); ti.append(state.ipos[str(iid)]); tr.append(float(r)); where.append((a, b))
        p0, p1, _, _ = RS.predict(state.user, state.item, state.rating, state.ts, len(state.uids), state.knn, state.nb,
                                  np.array(tu, dtype=np.int32), np.array(ti, dtype=np.int32), None, self.alpha)
        p0, p1 = p0.cpu().numpy(), p1.cpu().numpy()
        out = [(uid, [() for _ in lst]) for uid, lst in test]
        for q, (a, b) in enumerate(where):
            if p0[q] >= 0:
                iid, r, _t = test[a][1][b]
                out[a][1][b] = (iid, r, float(p0[q]), float(p1[q]))
        return LocalRDD(out)

    def calculate_mae(self, rdd):
        """'mae without decay; mae with decay' -- recommenderPrediction.py:116-139."""
        a = b = n = 0.0
        for _uid, pairs in records_of(rdd):
            for p in pairs:
                if p != ():
                    a += abs(p[1] - p[2]); b += abs(p[1] - p[3]); n += 1
        return str(1.0 * a / n) + "; " + str(b / n)


# ---- pipeline glue (assist.py:153-207) --------------------------------------------------------------------------
def recommender_calculate_sim_pipeline(sc, cross_sim_tool, alterEgo_profile):
    """assist.py:153-175: (user profile, item profile, their dicts, user info, item info, similarity RDD)."""
    state = ProfileState(alterEgo_profile)
    flat = LocalRDD(state.records)
    user_based = cross_sim_tool.build_sthbased_profile(flat, "user")
    item_based = cross_sim_tool.build_sthbased_profile(flat, "item")
    sims = cross_sim_tool.calculate_sim(state)
    info = RS.item_info(state.item, state.rating, len(state.iids)).cpu().numpy()
    item_info = {str(s): (info[n, 0], info[n, 1], int(info[n, 2])) for n, s in enumerate(state.iids)}
    user_info = {}
    for uid, lst in user_based.collect():
        r = np.array([x[1] for x in lst], dtype=np.float64)
        user_info[uid] = (1.0 * np.average(r), np.sqrt(np.sum(r ** 2)), len(r))
    return (user_based, item_based, Broadcast(user_based.collectAsMap()), Broadcast(item_based.collectAsMap()),
            Broadcast(user_info), Broadcast(item_info), sims)


def recommender_privacy_pipeline(policy_tool, alterEgo_sim, is_private):
    """assist.py:178-192."""
    if is_private:
        return policy_tool.noise_perturbation(policy_tool.private_neighbor_selection(alterEgo_sim))
    return policy_tool.nonnoise_perturbation(policy_tool.nonprivate_neighbor_selection(alterEgo_sim))


def recommender_prediction_pipeline(recommender_tool, cross_sim_tool, testRDD, simpair_dict_bd,
                                    user_based_dict_bd, item_based_dict_bd, user_info_bd, item_info_bd):
    """assist.py:195-207 (item-based methods)."""
    if "user" in cross_sim_tool.method:
        raise ValueError("user-based recommendation is not offered")
    predicted = recommender_tool.item_based_recommendation(testRDD, item_based_dict_bd, simpair_dict_bd, item_info_bd)
    return recommender_tool.calculate_mae(predicted)
