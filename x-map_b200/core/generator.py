"""Generator facade -- reference class xmap/core/generator.py:6-157.

`private_mode` selects what "private" means: 'argmax' reproduces the reference as it
behaves under Python 3 (weighted_pick returns index 0 for a `map` object,
generator.py:66-67), 'exp_mech' is the exponential mechanism the code intends
(generator.py:42-75, tech report Thm 1).  Draws come from Philox(seed, row) unless
`uniforms` (one per X-SIM row, ascending target index) are injected."""
import os

import numpy as np
import torch

from .. import generate as G
from ..extend import XsimResult
from ..rdd import LocalRDD, records_of
from ..session import session_of


class Generator(object):
    def __init__(self, mapping_range, privacy_epsilon, sim_method, rpo,
                 private_mode="argmax", seed=None, uniforms=None):
        self.mapping_range = mapping_range
        self.privacy_epsilon = privacy_epsilon
        self.sim_method = sim_method
        self.rpo = rpo
        self.private_mode = private_mode
        # seed=None (default): fresh entropy per tool, and every mapping call advances the Philox key, so
        # repeated releases are independent like the reference's unseeded np.random (generator.py:60-70);
        # an explicit seed keeps the draws reproducible (tests)
        self._fresh = seed is None
        self.seed = int.from_bytes(os.urandom(8), "little") if seed is None else seed
        self._calls = 0
        self.uniforms = uniforms
        self.single_candidate_rows = 0     # rows where the reference would raise (generator.py:110)

    def global_sentivity(self):
        return G.global_sensitivity(self.sim_method)

    # ---- mapping -----------------------------------------------------------
    def _xres(self, rdd, session):
        h = getattr(rdd, "handle", None)
        if h is not None and hasattr(h, "result"):
            return h.result
        return _encode_xsim_rows(records_of(rdd), session)

    def _map(self, rdd, session, mode, topn=G.NONPRIVATE_TOPN):
        xres = self._xres(rdd, session)
        seed = self.seed
        if self._fresh:
            seed = (self.seed + 0x9E3779B97F4A7C15 * self._calls) & (2 ** 64 - 1)
            self._calls += 1
        ch = G.choose_mapping(xres, mode, self.privacy_epsilon, self.mapping_range, self.sim_method,
                              self.uniforms, seed, topn=topn)
        if mode == "nonprivate":
            self.single_candidate_rows = int((xres.top_len == 1).sum().item())
        return xres, ch

    def cross_private_mapping(self, rdd, session=None):
        """(target iid, chosen source iid)* -- generator.py:27-98."""
        session = session or rdd.handle.session
        xres, ch = self._map(rdd, session, self.private_mode)
        return LocalRDD(_pairs(session, xres, ch))

    def cross_nonprivate_mapping(self, rdd, topn=4, session=None):
        """generator.py:100-111: one of the first `topn` candidates by |xsim| (the X-SIM stage keeps top_m = 10 of
        them, so topn <= 10 unless extender_pipeline ran with a larger top_m)."""
        session = session or rdd.handle.session
        xres, ch = self._map(rdd, session, "nonprivate", topn=topn)
        return LocalRDD(_pairs(session, xres, ch))

    # ---- profile rewrite -----------------------------------------------------
    def build_alterEgo(self, trainRDD, mapping_dict):
        """(uid, iid, rating, time)*: untouched "T:" ratings then the mapped, mean-merged
        source ratings -- generator.py:140-157."""
        sess = session_of(trainRDD)
        enc = sess.enc
        ipos = {str(s): n for n, s in enumerate(enc.iids)}
        mp = np.full(enc.n_items, -1, dtype=np.int32)
        for s, t in mapping_dict.items():
            if str(s) in ipos:
                mp[ipos[str(s)]] = ipos[str(t)]
        return LocalRDD(alterego_records(sess, torch.as_tensor(mp).to(sess.device)))


def alterego_mapping(privatemap_tool, sess, extended_simRDD, private):
    """The {source: target} item map generator_pipeline applies (assist.py:136-150): [n_items] int32 on the device,
    -1 for an unmapped item.  private selects the tool's private_mode, else the non-private mapping."""
    mode = privatemap_tool.private_mode if private else "nonprivate"
    xres, chosen = privatemap_tool._map(extended_simRDD, sess, mode)
    return G.invert_mapping(xres.start_item, chosen, sess.enc.n_items)


def alterego_records(sess, mapping):
    enc = sess.enc
    ou, oi, orr, ot = G.build_alterego(sess.layout, np.arange(len(enc.user), dtype=np.int64), mapping)
    ou, oi, orr, ot = ou.cpu().numpy(), oi.cpu().numpy(), orr.cpu().numpy(), ot.cpu().numpy()
    uids, iids, times = enc.uids, enc.iids, enc.times
    out = [(str(uids[u]), str(iids[i]), float(r), times[q])
           for q, (u, i, r) in enumerate(zip(enc.user, enc.item, enc.rating)) if enc.has_T[i]]
    out.extend((str(uids[u]), str(iids[i]), r, times[t]) for u, i, r, t in zip(ou, oi, orr, ot))
    return out


def _pairs(session, xres, chosen):
    iids = session.enc.iids
    st, ch = xres.start_item.cpu().numpy(), chosen.cpu().numpy()
    return [(str(iids[t]), str(iids[s])) for t, s in zip(st, ch) if s >= 0]


def _encode_xsim_rows(rows, session, top_m=10):
    """(iid_T, [(iid_S, xsim)*])* records (e.g. produced elsewhere) -> device top-m tables,
    ordered by |xsim| desc with ties to the smaller item index, rows by ascending target."""
    ipos = {str(s): n for n, s in enumerate(session.enc.iids)}
    enc_rows = sorted((ipos[str(t)], [(ipos[str(s)], float(x)) for s, x in lst]) for t, lst in rows)
    n = len(enc_rows)
    te = np.full((n, top_m), -1, np.int32); tx = np.zeros((n, top_m)); tl = np.zeros(n, np.int32)
    cnt = np.zeros(n, np.int32)
    for r, (_, lst) in enumerate(enc_rows):
        lst = sorted(lst, key=lambda p: (-abs(p[1]), p[0]))[:top_m]
        cnt[r] = len(enc_rows[r][1]); tl[r] = len(lst)
        te[r, :len(lst)] = [p[0] for p in lst]; tx[r, :len(lst)] = [p[1] for p in lst]
    dev = session.device
    T = lambda a: torch.as_tensor(a).to(dev)
    return XsimResult(T(np.array([t for t, _ in enc_rows], dtype=np.int32)), T(cnt),
                      torch.zeros(n, dtype=torch.int64, device=dev), T(te), T(tx), T(tl), 0)
