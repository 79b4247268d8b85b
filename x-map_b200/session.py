"""Per-training-set device state shared by the pipeline facades.

The reference threads one trainRDD through three pipelines
(twodomain_demo.py:87-105).  The facades encode it once, keep the layout in
HBM, and attach the session to the RDD object they were given (and to every
lazy RDD they return) so that the next stage finds the device-resident result
instead of re-encoding Python records.
"""
import numpy as np
import torch

from . import encode as ENC
from . import engine as E
from .rdd import records_of


class Session(object):
    def __init__(self, enc, device="cuda", user=None, item=None, rating=None, meta=None):
        """enc: the host-side Encoded.  user / item / rating / meta: the same arrays and item codes already on the
        device (ingest.clean_split_pipeline), used instead of copying enc's."""
        self.enc = enc
        self.device = torch.device(device)
        dev = lambda t, a: a if t is None else t
        self.layout = E.build_layout(dev(user, enc.user), dev(item, enc.item), dev(rating, enc.rating), enc.n_users,
                                     enc.n_items, device=self.device)
        T = lambda a, dt: torch.as_tensor(a, dtype=dt).to(self.device)
        self.meta = meta if meta is not None else E.ItemMeta(
            T(enc.prefix_code, torch.int32), T(enc.dom_code, torch.uint8), T(enc.contains, torch.uint8),
            T(enc.has_S, torch.bool), T(enc.has_T, torch.bool))
        self.sim_engine = None      # engine.SimEngine once similarity has run
        self.tables = None
        self.xsim = None            # (plan, engine, result)

    # ---- stage 1 -----------------------------------------------------------
    def similarity(self, method, num_atleast, k):
        eng = self.sim_engine
        if eng is None or (eng.method, eng.num_atleast, eng.k) != (method, int(num_atleast), int(k)):
            eng = E.SimEngine(self.layout, self.meta, method, num_atleast, k)
            self.tables = eng.run()
            self.sim_engine = eng
        return self.tables

    def user_info(self):
        """{uid: (average, norm2)} as BaselinerSim.get_universal_user_info (baselinerSim.py:17-38)."""
        enc = self.enc
        mu = self.layout.user_mu.cpu().numpy()
        s2 = np.bincount(enc.user, weights=enc.rating * enc.rating, minlength=enc.n_users)
        return [(str(u), (float(a), float(np.sqrt(b)))) for u, a, b in zip(enc.uids, mu, s2)]

    def item_info(self):
        """{iid: (average, norm2, adjusted norm2, count)} (baselinerSim.py:40-82)."""
        st = self.layout.item_stats.cpu().numpy()
        return [(str(i), tuple(float(x) for x in row)) for i, row in zip(self.enc.iids, st)]


def session_of(rdd, device="cuda"):
    """Find or create the Session of a train RDD (records (uid, [(iid, rating, time)]))."""
    s = getattr(rdd, "_xmap_session", None)
    if s is None:
        s = Session(ENC.encode_records(records_of(rdd)), device)
        try:
            rdd._xmap_session = s
        except AttributeError:
            pass
    return s
