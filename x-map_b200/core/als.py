"""MLlib-shaped explicit ALS (pyspark.mllib.recommendation.ALS.train / MatrixFactorizationModel), the recommender the
reference README feeds the AlterEgo profile to, served by als.py on the GPU (DESIGN.md section 3.8).

    model = ALS.train(alterego_records, 10, iterations=5, lambda_=0.01)
    model.predict(uid, iid); model.recommendProducts(uid, 10)

Ids are numbered by np.unique and every result is keyed by the original ids.  Divergences from MLlib (DESIGN.md
section 6): the initial factors come from Philox4x32-10 (seed None means 0), `num` is at most 64, ties in a list go
to the smaller product id, there is no NNLS (nonnegative=True raises) and no implicit feedback."""
from collections import namedtuple

import numpy as np
import torch

from .. import als as A
from .. import _native as N
from ..rdd import LocalRDD, records_of

Rating = namedtuple("Rating", ["user", "product", "rating"])


class MatrixFactorizationModel(object):
    """The trained factors with the id arrays that number them (users[k] is user index k, products[k] item index k)."""

    def __init__(self, model, users, products):
        self.model, self.users, self.products = model, users, products
        self.rank = model.rank
        self._upos = {u: k for k, u in enumerate(users)}
        self._ppos = {p: k for k, p in enumerate(products)}

    def predict(self, user, product):
        """The score of one (user, product) pair: sum_k x_u[k] y_p[k] in fp64.  Unknown ids raise KeyError."""
        s = A.predict(self.model, torch.tensor([self._upos[user]]), torch.tensor([self._ppos[product]]))
        return float(s.item())

    def predictAll(self, user_product):
        """Rating(user, product, score) for every pair of known ids (pairs with an unknown id are dropped, as
        MLlib's join drops them)."""
        pairs = [(u, p) for u, p in records_of(user_product) if u in self._upos and p in self._ppos]
        if not pairs:
            return LocalRDD([])
        s = A.predict(self.model, torch.tensor([self._upos[u] for u, _ in pairs]),
                      torch.tensor([self._ppos[p] for _, p in pairs])).cpu().tolist()
        return LocalRDD([Rating(u, p, v) for (u, p), v in zip(pairs, s)])

    def _lists(self, num, users):
        if isinstance(num, bool) or int(num) != num or not 1 <= int(num) <= N.TOPN_MAX:
            raise ValueError("num must be an integer in [1, %d] (a limit of this implementation), got %r"
                             % (N.TOPN_MAX, num))
        top = A.top_n(self.model, int(num), users=users, exclude_rated=False)
        idx, score, ln = top.idx.cpu().numpy(), top.score.cpu().numpy(), top.len.cpu().numpy()
        return idx, score, ln

    def recommendProducts(self, user, num):
        """The num products of highest score for user, best first (rated products included, as in MLlib)."""
        u = self._upos[user]
        idx, score, ln = self._lists(num, torch.tensor([u]))
        return [Rating(user, self.products[idx[u, p]], float(score[u, p])) for p in range(ln[u])]

    def recommendProductsForUsers(self, num):
        """(user, [Rating]) for every user."""
        idx, score, ln = self._lists(num, None)
        return LocalRDD([(user, [Rating(user, self.products[idx[u, p]], float(score[u, p])) for p in range(ln[u])])
                         for u, user in enumerate(self.users)])

    def userFeatures(self):
        return LocalRDD(list(zip(self.users, self.model.user_factors.cpu().double().tolist())))

    def productFeatures(self):
        return LocalRDD(list(zip(self.products, self.model.item_factors.cpu().double().tolist())))


class ALS(object):
    @classmethod
    def train(cls, ratings, rank, iterations=5, lambda_=0.01, blocks=-1, nonnegative=False, seed=None):
        """ratings: an RDD or list of (user, product, rating), or the flat AlterEgo records (uid, iid, rating, time)
        of which the first three fields are used.  blocks is Spark partitioning and has no effect here."""
        if nonnegative:
            raise ValueError("nonnegative=True (NNLS) is not offered")
        recs = records_of(ratings)
        users, user = np.unique(np.array([r[0] for r in recs]), return_inverse=True)
        products, item = np.unique(np.array([r[1] for r in recs]), return_inverse=True)
        rating = np.array([float(r[2]) for r in recs], dtype=np.float64)
        model = A.train(torch.from_numpy(user.astype(np.int64)), torch.from_numpy(item.astype(np.int64)),
                        torch.from_numpy(rating), len(users), len(products), rank, iterations, lambda_, seed=seed)
        return MatrixFactorizationModel(model, users.tolist(), products.tolist())
