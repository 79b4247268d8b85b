"""Host side of the user-based stage (usersim.py): the fixed-point scale, the norm exponents and the emit block plan,
and the definition itself -- cosine_user is cosine_item on the transposed arrays -- stated in numpy and pinned to
oracle/restate.recommender_cosine_item."""
import numpy as np
import pytest
import torch

from oracle import restate as R


def _user_pairs(user, item, rating, n_users, num_atleast):
    """cosine_user by its definition: every item emits the ordered pairs of distinct records on it; n and sim per
    (u, v).  (The local sensitivity is pinned on the device against recsim's pair kernel, NaN rule included.)"""
    norm2 = np.sqrt(np.bincount(user, weights=rating * rating, minlength=n_users))
    ent = {}
    for i in np.unique(item):
        recs = np.flatnonzero(item == i)                   # list order
        for x in range(len(recs)):
            for y in range(x + 1, len(recs)):
                a, b = recs[x], recs[y]
                ent.setdefault((user[a], user[b]), []).append((rating[a], rating[b]))
                ent.setdefault((user[b], user[a]), []).append((rating[b], rating[a]))
    out = {}
    N = float(num_atleast)
    for (u, v), es in ent.items():
        inner = 0.0
        for ra, rb in es:
            inner += ra * rb
        nn = norm2[u] * norm2[v]
        n = len(es)
        sim = (inner / nn if nn != 0 else 0.0) * min(n, num_atleast) / N
        out[(u, v)] = (n, sim)
    return out


def test_definition_is_cosine_item_transposed():
    rng = np.random.default_rng(2)
    nU, nI, n = 40, 25, 300
    user, item = rng.integers(0, nU, n), rng.integers(0, nI, n)
    rating = rng.integers(1, 11, n) * 0.5
    d = rng.choice(n, 15, replace=False)                  # duplicate records: self pairs
    user, item = np.concatenate([user, user[d]]), np.concatenate([item, item[d]])
    rating = np.concatenate([rating, rng.integers(1, 6, 15).astype(np.float64)])
    P = R.recommender_cosine_item(item, user, rating, nU, 5)
    mine = _user_pairs(user, item, rating, nU, 5)
    assert len(mine) == len(P["i"])
    assert any(u == v for u, v in mine)
    for q in range(len(P["i"])):
        n, sim = mine[(P["i"][q], P["j"][q])]
        assert n == P["n"][q] and sim == P["sim"][q]


def test_scale_base_and_exponents():
    from xmap_b200 import usersim
    assert [usersim.scale_base(m) for m in (1, 2, 3, 4, 5)] == [62, 61, 60, 60, 59]
    e = usersim.norm_exponents(torch.tensor([0.0, 0.5, 1.0, 1.5, 2.0, 1000.0], dtype=torch.float64))
    assert e.tolist() == [0, 0, 1, 1, 2, 10]           # 2^(E-1) <= norm < 2^E


def test_emit_blocks_plan_respects_the_budget():
    from xmap_b200 import recsim
    bound = torch.tensor([3, 0, 7, 1, 1, 10, 2], dtype=torch.int64)
    budget = 10 * recsim.ENTRY_BYTES
    b = recsim.pass_plan(bound, budget)
    assert b[0] == 0 and b[-1] == len(bound)
    for lo, hi in zip(b[:-1], b[1:]):
        assert hi > lo and int(bound[lo:hi].sum()) * recsim.ENTRY_BYTES <= budget
    with pytest.raises(ValueError):
        recsim.pass_plan(torch.tensor([11]), budget)
