"""CPU: the pass plan of the RecommenderSim stage (recsim.row_entries, recsim.pass_plan)."""
import numpy as np
import pytest


def _numpy_row_entries(user, item, n_items):
    d = np.bincount(user)
    out = np.zeros(n_items, dtype=np.int64)
    np.add.at(out, item, d[user] - 1)
    return out


def test_row_entries_against_numpy():
    from xmap_b200 import recsim
    rng = np.random.default_rng(4)
    nU, nI, n = 700, 90, 9000
    user = rng.integers(0, nU, n)
    item = rng.choice(nI - 3, n, p=np.r_[1.0 / np.arange(1, nI - 2)] / np.sum(1.0 / np.arange(1, nI - 2)))
    user[:3], item[:3] = nU + 5, nI - 1                     # a user with three records of one item: self pairs
    want = _numpy_row_entries(user, item, nI)
    got = recsim.row_entries(user, item, nI).numpy()
    assert np.array_equal(got, want)
    # every user with d records owns d (d - 1) entries, each counted on the item of its first record
    d = np.bincount(user)
    assert int(got.sum()) == int((d * (d - 1)).sum()) and got[nI - 2] == 0 and got[nI - 1] > 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_pass_plan_blocks(seed):
    from xmap_b200 import recsim
    import torch
    rng = np.random.default_rng(seed)
    ent = rng.zipf(1.6, 3000).astype(np.int64) * rng.integers(0, 2, 3000)
    ent[[0, 17, 2999]] = 0
    B = recsim.ENTRY_BYTES
    big = int(ent.max()) * B
    for budget in (big, big + 3, 2 * big, max(big, int(ent.sum()) * B // 5), int(ent.sum()) * B, 10 ** 18):
        for lo, hi in ((0, len(ent)), (17, 2000), (40, 41), (5, 5)):
            b = recsim.pass_plan(torch.as_tensor(ent), budget, lo, hi)
            assert b[0] == lo and b[-1] == hi and len(b) >= 2
            assert all(b[q] < b[q + 1] for q in range(len(b) - 1)) or (lo == hi and b == [lo, hi])
            cost = [int(ent[b[q]:b[q + 1]].sum()) * B for q in range(len(b) - 1)]
            assert max(cost) <= budget
            # each block is as long as the budget allows: adding the next row would exceed it
            assert all(cost[q] + int(ent[b[q + 1]]) * B > budget for q in range(len(b) - 2))
    assert recsim.pass_plan(torch.as_tensor(ent), 10 ** 18) == [0, len(ent)]


def test_pass_plan_refuses_a_row_over_the_budget():
    from xmap_b200 import recsim
    import torch
    ent = torch.tensor([3, 0, 9, 4])
    B = recsim.ENTRY_BYTES
    assert recsim.pass_plan(ent, 9 * B) == [0, 2, 3, 4]
    with pytest.raises(ValueError, match="item row 2 has 9 co-rating entries"):
        recsim.pass_plan(ent, 9 * B - 1)
    with pytest.raises(ValueError, match="item row 2"):
        recsim.pass_plan(ent, 9 * B - 1, 0, 2)              # every row is checked, whatever the range
