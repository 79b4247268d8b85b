"""CPU: the numpy restatement of explicit ALS (tests/als_exact.py) -- its solve within a Cholesky forward-error bound of
the exact solution, its segmented sums, its accuracy on a planted low-rank matrix -- and the argument checks of als.py
that run before any launch."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from tests import als_exact as AX


def _exact_solve(A, b):
    """Gaussian elimination in rationals: the exact solution of the fp64 system."""
    n = len(b)
    M = [[Fraction(float(A[i, j])) for j in range(n)] + [Fraction(float(b[i]))] for i in range(n)]
    for c in range(n):
        p = next(r for r in range(c, n) if M[r][c] != 0)
        M[c], M[p] = M[p], M[c]
        for r in range(n):
            if r != c and M[r][c] != 0:
                f = M[r][c] / M[c][c]
                M[r] = [x - f * y for x, y in zip(M[r], M[c])]
    return [M[i][n] / M[i][i] for i in range(n)]


@pytest.mark.parametrize("r", [1, 4, 9])
def test_solve_within_cholesky_bound(r):
    """Bound.  With u = 2^-53 and gamma_k = k u / (1 - k u), the Cholesky solve of an SPD system of order n computes
    x^ with (A + dA) x^ = b, |dA| <= gamma_(3n+1) |R^T| |R| (Higham, Accuracy and Stability of Numerical Algorithms,
    2nd ed., Thm 10.4), R the computed factor.  R^T R = A + dA1 with |dA1| <= gamma_(n+1) |R^T| |R| (Thm 10.3), and
    || |R^T| |R| ||_2 <= || |R| ||_2^2 <= n ||R||_2^2, so ||R||_2^2 <= ||A||_2 / (1 - n gamma_(n+1)) and
        ||dA||_2 <= eps ||A||_2,   eps = n gamma_(3n+1) / (1 - n gamma_(n+1)).
    Then x^ - x = -A^-1 dA x^, so ||x^ - x||_2 <= kappa_2(A) eps ||x^||_2, x the exact solution."""
    rng = np.random.default_rng(r)
    u = 2.0 ** -53
    g = lambda k: k * u / (1 - k * u)
    eps = r * g(3 * r + 1) / (1 - r * g(r + 1))
    n_rows = 30
    user = np.repeat(np.arange(n_rows), 3 * r)
    item = rng.integers(0, 50, len(user))
    Y = rng.standard_normal((50, r)).astype(np.float32)
    rating = rng.integers(0, 16, len(user)) / 3.0
    A, b, cnt = AX.normal_equations(user, item, rating, n_rows, Y, 0.01)
    x, bad = AX.cholesky_solve(A, b)
    assert not bad.any()
    worst = 0.0
    for q in range(n_rows):
        ex = np.array([float(v) for v in _exact_solve(A[q], b[q])])
        kappa = np.linalg.cond(A[q], 2)
        err = np.linalg.norm(x[q] - ex)
        assert err <= kappa * eps * np.linalg.norm(x[q]), q
        worst = max(worst, err / (kappa * eps * np.linalg.norm(x[q])))
    # the solution of np.linalg.solve on the same fp64 system is near both
    ref = np.linalg.solve(A, b[..., None])[..., 0]
    assert np.allclose(x, ref, rtol=1e-9, atol=1e-12)
    print("r=%d: worst error / bound = %.3g" % (r, worst))


def test_segment_sums_sequential_below_S():
    rng = np.random.default_rng(3)
    r = 5
    Y = rng.standard_normal((40, r)).astype(np.float32)
    for n in (1, 2, 37, AX.S):
        col = rng.integers(0, 40, n)
        rat = rng.integers(0, 16, n) / 3.0
        P, B = AX.segment_sums(col, rat, np.array([0]), np.array([n]), Y)
        I, J = AX.tri(r)
        a, bb = np.zeros(len(I)), np.zeros(r)
        for k in range(n):
            y = Y[col[k]].astype(np.float64)
            for t in range(len(I)):
                a[t] = a[t] + y[I[t]] * y[J[t]]
            for p in range(r):
                bb[p] = bb[p] + rat[k] * y[p]
        assert np.array_equal(P[0].view(np.int64), a.view(np.int64)) and np.array_equal(B[0].view(np.int64),
                                                                                       bb.view(np.int64))


def test_segments_cut_rows_at_S():
    S = AX.S
    row = np.r_[np.zeros(S - 1, np.int64), np.ones(S, np.int64), np.full(S + 1, 2), np.full(3 * S + 1, 4)]
    o, cnt, seg_row, seg_lo, seg_n = AX.segments(row, 6)
    assert seg_row.tolist() == [0, 1, 2, 2, 4, 4, 4, 4]
    assert seg_n.tolist() == [S - 1, S, S, 1, S, S, S, 1]
    assert seg_lo.tolist() == [0, S - 1, 2 * S - 1, 3 * S - 1, 3 * S, 4 * S, 5 * S, 6 * S]


def test_planted_low_rank_rmse_approaches_noise():
    """A rank-5 matrix plus Gaussian noise of sigma 0.1, 30 % of it observed: the restatement's held-out RMSE comes
    down to sigma (the GPU computes the same bits)."""
    rng = np.random.default_rng(0)
    nU, nI, k, sigma = 400, 300, 5, 0.1
    U = rng.standard_normal((nU, k))
    V = rng.standard_normal((nI, k))
    obs = rng.random((nU, nI)) < 0.3
    uu, ii = np.nonzero(obs)
    R = (U @ V.T)[uu, ii] + sigma * rng.standard_normal(len(uu))
    held = rng.random(len(uu)) < 0.1
    X0 = rng.standard_normal((nU, k)).astype(np.float32)
    Y, X = AX.train(uu[~held], ii[~held], R[~held], nU, nI, X0, 10, 0.01)[-1]
    pred = AX.score(X, Y, np.bincount(uu[~held], minlength=nU), np.bincount(ii[~held], minlength=nI), uu[held],
                    ii[held])
    rmse = np.sqrt(np.mean((pred - R[held]) ** 2))
    assert sigma * 0.9 < rmse < sigma * 1.3, rmse


def test_argument_checks_before_any_launch():
    from xmap_b200 import als
    u, i, r = torch.tensor([0, 1]), torch.tensor([1, 0]), torch.tensor([1.0, 2.0])
    ok = dict(rank=3, iterations=1, lam=0.1, device="cpu")
    bad = [dict(rank=0), dict(rank=65), dict(rank=2.5), dict(iterations=0), dict(lam=-0.1), dict(lam=float("nan")),
           dict(lam=True), dict(seed=-1), dict(init=torch.zeros((2, 3), dtype=torch.float64)),
           dict(init=torch.zeros((3, 3), dtype=torch.float32))]
    for b in bad:
        with pytest.raises(ValueError):
            als.train(u, i, r, 2, 2, **dict(ok, **b))
    for args in ((torch.tensor([0, 2]), i, r), (u, torch.tensor([0, -1]), r), (u, i, torch.tensor([1.0])),
                 (u, i, torch.tensor([1.0, float("inf")])), (u.double(), i, r), (u[:1], i, r)):
        with pytest.raises(ValueError):
            als.train(*args, 2, 2, **ok)
    m = als.AlsModel(torch.zeros((2, 3)), torch.zeros((2, 3)), torch.ones(2, dtype=torch.int64),
                     torch.ones(2, dtype=torch.int64), 3, 0.1, 1, None)
    for kw in (dict(n=0), dict(n=65), dict(n=3, candidates=torch.tensor([1, 0])), dict(n=3, users=torch.tensor([2])),
               dict(n=3, users=torch.tensor([1, 1])), dict(n=3, candidates=torch.tensor([0.5])),
               dict(n=3, user=None)):
        args = dict(user=u, item=i)
        args.update(kw)
        with pytest.raises(ValueError):
            als.top_n(m, **args)
    with pytest.raises(ValueError):
        als.predict(m, torch.tensor([2]), torch.tensor([0]))
    from xmap_b200.core import ALS
    with pytest.raises(ValueError):
        ALS.train([("a", "b", 1.0)], 2, nonnegative=True)
