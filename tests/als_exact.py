"""Numpy restatement of explicit ALS as DESIGN.md section 3.8 defines it: the same fp64 operations in the same order,
so the device factors, scores and lists equal it bit for bit.

numpy's elementwise +, -, *, / and sqrt are correctly rounded, as are __dadd_rn, __dsub_rn, __dmul_rn, __ddiv_rn and
__dsqrt_rn.  The product of two fp32 values is exact in fp64, so a + y_i * y_j here rounds once, as the kernel's fma
does.  Packed entries are in the kernels' order: the lower triangle column by column."""
import numpy as np

from xmap_b200._native import ALS_SEGMENT as S


def tri(r):
    """(i, j) of the packed entries, i >= j, column-major: column j holds rows j .. r-1."""
    I = np.concatenate([np.arange(j, r) for j in range(r)])
    J = np.concatenate([np.full(r - j, j) for j in range(r)])
    return I, J


def segments(row, n_rows):
    """Records stably sorted by row, cut into segments of S: (order, count, seg_row, seg_lo, seg_n)."""
    o = np.argsort(row, kind="stable")
    cnt = np.bincount(row, minlength=n_rows).astype(np.int64)
    ptr = np.zeros(n_rows + 1, np.int64)
    ptr[1:] = np.cumsum(cnt)
    nseg = (cnt + S - 1) // S
    seg_row = np.repeat(np.arange(n_rows), nseg)
    k = np.arange(len(seg_row)) - np.repeat(np.cumsum(nseg) - nseg, nseg)
    seg_lo = ptr[seg_row] + k * S
    seg_n = np.minimum(cnt[seg_row] - k * S, S)
    return o, cnt, seg_row, seg_lo, seg_n


def segment_sums(col_s, rat_s, seg_lo, seg_n, Y):
    """Per segment, (A packed, b) summed over its records in list order from +0.0."""
    r = Y.shape[1]
    I, J = tri(r)
    Y64 = Y.astype(np.float64)
    P = np.zeros((len(seg_lo), len(I)))
    B = np.zeros((len(seg_lo), r))
    order = np.argsort(-seg_n, kind="stable")          # the segments still running at step j are a prefix
    for j in range(int(seg_n.max()) if len(seg_n) else 0):
        act = order[:int((seg_n > j).sum())]
        idx = seg_lo[act] + j
        y = Y64[col_s[idx]]
        P[act] = P[act] + y[:, I] * y[:, J]
        B[act] = B[act] + rat_s[idx][:, None] * y
    return P, B


def normal_equations(row, col, rating, n_rows, Y, lam):
    """A (full symmetric [n_rows, r, r]), b, count: the segment partials added in segment order, lam * n on the
    diagonal last."""
    r = Y.shape[1]
    o, cnt, seg_row, seg_lo, seg_n = segments(row, n_rows)
    P, B = segment_sums(col[o], rating[o], seg_lo, seg_n, Y)
    I, J = tri(r)
    Ap = np.zeros((n_rows, len(I)))
    b = np.zeros((n_rows, r))
    first = np.full(n_rows, -1, np.int64)
    for s in range(len(seg_row) - 1, -1, -1):
        first[seg_row[s]] = s
    nseg = (cnt + S - 1) // S
    for k in range(int(nseg.max()) if n_rows else 0):
        rows = np.flatnonzero(nseg > k)
        if k == 0:
            Ap[rows], b[rows] = P[first[rows]], B[first[rows]]
        else:
            Ap[rows] = Ap[rows] + P[first[rows] + k]
            b[rows] = b[rows] + B[first[rows] + k]
    diag = np.flatnonzero(I == J)
    Ap[:, diag] = Ap[:, diag] + (np.float64(lam) * cnt.astype(np.float64))[:, None]
    A = np.zeros((n_rows, r, r))
    A[:, I, J] = Ap
    A[:, J, I] = Ap
    return A, b, cnt


def cholesky_solve(A, b):
    """Column Cholesky (every inner sum in index order from the entry of A), forward substitution (k ascending),
    back substitution (k descending).  Returns (x fp64, bad rows: a pivot not > 0 or NaN)."""
    R, r = b.shape
    L = np.zeros_like(A)
    bad = np.zeros(R, bool)
    with np.errstate(invalid="ignore", divide="ignore"):
        for j in range(r):
            s = A[:, j, j].copy()
            col = A[:, j + 1:, j].copy()
            for k in range(j):
                s = s - L[:, j, k] * L[:, j, k]
                col = col - L[:, j + 1:, k] * L[:, j, k][:, None]
            bad |= ~(s > 0)
            d = np.sqrt(s)
            L[:, j, j] = d
            L[:, j + 1:, j] = col / d[:, None]
        z = b.copy()
        for k in range(r):
            z[:, k] = z[:, k] / L[:, k, k]
            z[:, k + 1:] = z[:, k + 1:] - L[:, k + 1:, k] * z[:, k][:, None]
        for k in range(r - 1, -1, -1):
            z[:, k] = z[:, k] / L[:, k, k]
            z[:, :k] = z[:, :k] - L[:, k, :k] * z[:, k][:, None]
    return z, bad


def half_step(row, col, rating, n_rows, Y, lam):
    """New fp32 factors of every row from the other side's factors Y; rows without records stay zero."""
    A, b, cnt = normal_equations(row, col, rating, n_rows, Y, lam)
    have = cnt > 0
    x, bad = cholesky_solve(A[have], b[have])
    out = np.zeros((n_rows, Y.shape[1]), np.float32)
    out[have] = x.astype(np.float32)
    return out, np.flatnonzero(have)[bad]


def train(user, item, rating, n_users, n_items, init, iterations, lam):
    """[(item factors, user factors)] after every iteration, from the initial user factors."""
    X, out = init.astype(np.float32), []
    for _ in range(iterations):
        Y, bad = half_step(item, user, rating, n_items, X, lam)
        assert not len(bad), bad
        X, bad = half_step(user, item, rating, n_users, Y, lam)
        assert not len(bad), bad
        out.append((Y, X))
    return out


def score(X, Y, x_n, y_n, pu, pi):
    """sum_k x[k] y[k] in fp64 from +0.0, component order; NaN where a side has no records."""
    s = np.zeros(len(pu))
    X64, Y64 = X.astype(np.float64), Y.astype(np.float64)
    for k in range(X.shape[1]):
        s = s + X64[pu, k] * Y64[pi, k]
    s[(x_n[pu] == 0) | (y_n[pi] == 0)] = np.nan
    return s


def top_n(X, Y, x_n, y_n, n, users, cand, rated=None):
    """{user: [(item, score)]} by brute force: score descending, then the smaller item (-0.0 equals 0.0), no NaN."""
    out = {}
    cand = np.asarray(cand)
    cand = cand[y_n[cand] > 0]
    for u in users:
        c = cand if rated is None else np.setdiff1d(cand, rated.get(int(u), ()))
        s = score(X, Y, x_n, y_n, np.full(len(c), u), c)
        lst = sorted(((float(v), int(i)) for v, i in zip(s, c) if v == v), key=lambda e: (-e[0], e[1]))
        out[int(u)] = [(i, v) for v, i in lst[:n]]
    return out
