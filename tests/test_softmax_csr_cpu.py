"""CPU tests of the softmax-regression reference (tests/softmax_csr_reference.py): against an independent float64
statement, finite differences, the binary reference at K = 2, the Kronecker expansion against np.kron, and a whole
run through the host mirror of the engine."""
import math

import numpy as np
import scipy.sparse as sp
from scipy.special import logsumexp

import cgoptim_b200 as cg
from oracle import oracle as O

from helpers import make_pair
from logreg_csr_reference import L, LogRegCSR
from numpy_workspace import NumpyObjective
from softmax_csr_reference import SoftmaxCSR, kron_csr


def random_csr(N, d, seed, maxlen=6, long_rows=()):
    """ragged rows (some empty), unsorted columns, plus rows of the given lengths"""
    rng = np.random.default_rng(seed)
    rows = [list(rng.integers(0, d, int(rng.integers(0, maxlen + 1)))) for _ in range(N)]
    for i, n in enumerate(long_rows):
        rows[i] = list(rng.integers(0, d, n))
    rowptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col = np.concatenate([np.asarray(r, dtype=np.int64) for r in rows]).astype(np.int32)
    val = rng.uniform(-1.0, 1.0, col.size)
    return rowptr, col, val


def dense(N, d, rowptr, col, val):
    return sp.csr_matrix((val, col, rowptr), shape=(N, d)).toarray()


def independent_fg(A, y, W, lam):
    """float64 NumPy / SciPy statement of f and ∇f (W: d × K)"""
    N = A.shape[0]
    Z = A @ W
    lse = logsumexp(Z, axis=1)
    f = np.mean(lse - Z[np.arange(N), y]) + 0.5 * lam * np.sum(W * W)
    P = np.exp(Z - lse[:, None])
    P[np.arange(N), y] -= 1.0
    return f, A.T @ P / N + lam * W


def test_reference_matches_independent_statement():
    N, d, K, lam = 700, 40, 5, 1e-3
    rowptr, col, val = random_csr(N, d, 1)
    y = np.random.default_rng(2).integers(0, K, N)
    ref = SoftmaxCSR(N, d, K, rowptr, col, val, y, lam)
    A = dense(N, d, rowptr, col, val)
    rng = np.random.default_rng(3)
    for scale in (0.0, 0.3, 3.0):
        W = scale * rng.standard_normal((d, K))
        f, g = ref.fdf(W.ravel())
        fi, gi = independent_fg(A, y, W, lam)
        assert abs(f - fi) <= 1e-13 * abs(fi)
        assert np.max(np.abs(g - gi.ravel())) <= 1e-13 * np.max(np.abs(gi))


def test_gradient_matches_finite_differences():
    N, d, K = 300, 12, 4
    rowptr, col, val = random_csr(N, d, 4)
    y = np.random.default_rng(5).integers(0, K, N)
    ref = SoftmaxCSR(N, d, K, rowptr, col, val, y, 1e-2)
    w = 0.3 * np.random.default_rng(6).standard_normal(d * K)
    f, g = ref.fdf(w)
    h = 1e-6
    for j in range(d * K):
        e = np.zeros(d * K)
        e[j] = h
        fd = (ref.fdf(w + e)[0] - ref.fdf(w - e)[0]) / (2 * h)
        assert abs(fd - g[j]) <= 1e-7 * max(1.0, abs(g[j]))
    assert math.isfinite(f)


def test_two_classes_equal_binary_logistic_regression():
    """K = 2 with W = [0 | w]: the softmax loss is the binary logistic loss with labels 1 → +1, 0 → −1"""
    N, d, lam = 3000, 50, 1e-3
    rowptr, col, val = random_csr(N, d, 7, long_rows=(L + 5,))
    y = np.random.default_rng(8).integers(0, 2, N)
    sm = SoftmaxCSR(N, d, 2, rowptr, col, val, y, lam)
    lr = LogRegCSR(N, d, rowptr, col, val, np.where(y == 1, 1.0, -1.0), lam)
    lr.set_trial_site(2, 4)
    O.set_cgo_order(G=296)
    for mode in ("seq", "cgo"):
        sm.set_sum_mode(mode)
        lr.set_sum_mode(mode)
        w = 0.5 * np.random.default_rng(9).standard_normal(d)
        W = np.stack([np.zeros(d), w], 1)
        fs, gs = sm.fdf(W.ravel())
        fb, gb = lr.fdf(w)
        assert abs(fs - fb) <= 1e-13 * abs(fb)
        assert np.max(np.abs(gs.reshape(d, 2)[:, 1] - gb)) <= 1e-13 * np.max(np.abs(gb))


def test_kron_expansion_matches_numpy_kron():
    N, d, K = 9, 7, 3
    rowptr, col, val = random_csr(N, d, 10)
    rp, ci, va = kron_csr(N, rowptr, col, val, K)
    E = sp.csr_matrix((va.copy(), ci.copy(), rp.copy()), shape=(N * K, d * K))
    E.sum_duplicates()
    assert np.array_equal(E.toarray(), np.kron(dense(N, d, rowptr, col, val), np.eye(K)))
    for i in range(N):                                       # storage order kept row by row
        for k in range(K):
            r = i * K + k
            assert np.array_equal(ci[rp[r]:rp[r + 1]], col[rowptr[i]:rowptr[i + 1]].astype(np.int64) * K + k)
            assert np.array_equal(va[rp[r]:rp[r + 1]], val[rowptr[i]:rowptr[i + 1]])


def test_whole_run_through_the_host_mirror():
    N, d, K, lam = 400, 10, 3, 1e-3
    rng = np.random.default_rng(11)
    rowptr, col, val = random_csr(N, d - 1, 12)
    cnt = np.diff(rowptr) + 1                                # plus an intercept column
    rp1 = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    last = rp1[1:] - 1
    mask = np.ones(rp1[-1], dtype=bool)
    mask[last] = False
    ci1, va1 = np.empty(rp1[-1], dtype=np.int32), np.empty(rp1[-1])
    ci1[mask], va1[mask] = col, val
    ci1[last], va1[last] = d - 1, 1.0
    y = rng.integers(0, K, N)
    ref = SoftmaxCSR(N, d, K, rp1, ci1, va1, y, lam)
    O.set_cgo_order(G=296)
    _, cfg, ls = make_pair("LBFGS", eps=1e-8, max_iters=500, c1=1e-4, c2=0.9)
    res = cg.minimizeobjective(NumpyObjective(ref), np.zeros(d * K), cfg, ls)
    assert res.status == "success"
    assert abs(ref.fdf(np.zeros(d * K))[0] - math.log(K)) <= 1e-14 * math.log(K)
    A = dense(N, d, rp1, ci1, va1)
    _, g = independent_fg(A, y, res.minimizer.reshape(d, K), lam)
    assert np.max(np.abs(g)) <= 1e-6
