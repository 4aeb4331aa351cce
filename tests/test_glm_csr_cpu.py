"""CPU tests of the weighted / intercept reference (tests/glm_csr_reference.py): against an independent NumPy / SciPy
statement, finite differences, the references without the options, duplicated rows, an explicit ones column, and
whole runs through the host mirror of the engine and through SciPy's L-BFGS-B."""
import math

import numpy as np
import pytest
import scipy.optimize
import scipy.sparse as sp
from scipy.special import logsumexp

import cgoptim_b200 as cg
from oracle import oracle as O

from glm_csr_reference import LogRegGlmCSR, SoftmaxGlmCSR
from helpers import make_pair
from logreg_csr_reference import L, LogRegCSR
from numpy_workspace import NumpyObjective
from softmax_csr_reference import SoftmaxCSR


def random_csr(N, d, seed, maxlen=6, long_rows=()):
    """ragged rows (some empty), unsorted columns, plus rows of the given lengths"""
    rng = np.random.default_rng(seed)
    rows = [list(rng.integers(0, d, int(rng.integers(0, maxlen + 1)))) for _ in range(N)]
    for i, n in enumerate(long_rows):
        rows[i] = list(rng.integers(0, d, n))
    rowptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col = np.concatenate([np.asarray(r, dtype=np.int64) for r in rows]).astype(np.int32)
    return rowptr, col, rng.uniform(-1.0, 1.0, col.size)


def with_ones_column(N, d, rowptr, col, val):
    """A with a column of ones appended as feature d, stored last in every row"""
    cnt = np.diff(rowptr) + 1
    rp1 = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    last = rp1[1:] - 1
    mask = np.ones(rp1[-1], dtype=bool)
    mask[last] = False
    ci1, va1 = np.empty(rp1[-1], dtype=np.int32), np.empty(rp1[-1])
    ci1[mask], va1[mask] = col, val
    ci1[last], va1[last] = d, 1.0
    return rp1, ci1, va1


def dense(N, d, rowptr, col, val):
    return sp.csr_matrix((val, col, rowptr), shape=(N, d)).toarray()


def make(K, N, d, rowptr, col, val, y, lam, s=None, icpt=False):
    if K == 1:
        return LogRegGlmCSR(N, d, rowptr, col, val, y, lam, sample_weight=s, fit_intercept=icpt)
    return SoftmaxGlmCSR(N, d, K, rowptr, col, val, y, lam, sample_weight=s, fit_intercept=icpt)


def labels(K, N, seed):
    y = np.random.default_rng(seed).integers(0, max(K, 2), N)
    return np.where(y == 1, 1.0, -1.0) if K == 1 else y


def independent_fg(K, A, y, s, x, lam, icpt):
    """float64 NumPy / SciPy statement of f and ∇f; K = 1: binary with y ∈ {±1}"""
    N, d = A.shape
    S = math.fsum(s)
    Kc = max(K, 1)
    W = x[:d * Kc].reshape(d, Kc)
    b = x[d * Kc:] if icpt else np.zeros(Kc)
    Z = A @ W + b
    if K == 1:
        t = -y * Z[:, 0]
        f = np.dot(s, np.logaddexp(0.0, t)) / S
        C = (s * -y / (1.0 + np.exp(-t)))[:, None]
    else:
        lse = logsumexp(Z, axis=1)
        f = np.dot(s, lse - Z[np.arange(N), y]) / S
        C = np.exp(Z - lse[:, None])
        C[np.arange(N), y] -= 1.0
        C = C * s[:, None]
    f = f + 0.5 * lam * np.sum(W * W)
    g = (A.T @ C) / S + lam * W
    return f, np.concatenate([g.ravel(), C.sum(0) / S]) if icpt else g.ravel()


@pytest.mark.parametrize("K", [1, 2, 5])
@pytest.mark.parametrize("icpt", [False, True])
def test_reference_matches_independent_statement(K, icpt):
    N, d, lam = 700, 40, 1e-3
    rowptr, col, val = random_csr(N, d, 1)
    y = labels(K, N, 2)
    s = np.random.default_rng(3).uniform(0.0, 3.0, N)
    ref = make(K, N, d, rowptr, col, val, y, lam, s, icpt)
    A = dense(N, d, rowptr, col, val)
    rng = np.random.default_rng(4)
    for scale in (0.0, 0.3, 3.0):
        x = scale * rng.standard_normal(ref.n)
        f, g = ref.fdf(x)
        fi, gi = independent_fg(K, A, y, s, x, lam, icpt)
        assert abs(f - fi) <= 1e-13 * abs(fi)
        assert np.max(np.abs(g - gi)) <= 1e-13 * np.max(np.abs(gi))


@pytest.mark.parametrize("K", [1, 3])
def test_finite_differences(K):
    """∇f in w and b with non-uniform weights, and ∂f/∂s_i = (s-free loss ℓ_i − Σ s ℓ / S) / S"""
    N, d, lam = 300, 12, 1e-2
    rowptr, col, val = random_csr(N, d, 5)
    y = labels(K, N, 6)
    s = np.random.default_rng(7).uniform(0.1, 2.0, N)
    ref = make(K, N, d, rowptr, col, val, y, lam, s, True)
    x = 0.3 * np.random.default_rng(8).standard_normal(ref.n)
    f, g = ref.fdf(x)
    h = 1e-6
    for j in range(ref.n):
        e = np.zeros(ref.n)
        e[j] = h
        fd = (ref.fdf(x + e)[0] - ref.fdf(x - e)[0]) / (2 * h)
        assert abs(fd - g[j]) <= 1e-7 * max(1.0, abs(g[j]))
    lp, _ = ref.loss_and_c(x)
    Lw = np.dot(s, lp) / math.fsum(s)
    for i in (0, 17, N - 1):
        fs = []
        for sign in (1, -1):
            s2 = s.copy()
            s2[i] += sign * h
            fs.append(make(K, N, d, rowptr, col, val, y, lam, s2, True).fdf(x)[0])
        assert abs((fs[0] - fs[1]) / (2 * h) - (lp[i] - Lw) / math.fsum(s)) <= 1e-7


@pytest.mark.parametrize("K", [1, 4])
@pytest.mark.parametrize("mode", ["seq", "cgo"])
def test_unit_weights_equal_the_references_without_options(K, mode):
    N, d, lam = 3000, 30, 1e-3
    rowptr, col, val = random_csr(N, d, 9, long_rows=(L + 3,))
    y = labels(K, N, 10)
    if K == 1:
        base = LogRegCSR(N, d, rowptr, col, val, y, lam)
        base.set_trial_site(2, 4)
    else:
        base = SoftmaxCSR(N, d, K, rowptr, col, val, y, lam)
    O.set_cgo_order(G=296)
    x = 0.4 * np.random.default_rng(11).standard_normal(d * K)
    base.set_sum_mode(mode)
    fb, gb = base.fdf(x)
    for s in (None, np.ones(N)):
        ref = make(K, N, d, rowptr, col, val, y, lam, s)
        ref.set_sum_mode(mode)
        f, g = ref.fdf(x)
        assert f == fb and np.array_equal(g, gb)


@pytest.mark.parametrize("K", [1, 3])
def test_integer_weights_match_duplicated_rows(K):
    N, d, lam = 400, 20, 1e-3
    rowptr, col, val = random_csr(N, d, 12)
    y = labels(K, N, 13)
    s = np.random.default_rng(14).integers(0, 4, N).astype(np.float64)
    rows = np.repeat(np.arange(N), s.astype(np.int64))
    lens = np.diff(rowptr)[rows]
    rp2 = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    take = np.concatenate([np.arange(rowptr[i], rowptr[i + 1]) for i in rows])
    ref = make(K, N, d, rowptr, col, val, y, lam, s, True)
    dup = make(K, rows.size, d, rp2, col[take], val[take], y[rows], lam, None, True)
    x = 0.5 * np.random.default_rng(15).standard_normal(ref.n)
    f, g = ref.fdf(x)
    f2, g2 = dup.fdf(x)
    assert abs(f - f2) <= 1e-12 * abs(f2)
    assert np.max(np.abs(g - g2)) <= 1e-12 * np.max(np.abs(g2))


@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("G", [1, 3, 296])
def test_intercept_equals_an_explicit_ones_column(K, G):
    """λ = 0, N > CGO_LONG_ROW, every row of A shorter than CGO_LONG_ROW: bit for bit"""
    N, d = L + 300, 25
    rowptr, col, val = random_csr(N, d, 16, maxlen=9, long_rows=(L - 1,))
    y = labels(K, N, 17)
    rp1, ci1, va1 = with_ones_column(N, d, rowptr, col, val)
    O.set_cgo_order(G=G)
    s = np.random.default_rng(18).uniform(0.5, 2.0, N)
    for w in (None, s):
        ref = make(K, N, d, rowptr, col, val, y, 0.0, w, True)
        ones = make(K, N, d + 1, rp1, ci1, va1, y, 0.0, w, False)
        for mode in ("seq", "cgo"):
            ref.set_sum_mode(mode)
            ones.set_sum_mode(mode)
            x = 0.3 * np.random.default_rng(19).standard_normal(ref.n)
            f, g = ref.fdf(x)
            f1, g1 = ones.fdf(x)
            assert f == f1 and np.array_equal(g, g1)
    O.set_cgo_order(G=296)


@pytest.mark.parametrize("K", [1, 3])
def test_whole_run_through_the_host_mirror(K):
    N, d, lam = 400, 10, 1e-3
    rowptr, col, val = random_csr(N, d, 20)
    y = labels(K, N, 21)
    s = np.random.default_rng(22).uniform(0.0, 2.0, N)
    ref = make(K, N, d, rowptr, col, val, y, lam, s, True)
    O.set_cgo_order(G=296)
    _, cfg, ls = make_pair("LBFGS", eps=1e-8, max_iters=500, c1=1e-4, c2=0.9)
    res = cg.minimizeobjective(NumpyObjective(ref), np.zeros(ref.n), cfg, ls)
    assert res.status == "success"
    _, g = independent_fg(K, dense(N, d, rowptr, col, val), y, s, res.minimizer, lam, True)
    assert np.max(np.abs(g)) <= 1e-6


@pytest.mark.parametrize("K", [1, 3])
def test_converged_fit_matches_scipy(K):
    N, d, lam = 300, 8, 1e-2
    rowptr, col, val = random_csr(N, d, 23)
    y = labels(K, N, 24)
    s = np.random.default_rng(25).uniform(0.2, 3.0, N)
    ref = make(K, N, d, rowptr, col, val, y, lam, s, True)
    A = dense(N, d, rowptr, col, val)
    O.set_cgo_order(G=296)
    _, cfg, ls = make_pair("LBFGS", eps=1e-10, max_iters=1000, c1=1e-4, c2=0.9)
    res = cg.minimizeobjective(NumpyObjective(ref), np.zeros(ref.n), cfg, ls)
    sp_res = scipy.optimize.minimize(lambda x: independent_fg(K, A, y, s, x, lam, True), np.zeros(ref.n), jac=True,
                                     method="L-BFGS-B", options={"gtol": 1e-12, "ftol": 1e-15, "maxiter": 5000})
    assert np.max(np.abs(res.minimizer - sp_res.x)) <= 1e-6
    assert abs(res.objective - sp_res.fun) <= 1e-6 * abs(sp_res.fun)
