"""CPU tests of the reference for logistic regression on a host CSR (tests/logreg_csr_reference.py): the same numbers
and runs as the oracle's synthetic objective on the same matrix, the long-row rule of include/cgoptim.h against an
independent NumPy restatement and the exact-reference bound, the gradient, and the minimiser of a problem with an
intercept."""
import math

import numpy as np
import pytest
from scipy.optimize import minimize as sp_minimize

import cgoptim_b200 as cg
from oracle import oracle as O

import exact_reference as X
from helpers import assert_same_run, make_pair
from logreg_csr_reference import L, LogRegCSR
from numpy_workspace import NumpyObjective


def canonical_sum(terms, G, U=4):
    """the canonical order of include/cgoptim.h with V = 1: item k goes to lane k % 256 of virtual CTA
    (k // (256 U)) % G; lanes add their items in index order from +0.0, a CTA combines its lanes by the xor
    butterfly and then over the 8 warps, and the grid combines the CTA partials the same way"""
    terms = np.asarray(terms, dtype=np.float64)
    tile = 256 * U
    ntiles = max(-(-terms.size // tile), 1)
    rounds = -(-ntiles // G)
    padded = np.zeros(rounds * G * tile)
    padded[:terms.size] = terms
    items = padded.reshape(rounds, G, U, 256)
    acc = np.zeros((G, 256))
    for r in range(rounds):
        for j in range(U):
            acc = acc + items[r, :, j, :]

    def combine(lanes):                                  # lanes: (..., 256)
        v = lanes.reshape(lanes.shape[:-1] + (8, 32)).copy()
        idx = np.arange(32)
        for off in (16, 8, 4, 2, 1):
            v = v + v[..., idx ^ off]
        w = v[..., 0]
        s = w[..., 0]
        for k in range(1, 8):
            s = s + w[..., k]
        return s

    P = combine(acc)[:min(ntiles, G)]
    lanes = np.zeros(256)
    for c in range(P.size):
        lanes[c % 256] = lanes[c % 256] + P[c]
    return float(combine(lanes))


def sequential_sum(terms):
    s = 0.0
    for t in np.asarray(terms, dtype=np.float64):
        s = s + t
    return s


def synthetic_pair(N, d, K, lam, seed=24):
    syn = O.Objective.logreg(N, d, K, seed, lam)
    rp, ci, va = syn.csr(False)
    csr = LogRegCSR(N, d, rp, ci, va, syn.rhs(), lam)
    return syn, csr


@pytest.mark.parametrize("N,d,K", [(300, 64, 5), (1000, 200, 20), (33, 7, 3)])
def test_csr_constructor_matches_synthetic(N, d, K):
    syn, csr = synthetic_pair(N, d, K, 1e-3)
    for t in (False, True):
        for a, b in zip(syn.csr(t), csr.csr(t)):
            assert np.array_equal(a, b)
    w = 0.3 * np.random.default_rng(2).standard_normal(d)
    for mode, sites in (("seq", [(1, 1)]), ("cgo", [(1, 1), (2, 4)])):
        for site in sites:
            for o in (syn, csr):
                o.set_sum_mode(mode)
                o.set_trial_site(*site)
            fs, gs = syn.fdf(w)
            fc, gc = csr.fdf(w)
            assert fs == fc and np.array_equal(gs, gc), (mode, site)


@pytest.mark.parametrize("flavour", ["LBFGS", "HagerZhang"])
def test_runs_match_the_oracle_on_the_synthetic_matrix(flavour):
    """the host mirror of the engine on the reference runs the oracle's own minimisation bit for bit"""
    N, d, K, lam = 2000, 150, 8, 1e-3
    ocfg, cfg, ls = make_pair(flavour, max_iters=40, c1=1e-4, c2=0.9)
    syn, csr = synthetic_pair(N, d, K, lam)
    for site in ((1, 1), (2, 4)):
        syn.set_trial_site(*site)
        csr.set_trial_site(*site)
        ora = O.minimize(syn, np.zeros(d), ocfg)
        ret = cg.minimizeobjective(NumpyObjective(csr), np.zeros(d), cfg, ls)
        assert_same_run(ret, ora, what=f"{flavour} {site}")


def _long_rows_csr(lengths, d, seed):
    """a sample row for every length (its columns drawn with repeats and out of order) plus short rows"""
    rng = np.random.default_rng(seed)
    rows = [rng.integers(0, d, n) for n in lengths] + [rng.integers(0, d, rng.integers(0, 6)) for _ in range(40)]
    rowptr = np.concatenate([[0], np.cumsum([r.size for r in rows])]).astype(np.int64)
    col = np.concatenate(rows).astype(np.int32)
    val = rng.uniform(-1.0, 1.0, col.size)
    y = np.where(rng.random(len(rows)) < 0.5, -1.0, 1.0)
    return len(rows), rowptr, col, val, y


@pytest.mark.parametrize("G", [296, 3])
def test_long_rows_follow_the_canonical_order(G):
    lengths = [L - 1, L, L + 1, 3 * L]
    d = 5000
    N, rowptr, col, val, y = _long_rows_csr(lengths, d, 7)
    # Aᵀ: features 0..3 appear in exactly `lengths` samples (a column of that many entries)
    NT = 3 * L + 10
    rng = np.random.default_rng(8)
    rowsT = [np.sort(rng.choice(NT, n, replace=False)) for n in lengths]
    trip = [(i, j) for j, r in enumerate(rowsT) for i in r]
    trip += [(i, 4 + int(rng.integers(0, 60))) for i in range(NT)]
    trip.sort()
    ri = np.array([t[0] for t in trip])
    rpT = np.searchsorted(ri, np.arange(NT + 1)).astype(np.int64)
    colT = np.array([t[1] for t in trip], dtype=np.int32)
    valT = rng.uniform(-1.0, 1.0, colT.size)
    yT = np.where(rng.random(NT) < 0.5, -1.0, 1.0)
    O.set_cgo_order(G=G)
    try:
        for (n, nf, rp, ci, va, yy), transposed in (((N, d, rowptr, col, val, y), False), ((NT, 64, rpT, colT, valT, yT), True)):
            ora = LogRegCSR(n, nf, rp, ci, va, yy, 1e-4)
            orp, oci, ova = ora.csr(transposed)
            x = np.random.default_rng(9).uniform(-1.0, 1.0, n if transposed else nf)
            seq = ora.spmv(x, transposed)
            ora.set_trial_site(2, 4)
            got = ora.spmv(x, transposed)
            for r in range(orp.size - 1):
                terms = ova[orp[r]:orp[r + 1]] * x[oci[orp[r]:orp[r + 1]]]
                if terms.size > L:
                    assert got[r] == canonical_sum(terms, G), (transposed, r, terms.size)
                    exact = X.exact_dot(ova[orp[r]:orp[r + 1]], x[oci[orp[r]:orp[r + 1]]])
                    assert abs(got[r] - exact) <= X.canonical_bound(terms.size, G, (1, 4), float(np.abs(terms).sum()))
                else:
                    assert got[r] == sequential_sum(terms) == seq[r]
            assert sorted(np.diff(orp)[np.diff(orp) > L - 2].tolist()) == [L - 1, L, L + 1, 3 * L]
    finally:
        O.set_cgo_order(G=296)


def test_gradient_matches_finite_differences():
    N, d = 400, 30
    rng = np.random.default_rng(3)
    N_, rowptr, col, val, y = _long_rows_csr([50] * 5, d, 4)
    ora = LogRegCSR(N_, d, rowptr, col, val, y, 1e-2)
    w = 0.2 * rng.standard_normal(d)
    f, g = ora.fdf(w)
    h = 1e-6
    for j in range(d):
        e = np.zeros(d)
        e[j] = h
        fd = (ora.fdf(w + e)[0] - ora.fdf(w - e)[0]) / (2 * h)
        assert abs(fd - g[j]) <= 1e-7 * max(1.0, abs(g[j]))
    assert math.isfinite(f)


def test_intercept_minimiser_matches_scipy():
    """a column of ones is the intercept; λ penalises it like every other weight"""
    rng = np.random.default_rng(11)
    N, d, lam = 300, 8, 1e-3
    X_ = rng.standard_normal((N, d))
    X_[rng.random((N, d)) < 0.5] = 0.0
    X_ = np.hstack([X_, np.ones((N, 1))])
    w_true = rng.standard_normal(d + 1)
    y = np.where(X_ @ w_true + 0.5 * rng.standard_normal(N) >= 0.0, 1.0, -1.0)
    nz = X_ != 0.0
    rowptr = np.concatenate([[0], np.cumsum(nz.sum(1))]).astype(np.int64)
    col = np.nonzero(nz)[1].astype(np.int32)
    val = X_[nz]
    ora = LogRegCSR(N, d + 1, rowptr, col, val, y, lam)
    _, cfg, ls = make_pair("LBFGS", eps=1e-12, max_iters=500, c1=1e-4, c2=0.9)
    res = cg.minimizeobjective(NumpyObjective(ora), np.zeros(d + 1), cfg, ls)

    def fg(w):
        z = X_ @ w
        t = -y * z
        f = np.mean(np.logaddexp(0.0, t)) + 0.5 * lam * w @ w
        s = 0.5 * (1.0 + np.tanh(0.5 * t))
        return f, X_.T @ (-y * s) / N + lam * w
    ref = sp_minimize(fg, np.zeros(d + 1), jac=True, method="L-BFGS-B", options={"gtol": 1e-12, "ftol": 0.0, "maxiter": 10000})
    assert np.max(np.abs(res.minimizer - ref.x)) <= 1e-6
    assert ora.fdf(np.zeros(d + 1))[0] == pytest.approx(math.log(2.0), rel=1e-12)
