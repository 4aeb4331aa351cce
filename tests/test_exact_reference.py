"""The exact references of tests/exact_reference.py checked on the CPU: that they are exact, that the canonical
order (as the oracle restates it) stays inside the a-priori bound at every shape the GPU sweep uses, that the bound
is tight enough to catch a dropped or repeated tile there, and the L-BFGS history of the NumPy mirror against a
dense extended-precision BFGS inverse, rejections included."""
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle as O

import exact_reference as X
from numpy_workspace import NumpyObjective


def test_exact_dot_is_correctly_rounded():
    rng = np.random.default_rng(3)
    for n in (1, 2, 7, 1000):
        a = rng.standard_normal(n) * 10.0 ** rng.integers(-8, 8, n)
        b = rng.standard_normal(n) * 10.0 ** rng.integers(-8, 8, n)
        exact = sum(Fraction(float(p)) * Fraction(float(q)) for p, q in zip(a, b))
        assert X.exact_dot(a, b) == float(exact)
        assert X.exact_sum(a) == float(sum(Fraction(float(p)) for p in a))
    # catastrophic cancellation: the fp64 sum is 0, the exact one is not
    a = np.array([1e16, 1.0, -1e16])
    assert X.exact_sum(a) == 1.0 and X.exact_dot(a, np.ones(3)) == 1.0


def _tiles(n):
    """element ranges of the first, a middle and the last BLAS-1 tile"""
    nt = -(-n // X.T)
    return sorted({(k * X.T, min((k + 1) * X.T, n)) for k in (0, nt // 2, nt - 1)})


@pytest.mark.parametrize("G,n", X.SWEEP_EVEN + X.SWEEP_ODD)
def test_oracle_canonical_dot_within_bound_and_bound_catches_a_lost_tile(G, n):
    rng = np.random.default_rng(n + G)
    a, b = rng.uniform(0.5, 1.5, n), rng.uniform(0.5, 1.5, n)
    a[::3] *= -1.0                                   # cancellation in the dot; the sum of squares has none
    O.set_cgo_order(G, 1)
    O.set_site(2, 4)
    try:
        for u, v in ((a, b), (a, a)):
            got = O.dot(u, v, "cgo")
            bound = X.canonical_bound(n, G, (2, 4), X.exact_dot(np.abs(u), np.abs(v)))
            assert abs(got - X.exact_dot(u, v)) <= bound
        exact = X.exact_sumsq(a)
        bound = X.canonical_bound(n, G, (2, 4), exact)
        for lo, hi in _tiles(n):
            dropped, twice = a.copy(), a.copy()
            dropped[lo:hi] = 0.0
            twice[lo:hi] *= np.sqrt(2.0)             # (√2 a)² counts the tile's terms twice, up to rounding
            assert abs(O.dot(dropped, dropped, "cgo") - exact) > bound, (lo, hi)
            assert abs(O.dot(twice, twice, "cgo") - exact) > bound, (lo, hi)
    finally:
        O.set_cgo_order(296, 1)


def test_canonical_depth_follows_the_tree():
    # one tile, G = 1: 8 terms per lane, 5 + 7 for the CTA, one finish addition, 5 + 7 for the finish
    assert X.canonical_depth(1, 1) == 8 + 12 + 1 + 12
    assert X.canonical_depth(X.T, 296) == 8 + 12 + 1 + 12
    assert X.canonical_depth(X.T + 1, 1) == 16 + 12 + 1 + 12           # two tiles on virtual CTA 0
    assert X.canonical_depth(297 * X.T, 296) == 16 + 12 + 2 + 12       # (G+1)·T wraps; 296 partials
    assert X.canonical_depth(8193 * X.T, 8192) == 16 + 12 + 32 + 12
    assert X.canonical_depth(3000, 296, (1, 1)) == 1 + 12 + 1 + 12     # rows: one per lane, 12 tiles
    assert X.canonical_depth(3000, 3, (1, 1)) == 4 + 12 + 1 + 12       # 12 tiles over 3 virtual CTAs


# --------------------------------------------------------------------------------------------- L-BFGS
def _reject_script(m):
    """rejections at count < m (m > 1), at count == m, and twice in a row at count == m"""
    return {1, m + 2, 2 * m + 4, 2 * m + 5}, 2 * m + 8


@pytest.mark.parametrize("n", [100, 101])
@pytest.mark.parametrize("m", [1, 3, 64])
def test_lbfgs_mirror_matches_dense_bfgs_with_rejections(m, n):
    """The NumPy mirror of the device history (tests/numpy_workspace.py), driven through the same calls as the
    device: every direction equals −H g of the textbook history to 1e-10 (it agrees to ~5e-16), also right after a
    rejected pair.  The test checks its own power: at every rejection with a full history, dropping the oldest pair
    as well must move the textbook direction by more than 1e-6, so a history that loses a pair there cannot pass."""
    rp, ci, va, b = X.well_conditioned_ls(n, 11 + n)
    obj = NumpyObjective(O.Objective.sparse_ls_csr(n, n, rp, ci, va, b))
    ws = obj.make_workspace(np.zeros(n), lbfgs_m=m)
    reject, steps = _reject_script(m)
    errs, counts, power = X.drive_lbfgs(ws, m, steps, reject, a=0.05)
    assert counts[-3:] == [m, m, m] and (m == 1 or counts[0] < m)
    assert len(power) >= 3 and min(power) > 1e-6, power
    bad = [(k, e) for k, e in enumerate(errs) if not e <= 1e-10]
    assert not bad, f"steps where u != −H g (step, rel. error): {bad[:6]}"


def test_lbfgs_natural_rejection_at_full_history_oracle_matches_mirror():
    """A whole run in which a pair is rejected with the history full, with no forcing: the oracle's own history
    (cgo_oracle.c lbfgs_push / lbfgs_updatedir) must reproduce the run of the host engine over the NumPy mirror bit
    for bit — the mirror being the history the dense-BFGS test above pins to the textbook.  An oracle that drops its
    oldest pair on that rejection restarts from −g there and leaves the mirror's trace."""
    import cgoptim_b200 as cg
    from helpers import assert_same_run, natural_lbfgs_rejection_case
    ocfg, cfg, ls, x0 = natural_lbfgs_rejection_case()
    ora = O.minimize(O.Objective.rosenbrock_chained(2), x0, ocfg)
    mirror = NumpyObjective(O.Objective.rosenbrock_chained(2))
    log, make = [], mirror.make_workspace

    def counting(*a, **k):
        ws = make(*a, **k)
        commit = ws.lbfgs_commit_pair

        def counted(c, rho=0.0, gamma=1.0):
            log.append((bool(c), ws.count))
            commit(c, rho, gamma)
        ws.lbfgs_commit_pair = counted
        return ws
    mirror.make_workspace = counting
    with np.errstate(all="ignore"):
        ret = cg.minimizeobjective(mirror, x0, cfg, ls)
    first = next(i for i, (c, k) in enumerate(log) if not c and k == 1)
    assert first < len(log) - 5, "the rejection at full history must not be the run's last step"
    assert_same_run(ret, ora, what="LBFGS(1) + Backtracking, chained Rosenbrock n = 2")
