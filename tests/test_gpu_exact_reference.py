"""The kernels against exact references (tests/exact_reference.py), at the edges of their tiling.

Elementwise outputs (xp, g⁺, u) are IEEE +, −, ×, ÷ with contraction off on both sides, so they must equal NumPy
bit for bit.  Every reduced scalar must lie within the a-priori canonical-order bound of its correctly rounded
value, and still equal the oracle bit for bit (which the bound alone would not notice if the order changed).
L-BFGS directions are compared with a dense extended-precision BFGS inverse, and the CSR kernels with exact row
sums at the extremes of their shared-memory ring."""
import ctypes as C

import numpy as np
import pytest

import cgoptim_b200 as cg
import cgoptim_b200._capi as capi
from oracle import oracle as O

import exact_reference as X
from helpers import assert_same_run, make_pair, natural_lbfgs_rejection_case

pytestmark = pytest.mark.gpu
T = X.T


@pytest.fixture(scope="module")
def ctx():
    c = cg.Context(0)
    yield c
    c.close()


def _within(got, exact, bound, what):
    assert abs(got - exact) <= bound, f"{what}: |{got!r} − {exact!r}| = {abs(got - exact):.3e} > bound {bound:.3e}"


def _check_sum(got, a, b, n, G, site, what):
    """a reduced dot: within the canonical bound of the exact value, and the oracle's canonical value bit for bit"""
    _within(got, X.exact_dot(a, b), X.canonical_bound(n, G, site, X.exact_dot(np.abs(a), np.abs(b))), what)
    O.set_site(*site)
    try:
        ora = O.dot(a, b, "cgo")
    finally:
        O.set_site(2, 4)
    assert got == ora, f"{what}: differs from the oracle's canonical order"


def _check_trial_pack(P, G, n, site, u, g, gp, phi, phi_ref):
    """phi: (exact, bound, oracle value) of CGO_P_PHI; the other eight slots from the vectors"""
    exact, bound, ora = phi_ref
    _within(phi, exact, bound, "phi")
    assert phi == ora, "phi differs from the oracle"
    y = gp - g
    for slot, (a, b) in enumerate([(gp, u), (gp, gp), (y, y), (u, y), (y, gp), (gp, g), (u, g), (u, u)], start=1):
        _check_sum(float(P[slot]), a, b, n, G, site, f"pack slot {slot}")


def _rosen_numpy(xp):
    """extended Rosenbrock, the kernel's arithmetic (blas1.cu RosenTrial) in NumPy: per-pair f and g⁺"""
    p1, p2 = xp[0::2], xp[1::2]
    t = p2 - p1 * p1
    om = 1.0 - p1
    f = (100.0 * t) * t + om * om
    gp = np.empty_like(xp)
    gp[0::2] = (-400.0 * p1) * t - 2.0 * om
    gp[1::2] = 200.0 * t
    return f, gp


def _bidiagonal(n, seed):
    """square n×n CSR: diagonal in [1, 2], superdiagonal in [−½, ½]"""
    rng = np.random.default_rng(seed)
    lens = np.full(n, 2, dtype=np.int64)
    lens[-1] = 1
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.empty(rowptr[-1], dtype=np.int32)
    val = np.empty(rowptr[-1])
    col[rowptr[:-1]] = np.arange(n)
    val[rowptr[:-1]] = rng.uniform(1.0, 2.0, n)
    col[rowptr[:-1][:-1] + 1] = np.arange(1, n)
    val[rowptr[:-1][:-1] + 1] = rng.uniform(-0.5, 0.5, n - 1)
    return rowptr, col, val, rng.standard_normal(n)


def _sweep_one(ctx, obj, G, n, x0, site, phi_of):
    """reset_direction, a trial, the L-BFGS stage dots, literal β, ‖u + g‖², update_dir(β) and the fused trial,
    each checked elementwise against NumPy and per reduced scalar against the exact value and the oracle.
    phi_of(xp) -> ((exact, bound, oracle phi), oracle g⁺)."""
    ws = obj.make_workspace(x0, lbfgs_m=1, fuse_direction=False)
    try:
        x, g = ws.download_vector("x"), ws.download_vector("df_x")
        assert np.array_equal(x, x0)
        ws.reset_direction()
        u = ws.download_vector("u")
        assert np.array_equal(u, -g)
        _check_sum(float(ws.dpack[0]), g, u, n, G, (2, 4), "reset g·u")
        _check_sum(float(ws.dpack[1]), u, u, n, G, (2, 4), "reset u·u")

        a = 1e-3
        ws.eval_trial(a)
        xp, gp = ws.download_vector("xp"), ws.download_vector("df_xp")
        assert np.array_equal(xp, x + a * u)
        phi_ref, gp_ora = phi_of(xp)
        assert np.array_equal(gp, gp_ora)
        _check_trial_pack(ws.pack, G, n, site, u, g, gp, float(ws.pack[0]), phi_ref)

        sy, yy = ws.lbfgs_stage_pair()
        s, y = xp - x, gp - g
        _check_sum(float(sy), s, y, n, G, (2, 4), "L-BFGS s·y")
        _check_sum(float(yy), y, y, n, G, (2, 4), "L-BFGS y·y")
        ws.lbfgs_commit_pair(False)

        R, m = 1.7, 0.3
        _check_sum(float(ws.beta_literal(R, m)), y - m * u, gp / R, n, G, (2, 4), "literal β")

        beta = 0.37
        ws.update_dir(beta)
        u2 = ws.download_vector("u")
        assert np.array_equal(u2, -g + beta * u)
        _check_sum(float(ws.dpack[0]), g, u2, n, G, (2, 4), "update_dir g·u")
        _check_sum(float(ws.dpack[1]), u2, u2, n, G, (2, 4), "update_dir u·u")
        v = C.c_double()                             # u2 + g = β u ≠ 0 (right after reset_direction it is 0)
        capi.check(capi.lib().cgo_norm_sq_u_plus_g(ws.h, C.byref(v)))
        _check_sum(v.value, u2 + g, u2 + g, n, G, (2, 4), "‖u + g‖²")

        ws.fuse_direction = True                     # u = −g + βu rides on the next trial
        beta, a = -0.21, 2e-3
        ws.update_dir(beta)
        ws.hint_first_trial(a)
        ws.eval_trial(a)
        u3, xp, gp = ws.download_vector("u"), ws.download_vector("xp"), ws.download_vector("df_xp")
        assert np.array_equal(u3, -g + beta * u2)
        assert np.array_equal(xp, x + a * u3)
        phi_ref, gp_ora = phi_of(xp)
        assert np.array_equal(gp, gp_ora)
        _check_trial_pack(ws.pack, G, n, site, u3, g, gp, float(ws.pack[0]), phi_ref)
        _check_sum(float(ws.pack[9]), g, u3, n, G, (2, 4), "fused trial g·u")
        _check_sum(float(ws.pack[10]), u3, u3, n, G, (2, 4), "fused trial u·u")
    finally:
        ws.close()


@pytest.mark.parametrize("G,n", X.SWEEP_EVEN)
def test_blas1_and_trial_vs_exact_even_n(ctx, G, n):
    """extended Rosenbrock (one fused kernel per trial, V = 2, U = 4)"""
    ctx.set_reduction_ctas(G)
    O.set_cgo_order(G, 1)
    obj = None
    try:
        obj = cg.RosenbrockGPU(n, ctx)
        oo = O.Objective.rosenbrock(n)
        oo.set_sum_mode("cgo")

        def phi_of(xp):
            f, gp = _rosen_numpy(xp)
            return (X.exact_sum(f), X.canonical_bound(n, G, (2, 4), X.exact_sum(np.abs(f))), oo.fdf(xp)[0]), gp

        _sweep_one(ctx, obj, G, n, obj.default_x0(24, 0.1), (2, 4), phi_of)
    finally:
        if obj is not None:
            obj.close()
        ctx.set_reduction_ctas(296)
        O.set_cgo_order(296, 1)


def _csr_phi_of(ora, rowptr, col, val, b, G, site):
    nrows = rowptr.size - 1

    def phi_of(xp):
        r = ora.spmv(xp) - b                              # the residual the kernels form (bit-exact SpMV)
        f, g = ora.fdf(xp)
        rr = X.exact_sumsq(r)
        return (0.5 * rr, 0.5 * X.canonical_bound(nrows, G, site, rr), f), g
    return phi_of


@pytest.mark.parametrize("G,n", X.SWEEP_ODD)
def test_blas1_and_trial_vs_exact_odd_n(ctx, G, n):
    """CSR least squares with an odd column count: the BLAS-1 ops' half-filled last double2 (v2 = false)"""
    ctx.set_reduction_ctas(G)
    O.set_cgo_order(G, 1)
    obj = None
    try:
        rowptr, col, val, b = _bidiagonal(n, n)
        obj = cg.SparseLSGPU_from_csr(n, n, rowptr, col, val, b, ctx)
        ora = O.Objective.sparse_ls_csr(n, n, rowptr, col, val, b)
        ora.set_trial_site(*obj.trial_site)
        ora.set_sum_mode("cgo")
        x0 = np.random.default_rng(n).uniform(-1.0, 1.0, n)
        _sweep_one(ctx, obj, G, n, x0, obj.trial_site, _csr_phi_of(ora, rowptr, col, val, b, G, obj.trial_site))
    finally:
        if obj is not None:
            obj.close()
        ctx.set_reduction_ctas(296)
        O.set_cgo_order(296, 1)


def _random_csr(nrows, ncols, per_row, seed):
    rng = np.random.default_rng(seed)
    rowptr = np.arange(0, nrows * per_row + 1, per_row, dtype=np.int64)
    col = rng.integers(0, ncols, nrows * per_row).astype(np.int32)
    col[::per_row] = np.arange(nrows) % ncols                  # every column gathered at least once
    return rowptr, col, rng.standard_normal(nrows * per_row), rng.standard_normal(nrows)


@pytest.mark.parametrize("flavour,linesearch,beta_form", [("LBFGS", "Wolfe", "fused"),
                                                          ("HagerZhang", "StrongWolfeBisection", "literal"),
                                                          ("HagerZhang", "YuanWeiLuWolfe", "fused")])
def test_whole_run_odd_n_matches_oracle(ctx, flavour, linesearch, beta_form):
    """odd n through a whole run: L-BFGS (LbfgsStage / LbfgsStep at v2 = false), literal β (BetaLiteral) and
    YuanWeiLuWolfe (its own acceptance test; ‖u + g‖², NormUPlusG, is checked by value in the sweep above)"""
    nrows, ncols = 4001, T + 1
    rowptr, col, val, b = _random_csr(nrows, ncols, 5, 9)
    obj = cg.SparseLSGPU_from_csr(nrows, ncols, rowptr, col, val, b, ctx)
    try:
        ora = O.Objective.sparse_ls_csr(nrows, ncols, rowptr, col, val, b)
        ora.set_trial_site(*obj.trial_site)
        ocfg, cfg, ls = make_pair(flavour, linesearch, max_iters=40, beta_form=beta_form)
        ret = cg.minimizeobjective(obj, np.zeros(ncols), cfg, ls, beta_form=beta_form)
    finally:
        obj.close()
    assert_same_run(ret, O.minimize(ora, np.zeros(ncols), ocfg), what=f"{flavour}/{linesearch}/{beta_form}")


# --------------------------------------------------------------------------------------------- L-BFGS
@pytest.mark.parametrize("n", [100, 101])
@pytest.mark.parametrize("m", [1, 3, 64])
def test_lbfgs_device_matches_dense_bfgs_with_rejections(ctx, m, n):
    """cgo_lbfgs_stage_pair / _commit_pair / _update_dir driven by hand, the ring wrapping (2m + 8 steps), rejected
    pairs (commit = 0) at count < m, at count == m and twice in a row: after every step u = −H g of the pairs the
    textbook keeps, H the dense inverse-BFGS matrix in extended precision, to 1e-10 relative.  At every rejection
    with a full history the textbook direction without the oldest pair is more than 1e-6 away, so a device history
    that lost that pair (or mis-indexed its ring) would fail."""
    rp, ci, va, b = X.well_conditioned_ls(n, 11 + n)
    obj = cg.SparseLSGPU_from_csr(n, n, rp, ci, va, b, ctx)
    ws = obj.make_workspace(np.zeros(n), lbfgs_m=m, fuse_direction=False)
    reject, steps = {1, m + 2, 2 * m + 4, 2 * m + 5}, 2 * m + 8
    try:
        errs, counts, power = X.drive_lbfgs(ws, m, steps, reject, a=0.05)
    finally:
        ws.close()
        obj.close()
    assert counts[-3:] == [m, m, m] and (m == 1 or counts[0] < m)
    assert len(power) >= 3 and min(power) > 1e-6, power
    bad = [(k, e) for k, e in enumerate(errs) if not e <= 1e-10]
    assert not bad, f"steps where u != −H g (step, rel. error): {bad[:6]}"


def test_lbfgs_natural_rejection_at_full_history_matches_oracle(ctx):
    """a whole run in which getβ rejects a pair with the one-pair history full (helpers.natural_lbfgs_rejection_case):
    the device history must follow the oracle's bit for bit through and after the rejection"""
    ocfg, cfg, ls, x0 = natural_lbfgs_rejection_case()
    obj = cg.RosenbrockChainedGPU(2, ctx)
    try:
        ret = cg.minimizeobjective(obj, x0, cfg, ls)
    finally:
        obj.close()
    assert_same_run(ret, O.minimize(O.Objective.rosenbrock_chained(2), x0, ocfg), what="natural rejection, LBFGS(1)")


# --------------------------------------------------------------------------------------------- CSR ring
def _ts_layout(nops=0, budget=115200, nd=3, lanes=256, maxk=12, nw=8):
    """RING and CHMAX of TsLayout<NOPS> (csr.cu): the ring of k_csr_rows holds RING entries, a tile longer than
    CHMAX entries streams in CHMAX chunks, TS_ND = nd descriptors"""
    desc = (lanes + 2) * 8 + nops * lanes * 8
    tail = 2 * nd * 8 + nd * 4 + maxk * nw * 8
    ring = ((budget - nd * desc - tail - 64) // 12) & ~3
    return ring, (ring // 2) & ~3


RING, CHMAX = _ts_layout()


def _csr_from_lens(lens, ncols, seed, force_col=None):
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, dtype=np.int64)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, ncols, int(rowptr[-1])).astype(np.int32)
    if force_col is not None:
        col[rowptr[:-1][lens > 0]] = force_col
    return rowptr, col, rng.standard_normal(int(rowptr[-1])), rng.standard_normal(lens.size)


def _ring_cases():
    long_row = 50_000                                              # > TS_ND·CHMAX in one tile
    lens_f = np.full(512, 3)
    lens_f[250], lens_f[251:256] = 20_000, 0                       # empty tile tail after a long row
    return {
        "one_row_50000": ([long_row], 50_001, None),
        "tile_256x60": ([60] * 256, 999, None),                    # row boundaries inside the chunks
        "tile_over_ring": ([RING // 256 + 4] * 256 + [2] * 256, 4097, None),
        "nnz_0": ([0] * 300, 301, None),
        "one_column_every_row": ([4] * 3000, 7, 3),
        "empty_rows_after_long_row": (lens_f, 3001, None),
    }


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("case", list(_ring_cases()))
def test_csr_ring_and_chunk_extremes_vs_exact(mode, case):
    """k_csr_rows (mode 1) and k_spmv_direct (mode 2) at the extremes of the ring: SpMV and SpMVᵀ bit-exact
    against the oracle and within γ_len·Σ|a_ij x_j| of the exact row sums; f and g at x within the canonical bound
    of ½ Σ r² and of the exact Aᵀr; a second evaluation identical bit for bit."""
    assert CHMAX * 3 < 50_000 and 60 * 256 > CHMAX and (RING // 256 + 4) * 256 > RING
    lens, ncols, force_col = _ring_cases()[case]
    rowptr, col, val, b = _csr_from_lens(lens, ncols, 17, force_col)
    nrows = rowptr.size - 1
    c = cg.Context(0)
    c.set_csr_mode(mode)
    try:
        obj = cg.SparseLSGPU_from_csr(nrows, ncols, rowptr, col, val, b, c)
        ora = O.Objective.sparse_ls_csr(nrows, ncols, rowptr, col, val, b)
        ora.set_trial_site(*obj.trial_site)
        ora.set_sum_mode("cgo")
        rpT, ciT, vaT = ora.csr(True)
        rng = np.random.default_rng(3)
        x, yv = rng.standard_normal(ncols), rng.standard_normal(nrows)
        for A, v, t in (((rowptr, col, val), x, False), ((rpT, ciT, vaT), yv, True)):
            got = obj.spmv(v, transposed=t)
            assert np.array_equal(got, ora.spmv(v, transposed=t)), f"transposed={t}: differs from the oracle"
            assert np.array_equal(got, obj.spmv(v, transposed=t)), f"transposed={t}: not run-to-run identical"
            err = np.abs(got - X.exact_spmv_rows(*A, v))
            bound = X.exact_spmv_row_bound(*A, v)
            assert np.all(err <= bound), f"transposed={t}: rows {np.nonzero(err > bound)[0][:5]} outside the bound"
        r = obj.spmv(x) - b
        f_ora, g_ora = ora.fdf(x)
        for _ in range(2):
            ws = obj.make_workspace(x, fuse_direction=False)
            f, g = ws.f_x0, np.array(ws.download()[1])
            ws.close()
            assert f == f_ora and np.array_equal(g, g_ora)
        rr = X.exact_sumsq(r)
        _within(float(f), 0.5 * rr, 0.5 * X.canonical_bound(nrows, 296, obj.trial_site, rr), "f")
        err = np.abs(g - X.exact_spmv_rows(rpT, ciT, vaT, r))
        assert np.all(err <= X.exact_spmv_row_bound(rpT, ciT, vaT, r)), "g outside the row bound"
        obj.close()
    finally:
        c.close()
