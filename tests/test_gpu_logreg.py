"""GPU parity tests of the CSR logistic-regression objective (BASELINE.json configs[3], L-BFGS).
The generator, CSR, transpose and all IEEE arithmetic are bit-exact against the oracle; the loss
uses exp / log1p, whose CUDA and glibc implementations may differ in the last ulp, so f and g are
compared at 1e-13 relative and whole L-BFGS traces at north_star's 1e-10."""
import numpy as np
import pytest

import cgoptim_b200 as cg
from oracle import oracle as O

from helpers import make_pair

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = cg.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("N,d,K", [(3000, 500, 20), (10_000, 4000, 7), (257, 64, 4)])
def test_generator_labels_transpose_bit_exact(ctx, N, d, K):
    obj = cg.LogRegGPU(N, d, K, 24, 1e-4, ctx)
    ora = O.Objective.logreg(N, d, K, 24, 1e-4)
    rp, ci, va, y = obj.csr(False)
    orp, oci, ova = ora.csr(False)
    assert np.array_equal(rp, orp) and np.array_equal(ci, oci) and np.array_equal(va, ova)
    assert np.array_equal(y, ora.rhs()) and set(np.unique(y)) <= {-1.0, 1.0}
    rpT, ciT, vaT, _ = obj.csr(True)
    orpT, ociT, ovaT = ora.csr(True)
    assert np.array_equal(rpT, orpT) and np.array_equal(ciT, ociT) and np.array_equal(vaT, ovaT)
    x = np.random.default_rng(0).standard_normal(d)
    assert np.array_equal(obj.spmv(x), ora.spmv(x))                 # margins: IEEE only, bit-exact
    obj.close()


@pytest.mark.parametrize("N,d,K", [(3000, 500, 20), (20_000, 3000, 20)])
def test_f_and_g_match_oracle(ctx, N, d, K):
    lam = 1e-4
    obj = cg.LogRegGPU(N, d, K, 24, lam, ctx)
    ora = O.Objective.logreg(N, d, K, 24, lam)
    ora.set_trial_site(*obj.trial_site)
    ora.set_sum_mode("cgo")
    rng = np.random.default_rng(1)
    for scale in (0.0, 0.1, 3.0, 40.0):                             # incl. saturated sigmoids
        w = scale * rng.standard_normal(d)
        ws = obj.make_workspace(w, fuse_direction=False)
        f, g = ora.fdf(w)
        assert abs(ws.f_x0 - f) <= 1e-13 * max(abs(f), 1e-300)
        gd = ws.download()[1]
        assert np.max(np.abs(gd - g)) <= 1e-13 * np.max(np.abs(g))
        ws.close()
    obj.close()


def test_gradient_matches_finite_differences(ctx):
    N, d = 2000, 60
    obj = cg.LogRegGPU(N, d, 6, 5, 1e-3, ctx)
    w = 0.3 * np.random.default_rng(2).standard_normal(d)
    ws = obj.make_workspace(w, fuse_direction=False)
    g = ws.download()[1]
    ws.close()
    h = 1e-5
    for i in (0, 7, 59):
        e = np.zeros(d); e[i] = h
        a = obj.make_workspace(w + e, fuse_direction=False); fp = a.f_x0; a.close()
        b = obj.make_workspace(w - e, fuse_direction=False); fm = b.f_x0; b.close()
        assert abs((fp - fm) / (2 * h) - g[i]) <= 1e-7 * max(1.0, abs(g[i]))
    obj.close()


@pytest.mark.parametrize("flavour", ["LBFGS", "HagerZhang"])
def test_lbfgs_run_matches_oracle(ctx, flavour):
    """cfg 4 shape at test size: L-BFGS m = 10, StrongWolfe(c1 = 1e-4, c2 = 0.9), w0 = 0."""
    N, d, lam = 20_000, 2000, 1e-4
    ocfg, cfg, ls = make_pair(flavour, "StrongWolfeBisection", eps=1e-6, max_iters=60, c1=1e-4, c2=0.9, lbfgs_m=10)
    obj = cg.LogRegGPU(N, d, 20, 24, lam, ctx)
    ora = O.minimize(O.Objective.logreg(N, d, 20, 24, lam), np.zeros(d), ocfg)
    ret = cg.minimizeobjective(obj, np.zeros(d), cfg, ls)
    k = min(50, len(ora.trace_objective), len(ret.trace.objective))
    assert k >= 10
    assert np.array_equal(ret.trace.step_size[:k], ora.trace_step_size[:k])          # identical decisions
    assert np.array_equal(ret.trace.objective_evals[:k], ora.trace_objective_evals[:k])
    np.testing.assert_allclose(ret.trace.objective[:k], ora.trace_objective[:k], rtol=1e-10)
    np.testing.assert_allclose(ret.trace.grad_norm[:k], ora.trace_grad_norm[:k], rtol=1e-8)
    assert ret.status == ora.status and abs(ret.iters_ran - ora.iters_ran) <= 2
    assert abs(ret.objective - ora.objective) <= 1e-8 * abs(ora.objective)
    assert ret.trace.objective[k - 1] < 0.9 * ret.trace.objective[0]
    obj.close()


def test_run_to_run_reproducible(ctx):
    N, d = 50_000, 5000
    _, cfg, ls = make_pair("LBFGS", max_iters=15, c1=1e-4, c2=0.9)
    obj = cg.LogRegGPU(N, d, 20, 24, 1e-6, ctx)
    a = cg.minimizeobjective(obj, np.zeros(d), cfg, ls)
    b = cg.minimizeobjective(obj, np.zeros(d), cfg, ls)
    assert np.array_equal(a.trace.objective, b.trace.objective) and np.array_equal(a.minimizer, b.minimizer)
    obj.close()


@pytest.mark.parametrize("block_elems", [700, 64, 2999])
def test_column_blocked_passes_are_bit_identical(block_elems):
    """Large random gathers are evaluated one L2-sized column block per pass (csr.cu CsrBlocked);
    passes chain the row sums, so f, g and whole runs must not change by a single bit."""
    N, d, lam = 20_000, 3000, 1e-4
    c0, c1, c2, c3 = cg.Context(0), cg.Context(0), cg.Context(0), cg.Context(0)
    c0.set_gather_block_bytes(0)
    c0.set_csr_mode(2)                       # single pass through k_spmv_direct: same kernels, same order of the dots
    c1.set_gather_block_bytes(8 * block_elems)
    c2.set_gather_block_bytes(0)             # single pass through the fused k_csr_rows (dots in the row-per-lane order)
    c3.set_gather_block_bytes(8 * block_elems)
    c3.set_csr_mode(1)                       # forced k_csr_rows: column blocks apply to k_spmv_direct only
    a, b = cg.LogRegGPU(N, d, 20, 24, lam, c0), cg.LogRegGPU(N, d, 20, 24, lam, c1)
    f, h = cg.LogRegGPU(N, d, 20, 24, lam, c2), cg.LogRegGPU(N, d, 20, 24, lam, c3)
    assert a.csr_blocks(False) == 1 and a.csr_blocks(True) == 1
    assert b.csr_blocks(False) == -(-d // block_elems) and b.csr_blocks(True) == -(-N // block_elems)
    assert h.csr_blocks(False) == 1 and h.csr_blocks(True) == 1
    assert a.trial_site == b.trial_site == (2, 4) and f.trial_site == h.trial_site == (1, 1)
    w = 0.5 * np.random.default_rng(3).standard_normal(d)
    wa, wb = a.make_workspace(w, fuse_direction=False), b.make_workspace(w, fuse_direction=False)
    wf, wh = f.make_workspace(w, fuse_direction=False), h.make_workspace(w, fuse_direction=False)
    assert wa.f_x0 == wb.f_x0 and np.array_equal(wa.pack, wb.pack)
    assert np.array_equal(wa.download()[1], wb.download()[1])
    assert wh.f_x0 == wf.f_x0 and np.array_equal(wh.pack, wf.pack)
    assert np.array_equal(wh.download()[1], wf.download()[1])
    assert np.array_equal(wa.download()[1], wf.download()[1])          # the gradient does not depend on the kernel family
    assert abs(wf.f_x0 - wa.f_x0) <= 1e-14 * abs(wa.f_x0)              # the loss only through the order of its sum
    wa.close(); wb.close(); wf.close(); wh.close(); f.close(); h.close(); c2.close(); c3.close()
    _, cfg, ls = make_pair("LBFGS", max_iters=25, c1=1e-4, c2=0.9)
    ra = cg.minimizeobjective(a, np.zeros(d), cfg, ls)
    rb = cg.minimizeobjective(b, np.zeros(d), cfg, ls)
    assert ra.status == rb.status and np.array_equal(ra.trace.objective, rb.trace.objective)
    assert np.array_equal(ra.trace.step_size, rb.trace.step_size) and np.array_equal(ra.minimizer, rb.minimizer)
    a.close(); b.close(); c0.close(); c1.close()


def test_full_size_properties_cfg4():
    """BASELINE.json configs[3] at its full size (5e7 samples × 2e7 features, 1e9 nonzeros, column-blocked
    storage), through properties that need no oracle run: f(0) = log 2 (every sample contributes
    log1p(e⁰)); the column-blocked passes are in use; L-BFGS decreases f monotonically; two runs are
    bit-identical."""
    import torch
    if torch.cuda.get_device_properties(0).total_memory < 100e9:
        pytest.skip("needs a 180 GB B200")
    c = cg.Context(0)
    N, d = 50_000_000, 20_000_000
    obj = cg.LogRegGPU(N, d, 20, 24, 1e-6, c)
    assert obj.csr_blocks(False) == 4 and obj.csr_blocks(True) == 10
    _, cfg, ls = make_pair("LBFGS", max_iters=3, c1=1e-4, c2=0.9, lbfgs_m=10)
    w0 = np.zeros(d)
    r1 = cg.minimizeobjective(obj, w0, cfg, ls)
    r2 = cg.minimizeobjective(obj, w0, cfg, ls)
    ws = obj.make_workspace(w0, fuse_direction=False)
    assert abs(ws.f_x0 - np.log(2.0)) <= 1e-12
    ws.close()
    assert r1.trace.objective[0] < np.log(2.0) and np.all(np.diff(r1.trace.objective) < 0)
    assert np.array_equal(r1.trace.objective, r2.trace.objective) and np.array_equal(r1.minimizer, r2.minimizer)
    obj.close(); c.close()
