"""GPU tests of logistic regression on the caller's CSR (LogRegGPU_from_csr): the same objective as the synthetic
constructor on the same matrix, ragged user data with an intercept column and long rows against the oracle, the
launches the long rows add, whole runs, rejected input and a production-size check."""
import math

import numpy as np
import pytest

import cgoptim_b200 as cg
from oracle import oracle as O

import exact_reference as X
from helpers import make_pair
from logreg_csr_reference import L, LogRegCSR
from numpy_workspace import NumpyObjective
from test_gpu_csr_paths import _measure

pytestmark = pytest.mark.gpu

CONTEXTS = ["default", "blocked", "mode1", "mode2"]


def _ctx(name):
    c = cg.Context(0)
    c.timing(True)
    if name == "blocked":
        c.set_gather_block_bytes(8 * 700)
    elif name == "mode1":
        c.set_csr_mode(1)
    elif name == "mode2":
        c.set_csr_mode(2)
    return c


def _eval(obj, x0):
    """(launch counts of x0, trial and fused trial, f(x0), g(x0), the trial's pack and g⁺)"""
    box = {}
    counts = [_measure(obj.ctx, lambda: box.setdefault("ws", obj.make_workspace(x0, fuse_direction=True)))]
    ws = box["ws"]
    f0, g0 = ws.f_x0, ws.download()[1]
    ws.reset_direction()
    counts.append(_measure(obj.ctx, lambda: ws.eval_trial(1e-3)))
    pack, gp = np.array(ws.pack, copy=True), ws.download_vector("df_xp")
    ws.accept()

    def fused():
        ws.update_dir(0.3)
        ws.hint_first_trial(1e-3)
        ws.eval_trial(1e-3)
    counts.append(_measure(obj.ctx, fused))
    ws.close()
    return counts, f0, g0, pack, gp


@pytest.mark.parametrize("ctxname", CONTEXTS)
@pytest.mark.parametrize("N,d,K", [(3000, 500, 20), (20000, 3000, 20), (257, 64, 4)])
def test_same_matrix_two_constructors(ctxname, N, d, K):
    ctx = _ctx(ctxname)
    lam = 1e-4
    syn = cg.LogRegGPU(N, d, K, 24, lam, ctx)
    rp, ci, va, y = syn.csr(False)
    usr = cg.LogRegGPU_from_csr(N, d, rp, ci, va, y, lam, ctx)
    assert syn.trial_site == usr.trial_site
    assert syn.bytes_per_eval == usr.bytes_per_eval
    for t in (False, True):
        assert syn.csr_blocks(t) == usr.csr_blocks(t)
        for a, b in zip(syn.csr(t), usr.csr(t)):
            assert np.array_equal(a, b)
    rng = np.random.default_rng(1)
    x, c = rng.standard_normal(d), rng.standard_normal(N)
    assert np.array_equal(syn.spmv(x), usr.spmv(x)) and np.array_equal(syn.spmv(c, True), usr.spmv(c, True))
    x0 = 0.1 * rng.standard_normal(d)
    es, eu = _eval(syn, x0), _eval(usr, x0)
    assert es[0] == eu[0]                                             # launches by class, x0 / trial / fused trial
    assert es[1] == eu[1] and np.array_equal(es[2], eu[2])
    assert np.array_equal(es[3], eu[3]) and np.array_equal(es[4], eu[4])       # the trial's pack and g⁺
    _, cfg, ls = make_pair("LBFGS", max_iters=25, c1=1e-4, c2=0.9)
    ra = cg.minimizeobjective(syn, np.zeros(d), cfg, ls)
    rb = cg.minimizeobjective(usr, np.zeros(d), cfg, ls)
    assert np.array_equal(ra.trace.objective, rb.trace.objective) and np.array_equal(ra.trace.step_size, rb.trace.step_size)
    assert np.array_equal(ra.minimizer, rb.minimizer)
    syn.close(); usr.close(); ctx.close()


def ragged_intercept_data(seed=3, N=6000, d=301):
    """empty rows and columns, unsorted and duplicate columns, a ones column (the intercept, last feature), a
    sample row longer than L and rows of exactly L and L + 1 entries"""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(N):
        k = int(rng.integers(0, 9)) if i % 97 else 0
        r = list(rng.integers(0, d - 11, k))                   # features d−11 .. d−2 stay empty
        if k > 2:
            r.append(r[0])                                     # a duplicate
        rows.append(r + [d - 1])                               # intercept, after the others
    rows[5] = list(rng.integers(0, d - 11, L))
    rows[6] = list(rng.integers(0, d - 11, L + 1))
    rows[7] = list(rng.integers(0, d - 11, 3 * L + 17))
    rows[8] = []                                               # a sample without features
    rowptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col = np.concatenate([np.asarray(r, dtype=np.int64) for r in rows]).astype(np.int32)
    val = rng.uniform(-1.0, 1.0, col.size)
    val[col == d - 1] = 1.0
    y = np.where(rng.random(N) < 0.4, -1.0, 1.0)
    return N, d, rowptr, col, val, y


@pytest.mark.parametrize("ctxname", CONTEXTS)
@pytest.mark.parametrize("shape", [(6000, 301), (23, 9)])
def test_ragged_user_data_against_oracle(ctxname, shape):
    N, d = shape
    if N < 32:                                                 # N < 32, odd nfeat, no long rows
        rng = np.random.default_rng(4)
        lens = rng.integers(0, 5, N)
        rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        col = rng.integers(0, d, int(rowptr[-1])).astype(np.int32)
        val = rng.uniform(-1, 1, col.size)
        y = np.where(rng.random(N) < 0.5, -1.0, 1.0)
    else:
        N, d, rowptr, col, val, y = ragged_intercept_data(N=N, d=d)
    ctx = _ctx(ctxname)
    lam = 1e-4
    obj = cg.LogRegGPU_from_csr(N, d, rowptr, col, val, y, lam, ctx)
    ora = LogRegCSR(N, d, rowptr, col, val, y, lam)
    ora.set_trial_site(*obj.trial_site)
    ora.set_sum_mode("cgo")
    O.set_cgo_order(G=296)
    for t in (False, True):
        rp, ci, va, yy = obj.csr(t)
        orp, oci, ova = ora.csr(t)
        assert np.array_equal(rp, orp) and np.array_equal(ci, oci) and np.array_equal(va, ova)
    assert np.array_equal(yy, y)
    assert obj.csr_blocks(False) == 1                          # unsorted rows: A stays single-pass
    rng = np.random.default_rng(5)
    x = rng.standard_normal(d)
    assert np.array_equal(obj.spmv(x), ora.spmv(x))            # margins (long rows included)
    c = rng.standard_normal(N)
    assert np.array_equal(obj.spmv(c, True), ora.spmv(c, True))
    lens = np.diff(rowptr)
    for scale in (0.0, 0.1, 3.0, 40.0):
        w = scale * rng.standard_normal(d)
        ws = obj.make_workspace(w, fuse_direction=False)
        f, g = ora.fdf(w)
        assert abs(ws.f_x0 - f) <= 1e-13 * max(abs(f), 1e-300)
        gd = ws.download()[1]
        assert np.max(np.abs(gd - g)) <= 1e-13 * max(np.max(np.abs(g)), 1e-300)
        ws.close()
    if N > L and ctxname != "mode1":
        # the intercept's gradient entry: a row of Aᵀ with N entries, summed in the canonical order
        cvec = rng.uniform(-1, 1, N)
        gT = obj.spmv(cvec, True)
        rpT, ciT, vaT, _ = obj.csr(True)
        j = d - 1
        terms = vaT[rpT[j]:rpT[j + 1]] * cvec[ciT[rpT[j]:rpT[j + 1]]]
        assert terms.size > L
        exact = X.exact_dot(vaT[rpT[j]:rpT[j + 1]], cvec[ciT[rpT[j]:rpT[j + 1]]])
        assert abs(gT[j] - exact) <= X.canonical_bound(terms.size, 296, (1, 4), float(np.abs(terms).sum()))
        assert (lens > L).sum() == 2
    obj.close(); ctx.close()


@pytest.mark.parametrize("ctxname", ["default", "mode2", "mode1"])
def test_long_rows_add_two_launches_per_matrix(ctxname):
    ctx = _ctx(ctxname)
    N, d, rowptr, col, val, y = ragged_intercept_data()
    with_long = cg.LogRegGPU_from_csr(N, d, rowptr, col, val, y, 1e-4, ctx)
    keep = np.ones(N, dtype=bool)
    keep[[6, 7]] = False                                       # no sample row longer than L
    rows = [col[rowptr[i]:rowptr[i + 1]] for i in range(N) if keep[i]]
    vals = [val[rowptr[i]:rowptr[i + 1]] for i in range(N) if keep[i]]
    rp2 = np.concatenate([[0], np.cumsum([r.size for r in rows])]).astype(np.int64)
    only_t = cg.LogRegGPU_from_csr(int(keep.sum()), d, rp2, np.concatenate(rows), np.concatenate(vals), y[keep], 1e-4, ctx)
    rp3 = np.arange(N + 1, dtype=np.int64) * 2                  # short rows everywhere: two features each
    c3 = np.stack([np.arange(N) % (d - 1), np.full(N, d - 1)], 1).ravel().astype(np.int32)
    c3[1::2] = (np.arange(N) * 7) % (d - 1)
    short = cg.LogRegGPU_from_csr(N, d, rp3, c3, np.ones(2 * N), y, 1e-4, ctx)
    x0 = np.zeros(d)
    counts = {k: _eval(o, x0)[0][1] for k, o in (("long", with_long), ("only_t", only_t), ("short", short))}
    ctx.set_csr_mode(2)
    ref = cg.LogRegGPU_from_csr(N, d, rp3, c3, np.ones(2 * N), y, 1e-4, ctx)
    base = _eval(ref, x0)[0][1]                                # k_spmv_direct without long rows
    if ctxname == "mode1":
        for k in counts:
            assert counts[k] == ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3)
    else:
        bc, bl = base
        assert counts["long"] == ({**bc, "spmv": bc["spmv"] + 2, "spmvT": bc["spmvT"] + 2}, bl + 4)
        assert counts["only_t"] == ({**bc, "spmvT": bc["spmvT"] + 2}, bl + 2)
        if ctxname == "default":
            assert counts["short"] == ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3)
    for o in (with_long, only_t, short, ref):
        o.close()
    ctx.close()


@pytest.mark.parametrize("flavour,ctxname", [("LBFGS", "default"), ("HagerZhang", "default"), ("LBFGS", "mode1")])
def test_runs_match_oracle_and_repeat(flavour, ctxname):
    N, d, rowptr, col, val, y = ragged_intercept_data()
    lam = 1e-4
    ctx = _ctx(ctxname)
    _, cfg, ls = make_pair(flavour, "StrongWolfeBisection", eps=1e-6, max_iters=60, c1=1e-4, c2=0.9, lbfgs_m=10)
    obj = cg.LogRegGPU_from_csr(N, d, rowptr, col, val, y, lam, ctx)
    ref = LogRegCSR(N, d, rowptr, col, val, y, lam)
    ref.set_trial_site(*obj.trial_site)
    O.set_cgo_order(G=296)
    ora = cg.minimizeobjective(NumpyObjective(ref), np.zeros(d), cfg, ls)     # the host mirror on the reference
    ret = cg.minimizeobjective(obj, np.zeros(d), cfg, ls)
    k = min(50, len(ora.trace.objective), len(ret.trace.objective))
    assert k >= 10
    assert np.array_equal(ret.trace.step_size[:k], ora.trace.step_size[:k])
    assert np.array_equal(ret.trace.objective_evals[:k], ora.trace.objective_evals[:k])
    np.testing.assert_allclose(ret.trace.objective[:k], ora.trace.objective[:k], rtol=1e-10)
    np.testing.assert_allclose(ret.trace.grad_norm[:k], ora.trace.grad_norm[:k], rtol=1e-8)
    assert ret.status == ora.status and abs(ret.iters_ran - ora.iters_ran) <= 2
    assert abs(ret.objective - ora.objective) <= 1e-8 * abs(ora.objective)
    ws = obj.make_workspace(np.zeros(d))
    assert ws.f_x0 == pytest.approx(math.log(2.0), rel=1e-12)                # f(0) = log 2 for any data
    ws.close()
    again = cg.minimizeobjective(obj, np.zeros(d), cfg, ls)
    assert np.array_equal(again.trace.objective, ret.trace.objective) and np.array_equal(again.minimizer, ret.minimizer)
    obj.close(); ctx.close()


def _reject(*args, lam=1e-4):
    with pytest.raises(cg.CgoError):
        cg.LogRegGPU_from_csr(*args, lam=lam)


def test_rejected_input():
    rp = np.array([0, 2, 3], dtype=np.int64)
    ci = np.array([0, 1, 2], dtype=np.int32)
    va = np.ones(3)
    y = np.array([1.0, -1.0])
    obj = cg.LogRegGPU_from_csr(2, 3, rp, ci, va, y)            # accepted as given
    obj.close()
    _reject(0, 3, np.zeros(1, np.int64), ci[:0], va[:0], y[:0])
    _reject(2, 0, rp, ci, va, y)
    _reject(2, 1 << 31, rp, ci, va, y)
    _reject(2, 3, np.array([1, 2, 3], dtype=np.int64), ci, va, y)
    _reject(2, 3, np.array([0, 3, 2], dtype=np.int64), ci, va, y)
    _reject(2, 3, rp, np.array([0, 1, 3], dtype=np.int32), va, y)
    _reject(2, 3, rp, np.array([0, -1, 2], dtype=np.int32), va, y)
    for bad in (0.0, 2.0, float("nan")):
        _reject(2, 3, rp, ci, va, np.array([1.0, bad]))
    for lam in (-1e-3, float("inf"), float("nan")):
        _reject(2, 3, rp, ci, va, y, lam=lam)


def test_production_size_matches_synthetic():
    import torch
    if torch.cuda.get_device_properties(0).total_memory < 100e9:
        pytest.skip("needs a GPU with 100 GB")
    N = d = 10_000_000
    ctx = cg.Context(0)
    syn = cg.LogRegGPU(N, d, 20, 24, 1e-6, ctx)
    ctx.set_gather_block_bytes(0)
    flat = cg.LogRegGPU(N, d, 20, 24, 1e-6, ctx)                 # keeps the single-pass copy for download
    ctx.set_gather_block_bytes(40 << 20)
    rp, ci, va, y = flat.csr(False)
    flat.close()
    usr = cg.LogRegGPU_from_csr(N, d, rp, ci, va, y, 1e-6, ctx)
    _, cfg, ls = make_pair("LBFGS", max_iters=3, c1=1e-4, c2=0.9)
    ra = cg.minimizeobjective(syn, np.zeros(d), cfg, ls)
    rb = cg.minimizeobjective(usr, np.zeros(d), cfg, ls)
    assert np.array_equal(ra.trace.objective, rb.trace.objective) and np.array_equal(ra.minimizer, rb.minimizer)
    assert np.array_equal(ra.gradient, rb.gradient)
    syn.close(); usr.close()
    # the same matrix with a ones column appended (the intercept): f(0) = log 2 and f decreases
    cnt = np.diff(rp) + 1
    rp1 = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    ci1 = np.empty(rp1[-1], dtype=np.int32)
    va1 = np.empty(rp1[-1])
    last = rp1[1:] - 1
    mask = np.ones(rp1[-1], dtype=bool)
    mask[last] = False
    ci1[mask], va1[mask] = ci, va
    ci1[last], va1[last] = d, 1.0
    del ci, va
    one = cg.LogRegGPU_from_csr(N, d + 1, rp1, ci1, va1, y, 1e-6, ctx)
    ws = one.make_workspace(np.zeros(d + 1))
    f0 = ws.f_x0
    ws.close()
    assert f0 == pytest.approx(math.log(2.0), rel=1e-12)
    r1 = cg.minimizeobjective(one, np.zeros(d + 1), cfg, ls)
    f = np.concatenate([[f0], r1.trace.objective])
    assert np.all(np.diff(f) < 0)
    one.close(); ctx.close()
