"""GPU tests of per-sample weights and the unpenalised intercept of logistic and softmax regression on the caller's
CSR (LogRegGPU_from_csr / SoftmaxRegGPU_from_csr with sample_weight and fit_intercept): the transposed hook (Aᵀc and
the unit row) bit for bit against tests/glm_csr_reference.py and f, g to 1e-13 (the device's exp, log and log1p are
not the C library's, so a loss term or c may differ in its last bit, as for the objectives without the options);
bit for bit between device objectives: the old constructors against the new entry points with neither option,
all-ones weights against none, the intercept against an explicit ones column; whole runs, the launches of a trial
and rejected input."""
import ctypes as C

import numpy as np
import pytest

import cgoptim_b200 as cg
from cgoptim_b200._capi import check, lib
from cgoptim_b200.device import DeviceObjective
from oracle import oracle as O

from glm_csr_reference import LogRegGlmCSR, SoftmaxGlmCSR
from helpers import make_pair
from logreg_csr_reference import L
from numpy_workspace import NumpyObjective
from test_gpu_csr_paths import _measure
from test_gpu_softmax_csr import edge_data

pytestmark = pytest.mark.gpu


def _ctx(G=296, block_bytes=None, mode=None):
    c = cg.Context(0)
    c.timing(True)
    c.set_reduction_ctas(G)
    if block_bytes is not None:
        c.set_gather_block_bytes(block_bytes)
    if mode is not None:
        c.set_csr_mode(mode)
    return c


def data(K, N, d=51, seed=1, popular=False):
    """edge_data without its ones column: ragged, empty, unsorted and duplicate entries, rows of L and L + 1
    entries.  popular: feature d − 1 in every row with a random value (a long row of Aᵀ when N > L).  K = 1: binary
    labels ±1"""
    rowptr, col, val, y = edge_data(N, d, max(K, 2), seed, intercept=popular)
    if popular:
        val[col == d - 1] = np.random.default_rng(seed + 100).uniform(-1.0, 1.0, int(np.sum(col == d - 1)))
    return rowptr, col, val, (np.where(y == 1, 1.0, -1.0) if K == 1 else y)


def gpu(K, N, d, rowptr, col, val, y, lam, ctx, s=None, icpt=False):
    if K == 1:
        return cg.LogRegGPU_from_csr(N, d, rowptr, col, val, y, lam, ctx, sample_weight=s, fit_intercept=icpt)
    return cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, lam, ctx, sample_weight=s, fit_intercept=icpt)


def ref(K, N, d, rowptr, col, val, y, lam, s=None, icpt=False):
    if K == 1:
        r = LogRegGlmCSR(N, d, rowptr, col, val, y, lam, sample_weight=s, fit_intercept=icpt)
    else:
        r = SoftmaxGlmCSR(N, d, K, rowptr, col, val, y, lam, sample_weight=s, fit_intercept=icpt)
    r.set_sum_mode("cgo")
    return r


def fg(obj, x):
    ws = obj.make_workspace(x, fuse_direction=False)
    f, g = ws.f_x0, ws.download()[1]
    ws.close()
    return f, g


@pytest.mark.parametrize("popular", [False, True])
@pytest.mark.parametrize("N", [L - 1, L + 1, 5000])
@pytest.mark.parametrize("K", [1, 2, 3, 8, 33])
def test_f_g_and_hook_against_reference(K, N, popular):
    d, lam = 51, 1e-3
    rowptr, col, val, y = data(K, N, popular=popular)
    s = np.random.default_rng(N).uniform(0.0, 3.0, N)
    s[::11] = 0.0
    r = ref(K, N, d, rowptr, col, val, y, lam, s, True)
    rng = np.random.default_rng(K)
    x = 0.3 * rng.standard_normal(r.n)
    c = rng.standard_normal(N * K)
    for G in (1, 3, 296):
        O.set_cgo_order(G=G)
        f, g = r.fdf(x)
        qr = r.spmv(c, True)
        for bb in (None, 8 * K * 20):                       # single pass; Aᵀ in blocks of 20 samples
            ctx = _ctx(G, bb)
            obj = gpu(K, N, d, rowptr, col, val, y, lam, ctx, s, True)
            assert obj.n_local == r.n and obj.trial_site == (2, 4)
            assert obj.csr_blocks(True) == (1 if bb is None else -(-N // 20))
            assert np.array_equal(obj.spmv(c, True), qr)
            assert np.array_equal(obj.spmv(x), r.spmv(x))
            fo, go = fg(obj, x)
            assert abs(fo - f) <= 1e-13 * abs(f)
            assert np.max(np.abs(go - g)) <= 1e-13 * np.max(np.abs(g))
            obj.close(); ctx.close()
    O.set_cgo_order(G=296)


def _old(K, N, d, rowptr, col, val, y, lam, ctx):
    """the constructors without the options, called directly"""
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.float64)
    h = C.c_void_p()
    if K == 1:
        y = np.ascontiguousarray(y, dtype=np.float64)
        check(lib().cgo_obj_logreg_create_csr(ctx.h, N, d, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data,
                                              y.ctypes.data, lam, C.byref(h)))
        return DeviceObjective(ctx, h)
    y = np.ascontiguousarray(y, dtype=np.int32)
    check(lib().cgo_obj_softmax_create_csr(ctx.h, N, d, K, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data,
                                           y.ctypes.data, lam, C.byref(h)))
    obj = DeviceObjective(ctx, h)
    obj.nclasses = K
    return obj


def _trial_record(obj, x0):
    """(launches of x0, trial and fused trial, f, g, the trial's pack and g⁺)"""
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


@pytest.mark.parametrize("case", ["logreg_csr_rows", "logreg_direct", "softmax"])
def test_no_options_equal_the_old_constructors(case):
    """with (None, False) the new entry points build the objective the old constructors build: kernel family, launches,
    f, g and whole runs"""
    if case == "logreg_csr_rows":                          # short rows, coalescing gathers: the fused k_csr_rows
        K, N, d = 1, 3000, 40
        rng = np.random.default_rng(3)
        rowptr = np.arange(N + 1, dtype=np.int64) * 6
        col = np.sort(rng.integers(0, d, (N, 6)), axis=1).ravel().astype(np.int32)
        val = rng.uniform(-1.0, 1.0, col.size)
        y = np.where(rng.random(N) < 0.5, -1.0, 1.0)
    else:
        K, N, d = (1 if case == "logreg_direct" else 5), 1500, 51
        rowptr, col, val, y = data(K, N)
    ctx = _ctx()
    old = _old(K, N, d, rowptr, col, val, y, 1e-4, ctx)
    new = gpu(K, N, d, rowptr, col, val, y, 1e-4, ctx)
    assert old.trial_site == new.trial_site == ((1, 1) if case == "logreg_csr_rows" else (2, 4))
    assert old.bytes_per_eval == new.bytes_per_eval and old.n_local == new.n_local == d * K
    x0 = 0.1 * np.random.default_rng(4).standard_normal(d * K)
    ro, rn = _trial_record(old, x0), _trial_record(new, x0)
    assert ro[0] == rn[0] and ro[1] == rn[1]
    for a, b in zip(ro[2:], rn[2:]):
        assert np.array_equal(a, b)
    _, cfg, ls = make_pair("LBFGS", max_iters=25, c1=1e-4, c2=0.9)
    ra = cg.minimizeobjective(old, np.zeros(d * K), cfg, ls)
    rb = cg.minimizeobjective(new, np.zeros(d * K), cfg, ls)
    assert np.array_equal(ra.trace.objective, rb.trace.objective) and np.array_equal(ra.trace.step_size, rb.trace.step_size)
    assert np.array_equal(ra.minimizer, rb.minimizer)
    old.close(); new.close(); ctx.close()


@pytest.mark.parametrize("K", [1, 4])
@pytest.mark.parametrize("icpt", [False, True])
def test_all_ones_weights_equal_no_weights(K, icpt):
    N, d = 3000, 51
    rowptr, col, val, y = data(K, N, popular=True)
    ctx = _ctx()
    a = gpu(K, N, d, rowptr, col, val, y, 1e-3, ctx, None, icpt)
    b = gpu(K, N, d, rowptr, col, val, y, 1e-3, ctx, np.ones(N), icpt)
    x = 0.4 * np.random.default_rng(5).standard_normal(a.n_local)
    fa, ga = fg(a, x)
    fb, gb = fg(b, x)
    assert fa == fb and np.array_equal(ga, gb)
    a.close(); b.close(); ctx.close()


def with_ones_column(N, d, rowptr, col, val):
    cnt = np.diff(rowptr) + 1
    rp1 = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    last = rp1[1:] - 1
    mask = np.ones(rp1[-1], dtype=bool)
    mask[last] = False
    ci1, va1 = np.empty(rp1[-1], dtype=np.int32), np.empty(rp1[-1])
    ci1[mask], va1[mask] = col, val
    ci1[last], va1[last] = d, 1.0
    return rp1, ci1, va1


@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("weighted", [False, True])
def test_intercept_equals_an_explicit_ones_column(K, weighted):
    """λ = 0, N > CGO_LONG_ROW and every row of A shorter than CGO_LONG_ROW: f, g and whole runs bit for bit"""
    N, d = 4000, 51
    rng = np.random.default_rng(6)
    lens = rng.integers(0, 9, N)
    lens[3] = L - 1
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, d, rowptr[-1]).astype(np.int32)
    val = rng.uniform(-1.0, 1.0, col.size)
    y = rng.integers(0, max(K, 2), N)
    y = np.where(y == 1, 1.0, -1.0) if K == 1 else y
    s = rng.uniform(0.2, 2.0, N) if weighted else None
    rp1, ci1, va1 = with_ones_column(N, d, rowptr, col, val)
    ctx = _ctx()
    a = gpu(K, N, d, rowptr, col, val, y, 0.0, ctx, s, True)
    b = gpu(K, N, d + 1, rp1, ci1, va1, y, 0.0, ctx, s, False)
    assert b.trial_site == (2, 4)
    x = 0.3 * rng.standard_normal(a.n_local)
    fa, ga = fg(a, x)
    fb, gb = fg(b, x)
    assert fa == fb and np.array_equal(ga, gb)
    _, cfg, ls = make_pair("LBFGS", max_iters=30, c1=1e-4, c2=0.9)
    ra = cg.minimizeobjective(a, np.zeros(a.n_local), cfg, ls)
    rb = cg.minimizeobjective(b, np.zeros(b.n_local), cfg, ls)
    assert np.array_equal(ra.trace.objective, rb.trace.objective) and np.array_equal(ra.minimizer, rb.minimizer)
    a.close(); b.close(); ctx.close()


@pytest.mark.parametrize("flavour", ["HagerZhang", "LBFGS"])
@pytest.mark.parametrize("K", [1, 4])
def test_runs_match_reference(flavour, K):
    N, d, lam = 1500, 51, 1e-3
    rowptr, col, val, y = data(K, N, seed=6, popular=True)
    s = np.random.default_rng(7).uniform(0.0, 2.0, N)
    ctx = _ctx()
    _, cfg, ls = make_pair(flavour, "StrongWolfeBisection", eps=1e-6, max_iters=60, c1=1e-4, c2=0.9, lbfgs_m=10)
    obj = gpu(K, N, d, rowptr, col, val, y, lam, ctx, s, True)
    r = ref(K, N, d, rowptr, col, val, y, lam, s, True)
    O.set_cgo_order(G=296)
    ora = cg.minimizeobjective(NumpyObjective(r), np.zeros(r.n), cfg, ls)
    ret = cg.minimizeobjective(obj, np.zeros(r.n), cfg, ls)
    k = min(50, len(ora.trace.objective), len(ret.trace.objective))
    assert k >= 10
    assert np.array_equal(ret.trace.step_size[:k], ora.trace.step_size[:k])
    assert np.array_equal(ret.trace.objective_evals[:k], ora.trace.objective_evals[:k])
    np.testing.assert_allclose(ret.trace.objective[:k], ora.trace.objective[:k], rtol=1e-10)
    # ‖g‖ falls by orders of magnitude: last-bit differences of c are relative to the first gradient's scale
    np.testing.assert_allclose(ret.trace.grad_norm[:k], ora.trace.grad_norm[:k], rtol=1e-8, atol=1e-9 * ora.trace.grad_norm[0])
    assert ret.status == ora.status and abs(ret.iters_ran - ora.iters_ran) <= 2
    assert abs(ret.objective - ora.objective) <= 1e-8 * abs(ora.objective)
    again = cg.minimizeobjective(obj, np.zeros(r.n), cfg, ls)
    assert np.array_equal(again.trace.objective, ret.trace.objective) and np.array_equal(again.minimizer, ret.minimizer)
    obj.close(); ctx.close()


@pytest.mark.parametrize("K", [1, 7])
def test_launches_site_and_bytes(K):
    """one trial: K_a with P, A and its long row (two kernels), the loss, Aᵀ and the unit row (two kernels), the
    combine pass.  Bytes: the matrices, 8N for the weights and 8NK for the intercept's read of c"""
    N, d = 1500, 51
    rowptr, col, val, y = data(K, N)
    s = np.random.default_rng(1).uniform(0.5, 1.5, N)
    out = {}
    for name, bb in (("single", None), ("blocked", 8 * K * 100)):
        ctx = _ctx(block_bytes=bb)
        obj = gpu(K, N, d, rowptr, col, val, y, 1e-4, ctx, s, True)
        ro = _trial_record(obj, 0.1 * np.random.default_rng(2).standard_normal(obj.n_local))
        ws = obj.make_workspace(np.zeros(obj.n_local))
        with pytest.raises(cg.CgoError):
            ws.hessvec_dir()
        ws.close()
        out[name] = (obj.trial_site, obj.bytes_per_eval, ro[0])
        obj.close(); ctx.close()
    one = ({"axpy": 1, "other": 2, "spmv": 3, "spmvT": 3}, 9)
    blk = ({"axpy": 1, "other": 2, "spmv": 3, "spmvT": 17}, 23)
    nbytes = {1: 269672.0, 7: 573128.0}[K]
    assert out["single"] == ((2, 4), nbytes, [one, one, one])
    assert out["blocked"] == ((2, 4), nbytes, [blk, blk, blk])


def _raw(K, N, d, rowptr, col, val, y, s, icpt, ctx):
    """the new entry points called directly (fit_intercept unchecked by Python)"""
    h = C.c_void_p()
    sp = None if s is None else np.ascontiguousarray(s, dtype=np.float64)
    sptr = None if sp is None else sp.ctypes.data
    if K == 1:
        yy = np.ascontiguousarray(y, dtype=np.float64)
        return lib().cgo_obj_logreg_create_csr_ex(ctx.h, N, d, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data,
                                                  yy.ctypes.data, sptr, icpt, 1e-4, C.byref(h)), h
    yy = np.ascontiguousarray(y, dtype=np.int32)
    return lib().cgo_obj_softmax_create_csr_ex(ctx.h, N, d, K, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data,
                                               yy.ctypes.data, sptr, icpt, 1e-4, C.byref(h)), h


@pytest.mark.parametrize("K", [1, 3])
def test_rejected_input(K):
    rp = np.array([0, 2, 3], dtype=np.int64)
    ci = np.array([0, 1, 2], dtype=np.int32)
    va = np.ones(3)
    y = np.array([1.0, -1.0]) if K == 1 else np.array([0, 2])
    ctx = _ctx()
    for s, icpt in ((None, True), (np.array([0.5, 2.0]), False), (np.array([0.0, 2.0]), True)):
        gpu(K, 2, 3, rp, ci, va, y, 1e-4, ctx, s, icpt).close()          # accepted as given

    def reject(s=None, icpt=True, c=ctx, d=3):
        with pytest.raises(cg.CgoError):
            gpu(K, 2, d, rp, ci, va, y, 1e-4, c, s, icpt)
    for bad in (-1.0, float("nan"), float("inf"), -0.5e-300):
        reject(np.array([1.0, bad]))
        reject(np.array([bad, 1.0]), icpt=False)
    reject(np.zeros(2))                                                     # S = 0
    reject(np.array([1.5e308, 1.5e308]))                                    # S overflows
    reject(np.ones(3))                                                      # Python: wrong size
    reject(icpt=2)
    reject(d=(1 << 31) - 2)                                                 # nfeat + 1 overflows int32
    for icpt in (2, -1):
        rc, _ = _raw(K, 2, 3, rp, ci, va, y, None, icpt, ctx)
        assert rc != 0 and "fit_intercept" in lib().cgo_last_error().decode()
    rc, _ = _raw(K, 2, 3, rp, ci, va, y, np.array([1.0, -1.0]), 0, ctx)
    assert rc != 0 and "sample 1" in lib().cgo_last_error().decode()
    m1 = _ctx(mode=1)
    reject(np.ones(2), icpt=False, c=m1)
    reject(None, icpt=True, c=m1)
    if K == 1:
        gpu(K, 2, 3, rp, ci, va, y, 1e-4, m1).close()                        # mode 1 without the options
    m1.close(); ctx.close()
