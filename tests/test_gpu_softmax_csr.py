"""GPU tests of softmax regression on the caller's CSR (SoftmaxRegGPU_from_csr): the K-column SpMM bit for bit against
the SpMV of the Kronecker-expanded matrix (reference and k_spmv_direct), column blocks, f and g, K = 2 against
binary logistic regression, whole runs, the launches of a trial, rejected input and a size where blocks engage."""
import numpy as np
import pytest

import cgoptim_b200 as cg
from oracle import oracle as O

from helpers import make_pair
from logreg_csr_reference import L
from numpy_workspace import NumpyObjective
from softmax_csr_reference import SoftmaxCSR, kron_csr
from test_gpu_csr_paths import _measure

pytestmark = pytest.mark.gpu


def edge_data(N, d, K, seed=1, intercept=True):
    """ragged rows with empty ones, unsorted and duplicate columns, rows of exactly L and L + 1 entries and an
    intercept column (the last feature: a row of Aᵀ with N entries); labels in [0, K)"""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(N):
        k = int(rng.integers(0, 7)) if i % 13 else 0
        r = list(rng.integers(0, d - 3, k))
        if k > 2:
            r.append(r[0])
        rows.append(r + ([d - 1] if intercept else []))
    rows[3] = list(rng.integers(0, d - 3, L))
    rows[4] = list(rng.integers(0, d - 3, L + 1))
    rows[5] = []
    rowptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    col = np.concatenate([np.asarray(r, dtype=np.int64) for r in rows]).astype(np.int32)
    val = rng.uniform(-1.0, 1.0, col.size)
    if intercept:
        val[col == d - 1] = 1.0
    return rowptr, col, val, rng.integers(0, K, N)


def _ctx(G=296, block_bytes=None):
    c = cg.Context(0)
    c.timing(True)
    c.set_reduction_ctas(G)
    if block_bytes is not None:
        c.set_gather_block_bytes(block_bytes)
    return c


@pytest.mark.parametrize("G", [1, 3, 296])
@pytest.mark.parametrize("K", [2, 3, 7, 8, 32, 33])
def test_spmm_bit_exact(K, G):
    N, d = 1500, 51                                         # d odd: d·K odd for odd K
    rowptr, col, val, y = edge_data(N, d, K)
    ref = SoftmaxCSR(N, d, K, rowptr, col, val, y)
    O.set_cgo_order(G=G)
    rng = np.random.default_rng(K)
    W, C = rng.standard_normal(d * K), rng.standard_normal(N * K)
    Zr, Gr = ref.spmv(W), ref.spmv(C, True)
    ctx = _ctx(G)
    obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, 1e-4, ctx)
    assert obj.csr_blocks(False) == 1 and obj.csr_blocks(True) == 1
    assert np.array_equal(obj.spmv(W), Zr) and np.array_equal(obj.spmv(C, True), Gr)
    # column blocks of 20 features / samples: the same bits (A's rows are unsorted: only Aᵀ is blocked)
    cb = _ctx(G, block_bytes=8 * K * 20)
    blk = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, 1e-4, cb)
    assert blk.csr_blocks(False) == 1 and blk.csr_blocks(True) == 75
    assert np.array_equal(blk.spmv(W), Zr) and np.array_equal(blk.spmv(C, True), Gr)
    srt = np.concatenate([np.sort(col[rowptr[i]:rowptr[i + 1]]) for i in range(N)]).astype(np.int32)
    ref_s = SoftmaxCSR(N, d, K, rowptr, srt, val, y)          # sorted rows: A is blocked too
    sb = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, srt, val, y, 1e-4, cb)
    assert sb.csr_blocks(False) == 3
    assert np.array_equal(sb.spmv(W), ref_s.spmv(W)) and np.array_equal(sb.spmv(C, True), ref_s.spmv(C, True))
    # k_spmv_direct on the expanded matrix: the same bits on every row of at most L entries
    ctx.set_csr_mode(2)
    erp, eci, eva = kron_csr(N, rowptr, col, val, K)
    ls = cg.SparseLSGPU_from_csr(N * K, d * K, erp, eci.astype(np.int32), eva, np.zeros(N * K), ctx)
    assert ls.trial_site == (2, 4)
    short = np.diff(erp) <= L
    assert np.array_equal(ls.spmv(W)[short], Zr[short])
    erpT, _, _, _ = ls.csr(True)
    shortT = np.diff(erpT) <= L
    assert not shortT.all() and np.array_equal(ls.spmv(C, True)[shortT], Gr[shortT])
    for o in (obj, blk, sb, ls):
        o.close()
    ctx.close(); cb.close()


@pytest.mark.parametrize("K", [2, 5])
def test_no_entries(K):
    N, d = 40, 7
    rowptr = np.zeros(N + 1, dtype=np.int64)
    y = np.arange(N) % K
    ctx = _ctx()
    obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, np.zeros(0, np.int32), np.zeros(0), y, 1e-3, ctx)
    assert np.array_equal(obj.spmv(np.ones(d * K)), np.zeros(N * K))
    assert np.array_equal(obj.spmv(np.ones(N * K), True), np.zeros(d * K))
    ws = obj.make_workspace(np.zeros(d * K))
    assert ws.f_x0 == pytest.approx(np.log(K), rel=1e-13)
    ws.close(); obj.close(); ctx.close()


@pytest.mark.parametrize("K", [3, 33])
def test_f_and_g_against_reference(K):
    N, d, lam = 1500, 51, 1e-3
    rowptr, col, val, y = edge_data(N, d, K, seed=2)
    ref = SoftmaxCSR(N, d, K, rowptr, col, val, y, lam)
    ref.set_sum_mode("cgo")
    O.set_cgo_order(G=296)
    ctx = _ctx()
    obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, lam, ctx)
    assert obj.trial_site == (2, 4)
    rng = np.random.default_rng(3)
    for scale in (0.0, 0.1, 3.0, 40.0):
        w = scale * rng.standard_normal(d * K)
        assert np.array_equal(obj.spmv(w), ref.spmv(w))                     # Z
        _, Cr = ref.loss_and_c(w)
        assert np.array_equal(obj.spmv(Cr, True), ref.spmv(Cr, True))     # Aᵀ C for the reference's C
        f, g = ref.fdf(w)
        ws = obj.make_workspace(w, fuse_direction=False)
        assert abs(ws.f_x0 - f) <= 1e-13 * abs(f)
        gd = ws.download()[1]
        assert np.max(np.abs(gd - g)) <= 1e-13 * np.max(np.abs(g))
        ws.close()
    obj.close(); ctx.close()


def test_two_classes_equal_binary_logistic_regression():
    N, d, lam = 3000, 40, 1e-3
    rowptr, col, val, y = edge_data(N, d, 2, seed=4)
    ctx = _ctx()
    sm = cg.SoftmaxRegGPU_from_csr(N, d, 2, rowptr, col, val, y, lam, ctx)
    lr = cg.LogRegGPU_from_csr(N, d, rowptr, col, val, np.where(y == 1, 1.0, -1.0), lam, ctx)
    w = 0.5 * np.random.default_rng(5).standard_normal(d)
    ws, wb = sm.make_workspace(np.stack([np.zeros(d), w], 1).ravel()), lr.make_workspace(w)
    assert abs(ws.f_x0 - wb.f_x0) <= 1e-13 * abs(wb.f_x0)
    gs, gb = ws.download()[1].reshape(d, 2)[:, 1], wb.download()[1]
    assert np.max(np.abs(gs - gb)) <= 1e-13 * np.max(np.abs(gb))
    ws.close(); wb.close(); sm.close(); lr.close(); ctx.close()


@pytest.mark.parametrize("flavour", ["HagerZhang", "LBFGS"])
def test_runs_match_reference(flavour):
    N, d, K, lam = 1500, 51, 4, 1e-3
    rowptr, col, val, y = edge_data(N, d, K, seed=6)
    ctx = _ctx()
    _, cfg, ls = make_pair(flavour, "StrongWolfeBisection", eps=1e-6, max_iters=60, c1=1e-4, c2=0.9, lbfgs_m=10)
    obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, lam, ctx)
    ref = SoftmaxCSR(N, d, K, rowptr, col, val, y, lam)
    O.set_cgo_order(G=296)
    ora = cg.minimizeobjective(NumpyObjective(ref), np.zeros(d * K), cfg, ls)
    ret = cg.minimizeobjective(obj, np.zeros(d * K), cfg, ls)
    k = min(50, len(ora.trace.objective), len(ret.trace.objective))
    assert k >= 10
    assert np.array_equal(ret.trace.step_size[:k], ora.trace.step_size[:k])
    assert np.array_equal(ret.trace.objective_evals[:k], ora.trace.objective_evals[:k])
    np.testing.assert_allclose(ret.trace.objective[:k], ora.trace.objective[:k], rtol=1e-10)
    np.testing.assert_allclose(ret.trace.grad_norm[:k], ora.trace.grad_norm[:k], rtol=1e-8)
    assert ret.status == ora.status and abs(ret.iters_ran - ora.iters_ran) <= 2
    assert abs(ret.objective - ora.objective) <= 1e-8 * abs(ora.objective)
    again = cg.minimizeobjective(obj, np.zeros(d * K), cfg, ls)
    assert np.array_equal(again.trace.objective, ret.trace.objective) and np.array_equal(again.minimizer, ret.minimizer)
    obj.close(); ctx.close()


def test_launches_site_and_bytes():
    """one trial: K_a, the SpMM of A and its long row (two kernels), softmax, the SpMM of Aᵀ and the intercept's long
    row (two kernels), /N + λW"""
    N, d, K = 1500, 51, 7
    rowptr, col, val, y = edge_data(N, d, K)
    out = {}
    for name, bb in (("single", None), ("blocked", 8 * K * 100)):
        ctx = _ctx(block_bytes=bb)
        obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, 1e-4, ctx)
        x0 = 0.1 * np.random.default_rng(1).standard_normal(d * K)
        box = {}
        ops = {"x0": _measure(ctx, lambda: box.setdefault("ws", obj.make_workspace(x0, fuse_direction=True)))}
        ws = box["ws"]
        ws.reset_direction()
        ops["trial"] = _measure(ctx, lambda: ws.eval_trial(1e-3))
        ws.accept()

        def fused():
            ws.update_dir(0.3)
            ws.hint_first_trial(1e-3)
            ws.eval_trial(1e-3)
        ops["fused_trial"] = _measure(ctx, fused)
        with pytest.raises(cg.CgoError):
            ws.hessvec_dir()
        ws.close()
        out[name] = (obj.trial_site, obj.bytes_per_eval, ops)
        obj.close(); ctx.close()
    one = ({"axpy": 1, "other": 2, "spmv": 3, "spmvT": 3}, 9)
    assert out["single"] == ((2, 4), 512440.0, {"x0": one, "trial": one, "fused_trial": one})
    blk = ({"axpy": 1, "other": 2, "spmv": 3, "spmvT": 17}, 23)
    assert out["blocked"] == ((2, 4), 512440.0, {"x0": blk, "trial": blk, "fused_trial": blk})


def _reject(*args, lam=1e-4, ctx=None):
    with pytest.raises(cg.CgoError):
        cg.SoftmaxRegGPU_from_csr(*args, lam=lam, ctx=ctx)


def test_rejected_input():
    rp = np.array([0, 2, 3], dtype=np.int64)
    ci = np.array([0, 1, 2], dtype=np.int32)
    va = np.ones(3)
    y = np.array([0, 2])
    obj = cg.SoftmaxRegGPU_from_csr(2, 3, 3, rp, ci, va, y)      # accepted as given
    obj.close()
    _reject(0, 3, 3, np.zeros(1, np.int64), ci[:0], va[:0], y[:0])
    _reject(2, 0, 3, rp, ci, va, y)
    _reject(2, 1 << 31, 3, rp, ci, va, y)
    _reject(2, 3, 3, np.array([1, 2, 3], dtype=np.int64), ci, va, y)
    _reject(2, 3, 3, np.array([0, 3, 2], dtype=np.int64), ci, va, y)
    _reject(2, 3, 3, rp, np.array([0, 1, 3], dtype=np.int32), va, y)
    _reject(2, 3, 3, rp, np.array([0, -1, 2], dtype=np.int32), va, y)
    for K in (1, 257):
        _reject(2, 3, K, rp, ci, va, np.array([0, 0]))
    for bad in (-1, 3):
        _reject(2, 3, 3, rp, ci, va, np.array([0, bad]))
    _reject(2, 3, 3, rp, ci, va, np.array([0.0, 1.0]))             # labels are integers
    for lam in (-1e-3, float("inf"), float("nan")):
        _reject(2, 3, 3, rp, ci, va, y, lam=lam)
    ctx = cg.Context(0)
    ctx.set_csr_mode(1)
    _reject(2, 3, 3, rp, ci, va, y, ctx=ctx)
    ctx.close()


def test_blocked_size():
    """N = d = 10⁶, K = 8, ten sorted features per sample and an intercept: d·K·8 and N·K·8 exceed the 40 MiB
    blocks.  Sampled rows of A W and Aᵀ C bit for bit; f and g against a float64 statement whose sums are exact to
    far below 1e-13 (scipy adds the short rows in storage order, as the kernels do)."""
    import scipy.sparse as sp
    N = d = 1_000_000
    K, lam = 8, 1e-6
    rng = np.random.default_rng(7)
    cols = np.sort(rng.integers(0, d - 1, (N, 10)), axis=1)
    col = np.concatenate([cols, np.full((N, 1), d - 1)], 1).ravel().astype(np.int32)
    val = rng.uniform(-1.0, 1.0, col.size)
    val[10::11] = 1.0
    rowptr = np.arange(N + 1, dtype=np.int64) * 11
    y = rng.integers(0, K, N)
    ctx = cg.Context(0)
    obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rowptr, col, val, y, lam, ctx)
    assert obj.csr_blocks(False) == 2 and obj.csr_blocks(True) == 2
    A = sp.csr_matrix((val, col, rowptr), shape=(N, d))
    W = 0.3 * rng.standard_normal((d, K))
    Z = obj.spmv(W.ravel()).reshape(N, K)
    rows = rng.integers(0, N, 2000)
    assert np.array_equal(Z[rows], (A[rows] @ W))
    C = rng.standard_normal((N, K))
    GT = obj.spmv(C.ravel(), True).reshape(d, K)
    AT = A.T.tocsr()                                           # rows of Aᵀ by ascending sample: the storage order
    feats = rng.integers(0, d - 1, 2000)
    assert np.array_equal(GT[feats], AT[feats] @ C)
    O.set_cgo_order(G=296)
    O.set_site(1, 4)
    for k in range(K):                                         # the intercept: a long row, canonical order
        assert GT[d - 1, k] == O.dot(np.ones(N), np.ascontiguousarray(C[:, k]), "cgo")
    ws = obj.make_workspace(W.ravel())
    Zs = A @ W
    m = Zs.max(1, keepdims=True)
    E = np.exp(Zs - m)
    s = E.sum(1, keepdims=True)
    f = np.mean((m[:, 0] + np.log(s[:, 0])) - Zs[np.arange(N), y]) + 0.5 * lam * np.sum(W * W)
    P = E / s
    P[np.arange(N), y] -= 1.0
    g = (A.T @ P) / N + lam * W
    assert abs(ws.f_x0 - f) <= 1e-13 * abs(f)
    assert np.max(np.abs(ws.download()[1] - g.ravel())) <= 1e-13 * np.max(np.abs(g))
    ws.close(); obj.close(); ctx.close()
