"""The kernels every single-GPU path of the CSR objectives launches, pinned as literals.

A CSR objective runs its trial either on the fused k_csr_rows, whose epilogues reduce the dots, or on
k_spmv_direct followed by BLAS-1 dot passes; logistic regression also runs column-blocked k_spmv_direct passes.
For each objective and each operation this file checks how many kernels of each timing class run, the total
kernel launch count, the reduction site and the bytes per evaluation, so that a restructuring of the
evaluation code that launches one kernel more, one less or of another family fails here."""
import numpy as np
import pytest

import cgoptim_b200 as cg

pytestmark = pytest.mark.gpu

A_STEP = 1e-3


@pytest.fixture(scope="module")
def ctx():
    c = cg.Context(0)
    c.timing(True)
    yield c
    c.close()


def _ragged_csr(nrows=6000, ncols=4000, seed=5):
    """rows of 1 to 12 entries at random columns: ragged slices, gathers that do not coalesce"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 13, nrows)
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, ncols, int(rowptr[-1])).astype(np.int32)
    val = rng.uniform(-1.0, 1.0, int(rowptr[-1]))
    b = rng.uniform(-1.0, 1.0, nrows)
    return nrows, ncols, rowptr, col, val, b


def _make(ctx, name):
    mode, block = {"ragged_mode1": (1, None), "ragged_mode2": (2, None), "lr_blocked": (0, 8 * 700),
                   "lr_mode2": (2, None)}.get(name, (0, None))
    ctx.set_csr_mode(mode)
    if block is not None:
        ctx.set_gather_block_bytes(block)
    try:
        if name == "ls_coh0":
            return cg.SparseLSGPU(20_000, 10, 256, 24, 0, ctx)
        if name == "ls_coh30":
            return cg.SparseLSGPU(20_000, 10, 256, 24, 30, ctx)
        if name.startswith("ragged"):
            return cg.SparseLSGPU_from_csr(*_ragged_csr(), ctx=ctx)
        return cg.LogRegGPU(5000, 3000, 20, 24, 1e-4, ctx)
    finally:
        ctx.set_csr_mode(0)
        ctx.set_gather_block_bytes(40 << 20)


def _measure(ctx, fn):
    """({timing class: kernels}, kernel launches) of what fn() runs"""
    ctx.timing_read(reset=True)
    l0 = ctx.kernel_launches
    fn()
    counts = {k: c for k, (_, c) in ctx.timing_read(reset=True).items() if c}
    return counts, ctx.kernel_launches - l0


def observe(ctx, name):
    obj = _make(ctx, name)
    n = obj.n_local
    x0 = 0.1 * np.random.default_rng(1).standard_normal(n)
    ops = {}
    box = {}
    ops["x0"] = _measure(ctx, lambda: box.setdefault("ws", obj.make_workspace(x0, fuse_direction=True)))
    ws = box["ws"]
    ws.reset_direction()
    ops["trial"] = _measure(ctx, lambda: ws.eval_trial(A_STEP))
    ops["accept"] = _measure(ctx, ws.accept)

    def fused():
        ws.update_dir(0.3)
        ws.hint_first_trial(A_STEP)
        ws.eval_trial(A_STEP)
    ops["fused_trial"] = _measure(ctx, fused)
    ws.accept()
    if not name.startswith("lr"):
        ops["hessvec"] = _measure(ctx, ws.hessvec_dir)
        wq = obj.make_workspace(x0, quadratic_linesearch=True)
        wq.reset_direction()
        wq.hessvec_dir()                                   # leaves r as scratch: the next begin re-forms A x − b
        ops["quad_begin_residual"] = _measure(ctx, lambda: wq.eval_trial(A_STEP))
        ops["quad_accept"] = _measure(ctx, wq.accept)
        wq.reset_direction()
        ops["quad_begin"] = _measure(ctx, lambda: wq.eval_trial(A_STEP))
        ops["quad_accept_2"] = _measure(ctx, wq.accept)
        wq.close()
    site, nbytes = obj.trial_site, obj.bytes_per_eval
    ws.close()
    obj.close()
    return {"site": site, "bytes": nbytes, "ops": ops}


EXPECTED = {
    "ls_coh0": {"site": (2, 4), "bytes": 6880016.0, "ops": {
        "x0": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "trial": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "hessvec": ({"other": 2, "spmv": 1, "spmvT": 1}, 4),
        "quad_begin_residual": ({"other": 1, "spmv": 2}, 3),
        "quad_accept": ({"axpy": 2, "other": 1, "spmvT": 1}, 4),
        "quad_begin": ({"other": 1, "spmv": 1}, 2),
        "quad_accept_2": ({"axpy": 2, "other": 1, "spmvT": 1}, 4),
    }},
    "ls_coh30": {"site": (1, 1), "bytes": 6560016.0, "ops": {
        "x0": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "trial": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "hessvec": ({"spmv": 1, "spmvT": 1}, 2),
        "quad_begin_residual": ({"spmv": 2}, 2),
        "quad_accept": ({"axpy": 2, "spmvT": 1}, 3),
        "quad_begin": ({"spmv": 1}, 1),
        "quad_accept_2": ({"axpy": 2, "spmvT": 1}, 3),
    }},
    "ragged_mode1": {"site": (1, 1), "bytes": 1354560.0, "ops": {
        "x0": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "trial": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "hessvec": ({"spmv": 1, "spmvT": 1}, 2),
        "quad_begin_residual": ({"spmv": 2}, 2),
        "quad_accept": ({"axpy": 2, "spmvT": 1}, 3),
        "quad_begin": ({"spmv": 1}, 1),
        "quad_accept_2": ({"axpy": 2, "spmvT": 1}, 3),
    }},
    "ragged_mode2": {"site": (2, 4), "bytes": 1434560.0, "ops": {
        "x0": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "trial": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "hessvec": ({"other": 2, "spmv": 1, "spmvT": 1}, 4),
        "quad_begin_residual": ({"other": 1, "spmv": 2}, 3),
        "quad_accept": ({"axpy": 2, "other": 1, "spmvT": 1}, 4),
        "quad_begin": ({"other": 1, "spmv": 1}, 2),
        "quad_accept_2": ({"axpy": 2, "other": 1, "spmvT": 1}, 4),
    }},
    "lr_single": {"site": (1, 1), "bytes": 2728016.0, "ops": {
        "x0": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "trial": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "spmv": 1, "spmvT": 1}, 3),
    }},
    "lr_blocked": {"site": (2, 4), "bytes": 2928016.0, "ops": {
        "x0": ({"axpy": 1, "other": 2, "spmv": 5, "spmvT": 8}, 16),
        "trial": ({"axpy": 1, "other": 2, "spmv": 5, "spmvT": 8}, 16),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "other": 2, "spmv": 5, "spmvT": 8}, 16),
    }},
    "lr_mode2": {"site": (2, 4), "bytes": 2928016.0, "ops": {
        "x0": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "trial": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
        "accept": ({}, 0),
        "fused_trial": ({"axpy": 1, "other": 2, "spmv": 1, "spmvT": 1}, 5),
    }},
}


@pytest.mark.parametrize("name", list(EXPECTED))
def test_launch_sequence(ctx, name):
    assert observe(ctx, name) == EXPECTED[name]
