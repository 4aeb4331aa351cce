"""Device context, objective handles and the device-resident LineSearchContainer.

The reference keeps `xp, df_xp, x, u` (src/types.jl:84-100) and `x, df_x`
(src/engine/optim.jl:20-21) as host Vectors.  Here they live in HBM behind a `cgo_state`; the
host sees them as `DeviceVector` tokens so that the engine and the line searches keep the
reference's call shapes (`evalϕdϕ_(xp, df_xp, fdf_, a, x, u)`, `dot(df_x, u)`,
`getβ(β_config, g_next, g, u)`, `updatedir_(u, df_x, β)`).

No CPU fallback: everything here goes through libcgoptim.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _capi as capi
from ._capi import (D_GU, D_UU, P_DIR_GU, P_DIR_UU, P_DPHI, P_GPG, P_GPGP, P_PHI, P_UG, P_UU, P_UY, P_YGP, P_YY,
                    PACK_LEN, CgoError, check, dptr, lib)

f64 = np.float64


class Context:
    """One GPU, one stream, optionally one rank of an NCCL communicator (`cgo_ctx`)."""

    def __init__(self, device: int = 0, stream_ptr: int = 0, reduction_ctas: Optional[int] = None):
        h = C.c_void_p()
        check(lib().cgo_ctx_create(device, C.c_void_p(stream_ptr) if stream_ptr else None, C.byref(h)))
        self.h = h
        self.device = device
        self.nranks, self.rank = 1, 0
        if reduction_ctas is not None:
            self.set_reduction_ctas(reduction_ctas)

    def set_reduction_ctas(self, G: int):
        check(lib().cgo_ctx_set_reduction_ctas(self.h, G))

    def set_gather_block_bytes(self, nbytes: int):
        """Column-block size for objectives with large random gathers (0 disables blocking)."""
        check(lib().cgo_ctx_set_gather_block_bytes(self.h, int(nbytes)))

    def trim_pools(self) -> int:
        """Give the pooled device blocks (vectors of closed workspaces) and the pooled pinned host buffers back;
        returns the device bytes freed."""
        v = C.c_int64()
        check(lib().cgo_ctx_trim_pools(self.h, C.byref(v)))
        capi.pinned_pool_clear()
        return v.value

    def set_csr_mode(self, mode: int):
        """SpMV kernel family of CSR objectives created afterwards: 0 per matrix, 1 fused k_csr_rows, 2 k_spmv_direct."""
        check(lib().cgo_ctx_set_csr_mode(self.h, int(mode)))

    @property
    def stream_ptr(self) -> int:
        s = C.c_void_p()
        check(lib().cgo_ctx_stream(self.h, C.byref(s)))
        return s.value or 0

    @property
    def sm_count(self) -> int:
        v = C.c_int()
        check(lib().cgo_ctx_sm_count(self.h, C.byref(v)))
        return v.value

    @property
    def kernel_launches(self) -> int:
        v = C.c_int64()
        check(lib().cgo_ctx_kernel_launches(self.h, C.byref(v)))
        return v.value

    KERNEL_CLASSES = ("trial", "direction", "axpy", "spmv", "spmvT", "lbfgs", "other", "batched")

    def timing(self, enable: bool):
        check(lib().cgo_ctx_timing(self.h, int(enable)))

    def timing_read(self, reset: bool = True):
        """{class: (total_ms, launches)} measured with CUDA events on the ctx stream."""
        ms = np.zeros(8)
        cnt = np.zeros(8, dtype=np.int64)
        check(lib().cgo_ctx_timing_read(self.h, dptr(ms), cnt.ctypes.data_as(C.POINTER(C.c_int64)), int(reset)))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.KERNEL_CLASSES)}

    # -- multi-GPU: one process per GPU; the 128-byte id travels over the host's own channel
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        check(lib().cgo_comm_get_unique_id(buf))
        return buf.raw

    def comm_init(self, nranks: int, rank: int, unique_id: bytes):
        buf = C.create_string_buffer(unique_id, 128)
        check(lib().cgo_ctx_comm_init(self.h, nranks, rank, buf))
        self.nranks, self.rank = nranks, rank

    def comm_init_torch(self):
        """Bootstrap the communicator through an initialised torch.distributed group."""
        import torch.distributed as dist
        nranks, rank = dist.get_world_size(), dist.get_rank()
        ids = [Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        self.comm_init(nranks, rank, ids[0])

    def barrier(self):
        check(lib().cgo_ctx_barrier(self.h))

    @property
    def peer_memory(self) -> bool:
        """True when halo exchanges run as peer-memory stores fused into the kernels (CUDA IPC)."""
        v = C.c_int()
        check(lib().cgo_ctx_peer_memory(self.h, C.byref(v)))
        return bool(v.value)

    def close(self):
        if self.h:
            lib().cgo_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


def shard_range(n: int, nranks: int, rank: int, align: int = 2):
    lo, hi = C.c_int64(), C.c_int64()
    check(lib().cgo_shard_range(n, nranks, rank, align, C.byref(lo), C.byref(hi)))
    return lo.value, hi.value


# ---------------------------------------------------------------------------------- objectives
class DeviceObjective:
    """Device-resident replacement of the user callback `fdf!(g, x) -> f`."""

    nclasses = 1        # columns of the vectors `spmv` multiplies (the softmax objective's K)
    intercept = 0       # 1: the state ends with an intercept row, which `spmv(transposed=True)` returns too

    def __init__(self, ctx: Context, handle: C.c_void_p):
        self.ctx, self.h = ctx, handle
        nl, ng, off = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib().cgo_obj_dims(self.h, C.byref(nl), C.byref(ng), C.byref(off)))
        self.n_local, self.n_global, self.offset = nl.value, ng.value, off.value

    @property
    def bytes_per_eval(self) -> float:
        v = C.c_double()
        check(lib().cgo_obj_bytes_per_eval(self.h, C.byref(v)))
        return v.value

    @property
    def trial_site(self):
        """(V, U) of the canonical reduction order the trial's dots follow (include/cgoptim.h)"""
        v, u = C.c_int32(), C.c_int32()
        check(lib().cgo_obj_reduction_site(self.h, C.byref(v), C.byref(u)))
        return v.value, u.value

    def default_x0(self, seed: int = 24, perturb: float = 0.0) -> np.ndarray:
        x0 = np.empty(self.n_local)
        check(lib().cgo_obj_default_x0(self.h, seed, perturb, dptr(x0)))
        return x0

    def make_workspace(self, x_initial, lbfgs_m: int = 0, fuse_direction: bool = True,
                       beta_form: str = "fused", quadratic_linesearch: bool = False):
        return DeviceLineSearchContainer(self, x_initial, lbfgs_m, fuse_direction, beta_form, quadratic_linesearch)

    # CSR test hooks
    def csr(self, transposed=False):
        """(rowptr, col, val, b) of A, or of the explicit transpose; b always has A's row count."""
        nr, nnz, nra = C.c_int64(), C.c_int64(), C.c_int64()
        check(lib().cgo_obj_csr_nnz(self.h, int(transposed), C.byref(nr), C.byref(nnz)))
        check(lib().cgo_obj_csr_nnz(self.h, 0, C.byref(nra), None))
        rp = np.empty(nr.value + 1, dtype=np.int64)
        ci = np.empty(nnz.value, dtype=np.int32)
        va = np.empty(nnz.value)
        b = np.empty(nra.value)
        check(lib().cgo_obj_csr_download(self.h, int(transposed), rp.ctypes.data, ci.ctypes.data,
                                         va.ctypes.data, b.ctypes.data))
        return rp, ci, va, b

    def csr_blocks(self, transposed=False) -> int:
        """passes one SpMV with this matrix takes (1 = not column-blocked)"""
        v = C.c_int32()
        check(lib().cgo_obj_csr_blocks(self.h, int(transposed), C.byref(v)))
        return v.value

    def spmv(self, x, transposed=False):
        nr, nnz = C.c_int64(), C.c_int64()
        check(lib().cgo_obj_csr_nnz(self.h, int(transposed), C.byref(nr), C.byref(nnz)))
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty((nr.value + (self.intercept if transposed else 0)) * self.nclasses)
        check(lib().cgo_obj_spmv(self.h, int(transposed), dptr(x), dptr(y)))
        return y

    def close(self):
        if self.h:
            lib().cgo_obj_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def RosenbrockGPU(n: int, ctx: Optional[Context] = None) -> DeviceObjective:
    """Extended Rosenbrock (pairs), SURVEY.md §8d cfg 1/2/5."""
    ctx = ctx or default_context()
    h = C.c_void_p()
    check(lib().cgo_obj_rosenbrock_create(ctx.h, n, C.byref(h)))
    return DeviceObjective(ctx, h)


class _DevArray:
    """a device pointer behind __cuda_array_interface__ (what torch.as_tensor wraps without a copy)"""

    def __init__(self, ptr: int, n: int, readonly: bool):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}   # (torch rejects the read-only flag)


class UserObjectiveGPU(DeviceObjective):
    """Any `fdf!(g, x) -> f` (src/engine/optim.jl:6-11) on the device: `fdf(g, x)` receives the gradient buffer and
    the trial point as torch.float64 CUDA tensors (views of the solver's own vectors — this rank's shard), fills `g`
    in place and returns f (a 0-dim CUDA tensor, or this rank's part of it when sharded).  It runs on the ctx stream
    (torch.cuda.stream is set around the call) and must not synchronise.  The reference's signature and order of
    arguments; the line search, β and the dots stay the library's (two BLAS-1 kernels per trial around the callback)."""

    def __init__(self, n: int, fdf, ctx: Optional[Context] = None):
        import torch
        ctx = ctx or default_context()
        self._torch, self._fdf = torch, fdf
        self._stream = torch.cuda.ExternalStream(ctx.stream_ptr, device=torch.device("cuda", ctx.device))
        self.last_error = None

        def trampoline(_user, _stream, n_local, offset, xp, g, f):
            try:
                dev = torch.device("cuda", ctx.device)
                with torch.cuda.stream(self._stream):
                    x_t = torch.as_tensor(_DevArray(xp, n_local, True), device=dev)
                    g_t = torch.as_tensor(_DevArray(g, n_local, False), device=dev)
                    f_t = torch.as_tensor(_DevArray(f, 1, False), device=dev)
                    val = fdf(g_t, x_t)
                    f_t.copy_(torch.as_tensor(val, dtype=torch.float64, device=dev).reshape(1))
                return 0
            except Exception as e:      # an exception must not cross the C ABI
                self.last_error = e
                return 1

        self._cb = capi.USER_FDF(trampoline)          # keep the thunk alive as long as the objective
        h = C.c_void_p()
        check(lib().cgo_obj_user_create(ctx.h, n, self._cb, None, C.byref(h)))
        super().__init__(ctx, h)


def RosenbrockChainedGPU(n: int, ctx: Optional[Context] = None) -> DeviceObjective:
    """The reference's own chained Rosenbrock (examples/helpers/test_funcs.jl:50-57) with its gradient."""
    ctx = ctx or default_context()
    h = C.c_void_p()
    check(lib().cgo_obj_rosenbrock_chained_create(ctx.h, n, C.byref(h)))
    return DeviceObjective(ctx, h)


def SparseLSGPU(n: int, nnz_per_row: int = 10, W: Optional[int] = None, seed: int = 24,
                coh_log2: int = 0, ctx: Optional[Context] = None) -> DeviceObjective:
    """½‖Ax − b‖² with the synthetic banded-random CSR of SURVEY.md §8d cfg 3."""
    ctx = ctx or default_context()
    if W is None:
        W = min(1 << 20, (n - 1) // 2)
    h = C.c_void_p()
    check(lib().cgo_obj_sparse_ls_create_synthetic(ctx.h, n, nnz_per_row, W, seed, coh_log2, C.byref(h)))
    return DeviceObjective(ctx, h)


def SparseLSGPU_from_csr(nrows, ncols, rowptr, col, val, b, ctx: Optional[Context] = None) -> DeviceObjective:
    ctx = ctx or default_context()
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    h = C.c_void_p()
    check(lib().cgo_obj_sparse_ls_create_csr(ctx.h, nrows, ncols, rowptr.ctypes.data, col.ctypes.data,
                                             val.ctypes.data, b.ctypes.data, C.byref(h)))
    return DeviceObjective(ctx, h)


def LogRegGPU(nsamples: int, nfeat: int, nnz_per_row: int = 20, seed: int = 24, lam: float = 1e-6,
              ctx: Optional[Context] = None) -> DeviceObjective:
    """CSR logistic regression, SURVEY.md §8d cfg 4."""
    ctx = ctx or default_context()
    h = C.c_void_p()
    check(lib().cgo_obj_logreg_create_synthetic(ctx.h, nsamples, nfeat, nnz_per_row, seed, lam, C.byref(h)))
    return DeviceObjective(ctx, h)


def _glm_options(nsamples, sample_weight, fit_intercept):
    """(weights pointer or None, the array that owns it, 0 / 1) of the GLM constructors"""
    if fit_intercept not in (False, True, 0, 1):
        raise CgoError(f"fit_intercept must be a bool (got {fit_intercept!r})")
    if sample_weight is None:
        return None, None, int(fit_intercept)
    sw = np.ascontiguousarray(sample_weight, dtype=np.float64)
    if sw.shape != (nsamples,):
        raise CgoError(f"sample_weight needs nsamples = {nsamples} entries (got shape {sw.shape})")
    return sw.ctypes.data, sw, int(fit_intercept)


def LogRegGPU_from_csr(nsamples, nfeat, rowptr, col, val, y, lam: float = 1e-6,
                       ctx: Optional[Context] = None, sample_weight=None, fit_intercept=False) -> DeviceObjective:
    """(1/S) Σ s_i log(1 + exp(−y_i (a_i·w + b))) + (λ/2)‖w‖² on the caller's CSR (0-based int64 row pointers, int32
    columns) and labels y_i ∈ {−1, +1}; single GPU.

    `sample_weight`: nsamples finite weights s_i >= 0 with a positive sum S, or None for s_i = 1 (S = nsamples).
    `fit_intercept`: fit b, which λ does not penalise.  The state is then (w, b) of length nfeat + 1: b is
    `minimizer[nfeat]`, where an explicit column of ones appended as feature nfeat would put its weight.  Without it
    there is no b; a column of ones in A is an intercept that λ penalises like the other weights.  Weights or an
    intercept need the k_spmv_direct kernel family (a ctx with csr_mode 1 rejects them)."""
    ctx = ctx or default_context()
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    if rowptr.size != nsamples + 1 or y.size != nsamples:
        raise CgoError(f"rowptr needs nsamples + 1 = {nsamples + 1} entries and y nsamples (got {rowptr.size}, {y.size})")
    if col.size < rowptr[-1] or val.size < rowptr[-1]:
        raise CgoError(f"col and val need rowptr[-1] = {rowptr[-1]} entries (got {col.size}, {val.size})")
    sw_ptr, _sw, icpt = _glm_options(nsamples, sample_weight, fit_intercept)
    h = C.c_void_p()
    check(lib().cgo_obj_logreg_create_csr_ex(ctx.h, nsamples, nfeat, rowptr.ctypes.data, col.ctypes.data,
                                             val.ctypes.data, y.ctypes.data, sw_ptr, icpt, lam, C.byref(h)))
    obj = DeviceObjective(ctx, h)
    obj.intercept = icpt
    return obj


def SoftmaxRegGPU_from_csr(nsamples, nfeat, nclasses, rowptr, col, val, labels, lam: float = 1e-6,
                           ctx: Optional[Context] = None, sample_weight=None, fit_intercept=False) -> DeviceObjective:
    """(1/S) Σ_i s_i [logsumexp(a_i W + b) − (a_i W + b)_{y_i}] + (λ/2)‖W‖² (multinomial logistic regression) on the
    caller's CSR (0-based int64 row pointers, int32 columns) and labels y_i ∈ [0, nclasses), 2 <= nclasses <= 256;
    single GPU.  The state vector is W (nfeat × nclasses) feature-major, w[j·K + k], of length nfeat·nclasses: a
    result's `minimizer.reshape(nfeat, nclasses)` is W.

    `sample_weight`: nsamples finite weights s_i >= 0 with a positive sum S, or None for s_i = 1 (S = nsamples).
    `fit_intercept`: fit b (one per class), which λ does not penalise.  The state then has nfeat + 1 rows:
    `minimizer.reshape(nfeat + 1, nclasses)[nfeat]` is b, where an explicit column of ones appended as feature nfeat
    would put its weights.  Without it there is no b; a column of ones in A is an intercept penalised like the
    other weights.  `spmv` takes and returns K-wide vectors: Z = A W (nfeat·K → nsamples·K) and Aᵀ C (nsamples·K →
    nfeat·K, followed by the K intercept sums Σ_i c_ik with an intercept)."""
    ctx = ctx or default_context()
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    val = np.ascontiguousarray(val, dtype=np.float64)
    labels = np.asarray(labels)
    if labels.size != nsamples or rowptr.size != nsamples + 1:
        raise CgoError(f"rowptr needs nsamples + 1 = {nsamples + 1} entries and labels nsamples (got {rowptr.size}, {labels.size})")
    if col.size < rowptr[-1] or val.size < rowptr[-1]:
        raise CgoError(f"col and val need rowptr[-1] = {rowptr[-1]} entries (got {col.size}, {val.size})")
    if not np.issubdtype(labels.dtype, np.integer) or labels.size and (labels.min() < -2**31 or labels.max() >= 2**31):
        raise CgoError("labels must be integers")
    labels = np.ascontiguousarray(labels, dtype=np.int32)
    sw_ptr, _sw, icpt = _glm_options(nsamples, sample_weight, fit_intercept)
    h = C.c_void_p()
    check(lib().cgo_obj_softmax_create_csr_ex(ctx.h, nsamples, nfeat, int(nclasses), rowptr.ctypes.data,
                                              col.ctypes.data, val.ctypes.data, labels.ctypes.data, sw_ptr, icpt, lam,
                                              C.byref(h)))
    obj = DeviceObjective(ctx, h)
    obj.nclasses = int(nclasses)
    obj.intercept = icpt
    return obj


class BoxBarrierGPU(DeviceObjective):
    """t·f0(x) − Σ log(ubs − x) − Σ log(x − lbs) around a device objective: the `fdf!` closure that
    primalbarriermethod! builds (src/engine/primal_barrier.jl:205-213, evalbarrier! :112-133) for the
    box constraints of examples/constrained.jl:17-47.  lbs / ubs are this rank's shard."""

    def __init__(self, inner: DeviceObjective, lbs, ubs, t: float = 1.0):
        lbs = np.ascontiguousarray(lbs, dtype=np.float64)
        ubs = np.ascontiguousarray(ubs, dtype=np.float64)
        if lbs.shape != (inner.n_local,) or ubs.shape != (inner.n_local,):
            raise ValueError("lbs / ubs must have the objective's (local) dimension")
        h = C.c_void_p()
        check(lib().cgo_obj_box_barrier_create(inner.ctx.h, inner.h, dptr(lbs), dptr(ubs), float(t), C.byref(h)))
        super().__init__(inner.ctx, h)
        self.inner, self.lbs, self.ubs, self.t = inner, lbs, ubs, float(t)

    def set_t(self, t: float):
        check(lib().cgo_obj_barrier_set_t(self.h, float(t)))
        self.t = float(t)

    def infeasible_count(self, x) -> int:
        """how many coordinates (over all ranks) have x − ub >= 0 or lb − x >= 0 (primal_barrier.jl:189)"""
        x = np.ascontiguousarray(x, dtype=np.float64)
        v = C.c_int64()
        check(lib().cgo_obj_barrier_infeasible(self.h, dptr(x), C.byref(v)))
        return v.value


# ---------------------------------------------------------------------------------- vectors
class DeviceVector:
    """Token for one of the device-resident vectors of a LineSearchContainer."""
    __slots__ = ("ws", "name")

    def __init__(self, ws, name: str):
        self.ws, self.name = ws, name

    def __repr__(self):
        return f"<DeviceVector {self.name} n={self.ws.n}>"


def dot(a: DeviceVector, b: DeviceVector):
    """LinearAlgebra.dot on device vectors.  Only the pairs the hot path needs exist:
    dot(df_x, u) (nocedal.jl:56, wolfe.jl:40, geometric.jl:43) and dot(u, u) (wolfe.jl:240,
    geometric.jl:52); both were produced by the kernel that last wrote u."""
    names = {a.name, b.name}
    if names == {"df_x", "u"}:
        return a.ws.dot_g_u()
    if names == {"u"}:
        return a.ws.dot_u_u()
    raise NotImplementedError(f"dot({a.name}, {b.name}) is not on the hot path")


class DeviceStart:
    """`x_initial` that already lives on the device: the iterate `x` of a live workspace.  minimizeobjective copies
    it device to device (cgo_state_create_from_state) instead of uploading a host vector."""
    __slots__ = ("ws",)

    def __init__(self, ws):
        self.ws = ws


class DeviceLineSearchContainer:
    """LineSearchContainer (types.jl:84-100) + x, df_x of optim.jl:20-21, resident in HBM.

    Construction performs optim.jl:20-26: copies x_initial to the device, evaluates
    f_x = fdf!(df_x, x) and ‖df_x‖.
    """

    def __init__(self, objective: DeviceObjective, x_initial, lbfgs_m=0, fuse_direction=True,
                 beta_form="fused", quadratic_linesearch=False):
        assert beta_form in ("fused", "literal")
        # SURVEY.md §8f N1 (CSR least squares only): the trials of a line search are evaluated from
        # r·v, v·v with v = A u (one SpMV per line search); the accepted step is materialised once
        self.quadratic = bool(quadratic_linesearch)
        self._q = None                        # (r·v, v·v, ½ r·r) of the current line search
        self._q_a = None                      # last trial step, not yet materialised
        if self.quadratic:
            fuse_direction = False            # there is no trial kernel for the direction update to ride on
        self.objective = objective
        self.n = objective.n_local
        self.fuse_direction = fuse_direction
        self.beta_form = beta_form
        self._buf = np.zeros(PACK_LEN)
        self.h = C.c_void_p()
        self.h2d_bytes = 0                    # host → device bytes this workspace cost (x_initial)
        if isinstance(x_initial, DeviceStart):
            src = x_initial.ws
            if src.h is None or not src.h or src.n != self.n:
                raise ValueError("DeviceStart: the source workspace is closed or has another dimension")
            check(lib().cgo_state_create_from_state(objective.ctx.h, objective.h, src.h, 0, lbfgs_m, C.byref(self.h), dptr(self._buf)))
        else:
            x0 = np.ascontiguousarray(x_initial, dtype=np.float64)
            if x0.shape != (objective.n_local,):
                raise ValueError(f"x_initial has shape {x0.shape}, objective shard has n={objective.n_local}")
            check(lib().cgo_state_create(objective.ctx.h, objective.h, dptr(x0), lbfgs_m, C.byref(self.h), dptr(self._buf)))
            self.h2d_bytes = 8 * self.n
        self.f_x0 = f64(self._buf[P_PHI])
        self.norm_df_x0 = np.sqrt(f64(self._buf[P_GPGP]))
        self.pack = self._buf.copy()          # last trial pack
        self.dpack = np.zeros(2)              # last direction pack {g·u, u·u}
        self._pending_beta = None             # lazily fused updatedir!
        self._hint = None
        self._cached = None                   # (a, pack) of a speculative first trial
        self.fdf_evals = 1
        self.xp, self.df_xp = DeviceVector(self, "xp"), DeviceVector(self, "df_xp")
        self.x, self.u = DeviceVector(self, "x"), DeviceVector(self, "u")
        self.df_x = DeviceVector(self, "df_x")

    # -- direction -------------------------------------------------------------------
    def reset_direction(self):
        """u = −df_x (cg_flavours.jl:28, wolfe.jl:129)."""
        self._pending_beta = None
        self._cached = None
        self._q = None
        check(lib().cgo_reset_direction(self.h, dptr(self._buf)))
        self.dpack = self._buf[:2].copy()

    def update_dir(self, β):
        """updatedir! (cg_flavours.jl:2-15).  With fuse_direction the kernel is deferred and
        fused into the first trial of the next line search."""
        self._cached = None
        self._q = None
        if self.fuse_direction:
            self._pending_beta = float(β)
        else:
            check(lib().cgo_update_dir(self.h, float(β), dptr(self._buf)))
            self.dpack = self._buf[:2].copy()

    def hint_first_trial(self, a):
        """The step the caller will evaluate first (lets the pending direction update ride on it)."""
        self._hint = float(a)

    def _materialize_direction(self):
        if self._pending_beta is None:
            return
        β, self._pending_beta = self._pending_beta, None
        if self._hint is not None and np.isfinite(self._hint):
            a = self._hint
            check(lib().cgo_eval_trial_fused_dir(self.h, β, a, dptr(self._buf)))
            pk = self._buf.copy()
            self._cached = (a, pk)
            self.dpack = np.array([pk[P_DIR_GU], pk[P_DIR_UU]])
        else:
            check(lib().cgo_update_dir(self.h, β, dptr(self._buf)))
            self.dpack = self._buf[:2].copy()
        self._hint = None

    def dot_g_u(self):
        self._materialize_direction()
        return f64(self.dpack[D_GU])

    def dot_u_u(self):
        self._materialize_direction()
        return f64(self.dpack[D_UU])

    def norm_u_plus_g(self):
        """norm(u + df_x) (wolfe.jl:123)"""
        self._materialize_direction()
        v = C.c_double()
        check(lib().cgo_norm_sq_u_plus_g(self.h, C.byref(v)))
        return np.sqrt(f64(v.value))

    # -- trial point -----------------------------------------------------------------
    def _quad_materialize(self):
        """the accepted step of a quadratic-aware line search: xp, r, g⁺ and the dot pack"""
        if self._q_a is not None:
            a, self._q_a = self._q_a, None
            check(lib().cgo_quad_accept(self.h, a, dptr(self._buf)))
            self.pack = self._buf.copy()
            self._q = None

    def eval_trial(self, a):
        """evalϕdϕ! (cg_utils.jl:3-22): returns (ϕ, dϕ); the full pack stays in self.pack."""
        self._materialize_direction()
        a = float(a)
        if self.quadratic:
            if self._q is None:               # first trial of this line search: v = A u
                check(lib().cgo_quad_begin(self.h, dptr(self._buf)))
                self._q = (f64(self._buf[0]), f64(self._buf[1]), f64(0.5) * f64(self._buf[2]))
            rv, vv, f0 = self._q
            a64 = f64(a)
            self._q_a = a
            self.fdf_evals += 1
            with np.errstate(all="ignore"):
                return f0 + a64 * rv + f64(0.5) * a64 * a64 * vv, rv + a64 * vv
        if self._cached is not None and self._cached[0] == a:
            self.pack = self._cached[1]
            self._cached = None
        else:
            self._cached = None
            check(lib().cgo_eval_trial(self.h, a, dptr(self._buf)))
            self.pack = self._buf.copy()
        self.fdf_evals += 1
        return f64(self.pack[P_PHI]), f64(self.pack[P_DPHI])

    def norm_df_xp(self):
        """norm(info.df_xp) (optim.jl:107)"""
        self._quad_materialize()
        return np.sqrt(f64(self.pack[P_GPGP]))

    def beta_literal(self, R, m):
        v = C.c_double()
        check(lib().cgo_beta_literal(self.h, float(R), float(m), C.byref(v)))
        return f64(v.value)

    def accept(self):
        """x[:] = info.xp; df_x[:] = info.df_xp; info.x[:] = x  (optim.jl:136-140): pointer swaps."""
        self._cached = None
        self._quad_materialize()
        check(lib().cgo_accept(self.h))

    # -- L-BFGS ----------------------------------------------------------------------
    def lbfgs_stage_pair(self):
        check(lib().cgo_lbfgs_stage_pair(self.h, dptr(self._buf)))
        return f64(self._buf[0]), f64(self._buf[1])

    def lbfgs_commit_pair(self, commit: bool, rho=0.0, gamma=1.0):
        check(lib().cgo_lbfgs_commit_pair(self.h, int(commit), float(rho), float(gamma)))

    def lbfgs_update_dir(self):
        self._cached = None
        self._pending_beta = None
        self._q = None
        check(lib().cgo_lbfgs_update_dir(self.h, dptr(self._buf)))
        self.dpack = self._buf[:2].copy()

    # -- curvature ------------------------------------------------------------------
    def hessvec_dir(self):
        """∇²f(x) u along the current direction (CSR least squares: Aᵀ(A u)) -> (u·Hu, hv on the host).
        u·Hu is what an exact line minimisation of a quadratic needs: a* = −(g·u)/(u·Hu)."""
        self._materialize_direction()
        check(lib().cgo_hessvec_dir(self.h, dptr(self._buf)))
        uHu = f64(self._buf[0])
        hv = np.empty(self.n)
        check(lib().cgo_download_vector(self.h, 5, dptr(hv)))
        return uHu, hv

    # -- solvesystem (src/engine/solve_system.jl) --------------------------------------
    def solvesys_begin(self):
        """x_next = copy(x_initial) (solve_system.jl:82)"""
        check(lib().cgo_solvesys_begin(self.h))

    def solvesys_project(self, m, fix_stale_iterate=False):
        """updateiteratesolvesys! (:237-253) + f_x_next = fdf!(info.df_xp, x_next) (:179):
        returns (f_x_next, norm(info.df_xp)); the pack holds the getβ dots."""
        self._materialize_direction()
        self._cached = None
        check(lib().cgo_solvesys_project(self.h, float(m), int(bool(fix_stale_iterate)), dptr(self._buf)))
        self.pack = self._buf.copy()
        self.fdf_evals += 1
        return f64(self.pack[P_PHI]), np.sqrt(f64(self.pack[P_GPGP]))

    def solvesys_accept(self, fix_stale_iterate=False):
        """x, x_next = x_next, x; df_x[:] = info.df_xp; info.x[:] = x (:196, :207-208)"""
        self._cached = None
        check(lib().cgo_solvesys_accept(self.h, int(bool(fix_stale_iterate))))

    def dot_df_xp_u(self):
        """dot(df_xp, u) (solve_system.jl:246): reduced by the trial kernel that produced df_xp"""
        return f64(self.pack[P_DPHI])

    # -- results ---------------------------------------------------------------------
    def download_trial(self):
        """info.xp, info.df_xp on the host (updateresult! with the container, types.jl:116-131)"""
        x, g = capi.pinned_empty(self.n), capi.pinned_empty(self.n)
        check(lib().cgo_download_vector(self.h, 3, dptr(x)))
        check(lib().cgo_download_vector(self.h, 4, dptr(g)))
        return x, g

    def download(self):
        x, g = capi.pinned_empty(self.n), capi.pinned_empty(self.n)
        check(lib().cgo_download(self.h, dptr(x), dptr(g)))
        return x, g

    def download_vector(self, name: str):
        which = {"x": 0, "df_x": 1, "u": 2, "xp": 3, "df_xp": 4}[name]
        if name == "u":
            self._materialize_direction()
        v = np.empty(self.n)
        check(lib().cgo_download_vector(self.h, which, dptr(v)))
        return v

    def close(self):
        if self.h:
            lib().cgo_state_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------- batched
STATUS_SYMBOLS = (
    "incomplete", "success", "increasing_objective", "max_iters_reached",
    "non_finite_objective_or_gradient_proposed", "non_descent_search_direction",
    "linesearch_a_max_overflow", "linesearch_max_iters_reached", "zoom_max_iters_reached",
    "accepted_non_finite_iterate", "cannot_find_initial_feasible_step", "max_step_length_reached",
    "cannot_find_feasible_step", "non_finite_step_proposed", "proposed_step_same_as_current_step",
    "step_bracket_precision_issue")


class BatchedResults:
    """Per-problem Results fields (types.jl:107-114) of a batched run, as arrays."""

    def __init__(self, objective, minimizer, grad_norm, iters_ran, status_code, fdf_evals):
        self.objective, self.minimizer, self.grad_norm = objective, minimizer, grad_norm
        self.iters_ran, self.status_code, self.fdf_evals = iters_ran, status_code, fdf_evals

    @property
    def status(self):
        return [STATUS_SYMBOLS[c] for c in self.status_code]


def batched_lanes(n: int) -> int:
    """Lanes (CTA size) the batched kernel gives a problem of dimension n: its reductions follow the
    canonical order with this many lanes and one tile (include/cgoptim.h)."""
    nw, npt = C.c_int32(), C.c_int32()
    check(lib().cgo_batched_layout(int(n), C.byref(nw), C.byref(npt)))
    return 32 * nw.value


def minimizeobjective_batched(x_initial, config, linesearch_config, ctx: Optional[Context] = None,
                              want_minimizer: bool = True) -> BatchedResults:
    """`minimizeobjective` (src/engine/optim.jl:6-171) for MANY independent extended-Rosenbrock
    problems at once (BASELINE.json configs[4]): `x_initial` is (nprob, n), one CTA solves one
    problem entirely on the device — any of the four CG flavours (cg_flavours.jl) with any of the
    line searches (StrongWolfeBisection, WolfeBisection{Wolfe | YuanWeiLuWolfe},
    Backtracking{Armijo}) — no communication between problems."""
    from .cg_flavours import HagerZhang, LiuStorrey, SallehAlhawarat, YuanWangSheng
    from .linesearch.geometric import Armijo, Backtracking
    from .linesearch.nocedal import StrongWolfeBisection
    from .linesearch.wolfe import Wolfe, WolfeBisection, YuanWeiLuWolfe
    ctx = ctx or default_context()
    X0 = np.ascontiguousarray(x_initial, dtype=np.float64)
    if X0.ndim != 2:
        raise ValueError("x_initial must be (nprob, n)")
    nprob, n = X0.shape
    β = config.β_config
    flav = {HagerZhang: 0, YuanWangSheng: 1, SallehAlhawarat: 2, LiuStorrey: 3}.get(type(β))
    if flav is None:
        raise TypeError(f"the batched solver has no {type(β).__name__} flavour")
    ls = linesearch_config
    bc = capi.BatchedConfig(eps=config.ϵ, max_iters=config.max_iters, flavour=flav, mu=getattr(β, "μ", 0.0),
                            c1=0.0, c2=0.0, growth=2.0, ls_max_iters=getattr(ls, "max_iters", 0), zoom_max_iters=0,
                            delta1=0.0, max_step_size=0.0, discount=0.5, feas_max_iters=0)
    if isinstance(ls, StrongWolfeBisection):
        bc.linesearch, bc.c1, bc.c2, bc.growth = 0, ls.c1, ls.c2, ls.a_max_growth_factor
        bc.zoom_max_iters = ls.zoom_max_iters
    elif isinstance(ls, WolfeBisection) and isinstance(ls.condition, (Wolfe, YuanWeiLuWolfe)):
        bc.linesearch = 2 if isinstance(ls.condition, YuanWeiLuWolfe) else 1
        bc.c1, bc.c2, bc.delta1 = ls.condition.c1, ls.condition.c2, getattr(ls.condition, "δ1", 0.0)
        bc.max_step_size, bc.feas_max_iters = ls.max_step_size, ls.feasibility_max_iters
    elif isinstance(ls, Backtracking) and isinstance(ls.condition, Armijo):
        bc.linesearch, bc.c1, bc.discount = 3, ls.condition.c1, ls.discount_factor
        bc.feas_max_iters = ls.feasibility_max_iters
    else:
        raise TypeError(f"no batched linesearch! method for {type(ls).__name__}")
    obj, gn = np.empty(nprob), np.empty(nprob)
    it, ev = np.empty(nprob, dtype=np.int64), np.empty(nprob, dtype=np.int64)
    st = np.empty(nprob, dtype=np.int32)
    xm = np.empty((nprob, n)) if want_minimizer else None
    check(lib().cgo_batched_minimize_rosenbrock(
        ctx.h, nprob, n, dptr(X0.reshape(-1)), C.byref(bc), dptr(obj), it.ctypes.data, st.ctypes.data,
        ev.ctypes.data, dptr(xm.reshape(-1)) if want_minimizer else None, dptr(gn)))
    return BatchedResults(obj, xm, gn, it, st, ev)
