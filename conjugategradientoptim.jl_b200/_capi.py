"""ctypes binding of libcgoptim.so (include/cgoptim.h).

This is the Python twin of julia/capi.jl: the same symbols a Julia host `ccall`s.  There is no
CPU fallback: if the library is missing, or no CUDA device is present, calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcgoptim.so")
PACK_LEN = 16
# pack indices (include/cgoptim.h)
P_PHI, P_DPHI, P_GPGP, P_YY, P_UY, P_YGP, P_GPG, P_UG, P_UU, P_DIR_GU, P_DIR_UU, P_XPXP = range(12)
D_GU, D_UU = 0, 1

_lib = None


class CgoError(RuntimeError):
    """CUDA / NCCL / argument error reported by libcgoptim (never a numerical status)."""


class BatchedConfig(C.Structure):
    _fields_ = [
        ("eps", C.c_double), ("max_iters", C.c_int64), ("flavour", C.c_int32), ("linesearch", C.c_int32),
        ("mu", C.c_double), ("c1", C.c_double), ("c2", C.c_double), ("growth", C.c_double),
        ("ls_max_iters", C.c_int64), ("zoom_max_iters", C.c_int64),
        ("delta1", C.c_double), ("max_step_size", C.c_double), ("discount", C.c_double),
        ("feas_max_iters", C.c_int64),
    ]


USER_FDF = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p)
_dp = C.POINTER(C.c_double)
_vp = C.c_void_p
_SIGS = {
    # name: (restype, argtypes)
    "cgo_last_error": (C.c_char_p, []),
    "cgo_version": (C.c_int, []),
    "cgo_ctx_create": (C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    "cgo_ctx_destroy": (C.c_int, [_vp]),
    "cgo_ctx_stream": (C.c_int, [_vp, C.POINTER(_vp)]),
    "cgo_ctx_set_reduction_ctas": (C.c_int, [_vp, C.c_int]),
    "cgo_ctx_set_gather_block_bytes": (C.c_int, [_vp, C.c_int64]),
    "cgo_ctx_set_csr_mode": (C.c_int, [_vp, C.c_int]),
    "cgo_ctx_trim_pools": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "cgo_ctx_sm_count": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "cgo_ctx_kernel_launches": (C.c_int, [_vp, C.POINTER(C.c_int64)]),
    "cgo_ctx_timing": (C.c_int, [_vp, C.c_int]),
    "cgo_ctx_timing_read": (C.c_int, [_vp, _dp, C.POINTER(C.c_int64), C.c_int]),
    "cgo_comm_get_unique_id": (C.c_int, [_vp]),
    "cgo_ctx_comm_init": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "cgo_ctx_barrier": (C.c_int, [_vp]),
    "cgo_ctx_peer_memory": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "cgo_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp)]),
    "cgo_host_free": (C.c_int, [_vp]),
    "cgo_shard_range": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "cgo_obj_user_create": (C.c_int, [_vp, C.c_int64, USER_FDF, _vp, C.POINTER(_vp)]),
    "cgo_obj_rosenbrock_create": (C.c_int, [_vp, C.c_int64, C.POINTER(_vp)]),
    "cgo_obj_rosenbrock_chained_create": (C.c_int, [_vp, C.c_int64, C.POINTER(_vp)]),
    "cgo_obj_sparse_ls_create_synthetic": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_uint64, C.c_int32, C.POINTER(_vp)]),
    "cgo_obj_sparse_ls_create_csr": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "cgo_obj_logreg_create_synthetic": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int32, C.c_uint64, C.c_double, C.POINTER(_vp)]),
    "cgo_obj_logreg_create_csr": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, C.c_double, C.POINTER(_vp)]),
    "cgo_obj_softmax_create_csr": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int32, _vp, _vp, _vp, _vp, C.c_double, C.POINTER(_vp)]),
    "cgo_obj_logreg_create_csr_ex": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp, C.c_int32, C.c_double,
                                               C.POINTER(_vp)]),
    "cgo_obj_softmax_create_csr_ex": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int32, _vp, _vp, _vp, _vp, _vp, C.c_int32,
                                                C.c_double, C.POINTER(_vp)]),
    "cgo_obj_box_barrier_create": (C.c_int, [_vp, _vp, _dp, _dp, C.c_double, C.POINTER(_vp)]),
    "cgo_obj_barrier_set_t": (C.c_int, [_vp, C.c_double]),
    "cgo_obj_barrier_infeasible": (C.c_int, [_vp, _dp, C.POINTER(C.c_int64)]),
    "cgo_obj_destroy": (C.c_int, [_vp]),
    "cgo_obj_dims": (C.c_int, [_vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "cgo_obj_reduction_site": (C.c_int, [_vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "cgo_obj_bytes_per_eval": (C.c_int, [_vp, _dp]),
    "cgo_obj_default_x0": (C.c_int, [_vp, C.c_uint64, C.c_double, _dp]),
    "cgo_obj_csr_nnz": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "cgo_obj_csr_blocks": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_int32)]),
    "cgo_obj_csr_download": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp]),
    "cgo_obj_spmv": (C.c_int, [_vp, C.c_int, _dp, _dp]),
    "cgo_state_create": (C.c_int, [_vp, _vp, _dp, C.c_int32, C.POINTER(_vp), _dp]),
    "cgo_state_create_from_state": (C.c_int, [_vp, _vp, _vp, C.c_int32, C.c_int32, C.POINTER(_vp), _dp]),
    "cgo_state_destroy": (C.c_int, [_vp]),
    "cgo_reset_direction": (C.c_int, [_vp, _dp]),
    "cgo_eval_trial": (C.c_int, [_vp, C.c_double, _dp]),
    "cgo_eval_trial_fused_dir": (C.c_int, [_vp, C.c_double, C.c_double, _dp]),
    "cgo_accept": (C.c_int, [_vp]),
    "cgo_update_dir": (C.c_int, [_vp, C.c_double, _dp]),
    "cgo_beta_literal": (C.c_int, [_vp, C.c_double, C.c_double, _dp]),
    "cgo_norm_sq_u_plus_g": (C.c_int, [_vp, _dp]),
    "cgo_lbfgs_stage_pair": (C.c_int, [_vp, _dp]),
    "cgo_lbfgs_commit_pair": (C.c_int, [_vp, C.c_int32, C.c_double, C.c_double]),
    "cgo_lbfgs_update_dir": (C.c_int, [_vp, _dp]),
    "cgo_solvesys_begin": (C.c_int, [_vp]),
    "cgo_solvesys_project": (C.c_int, [_vp, C.c_double, C.c_int32, _dp]),
    "cgo_solvesys_accept": (C.c_int, [_vp, C.c_int32]),
    "cgo_hessvec_dir": (C.c_int, [_vp, _dp]),
    "cgo_quad_begin": (C.c_int, [_vp, _dp]),
    "cgo_quad_accept": (C.c_int, [_vp, C.c_double, _dp]),
    "cgo_download": (C.c_int, [_vp, _dp, _dp]),
    "cgo_download_vector": (C.c_int, [_vp, C.c_int32, _dp]),
    "cgo_batched_layout": (C.c_int, [C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "cgo_batched_minimize_rosenbrock": (C.c_int, [_vp, C.c_int64, C.c_int32, _dp, C.POINTER(BatchedConfig), _dp, _vp, _vp, _vp, _dp, _dp]),
}
EXPORTED_SYMBOLS = sorted(_SIGS)


def lib():
    """Load libcgoptim.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CgoError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (nvcc, sm_100a).  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (rt, at) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = rt
            fn.argtypes = at
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise CgoError(f"libcgoptim error {rc}: {lib().cgo_last_error().decode(errors='replace')}")


class _PinnedBlock:
    """Owner of one cudaHostAlloc block.  Page-locking is slow (~1 s per GB), so a block whose
    last numpy view died goes back to a small free list and is handed out again by the next
    `pinned_empty` of the same size (Results of successive runs reuse the same host pages)."""
    POOL: dict = {}                  # nbytes -> [ptr, ...]
    POOL_BYTES = 0
    POOL_CAP = 16 << 30              # retained bytes; beyond it blocks are freed

    def __init__(self, nbytes: int):
        free = _PinnedBlock.POOL.get(nbytes)
        if free:
            self.ptr = free.pop()
            _PinnedBlock.POOL_BYTES -= nbytes
        else:
            p = C.c_void_p()
            check(lib().cgo_host_alloc(nbytes, C.byref(p)))
            self.ptr = p
        self.nbytes = nbytes

    def __del__(self):
        try:
            if self.ptr:
                if _PinnedBlock.POOL_BYTES + self.nbytes <= _PinnedBlock.POOL_CAP:
                    _PinnedBlock.POOL.setdefault(self.nbytes, []).append(self.ptr)
                    _PinnedBlock.POOL_BYTES += self.nbytes
                else:
                    lib().cgo_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def pinned_empty(n: int) -> np.ndarray:
    """float64 vector in page-locked host memory (device<->host copies run at PCIe speed)."""
    blk = _PinnedBlock(8 * max(int(n), 1))
    buf = (C.c_double * max(int(n), 1)).from_address(blk.ptr.value)
    buf._cgo_owner = blk                   # the numpy array keeps `buf` (its base) alive, `buf` the block
    return np.frombuffer(buf, dtype=np.float64, count=int(n))


def pinned_pool_clear():
    """Free every retained page-locked block."""
    for ptrs in _PinnedBlock.POOL.values():
        for p in ptrs:
            lib().cgo_host_free(p)
    _PinnedBlock.POOL.clear()
    _PinnedBlock.POOL_BYTES = 0


def dptr(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags.c_contiguous
    return a.ctypes.data_as(_dp)
