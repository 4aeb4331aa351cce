"""Reference of logistic regression on a host CSR (test infrastructure): f and g of `LogRegGPU_from_csr`, restated
in the arithmetic of the oracle's `logreg_fdf` (oracle/cgo_oracle.c), plus the long-row rule of include/cgoptim.h.

`LogRegCSR` has the interface of `oracle.Objective` that the tests and `numpy_workspace.NumpyObjective` use (n,
fdf, set_sum_mode, trial_site, set_trial_site, csr, rhs, spmv), so whole runs go through the host mirror of the
engine exactly as the oracle's own objectives do.  Every reduction is one of the oracle's (`O.dot`, `O.sum_cgo`), in
the order the oracle uses; `exp` and `log1p` are the C library's (`math`), as in the oracle.

Row sums: each row's products val_k · x[col_k] are added one by one in storage order from +0.0.  At trial site
(2, 4) — the k_spmv_direct family — a row with more than CGO_LONG_ROW entries is instead summed in the canonical
order with V = 1, U = 4 (the oracle's `dot` at site (1, 4), whose terms are exactly those products)."""
from __future__ import annotations

import math
import os
import re

import numpy as np

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def long_row_limit() -> int:
    """CGO_LONG_ROW, read from the public header"""
    with open(os.path.join(ROOT, "include", "cgoptim.h")) as f:
        return int(re.search(r"#define\s+CGO_LONG_ROW\s+(\d+)", f.read()).group(1))


L = long_row_limit()


def transpose(nrows, ncols, rowptr, col, val):
    """stable counting-sort transpose (the oracle's build_transpose): rows of Aᵀ sorted by source entry"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    src = np.repeat(np.arange(nrows, dtype=np.int64), np.diff(rowptr))
    order = np.argsort(col, kind="stable")
    rpT = np.zeros(ncols + 1, dtype=np.int64)
    np.cumsum(np.bincount(col, minlength=ncols), out=rpT[1:])
    return rpT, src[order].astype(np.int32), np.asarray(val, dtype=np.float64)[order]


class LogRegCSR:
    """(1/N) Σ log(1 + exp(−y_i a_i·w)) + (λ/2)‖w‖² on a host CSR"""

    def __init__(self, nsamples, nfeat, rowptr, col, val, y, lam=1e-6):
        self.nrows, self.n, self.lam = int(nsamples), int(nfeat), float(lam)
        self.rowptr = np.array(rowptr, dtype=np.int64)
        self.col = np.array(col, dtype=np.int32)
        self.val = np.array(val, dtype=np.float64)
        self.y = np.array(y, dtype=np.float64)
        self.T = transpose(self.nrows, self.n, self.rowptr, self.col, self.val)
        self.sum_mode, self.site = "seq", (1, 1)

    # the oracle.Objective interface
    def set_sum_mode(self, sum_mode="seq", threads=0):
        self.sum_mode = sum_mode

    def trial_site(self):
        return self.site

    def set_trial_site(self, V, U):
        self.site = (int(V), int(U))

    def csr(self, transposed=False):
        if transposed:
            return tuple(a.copy() for a in self.T)
        return self.rowptr.copy(), self.col.copy(), self.val.copy()

    def rhs(self):
        return self.y.copy()

    def spmv(self, x, transposed=False):
        rp, ci, va = self.T if transposed else (self.rowptr, self.col, self.val)
        x = np.ascontiguousarray(x, dtype=np.float64)
        lens = np.diff(rp)
        split = self.site == (2, 4)
        short = lens <= L if split else np.ones(lens.size, dtype=bool)
        y = np.zeros(lens.size)
        for k in range(int(lens[short].max(initial=0))):       # level k of every short row: storage order
            rows = np.nonzero(short & (lens > k))[0]
            p = rp[rows] + k
            y[rows] = y[rows] + va[p] * x[ci[p]]
        if split:
            O.set_site(1, 4)
            for r in np.nonzero(~short)[0]:
                y[r] = O.dot(va[rp[r]:rp[r + 1]], x[ci[rp[r]:rp[r + 1]]], "cgo")
            O.set_site(2, 4)
        return y

    def fdf(self, w):
        w = np.ascontiguousarray(w, dtype=np.float64)
        N = self.nrows
        z = self.spmv(w)
        lp, c = np.empty(N), np.empty(N)
        for i in range(N):
            yi = float(self.y[i])
            t = -yi * float(z[i])
            e = math.exp(-abs(t))
            lp[i] = (t if t > 0.0 else 0.0) + math.log1p(e)
            sg = 1.0 / (1.0 + e) if t >= 0.0 else e / (1.0 + e)
            c[i] = -yi * sg
        if self.sum_mode == "cgo":
            if self.site[0] == 2:
                O.set_site(2, 4)
                loss = O.dot(lp, np.ones(N), "cgo")
            else:
                loss = O.sum_cgo(lp, U=1, align=2)
        else:
            loss = O.dot(lp, np.ones(N), self.sum_mode)
        loss = loss / float(N)
        g = self.spmv(c, transposed=True)
        O.set_site(2, 4)                                         # w·w is reduced by the BLAS-1 kernel K_a
        ww = O.dot(w, w, self.sum_mode)
        g = g * (1.0 / float(N)) + self.lam * w
        return loss + (0.5 * self.lam) * ww, g
