"""Reference of multinomial (softmax) logistic regression on a host CSR (test infrastructure): f and g of
`SoftmaxRegGPU_from_csr`.

W is nfeat × K, stored feature-major (w[j·K + k]).  Z = A W is the SpMV of the Kronecker-expanded matrix A ⊗ I_K on
the flat W: its row (i, k) holds row i's entries in storage order at columns col·K + k.  Aᵀ C is likewise the SpMV
of the transpose of that matrix, whose rows keep the storage order of Aᵀ.  So every row sum comes from
`LogRegCSR.spmv` on the expanded matrix, long-row rule at site (2, 4) included.  The loss and C follow the kernel's
order with `math.exp` / `math.log`; the loss is reduced like the binary loss at site (2, 4), and ‖W‖² like the binary
reference reduces ‖w‖².

`SoftmaxCSR` has the interface of `oracle.Objective` (n, fdf, set_sum_mode, trial_site, set_trial_site, csr, rhs,
spmv), so whole runs go through the host mirror of the engine (`numpy_workspace`)."""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle as O

from logreg_csr_reference import LogRegCSR


def kron_csr(nrows, rowptr, col, val, K):
    """(rowptr, col, val) of A ⊗ I_K: row i·K + k holds row i's entries in storage order at columns col·K + k"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    col = np.asarray(col, dtype=np.int64)
    val = np.asarray(val, dtype=np.float64)
    lens = np.repeat(np.diff(rowptr), K)
    rp = np.zeros(nrows * K + 1, dtype=np.int64)
    np.cumsum(lens, out=rp[1:])
    erow = np.repeat(np.arange(nrows * K, dtype=np.int64), lens)
    p = rowptr[erow // K] + (np.arange(rp[-1], dtype=np.int64) - rp[erow])
    return rp, (col[p] * K + erow % K).astype(np.int64), val[p]


def softmax_rows(Z, y, K):
    """(ℓ, C) from Z (N·K, row-major) in the kernel's order: m = max_k z_k, s = Σ exp(z_k − m) from +0.0,
    ℓ = (m + log s) − z_y, c_k = exp(z_k − m) / s − [k = y]"""
    N = y.size
    loss, C = np.empty(N), np.empty(N * K)
    for i in range(N):
        z = [float(v) for v in Z[i * K:(i + 1) * K]]
        lab = int(y[i])
        m = z[0]
        for v in z[1:]:
            m = v if v > m else m
        s = 0.0
        for v in z:
            s = s + math.exp(v - m)
        loss[i] = (m + math.log(s)) - z[lab]
        for k in range(K):
            p = math.exp(z[k] - m) / s
            C[i * K + k] = p - 1.0 if k == lab else p
    return loss, C


class SoftmaxCSR:
    """(1/N) Σ_i [logsumexp(a_i W) − (a_i W)_{y_i}] + (λ/2)‖W‖² on a host CSR, labels in [0, K)"""

    def __init__(self, nsamples, nfeat, nclasses, rowptr, col, val, labels, lam=1e-6):
        self.nrows, self.nfeat, self.K, self.lam = int(nsamples), int(nfeat), int(nclasses), float(lam)
        self.n = self.nfeat * self.K
        self.rowptr = np.array(rowptr, dtype=np.int64)
        self.col = np.array(col, dtype=np.int32)
        self.val = np.array(val, dtype=np.float64)
        self.y = np.array(labels, dtype=np.int64)
        erp, ecol, evl = kron_csr(self.nrows, self.rowptr, self.col, self.val, self.K)
        self.E = LogRegCSR(self.nrows * self.K, self.n, erp, ecol, evl, np.ones(self.nrows * self.K), lam)
        self.sum_mode = "seq"
        self.set_trial_site(2, 4)

    # the oracle.Objective interface
    def set_sum_mode(self, sum_mode="seq", threads=0):
        self.sum_mode = sum_mode

    def trial_site(self):
        return self.E.trial_site()

    def set_trial_site(self, V, U):
        self.E.set_trial_site(V, U)

    def csr(self, transposed=False):
        """A or Aᵀ (not expanded), as the GPU objective's download returns them"""
        if transposed:
            from logreg_csr_reference import transpose
            return transpose(self.nrows, self.nfeat, self.rowptr, self.col, self.val)
        return self.rowptr.copy(), self.col.copy(), self.val.copy()

    def rhs(self):
        return self.y.astype(np.float64)

    def spmv(self, x, transposed=False):
        """Z = A W (nfeat·K → N·K) or Aᵀ C (N·K → nfeat·K)"""
        return self.E.spmv(x, transposed)

    def loss_and_c(self, w):
        return softmax_rows(self.spmv(np.ascontiguousarray(w, dtype=np.float64)), self.y, self.K)

    def fdf(self, w):
        w = np.ascontiguousarray(w, dtype=np.float64)
        N = self.nrows
        lp, C = self.loss_and_c(w)
        if self.sum_mode == "cgo":
            O.set_site(2, 4)
            loss = O.dot(lp, np.ones(N), "cgo")
        else:
            loss = O.dot(lp, np.ones(N), self.sum_mode)
        loss = loss / float(N)
        g = self.spmv(C, transposed=True)
        O.set_site(2, 4)                                         # W·W is reduced by the BLAS-1 kernel K_a
        ww = O.dot(w, w, self.sum_mode)
        g = g * (1.0 / float(N)) + self.lam * w
        return loss + (0.5 * self.lam) * ww, g
