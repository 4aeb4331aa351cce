"""Reference of logistic and softmax regression with per-sample weights and an unpenalised intercept on a host CSR
(test infrastructure): f and g of `LogRegGPU_from_csr` / `SoftmaxRegGPU_from_csr` with `sample_weight` and
`fit_intercept`, restating the arithmetic contract of include/cgoptim.h.

- Margins: the row sums of A exactly as the references without the options compute them (`LogRegCSR.spmv`, long
  rows included), then z_i + b (z_ik + b_k).
- Loss: s_i·ℓ_i reduced at site (2, 4); c_i = s_i·(−y_i σ_i), c_ik = s_i·(p_ik − [k = y_i]).
- Intercept gradient: the unit row, a row of Aᵀ with entry 1.0 at every sample, summed in the long-row order (the
  oracle's `dot` at site (1, 4)) whatever N is.
- Scaling: invS = 1.0 / S with S = math.fsum(s); a feature's gradient is q_j·invS + λ w_j, an intercept's q_j·invS;
  f = Σ/S + (λ/2)·P, where P is the site-(2, 4) dot of the state with itself with every intercept coordinate zeroed
  (each contributes +0.0 instead of its square).

Both classes have the interface of `oracle.Objective` (n, fdf, set_sum_mode, trial_site, set_trial_site, csr, rhs,
spmv), so whole runs go through the host mirror of the engine (`numpy_workspace`)."""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle as O

from logreg_csr_reference import LogRegCSR
from softmax_csr_reference import SoftmaxCSR, softmax_rows


def _weights(N, sample_weight):
    s = np.ones(N) if sample_weight is None else np.array(sample_weight, dtype=np.float64)
    assert s.shape == (N,)
    return s, (float(N) if sample_weight is None else math.fsum(s))


def unit_row_sum(c):
    """Σ_i 1.0 · c_i in the long-row order (V = 1, U = 4, the oracle's G)"""
    O.set_site(1, 4)
    q = O.dot(np.ones(c.size), np.ascontiguousarray(c, dtype=np.float64), "cgo")
    O.set_site(2, 4)
    return q


class _Glm:
    """what the binary and the softmax objectives share: sum mode, site, weights, scaling, P"""

    def _init_glm(self, N, nfeat, K, lam, sample_weight, fit_intercept):
        self.nrows, self.nfeat, self.K, self.lam = int(N), int(nfeat), int(K), float(lam)
        self.icpt = bool(fit_intercept)
        self.npen = self.nfeat * self.K
        self.n = self.npen + (self.K if self.icpt else 0)
        self.s, self.S = _weights(self.nrows, sample_weight)
        self.sum_mode = "seq"

    def set_sum_mode(self, sum_mode="seq", threads=0):
        self.sum_mode = sum_mode

    def trial_site(self):
        return (2, 4)

    def set_trial_site(self, V, U):
        assert (V, U) == (2, 4), "the objective runs on k_spmv_direct / the SpMM only"

    def _reduce(self, lp):
        O.set_site(2, 4)
        return O.dot(lp, self.s, self.sum_mode)

    def _finish(self, x, loss, q):
        """f and g from the weighted loss sum and q (Aᵀc, then the intercept sums)"""
        O.set_site(2, 4)                                       # P is reduced by the BLAS-1 kernel K_a
        xm = x.copy()
        xm[self.npen:] = 0.0
        P = O.dot(xm, xm, self.sum_mode)
        invS = 1.0 / self.S
        g = q * invS
        g[:self.npen] = g[:self.npen] + self.lam * x[:self.npen]
        return loss / self.S + (0.5 * self.lam) * P, g


class LogRegGlmCSR(_Glm):
    """(1/S) Σ s_i log(1 + exp(−y_i (a_i·w + b))) + (λ/2)‖w‖² on a host CSR; state (w[, b])"""

    def __init__(self, nsamples, nfeat, rowptr, col, val, y, lam=1e-6, sample_weight=None, fit_intercept=False):
        self._init_glm(nsamples, nfeat, 1, lam, sample_weight, fit_intercept)
        self.base = LogRegCSR(nsamples, nfeat, rowptr, col, val, y, lam)
        self.base.set_trial_site(2, 4)
        self.y = self.base.y

    def csr(self, transposed=False):
        return self.base.csr(transposed)

    def rhs(self):
        return self.y.copy()

    def spmv(self, x, transposed=False):
        """A times the feature part, or (Aᵀ c, the intercept's sum): what `DeviceObjective.spmv` returns"""
        if not transposed:
            return self.base.spmv(np.ascontiguousarray(x, dtype=np.float64)[:self.nfeat])
        q = self.base.spmv(x, True)
        return np.append(q, unit_row_sum(x)) if self.icpt else q

    def loss_and_c(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        z = self.spmv(x)
        if self.icpt:
            z = z + x[self.nfeat]
        lp, c = np.empty(self.nrows), np.empty(self.nrows)
        for i in range(self.nrows):
            yi, si = float(self.y[i]), float(self.s[i])
            t = -yi * float(z[i])
            e = math.exp(-abs(t))
            lp[i] = (t if t > 0.0 else 0.0) + math.log1p(e)
            sg = 1.0 / (1.0 + e) if t >= 0.0 else e / (1.0 + e)
            c[i] = si * (-yi * sg)
        return lp, c

    def fdf(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        lp, c = self.loss_and_c(x)
        return self._finish(x, self._reduce(lp), self.spmv(c, True))


class SoftmaxGlmCSR(_Glm):
    """(1/S) Σ_i s_i [logsumexp(a_i W + b) − (a_i W + b)_{y_i}] + (λ/2)‖W‖² on a host CSR; state W[, b] feature-major"""

    def __init__(self, nsamples, nfeat, nclasses, rowptr, col, val, labels, lam=1e-6, sample_weight=None,
                 fit_intercept=False):
        self._init_glm(nsamples, nfeat, nclasses, lam, sample_weight, fit_intercept)
        self.base = SoftmaxCSR(nsamples, nfeat, nclasses, rowptr, col, val, labels, lam)
        self.y = self.base.y

    def csr(self, transposed=False):
        return self.base.csr(transposed)

    def rhs(self):
        return self.base.rhs()

    def spmv(self, x, transposed=False):
        """Z = A W of the feature part, or (Aᵀ C, the K intercept sums)"""
        if not transposed:
            return self.base.spmv(np.ascontiguousarray(x, dtype=np.float64)[:self.npen])
        q = self.base.spmv(x, True)
        if not self.icpt:
            return q
        C = np.ascontiguousarray(x, dtype=np.float64).reshape(self.nrows, self.K)
        return np.concatenate([q, [unit_row_sum(C[:, k]) for k in range(self.K)]])

    def loss_and_c(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        Z = self.spmv(x)
        if self.icpt:
            Z = Z + np.tile(x[self.npen:], self.nrows)
        lp, C = softmax_rows(Z, self.y, self.K)
        return lp, C * np.repeat(self.s, self.K)

    def fdf(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        lp, C = self.loss_and_c(x)
        return self._finish(x, self._reduce(lp), self.spmv(C, True))
