"""Exact references and a-priori error bounds for the device reductions (test infrastructure).

The bit-exact tests compare the kernels with oracle/cgo_oracle.c, which follows the kernels' own reduction tree.
The references here do not: `exact_dot` / `exact_sum` are the correctly rounded values of the fp64 inputs, and
`canonical_bound` is the classical bound γ_{D+1}·Σ|terms| (Higham, Accuracy and Stability, §3.1 and §4.2) on the
error of ANY fp64 summation tree in which no term passes through more than D additions.  D is worked out from the
canonical order of include/cgoptim.h and reduce.cuh, not fitted.  It is tight enough to catch a kernel that drops
or repeats a tile (tests/test_exact_reference.py shows it at every shape of the GPU sweep), even when the oracle
shares the mistake; it is far too loose to notice a reduction tree that is merely somewhat deeper than the spec,
which is what the bit-exact comparison with the oracle is for.
"""
from __future__ import annotations

import math

import numpy as np

U_ROUND = 2.0 ** -53          # unit roundoff of fp64
B = 256                       # lanes per virtual CTA (CGO_B)
T = 2048                      # elements per BLAS-1 tile: B lanes × U = 4 double2 loads × V = 2
_SPLIT = 134217729.0          # 2^27 + 1 (Veltkamp)


def _split(a):
    c = _SPLIT * a
    hi = c - (c - a)
    return hi, a - hi


def _two_products(a, b):
    """p + e == a·b exactly (Dekker's TwoProduct; NumPy does not contract a*b+c into an FMA)"""
    a = np.ascontiguousarray(a, dtype=np.float64).ravel()
    b = np.ascontiguousarray(b, dtype=np.float64).ravel()
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact_dot(a, b) -> float:
    """Σ a_i b_i correctly rounded (|a_i b_i| must stay clear of overflow and of the subnormal range)"""
    p, e = _two_products(a, b)
    return math.fsum(np.concatenate([p, e]))


def exact_sumsq(a) -> float:
    return exact_dot(a, a)


def exact_sum(a) -> float:
    return math.fsum(np.ascontiguousarray(a, dtype=np.float64).ravel())


def _sweep(G, ns):
    return [(G, n) for n in sorted(set(ns))]


# (G, n) at the tiling edges: one tile and a lane's first load (1..3), the tile size T, one tile per virtual CTA
# (G·T), the first wrap back to virtual CTA 0 ((G+1)·T); G = 8192 = CGO_GMAX makes every physical CTA loop over
# ~28 virtual ones.  Even n for the even-only objectives (Rosenbrock), odd n for the CSR ones.  At G = 8192 only
# (G+1)·T of the large sizes: it fills every virtual CTA and wraps, and each 16.8M-element shape costs about 100 s
# of exact host-side sums.
SWEEP_EVEN = [c for G in (1, 2, 3, 296) for c in _sweep(G, [2, T - 2, T, T + 2, G * T, G * T + 2, (G + 1) * T])] + \
    _sweep(8192, [2, T + 2, 8193 * T])
SWEEP_ODD = [c for G in (1, 2, 3, 296) for c in _sweep(G, [1, 3, T - 1, T + 1, G * T - 1, G * T + 1])] + \
    _sweep(8192, [3, T + 1, 4 * T + 1])


def gamma(k: int) -> float:
    return k * U_ROUND / (1.0 - k * U_ROUND)


def canonical_depth(n: int, G: int, site=(2, 4)) -> int:
    """Additions a term can pass through in the canonical reduction of n items at reduction site (V, U):
      - the lane's sequential additions over its tiles: V·U terms per tile, ⌈ntiles/G⌉ tiles;
      - the xor butterfly inside a warp (16, 8, 4, 2, 1): 5;
      - the sequential combine of the 8 warps: 7;
      - the last block's lane t adding partials t, t+256, …: ⌈nact/256⌉;
      - the butterfly and warp combine of that finish: 5 + 7."""
    V, U = site
    nq = -(-n // V)
    ntiles = max(-(-nq // (B * U)), 1)
    nact = min(ntiles, G)
    return V * U * -(-ntiles // G) + 5 + 7 + -(-nact // B) + 5 + 7


def canonical_bound(n: int, G: int, site, terms_abs_sum: float) -> float:
    """|computed − exact| for a canonical-order sum of n items whose terms are rounded once (a product, or an
    elementwise value formed before the sum: one more rounding than the depth)"""
    return gamma(canonical_depth(n, G, site) + 1) * terms_abs_sum


def exact_spmv_rows(rowptr, col, val, x):
    """(A x)_i correctly rounded for every row"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    p, e = _two_products(np.asarray(val, dtype=np.float64), np.asarray(x, dtype=np.float64)[np.asarray(col, dtype=np.int64)])
    out = np.empty(rowptr.size - 1)
    for i in range(out.size):
        lo, hi = rowptr[i], rowptr[i + 1]
        out[i] = math.fsum(np.concatenate([p[lo:hi], e[lo:hi]])) if hi > lo else 0.0
    return out


def exact_spmv_row_bound(rowptr, col, val, x):
    """per-row bound γ_len·Σ_j |a_ij x_j| on the error of any fp64 evaluation of the row sum (a row of `len`
    entries summed sequentially from +0.0: every product is rounded once and passes through at most len − 1
    additions)"""
    rowptr = np.asarray(rowptr, dtype=np.int64)
    ax = np.abs(np.asarray(val, dtype=np.float64) * np.asarray(x, dtype=np.float64)[np.asarray(col, dtype=np.int64)])
    cs = np.concatenate([[0.0], np.cumsum(ax)])
    lens = np.diff(rowptr)
    absrow = cs[rowptr[1:]] - cs[rowptr[:-1]]
    # (the cumulative sum of |terms| is itself rounded: 2× covers it for any length used in the tests)
    return np.array([gamma(int(k)) for k in lens]) * absrow * 2.0


# ---------------------------------------------------------------------------------------------- L-BFGS
def dense_lbfgs_direction(pairs, gam, g):
    """−H g with H the inverse-BFGS matrix of the kept (s, y) pairs (oldest first), H₀ = γ I, built densely in
    np.longdouble by the product form H ← (I − ρ s yᵀ) H (I − ρ y sᵀ) + ρ s sᵀ (Nocedal & Wright (6.17), (7.19))"""
    L = np.longdouble
    n = len(g)
    H = np.eye(n, dtype=L) * L(gam)
    for s, y in pairs:
        s, y = np.asarray(s, dtype=L), np.asarray(y, dtype=L)
        rho = L(1) / (s @ y)
        Hy = H @ y                                   # (H is symmetric)
        yHy = y @ Hy
        H = H - rho * (np.outer(s, Hy) + np.outer(Hy, s)) + (rho * rho * yHy + rho) * np.outer(s, s)
    return -(H @ np.asarray(g, dtype=L))


def drive_lbfgs(ws, m, steps, reject, a):
    """Drives an L-BFGS workspace by hand: trial at step a along u, stage (s, y), commit unless the step index is in
    `reject` (or s·y <= 0), accept, two-loop direction.  After every step the device direction u is compared with the
    dense extended-precision −H g over the pairs the textbook keeps (a rejection leaves them unchanged).
    Returns the relative 2-norm error per step, the history length before each rejection, and, for each rejection
    at count == m, how far (relative 2-norm) the textbook direction moves when the oldest pair is dropped as well:
    the margin by which the error check tells the textbook history from one that loses a pair on a rejection."""
    ws.reset_direction()
    pairs, gam = [], 1.0
    errs, count_at_reject, power = [], [], []
    for k in range(steps):
        x, g = ws.download_vector("x"), ws.download_vector("df_x")
        ws.eval_trial(a)
        xp, gp = ws.download_vector("xp"), ws.download_vector("df_xp")
        sy, yy = ws.lbfgs_stage_pair()
        if k in reject or not sy > 0.0:
            count_at_reject.append(len(pairs))
            ws.lbfgs_commit_pair(False)
        else:
            ws.lbfgs_commit_pair(True, 1.0 / sy, sy / yy)
            s, y = xp - x, gp - g
            pairs = (pairs + [(s, y)])[-m:]
            L = np.longdouble
            gam = (np.asarray(s, L) @ np.asarray(y, L)) / (np.asarray(y, L) @ np.asarray(y, L))
        ws.accept()
        ws.lbfgs_update_dir()
        u = ws.download_vector("u")
        ref = dense_lbfgs_direction(pairs, gam, gp) if pairs else -np.asarray(gp, dtype=np.longdouble)
        nref = np.linalg.norm(ref.astype(np.float64))
        errs.append(float(np.linalg.norm((u - ref).astype(np.float64)) / nref))
        if k in reject and len(pairs) == m:
            lost = dense_lbfgs_direction(pairs[1:], gam, gp) if m > 1 else -np.asarray(gp, dtype=np.longdouble)
            power.append(float(np.linalg.norm((lost - ref).astype(np.float64)) / nref))
    return errs, count_at_reject, power


def well_conditioned_ls(n, seed):
    """a dense n×n least-squares problem with singular values spread geometrically over [1, 10] as CSR
    (rowptr, col, val, b): well conditioned, yet with n > m = 64 and that spread the 64 newest pairs do not pin the
    inverse Hessian, so losing the oldest one moves the direction far above the tests' tolerance"""
    rng = np.random.default_rng(seed)
    q1, _ = np.linalg.qr(rng.standard_normal((n, n)))
    q2, _ = np.linalg.qr(rng.standard_normal((n, n)))
    A = (q1 * np.geomspace(1.0, 10.0, n)) @ q2.T
    rowptr = np.arange(0, n * n + 1, n, dtype=np.int64)
    col = np.tile(np.arange(n, dtype=np.int32), n)
    return rowptr, col, A.ravel().copy(), rng.standard_normal(n)
