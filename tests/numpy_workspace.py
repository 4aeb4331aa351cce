"""TEST-ONLY numpy stand-in for DeviceLineSearchContainer.

Lets the host mirror (engine, line searches, β flavours) be checked against the C oracle on a
machine without a GPU.  It is NOT shipped and NOT a CPU fallback: the product package cannot
reach this module (it lives in tests/ and computes with the oracle's own fdf and canonical
sums)."""
from __future__ import annotations

import numpy as np

from oracle import oracle as O

f64 = np.float64
P_PHI, P_DPHI, P_GPGP, P_YY, P_UY, P_YGP, P_GPG, P_UG, P_UU = range(9)


class _Vec:
    def __init__(self, ws, name):
        self.ws, self.name = ws, name


class NumpyObjective:
    def __init__(self, oracle_objective, sum_mode="cgo"):
        self.o = oracle_objective
        self.sum_mode = sum_mode
        self.o.set_sum_mode(sum_mode)
        self.n_local = self.o.n

    def make_workspace(self, x_initial, lbfgs_m=0, fuse_direction=True, beta_form="fused"):
        return NumpyWorkspace(self, x_initial, lbfgs_m, fuse_direction, beta_form)


class NumpyBoxBarrier(NumpyObjective):
    """numpy stand-in of BoxBarrierGPU (the oracle's box_barrier objective)"""

    def __init__(self, f0: NumpyObjective, lbs, ubs, t=1.0):
        self.f0, self.lbs, self.ubs = f0, np.asarray(lbs, dtype=np.float64), np.asarray(ubs, dtype=np.float64)
        super().__init__(O.Objective.box_barrier(f0.o, self.lbs, self.ubs, t), f0.sum_mode)

    def set_t(self, t):
        self.o.set_t(t)

    def infeasible_count(self, x):
        x = np.asarray(x, dtype=np.float64)
        return int(np.sum((x - self.ubs >= 0.0) | (self.lbs - x >= 0.0)))

    def close(self):
        pass


class NumpyWorkspace:
    def __init__(self, obj, x_initial, lbfgs_m, fuse_direction, beta_form):
        self.obj, self.o = obj, obj.o
        self.n = self.o.n
        self.beta_form = beta_form
        self.fuse_direction = fuse_direction
        self.sm = obj.sum_mode
        self.site = self.o.trial_site()
        if hasattr(x_initial, "ws"):          # DeviceStart: the iterate of a live workspace
            x_initial = x_initial.ws.x_
        self.x_ = np.array(x_initial, dtype=np.float64)
        f, g = self.o.fdf(self.x_)
        self.g_ = g
        self.u_ = np.zeros(self.n)
        self.xp_ = self.x_.copy()
        self.gp_ = g.copy()
        self.f_x0 = f64(f)
        self.norm_df_x0 = np.sqrt(f64(self._tdot(g, g)))
        self.pack = np.zeros(16)
        self.dpack = np.zeros(2)
        self._pending = None
        self.xp, self.df_xp, self.x, self.u, self.df_x = (_Vec(self, n) for n in ("xp", "df_xp", "x", "u", "df_x"))
        self.m = lbfgs_m
        # a ring of m + 1 slots: a pair is staged into the one no live pair occupies
        self.S, self.Y, self.rho = [None] * (lbfgs_m + 1), [None] * (lbfgs_m + 1), [0.0] * (lbfgs_m + 1)
        self.count, self.head, self.gamma, self.staged = 0, 0, 1.0, -1

    def _bdot(self, a, b):
        O.set_site(2, 4)
        return O.dot(a, b, self.sm)

    def _tdot(self, a, b):
        O.set_site(*self.site)
        r = O.dot(a, b, self.sm)
        O.set_site(2, 4)
        return r

    def _dirpack(self):
        self.dpack = np.array([self._bdot(self.g_, self.u_), self._bdot(self.u_, self.u_)])

    def reset_direction(self):
        self._pending = None
        self.u_ = -self.g_
        self._dirpack()

    def update_dir(self, β):
        self._pending = float(β)      # applied lazily like the fused device path (same bits)

    def hint_first_trial(self, a):
        pass

    def _mat(self):
        if self._pending is not None:
            β, self._pending = self._pending, None
            self.u_ = -self.g_ + β * self.u_
            self._dirpack()

    def dot_g_u(self):
        self._mat()
        return f64(self.dpack[0])

    def dot_u_u(self):
        self._mat()
        return f64(self.dpack[1])

    def norm_u_plus_g(self):
        self._mat()
        t = self.u_ + self.g_
        return np.sqrt(f64(self._bdot(t, t)))

    def eval_trial(self, a):
        self._mat()
        a = float(a)
        self.xp_ = self.x_ + a * self.u_
        with np.errstate(all="ignore"):
            f, gp = self.o.fdf(self.xp_)
            self.gp_ = gp
            y = gp - self.g_
            P = self.pack = np.zeros(16)
            P[P_PHI] = f
            P[P_DPHI] = self._tdot(gp, self.u_)
            P[P_GPGP] = self._tdot(gp, gp)
            P[P_YY] = self._tdot(y, y)
            P[P_UY] = self._tdot(self.u_, y)
            P[P_YGP] = self._tdot(y, gp)
            P[P_GPG] = self._tdot(gp, self.g_)
            P[P_UG] = self._tdot(self.u_, self.g_)
            P[P_UU] = self._tdot(self.u_, self.u_)
        return f64(P[P_PHI]), f64(P[P_DPHI])

    def norm_df_xp(self):
        return np.sqrt(f64(self.pack[P_GPGP]))

    # solvesystem (src/engine/solve_system.jl): same call shapes as DeviceLineSearchContainer
    def solvesys_begin(self):
        self.xn_ = self.x_.copy()

    def solvesys_project(self, m, fix_stale_iterate=False):
        self._mat()
        base = self.x_ if fix_stale_iterate else self.xn_
        with np.errstate(all="ignore"):
            self.xn_ = base + float(m) * self.gp_
        x_saved, self.x_ = self.x_, self.xn_
        f, _ = self.eval_trial(0.0)          # xp = x_next + 0·u, like the device path
        self.x_ = x_saved
        return f, self.norm_df_xp()

    def solvesys_accept(self, fix_stale_iterate=False):
        self.accept()
        if not fix_stale_iterate:
            self.xn_ = self.xp_.copy()       # the old x

    def dot_df_xp_u(self):
        return f64(self.pack[P_DPHI])

    def download_trial(self):
        return self.xp_.copy(), self.gp_.copy()

    def beta_literal(self, R, m):
        with np.errstate(all="ignore"):
            y = self.gp_ - self.g_
            tmp2 = self.gp_ / R
            tmp1 = y - m * self.u_
            return f64(self._bdot(tmp1, tmp2))

    def accept(self):
        self.x_old = self.x_
        self.x_, self.xp_ = self.xp_, self.x_
        self.g_, self.gp_ = self.gp_, self.g_

    # L-BFGS (staging happens before accept: xp_ is the new point, x_ the old)
    def lbfgs_stage_pair(self):
        slot = (self.head + 1) % (self.m + 1)
        self.S[slot] = self.xp_ - self.x_
        self.Y[slot] = self.gp_ - self.g_
        self.staged = slot
        return f64(self._bdot(self.S[slot], self.Y[slot])), f64(self._bdot(self.Y[slot], self.Y[slot]))

    def lbfgs_commit_pair(self, commit, rho=0.0, gamma=1.0):
        if commit:
            self.head = self.staged
            self.count = min(self.count + 1, self.m)
            self.rho[self.staged] = float(rho)
            self.gamma = float(gamma)
        self.staged = -1             # a rejected pair leaves the history unchanged

    def lbfgs_update_dir(self):
        self._pending = None
        if self.count == 0:
            return self.reset_direction()
        q = self.g_.copy()
        alpha = {}
        slots = [(self.head - k) % (self.m + 1) for k in range(self.count)]
        for s in slots:
            alpha[s] = self.rho[s] * self._bdot(self.S[s], q)
            q = q - alpha[s] * self.Y[s]
        q = self.gamma * q
        for s in reversed(slots):
            be = self.rho[s] * self._bdot(self.Y[s], q)
            q = q + self.S[s] * (alpha[s] - be)
        self.u_ = -q
        self._dirpack()

    def download(self):
        return self.x_.copy(), self.g_.copy()

    def download_vector(self, name):
        self._mat()
        return {"x": self.x_, "df_x": self.g_, "u": self.u_, "xp": self.xp_, "df_xp": self.gp_}[name].copy()

    def close(self):
        pass
