"""Quasi-Newton direction plugin — the slot of src/qn_flavours.jl.

The reference's `BroydenFamily` (qn_flavours.jl:53-90) keeps a dense n×n matrix, costs O(n³) per
iteration and, because it sets `s = B\\y` (:81), is a mathematical no-op (SURVEY.md §0): the matrix is
not built; `BroydenFamily` below is kept as what that update computes.  `LBFGS(m)` is the new flavour behind the same four-method plugin interface
(initializeβ, initializeLineSearchContainer!, getβ, updatedir!): textbook two-loop recursion
(Nocedal & Wright Alg. 7.4/7.5) over the m stored (s, y) pairs, s = xp − x, y = g⁺ − g,
H₀ = (s·y / y·y) I, pair kept only when s·y > 0; a rejected pair leaves the history unchanged.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .cg_flavours import LBFGSHistoryToken
from .cg_types import QNβConfig

f64 = np.float64


@dataclass(frozen=True)
class LBFGS(QNβConfig):
    m: int = 10

    def __post_init__(self):
        assert 1 <= self.m <= 64


def getβ_lbfgs(β_config: LBFGS, ws) -> LBFGSHistoryToken:
    """Called at optim.jl:130, i.e. before x ← xp: stage (s, y) from (xp − x, g⁺ − g)."""
    sy, yy = ws.lbfgs_stage_pair()
    with np.errstate(all="ignore"):
        if sy > 0.0:
            ws.lbfgs_commit_pair(True, f64(1.0) / sy, sy / yy)
        else:
            ws.lbfgs_commit_pair(False)
    return LBFGSHistoryToken()


@dataclass(frozen=True)
class BroydenFamily(QNβConfig):
    """The reference's quasi-Newton config (qn_flavours.jl:53-62), kept so that code written against it still runs.
    Its update sets `s = B\\y` (:81), which makes `B_new − B` vanish identically (`Bs = y` ⇒ `−Bs Bsᵀ/sᵀBs + y yᵀ/sᵀy
    = 0`, and v = 0): B stays the identity it starts as, and `u = B\\(−g)` (:13-19) is the steepest-descent
    direction (SURVEY.md §0; verified numerically there to O(1e-16)).  The dense n×n matrix with its O(n³)
    factorisation per iteration is therefore not built here: this flavour returns β = 0, i.e. u = −g, which is
    what the reference computes.  Use LBFGS(m) for an actual quasi-Newton direction."""
    θ: float = 0.0
    N: int = 0


def setupBroydenFamily(θ, N: int) -> BroydenFamily:
    """qn_flavours.jl:55-62 (only the lower bound on θ is asserted there: `@assert zero(T) <= θ #<= one(T)`)"""
    assert 0.0 <= θ
    return BroydenFamily(float(θ), int(N))
