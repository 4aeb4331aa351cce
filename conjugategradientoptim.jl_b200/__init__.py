"""conjugategradientoptim.jl_b200 — B200-native hot path of ConjugateGradientOptim.jl.

Host mirror (Python; Julia is not installed in the build image — see julia/ for the Julia twin)
of the reference's public API over the C ABI of include/cgoptim.h.  Export list follows
src/ConjugateGradientOptim.jl:23-29 plus the names the reference reaches qualified
(examples/min.jl:18-43).
"""
from ._capi import CgoError, EXPORTED_SYMBOLS, LIB_PATH  # noqa: F401
from .cg_types import (CGConfig, CGβConfig, DisableTrace, EnableTrace, LineSearchConfig,  # noqa: F401
                       QNβConfig, Results, TraceContainer, TraceTrait, setupCGConfig, setuptrace,
                       βConfig)
from .cg_flavours import (HagerZhang, LiuStorrey, SallehAlhawarat, YuanWangSheng, getβ,  # noqa: F401
                          initializeLineSearchContainer_, initializeβ, updatedir_)
from .qn_flavours import LBFGS, BroydenFamily, setupBroydenFamily  # noqa: F401
from .cg_utils import evalϕdϕ_  # noqa: F401
from .linesearch import (Armijo, Backtracking, StrongWolfeBisection, Wolfe, WolfeBisection,  # noqa: F401
                         YuanWeiLuWolfe, setupStrongWolfeBisection)
from .engine import (BoxConstraint, CvxInequalityConstraint, LinesearchSolveSys, MinimizerRun,  # noqa: F401
                     PrimalBarrierConfig, PrimalBarrierResults, getNconstraints, minimizeobjective,
                     minimizeobjectivererun, primalbarriermethod_, setupCvxInequalityConstraint,
                     setupLinesearchSolveSys, setupPrimalBarrierConfig, solvesystem, verifyt0)
from .engine.optim import linesearch_  # noqa: F401
from .device import (Context, DeviceLineSearchContainer, DeviceObjective, DeviceStart, DeviceVector,  # noqa: F401
                     BoxBarrierGPU, LogRegGPU, LogRegGPU_from_csr, RosenbrockChainedGPU, RosenbrockGPU, SoftmaxRegGPU_from_csr, SparseLSGPU, SparseLSGPU_from_csr, UserObjectiveGPU, default_context,
                     dot, shard_range, BatchedResults, minimizeobjective_batched, batched_lanes)
from .device import DeviceLineSearchContainer as LineSearchContainer  # noqa: F401
