# B200CGOptim — Julia host of the B200-native hot path of ConjugateGradientOptim.jl.
#
# It ADDS METHODS to the reference package's own generic functions (`minimizeobjective`,
# `minimizeobjectivererun`, `linesearch!`, `getβ`, `updatedir!`, `evalϕdϕ!`, …) for the case where
# `fdf!` is a device-objective handle instead of a closure, and re-uses the reference's own
# config / result types (src/types.jl: CGConfig, Results, TraceContainer, EnableTrace, …; the
# line-search and flavour configs).  Every line that touches a vector in the reference is one
# `ccall` into libcgoptim.so (include/cgoptim.h); all scalar logic stays here in Julia.
#
# STATUS: Julia is not installed in the build image nor on the GPU box, so this package has not
# been executed.  It is kept structurally identical to the Python host
# (conjugategradientoptim.jl_b200/), which IS tested bit-for-bit against the oracle on a B200.
# (Set the `ConjugateGradientOptim` UUID in Project.toml to the one of your checkout.)
module B200CGOptim

import ConjugateGradientOptim
const CGO = ConjugateGradientOptim
import ConjugateGradientOptim: CGConfig, Results, TraceContainer, EnableTrace, DisableTrace,
    LineSearchConfig, βConfig, CGβConfig, QNβConfig, setuptrace, resizetrace!, updatetrace!,
    StrongWolfeBisection, WolfeBisection, Backtracking, Wolfe, YuanWeiLuWolfe, Armijo,
    HagerZhang, YuanWangSheng, SallehAlhawarat, LiuStorrey,
    minimizeobjective, minimizeobjectivererun, linesearch!, evalϕdϕ!, getβ, updatedir!,
    initializeβ, initializeLineSearchContainer!, evalwolfeconditions, evalbacktrackcondition

export Context, RosenbrockGPU, RosenbrockChainedGPU, UserObjectiveGPU, SparseLSGPU, LogRegGPU, SoftmaxRegGPU, LBFGS, DeviceObjective,
    DeviceStart, trial_site, set_csr_mode!, trim_pools!,
    BoxConstraint, BoxBarrierGPU, BatchedConfig, minimizeobjective_batched

include("capi.jl")
include("device.jl")
include("flavours.jl")
include("linesearch.jl")
include("optim.jl")
include("extras.jl")     # solvesystem, primalbarriermethod!, batched solver

end # module
