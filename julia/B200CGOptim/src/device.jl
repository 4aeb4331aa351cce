# Device context, objective handles and the device-resident LineSearchContainer
# (src/types.jl:84-100: xp, df_xp, x, u — plus x, df_x of src/engine/optim.jl:20-21).

mutable struct Context
    h::Ptr{Cvoid}
    nranks::Int
    rank::Int
    function Context(device::Integer = 0; reduction_ctas::Union{Nothing,Integer} = nothing)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:cgo_ctx_create, LIBCGOPTIM[]), Cint, (Cint, Ptr{Cvoid}, Ref{Ptr{Cvoid}}), device, C_NULL, h))
        ctx = new(h[], 1, 0)
        reduction_ctas === nothing ||
            check(ccall((:cgo_ctx_set_reduction_ctas, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Cint), ctx.h, reduction_ctas))
        finalizer(c -> (c.h == C_NULL || ccall((:cgo_ctx_destroy, LIBCGOPTIM[]), Cint, (Ptr{Cvoid},), c.h); c.h = C_NULL), ctx)
        return ctx
    end
end

# multi-GPU: one Julia process per GPU; rank 0 creates the 128-byte id, the host ships it
# (MPI.jl, Distributed, a file) and every rank calls comm_init!.
function comm_unique_id()
    id = zeros(UInt8, 128)
    check(ccall((:cgo_comm_get_unique_id, LIBCGOPTIM[]), Cint, (Ptr{UInt8},), id))
    return id
end
function comm_init!(ctx::Context, nranks::Integer, rank::Integer, id::Vector{UInt8})
    check(ccall((:cgo_ctx_comm_init, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{UInt8}), ctx.h, nranks, rank, id))
    ctx.nranks, ctx.rank = nranks, rank
    return ctx
end

"Device-resident replacement of the user callback `fdf!(g, x) -> f` (optim.jl:25, cg_utils.jl:18)."
mutable struct DeviceObjective
    ctx::Context
    h::Ptr{Cvoid}
    n_local::Int
    n_global::Int
    offset::Int
end
function _wrap(ctx::Context, h::Ptr{Cvoid})
    nl, ng, off = Ref{Int64}(0), Ref{Int64}(0), Ref{Int64}(0)
    check(ccall((:cgo_obj_dims, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int64}, Ref{Int64}), h, nl, ng, off))
    obj = DeviceObjective(ctx, h, nl[], ng[], off[])
    finalizer(o -> (o.h == C_NULL || ccall((:cgo_obj_destroy, LIBCGOPTIM[]), Cint, (Ptr{Cvoid},), o.h); o.h = C_NULL), obj)
    return obj
end
"Extended Rosenbrock (pairs), SURVEY.md §8d cfg 1/2."
function RosenbrockGPU(n::Integer, ctx::Context)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_obj_rosenbrock_create, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.h, n, h))
    return _wrap(ctx, h[])
end
"The reference's own chained Rosenbrock, rosenbrockfunc (examples/helpers/test_funcs.jl:50-57), with its gradient."
function RosenbrockChainedGPU(n::Integer, ctx::Context)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_obj_rosenbrock_chained_create, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.h, n, h))
    return _wrap(ctx, h[])
end
"""
ANY `fdf!(g, x) -> f` on the device (include/cgoptim.h cgo_obj_user_create).  `fdf_dev(stream, n_local, offset, xp, g, f)`
receives raw device pointers (`Ptr{Float64}`; wrap them with `unsafe_wrap(CuArray, …)` under CUDA.jl, or launch your
own kernels) and must enqueue on `stream` the work that fills `g` with ∇f(xp) and `f[1]` with this rank's part of f.
It returns nothing; an exception is reported as a failed trial, never thrown across the C ABI.
"""
function UserObjectiveGPU(n::Integer, fdf_dev, ctx::Context)
    function thunk(user::Ptr{Cvoid}, stream::Ptr{Cvoid}, n_local::Int64, offset::Int64,
                   xp::Ptr{Float64}, g::Ptr{Float64}, f::Ptr{Float64})::Cint
        try
            fdf_dev(stream, n_local, offset, xp, g, f)
            return Cint(0)
        catch
            return Cint(1)
        end
    end
    cb = @cfunction($thunk, Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_obj_user_create, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Int64, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Ptr{Cvoid}}),
                ctx.h, n, cb, C_NULL, h))
    obj = _wrap(ctx, h[])
    USER_THUNKS[obj.h] = cb          # keep the closure alive as long as the objective
    return obj
end
const USER_THUNKS = Dict{Ptr{Cvoid},Any}()
"(V, U) of the canonical reduction order the objective's trial dots follow (include/cgoptim.h)."
function trial_site(obj::DeviceObjective)
    v, u = Ref{Int32}(0), Ref{Int32}(0)
    check(ccall((:cgo_obj_reduction_site, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Ref{Int32}, Ref{Int32}), obj.h, v, u))
    return Int(v[]), Int(u[])
end
set_csr_mode!(ctx::Context, mode::Integer) = check(ccall((:cgo_ctx_set_csr_mode, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Cint), ctx.h, mode))
function trim_pools!(ctx::Context)
    freed = Ref{Int64}(0)
    check(ccall((:cgo_ctx_trim_pools, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Ref{Int64}), ctx.h, freed))
    return freed[]
end
"½‖Ax − b‖², synthetic banded CSR (cfg 3), or from a host CSR (0-based int64 rowptr, int32 col)."
function SparseLSGPU(n::Integer, ctx::Context; nnz_per_row = 10, W = min(1 << 20, (n - 1) ÷ 2), seed = 24, coh_log2 = 0)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_obj_sparse_ls_create_synthetic, LIBCGOPTIM[]), Cint,
        (Ptr{Cvoid}, Int64, Int32, Int64, UInt64, Int32, Ref{Ptr{Cvoid}}), ctx.h, n, nnz_per_row, W, seed, coh_log2, h))
    return _wrap(ctx, h[])
end
function SparseLSGPU(nrows::Integer, ncols::Integer, rowptr::Vector{Int64}, col::Vector{Int32},
                     val::Vector{Float64}, b::Vector{Float64}, ctx::Context)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_obj_sparse_ls_create_csr, LIBCGOPTIM[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
        ctx.h, nrows, ncols, rowptr, col, val, b, h))
    return _wrap(ctx, h[])
end
"CSR logistic regression (cfg 4)."
function LogRegGPU(nsamples::Integer, nfeat::Integer, ctx::Context; nnz_per_row = 20, seed = 24, λ = 1e-6)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_obj_logreg_create_synthetic, LIBCGOPTIM[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Int32, UInt64, Float64, Ref{Ptr{Cvoid}}), ctx.h, nsamples, nfeat, nnz_per_row, seed, λ, h))
    return _wrap(ctx, h[])
end
"CSR logistic regression on the caller's CSR (0-based int64 row pointers, int32 columns) and labels ±1; single GPU.
`sample_weight`: nsamples finite weights >= 0 with a positive sum S (`nothing`: unit weights, S = nsamples); the loss
is (1/S) Σ s_i ℓ_i.  `fit_intercept = true` fits b, which λ does not penalise: the state is (w, b), n = nfeat + 1,
and `x[nfeat + 1]` is b.  Without it, a column of ones in A is an intercept that λ penalises like the other weights."
function LogRegGPU(nsamples::Integer, nfeat::Integer, rowptr::Vector{Int64}, col::Vector{Int32},
                   val::Vector{Float64}, y::Vector{Float64}, ctx::Context; λ = 1e-6,
                   sample_weight::Union{Nothing, Vector{Float64}} = nothing, fit_intercept::Bool = false)
    sample_weight === nothing || length(sample_weight) == nsamples || throw(ArgumentError("sample_weight needs nsamples entries"))
    sw = sample_weight === nothing ? Ptr{Float64}(C_NULL) : pointer(sample_weight)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve sample_weight check(ccall((:cgo_obj_logreg_create_csr_ex, LIBCGOPTIM[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Float64,
         Ref{Ptr{Cvoid}}),
        ctx.h, nsamples, nfeat, rowptr, col, val, y, sw, Int32(fit_intercept), λ, h))
    return _wrap(ctx, h[])
end
"Softmax (multinomial logistic) regression on the caller's CSR (0-based int64 row pointers, int32 columns) and labels in
[0, nclasses), 2 <= nclasses <= 256; single GPU.  The state vector is W (nfeat × nclasses) feature-major, w[j·K + k]:
`permutedims(reshape(x, nclasses, nfeat))` is W.  `sample_weight` as for `LogRegGPU`.  `fit_intercept = true` fits
b_k, which λ does not penalise: the state has nfeat + 1 rows and `permutedims(reshape(x, nclasses, nfeat + 1))[end, :]`
is b.  Without it, a column of ones in A is an intercept whose weights λ penalises."
function SoftmaxRegGPU(nsamples::Integer, nfeat::Integer, nclasses::Integer, rowptr::Vector{Int64}, col::Vector{Int32},
                       val::Vector{Float64}, labels::Vector{Int32}, ctx::Context; λ = 1e-6,
                       sample_weight::Union{Nothing, Vector{Float64}} = nothing, fit_intercept::Bool = false)
    sample_weight === nothing || length(sample_weight) == nsamples || throw(ArgumentError("sample_weight needs nsamples entries"))
    sw = sample_weight === nothing ? Ptr{Float64}(C_NULL) : pointer(sample_weight)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve sample_weight check(ccall((:cgo_obj_softmax_create_csr_ex, LIBCGOPTIM[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Int32, Ptr{Int64}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}, Int32, Float64,
         Ref{Ptr{Cvoid}}),
        ctx.h, nsamples, nfeat, nclasses, rowptr, col, val, labels, sw, Int32(fit_intercept), λ, h))
    return _wrap(ctx, h[])
end

"Token for one of the device vectors of a workspace (keeps the reference's call shapes)."
struct DeviceVector{W}
    ws::W
    name::Symbol
end

"LineSearchContainer (types.jl:84-100) + x, df_x (optim.jl:20-21), resident in HBM."
mutable struct DeviceWorkspace
    obj::DeviceObjective
    h::Ptr{Cvoid}
    n::Int
    buf::Vector{Float64}          # scalar pack scratch
    pack::Vector{Float64}         # last trial pack
    dpack::Vector{Float64}        # {g·u, u·u} of the kernel that last wrote u
    f_x0::Float64
    norm_df_x0::Float64
    pending_β::Union{Nothing,Float64}     # lazily fused updatedir!
    hint::Union{Nothing,Float64}
    cached::Union{Nothing,Tuple{Float64,Vector{Float64}}}
    β_literal::Bool
end
"`x_initial` that already lives on the device: the iterate of a live workspace (cgo_state_create_from_state)."
struct DeviceStart
    ws::Any
end
# the restart of minimizeobjectivererun (optim.jl:191-201) / a centering step (primal_barrier.jl:215-247) without H2D
function DeviceWorkspace(obj::DeviceObjective, start::DeviceStart; lbfgs_m::Integer = 0, β_literal = false)
    buf = zeros(PACK_LEN)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:cgo_state_create_from_state, LIBCGOPTIM[]), Cint,
                (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Ref{Ptr{Cvoid}}, Ptr{Float64}),
                obj.ctx.h, obj.h, start.ws.h, 0, lbfgs_m, h, buf))
    ws = DeviceWorkspace(obj, h[], obj.n_local, buf, copy(buf), zeros(2), buf[P_PHI], sqrt(buf[P_GPGP]),
                         nothing, nothing, nothing, β_literal)
    finalizer(close!, ws)
    return ws
end
# optim.jl:20-26: x = copy(x_initial); f_x = fdf!(df_x, x); norm(df_x)
function DeviceWorkspace(obj::DeviceObjective, x_initial::Vector{Float64}; lbfgs_m::Integer = 0, β_literal = false)
    length(x_initial) == obj.n_local || throw(DimensionMismatch("x_initial vs objective shard"))
    buf = zeros(PACK_LEN)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve x_initial check(ccall((:cgo_state_create, LIBCGOPTIM[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Int32, Ref{Ptr{Cvoid}}, Ptr{Float64}),
        obj.ctx.h, obj.h, x_initial, lbfgs_m, h, buf))
    ws = DeviceWorkspace(obj, h[], obj.n_local, buf, copy(buf), zeros(2), buf[P_PHI], sqrt(buf[P_GPGP]),
                         nothing, nothing, nothing, β_literal)
    finalizer(close!, ws)
    return ws
end
close!(ws::DeviceWorkspace) = (ws.h == C_NULL || ccall((:cgo_state_destroy, LIBCGOPTIM[]), Cint, (Ptr{Cvoid},), ws.h); ws.h = C_NULL; nothing)

vec(ws::DeviceWorkspace, name::Symbol) = DeviceVector(ws, name)

function resetdirection!(ws::DeviceWorkspace)            # u = −df_x  (cg_flavours.jl:28, wolfe.jl:129)
    ws.pending_β = nothing; ws.cached = nothing
    check(ccall((:cgo_reset_direction, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Ptr{Float64}), ws.h, ws.buf))
    ws.dpack .= ws.buf[1:2]
    return nothing
end
function materializedirection!(ws::DeviceWorkspace)
    ws.pending_β === nothing && return nothing
    β = ws.pending_β; ws.pending_β = nothing
    if ws.hint !== nothing && isfinite(ws.hint)
        a = ws.hint
        check(ccall((:cgo_eval_trial_fused_dir, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Float64, Float64, Ptr{Float64}), ws.h, β, a, ws.buf))
        pk = copy(ws.buf)
        ws.cached = (a, pk)
        ws.dpack .= (pk[P_DIR_GU], pk[P_DIR_UU])
    else
        check(ccall((:cgo_update_dir, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Float64, Ptr{Float64}), ws.h, β, ws.buf))
        ws.dpack .= ws.buf[1:2]
    end
    ws.hint = nothing
    return nothing
end
dot_g_u(ws::DeviceWorkspace) = (materializedirection!(ws); ws.dpack[D_GU])
dot_u_u(ws::DeviceWorkspace) = (materializedirection!(ws); ws.dpack[D_UU])
function norm_u_plus_g(ws::DeviceWorkspace)              # norm(u + df_x), wolfe.jl:123
    materializedirection!(ws)
    v = Ref{Float64}(0.0)
    check(ccall((:cgo_norm_sq_u_plus_g, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Ref{Float64}), ws.h, v))
    return sqrt(v[])
end
function evaltrial!(ws::DeviceWorkspace, a::Float64)     # evalϕdϕ!, cg_utils.jl:3-22
    materializedirection!(ws)
    if ws.cached !== nothing && ws.cached[1] == a
        ws.pack = ws.cached[2]
    else
        check(ccall((:cgo_eval_trial, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Float64, Ptr{Float64}), ws.h, a, ws.buf))
        ws.pack = copy(ws.buf)
    end
    ws.cached = nothing
    return ws.pack[P_PHI], ws.pack[P_DPHI]
end
accept!(ws::DeviceWorkspace) = (ws.cached = nothing; check(ccall((:cgo_accept, LIBCGOPTIM[]), Cint, (Ptr{Cvoid},), ws.h)))
function download(ws::DeviceWorkspace)                   # Results.minimizer / .gradient
    x, g = Vector{Float64}(undef, ws.n), Vector{Float64}(undef, ws.n)
    check(ccall((:cgo_download, LIBCGOPTIM[]), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), ws.h, x, g))
    return x, g
end

# LinearAlgebra.dot on device vectors: only the pairs the hot path needs exist
# (dot(df_x,u): nocedal.jl:56, wolfe.jl:40, geometric.jl:43; dot(u,u): wolfe.jl:240, geometric.jl:52)
function devdot(a::DeviceVector, b::DeviceVector)
    names = (a.name, b.name)
    (names == (:df_x, :u) || names == (:u, :df_x)) && return dot_g_u(a.ws)
    names == (:u, :u) && return dot_u_u(a.ws)
    error("dot($(a.name), $(b.name)) is not on the hot path")
end
