# AdvancedHMCB200Ext.jl -- the reference-side binding of libahmc_b200 (include/ahmc_b200.h): one `ccall` wrapper per
# exported entry point (tests/test_abi.py checks names, arities and struct layouts against the header).
#
# STATUS: WRITTEN, NOT EXECUTED.  No `julia` binary exists in the build image (SURVEY.md section 8c), so this file has
# never been parsed or run; the same entry points are exercised from Python (advancedhmc.jl_b200/core.py) by the
# test-suite.  It is the package extension a maintainer would add next to ext/AdvancedHMCCUDAExt.jl.  Citations are
# relative to the AdvancedHMC.jl checkout.
#
# Plug-in points used (SURVEY.md section 8b):
#   * a new integrator type `B200Leapfrog{T} <: AbstractLeapfrog{T}` with its own `step` method -- the mechanism
#     ext/AdvancedHMCOrdinaryDiffEqSymplecticRKExt.jl:6-13 uses for `DiffEqIntegrator`;
#   * whole-transition overrides `transition(rng, h, tau, z)` (src/trajectory.jl:271-276, 344-390, 677-681) when the
#     integrator is a `B200Leapfrog`, so refresh + trajectory + MH / NUTS tree run as ONE kernel;
#   * `Hamiltonian`, `AbstractMetric`, the adaptors and `sample` (src/sampler.jl:159-248) are untouched; the pooled
#     multi-GPU adaptor (`B200PooledAdaptor`) is an additional `AbstractAdaptor`-shaped object for the many-chain case.
module AdvancedHMCB200Ext

using AdvancedHMC
using AdvancedHMC: AbstractLeapfrog, Hamiltonian, PhasePoint, DualValue, Trajectory, Transition, HMCKernel,
    UnitEuclideanMetric, DiagEuclideanMetric, DenseEuclideanMetric, EndPointTS, MultinomialTS, SliceTS,
    FixedNSteps, FixedIntegrationTime, GeneralisedNoUTurn, ClassicNoUTurn, StrictGeneralisedNoUTurn,
    DynamicTerminationCriterion, FullMomentumRefreshment, PartialMomentumRefreshment, step_size, nom_step_size, nsteps
using CUDA
using Random

const libahmc = get(ENV, "AHMC_B200_LIB", "libahmc_b200.so")

# ---- C structs (include/ahmc_b200.h) --------------------------------------------------------------
struct CMetric
    kind::Int32
    Minv::Ptr{Float64}
    chain_stride::Int64
    cholU::Ptr{Float64}
end
struct CPhasePoint
    theta::Ptr{Float64}
    r::Ptr{Float64}
    lp_value::Ptr{Float64}
    lp_gradient::Ptr{Float64}
    lk_value::Ptr{Float64}
    lk_gradient::Ptr{Float64}
    ld::Int64
end
struct CStats
    n_steps::Ptr{Int32}
    is_accept::Ptr{UInt8}
    acceptance_rate::Ptr{Float64}
    log_density::Ptr{Float64}
    hamiltonian_energy::Ptr{Float64}
    hamiltonian_energy_error::Ptr{Float64}
    max_hamiltonian_energy_error::Ptr{Float64}
    tree_depth::Ptr{Int32}
    numerical_error::Ptr{UInt8}
end
struct CRng
    seed::UInt64
    offset::UInt64
    normal_tape::Ptr{Float64}
    exp_tape::Ptr{Float64}
    exp_stride::Int64
    dir_tape::Ptr{UInt8}
    dir_stride::Int64
    partial_refresh_alpha::Float64
    temper_alpha::Float64
end
struct CAdaptCfg
    n_adapts::Int32; init_buffer::Int32; term_buffer::Int32; window_size::Int32
    delta::Float64; gamma::Float64; t0::Float64; kappa::Float64
    adapt_metric::Int32; n_min::Int32
    eps_chain::Ptr{Float64}; Minv_chain::Ptr{Float64}; eps_trace::Ptr{Float64}
end
struct CPooledCfg
    n_adapts::Int32; init_buffer::Int32; term_buffer::Int32; window_size::Int32
    delta::Float64; gamma::Float64; t0::Float64; kappa::Float64; eps0::Float64
    adapt_metric::Int32; n_min::Int32
end

const FLAG_HOST_BUFFERS = 0x1 % UInt32
const FLAG_COMPAT_BREAK_ALL = 0x2 % UInt32
const FLAG_ASYNC = 0x4 % UInt32
const FLAG_EXACT_CHECKS = 0x8 % UInt32
const FLAG_NO_REFRESH = 0x10 % UInt32
const FLAG_NUTS_SLICE_TS = 0x20 % UInt32
const FLAG_NUTS_CLASSIC = 0x40 % UInt32
const FLAG_NUTS_STRICT = 0x80 % UInt32

# device pointer of a CuArray as the plain `Ptr` the C structs carry (`pointer(::CuArray)` is a `CuPtr`)
dptr(x::CuArray{T}) where {T} = reinterpret(Ptr{T}, pointer(x))
dptr(::Nothing) = C_NULL

# ---- context -------------------------------------------------------------------------------------------
mutable struct B200Context
    h::Ptr{Cvoid}
end
const CTX = Ref{Union{Nothing,B200Context}}(nothing)

b200_version() = unsafe_string(ccall((:ahmc_version, libahmc), Cstring, ()))

function context()
    if CTX[] === nothing
        out = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:ahmc_create, libahmc), Cint, (Ref{Ptr{Cvoid}}, Int32, Ptr{Cvoid}), out, CUDA.deviceid(), CUDA.stream().handle)
        rc == 0 || error("ahmc_create failed ($rc)")
        CTX[] = B200Context(out[])
    end
    return CTX[]
end

function destroy_context()
    CTX[] === nothing && return nothing
    ccall((:ahmc_destroy, libahmc), Cint, (Ptr{Cvoid},), CTX[].h)
    CTX[] = nothing
    return nothing
end

last_error() = unsafe_string(ccall((:ahmc_last_error, libahmc), Cstring, (Ptr{Cvoid},), context().h))

"Negative return codes become Julia exceptions: AHMC_ERR_INVALID -> ArgumentError (hamiltonian.jl:55-57, :94)."
check(rc) = rc == 0 ? nothing : (msg = last_error(); rc == -1 ? throw(ArgumentError(msg)) : error("ahmc error $rc: $msg"))

b200_synchronize() = check(ccall((:ahmc_synchronize, libahmc), Cint, (Ptr{Cvoid},), context().h))
b200_stream() = ccall((:ahmc_stream, libahmc), Ptr{Cvoid}, (Ptr{Cvoid},), context().h)
b200_launch_count() = ccall((:ahmc_launch_count, libahmc), Int64, (Ptr{Cvoid},), context().h)
b200_last_transport() = unsafe_string(ccall((:ahmc_last_transport, libahmc), Cstring, (Ptr{Cvoid},), context().h))

# ---- models ----------------------------------------------------------------------------------------------
"Target handle: replaces the `ℓπ` / `∂ℓπ∂θ` closures (src/hamiltonian.jl:45-48) inside the fused kernels."
mutable struct B200Target
    handle::Ptr{Cvoid}
    D::Int
    keep::Any   # callback targets: the closure and its @cfunction must outlive the handle
end

"Built-in device target: kind 0 std-normal, 1 diagonal Gaussian (p0 = mean, p1 = 1/s^2), 2 dense Gaussian (p1 = precision), 3 funnel."
function B200Target(kind::Integer, D::Integer; p0::Union{Nothing,Vector{Float64}}=nothing,
                    p1::Union{Nothing,Array{Float64}}=nothing, c0=0.0)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve p0 p1 check(ccall((:ahmc_model_create, libahmc), Cint,
                                   (Ptr{Cvoid}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Float64, Ref{Ptr{Cvoid}}),
                                   context().h, kind, D, p0 === nothing ? C_NULL : pointer(p0),
                                   p1 === nothing ? C_NULL : pointer(p1), c0, out))
    return B200Target(out[], D, nothing)
end

# trampoline of a user closure f(θ::CuMatrix) -> (ℓπ::CuVector, ∇ℓπ::CuMatrix): runs on the library's stream
function _logp_grad_trampoline(user::Ptr{Cvoid}, theta::Ptr{Float64}, lp::Ptr{Float64}, grad::Ptr{Float64}, D::Int32,
                               N::Int64, ld::Int64, stream::Ptr{Cvoid})::Cint
    try
        f = unsafe_pointer_to_objref(user)[]
        θ = unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, theta), (Int(ld), Int(N)))
        v, g = f(view(θ, 1:Int(D), :))
        copyto!(unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, lp), (Int(N),)), v)
        copyto!(view(unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, grad), (Int(ld), Int(N))), 1:Int(D), :), g)
        return Cint(0)
    catch
        return Cint(1)   # never throw across the C ABI
    end
end

"Callback target: an arbitrary Julia closure `θ -> (ℓπ, ∇ℓπ)` on CuArrays, called once per leapfrog step (split-step mode)."
function B200Target(f::Function, D::Integer)
    box = Ref{Any}(f)
    cfn = @cfunction(_logp_grad_trampoline, Cint,
                     (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Int64, Int64, Ptr{Cvoid}))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ahmc_model_create_callback, libahmc), Cint, (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Ptr{Cvoid}}),
                context().h, D, cfn, pointer_from_objref(box), out))
    return B200Target(out[], D, (box, cfn))
end

"""
User target as CUDA source compiled at run time INTO the fused kernels (ahmc_model_create_user): `src` defines
`__device__ double ahmc_user_logp_grad(const double* theta, double* grad, int D, const double* params)` (or the
coordinate-wise contract, see include/ahmc_b200.h).  Unlike a callback target it runs inside NUTS and costs no host round trip.
"""
function B200Target(src::String, D::Integer; params::Vector{Float64}=Float64[], c0=0.0)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve params check(ccall((:ahmc_model_create_user, libahmc), Cint,
                                    (Ptr{Cvoid}, Int32, Cstring, Ptr{Float64}, Int32, Float64, Ref{Ptr{Cvoid}}),
                                    context().h, D, src, isempty(params) ? C_NULL : pointer(params), length(params), c0, out))
    return B200Target(out[], D, nothing)
end
"compile-only check of a user target (no GPU needed); returns the NVRTC log (empty = compiles)"
function b200_user_source_check(src::String, D::Integer; kernel::Integer=1, metric_kind::Integer=1)
    log = zeros(UInt8, 8192)
    rc = GC.@preserve log ccall((:ahmc_user_source_check, libahmc), Cint, (Cstring, Int32, Int32, Int32, Ptr{UInt8}, Int64),
                                src, kernel, metric_kind, D, pointer(log), length(log))
    return rc == 0 ? "" : unsafe_string(pointer(log))
end

function destroy!(t::B200Target)
    check(ccall((:ahmc_model_destroy, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), context().h, t.handle))
    t.handle = C_NULL
    return nothing
end

# ---- the integrator plug-in (src/integrator.jl:49-60 interface) -------------------------------------
struct B200Leapfrog{T<:AdvancedHMC.AbstractScalarOrVec{<:AbstractFloat}} <: AbstractLeapfrog{T}
    ϵ::T
    target::B200Target
    α::Float64          # 0: `Leapfrog(ϵ)`; > 0: `TemperedLeapfrog(ϵ, α)` (src/integrator.jl:174-209), in `step` and in transitions
end
B200Leapfrog(ϵ, target::B200Target) = B200Leapfrog(ϵ, target, 0.0)
AdvancedHMC.update_nom_step_size(lf::B200Leapfrog, ϵ) = B200Leapfrog(ϵ, lf.target, lf.α)
temper_alpha(lf::B200Leapfrog) = lf.α

cmetric(m::UnitEuclideanMetric, N) = CMetric(0, C_NULL, 0, C_NULL)
cmetric(m::DiagEuclideanMetric, N) = CMetric(1, dptr(m.M⁻¹), ndims(m.M⁻¹) == 2 ? size(m.M⁻¹, 1) : 0, C_NULL)
# Dense: the caller keeps `U = CuArray(Matrix(m.cholM⁻¹))` alive for the duration of the call
cmetric(m::DenseEuclideanMetric, N, U::CuMatrix{Float64}) = CMetric(2, dptr(m.M⁻¹), 0, dptr(U))
dense_factor(m::DenseEuclideanMetric) = CuArray(Matrix(m.cholM⁻¹))
dense_factor(m) = nothing
metric_desc(m::DenseEuclideanMetric, N, U) = cmetric(m, N, U)
metric_desc(m, N, U) = cmetric(m, N)

cpp(z::PhasePoint{<:CuArray}; lk_gradient::Bool=true) =
    CPhasePoint(dptr(z.θ), dptr(z.r), dptr(z.ℓπ.value), dptr(z.ℓπ.gradient), dptr(z.ℓκ.value),
                lk_gradient ? dptr(z.ℓκ.gradient) : C_NULL, size(z.θ, 1))

fresh_pp(z::PhasePoint) = PhasePoint(similar(z.θ), similar(z.r), DualValue(similar(z.ℓπ.value), similar(z.ℓπ.gradient)),
                                     DualValue(similar(z.ℓκ.value), similar(z.ℓκ.gradient)))

refresh_alpha(::FullMomentumRefreshment) = 0.0
refresh_alpha(r::PartialMomentumRefreshment) = Float64(r.α)

eps_args(ϵ::AbstractFloat) = (Float64(ϵ), Ptr{Float64}(C_NULL))
eps_args(ϵ::CuVector{Float64}) = (0.0, dptr(ϵ))

# key drawn from the Julia rng; the transition's refreshment and integrator options ride in the same struct
philox(rng, κ) = CRng(rand(rng, UInt64), 0, C_NULL, C_NULL, 0, C_NULL, 0, refresh_alpha(κ.refreshment), temper_alpha(κ.τ.integrator))

"`phasepoint(h, θ, r)` (src/hamiltonian.jl:115-119) for a B200 target."
function b200_phasepoint(t::B200Target, h::Hamiltonian, θ::CuMatrix{Float64}, r::CuMatrix{Float64})
    D, N = size(θ)
    z = PhasePoint(θ, r, DualValue(CUDA.zeros(Float64, N), similar(θ)), DualValue(CUDA.zeros(Float64, N), similar(θ)))
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zc = Ref(cpp(z))
    GC.@preserve z U check(ccall((:ahmc_phasepoint_f64, libahmc), Cint,
                                 (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Ref{CPhasePoint}, UInt32),
                                 context().h, t.handle, md, D, N, zc, 0))
    return z
end

"`step` for CuArray phase points: replaces src/integrator.jl:216-265 (about 10 broadcast kernels and 4 host-syncing
`all(isfinite)` per step) with ONE fused kernel for all n_steps; `full_trajectory = Val(true)` (:229, 249-261) returns
the `Vector{PhasePoint}` of every step (views into one device slab)."
function AdvancedHMC.step(lf::B200Leapfrog, h::Hamiltonian, z::PhasePoint{<:CuMatrix{Float64}}, n_steps::Int=1;
                          fwd::Bool=n_steps > 0, full_trajectory::Val{FullTraj}=Val(false)) where {FullTraj}
    D, N = size(z.θ)
    ϵ, ϵp = eps_args(step_size(lf))
    n = fwd ? abs(n_steps) : -abs(n_steps)
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zi = Ref(cpp(z))
    if FullTraj
        L = abs(n_steps)
        θs = CUDA.zeros(Float64, D, N, L); rs = similar(θs); gs = similar(θs); drs = similar(θs)
        lps = CUDA.zeros(Float64, N, L); lks = similar(lps)
        done = CUDA.zeros(Int32, N)
        tc = Ref(CPhasePoint(dptr(θs), dptr(rs), dptr(lps), dptr(gs), dptr(lks), dptr(drs), D))
        GC.@preserve z U θs rs gs drs lps lks done begin
            check(ccall((:ahmc_leapfrog_trajectory_f64, libahmc), Cint,
                        (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Float64,
                         Ref{CPhasePoint}, Ref{CPhasePoint}, Int64, Ptr{Int32}, UInt32),
                        context().h, lf.target.handle, md, D, N, ϵ, ϵp, n, lf.α, zi, tc, D * N, dptr(done), 0))
        end
        nmax = Int(maximum(Array(done)))   # like `resize!(res, i)` on an early break (integrator.jl:252-258)
        return [PhasePoint(θs[:, :, i], rs[:, :, i], DualValue(lps[:, i], gs[:, :, i]), DualValue(lks[:, i], drs[:, :, i]))
                for i in 1:nmax]
    end
    zout = fresh_pp(z); zo = Ref(cpp(zout))
    GC.@preserve z zout U begin
        check(ccall((:ahmc_leapfrog_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Float64,
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ptr{UInt32}, Ptr{Int32}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, n, lf.α, zi, zo, C_NULL, C_NULL, 0))
    end
    return zout
end

"`step` on HOST matrices (the CPU path's own argument types): the library stages / streams the buffers over PCIe
(AHMC_FLAG_HOST_BUFFERS); `z.ℓπ.gradient` is not uploaded (recomputed on the device for built-in targets)."
function AdvancedHMC.step(lf::B200Leapfrog, h::Hamiltonian, z::PhasePoint{<:Matrix{Float64}}, n_steps::Int=1;
                          fwd::Bool=n_steps > 0, full_trajectory::Val{FullTraj}=Val(false)) where {FullTraj}
    FullTraj && throw(ArgumentError("full_trajectory on host matrices: move the phase point to the device (CuArray) first"))
    h.metric isa DenseEuclideanMetric && throw(ArgumentError("host-buffer step: Unit / Diag metrics (move a Dense problem to the device)"))
    D, N = size(z.θ)
    zout = fresh_pp(z)
    ϵ, ϵp = step_size(lf) isa AbstractFloat ? (Float64(step_size(lf)), Ptr{Float64}(C_NULL)) : (0.0, pointer(step_size(lf)))
    n = fwd ? abs(n_steps) : -abs(n_steps)
    Mi = h.metric isa DiagEuclideanMetric ? h.metric.M⁻¹ : nothing
    md = Ref(Mi === nothing ? CMetric(0, C_NULL, 0, C_NULL) : CMetric(1, pointer(Mi), ndims(Mi) == 2 ? size(Mi, 1) : 0, C_NULL))
    zi = Ref(CPhasePoint(pointer(z.θ), pointer(z.r), C_NULL, C_NULL, C_NULL, C_NULL, D))
    zo = Ref(CPhasePoint(pointer(zout.θ), pointer(zout.r), pointer(zout.ℓπ.value), pointer(zout.ℓπ.gradient),
                         pointer(zout.ℓκ.value), pointer(zout.ℓκ.gradient), D))
    GC.@preserve z zout Mi lf begin
        check(ccall((:ahmc_leapfrog_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Float64,
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ptr{UInt32}, Ptr{Int32}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, n, lf.α, zi, zo, C_NULL, C_NULL, FLAG_HOST_BUFFERS))
    end
    return zout
end

"`rand_momentum(rng, metric, kinetic, θ)` (src/metric.jl:290-320) on the device (Philox stream keyed from `rng`)."
function b200_rand_momentum(rng, h::Hamiltonian, θ::CuMatrix{Float64})
    D, N = size(θ)
    r = similar(θ)
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U))
    rg = Ref(CRng(rand(rng, UInt64), 0, C_NULL, C_NULL, 0, C_NULL, 0, 0.0, 0.0))
    GC.@preserve r U check(ccall((:ahmc_rand_momentum_f64, libahmc), Cint,
                                 (Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Ref{CRng}, Ptr{Float64}, Int64, UInt32),
                                 context().h, md, D, N, rg, dptr(r), D, 0))
    return r
end

"`find_good_stepsize(rng, h, θ)` (src/trajectory.jl:768-837) for every column of θ at once, the whole search in one launch."
function b200_find_good_stepsize(rng, t::B200Target, h::Hamiltonian, θ::CuMatrix{Float64}; initial_step_size=0.1, max_n_iters::Int=100)
    D, N = size(θ)
    z = b200_phasepoint(t, h, θ, CUDA.zeros(Float64, D, N))
    ϵ = CUDA.zeros(Float64, N)
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zc = Ref(cpp(z; lk_gradient=false))
    rg = Ref(CRng(rand(rng, UInt64), 0, C_NULL, C_NULL, 0, C_NULL, 0, 0.0, 0.0))
    GC.@preserve z ϵ U check(ccall((:ahmc_find_good_stepsize_f64, libahmc), Cint,
                                   (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Ref{CPhasePoint}, Ref{CRng}, Float64, Int32,
                                    Ptr{Float64}, Ptr{Float64}, UInt32),
                                   context().h, t.handle, md, D, N, zc, rg, Float64(initial_step_size), max_n_iters, dptr(ϵ), C_NULL, 0))
    return ϵ
end

"Static HMC transition (src/trajectory.jl:271-300) as ONE kernel: refresh + L steps + MH + revert + flip."
function AdvancedHMC.transition(rng, h::Hamiltonian, κ::HMCKernel{R,<:Trajectory{EndPointTS,<:B200Leapfrog}},
                                z::PhasePoint{<:CuMatrix{Float64}}) where {R}
    τ = κ.τ; lf = τ.integrator
    D, N = size(z.θ)
    zout = fresh_pp(z)
    acc = CUDA.zeros(UInt8, N); α = CUDA.zeros(Float64, N); H = CUDA.zeros(Float64, N); dH = CUDA.zeros(Float64, N)
    nerr = CUDA.zeros(UInt8, N)
    st = Ref(CStats(C_NULL, dptr(acc), dptr(α), C_NULL, dptr(H), dptr(dH), C_NULL, C_NULL, dptr(nerr)))
    rg = Ref(philox(rng, κ))
    ϵ, ϵp = eps_args(step_size(lf))
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zi = Ref(cpp(z)); zo = Ref(cpp(zout; lk_gradient=false))
    GC.@preserve z zout acc α H dH nerr U begin
        check(ccall((:ahmc_hmc_transition_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Ref{CRng},
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ref{CStats}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, nsteps(τ), rg, zi, zo, st, 0))
    end
    tstat = merge((n_steps=nsteps(τ), is_accept=acc .== 1, acceptance_rate=α, log_density=zout.ℓπ.value,
                   hamiltonian_energy=H, hamiltonian_energy_error=dH, numerical_error=any(nerr .== 1)),
                  AdvancedHMC.stat(lf))
    return Transition(zout, tstat)
end

"Static transition with `MultinomialTS` (src/trajectory.jl:344-390): the direction split is ONE draw shared by all
chains (`rand_coupled`, :371-373), drawn here from the Julia rng."
function AdvancedHMC.transition(rng, h::Hamiltonian, κ::HMCKernel{R,<:Trajectory{MultinomialTS,<:B200Leapfrog,<:AdvancedHMC.StaticTerminationCriterion}},
                                z::PhasePoint{<:CuMatrix{Float64}}) where {R}
    τ = κ.τ; lf = τ.integrator
    D, N = size(z.θ)
    n = nsteps(τ)
    n_fwd = rand(rng, 0:n)
    zout = fresh_pp(z)
    α = CUDA.zeros(Float64, N); H = CUDA.zeros(Float64, N); dH = CUDA.zeros(Float64, N); off = CUDA.zeros(Int32, N)
    nerr = CUDA.zeros(UInt8, N)
    st = Ref(CStats(C_NULL, C_NULL, dptr(α), C_NULL, dptr(H), dptr(dH), C_NULL, dptr(off), dptr(nerr)))
    rg = Ref(philox(rng, κ))
    ϵ, ϵp = eps_args(step_size(lf))
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zi = Ref(cpp(z)); zo = Ref(cpp(zout; lk_gradient=false))
    GC.@preserve z zout α H dH off nerr U begin
        check(ccall((:ahmc_hmc_multinomial_transition_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Int32, Ref{CRng},
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ref{CStats}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, n, n_fwd, rg, zi, zo, st, 0))
    end
    tstat = merge((n_steps=n, is_accept=true, acceptance_rate=α, log_density=zout.ℓπ.value, hamiltonian_energy=H,
                   hamiltonian_energy_error=dH, numerical_error=any(nerr .== 1)), AdvancedHMC.stat(lf))
    return Transition(zout, tstat)
end

nuts_flags(::Type{TS}, ::Type{TC}) where {TS,TC} =
    (TS <: SliceTS ? FLAG_NUTS_SLICE_TS : 0x0 % UInt32) |
    (TC <: ClassicNoUTurn ? FLAG_NUTS_CLASSIC : TC <: StrictGeneralisedNoUTurn ? FLAG_NUTS_STRICT : 0x0 % UInt32)

"Many-chain NUTS (the reference's src/trajectory.jl:677-742 is scalar-only): MultinomialTS / SliceTS x the three
no-U-turn criteria (trajectory.jl:102-109, 551-557, 579-613) are flag bits of one entry point."
function AdvancedHMC.transition(rng, h::Hamiltonian, κ::HMCKernel{R,<:Trajectory{TS,<:B200Leapfrog,TC}},
                                z::PhasePoint{<:CuMatrix{Float64}}) where {R,TS<:Union{MultinomialTS,SliceTS},
                                                                          TC<:DynamicTerminationCriterion}
    τ = κ.τ; lf = τ.integrator; tc = τ.termination_criterion
    flags = nuts_flags(TS, TC)
    D, N = size(z.θ)
    zout = fresh_pp(z)
    ns = CUDA.zeros(Int32, N); α = CUDA.zeros(Float64, N); H = CUDA.zeros(Float64, N); dH = CUDA.zeros(Float64, N)
    mx = CUDA.zeros(Float64, N); td = CUDA.zeros(Int32, N); nerr = CUDA.zeros(UInt8, N)
    st = Ref(CStats(dptr(ns), C_NULL, dptr(α), C_NULL, dptr(H), dptr(dH), dptr(mx), dptr(td), dptr(nerr)))
    rg = Ref(philox(rng, κ))
    ϵ, ϵp = eps_args(step_size(lf))
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zi = Ref(cpp(z)); zo = Ref(cpp(zout; lk_gradient=false))
    GC.@preserve z zout ns α H dH mx td nerr U begin
        check(ccall((:ahmc_nuts_transition_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Float64, Ref{CRng},
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ref{CStats}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, tc.max_depth, tc.Δ_max, rg, zi, zo, st, flags))
    end
    tstat = merge((n_steps=ns, is_accept=true, acceptance_rate=α, log_density=zout.ℓπ.value, hamiltonian_energy=H,
                   hamiltonian_energy_error=dH, max_hamiltonian_energy_error=mx, tree_depth=td, numerical_error=nerr .== 1),
                  AdvancedHMC.stat(lf))
    return Transition(zout, tstat)
end

# ---- the un-adapted body of `sample` (src/sampler.jl:182-228) as ONE launch ------------------------------
"n_samples static-HMC transitions per chain in one persistent launch -> (draws D×N×n_samples, last phase point, α)."
function b200_sample_hmc(rng, h::Hamiltonian, κ::HMCKernel{R,<:Trajectory{EndPointTS,<:B200Leapfrog}}, z::PhasePoint{<:CuMatrix{Float64}},
                         n_samples::Int) where {R}
    τ = κ.τ; lf = τ.integrator
    D, N = size(z.θ)
    zout = fresh_pp(z)
    draws = CUDA.zeros(Float64, D, N, n_samples); α = CUDA.zeros(Float64, N * n_samples)
    st = Ref(CStats(C_NULL, C_NULL, dptr(α), C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL))
    rg = Ref(philox(rng, κ))
    ϵ, ϵp = eps_args(step_size(lf))
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zi = Ref(cpp(z)); zo = Ref(cpp(zout; lk_gradient=false))
    GC.@preserve z zout draws α U begin
        check(ccall((:ahmc_hmc_sample_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Int32, Ref{CRng},
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ptr{Float64}, Ref{CStats}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, nsteps(τ), n_samples, rg, zi, zo, dptr(draws), st, 0))
    end
    return draws, zout, reshape(α, N, n_samples)
end

"n_samples NUTS transitions per chain in one persistent launch (chains never wait for each other's trees)."
function b200_sample_nuts_fixed(rng, h::Hamiltonian, κ::HMCKernel{R,<:Trajectory{TS,<:B200Leapfrog,TC}}, z::PhasePoint{<:CuMatrix{Float64}},
                                n_samples::Int) where {R,TS<:Union{MultinomialTS,SliceTS},TC<:DynamicTerminationCriterion}
    τ = κ.τ; lf = τ.integrator; tc = τ.termination_criterion
    D, N = size(z.θ)
    zout = fresh_pp(z)
    draws = CUDA.zeros(Float64, D, N, n_samples); α = CUDA.zeros(Float64, N * n_samples); ns = CUDA.zeros(Int32, N * n_samples)
    st = Ref(CStats(dptr(ns), C_NULL, dptr(α), C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL))
    rg = Ref(philox(rng, κ))
    ϵ, ϵp = eps_args(step_size(lf))
    U = dense_factor(h.metric)
    md = Ref(metric_desc(h.metric, N, U)); zi = Ref(cpp(z)); zo = Ref(cpp(zout; lk_gradient=false))
    GC.@preserve z zout draws α ns U begin
        check(ccall((:ahmc_nuts_sample_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Float64, Ptr{Float64}, Int32, Float64, Int32, Ref{CRng},
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ptr{Float64}, Ref{CStats}, UInt32),
                    context().h, lf.target.handle, md, D, N, ϵ, ϵp, tc.max_depth, tc.Δ_max, n_samples, rg, zi, zo,
                    dptr(draws), st, nuts_flags(TS, TC)))
    end
    return draws, zout, reshape(α, N, n_samples), reshape(ns, N, n_samples)
end

"""
`sample(rng, h, κ, θ, n_samples, adaptor, n_adapts)` (src/sampler.jl:159-248) for many-chain NUTS with the reference's
vectorised adaptors -- `StanHMCAdaptor(WelfordVar((D, N)), NesterovDualAveraging(δ, ϵ::Vector))` -- as ONE launch
(ahmc_nuts_adapt_sample_f64): every chain adapts its own ϵ and diagonal M⁻¹ and never waits for another chain.
Returns (θ draws D×N×n_samples, final per-chain ϵ, per-chain M⁻¹ D×N).
"""
function b200_sample_nuts(rng, h::Hamiltonian, lf::B200Leapfrog, tc::GeneralisedNoUTurn, θ::CuMatrix{Float64},
                          n_samples::Int, n_adapts::Int; δ=0.8, adapt_metric=true, init_buffer=75, term_buffer=50,
                          window_size=25)
    D, N = size(θ)
    z = b200_phasepoint(lf.target, h, θ, CUDA.zeros(Float64, D, N))
    zout = fresh_pp(z)
    ϵ = CUDA.fill(Float64(first(step_size(lf))), N); Minv = CUDA.ones(Float64, D, N)
    draws = CUDA.zeros(Float64, D, N, n_samples)
    α = CUDA.zeros(Float64, N * n_samples)
    st = Ref(CStats(C_NULL, C_NULL, dptr(α), C_NULL, C_NULL, C_NULL, C_NULL, C_NULL, C_NULL))
    cfg = Ref(CAdaptCfg(n_adapts, init_buffer, term_buffer, window_size, δ, 0.05, 10.0, 0.75, adapt_metric ? 1 : 0, 10,
                        dptr(ϵ), dptr(Minv), C_NULL))
    rg = Ref(CRng(rand(rng, UInt64), 0, C_NULL, C_NULL, 0, C_NULL, 0, 0.0, 0.0))
    md = Ref(cmetric(h.metric, N)); zi = Ref(cpp(z)); zo = Ref(cpp(zout; lk_gradient=false))
    GC.@preserve z zout ϵ Minv draws α begin
        check(ccall((:ahmc_nuts_adapt_sample_f64, libahmc), Cint,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Ref{CMetric}, Int32, Int64, Int32, Float64, Int32, Ref{CAdaptCfg}, Ref{CRng},
                     Ref{CPhasePoint}, Ref{CPhasePoint}, Ptr{Float64}, Ref{CStats}, UInt32),
                    context().h, lf.target.handle, md, D, N, tc.max_depth, tc.Δ_max, n_samples, cfg, rg, zi, zo,
                    dptr(draws), st, 0))
    end
    return draws, ϵ, Minv
end

# ---- adaptor statistics and the pooled multi-GPU adaptor (src/adaptation/*.jl) -----------------------------
"Pooled adaptor record of one iteration: [N, sum min(1,α), mean(θ), M2(θ)] (ahmc_adapt_summary_f64)."
function b200_adapt_summary(θ::CuMatrix{Float64}, α::CuVector{Float64})
    D, N = size(θ)
    out = CUDA.zeros(Float64, 2 + 2D)
    GC.@preserve θ α out check(ccall((:ahmc_adapt_summary_f64, libahmc), Cint,
                                     (Ptr{Cvoid}, Int32, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, UInt32),
                                     context().h, D, N, dptr(θ), D, dptr(α), dptr(out), 0))
    return out
end

"Dense second moment Σ_c (θ_c − mean)(θ_c − mean)ᵀ for the pooled `WelfordCov` (massmatrix.jl:286-340)."
function b200_adapt_cov(θ::CuMatrix{Float64}, mean::CuVector{Float64})
    D, N = size(θ)
    out = CUDA.zeros(Float64, D, D)
    GC.@preserve θ mean out check(ccall((:ahmc_adapt_cov_f64, libahmc), Cint,
                                        (Ptr{Cvoid}, Int32, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, UInt32),
                                        context().h, D, N, dptr(θ), D, dptr(mean), dptr(out), 0))
    return out
end

"NCCL communicator of the ranks that share one adaptation (one Julia process per GPU)."
mutable struct B200Comm
    h::Ptr{Cvoid}
    nranks::Int
    rank::Int
end
"rank 0: 128 bytes to broadcast to the other ranks (MPI.jl `bcast`, Distributed `remotecall`, a file ...)"
function b200_comm_unique_id()
    id = zeros(UInt8, 128)
    GC.@preserve id check(ccall((:ahmc_comm_unique_id, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), context().h, pointer(id)))
    return id
end
function B200Comm(id::Vector{UInt8}, nranks::Integer, rank::Integer)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve id check(ccall((:ahmc_comm_create, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Ref{Ptr{Cvoid}}),
                                context().h, pointer(id), nranks, rank, out))
    return B200Comm(out[], nranks, rank)
end
"wrap a communicator the host already owns, e.g. `NCCL.Communicator(...).handle`"
function B200Comm(nccl_handle::Ptr{Cvoid}, nranks::Integer, rank::Integer)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ahmc_comm_from_nccl, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Ref{Ptr{Cvoid}}),
                context().h, nccl_handle, nranks, rank, out))
    return B200Comm(out[], nranks, rank)
end
function destroy!(c::B200Comm)
    check(ccall((:ahmc_comm_destroy, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), context().h, c.h))
    c.h = C_NULL
    return nothing
end

"all-gather of a small device record over the ranks (rank order), on the library's stream"
function b200_allgather(c::Union{Nothing,B200Comm}, record::CuVector{Float64})
    n = length(record)
    out = CUDA.zeros(Float64, n, c === nothing ? 1 : c.nranks)
    GC.@preserve record out check(ccall((:ahmc_adapt_allgather_f64, libahmc), Cint,
                                        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, UInt32),
                                        context().h, c === nothing ? C_NULL : c.h, dptr(record), n, dptr(out), 0))
    return out
end

"""
Pooled `StanHMCAdaptor(WelfordVar, NesterovDualAveraging)` resident on the device (stepsize.jl:178-210,
massmatrix.jl:141-157, stan_adaptor.jl:13-50, 137-159; pooling across chains and ranks is new, `Adaptation.jl:52`).
`ϵ` (length N, all entries equal) and `M⁻¹` (length D) are CuArray views of the buffers the library updates in place:
build `B200Leapfrog(a.ϵ, target)` and `DiagEuclideanMetric(a.M⁻¹)` once, then per warm-up iteration call
`t = transition(rng, h, κ, t.z); adapt!(a, comm, t.z.θ, t.stat.acceptance_rate)` -- nothing is copied to the host.
"""
mutable struct B200PooledAdaptor
    h::Ptr{Cvoid}
    D::Int
    N::Int
    ϵ::CuVector{Float64}
    M⁻¹::CuVector{Float64}
end
function B200PooledAdaptor(D::Integer, N::Integer, n_adapts::Integer, ϵ0::Real; δ=0.8, adapt_metric=true, init_buffer=75,
                           term_buffer=50, window_size=25, γ=0.05, t_0=10.0, κ=0.75, n_min=10,
                           M⁻¹0::Union{Nothing,Vector{Float64}}=nothing)
    cfg = Ref(CPooledCfg(n_adapts, init_buffer, term_buffer, window_size, δ, γ, t_0, κ, ϵ0, adapt_metric ? 1 : 0, n_min))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve M⁻¹0 check(ccall((:ahmc_pooled_create, libahmc), Cint,
                                  (Ptr{Cvoid}, Int32, Int64, Ref{CPooledCfg}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
                                  context().h, D, N, cfg, M⁻¹0 === nothing ? C_NULL : pointer(M⁻¹0), out))
    pe = ccall((:ahmc_pooled_eps, libahmc), Ptr{Float64}, (Ptr{Cvoid},), out[])
    pm = ccall((:ahmc_pooled_minv, libahmc), Ptr{Float64}, (Ptr{Cvoid},), out[])
    ϵ = unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, pe), (Int(N),))
    Mi = unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, pm), (Int(D),))
    return B200PooledAdaptor(out[], D, N, ϵ, Mi)
end
"`adapt!(adaptor, θ, α)` of the next iteration (sampler.jl:72-90 glue): K5 record -> all-gather -> merge + adaptor update"
function AdvancedHMC.Adaptation.adapt!(a::B200PooledAdaptor, c::Union{Nothing,B200Comm}, θ::CuMatrix{Float64}, α::CuVector{Float64})
    GC.@preserve θ α check(ccall((:ahmc_adapt_exchange_f64, libahmc), Cint,
                                 (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, UInt32),
                                 context().h, c === nothing ? C_NULL : c.h, a.h, a.D, a.N, dptr(θ), a.D, dptr(α), C_NULL, FLAG_ASYNC))
    return nothing
end
"synchronising read-back: (ϵ, M⁻¹, iterations done)"
function b200_pooled_state(a::B200PooledAdaptor)
    ϵ = Ref{Float64}(0.0); it = Ref{Int32}(0); Mi = zeros(Float64, a.D)
    GC.@preserve Mi check(ccall((:ahmc_pooled_state, libahmc), Cint,
                                (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float64}, Ptr{Float64}, Ref{Int32}, Ptr{Float64}),
                                context().h, a.h, ϵ, pointer(Mi), it, C_NULL))
    return ϵ[], Mi, Int(it[])
end
function destroy!(a::B200PooledAdaptor)
    check(ccall((:ahmc_pooled_destroy, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), context().h, a.h))
    a.h = C_NULL
    return nothing
end

"""
Pooled `StanHMCAdaptor(WelfordCov, NesterovDualAveraging)` resident on the device (massmatrix.jl:286-340): the dense form of
`B200PooledAdaptor`.  `M⁻¹` and `U` (upper, `U'U = M⁻¹`) are D x D CuArray views of the buffers the library updates in place
at window ends (the new estimate is factorised on the device; a failed factorisation keeps both and is reported by
`b200_pooled_state(::B200PooledDenseAdaptor)` as `failed_iteration`).  Build the metric once from them, e.g.
`DenseEuclideanMetric(a.M⁻¹)` with the transition calls passing `CMetric(METRIC_DENSE, dptr(a.M⁻¹), 0, dptr(a.U))`.
Like the rest of this file, written but not executed.
"""
mutable struct B200PooledDenseAdaptor
    h::Ptr{Cvoid}
    D::Int
    N::Int
    ϵ::CuVector{Float64}
    M⁻¹::CuMatrix{Float64}
    U::CuMatrix{Float64}
end
function b200_pooled_adaptor(D::Integer, N::Integer, n_adapts::Integer, ϵ0::Real, M⁻¹0::Union{Nothing,Matrix{Float64}};
                             δ=0.8, adapt_metric=true, init_buffer=75, term_buffer=50, window_size=25, γ=0.05, t_0=10.0,
                             κ=0.75, n_min=10)
    cfg = Ref(CPooledCfg(n_adapts, init_buffer, term_buffer, window_size, δ, γ, t_0, κ, ϵ0, adapt_metric ? 1 : 0, n_min))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve M⁻¹0 check(ccall((:ahmc_pooled_create_dense, libahmc), Cint,
                                  (Ptr{Cvoid}, Int32, Int64, Ref{CPooledCfg}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
                                  context().h, D, N, cfg, M⁻¹0 === nothing ? C_NULL : pointer(M⁻¹0), out))
    pe = ccall((:ahmc_pooled_eps, libahmc), Ptr{Float64}, (Ptr{Cvoid},), out[])
    pm = ccall((:ahmc_pooled_minv, libahmc), Ptr{Float64}, (Ptr{Cvoid},), out[])
    pu = ccall((:ahmc_pooled_cholu, libahmc), Ptr{Float64}, (Ptr{Cvoid},), out[])
    ϵ = unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, pe), (Int(N),))
    Mi = unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, pm), (Int(D), Int(D)))  # column-major, as Julia's
    U = unsafe_wrap(CuArray, reinterpret(CuPtr{Float64}, pu), (Int(D), Int(D)))
    return B200PooledDenseAdaptor(out[], D, N, ϵ, Mi, U)
end
function AdvancedHMC.Adaptation.adapt!(a::B200PooledDenseAdaptor, c::Union{Nothing,B200Comm}, θ::CuMatrix{Float64}, α::CuVector{Float64})
    GC.@preserve θ α check(ccall((:ahmc_adapt_exchange_f64, libahmc), Cint,
                                 (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, UInt32),
                                 context().h, c === nothing ? C_NULL : c.h, a.h, a.D, a.N, dptr(θ), a.D, dptr(α), C_NULL, FLAG_ASYNC))
    return nothing
end
"synchronising read-back: (ϵ, M⁻¹, U, iterations done, failed_iteration); failed_iteration = 0 when every factorisation succeeded"
function b200_pooled_state(a::B200PooledDenseAdaptor)
    ϵ = Ref{Float64}(0.0); it = Ref{Int32}(0); failed = Ref{Int32}(0)
    Mi = zeros(Float64, a.D, a.D); U = zeros(Float64, a.D, a.D)
    GC.@preserve Mi U check(ccall((:ahmc_pooled_state_dense, libahmc), Cint,
                                  (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Int32}, Ptr{Float64}, Ref{Int32}),
                                  context().h, a.h, ϵ, pointer(Mi), pointer(U), it, C_NULL, failed))
    return ϵ[], Mi, U, Int(it[]), Int(failed[])
end
function destroy!(a::B200PooledDenseAdaptor)
    check(ccall((:ahmc_pooled_destroy, libahmc), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), context().h, a.h))
    a.h = C_NULL
    return nothing
end

end # module
