# LinearMixingModelsB200.jl -- the reference-side binding of liblmm.so (include/lmm.h).
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia.  This is the shim a
# maintainer loads next to LinearMixingModels.jl: it keeps the reference's exported types
# (ILMM, OILMM, Orthogonal, IndependentMOGP; src/LinearMixingModels.jl:21-24) and overrides the
# method *bodies* of the hot path with `ccall`s.  The Python host mirror
# (linearmixingmodels.jl_b200/api.py) exercises exactly the same exports with the same buffer
# layouts (column-major, by-outputs vectors), so every ccall below has a tested ctypes twin.
module LinearMixingModelsB200

using LinearAlgebra, Random
using AbstractGPs, KernelFunctions, FillArrays
using LinearMixingModels
using LinearMixingModels: ILMM, OILMM, Orthogonal, IndependentMOGP, unpack, noise_var

const liblmm = get(ENV, "LIBLMM", joinpath(@__DIR__, "..", "liblmm.so"))

struct KernelTerm        # lmm_kernel_term: one further term of a KernelSum / KernelProduct
    kind::Int32
    reserved::Int32
    variance::Float64
    inv_lengthscale::Float64
    param::Float64
    ard::Ptr{Float64}
end

struct GpDesc            # lmm_gp_desc
    kind::Int32
    compose::Int32       # 0 single kernel, 1 KernelSum, 2 KernelProduct over this term and `extra`
    variance::Float64
    inv_lengthscale::Float64
    mean_const::Float64
    ard::Ptr{Float64}    # ARDTransform multipliers (D values, kept alive by the caller with GC.@preserve) or C_NULL
    param::Float64       # α of RationalQuadraticKernel, r of PeriodicKernel
    n_extra::Int32
    reserved2::Int32
    extra::Ptr{KernelTerm}
end

const CTX = Ref{Ptr{Cvoid}}(C_NULL)
function ctx()
    if CTX[] == C_NULL
        h = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:lmm_ctx_create, liblmm), Cint, (Cint, Ptr{Ptr{Cvoid}}), 0, h)
        rc == 0 || error("lmm_ctx_create failed ($rc): a CUDA device is required (no CPU fallback)")
        CTX[] = h[]
    end
    return CTX[]
end
lasterr() = unsafe_string(ccall((:lmm_last_error, liblmm), Cstring, (Ptr{Cvoid},), ctx()))

function check(rc::Integer)
    rc == 0 && return nothing
    rc > 0 && throw(PosDefException(rc))                                   # LAPACK info
    rc == -2 && error("out dim of x != out dim of f.")                     # src/ilmm.jl:52
    rc == -6 && throw(ArgumentError("`U` is not an orthogonal matrix"))    # src/orthogonal_matrix.jl:22
    rc == -7 && throw(OutOfMemoryError())
    (rc == -1 || rc == -3) && throw(ArgumentError(lasterr()))
    error("liblmm error $rc: $(lasterr())")
end

# --- kernel / GP description ------------------------------------------------------------------
kind(::SqExponentialKernel) = Int32(0)
kind(::Matern32Kernel) = Int32(1)
kind(::Matern52Kernel) = Int32(2)
kind(::ExponentialKernel) = Int32(3)          # == Matern12Kernel
kind(::RationalQuadraticKernel) = Int32(4)    # α travels in GpDesc.param
kind(::PeriodicKernel) = Int32(5)             # r travels in GpDesc.param (one r for all dimensions)
shape(k) = 1.0
shape(k::RationalQuadraticKernel) = Float64(only(k.α))   # KernelFunctions default α = 2
function shape(k::PeriodicKernel)
    all(==(first(k.r)), k.r) || throw(ArgumentError("PeriodicKernel with per-dimension r is not supported by liblmm"))
    return Float64(first(k.r))
end
# One scaled, stretched base kernel: (kind, variance, inv_lengthscale, shape parameter, ARD multipliers or nothing)
const Term = Tuple{Int32,Float64,Float64,Float64,Union{Nothing,Vector{Float64}}}
# describe(k) -> (op, terms): op 0 single kernel, 1 KernelSum, 2 KernelProduct (flat, at most 4 terms)
describe(k::KernelFunctions.SimpleKernel) = (Int32(0), Term[(kind(k), 1.0, 1.0, shape(k), nothing)])
function describe(k::ScaledKernel)
    op, ts = describe(k.kernel)
    c = Float64(only(k.σ²))
    if op == 1                       # c (k1 + k2) = c k1 + c k2
        return op, Term[(t[1], t[2] * c, t[3], t[4], t[5]) for t in ts]
    end
    t = ts[1]                        # single kernel or product: the factor goes to the first term
    return op, Term[(t[1], t[2] * c, t[3], t[4], t[5]); ts[2:end]]
end
function describe(k::TransformedKernel{<:Kernel,<:ScaleTransform})
    op, ts = describe(k.kernel)      # the transformed inputs feed every term of a composite
    s = Float64(only(k.transform.s))
    return op, Term[(t[1], t[2], t[3] * s, t[4], t[5]) for t in ts]
end
# `k ∘ ARDTransform(v)`: inputs are multiplied by v per dimension before distances are taken -> the terms' ard vectors
function describe(k::TransformedKernel{<:Kernel,<:ARDTransform})
    op, ts = describe(k.kernel)
    v = Vector{Float64}(k.transform.v)
    length(v) <= 8 || throw(ArgumentError("ARDTransform with more than 8 dimensions is not supported by liblmm"))
    return op, Term[(t[1], t[2], t[3], t[4], t[5] === nothing ? copy(v) : t[5] .* v) for t in ts]
end
function combine(op::Int32, parts)
    ts = Term[]
    for q in parts
        o, t = describe(q)
        (o == 0 || o == op) || throw(ArgumentError("liblmm supports flat sums or flat products of base kernels"))
        append!(ts, t)
    end
    length(ts) <= 4 || throw(ArgumentError("a composite kernel has at most 4 terms"))
    return (length(ts) > 1 ? op : Int32(0)), ts
end
describe(k::KernelSum) = combine(Int32(1), k.kernels)          # `k1 + k2`
describe(k::KernelProduct) = combine(Int32(2), k.kernels)      # `k1 * k2`
describe(k) = throw(ArgumentError("kernel $(typeof(k)) is not supported by liblmm (no CPU fallback)"))
meanconst(::AbstractGPs.ZeroMean) = 0.0
meanconst(m::AbstractGPs.ConstMean) = Float64(m.c)
# The C descriptors of a vector of latents plus the objects that must stay rooted while the library reads them (the ARD
# vectors GpDesc.ard / KernelTerm.ard point into, the KernelTerm arrays GpDesc.extra points into): every ccall that takes
# `descs` runs under `GC.@preserve keep`.
function gpdescs(fs::AbstractVector)
    keep = Any[]
    ardptr(a) = a === nothing ? Ptr{Float64}(C_NULL) : (push!(keep, a); pointer(a))
    descs = map(fs) do f
        op, ts = describe(f.kernel)
        t0 = ts[1]
        extra = KernelTerm[KernelTerm(t[1], 0, t[2], t[3], t[4], ardptr(t[5])) for t in ts[2:end]]
        px = isempty(extra) ? Ptr{KernelTerm}(C_NULL) : (push!(keep, extra); pointer(extra))
        p = ardptr(t0[5])
        GpDesc(t0[1], op, t0[2], t0[3], meanconst(f.mean), p, t0[4], length(extra), 0, px)
    end
    return Vector{GpDesc}(descs), keep
end

points(x::AbstractVector{<:Real}) = (collect(Float64, x), 1)
points(x::ColVecs) = (Matrix{Float64}(x.X), size(x.X, 1))              # D x N column-major
points(x::RowVecs) = (Matrix{Float64}(permutedims(x.X)), size(x.X, 2))

# --- device-resident posterior -----------------------------------------------------------------
# y / σ²: the training data and noise the handle was conditioned on (empty / NaN when unknown, e.g. a loaded handle); the
# gradient through the conditioning (lmm_post_logpdf_grad_full) needs them.
mutable struct DevicePosterior
    handle::Ptr{Cvoid}
    y::Vector{Float64}
    σ²::Float64
    function DevicePosterior(h, y::Vector{Float64} = Float64[], σ²::Float64 = NaN)
        p = new(h, y, σ²)
        finalizer(q -> ccall((:lmm_post_free, liblmm), Cint, (Ptr{Cvoid},), q.handle), p)
        return p
    end
end
# A latent of the posterior OILMM: behaves as an AbstractGP whose (α, C, x, δ) live on the GPU.
struct DeviceLatentPosterior{Tf<:GP} <: AbstractGPs.AbstractGP
    owner::DevicePosterior
    index::Int
    prior::Tf
end

# --- logpdf(fx::FiniteGP{<:OILMM}, y)   replaces src/oilmm.jl:79-93 ------------------------------
function AbstractGPs.logpdf(fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    U = Matrix{Float64}(H.U); S = Vector{Float64}(diag(H.S)); yv = Vector{Float64}(y)
    out = Ref{Float64}(0.0); il = Ref{Cint}(-1)
    rc = GC.@preserve keep ccall((:lmm_oilmm_logpdf, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64,
         Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, U, S, size(U, 1), Float64(σ²), yv, fx.x.out_dim, out, C_NULL, il)
    check(rc)
    return out[]
end

# --- posterior(fx::FiniteGP{<:OILMM}, y)   replaces src/oilmm.jl:116-134 -------------------------
function AbstractGPs.posterior(fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    U = Matrix{Float64}(H.U); S = Vector{Float64}(diag(H.S)); yv = Vector{Float64}(y)
    h = Ref{Ptr{Cvoid}}(C_NULL); il = Ref{Cint}(-1)
    rc = GC.@preserve keep ccall((:lmm_oilmm_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64,
         Ptr{Float64}, Cint, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, U, S, size(U, 1), Float64(σ²), yv, fx.x.out_dim, h, C_NULL, C_NULL, il)
    check(rc)
    owner = DevicePosterior(h[], yv, Float64(σ²))
    latents = [DeviceLatentPosterior(owner, i - 1, f) for (i, f) in enumerate(fs.fs)]
    return ILMM(IndependentMOGP(latents), H)          # an OILMM whose latents are (device) posteriors
end

const PosteriorOILMM = ILMM{<:IndependentMOGP{<:Vector{<:DeviceLatentPosterior}},<:Orthogonal}

# --- mean_and_var(post(x*, σ²))   replaces src/oilmm.jl:57-76 on posterior latents ---------------
function AbstractGPs.mean_and_var(fx::FiniteGP{<:PosteriorOILMM})
    fs, H, σ², x = unpack(fx)
    X, _ = points(x)
    n = length(x) * fx.x.out_dim
    M = Vector{Float64}(undef, n); V = Vector{Float64}(undef, n)
    rc = ccall((:lmm_post_mean_and_var, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}),
        fs.fs[1].owner.handle, X, length(x), Float64(σ²), M, V)
    check(rc)
    return M, V
end

# --- logpdf(post(x*, σ²), y*)   (test/oilmm.jl:84) ----------------------------------------------
function AbstractGPs.logpdf(fx::FiniteGP{<:PosteriorOILMM}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, _ = points(x)
    out = Ref{Float64}(0.0); il = Ref{Cint}(-1)
    rc = ccall((:lmm_post_logpdf, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        fs.fs[1].owner.handle, X, length(x), Float64(σ²), Vector{Float64}(y), out, il)
    check(rc)
    return out[]
end

# --- rand(rng, fx)   replaces src/oilmm.jl:40-54: normals drawn in the reference's order ----------
function AbstractGPs.rand(rng::AbstractRNG, fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    m, p, N = length(descs), size(H, 1), length(x)
    zl = randn(rng, N * m)          # latent 1..m, N draws each  (src/oilmm.jl:47)
    zn = randn(rng, N * p)          # then the observation noise (src/oilmm.jl:53)
    out = Vector{Float64}(undef, N * p); il = Ref{Cint}(-1)
    rc = GC.@preserve keep ccall((:lmm_oilmm_rand, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint,
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, m, X, N, D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), p, Float64(σ²), fx.x.out_dim, zl, zn, out, il)
    check(rc)
    return out
end

# --- general ILMM: logpdf replaces src/ilmm.jl:150-163 ------------------------------------------
function AbstractGPs.logpdf(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}},<:Matrix{Float64}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    out = Ref{Float64}(0.0); info = Ref{Cint}(0)
    rc = GC.@preserve keep ccall((:lmm_ilmm_logpdf, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint, Cint,
         Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, H, size(H, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, 0, out, info)
    check(rc)
    return out[]
end

# --- IndependentMOGP: logpdf replaces src/independent_mogp.jl:74-80 -----------------------------
function AbstractGPs.logpdf(ft::FiniteGP{<:IndependentMOGP{<:Vector{<:GP}},<:MOInputIsotopicByOutputs,<:Diagonal{<:Real,<:Fill}},
                            y::AbstractVector{<:Real})
    X, D = points(ft.x.x)
    descs, keep = gpdescs(ft.f.fs)
    out = Ref{Float64}(0.0); il = Ref{Cint}(-1)
    rc = GC.@preserve keep ccall((:lmm_imogp_logpdf, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(ft.x.x), D, Float64(ft.Σy[1]), Vector{Float64}(y), ft.x.out_dim, out, C_NULL, il)
    check(rc)
    return out[]
end

# --- mean_and_cov / cov(post(x*, σ²))   replaces src/ilmm.jl:132-139,147 on posterior latents -----
function AbstractGPs.mean_and_cov(fx::FiniteGP{<:PosteriorOILMM})
    fs, H, σ², x = unpack(fx)
    X, _ = points(x)
    n = length(x) * fx.x.out_dim
    M = Vector{Float64}(undef, n); C = Matrix{Float64}(undef, n, n)
    check(ccall((:lmm_post_mean_and_cov, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}),
        fs.fs[1].owner.handle, X, length(x), Float64(σ²), M, C))
    return M, C
end
AbstractGPs.cov(fx::FiniteGP{<:PosteriorOILMM}) = mean_and_cov(fx)[2]

# --- mean_and_cov on prior latents (OILMM and general ILMM): H passed explicitly -------------------
function AbstractGPs.mean_and_cov(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    Hm = Matrix{Float64}(collect(H))            # U*sqrt(S) for an Orthogonal
    n = length(x) * fx.x.out_dim
    M = Vector{Float64}(undef, n); C = Matrix{Float64}(undef, n, n)
    check(GC.@preserve keep ccall((:lmm_prior_mean_and_cov, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Float64, Cint, Ptr{Float64}, Ptr{Float64}),
        ctx(), descs, length(descs), X, length(x), D, Hm, size(Hm, 1), Float64(σ²), 1e-18, fx.x.out_dim, M, C))
    return M, C
end

# --- posterior(post(x2, σ²), y2): sequential conditioning ------------------------------------------
function AbstractGPs.posterior(fx::FiniteGP{<:PosteriorOILMM}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, _ = points(x)
    h = Ref{Ptr{Cvoid}}(C_NULL); il = Ref{Cint}(-1)
    check(ccall((:lmm_post_condition, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Ptr{Cvoid}}, Ptr{Cint}),
        fs.fs[1].owner.handle, X, length(x), Float64(σ²), Vector{Float64}(y), h, il))
    owner = DevicePosterior(h[])
    return ILMM(IndependentMOGP([DeviceLatentPosterior(owner, f.index, f.prior) for f in fs.fs]), H)
end

# --- rand(rng, post(x*, σ²)) ------------------------------------------------------------------------
function AbstractGPs.rand(rng::AbstractRNG, fx::FiniteGP{<:PosteriorOILMM})
    fs, H, σ², x = unpack(fx)
    X, _ = points(x)
    m, p, N = length(fs.fs), size(H, 1), length(x)
    zl = randn(rng, N * m); zn = randn(rng, N * p)
    out = Vector{Float64}(undef, N * p); il = Ref{Cint}(-1)
    check(ccall((:lmm_post_rand, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        fs.fs[1].owner.handle, X, N, Float64(σ²), zl, zn, out, il))
    return out
end

# --- rrule for logpdf (keeps `Zygote.gradient(logpdf, fx, y)` working: test/oilmm.jl:31-32) ---------
# The ccall is opaque to AD, so the pullback comes from `lmm_oilmm_logpdf_grad_terms` (batched potri +
# fused kernel-gradient reductions), which accepts every latent kernel the value path does (KernelSum /
# KernelProduct, PeriodicKernel, RationalQuadraticKernel).  Tangents are returned for y, σ² and, per latent,
# the hyper-parameters of every kernel term (gt) and the constant mean; mapping them back onto the nested
# kernel structs (ScaledKernel.σ², ScaleTransform.s, PeriodicKernel.r, ConstMean.c) is mechanical and omitted here.
const GRAD_TERM_DOUBLES = 4 * 11   # LMM_MAX_TERMS * LMM_GRAD_TERM_STRIDE doubles of grad_terms per latent
using ChainRulesCore
function ChainRulesCore.rrule(::typeof(AbstractGPs.logpdf), fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}},
                              y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs); m = length(descs)
    out = Ref{Float64}(0.0); gs2 = Ref{Float64}(0.0); il = Ref{Cint}(-1)
    gl = Matrix{Float64}(undef, 3, m)            # column i = (d/dvariance, d/dinv_lengthscale, d/dmean) of latent i
    gy = Vector{Float64}(undef, length(y))
    gU = Matrix{Float64}(undef, size(H, 1), m); gS = Vector{Float64}(undef, m)   # tangents of H.U and H.S.diag
    gt = Matrix{Float64}(undef, GRAD_TERM_DOUBLES, m)   # column i: latent i's terms, 11 slots each (variance, s, param, ard[1:8])
    check(GC.@preserve keep ccall((:lmm_oilmm_logpdf_grad_terms, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, m, X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
        Vector{Float64}(y), fx.x.out_dim, out, gl, C_NULL #= grad_ard (m x D, row-major): pass a Matrix{Float64}(undef, D, m) to receive d/d ARD multipliers =#, gs2, gy, gU, gS, gt, il))
    function logpdf_pullback(Δ)
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
        return NoTangent(), Tangent{typeof(fx)}(; Σy = Σy_tangent), Δ .* gy
    end
    return out[], logpdf_pullback
end

# --- rrule for the general-ILMM logpdf (test/ilmm.jl:31 `gradient(logpdf, ilmmx, y_train)`) -------
function ChainRulesCore.rrule(::typeof(AbstractGPs.logpdf), fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}},<:Matrix{Float64}}},
                              y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs); m = length(descs)
    out = Ref{Float64}(0.0); gs2 = Ref{Float64}(0.0); info = Ref{Cint}(0)
    gl = Matrix{Float64}(undef, 3, m); gy = Vector{Float64}(undef, length(y)); gH = similar(H)
    gt = Matrix{Float64}(undef, GRAD_TERM_DOUBLES, m)
    check(GC.@preserve keep ccall((:lmm_ilmm_logpdf_grad_terms, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, m, X, length(x), D, H, size(H, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, out, gl, C_NULL, gs2, gy, gH, gt, info))
    function logpdf_pullback(Δ)
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
        f_tangent = Tangent{typeof(fx.f)}(; H = Δ .* gH)
        return NoTangent(), Tangent{typeof(fx)}(; f = f_tangent, Σy = Σy_tangent), Δ .* gy
    end
    return out[], logpdf_pullback
end

# --- leave-one-input-out cross-validation (lmm_oilmm_loo / lmm_imogp_loo) --------------------------------------------
# loo_logpdf(fx, y) = Σ_i log p(y_i | y_{-i}) with y_i all outputs at input x_i (closed form, no refits);
# loo_mean_and_var(fx, y) = the LOO predictive marginals, by outputs.  Outputs left at C_NULL are not computed; without a
# gradient output only the value path runs.
const LOOFiniteGP = Union{FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}},
                          FiniteGP{<:IndependentMOGP{<:Vector{<:GP}},<:MOInputIsotopicByOutputs,<:Diagonal{<:Real,<:Fill}}}

function _loo(fx::LOOFiniteGP, y::AbstractVector{<:Real}; out=C_NULL, M=C_NULL, V=C_NULL, gl=C_NULL, gs2=C_NULL, gy=C_NULL,
              gU=C_NULL, gS=C_NULL, gt=C_NULL)
    il = Ref{Cint}(-1)
    if fx.f isa OILMM
        fs, H, σ², x = unpack(fx)
        X, D = points(x)
        descs, keep = gpdescs(fs.fs)
        check(GC.@preserve keep ccall((:lmm_oilmm_loo, liblmm), Cint,
            (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
            ctx(), descs, length(descs), X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
            Vector{Float64}(y), fx.x.out_dim, out, M, V, gl, C_NULL, gs2, gy, gU, gS, gt, il))
    else
        X, D = points(fx.x.x)
        descs, keep = gpdescs(fx.f.fs)
        check(GC.@preserve keep ccall((:lmm_imogp_loo, liblmm), Cint,
            (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ptr{Float64}, Cint,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
            ctx(), descs, length(descs), X, length(fx.x.x), D, Float64(fx.Σy[1]), Vector{Float64}(y), fx.x.out_dim,
            out, M, V, gl, C_NULL, gs2, gy, gt, il))
    end
    return nothing
end

function loo_logpdf(fx::LOOFiniteGP, y::AbstractVector{<:Real})
    out = Ref{Float64}(0.0)
    _loo(fx, y; out = out)
    return out[]
end

function loo_mean_and_var(fx::LOOFiniteGP, y::AbstractVector{<:Real})
    M = Vector{Float64}(undef, length(y)); V = Vector{Float64}(undef, length(y))
    _loo(fx, y; M = M, V = V)
    return M, V
end

# The pullback gives the σ² and y tangents; the per-term kernel tangents (gt), the means (gl row 3) and, for an OILMM, U / S
# are computed as in the logpdf rrule and, as there, not mapped onto the kernel structs.
function ChainRulesCore.rrule(::typeof(loo_logpdf), fx::LOOFiniteGP, y::AbstractVector{<:Real})
    orth = fx.f isa OILMM
    m = length((orth ? fx.f.f : fx.f).fs)
    out = Ref{Float64}(0.0); gs2 = Ref{Float64}(0.0)
    gl = Matrix{Float64}(undef, 3, m); gy = Vector{Float64}(undef, length(y))
    gt = Matrix{Float64}(undef, GRAD_TERM_DOUBLES, m)
    gU = orth ? Matrix{Float64}(undef, size(fx.f.H, 1), m) : C_NULL
    gS = orth ? Vector{Float64}(undef, m) : C_NULL
    _loo(fx, y; out = out, gl = gl, gs2 = gs2, gy = gy, gU = gU, gS = gS, gt = gt)
    function loo_pullback(Δ)
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
        return NoTangent(), Tangent{typeof(fx)}(; Σy = Σy_tangent), Δ .* gy
    end
    return out[], loo_pullback
end

# --- rrule for logpdf(post(x*, σ²), y*) (test/oilmm.jl:32 `gradient(logpdf, po, y_test)`) -----------------------------
# Through the conditioning (lmm_post_logpdf_grad_full): besides the Σy and y* tangents, the posterior's latents get a tangent
# on their `prior` (per-term hyper-parameters gt as in the prior rrule, mapping onto the kernel structs omitted as there; the
# constant means), H gets U / S, and the owner gets (σ², y) of the training data -- the rrule of `posterior` below maps those
# back onto the prior FiniteGP and the training y.  A handle that does not know its training data (a loaded one) gives the
# σ² and y* tangents only (lmm_post_logpdf_grad).
function ChainRulesCore.rrule(::typeof(AbstractGPs.logpdf), fx::FiniteGP{<:PosteriorOILMM}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    owner = fs.fs[1].owner
    out = Ref{Float64}(0.0); gs2 = Ref{Float64}(0.0); il = Ref{Cint}(-1)
    gy = Vector{Float64}(undef, length(y))
    if isempty(owner.y)
        check(ccall((:lmm_post_logpdf_grad, liblmm), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
            owner.handle, X, length(x), Float64(σ²), Vector{Float64}(y), out, gs2, gy, il))
        function logpdf_pullback(Δ)
            Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
            return NoTangent(), Tangent{typeof(fx)}(; Σy = Σy_tangent), Δ .* gy
        end
        return out[], logpdf_pullback
    end
    m = length(fs.fs); p = size(H, 1)
    gl = Matrix{Float64}(undef, 3, m); gt = Matrix{Float64}(undef, GRAD_TERM_DOUBLES, m)
    gts2 = Ref{Float64}(0.0); gyt = Vector{Float64}(undef, length(owner.y))
    gU = Matrix{Float64}(undef, p, m); gS = Vector{Float64}(undef, m)
    check(ccall((:lmm_post_logpdf_grad_full, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        owner.handle, X, length(x), Float64(σ²), Vector{Float64}(y), owner.y, out, gs2, gy, gl, C_NULL, gt, gts2, gyt, gU, gS, il))
    function logpdf_full_pullback(Δ)
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
        owner_tangent = Tangent{DevicePosterior}(; y = Δ .* gyt, σ² = Δ * gts2[])
        lat_tangents = [Tangent{typeof(f)}(; owner = owner_tangent, prior = Tangent{typeof(f.prior)}(; mean = Tangent{typeof(f.prior.mean)}(; c = Δ * gl[3, i])))
                        for (i, f) in enumerate(fs.fs)]
        f_tangent = Tangent{typeof(fx.f)}(; f = Tangent{typeof(fs)}(; fs = lat_tangents),
                                          H = Tangent{typeof(H)}(; U = Δ .* gU, S = Tangent{typeof(H.S)}(; diag = Δ .* gS)))
        return NoTangent(), Tangent{typeof(fx)}(; f = f_tangent, Σy = Σy_tangent), Δ .* gy
    end
    return out[], logpdf_full_pullback
end

# --- rrule for posterior(fx::FiniteGP{<:OILMM}, y): maps the posterior's tangent back onto fx and y ---------------------
# The latents' `prior` tangents become the prior's latents, H stays H, and the owner's stored (σ², y) become Σy and y.
function ChainRulesCore.rrule(::typeof(AbstractGPs.posterior), fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}},
                              y::AbstractVector{<:Real})
    post = AbstractGPs.posterior(fx, y)
    function posterior_pullback(Δpost)
        Δ = unthunk(Δpost)
        Δ isa AbstractZero && return NoTangent(), NoTangent(), NoTangent()
        lat = Δ.f isa AbstractZero ? nothing : Δ.f.fs
        prior_fs = lat === nothing ? NoTangent() : [t isa AbstractZero ? NoTangent() : t.prior for t in lat]
        owner = lat === nothing ? nothing : findfirst(t -> !(t isa AbstractZero) && !(t.owner isa AbstractZero), lat)
        ow = owner === nothing ? nothing : lat[owner].owner
        f_tangent = Tangent{typeof(fx.f)}(; f = Tangent{typeof(fx.f.f)}(; fs = prior_fs), H = Δ.H)
        if ow === nothing
            return NoTangent(), Tangent{typeof(fx)}(; f = f_tangent), NoTangent()
        end
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = ow.σ²))
        return NoTangent(), Tangent{typeof(fx)}(; f = f_tangent, Σy = Σy_tangent), ow.y
    end
    return post, posterior_pullback
end

# --- IndependentMOGP with Σy = Diagonal(v) or a dense Σy (AbstractGPs generic FiniteGP path,
#     test/independent_mogp.jl:72-75; by-features callers reorder Σy first, src/independent_mogp.jl:149-159) ---
noise_arg(Σy::Diagonal) = (Vector{Float64}(Σy.diag), Cint(1))      # LMM_NOISE_DIAG
noise_arg(Σy::AbstractMatrix) = (Matrix{Float64}(Σy), Cint(2))     # LMM_NOISE_DENSE
function AbstractGPs.logpdf(ft::FiniteGP{<:IndependentMOGP{<:Vector{<:GP}},<:MOInputIsotopicByOutputs}, y::AbstractVector{<:Real})
    X, D = points(ft.x.x)
    descs, keep = gpdescs(ft.f.fs)
    Σ, kind = noise_arg(ft.Σy)
    out = Ref{Float64}(0.0); il = Ref{Cint}(-1)
    check(GC.@preserve keep ccall((:lmm_imogp_posterior_noise, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(ft.x.x), D, Σ, kind, Vector{Float64}(y), ft.x.out_dim, C_NULL, out, il))
    return out[]
end

# --- mean_and_var on PRIOR latents   replaces src/oilmm.jl:57-76 (OILMM) and src/ilmm.jl:108-130 (general H) ---------
function AbstractGPs.mean_and_var(fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    n = length(x) * fx.x.out_dim
    M = Vector{Float64}(undef, n); V = Vector{Float64}(undef, n)
    check(GC.@preserve keep ccall((:lmm_oilmm_prior_mean_and_var, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Ptr{Float64}, Ptr{Float64}),
        ctx(), descs, length(descs), X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
        fx.x.out_dim, M, V))
    return M, V
end
function AbstractGPs.mean_and_var(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}},<:Matrix{Float64}}})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    n = length(x) * fx.x.out_dim
    M = Vector{Float64}(undef, n); V = Vector{Float64}(undef, n)
    check(GC.@preserve keep ccall((:lmm_ilmm_prior_mean_and_var, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Cint, Ptr{Float64}, Ptr{Float64}),
        ctx(), descs, length(descs), X, length(x), D, H, size(H, 1), Float64(σ²), fx.x.out_dim, M, V))
    return M, V
end
AbstractGPs.mean(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}}) = mean_and_var(fx)[1]     # src/ilmm.jl:142
AbstractGPs.var(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}}) = mean_and_var(fx)[2]      # src/ilmm.jl:145
AbstractGPs.mean(fx::FiniteGP{<:PosteriorOILMM}) = mean_and_var(fx)[1]
AbstractGPs.var(fx::FiniteGP{<:PosteriorOILMM}) = mean_and_var(fx)[2]

# --- general ILMM: posterior replaces src/ilmm.jl:184-198 (one (mN)² factor; POST_ILMM handle) and rand src/ilmm.jl:78-87 ---
const PosteriorILMM = ILMM{<:IndependentMOGP{<:Vector{<:DeviceLatentPosterior}},<:Matrix{Float64}}
function AbstractGPs.posterior(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}},<:Matrix{Float64}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    h = Ref{Ptr{Cvoid}}(C_NULL); info = Ref{Cint}(0)
    check(GC.@preserve keep ccall((:lmm_ilmm_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, H, size(H, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, h, C_NULL, info))
    owner = DevicePosterior(h[])
    return ILMM(IndependentMOGP([DeviceLatentPosterior(owner, i - 1, f) for (i, f) in enumerate(fs.fs)]), H)
end
# every lmm_post_* entry point dispatches on the handle's kind, so the posterior methods above serve both aliases
for f in (:mean_and_var, :mean_and_cov, :cov, :mean, :var)
    @eval AbstractGPs.$f(fx::FiniteGP{<:PosteriorILMM}) = invoke(AbstractGPs.$f, Tuple{FiniteGP{<:PosteriorOILMM}}, fx)
end
function AbstractGPs.rand(rng::AbstractRNG, fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}},<:Matrix{Float64}}})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    m, p, N = length(descs), size(H, 1), length(x)
    zl = randn(rng, N * m); zn = randn(rng, N * p)       # latent draws (src/ilmm.jl:84), then the noise (:86)
    out = Vector{Float64}(undef, N * p); il = Ref{Cint}(-1)
    check(GC.@preserve keep ccall((:lmm_ilmm_rand, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Cint,
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, m, X, N, D, H, p, Float64(σ²), fx.x.out_dim, zl, zn, out, il))
    return out
end
# rand(rng, fx, n) / rand(fx) (src/ilmm.jl:90-106): columns are independent draws in the reference's order
AbstractGPs.rand(rng::AbstractRNG, fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, n::Int) = hcat((rand(rng, fx) for _ in 1:n)...)
AbstractGPs.rand(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}}) = rand(Random.GLOBAL_RNG, fx)

# --- IndependentMOGP: posterior replaces src/independent_mogp.jl:119-126, rand :85-98 ------------------------------
function AbstractGPs.posterior(ft::FiniteGP{<:IndependentMOGP{<:Vector{<:GP}},<:MOInputIsotopicByOutputs,<:Diagonal{<:Real,<:Fill}},
                               y::AbstractVector{<:Real})
    X, D = points(ft.x.x)
    descs, keep = gpdescs(ft.f.fs)
    h = Ref{Ptr{Cvoid}}(C_NULL); il = Ref{Cint}(-1)
    check(GC.@preserve keep ccall((:lmm_imogp_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Float64, Ptr{Float64}, Cint, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(ft.x.x), D, Float64(ft.Σy[1]), Vector{Float64}(y), ft.x.out_dim, h, C_NULL, il))
    owner = DevicePosterior(h[])
    return IndependentMOGP([DeviceLatentPosterior(owner, i - 1, f) for (i, f) in enumerate(ft.f.fs)])
end
function AbstractGPs.rand(rng::AbstractRNG, ft::FiniteGP{<:IndependentMOGP{<:Vector{<:GP}},<:MOInputIsotopicByOutputs,<:Diagonal{<:Real,<:Fill}})
    X, D = points(ft.x.x)
    descs, keep = gpdescs(ft.f.fs)
    N = length(ft.x.x); m = length(descs)
    z = randn(rng, N * m); out = Vector{Float64}(undef, N * m); il = Ref{Cint}(-1)
    check(GC.@preserve keep ccall((:lmm_imogp_rand, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Float64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, m, X, N, D, Float64(ft.Σy[1]), ft.x.out_dim, z, out, il))
    return out
end
# by-features inputs (src/independent_mogp.jl:134-229): the permutation the reference builds with
# `vec(reshape(1:pN, N, p)')` comes from lmm_reorder_indices; y is permuted, the by-outputs method called, results permuted back
function reorder(N::Int, p::Int, direction::Int)
    idx = Vector{Int64}(undef, N * p)
    check(ccall((:lmm_reorder_indices, liblmm), Cint, (Cint, Cint, Cint, Ptr{Int64}), N, p, direction, idx))
    return idx .+ 1
end

# --- hyper-parameter sweep (BASELINE config 5): n_sweep logpdfs of the same data, every latent's inverse lengthscale scaled ---
function logpdf_sweep(fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real}, scales::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    out = Vector{Float64}(undef, length(scales)); il = Ref{Cint}(-1)
    check(GC.@preserve keep ccall((:lmm_oilmm_logpdf_sweep, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
        Vector{Float64}(y), fx.x.out_dim, Vector{Float64}(scales), length(scales), out, il))
    return out
end

# --- missing data (not in the reference, examples/oilmm_and_ilmm.ipynb:112): NaN entries of y are unobserved ---------
function posterior_missing(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    Hm = Matrix{Float64}(collect(H))
    h = Ref{Ptr{Cvoid}}(C_NULL); lp = Ref{Float64}(0.0); nobs = Ref{Cint}(0); info = Ref{Cint}(0)
    check(GC.@preserve keep ccall((:lmm_ilmm_masked_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, Hm, size(Hm, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, h, lp, nobs, info))
    return DevicePosterior(h[]), lp[], Int(nobs[])
end

# An OILMM whose mask is per input (whole time steps missing) stays an OILMM on the observed inputs: a full posterior.
function posterior_missing(fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    h = Ref{Ptr{Cvoid}}(C_NULL); lp = Ref{Float64}(0.0); nobs = Ref{Cint}(0); il = Ref{Cint}(-1)
    rc = GC.@preserve keep ccall((:lmm_oilmm_masked_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
        Vector{Float64}(y), fx.x.out_dim, h, lp, nobs, il)
    if rc == -3   # the mask is not per-input: the dense model (method above) on H = U sqrt(S)
        return invoke(posterior_missing, Tuple{FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}},AbstractVector{<:Real}}, fx, y)
    end
    check(rc)
    owner = DevicePosterior(h[])
    return ILMM(IndependentMOGP([DeviceLatentPosterior(owner, i - 1, f) for (i, f) in enumerate(fs.fs)]), H), lp[], Int(nobs[])
end

# logpdf of the observed (non-NaN) entries of y: the value of posterior_missing without keeping the factor
function logpdf_missing(fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    Hm = Matrix{Float64}(collect(H))
    lp = Ref{Float64}(0.0); nobs = Ref{Cint}(0); info = Ref{Cint}(0)
    check(GC.@preserve keep ccall((:lmm_ilmm_masked_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, Hm, size(Hm, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, C_NULL, lp, nobs, info))
    return lp[]
end
function logpdf_missing(fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs)
    lp = Ref{Float64}(0.0); nobs = Ref{Cint}(0); il = Ref{Cint}(-1)
    rc = GC.@preserve keep ccall((:lmm_oilmm_masked_posterior, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Ptr{Cvoid}}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
        ctx(), descs, length(descs), X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
        Vector{Float64}(y), fx.x.out_dim, C_NULL, lp, nobs, il)
    if rc == -3   # the mask is not per-input: the dense model on H = U sqrt(S)
        return invoke(logpdf_missing, Tuple{FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}}}},AbstractVector{<:Real}}, fx, y)
    end
    check(rc)
    return lp[]
end

# rrules of logpdf_missing, modelled on the two logpdf rrules above.  NaN entries of y get a zero tangent.
function ChainRulesCore.rrule(::typeof(logpdf_missing), fx::FiniteGP{<:ILMM{<:IndependentMOGP{<:Vector{<:GP}},<:Matrix{Float64}}},
                              y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs); m = length(descs)
    out = Ref{Float64}(0.0); gs2 = Ref{Float64}(0.0); nobs = Ref{Cint}(0); info = Ref{Cint}(0)
    gl = Matrix{Float64}(undef, 3, m); gy = Vector{Float64}(undef, length(y)); gH = similar(H)
    gt = Matrix{Float64}(undef, GRAD_TERM_DOUBLES, m)
    check(GC.@preserve keep ccall((:lmm_ilmm_masked_logpdf_grad, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
        ctx(), descs, m, X, length(x), D, H, size(H, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, out, gl, C_NULL, gs2, gy, gH, gt,
        nobs, info))
    function logpdf_missing_pullback(Δ)
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
        f_tangent = Tangent{typeof(fx.f)}(; H = Δ .* gH)
        return NoTangent(), Tangent{typeof(fx)}(; f = f_tangent, Σy = Σy_tangent), Δ .* gy
    end
    return out[], logpdf_missing_pullback
end
function ChainRulesCore.rrule(::typeof(logpdf_missing), fx::FiniteGP{<:OILMM{<:IndependentMOGP{<:Vector{<:GP}}}}, y::AbstractVector{<:Real})
    fs, H, σ², x = unpack(fx)
    X, D = points(x)
    descs, keep = gpdescs(fs.fs); m = length(descs)
    out = Ref{Float64}(0.0); gs2 = Ref{Float64}(0.0); nobs = Ref{Cint}(0); il = Ref{Cint}(-1)
    gl = Matrix{Float64}(undef, 3, m); gy = Vector{Float64}(undef, length(y))
    gU = Matrix{Float64}(undef, size(H, 1), m); gS = Vector{Float64}(undef, m)
    gt = Matrix{Float64}(undef, GRAD_TERM_DOUBLES, m)
    rc = GC.@preserve keep ccall((:lmm_oilmm_masked_logpdf_grad, liblmm), Cint,
        (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
        ctx(), descs, m, X, length(x), D, Matrix{Float64}(H.U), Vector{Float64}(diag(H.S)), size(H, 1), Float64(σ²),
        Vector{Float64}(y), fx.x.out_dim, out, gl, C_NULL, gs2, gy, gU, gS, gt, nobs, il)
    if rc == -3   # the mask is not per-input: the dense model on H = U sqrt(S), whose gradient is w.r.t. H
        Hm = Matrix{Float64}(collect(H)); gH = similar(Hm); info = Ref{Cint}(0)
        rc = GC.@preserve keep ccall((:lmm_ilmm_masked_logpdf_grad, liblmm), Cint,
            (Ptr{Cvoid}, Ptr{GpDesc}, Cint, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Cint,
             Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}, Ptr{Cint}),
            ctx(), descs, m, X, length(x), D, Hm, size(Hm, 1), Float64(σ²), Vector{Float64}(y), fx.x.out_dim, out, gl, C_NULL, gs2, gy, gH, gt,
            nobs, info)
    end
    check(rc)
    function logpdf_missing_pullback(Δ)
        Σy_tangent = Tangent{typeof(fx.Σy)}(; diag = Tangent{typeof(fx.Σy.diag)}(; value = Δ * gs2[]))
        return NoTangent(), Tangent{typeof(fx)}(; Σy = Σy_tangent), Δ .* gy
    end
    return out[], logpdf_missing_pullback
end

# --- one latent of a posterior on its own: mean_and_var(get_latent_gp(post).fs[i](x*, σ²)), the call src/oilmm.jl:61 makes ---
function AbstractGPs.mean_and_var(fx::FiniteGP{<:DeviceLatentPosterior})
    X, _ = points(fx.x)
    n = length(fx.x)
    M = Vector{Float64}(undef, n); V = Vector{Float64}(undef, n)
    check(ccall((:lmm_post_latent_mean_and_var, liblmm), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Float64}, Cint, Float64, Ptr{Float64}, Ptr{Float64}),
        fx.f.owner.handle, fx.f.index, X, n, Float64(noise_var(fx.Σy)), M, V))
    return M, V
end

# --- tunables and teardown ------------------------------------------------------------------------------------------
set_option(key::AbstractString, value::Real) = check(ccall((:lmm_ctx_set_option, liblmm), Cint, (Ptr{Cvoid}, Cstring, Float64), ctx(), key, Float64(value)))
version() = unsafe_string(ccall((:lmm_version, liblmm), Cstring, ()))
function __init__()
    atexit() do
        CTX[] == C_NULL || ccall((:lmm_ctx_destroy, liblmm), Cint, (Ptr{Cvoid},), CTX[])
        CTX[] = C_NULL
    end
end

# --- serialisable posterior: the on-disk form of a DevicePosterior -----------------------------------
save_posterior(p::DevicePosterior, path::AbstractString) = check(ccall((:lmm_post_save, liblmm), Cint, (Ptr{Cvoid}, Cstring), p.handle, path))
function load_posterior(path::AbstractString)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:lmm_post_load, liblmm), Cint, (Ptr{Cvoid}, Cstring, Ptr{Ptr{Cvoid}}), ctx(), path, h))
    return DevicePosterior(h[])
end

# PosteriorGP field access (α, C, δ) for one latent -- `lmm_post_export`
function export_latent(f::DeviceLatentPosterior, N::Int)
    L = Matrix{Float64}(undef, N, N); α = Vector{Float64}(undef, N); δ = Vector{Float64}(undef, N)
    check(ccall((:lmm_post_export, liblmm), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                f.owner.handle, f.index, L, α, δ))
    return (α = α, C = Cholesky(LowerTriangular(L)), δ = δ)
end

end # module
