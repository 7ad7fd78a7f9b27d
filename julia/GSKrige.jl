# GSKrige.jl — Julia shim that keeps `solve(problem, KrigingSolver(...))` drop-in while the per-location
# loops run in libgskrige.so (B200, sm_100a). It mirrors the host logic of the reference
# (GeoStatsSolvers.jl v0.7.16, src/estimation/krig.jl:76-164, src/ui.jl:11-50, src/utils.jl:5-15) and
# replaces exactly two functions — exactsolve (krig.jl:166-186) and approxsolve (krig.jl:188-234) — by a
# single `ccall` each. NOTE: Julia is not installed in the build or GPU images of this repository, so this
# file is NOT executed by the test-suite (UNTESTED until julia/verify_semantics.jl and a smoke call have run under a real
# Julia install with the pinned packages); geostatssolvers.jl_b200/host.py is the same logic in Python and
# is what the tests exercise. julia/verify_semantics.jl prints the third-party behaviours (SURVEY V1-V9)
# a maintainer with a Julia install should confirm.
module GSKrige

using GeoStatsBase, GeoStatsModels, Variography, Meshes, GeoTables, Tables, Unitful, Distances
import GeoStatsSolvers                       # kriging_ui / searcher_ui (src/ui.jl) and the solver types are the reference's own
import GeoStatsSolvers: KrigingSolver, IDWSolver, LWRSolver, SGS
using Random
import GeoStatsBase: solve, preprocess

# `north_star` spells the solver `Kriging(...)` (the name older GeoStats releases used); the reference's type is
# `KrigingSolver` (src/estimation/krig.jl:64)
const Kriging = KrigingSolver

const LIB = get(ENV, "GSKRIGE_LIB", joinpath(@__DIR__, "..", "geostatssolvers.jl_b200", "csrc", "libgskrige.so"))

# ---- struct gsk_problem (include/gskrige.h), field for field -----------------------------------------
struct GskProblem
  abi_version::Int32
  dim::Int32
  n_samples::Int64
  coords::NTuple{3,Ptr{Float64}}
  values::Ptr{Float64}
  grid_dims::NTuple{3,Int64}
  grid_origin::NTuple{3,Float64}
  grid_spacing::NTuple{3,Float64}
  n_points::Int64
  point_coords::NTuple{3,Ptr{Float64}}
  target_first::Int64
  target_count::Int64
  n_support::Int32
  support_offsets::NTuple{3,Ptr{Float64}}
  vario_kind::Int32
  vario_range::Float64
  vario_sill::Float64
  vario_nugget::Float64
  gaussian_nugget_eps::Float64
  estimator::Int32
  sk_mean::Float64
  uk_degree::Int32
  min_neighbors::Int32
  max_neighbors::Int32
  ball_radius::Float64
  flags::UInt32
  target_order::Ptr{Int64}
  solver::Int32
  idw_exponent::Float64
  lwr_weightfun::Int32
end

mutable struct Context
  handle::Ptr{Cvoid}
  function Context(device::Integer=0)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:gsk_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint), h, device)
    rc == 0 || error("libgskrige: ", unsafe_string(ccall((:gsk_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL)))
    ctx = new(h[])
    finalizer(c -> ccall((:gsk_destroy, LIB), Cvoid, (Ptr{Cvoid},), c.handle), ctx)
  end
end

const DEFAULT = Ref{Union{Nothing,Context}}(nothing)
context() = (DEFAULT[] === nothing && (DEFAULT[] = Context(0)); DEFAULT[])

check(ctx, rc) = rc == 0 ? nothing :
  (msg = unsafe_string(ccall((:gsk_last_error, LIB), Cstring, (Ptr{Cvoid},), ctx.handle));
   rc == -2 ? throw(ArgumentError("unsupported by the B200 Kriging path (no CPU fallback): $msg")) : error("libgskrige ($rc): $msg"))

# ---- what crosses the ABI ------------------------------------------------------------------------------
variokind(::GaussianVariogram) = Int32(0)
variokind(::SphericalVariogram) = Int32(1)
variokind(::ExponentialVariogram) = Int32(2)
variokind(γ) = throw(ArgumentError("variogram $(typeof(γ)) is not supported by the B200 Kriging path"))

function support_offsets(pdomain::CartesianGrid, γ)
  dim = embeddim(pdomain)
  sp = collect(Float64, ustrip.(spacing(pdomain)))
  sig = (Cint, Ptr{Float64}, Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint)
  n = ccall((:gsk_default_support, LIB), Cint, sig, dim, sp, ustrip(range(γ)), C_NULL, C_NULL, C_NULL, 0)   # count only
  n > 0 || throw(ArgumentError("the block support of this cell size / variogram range is too large for the B200 Kriging path"))
  bufs = [zeros(n) for _ in 1:3]
  m = ccall((:gsk_default_support, LIB), Cint, sig, dim, sp, ustrip(range(γ)), bufs[1], bufs[2], bufs[3], n)
  m == n || error("gsk_default_support failed")
  bufs[1:dim]
end
support_offsets(pdomain, γ) = [zeros(1) for _ in 1:embeddim(pdomain)]  # PointSet targets: point support

"""
the visiting order of `path` as 0-based linear indices (what `traverse(pdomain, path)` yields, krig.jl:179,204), or
`nothing` for LinearPath. The reference returns its predictions in this order without permuting back; passing the
order across the ABI (gsk_problem.target_order) reproduces exactly that.
"""
pathorder(pdomain, ::LinearPath) = nothing
pathorder(pdomain, path) = Int64[i - 1 for i in traverse(pdomain, path)]

"one ccall: replaces exactsolve / approxsolve (krig.jl:166-234) — or the IDW / LWR loops (idw.jl:112-142, lwr.jl:113-146)"
function krige(samples, pdomain, var, estimator, searcher, minneighbors, islocal::Bool; ctx=context(), path=LinearPath(),
               devices=nothing, solverkind::Int32=Int32(0), exponent::Float64=1.0, γ=nothing)
  γ = isnothing(estimator) ? γ : estimator.γ
  sdom = domain(samples)
  dim = embeddim(sdom)
  n = nelements(sdom)
  X = [Float64[ustrip(coordinates(centroid(sdom, i))[d]) for i in 1:n] for d in 1:dim]       # SoA
  z = collect(Float64, ustrip.(getproperty(samples, var)))
  sup = (isnothing(γ) || solverkind != 0) ? [zeros(1) for _ in 1:dim] : support_offsets(pdomain, γ)
  T = nelements(pdomain)
  isgrid = pdomain isa CartesianGrid
  P = isgrid ? [Float64[] for _ in 1:dim] : [Float64[ustrip(coordinates(centroid(pdomain, i))[d]) for i in 1:T] for d in 1:dim]
  order = pathorder(pdomain, path)
  tup(v, fill) = ntuple(d -> d <= length(v) ? v[d] : fill, 3)
  ptrs(v) = ntuple(d -> d <= length(v) ? pointer(v[d]) : Ptr{Float64}(C_NULL), 3)
  est, skmean, deg = isnothing(estimator) ? (Int32(1), 0.0, Int32(0)) :
                     estimator isa GeoStatsModels.SimpleKriging ? (Int32(0), Float64(ustrip(estimator.μ)), Int32(0)) :
                     estimator isa GeoStatsModels.UniversalKriging ? (Int32(2), 0.0, Int32(maximum(estimator.exponents))) :
                     estimator isa GeoStatsModels.OrdinaryKriging ? (Int32(1), 0.0, Int32(0)) :
                     throw(ArgumentError("ExternalDriftKriging (`drifts`) is not supported by the B200 Kriging path"))
  k = islocal ? Int32(maxneighbors(searcher)) : Int32(0)            # the CLAMPED k (ui.jl:16-23)
  radius = (islocal && searcher isa KBallSearch) ? Float64(ustrip(Meshes.radius(searcher.ball))) : NaN
  μ = Vector{Float64}(undef, T); σ² = Vector{Float64}(undef, T); nn = Vector{Int32}(undef, T)
  GC.@preserve X z sup P μ σ² nn order begin
    prob = GskProblem(2, dim, n, ptrs(X), pointer(z),
      isgrid ? tup(collect(Int64, size(pdomain)), 1) : (0, 1, 1),
      isgrid ? tup(collect(Float64, ustrip.(coordinates(minimum(pdomain)))), 0.0) : (0.0, 0.0, 0.0),
      isgrid ? tup(collect(Float64, ustrip.(spacing(pdomain))), 1.0) : (1.0, 1.0, 1.0),
      isgrid ? 0 : T, ptrs(P), 0, -1, length(sup[1]), ptrs(sup),
      isnothing(γ) ? Int32(1) : variokind(γ), isnothing(γ) ? 1.0 : ustrip(range(γ)), isnothing(γ) ? 1.0 : ustrip(sill(γ)),
      isnothing(γ) ? 0.0 : ustrip(nugget(γ)), 1e-6,
      est, skmean, deg, Int32(minneighbors), k, radius, UInt32(3),
      isnothing(order) ? Ptr{Int64}(C_NULL) : pointer(order), solverkind, exponent, Int32(0))
    if isnothing(devices)
      check(ctx, ccall((:gsk_krige, LIB), Cint,
        (Ptr{Cvoid}, Ref{GskProblem}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
        ctx.handle, prob, μ, σ², nn, C_NULL))
    else
      # all GPUs of the box from this one process: the target range is cut into one contiguous piece per device
      # (samples replicated, one host thread and one cached context per piece), results land in μ / σ² directly
      devs = collect(Cint, devices)
      err = zeros(UInt8, 512)
      rc = ccall((:gsk_krige_multi, LIB), Cint,
        (Ptr{Cint}, Cint, Ref{GskProblem}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{UInt8}, Cint),
        devs, length(devs), prob, μ, σ², nn, C_NULL, err, 512)
      rc == 0 || (rc == -2 ? throw(ArgumentError("unsupported by the B200 Kriging path: " * unsafe_string(pointer(err)))) :
                             error("libgskrige ($rc): " * unsafe_string(pointer(err))))
    end
  end
  if islocal && any(<(max(minneighbors, 1)), nn)                    # krig.jl:213-214 → (missing, missing)
    miss = nn .< max(minneighbors, 1)
    return ifelse.(miss, missing, μ), ifelse.(miss, missing, σ²)
  end
  μ, σ²
end

# ---- the reference's host logic, unchanged in behaviour (krig.jl:76-164) -------------------------------
elunit(x) = typeunit(eltype(x))
typeunit(::Type) = NoUnits
typeunit(::Type{Q}) where {Q<:Quantity} = unit(Q)
uadjust(x) = uadjust(elunit(x), x)
uadjust(::Unitful.Units, x) = x
uadjust(U::Unitful.AffineUnits, x) = uconvert.(absoluteunit(U), x)

"""
drop-in for GeoStatsSolvers.solve(problem, ::KrigingSolver); `solver` is the reference's own solver object.
`devices = 0:7` drives all GPUs of the box from this process (gsk_krige_multi).
"""
function solve_b200(problem::EstimationProblem, solver::KrigingSolver; ctx=context(), devices=nothing)
  pdata = data(problem); dtable = values(pdata); ddomain = domain(pdata); pdomain = domain(problem)
  μs = []; σs = []
  for covars in covariables(problem, solver), var in covars.names
    p = covars.params[Set([var])]
    p.distance isa Euclidean || throw(ArgumentError("non-Euclidean `distance` is not supported by the B200 Kriging path"))
    z = uadjust(Tables.getcolumn(Tables.columns(dtable), var))                     # krig.jl:94
    inds = findall(!ismissing, z)                                                  # krig.jl:97
    isempty(inds) && throw(AssertionError("all samples of $var are missing, aborting..."))   # krig.jl:100-102
    samples = georef((; var => collect(skipmissing(z))), view(ddomain, inds))      # krig.jl:105-107
    estimator = GeoStatsSolvers.kriging_ui(pdomain, p.variogram, p.mean, p.degree, p.drifts)        # ui.jl:40-50
    searcher = GeoStatsSolvers.searcher_ui(domain(samples), p.maxneighbors, p.distance, p.neighborhood)  # ui.jl:11-32 (warns + clamps)
    varμ, varσ = krige(samples, pdomain, var, estimator, searcher, p.minneighbors, !isnothing(p.maxneighbors);
                       ctx, path=p.path, devices)                                  # krig.jl:151-157
    u = elunit(z)
    push!(μs, var => (u == NoUnits ? varμ : varμ .* u))
    push!(σs, Symbol(var, "_variance") => (u == NoUnits ? varσ : varσ .* u^2))      # krig.jl:160
  end
  georef((; μs..., σs...), pdomain)                                                # krig.jl:163
end

"""
leave-one-out cross-validation of `data` with `solver` (what GeoStatsValidation's `LeaveOneOut` computes by solving one
fold per sample): per variable one gsk_krige_loo call; row i is sample i kriged at its own location from the other
non-missing samples. Returns `var` and `var_variance` on the data domain in data order, `missing` where the value is
missing or fewer than `minneighbors` neighbours remain. Each fold holds n − 1 samples, so `maxneighbors` is clamped to
n − 1 by the fold's own `searcher_ui`; `path` does not apply.
"""
function leaveoneout_b200(data, solver::KrigingSolver; ctx=context())
  dtable = values(data); ddomain = domain(data)
  μs = []; σs = []
  for covars in covariables(EstimationProblem(data, ddomain, Tables.columnnames(Tables.columns(dtable))), solver),
      var in covars.names
    p = covars.params[Set([var])]
    p.distance isa Euclidean || throw(ArgumentError("non-Euclidean `distance` is not supported by the B200 Kriging path"))
    z = uadjust(Tables.getcolumn(Tables.columns(dtable), var))
    inds = findall(!ismissing, z)
    n = length(inds)
    n >= 2 || throw(AssertionError("leave-one-out of $var needs at least two non-missing samples"))
    sdom = view(ddomain, inds)
    estimator = GeoStatsSolvers.kriging_ui(sdom, p.variogram, p.mean, p.degree, p.drifts)
    islocal = !isnothing(p.maxneighbors)
    fold = view(ddomain, inds[1:n-1])                                              # any fold: n − 1 samples
    searcher = GeoStatsSolvers.searcher_ui(fold, p.maxneighbors, p.distance, p.neighborhood)  # the fold's clamp + warning
    γ = estimator.γ
    dim = embeddim(sdom)
    X = [Float64[ustrip(coordinates(centroid(sdom, i))[d]) for i in 1:n] for d in 1:dim]
    zs = collect(Float64, ustrip.(z[inds]))
    est, skmean, deg = estimator isa GeoStatsModels.SimpleKriging ? (Int32(0), Float64(ustrip(estimator.μ)), Int32(0)) :
                       estimator isa GeoStatsModels.UniversalKriging ? (Int32(2), 0.0, Int32(maximum(estimator.exponents))) :
                       estimator isa GeoStatsModels.OrdinaryKriging ? (Int32(1), 0.0, Int32(0)) :
                       throw(ArgumentError("ExternalDriftKriging (`drifts`) is not supported by the B200 Kriging path"))
    k = islocal ? Int32(maxneighbors(searcher)) : Int32(0)
    radius = (islocal && searcher isa KBallSearch) ? Float64(ustrip(Meshes.radius(searcher.ball))) : NaN
    ptrs(v) = ntuple(d -> d <= length(v) ? pointer(v[d]) : Ptr{Float64}(C_NULL), 3)
    μ = Vector{Float64}(undef, n); σ² = Vector{Float64}(undef, n); nn = Vector{Int32}(undef, n)
    GC.@preserve X zs μ σ² nn begin
      prob = GskProblem(2, dim, n, ptrs(X), pointer(zs), (0, 1, 1), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0),
        0, ntuple(_ -> Ptr{Float64}(C_NULL), 3), 0, -1, 1, ntuple(_ -> Ptr{Float64}(C_NULL), 3),
        variokind(γ), ustrip(range(γ)), ustrip(sill(γ)), ustrip(nugget(γ)), 1e-6,
        est, skmean, deg, Int32(p.minneighbors), k, radius, UInt32(3), Ptr{Int64}(C_NULL), Int32(0), 1.0, Int32(0))
      check(ctx, ccall((:gsk_krige_loo, LIB), Cint,
        (Ptr{Cvoid}, Ref{GskProblem}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
        ctx.handle, prob, μ, σ², nn, C_NULL))
    end
    T = nelements(ddomain)
    varμ = Vector{Union{Missing,Float64}}(missing, T); varσ = Vector{Union{Missing,Float64}}(missing, T)
    ok = nn .>= max(p.minneighbors, 1)
    varμ[inds[ok]] .= μ[ok]; varσ[inds[ok]] .= σ²[ok]
    u = elunit(z)
    push!(μs, var => (u == NoUnits ? varμ : varμ .* u))
    push!(σs, Symbol(var, "_variance") => (u == NoUnits ? varσ : varσ .* u^2))
  end
  georef((; μs..., σs...), ddomain)
end

"drop-in for GeoStatsSolvers.solve(problem, ::IDWSolver) (idw.jl:59-148) and ::LWRSolver (lwr.jl:62-152)"
function solve_b200(problem::EstimationProblem, solver::Union{IDWSolver,LWRSolver}; ctx=context(), devices=nothing)
  pdata = data(problem); dtable = values(pdata); ddomain = domain(pdata); pdomain = domain(problem)
  isidw = solver isa IDWSolver
  μs = []; σs = []
  for covars in covariables(problem, solver), var in covars.names
    p = covars.params[Set([var])]
    p.distance isa Euclidean || throw(ArgumentError("non-Euclidean `distance` is not supported by the B200 path"))
    dvals = Tables.getcolumn(Tables.columns(dtable), var)
    dinds = findall(!ismissing, dvals)                                             # idw.jl:78 / lwr.jl:81
    sdom = view(ddomain, dinds)
    n = nelements(sdom)
    nmin = p.minneighbors
    nmax = isnothing(p.maxneighbors) ? n : min(p.maxneighbors, n)
    @assert n > 0 "estimation requires data"
    isidw && @assert p.exponent > 0 "exponent must be positive"
    @assert nmin ≤ nmax "invalid min/max number of neighbors"
    isidw || p.weightfun(0.5) == exp(-3 * 0.5^2) || throw(ArgumentError("only the default `weightfun` crosses the C ABI"))
    searcher = GeoStatsSolvers.searcher_ui(sdom, p.maxneighbors, p.distance, p.neighborhood)
    z = uadjust(collect(skipmissing(dvals)))
    samples = georef((; var => ustrip.(z)), sdom)
    μ, σ = krige(samples, pdomain, var, nothing, searcher, nmin, !isnothing(p.maxneighbors); ctx, path=p.path, devices,
                 solverkind=Int32(isidw ? 1 : 2), exponent=Float64(isidw ? p.exponent : 1.0))
    u = elunit(z)
    push!(μs, var => (u == NoUnits ? μ : μ .* u))
    if isidw
      push!(σs, Symbol(var, "_distance") => σ)                                      # idw.jl:146
    else
      push!(σs, Symbol(var, "_variance") => (u == NoUnits ? σ : σ .* u^2))           # lwr.jl:152
    end
  end
  georef((; μs..., σs...), pdomain)
end

"""
drop-in for GeoStatsSolvers.solve(problem, ::SGS) (sgs.jl:56-89 → seq.jl:76-141), one variable: the masked searches, the
Simple Kriging fits and the weights of every location of the path are computed at once (gsk_sgs_plan); the `nreals`
realisations are then one gsk_sgs_sample call. The draws are `randn(solver.rng)` in path order — the numbers
`rand(rng, Normal(μ, σ))` consumes in the reference's loop (seq.jl:110,130), so a seeded solver gives the same
realisations as the reference up to the rounding of the kriging systems.
"""
function solve_b200(problem::SimulationProblem, solver::SGS; ctx=context())
  pdata = data(problem); pdomain = domain(problem); pvars = variables(problem)
  N = nelements(pdomain); dim = embeddim(pdomain)
  X = [Float64[ustrip(coordinates(centroid(pdomain, i))[d]) for i in 1:N] for d in 1:dim]      # seq.jl:91
  buff, mask = GeoStatsBase.initbuff(pdomain, pvars, solver.init, data=pdata)                 # seq.jl:88
  reals = []
  for covars in covariables(problem, solver), var in covars.names
    p = covars.params[Set([var])]
    p.distance isa Euclidean || throw(ArgumentError("non-Euclidean `distance` is not supported by the B200 path"))
    γ = p.variogram
    searcher = GeoStatsSolvers.searcher_ui(pdomain, p.maxneighbors, p.distance, p.neighborhood)  # seq.jl:66
    radius = searcher isa KBallSearch ? Float64(ustrip(Meshes.radius(searcher.ball))) : NaN
    simulated = mask[var]
    visit = [i for i in traverse(pdomain, p.path) if !simulated[i]]                            # seq.jl:102-103
    rank = fill(Int64(-1), N); rank[visit] .= 0:(length(visit) - 1)
    vals = Float64[simulated[i] ? buff[var][i] : 0.0 for i in 1:N]
    nreals = GeoStatsBase.nreals(problem)
    z = zeros(N, nreals)
    for r in 1:nreals, i in visit
      z[i, r] = randn(solver.rng)
    end
    out = Matrix{Float64}(undef, N, nreals)
    GC.@preserve X rank vals z out begin
      ptrs = ntuple(d -> d <= dim ? pointer(X[d]) : Ptr{Float64}(C_NULL), 3)
      check(ctx, ccall((:gsk_sgs_plan, LIB), Cint,
        (Ptr{Cvoid}, Cint, Int64, Ref{NTuple{3,Ptr{Float64}}}, Ptr{Int64}, Cint, Float64, Float64, Float64, Float64, Float64,
         Cint, Cint, Float64),
        ctx.handle, dim, N, ptrs, rank, variokind(γ), ustrip(range(γ)), ustrip(sill(γ)), ustrip(nugget(γ)), 1e-6,
        Float64(p.mean), p.minneighbors, maxneighbors(searcher), radius))
      check(ctx, ccall((:gsk_sgs_sample, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        ctx.handle, nreals, vals, z, out))
    end
    push!(reals, var => [out[:, r] for r in 1:nreals])
  end
  Ensemble(pdomain, Dict(reals))
end

end # module
