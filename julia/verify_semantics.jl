# verify_semantics.jl — run on a machine WITH Julia and the pinned packages (GeoStatsSolvers 0.7.16 ⇒
# GeoStatsModels 0.2, Variography 0.22, Meshes 0.37) to close the [3P-RECALLED] checklist of SURVEY.md §8c.
# Each line prints what oracle/gsk_oracle.c and libgskrige.so assume; a mismatch means flipping the
# corresponding switch in gsk_problem (support offsets, gaussian_nugget_eps, flags) — no code change.
using GeoStatsSolvers, GeoStatsModels, Variography, Meshes, GeoTables, LinearAlgebra

println("V1 block support of a unit 2-D cell (expect 9 points at {0.25,0.5,0.75}²):")
q = Quadrangle((0.0, 0.0), (1.0, 0.0), (1.0, 1.0), (0.0, 1.0))
println(collect(Variography._sample(GaussianVariogram(range=35.0), q)))
println("V2 Gaussian nugget epsilon (expect γ(1e-9) ≈ 1e-6): ", GaussianVariogram(range=35.0)(1e-9))
println("V4 UK exponents degree 1, dim 3 (expect x,y,z,1): ", GeoStatsModels.UniversalKriging(GaussianVariogram(), 1, 3).exponents)
println("V4 UK exponents degree 2, dim 2 (expect x²,y²,x,y,xy,1): ", GeoStatsModels.UniversalKriging(GaussianVariogram(), 2, 2).exponents)
data = georef((; z=[1.0, 0.0, 1.0]), [(25.0, 25.0), (50.0, 75.0), (75.0, 50.0)])
grid = CartesianGrid((100, 100), (0.5, 0.5), (1.0, 1.0))
println("V9 centroid(grid, 1) (expect (1.0, 1.0)): ", centroid(grid, 1))
sol = solve(EstimationProblem(data, grid, :z), KrigingSolver(:z => (variogram=GaussianVariogram(range=35.0, nugget=0.0), maxneighbors=3)))
# compare with:  python -c "import gskrige, oracle_py; ..."  (tests/_cases.py: ref_problem_2d)
println("known answer: mean[1:3] = ", sol.z[1:3], "  var[1:3] = ", sol.z_variance[1:3])
println("expected from the oracle: mean[0:3] and var[0:3] of tests/_cases.ref_problem_2d(k=3)")

# leave-one-out: GSKrige.leaveoneout_b200 against the reference's folds — sample i deleted, kriged at its own location
# by KrigingSolver (what GeoStatsValidation's LeaveOneOut solves per fold). Needs libgskrige.so and a B200.
include(joinpath(@__DIR__, "GSKrige.jl"))
xy = [(Float64(i % 7) + 0.3 * (i % 3), Float64(i ÷ 7) + 0.2 * (i % 5)) for i in 0:48]
loodata = georef((; z=[sin(p[1] / 2) + cos(p[2] / 3) for p in xy]), xy)
for params in ((variogram=SphericalVariogram(range=4.0), maxneighbors=8), (variogram=ExponentialVariogram(range=5.0),))
  solver = KrigingSolver(:z => params)
  loo = GSKrige.leaveoneout_b200(loodata, solver)
  worst = 0.0
  for i in 1:length(xy)
    keep = setdiff(1:length(xy), i)
    fold = georef((; z=loodata.z[keep]), xy[keep])
    ref = solve(EstimationProblem(fold, PointSet([xy[i]]), :z), solver)
    worst = max(worst, abs(ref.z[1] - loo.z[i]), abs(ref.z_variance[1] - loo.z_variance[i]))
  end
  println("leave-one-out ", params, ": largest |reference fold − leaveoneout_b200| = ", worst, " (expect < 1e-9)")
end
