"""GPU parity of what round 2 added around the Kriging loop: the IDW / LWR solvers on the same search kernel
(ref src/estimation/idw.jl, lwr.jl), the values-only update and plan reuse the conditional-simulation callers need
(ref src/simulation/fft.jl:112-126,184-188), traversal orders, and block supports of any size."""
import numpy as np
import pytest

from conftest import assert_parity

pytestmark = pytest.mark.gpu


def _samples(rng, n, box):
    coords = [rng.uniform(0.0, b, n) for b in box]
    vals = np.sin(coords[0] / 7.0) + 0.3 * rng.standard_normal(n)
    return coords, vals


def _simple_spec(gsk, rng, dim, n, grid, **kw):
    coords, vals = _samples(rng, n, grid)
    return gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, **kw)


# ---- IDW / LWR: local (neighbour lists), global (every sample), ball, exponents, zero distance ----
@pytest.mark.parametrize("solver", ["idw", "lwr"])
@pytest.mark.parametrize("dim,grid,n,k", [(2, (60, 50), 400, 8), (3, (20, 18, 16), 900, 12), (1, (300,), 60, 5),
                                          (2, (40, 40), 90, 0), (3, (12, 12, 12), 64, 0)])
def test_idw_lwr_vs_oracle(gsk, ctx, oracle, solver, dim, grid, n, k):
    rng = np.random.default_rng(1000 * dim + n + k)
    sv = gsk.SOLVER_IDW if solver == "idw" else gsk.SOLVER_LWR
    for expo in ((1.0, 2.0, 1.5) if solver == "idw" else (1.0,)):
        spec = _simple_spec(gsk, rng, dim, n, grid, solver=sv, idw_exponent=expo, max_neighbors=k)
        mean, sig, nn = ctx.krige(spec, want_nneigh=True)
        om, osig, onn, _ = oracle.krige(spec, want_neighbors=True)
        assert np.array_equal(nn, onn)
        # IDW is a convex combination: rtol 1e-9 (north_star). LWR solves (d+1)×(d+1) normal equations in raw
        # coordinates — cond ~ (extent/spacing)^2 — on both sides with the same pivoting; the differences are the
        # 1-ulp differences of exp() amplified by that: a few 1e-10 relative at most on these sizes
        tol = 1e-9 if solver == "idw" else 2e-8
        np.testing.assert_allclose(mean, om, rtol=tol, atol=tol)
        np.testing.assert_allclose(sig, osig, rtol=tol, atol=tol)


def test_idw_zero_distance_and_ball(gsk, ctx, oracle):
    """idw.jl:127-130: a neighbour at distance zero returns its value and σ = 0; ball search + minneighbors → missing"""
    gx, gy = np.meshgrid(np.arange(0.5, 20.0, 4.0), np.arange(0.5, 20.0, 4.0))
    coords = [gx.ravel().copy(), gy.ravel().copy()]                 # samples exactly on cell centroids
    vals = np.arange(coords[0].size, dtype=np.float64)
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(20, 20), solver=gsk.SOLVER_IDW, idw_exponent=2.0, max_neighbors=4)
    mean, sig, nn = ctx.krige(spec, want_nneigh=True)
    om, osig, _, _ = oracle.krige(spec, want_neighbors=True)
    assert np.array_equal(mean, om) or np.allclose(mean, om, rtol=1e-12, atol=0)
    hits = osig == 0.0
    assert hits.sum() == coords[0].size and np.array_equal(sig == 0.0, hits)
    lin = (np.floor(coords[1]).astype(int)) * 20 + np.floor(coords[0]).astype(int)
    assert np.array_equal(mean[lin], vals)
    ball = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(20, 20), solver=gsk.SOLVER_IDW, max_neighbors=4,
                           ball_radius=1.5, min_neighbors=2)
    mean, sig, nn = ctx.krige(ball, want_nneigh=True)
    om, osig, onn, _ = oracle.krige(ball, want_neighbors=True)
    assert np.array_equal(nn, onn) and np.array_equal(np.isnan(mean), np.isnan(om)) and np.isnan(mean).any()
    ok = ~np.isnan(om)
    np.testing.assert_allclose(mean[ok], om[ok], rtol=1e-9)


def test_idw_lwr_through_solve_units_and_reference_problems(gsk, ctx):
    """ref test/estimation/idw.jl:2-41, test/estimation/lwr.jl:15-31,61-76 through the mirrored solvers"""
    data = gsk.georef({"z": [1.0, 0.0, 1.0]}, [(25.0, 25.0), (50.0, 75.0), (75.0, 50.0)])
    grid = gsk.CartesianGrid(100, 100)
    prob = gsk.EstimationProblem(data, grid, "z")
    sol = gsk.solve(prob, gsk.IDWSolver(z=dict(maxneighbors=3)), ctx=ctx)
    z = np.asarray(sol.z)
    assert z.shape == (10000,) and np.all((z >= 0.0) & (z <= 1.0)) and "z_distance" in sol.names()
    Z = gsk.asarray(sol, "z")
    assert abs(Z[24, 24] - 1.0) < 5e-2 and abs(Z[49, 74] - 0.0) < 5e-2 and abs(Z[74, 49] - 1.0) < 5e-2   # cf. idw.jl:71-73
    order = gsk.traverse(grid, gsk.MultiGridPath())
    solp = gsk.solve(prob, gsk.IDWSolver(z=dict(maxneighbors=3, path=gsk.MultiGridPath())), ctx=ctx)
    assert np.array_equal(np.asarray(solp.z), z[order])
    for T in (gsk.Quantities([1.0, 0.0, 1.0], gsk.K), gsk.Quantities([-272.15, -273.15, -272.15], gsk.degC)):
        d = gsk.georef({"T": T}, [(25.0, 25.0), (50.0, 75.0), (75.0, 50.0)])
        p5 = gsk.EstimationProblem(d, gsk.CartesianGrid(5, 5), "T")
        s1 = gsk.solve(p5, gsk.IDWSolver(), ctx=ctx)
        assert gsk.elunit(s1["T"]) == gsk.K                                         # idw.jl:33,40
        s2 = gsk.solve(p5, gsk.LWRSolver(), ctx=ctx)
        assert gsk.elunit(s2["T"]) == gsk.K and gsk.elunit(s2["T_variance"]) == gsk.K ** 2   # lwr.jl:67-68,75-76
    d4 = gsk.georef({"z": [1.0, 0.0, 1.0, 0.0]}, [(25.0, 25.0), (50.0, 75.0), (75.0, 50.0), (75.0, 25.0)])
    p4 = gsk.EstimationProblem(d4, grid, "z")
    for kk in (3, 4):
        s = gsk.solve(p4, gsk.LWRSolver(z=dict(maxneighbors=kk)), ctx=ctx)           # lwr.jl:20-28
        assert np.all(np.isfinite(np.asarray(s.z))) and np.all(np.asarray(s["z_variance"]) >= 0)
    with pytest.raises(gsk.UnsupportedOption):
        gsk.solve(p4, gsk.LWRSolver(z=dict(weightfun=lambda h: 1 - h)), ctx=ctx)


# ---- traversal order through the C ABI ----
def test_target_order_is_visiting_order(gsk, ctx, oracle):
    spec = gsk.synth.config_spec("C2", scale=0.06)
    T = spec.n_targets
    order = np.random.default_rng(5).permutation(T).astype(np.int64)
    lin_mean, lin_var, lin_nn, lin_idx = ctx.krige(spec, want_neighbors=True)
    import copy
    sp = copy.copy(spec)
    sp.target_order = order
    mean, var, nn, idx = ctx.krige(sp, want_neighbors=True)
    assert np.array_equal(nn, lin_nn[order]) and np.array_equal(idx, lin_idx[order])
    assert np.array_equal(mean, lin_mean[order]) and np.array_equal(var, lin_var[order])
    om, ov, onn, oidx = oracle.krige(sp, want_neighbors=True)
    assert np.array_equal(idx, oidx)
    assert_parity(mean, var, om, ov)
    part = sp.with_slab(100, 777)                                    # slabs count positions of the path
    pm, pv = ctx.krige(part)
    assert np.array_equal(pm, mean[100:877]) and np.array_equal(pv, var[100:877])
    bad = copy.copy(spec)
    bad.target_order = np.full(T, T, dtype=np.int64)
    with pytest.raises(gsk.GskError):
        ctx.krige(bad)


# ---- values-only update / plan reuse ----
@pytest.mark.parametrize("shape", ["local_grid", "local_points", "global", "global_sk", "global_uk2"])
def test_update_values_equals_fresh_call(gsk, shape):
    rng = np.random.default_rng(11)
    if shape.startswith("global"):
        spec = gsk.synth.config_spec("C1", grid=(30, 30), n=200)
        if shape != "global":   # the SK value column holds z − μ; UK2 refines 6 drift weights
            est, deg = (gsk.EST_SIMPLE, 0) if shape == "global_sk" else (gsk.EST_UNIVERSAL, 2)
            spec = gsk.ProblemSpec(coords=spec.coords, values=spec.values, grid_dims=spec.grid_dims,
                                   support=spec.support, **dict(spec.params, estimator=est, uk_degree=deg,
                                                                sk_mean=float(spec.values.mean())))
    else:
        spec = gsk.synth.config_spec("C3a", scale=0.08)
        if shape == "local_points":
            T = 3000
            pts = [rng.uniform(0.0, g, T) for g in spec.grid_dims]
            spec = gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=pts, **{k: v for k, v in spec.params.items()})
    new_vals = spec.values[::-1].copy() + 0.25
    import copy
    spec2 = copy.copy(spec)
    spec2.values = new_vals
    with gsk.Context(0) as fresh:
        want_mean, want_var = fresh.krige(spec2)
    T = spec.n_targets
    import torch
    d_mean = torch.empty(T, dtype=torch.float64, device="cuda")
    d_var = torch.empty(T, dtype=torch.float64, device="cuda")
    with gsk.Context(0) as c:
        c.plan(spec)
        c.execute(0, T, d_mean.data_ptr(), d_var.data_ptr())
        c.synchronize()
        first = c.timing()
        c.update_values(new_vals)
        c.execute(0, T, d_mean.data_ptr(), d_var.data_ptr())
        c.synchronize()
        second = c.timing()
        assert np.array_equal(d_mean.cpu().numpy(), want_mean, equal_nan=True)
        assert np.array_equal(d_var.cpu().numpy(), want_var, equal_nan=True)
        if not shape.startswith("global"):
            assert second["launches"] < first["launches"]            # the search (and the bin sort) was skipped
        with pytest.raises(gsk.GskError):
            c.update_values(new_vals[:-1])
    # the same through gsk_krige with GSK_FLAG_REUSE_PLAN: identical inputs → nothing re-planned; new values → values only
    with gsk.Context(0) as c:
        a = copy.copy(spec); a.params = dict(spec.params, flags=spec.params["flags"] | gsk.FLAG_REUSE_PLAN)
        b = copy.copy(spec2); b.params = dict(a.params)
        m1, v1 = c.krige(a)
        assert c.timing()["ms_plan"] > 0
        m1b, v1b = c.krige(a)
        assert c.timing()["ms_plan"] == 0 and np.array_equal(m1, m1b, equal_nan=True) and np.array_equal(v1, v1b, equal_nan=True)
        m2, v2 = c.krige(b)
        assert c.timing()["ms_plan"] == 0
        assert np.array_equal(m2, want_mean, equal_nan=True) and np.array_equal(v2, want_var, equal_nan=True)
        moved = copy.copy(b); moved.coords = [x.copy() for x in b.coords]; moved.coords[0][0] += 1e-9
        c.krige(moved)
        assert c.timing()["ms_plan"] > 0                             # other coordinates: a new plan


# ---- block supports of any size (anisotropic cells, ranges below the cell side) ----
@pytest.mark.parametrize("k,est,deg", [(8, "OK", 0), (32, "UK", 1), (64, "OK", 0), (0, "OK", 0)])
def test_large_block_support(gsk, ctx, oracle, k, est, deg):
    spacing = [10.0, 10.0, 1.0]
    sup = gsk.default_support(spacing, 100.0)                        # 30 × 30 × 3 = 2700 points (ADVICE round 1)
    assert sup[0].shape[0] == 2700
    assert all(np.array_equal(a, b) for a, b in zip(sup, gsk.default_support_py(spacing, 100.0)))
    rng = np.random.default_rng(k + 3)
    n = 150
    coords = [rng.uniform(0, 60, n), rng.uniform(0, 50, n), rng.uniform(0, 5, n)]
    vals = rng.standard_normal(n)
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(6, 5, 5), grid_spacing=spacing, support=sup,
                           vario_kind=gsk.VARIO_SPHERICAL, vario_range=100.0, max_neighbors=k,
                           estimator=gsk.EST_UNIVERSAL if est == "UK" else gsk.EST_ORDINARY, uk_degree=deg)
    mean, var, nn, idx = ctx.krige(spec, want_neighbors=True)
    om, ov, onn, oidx = oracle.krige(spec, want_neighbors=True)
    assert np.array_equal(nn, onn) and (k == 0 or np.array_equal(idx, oidx))
    assert_parity(mean, var, om, ov, atol_mean=1e-10, atol_var=1e-10)


def test_uk2_3d_k96_large_support_fits_or_reports(gsk, ctx, oracle):
    """ADVICE round 1: UK degree 2 in 3-D with k = 96 and n_support = 125 needed more shared memory than sm_100 has;
    the support now moves to global memory when it does not fit"""
    rng = np.random.default_rng(96)
    n = 400
    coords = [rng.uniform(0, 30, n) for _ in range(3)]
    vals = rng.standard_normal(n)
    sup = gsk.default_support([1.0, 1.0, 1.0], 0.6)                  # ceil(1/0.2) = 5 per axis → 125 points
    assert sup[0].shape[0] == 125
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(6, 6, 6), grid_origin=(12.0, 12.0, 12.0), support=sup,
                           vario_kind=gsk.VARIO_EXPONENTIAL, vario_range=25.0, max_neighbors=96,
                           estimator=gsk.EST_UNIVERSAL, uk_degree=2)
    mean, var, nn, idx = ctx.krige(spec, want_neighbors=True)
    om, ov, onn, oidx = oracle.krige(spec, want_neighbors=True)
    assert np.array_equal(idx, oidx)
    assert_parity(mean, var, om, ov, atol_mean=1e-6, atol_var=1e-6)  # k = 96, UK2: cond·eps floor as in test_more_edge_shapes


# ---- the first caller of the Kriging path: FFT Gaussian simulation with conditioning (ref src/simulation/fft.jl) ----
def _numpy_fftgs(gsk, oracle, grid, gamma, mu, data_coords, data_vals, noises, maxneighbors=None):
    """fft.jl:62-192 restated with numpy FFTs and the CPU oracle for the two Kriging solves"""
    from gskrige.simulation import variogram_values
    dims = grid.dims
    cents = grid.centroids()
    ccen = [grid.origin[a] + (dims[a] // 2 - 1 + 0.5) * grid.spacing[a] for a in range(len(dims))]
    h = np.sqrt(sum((cents[a] - ccen[a]) ** 2 for a in range(len(dims))))
    C = np.reshape(gamma.sill - variogram_values(gamma, h), dims, order="F")
    F = np.sqrt(np.abs(np.fft.fftn(np.fft.fftshift(C))))
    F.flat[0] = 0.0

    def sk(coords, vals):
        spec = gsk.ProblemSpec(coords=coords, values=vals, points=cents, vario_kind=gamma.kind, vario_range=gamma.range,
                               vario_sill=gamma.sill, vario_nugget=gamma.nugget, estimator=gsk.EST_SIMPLE, sk_mean=mu,
                               max_neighbors=maxneighbors or 0)
        return oracle.krige(spec)[0]

    zbar = sk(data_coords, data_vals)
    ijk = [np.clip(np.floor((data_coords[a] - grid.origin[a]) / grid.spacing[a]).astype(np.int64), 0, dims[a] - 1) for a in range(len(dims))]
    lin = ijk[0] + dims[0] * ijk[1]
    _, first = np.unique(lin, return_index=True)
    dinds = lin[np.sort(first)]
    out = []
    for U in noises:
        P = F * np.exp(1j * np.angle(np.fft.fftn(U)))
        Z = np.real(np.fft.ifftn(P))
        Z = np.sqrt(gamma.sill / (np.sum(Z * Z) / (Z.size - 1))) * Z + mu
        zu = Z.reshape(-1, order="F")
        out.append(zbar + (zu - sk([c[dinds] for c in cents], zu[dinds].copy())))
    return out, dinds


@pytest.mark.parametrize("maxneighbors", [None, 3])
def test_fftgs_conditional_simulation(gsk, oracle, maxneighbors):
    """ref test/simulation/fft.jl:27-37 (conditional simulation on CartesianGrid(100,100), three data; here 40×30 so that
    the oracle's global solves stay small) with explicit noise fields, against the numpy + oracle restatement"""
    grid = gsk.CartesianGrid(40, 30)
    gamma = gsk.GaussianVariogram(range=10.0)
    dcoords = [np.array([10.0, 20.2, 30.7, 5.5, 20.9]), np.array([10.0, 22.4, 14.1, 25.5, 22.1])]   # two data share a cell
    dvals = np.array([1.0, -1.0, 1.0, 0.3, -0.7])
    data = gsk.georef({"z": dvals}, np.stack(dcoords, 0))
    rng = np.random.default_rng(2022)
    noises = [rng.random(grid.dims) for _ in range(3)]
    params = dict(variogram=gamma) if maxneighbors is None else dict(variogram=gamma, maxneighbors=maxneighbors)
    solver = gsk.FFTGS(z=params, rng=1)
    problem = gsk.SimulationProblem(data, grid, "z", 3)
    with gsk.Context(0) as c:
        pre = gsk.simulation.preprocess_fftgs(problem, solver, c)
        want, dinds = _numpy_fftgs(gsk, oracle, grid, gamma, 0.0, dcoords, dvals, noises, maxneighbors)
        assert np.array_equal(pre["dinds"], dinds) and len(dinds) == 4
        plans = []
        for U, w in zip(noises, want):
            z = gsk.simulation.solvesingle_fftgs(problem, solver, pre, c, noise=U)
            plans.append(c.timing()["ms_plan"])
            # cuFFT vs pocketfft: 1e-13 relative on the field; the Gaussian SK systems amplify by their condition number
            np.testing.assert_allclose(z, w, rtol=1e-7, atol=1e-7)
            # conditioning: the simulated field honours the data at the data cells' centroids in expectation only
            # (fft.jl conditions on cell centroids); what must hold exactly is z = zbar + (zu - zbar_u) at every cell
            assert np.all(np.isfinite(z))
        assert plans[0] > 0 and plans[1] == 0 and plans[2] == 0      # realisations 2, 3: same coordinates → values only
        sols = gsk.solve(problem, solver, ctx=c)
        assert len(sols) == 3 and sols[0].z.shape == (1200,)
    # unconditional: realisations are rescaled to the sill
    sols = gsk.solve(gsk.SimulationProblem(grid, "z", 2), gsk.FFTGS(z=dict(variogram=gamma), rng=3))
    for s in sols:
        z = np.asarray(s.z)
        assert abs(np.sum(z * z) / (z.size - 1) - 1.0) < 1e-9


# ---- LU Gaussian simulation (ref src/simulation/lu.jl): dense joint factor + one triangular product per realisation ----
@pytest.mark.parametrize("conditional", [False, True])
def test_lugs_vs_numpy_cholesky(gsk, conditional):
    """lu.jl:118-133 (C11, C12, C22, L11, B12, d2, L22) and lusim (lu.jl:198-224) restated with numpy's Cholesky"""
    from gskrige.simulation import variogram_values, preprocess_lugs, lusim
    grid = gsk.CartesianGrid(24, 20)
    gamma = gsk.SphericalVariogram(range=9.0, sill=1.3, nugget=0.1)
    rng = np.random.default_rng(4)
    if conditional:
        dcoords = [np.array([3.2, 10.7, 20.1, 3.4, 15.5]), np.array([2.2, 11.3, 17.9, 2.6, 5.5])]   # data 0 and 3 share a cell
        dvals = np.array([0.8, -0.4, 1.1, 0.6, -1.2])
        problem = gsk.SimulationProblem(gsk.georef({"z": dvals}, np.stack(dcoords, 0)), grid, "z", 2)
    else:
        problem = gsk.SimulationProblem(grid, "z", 2)
    solver = gsk.LUGS(z=dict(variogram=gamma, mean=None if conditional else 2.5), rng=9)
    with gsk.Context(0) as c:
        pre = preprocess_lugs(problem, solver, "z", c)
        dlocs, slocs = pre["dlocs"], pre["slocs"]
        cents = np.stack(grid.centroids(), 1)
        cov = lambda A, B: gamma.sill - variogram_values(gamma, np.sqrt(((A[:, None, :] - B[None, :, :]) ** 2).sum(-1)))
        S = cents[slocs]
        C22 = cov(S, S)
        if conditional:
            assert len(dlocs) == 4 and pre["z1"].tolist() == [0.6, -1.2, -0.4, 1.1]       # the later datum wins its cell
            D = cents[dlocs]
            L11 = np.linalg.cholesky(cov(D, D))
            B12 = np.linalg.solve(L11, cov(D, S))
            d2 = B12.T @ np.linalg.solve(L11, pre["z1"])
            L22 = np.linalg.cholesky(C22 - B12.T @ B12)
        else:
            d2, L22 = 0.0, np.linalg.cholesky(C22)
        for _ in range(2):
            w = rng.standard_normal(len(slocs))
            y = lusim(c, pre, w)
            want = np.empty(grid.nelements())
            want[dlocs] = pre["z1"]
            want[slocs] = d2 + L22 @ w
            if not conditional:
                want += 2.5
            np.testing.assert_allclose(y, want, rtol=1e-9, atol=1e-10)
        w1, w2 = rng.standard_normal(len(slocs)), rng.standard_normal(len(slocs))
        y2 = lusim(c, pre, w2, rho=0.6, w1=w1)                                             # lu.jl:213
        np.testing.assert_allclose(y2[slocs] - (2.5 if not conditional else 0.0), d2 + L22 @ (0.6 * w1 + 0.8 * w2), rtol=1e-9, atol=1e-10)
        with pytest.raises(gsk.GskError):
            c.plan(gsk.synth.config_spec("C2", scale=0.05)) or c.lu_sample(w)               # a Kriging plan replaces the LU plan
        sols = gsk.solve(problem, solver, ctx=c)
        assert len(sols) == 2 and np.asarray(sols[0].z).shape == (480,)
    with pytest.raises(gsk.UnsupportedOption):
        gsk.LUGS(z=dict(factorization="lu")).params("z")
