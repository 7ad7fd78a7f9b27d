"""Parity tests proper: the CUDA path, called through the C ABI (libgskrige.so via ctypes), against
the CPU oracle on identical inputs — neighbour sets bit-exact, mean/variance rtol 1e-9 (Float64),
plus the reference's own known-answer checks through the mirrored `solve` API and the committed
golden vectors. Sizes are such that the oracle finishes in seconds; BASELINE-size cases are checked
on random target subsets and through size-independent properties."""
import numpy as np
import pytest

from _cases import CASES, GOLDEN, build_case, ref_problem_1d, ref_problem_2d
from conftest import assert_parity

pytestmark = pytest.mark.gpu


def _both(ctx, oracle, spec, search=None):
    search = oracle.SEARCH_KDTREE if search is None else search
    g = ctx.krige(spec, want_neighbors=True)
    o = oracle.krige(spec, search=search, want_neighbors=True)
    return g, o


def _check(gsk, ctx, oracle, spec, **tol):
    (mean, var, nn, idx), (om, ov, onn, oidx) = _both(ctx, oracle, spec)
    assert np.array_equal(nn, onn)
    if spec.params["max_neighbors"] > 0:
        assert np.array_equal(idx, oidx)          # bit-exact neighbour sets, sorted by (d², idx)
    assert_parity(mean, var, om, ov, scale=max(1.0, np.abs(spec.values).max()), sill=spec.params["vario_sill"], **tol)
    return mean, var


# ---- the reference's own tests, through the mirrored public API (test/estimation/krig.jl) ----
def test_reference_testset_through_solve(gsk, ctx):
    g35 = gsk.GaussianVariogram(range=35.0, nugget=0.0)
    data1d = gsk.georef({"z": [0.0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.4, 0.3, 0.2, 0.1, 0.0]}, np.arange(0.0, 101.0, 10.0)[None, :])
    prob1d = gsk.EstimationProblem(data1d, gsk.CartesianGrid(100), "z")
    for params in (dict(variogram=g35), dict(variogram=g35, maxneighbors=3),
                   dict(variogram=g35, maxneighbors=3, neighborhood=gsk.MetricBall(100.0))):
        sol = gsk.solve(prob1d, gsk.KrigingSolver(z=params), ctx=ctx)               # krig.jl:6-19 (smoke)
        assert np.all(np.isfinite(np.asarray(sol.z))) and np.all(np.asarray(sol["z_variance"]) >= 0)
    data2d = gsk.georef({"z": [1.0, 0.0, 1.0]}, [(25.0, 25.0), (50.0, 75.0), (75.0, 50.0)])
    grid2d = gsk.CartesianGrid((100, 100), (0.5, 0.5), (1.0, 1.0))
    prob2d = gsk.EstimationProblem(data2d, grid2d, "z")
    for params in (dict(variogram=g35), dict(variogram=g35, maxneighbors=3),
                   dict(variogram=g35, maxneighbors=3, neighborhood=gsk.MetricBall(100.0))):
        sol = gsk.solve(prob2d, gsk.KrigingSolver(z=params), ctx=ctx)
        Z = gsk.asarray(sol, "z")
        S = np.asarray(sol.z)
        for i, j, expected in GOLDEN["ref_checks"]:
            i, j = int(i), int(j)
            assert abs(Z[i - 1, j - 1] - expected) < 1e-3                          # krig.jl:35-37,50-52
            assert abs(S[(i - 1) + (j - 1) * 100] - expected) < 1e-3               # krig.jl:70-72 (LinearIndices)
    # custom path (krig.jl:78-90; the reference only checks that it runs): the reference maps over
    # traverse(grid, MultiGridPath()) and returns the predictions in VISITING order (krig.jl:204-231) — so must we;
    # `path_order=False` gives the same field in domain order
    base = dict(variogram=g35, maxneighbors=3, neighborhood=gsk.MetricBall(100.0))
    lin = gsk.solve(prob2d, gsk.KrigingSolver(z=base), ctx=ctx)
    for path in (gsk.MultiGridPath(), gsk.RandomPath(seed=2021)):
        order = gsk.traverse(grid2d, path)
        assert sorted(order.tolist()) == list(range(grid2d.nelements()))
        sol = gsk.solve(prob2d, gsk.KrigingSolver(z=dict(base, path=path)), ctx=ctx)
        assert np.array_equal(np.asarray(sol.z), np.asarray(lin.z)[order])
        assert np.array_equal(np.asarray(sol["z_variance"]), np.asarray(lin["z_variance"])[order])
        dom = gsk.solve(prob2d, gsk.KrigingSolver(z=dict(base, path=path)), ctx=ctx, path_order=False)
        assert np.array_equal(np.asarray(dom.z), np.asarray(lin.z))
    glob_lin = gsk.solve(prob2d, gsk.KrigingSolver(z=dict(variogram=g35)), ctx=ctx)
    glob_mg = gsk.solve(prob2d, gsk.KrigingSolver(z=dict(variogram=g35, path=gsk.MultiGridPath())), ctx=ctx)
    order = gsk.traverse(grid2d, gsk.MultiGridPath())
    np.testing.assert_allclose(np.asarray(glob_mg.z), np.asarray(glob_lin.z)[order], rtol=0, atol=1e-12)


@pytest.mark.parametrize("k,radius", [(0, None), (3, None), (3, 100.0)])
def test_reference_problems_vs_oracle(gsk, ctx, oracle, k, radius):
    _check(gsk, ctx, oracle, ref_problem_2d(gsk, k, radius), atol_mean=1e-11, atol_var=1e-11)
    _check(gsk, ctx, oracle, ref_problem_1d(gsk, k, radius), atol_mean=1e-7, atol_var=1e-9)  # 11 Gaussian samples at h/r=0.29: cond ~1e9


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_golden_vectors(gsk, ctx, case):
    name = case[0]
    spec = build_case(case)
    mean, var, nn, idx = ctx.krige(spec, want_neighbors=True)
    assert np.array_equal(nn, GOLDEN[f"{name}/nn"])
    if spec.params["max_neighbors"] > 0:
        assert np.array_equal(idx, GOLDEN[f"{name}/idx"])
    gauss = spec.params["vario_kind"] == gsk.VARIO_GAUSSIAN
    assert_parity(mean, var, GOLDEN[f"{name}/mean"], GOLDEN[f"{name}/var"], scale=np.abs(spec.values).max(),
                  atol_mean=2e-8 if gauss else None, atol_var=2e-9 if gauss else None)


# ---- BASELINE.json configs at oracle-friendly sizes ----
@pytest.mark.parametrize("name,scale", [("C2", 0.25), ("C3a", 0.16), ("C3b", 0.16), ("C5", 0.07)])
def test_local_configs_scaled(gsk, ctx, oracle, name, scale):
    _check(gsk, ctx, oracle, gsk.synth.config_spec(name, scale=scale))


def test_config_c1_full(gsk, ctx, oracle):
    """C1 at full size (500 samples → 100×100, global OK, Gaussian r=35). cond(C) ≈ 6e7 with the 1e-6
    nugget, so any two backward-stable solvers differ by ~cond·eps·|z| ≈ 1e-8 in the mean (LU vs
    Bunch–Kaufman vs long double: see DESIGN.md §Numerics); the floor below is that bound."""
    _check(gsk, ctx, oracle, gsk.synth.config_spec("C1"), atol_mean=2e-8, atol_var=1e-10)


def test_config_c4_reduced(gsk, ctx, oracle):
    """C4's shape (global OK, Spherical r=256) at n=1500 onto 96×96 — well conditioned → strict rtol."""
    _check(gsk, ctx, oracle, gsk.synth.config_spec("C4", grid=(96, 96), n=1500))


def test_config_c2_full_size_subset_and_properties(gsk, ctx, oracle):
    """C2 at BASELINE size (1e4 samples → 1000×1000, k=20): parity on 3 random row slabs, and
    size-independent properties on the whole field."""
    spec = gsk.synth.config_spec("C2")
    mean, var, nn, idx = ctx.krige(spec, want_neighbors=True)
    assert mean.shape == (1_000_000,) and np.all(nn == 20)
    assert np.all(np.isfinite(mean)) and np.all(var >= 0) and np.all(var <= 2.0)
    assert np.all((idx >= 0) & (idx < spec.n_samples))
    assert np.all(np.sort(idx, axis=1)[:, 1:] != np.sort(idx, axis=1)[:, :-1])      # no duplicate neighbour
    # distances of the reported neighbours are ascending
    ctr = spec.target_centers()
    sub = np.random.default_rng(5).choice(spec.n_targets, 20000, replace=False)
    dx = spec.coords[0][idx[sub]] - ctr[0][sub, None]
    dy = spec.coords[1][idx[sub]] - ctr[1][sub, None]
    d2 = dx * dx + dy * dy
    assert np.all(np.diff(d2, axis=1) >= 0)
    for first in (0, 333_000, 990_000):
        slab = spec.with_slab(first, 10_000)
        om, ov, onn, oidx = oracle.krige(slab, want_neighbors=True)
        assert np.array_equal(idx[first:first + 10_000], oidx)
        assert_parity(mean[first:first + 10_000], var[first:first + 10_000], om, ov, scale=2.0)
    # Ordinary Kriging is exact for constants: shifting z by c shifts the mean by c, variance unchanged
    shifted = gsk.synth.config_spec("C2")
    shifted.values = shifted.values + 7.5
    m2, v2 = ctx.krige(shifted.with_slab(500_000, 50_000))
    np.testing.assert_allclose(m2, mean[500_000:550_000] + 7.5, rtol=1e-12, atol=1e-12)
    np.testing.assert_array_equal(v2, var[500_000:550_000])


# ---- estimator × variogram × dimension matrix ----
@pytest.mark.parametrize("dim", [1, 2, 3])
@pytest.mark.parametrize("vk", [0, 1, 2])
@pytest.mark.parametrize("est,deg", [(0, 0), (1, 0), (2, 1), (2, 2)])
def test_matrix(gsk, ctx, oracle, dim, vk, est, deg):
    grid = {1: (300,), 2: (24, 20), 3: (10, 9, 8)}[dim]
    n = {1: 60, 2: 150, 3: 260}[dim]
    k = 10 if est == 2 and deg == 2 and dim == 3 else 8
    k = {1: 6, 2: k + 4, 3: k + 8}[dim]
    coords, vals = gsk.synth.make_samples(100 + dim, n, grid, seed_extra=vk * 10 + est)
    rng = {1: 40.0, 2: 9.0, 3: 6.0}[dim]
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, support=gsk.default_support_py([1.0] * dim, rng),
                           vario_kind=vk, vario_range=rng, vario_sill=1.3, vario_nugget=0.05, estimator=est,
                           uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=k)
    loose = vk == 0 or (est == 2 and deg == 2)    # Gaussian / quadratic drift in raw coordinates: cond ≳ 1e6
    mean, var = _check(gsk, ctx, oracle, spec, **(dict(atol_mean=1e-7, atol_var=1e-7) if loose else {}))
    if est == 1:   # k <= 20: the small kernel; UK of degree 0 is Ordinary Kriging bit for bit
        uk0 = gsk.ProblemSpec(coords=spec.coords, values=spec.values, grid_dims=grid, support=spec.support,
                              **dict(spec.params, estimator=2, uk_degree=0))
        m0, v0 = ctx.krige(uk0)
        assert np.array_equal(m0, mean, equal_nan=True) and np.array_equal(v0, var, equal_nan=True)


# ---- edge cases ----
def test_ball_and_min_neighbors_produce_missing(gsk, ctx, oracle):
    spec = gsk.synth.config_spec("C2", scale=0.2, ball_radius=9.0, min_neighbors=4)
    mean, var = _check(gsk, ctx, oracle, spec)
    assert np.isnan(mean).any() and (~np.isnan(mean)).any()
    spec3 = gsk.synth.config_spec("C3a", scale=0.12, ball_radius=7.0, min_neighbors=3)
    _check(gsk, ctx, oracle, spec3)


def test_point_targets_point_support(gsk, ctx, oracle):
    base = gsk.synth.config_spec("C2", scale=0.1)
    rng = np.random.default_rng(3)
    pts = [rng.uniform(-5, 105, 5000), rng.uniform(-5, 105, 5000)]   # unordered, partly outside the samples' box
    spec = gsk.ProblemSpec(coords=base.coords, values=base.values, points=pts, vario_kind=gsk.VARIO_SPHERICAL,
                           vario_range=50.0, max_neighbors=12)
    _check(gsk, ctx, oracle, spec)
    # targets ON samples (point support, nugget 0): exact interpolation, zero variance
    on = gsk.ProblemSpec(coords=base.coords, values=base.values, points=[c[:200] for c in base.coords],
                         vario_kind=gsk.VARIO_SPHERICAL, vario_range=50.0, max_neighbors=12)
    mean, var = ctx.krige(on)
    np.testing.assert_allclose(mean, base.values[:200], rtol=0, atol=1e-9)
    np.testing.assert_allclose(var, 0.0, atol=1e-9)
    glob = ctx.krige(gsk.ProblemSpec(coords=[c[:300] for c in base.coords], values=base.values[:300],
                                     points=[c[:50] for c in base.coords], vario_kind=gsk.VARIO_EXPONENTIAL,
                                     vario_range=30.0, max_neighbors=0))
    np.testing.assert_allclose(glob[0], base.values[:50], rtol=0, atol=1e-8)


def test_small_and_degenerate_inputs(gsk, ctx, oracle):
    # k = n (host clamp), k = 1, a single sample, collinear samples, far-away coordinates
    coords = [np.array([1.0, 4.0, 9.0, 2.5]), np.array([2.0, 2.0, 2.0, 2.0])]
    vals = np.array([0.3, 1.1, -0.4, 0.9])
    for k in (1, 2, 4):
        spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(12, 5), vario_kind=gsk.VARIO_EXPONENTIAL,
                               vario_range=5.0, max_neighbors=k)
        _check(gsk, ctx, oracle, spec)
    one = gsk.ProblemSpec(coords=[np.array([3.0])], values=np.array([2.0]), grid_dims=(7,), vario_kind=gsk.VARIO_SPHERICAL,
                          vario_range=4.0, max_neighbors=1)
    _check(gsk, ctx, oracle, one)
    big = gsk.synth.config_spec("C2", scale=0.1)
    big.coords = [c + 4.0e6 for c in big.coords]
    big.grid_origin = [4.0e6, 4.0e6]
    _check(gsk, ctx, oracle, big)
    empty = gsk.synth.config_spec("C2", scale=0.1).with_slab(10, 0)
    m, v = ctx.krige(empty)
    assert m.shape == (0,) and v.shape == (0,)


def test_clustered_samples_exact_neighbours(gsk, ctx, oracle):
    """Strongly non-uniform density: the ring expansion must still return the exact kNN."""
    rng = np.random.default_rng(11)
    c1 = rng.normal([20, 20], 1.5, (600, 2)); c2 = rng.normal([80, 70], 4.0, (300, 2)); c3 = rng.uniform(0, 100, (40, 2))
    xy = np.concatenate([c1, c2, c3])
    vals = np.sin(xy[:, 0] / 9.0) + 0.1 * rng.standard_normal(len(xy))
    spec = gsk.ProblemSpec(coords=[xy[:, 0], xy[:, 1]], values=vals, grid_dims=(100, 100),
                           support=gsk.default_support_py([1.0, 1.0], 30.0), vario_kind=gsk.VARIO_EXPONENTIAL,
                           vario_range=30.0, vario_nugget=0.02, max_neighbors=16)
    _check(gsk, ctx, oracle, spec)


def test_ties_fall_to_lower_index(gsk, ctx, oracle):
    """A regular sample lattice with targets on cell centres: many exactly tied distances."""
    gx, gy = np.meshgrid(np.arange(0.0, 20.0, 2.0), np.arange(0.0, 20.0, 2.0), indexing="ij")
    coords = [gx.ravel(), gy.ravel()]
    vals = np.cos(coords[0]) + coords[1] * 0.1
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(20, 20), grid_origin=(-0.5, -0.5),
                           vario_kind=gsk.VARIO_SPHERICAL, vario_range=8.0, max_neighbors=6)
    (mean, var, nn, idx), (om, ov, onn, oidx) = _both(ctx, oracle, spec, oracle.SEARCH_BRUTE)
    assert np.array_equal(idx, oidx)


@pytest.mark.parametrize("dim,k", [(2, 6), (2, 30), (3, 12), (3, 40)])
def test_ties_on_a_non_dyadic_lattice(gsk, ctx, oracle, dim, k):
    """Lattice coordinates that are not exactly representable (multiples of 0.3): mathematically tied distances come
    out of the rounding chain equal or a few ulps apart. The search keeps 64-bit keys (distance bits + sample index)
    that drop the low mantissa bits; every tile where those bits could matter must come back from the exact redo
    pass, so the lists still equal the oracle's (d², index) order bit for bit."""
    ax = np.arange(12) * 0.3
    g = np.meshgrid(*([ax] * dim), indexing="ij")
    coords = [c.ravel().copy() for c in g]
    rng = np.random.default_rng(5)
    perm = rng.permutation(len(coords[0]))           # index order unrelated to position
    coords = [c[perm] for c in coords]
    vals = np.cos(coords[0] * 3.0) + 0.1 * coords[-1]
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(36,) * dim, grid_origin=(-0.05,) * dim,
                           grid_spacing=(0.1,) * dim, vario_kind=gsk.VARIO_SPHERICAL, vario_range=2.0,
                           max_neighbors=k)
    (mean, var, nn, idx), (om, ov, onn, oidx) = _both(ctx, oracle, spec, oracle.SEARCH_BRUTE)
    assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)


@pytest.mark.parametrize("k", [3, 4, 24, 25])
def test_distances_that_differ_only_in_the_dropped_key_bits(gsk, ctx, oracle, k):
    """Pairs of samples placed symmetrically about a column of targets, one of each pair moved outwards by a few ulps
    and given the LOWER index: ordering by the truncated distance and then by index would put it first, the exact
    (d², index) order puts it second — also across the k-th / (k+1)-th boundary (k odd cuts a pair)."""
    rng = np.random.default_rng(9)
    npair = 16
    a = 0.37 + 1.13 * np.arange(1, npair + 1)        # half-distances of the pairs, increasing
    xs, ys = [], []
    for j in range(npair):
        far = 50.5 + a[j]
        far = np.nextafter(np.nextafter(far, np.inf), np.inf)
        xs += [far, 50.5 - a[j]]                      # lower index: (slightly) farther
        ys += [50.5, 50.5]
    filler = rng.uniform(0, 100, (9000, 2))               # n > 2^12: at least 13 dropped bits
    filler = filler[np.abs(filler[:, 1] - 50.5) > 30.0]   # far from the targets of interest
    x = np.concatenate([np.array(xs), filler[:, 0]]); y = np.concatenate([np.array(ys), filler[:, 1]])
    vals = np.sin(x / 7.0) + 0.05 * y
    spec = gsk.ProblemSpec(coords=[x, y], values=vals, grid_dims=(100, 100), vario_kind=gsk.VARIO_SPHERICAL,
                           vario_range=40.0, max_neighbors=k)
    (mean, var, nn, idx), (om, ov, onn, oidx) = _both(ctx, oracle, spec, oracle.SEARCH_BRUTE)
    assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)
    row = 50 * 100 + 50                               # the target at (50.5, 50.5): every pair is a near-tie there
    assert oidx[row, 0] == 1 and oidx[row, 1] == 0    # exact order: the nearer sample (index 1) first


def test_one_call_over_several_chunks_equals_slab_calls(gsk, ctx):
    """gsk_execute cuts a range into chunks of ~4M targets (search + solve per chunk, chunk edges on tile layers): a
    9M-target grid computed in ONE call must equal, bit for bit, the same grid computed slab by slab with slab edges
    that fall inside chunks and off the tile lattice."""
    spec = gsk.synth.config_spec("C2", grid=(3000, 3000), n=90_000)
    T = spec.n_targets
    mean, var = ctx.krige(spec)
    assert np.isfinite(mean).all() and np.isfinite(var).all()
    cuts = [0, 1_234_567, 4_194_304 + 11, 6_000_000, T]
    for a, b in zip(cuts[:-1], cuts[1:]):
        m, v = ctx.krige(spec.with_slab(a, b - a))
        assert np.array_equal(m, mean[a:b]) and np.array_equal(v, var[a:b])


# ---- sharding and the resident form ----
def test_slabs_equal_full(gsk, ctx):
    spec = gsk.synth.config_spec("C3a", scale=0.14)
    full = ctx.krige(spec)
    T = spec.n_targets
    for world in (2, 3, 8):
        parts = [ctx.krige(spec.with_slab(*gsk.slab_bounds(T, r, world))) for r in range(world)]
        assert np.array_equal(np.concatenate([p[0] for p in parts]), full[0])
        assert np.array_equal(np.concatenate([p[1] for p in parts]), full[1])


def test_resident_plan_execute_matches_one_shot(gsk, ctx):
    import torch
    spec = gsk.synth.config_spec("C2", scale=0.2)
    mean, var = ctx.krige(spec)
    T = spec.n_targets
    dm = torch.empty(T, dtype=torch.float64, device="cuda")
    dv = torch.empty(T, dtype=torch.float64, device="cuda")
    own = gsk.Context(0)
    own.set_stream(torch.cuda.current_stream().cuda_stream)
    own.plan(spec)
    own.execute(0, T, dm.data_ptr(), dv.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(dm.cpu().numpy(), mean) and np.array_equal(dv.cpu().numpy(), var)
    t = own.timing()
    assert t["launches"] >= 2 and t["targets"] == T
    with pytest.raises(gsk.GskError):
        gsk.Context(0).execute(0, 1, dm.data_ptr(), dv.data_ptr())      # execute before plan
    own.close()


def test_invalid_arguments_are_rejected(gsk, ctx):
    spec = gsk.synth.config_spec("C2", scale=0.1)
    bad = gsk.synth.config_spec("C2", scale=0.1)
    bad.params["max_neighbors"] = gsk.GSK_MAX_NEIGHBORS + 1
    with pytest.raises(gsk.GskError, match="GSK_MAX_NEIGHBORS"):
        ctx.krige(bad)
    few = gsk.ProblemSpec(coords=[c[:5] for c in spec.coords], values=spec.values[:5], grid_dims=(8, 8), max_neighbors=6)
    with pytest.raises(gsk.GskError, match="clamped"):
        ctx.krige(few)
    bad = gsk.synth.config_spec("C2", scale=0.1)
    bad.params["vario_range"] = 0.0
    with pytest.raises(gsk.GskError, match="vario_range"):
        ctx.krige(bad)
    bad = gsk.synth.config_spec("C2", scale=0.1)
    bad.coords[0][3] = np.nan
    with pytest.raises(gsk.GskError, match="finite"):
        ctx.krige(bad)
    bad = gsk.synth.config_spec("C2", scale=0.1)
    bad.params["vario_nugget"] = 1.5                      # above the sill: no positive-definite covariance
    with pytest.raises(gsk.GskError, match="nugget"):
        ctx.krige(bad)
    bad = gsk.synth.config_spec("C2", scale=0.1)
    bad.grid_spacing[1] = 0.0
    with pytest.raises(gsk.GskError, match="grid_spacing"):
        ctx.krige(bad)
    ctx.krige(spec)                                       # the context stays usable after rejected calls


# ---- BASELINE-size sample sets (full n), parity on slabs of targets -------------------------------
@pytest.mark.parametrize("name,slabs", [
    ("C3a", [(0, 4096), (8_000_000, 4096), (16_777_216 - 4096, 4096)]),
    ("C3b", [(5_000_000, 4096)]),
    ("C5", [(0, 2048), (67_000_000, 2048), (134_217_728 - 2048, 2048)]),
])
def test_full_size_samples_slab_parity(gsk, ctx, oracle, name, slabs):
    """C3/C5 with their full sample sets (1e5 / 1e6 samples, 256³ / 512³ grids): the oracle (KD-tree) and the
    GPU compute the same slabs of targets — first, middle and last rows of the grid (slab boundaries)."""
    spec = gsk.synth.config_spec(name)
    for first, count in slabs:
        slab = spec.with_slab(first, count)
        mean, var, nn, idx = ctx.krige(slab, want_neighbors=True)
        om, ov, onn, oidx = oracle.krige(slab, want_neighbors=True)
        assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)
        assert_parity(mean, var, om, ov, scale=3.0)


def test_config_c4_full_size_properties(gsk, ctx):
    """C4 at BASELINE size (2e4 samples, global OK, Spherical r=256): the oracle cannot factor a 20 001² system
    in test time, so the full-size path is checked through size-independent properties: with point support and
    zero nugget, kriging interpolates exactly at the samples (mean = z, variance = 0); the block-support field on
    a slab of the 2048² grid is finite, bounded by the data range up to the usual overshoot, and has variance in
    [0, 2·sill]; the same slab computed in two halves is bit-identical (sharding)."""
    spec = gsk.synth.config_spec("C4")
    n = spec.n_samples
    sel = np.arange(0, n, 97)
    on = gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=[c[sel] for c in spec.coords],
                         vario_kind=gsk.VARIO_SPHERICAL, vario_range=256.0, max_neighbors=0)
    mean, var = ctx.krige(on)
    np.testing.assert_allclose(mean, spec.values[sel], rtol=0, atol=5e-8)
    np.testing.assert_allclose(var, 0.0, atol=5e-8)
    first, count = 2048 * 1000, 4096
    m, v = ctx.krige(spec.with_slab(first, count))
    assert np.all(np.isfinite(m)) and m.min() > spec.values.min() - 0.5 and m.max() < spec.values.max() + 0.5
    assert np.all(v >= 0) and np.all(v <= 2.0)
    m1, v1 = ctx.krige(spec.with_slab(first, 1000))
    m2, v2 = ctx.krige(spec.with_slab(first + 1000, count - 1000))
    assert np.array_equal(np.concatenate([m1, m2]), m) and np.array_equal(np.concatenate([v1, v2]), v)


def test_unordered_point_targets_are_bin_sorted(gsk, ctx, oracle):
    """2e5 targets in random order: the library sorts them by bin internally (otherwise every CTA would scan
    all samples) and returns results in the caller's order; slabs of the list work too."""
    import time
    base = gsk.synth.config_spec("C2")
    rng = np.random.default_rng(9)
    pts = [rng.uniform(0, 1000, 200_000), rng.uniform(0, 1000, 200_000)]
    spec = gsk.ProblemSpec(coords=base.coords, values=base.values, points=pts, vario_kind=gsk.VARIO_SPHERICAL,
                           vario_range=50.0, max_neighbors=20)
    ctx.krige(spec.with_slab(0, 1000))          # warm-up
    t0 = time.perf_counter()
    mean, var, nn, idx = ctx.krige(spec, want_neighbors=True)
    dt = time.perf_counter() - t0
    assert dt < 2.0, f"unordered points took {dt:.2f}s"
    om, ov, onn, oidx = oracle.krige(spec, want_neighbors=True)
    assert np.array_equal(idx, oidx) and np.array_equal(nn, onn)
    assert_parity(mean, var, om, ov, scale=2.0)
    m2, v2 = ctx.krige(spec.with_slab(150_000, 12_345))
    assert np.array_equal(m2, mean[150_000:162_345]) and np.array_equal(v2, var[150_000:162_345])


def test_more_edge_shapes(gsk, ctx, oracle):
    """Non-unit spacing with a negative origin (block support scales with the cell), k at the library maximum
    (one warp per target configuration), every target missing (min_neighbors > what the ball can hold), and a
    slab that starts and ends in the middle of grid rows."""
    rng = np.random.default_rng(21)
    # 1) anisotropic spacing, negative origin
    coords = [rng.uniform(-50, 30, 700), rng.uniform(10, 90, 700)]
    vals = np.sin(coords[0] / 11.0) * np.cos(coords[1] / 7.0)
    spacing = [2.0, 0.5]
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(40, 160), grid_origin=(-50.0, 10.0), grid_spacing=spacing,
                           support=gsk.default_support_py(spacing, 12.0), vario_kind=gsk.VARIO_EXPONENTIAL,
                           vario_range=12.0, vario_nugget=0.1, max_neighbors=14)
    _check(gsk, ctx, oracle, spec)
    # 2) k = 96 (GSK_MAX_NEIGHBORS), Ordinary and Universal degree 2 (e = 12 extra rows)
    c3, v3 = gsk.synth.make_samples(55, 4000, (30, 30, 30))
    for est, deg in ((gsk.EST_ORDINARY, 0), (gsk.EST_UNIVERSAL, 2)):
        big = gsk.ProblemSpec(coords=c3, values=v3, grid_dims=(12, 12, 12), grid_origin=(9.0, 9.0, 9.0),
                              support=gsk.default_support_py([1.0] * 3, 8.0), vario_kind=gsk.VARIO_SPHERICAL,
                              vario_range=8.0, vario_nugget=0.05, estimator=est, uk_degree=deg, max_neighbors=96)
        _check(gsk, ctx, oracle, big, **(dict(atol_mean=1e-6, atol_var=1e-6) if deg == 2 else {}))
    # 3) everything missing
    none = gsk.synth.config_spec("C2", scale=0.1, ball_radius=0.5, min_neighbors=5)
    mean, var, nn, idx = ctx.krige(none, want_neighbors=True)
    assert np.isnan(mean).all() and np.isnan(var).all() and nn.max() < 5
    om, ov, onn, oidx = oracle.krige(none, want_neighbors=True)
    assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)
    # 4) slab cutting through rows
    base = gsk.synth.config_spec("C3b", scale=0.12)
    full = ctx.krige(base)
    cut = ctx.krige(base.with_slab(1234, 5677))
    assert np.array_equal(cut[0], full[0][1234:1234 + 5677]) and np.array_equal(cut[1], full[1][1234:1234 + 5677])


def test_execute_peers_stores_into_every_destination(gsk, ctx):
    """gsk_execute_peers (the fused result gather): with three destination buffers standing in for three ranks'
    symmetric-memory buffers, every buffer receives the slab at out_offset; local and global paths."""
    import torch
    for name, kw in (("C2", dict(scale=0.15)), ("C1", dict(grid=(30, 30), n=200))):
        spec = gsk.synth.config_spec(name, **kw)
        T = spec.n_targets
        first, count = T // 3, T // 2
        ref_m, ref_v = ctx.krige(spec.with_slab(first, count))
        own = gsk.Context(0)
        own.set_stream(torch.cuda.current_stream().cuda_stream)
        own.plan(spec)
        bufs = [torch.full((2, T), -7.0, dtype=torch.float64, device="cuda") for _ in range(3)]
        own.execute_peers(first, count, [b[0].data_ptr() for b in bufs], [b[1].data_ptr() for b in bufs],
                          out_offset=first)
        torch.cuda.synchronize()
        for b in bufs:
            got = b.cpu().numpy()
            assert np.array_equal(got[0, first:first + count], ref_m) and np.array_equal(got[1, first:first + count], ref_v)
            assert np.all(got[:, :first] == -7.0) and np.all(got[:, first + count:] == -7.0)
        with pytest.raises(gsk.GskError):
            own.execute_peers(first, count, [bufs[0][0].data_ptr()] * 9, [bufs[0][1].data_ptr()] * 9)
        own.close()


def test_krige_multi_single_process(gsk, ctx):
    """gsk_krige_multi: one process, several pieces (here three contexts on the one visible GPU) — the result
    must equal the single-context call bit for bit, local and global paths."""
    import torch
    ids = [0, 0, 0] if torch.cuda.device_count() < 2 else [0, 1, 0]
    for name, kw in (("C3b", dict(scale=0.12)), ("C1", dict(grid=(40, 30), n=250))):
        spec = gsk.synth.config_spec(name, **kw)
        ref = ctx.krige(spec, want_neighbors=True)
        got = gsk.krige_multi(spec, ids, want_neighbors=True)
        for a, b in zip(ref, got):
            if a is not None:
                assert np.array_equal(a, b, equal_nan=True)
        part = gsk.krige_multi(spec.with_slab(100, 777), [0, 0])
        assert np.array_equal(part[0], ref[0][100:877])
    with pytest.raises(gsk.GskError):
        gsk.krige_multi(spec, [99])
    gsk.load_library().gsk_krige_multi_release()          # the cached per-device contexts are given back …
    again = gsk.krige_multi(spec, [0, 0])                 # … and re-created on demand
    assert np.array_equal(again[0], ref[0])


def test_plain_c_host_end_to_end(gsk, oracle, tmp_path):
    """The C-ABI without Python in the process: examples/krige_c.c (C99) runs C2 at 1/20 scale from files."""
    import subprocess
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    lib_dir = root / "geostatssolvers.jl_b200" / "csrc"
    exe = tmp_path / "krige_c"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", f"-I{root / 'include'}",
                    str(root / "examples" / "krige_c.c"), f"-L{lib_dir}", "-lgskrige", f"-Wl,-rpath,{lib_dir}", "-lm",
                    "-o", str(exe)], check=True)
    spec = gsk.synth.config_spec("C2", scale=0.05)
    gx, gy = spec.grid_dims
    with open(tmp_path / "in.bin", "wb") as f:
        np.array([spec.n_samples, gx, gy, spec.params["max_neighbors"]], dtype="<i8").tofile(f)
        np.array([spec.params["vario_range"]], dtype="<f8").tofile(f)
        for a in (spec.coords[0], spec.coords[1], spec.values):
            np.ascontiguousarray(a, dtype="<f8").tofile(f)
    r = subprocess.run([str(exe), str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0, r.stderr
    T = gx * gy
    raw = (tmp_path / "out.bin").read_bytes()
    mean = np.frombuffer(raw, dtype="<f8", count=T)
    var = np.frombuffer(raw, dtype="<f8", count=T, offset=8 * T)
    nn = np.frombuffer(raw, dtype="<i4", count=T, offset=16 * T)
    om, ov, onn, _ = oracle.krige(spec, want_neighbors=True)
    assert np.array_equal(nn, onn)
    assert_parity(mean, var, om, ov, scale=max(1.0, np.abs(spec.values).max()))


@pytest.mark.parametrize("name", ["C3a", "C3b", "C5"])
def test_full_size_random_and_sample_cells(gsk, ctx, oracle, name):
    """SURVEY §8d parity procedure for the configs too large for a full-grid oracle run: with the FULL sample set,
    65 536 random grid cells plus (up to 65 536 of) the cells that contain a sample — the nearest neighbour is then
    closer than the block-support radius — evaluated as explicit point targets carrying the cell's block support."""
    spec = gsk.synth.config_spec(name)
    g = np.array(spec.grid_dims, dtype=np.int64)
    rng = np.random.default_rng(20240 + len(name) + int(g[0]))
    cells = [rng.integers(0, g[d], size=65536) for d in range(3)]
    sel = rng.permutation(spec.n_samples)[:65536]
    for d in range(3):
        own = np.clip(np.floor(spec.coords[d][sel]).astype(np.int64), 0, g[d] - 1)   # origin 0, spacing 1
        cells[d] = np.concatenate([cells[d], own])
    pts = [c.astype(np.float64) + 0.5 for c in cells]
    p = dict(spec.params)
    on = gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=pts, support=spec.support, **p)
    mean, var, nn, idx = ctx.krige(on, want_neighbors=True)
    om, ov, onn, oidx = oracle.krige(on, want_neighbors=True)
    assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)
    assert_parity(mean, var, om, ov, scale=3.0)
    # and the grid path gives the same numbers for the same cells (spot check on a slab)
    lin = int(cells[0][0] + g[0] * (cells[1][0] + g[1] * cells[2][0]))
    gm, gv = ctx.krige(spec.with_slab(lin, 1))[:2]
    np.testing.assert_allclose([gm[0], gv[0]], [mean[0], var[0]], rtol=1e-12, atol=1e-14)


def test_config_c4_full_size_golden(gsk, ctx):
    """C4 at FULL size (20 000 samples, the 20 001² system) against 4 096 golden targets solved with LAPACK
    dsytrf/dsytrs — the factorisation the reference itself calls — by tests/golden/make_golden_c4.py. The golden
    targets are reached through a traversal order that visits them first (the slab is then the first 4 096 positions)."""
    from pathlib import Path
    g = np.load(Path(__file__).parent / "golden" / "c4_full_4096.npz")
    spec = gsk.synth.config_spec("C4")
    T = spec.n_targets
    chosen = g["targets"]
    rest = np.setdiff1d(np.arange(T, dtype=np.int64), chosen, assume_unique=True)
    import copy
    sp = copy.copy(spec)
    sp.target_order = np.concatenate([chosen, rest])
    mean, var = ctx.krige(sp.with_slab(0, chosen.size))
    # Spherical(r = 256) on 20 000 samples: cond(C) ~ 1e6-1e7; Bunch–Kaufman on the indefinite (n+1)-system and
    # Cholesky + Schur complement on L⁻¹ are both backward stable, so they agree to ~cond·eps ≈ 1e-9 in the mean
    # (values of order 1): rtol 1e-9 with that absolute floor (north_star's tolerance, floor stated per SURVEY §8d)
    np.testing.assert_allclose(mean, g["mean"], rtol=1e-9, atol=2e-9)
    np.testing.assert_allclose(var, g["var"], rtol=1e-9, atol=2e-9)


@pytest.mark.parametrize("name", ["C2", "C3a", "C3b", "C5"])
def test_local_configs_full_size_golden(gsk, ctx, name):
    """The local BASELINE configs at their FULL sample counts against 1 024 golden targets each from the independent
    numpy + LAPACK restatement (tests/golden/make_golden_local.py: brute-force k-NN, dsytrf / dpotrf): neighbour
    lists bit-exact, mean and variance rtol 1e-9 (absolute floor 1e-12·scale for values that cross zero)."""
    from pathlib import Path
    g = np.load(Path(__file__).parent / "golden" / "local_full_1024.npz")
    spec = gsk.synth.config_spec(name)
    chosen = g[f"{name}/targets"]
    # the chosen cells as an explicit point list (their centroids, formed exactly as the library forms them) with the
    # grid's block support — the same targets without a 134M-entry traversal order for C5
    lin, pts = chosen.copy(), []
    for d in range(spec.dim):
        pts.append(spec.grid_origin[d] + ((lin % spec.grid_dims[d]).astype(np.float64) + 0.5) * spec.grid_spacing[d])
        lin //= spec.grid_dims[d]
    sp = gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=pts, support=spec.support, **spec.params)
    mean, var, nn, idx = ctx.krige(sp, want_neighbors=True)
    assert np.array_equal(idx, g[f"{name}/idx"])
    assert_parity(mean, var, g[f"{name}/mean"], g[f"{name}/var"], scale=max(1.0, np.abs(spec.values).max()))


# ---- the block-pool solve kernel (20 < k <= 64, at most 6 drift terms): both shapes, every model ----
@pytest.mark.parametrize("k", [21, 24, 31, 32, 33, 40, 57, 64])
@pytest.mark.parametrize("vk,nugget", [(0, 0.0), (1, 0.0), (1, 0.07), (2, 0.0), (2, 0.07)])
@pytest.mark.parametrize("dim,est,deg", [(3, 0, 0), (3, 1, 0), (3, 2, 1), (2, 1, 0), (2, 2, 1), (2, 2, 2), (1, 1, 0)])
def test_block_pool_matrix(gsk, ctx, oracle, k, vk, nugget, dim, est, deg):
    """k = 21 … 32 runs two targets per warp (4 neighbour blocks), k = 33 … 64 one warp per target (8 blocks); partial last
    blocks (k not a multiple of 8), no-nugget and nugget variants (the d² == 0 select), SK / OK / UK (up to 6 drift
    terms: UK degree 2 in 2-D), a ball that leaves some targets with fewer than k neighbours, 1-D to 3-D."""
    grid = {1: (160,), 2: (17, 13), 3: (8, 7, 6)}[dim]
    n = {1: 90, 2: 260, 3: 420}[dim]
    coords, vals = gsk.synth.make_samples(300 + dim, n, grid, seed_extra=k + 7 * vk + est)
    rng_ = {1: 50.0, 2: 11.0, 3: 7.0}[dim]
    radius = {1: 38.0, 2: 5.5, 3: 3.9}[dim] if (k % 8 == 0) else None     # roughly the k-NN radius: some targets get fewer
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, support=gsk.default_support_py([1.0] * dim, rng_),
                           vario_kind=vk, vario_range=rng_, vario_sill=1.2, vario_nugget=nugget, estimator=est,
                           uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=min(k, n), min_neighbors=3,
                           ball_radius=float("nan") if radius is None else radius)
    loose = vk == 0 or deg == 2 or (est == 2 and k >= 40)   # Gaussian / drift monomials in raw coordinates: cond ≳ 1e6
    _check(gsk, ctx, oracle, spec, **(dict(atol_mean=2e-7, atol_var=2e-7) if loose else {}))


# ---- the column-packed kernel where only it runs: configuration D (3-D UK2, 25 <= k <= 56) and E (64 < k <= 96, or
# more than 6 drift terms above k = 56) — the two configurations on the bottom-up row layout (RS % G != 0) ----
def _colpack_cases():
    cases = [(3, 2, 2, k, i % 3, (i // 3) % 2) for i, k in enumerate((25, 29, 32, 33, 40, 48, 49, 56, 57, 64))]
    for a, k in enumerate((65, 66, 72, 73, 80, 88, 89, 95, 96)):   # dimension × variogram: every pair over the ks
        cases += [((a + j) % 3 + 1 if deg < 2 else 2, est, deg, k, (a + 2 * j) % 3, (a + j) % 2)
                  for j, (est, deg) in enumerate(((0, 0), (1, 0), (2, 1), (2, 2)))]
    return [(dim, est, deg, k, vk, (0.0, 0.07)[g]) for dim, est, deg, k, vk, g in cases]


COLPACK = _colpack_cases()
# Every combination above fits the 227 KB of shared memory per CTA (the support offsets move to global memory when they
# do not): the largest, E with 12 extra rows in 3-D, needs 231 712 bytes of 232 448 — so none answers
# GSK_ERR_UNSUPPORTED, and the test fails if one does.
COLPACK_UNSUPPORTED = ()


def colpack_spec(gsk, dim, est, deg, k, vk, nugget):
    grid = {1: (300,), 2: (17, 13), 3: (8, 7, 6)}[dim]
    n = {1: 300, 2: 520, 3: 800}[dim]
    coords, vals = gsk.synth.make_samples(700 + dim, n, grid, seed_extra=k + 7 * vk + 3 * est + deg)
    rng_ = {1: 30.0, 2: 11.0, 3: 7.0}[dim]
    dens = n / np.prod(grid)
    knn_r = {1: k / (2 * dens), 2: np.sqrt(k / (np.pi * dens)), 3: (k / (4.18879 * dens)) ** (1 / 3)}[dim]
    c = 0 if est == 0 else (1 if est == 1 else len(gsk.uk_exponents(deg, dim)))
    return gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, support=gsk.default_support_py([1.0] * dim, rng_),
                           vario_kind=vk, vario_range=rng_, vario_sill=1.2, vario_nugget=nugget, estimator=est,
                           uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=k, min_neighbors=max(3, c + 10),
                           ball_radius=0.95 * knn_r if k % 8 == 0 else float("nan"))


def colpack_reference_rows(nn, k, mean):
    """≤ 32 targets: up to 16 with a partly filled list (ball), the rest full; none missing."""
    rng = np.random.default_rng(k)
    ok = ~np.isnan(mean)
    part, full = np.flatnonzero(ok & (nn < k)), np.flatnonzero(ok & (nn == k))
    part = rng.choice(part, min(16, part.size), replace=False)
    return np.sort(np.concatenate([part, rng.choice(full, min(32 - part.size, full.size), replace=False)]))


@pytest.mark.parametrize("dim,est,deg,k,vk,nugget", COLPACK,
                         ids=[f"d{c[0]}-e{c[1]}{c[2]}-k{c[3]}-v{c[4]}-g{c[5]}" for c in COLPACK])
def test_column_packed_matrix(gsk, ctx, oracle, dim, est, deg, k, vk, nugget):
    """Configurations D and E of local_solve.cuh against the oracle (neighbour lists bit-exact, parity rule on every
    target) and, on up to 32 targets, against the extended-precision reference at |gpu − ref| ≤ c·u·B + 2u·|ref|,
    c = 4(m + q) (derivation: tests/test_gpu_global_reference.py, oracle/extended_ref.py). For spherical and exponential
    variograms that bound must itself be below 1e-10 (relative to max(1, |z|), resp. the sill). k % 8 == 0 adds a ball
    just inside the k-NN radius, so some targets solve with fewer than k neighbours and some are missing."""
    import extended_ref as XR
    spec = colpack_spec(gsk, dim, est, deg, k, vk, nugget)
    if (dim, est, deg, k) in COLPACK_UNSUPPORTED:
        with pytest.raises(gsk.GskError) as err:
            ctx.krige(spec)
        assert err.value.code == -2
        return
    (mean, var, nn, idx), (om, ov, onn, oidx) = _both(ctx, oracle, spec)
    assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)
    scale = max(1.0, np.abs(spec.values).max())
    loose = vk == 0 or deg == 2 or (est == 2 and k >= 40)   # as the block-pool matrix: cond ≳ 1e6
    assert_parity(mean, var, om, ov, scale=scale, sill=1.2, **(dict(atol_mean=2e-7, atol_var=2e-7) if loose else {}))
    if k % 8 == 0:
        assert (nn < k).any()
    rows = colpack_reference_rows(nn, k, om)
    ref = XR.reference(spec, rows, oidx, onn)
    tm, tv = ref.tolerances(4)
    if vk != 0:
        assert tm.max() <= 1e-10 * scale and tv.max() <= 1e-10 * 1.2
    assert np.all(np.abs(mean[rows] - ref.mean) <= tm), np.max(np.abs(mean[rows] - ref.mean) / tm)
    assert np.all(np.abs(var[rows] - ref.var) <= tv), np.max(np.abs(var[rows] - ref.var) / tv)
    if est == 1:   # the column-packed c == 1 branch: UK of degree 0 is Ordinary Kriging bit for bit
        uk0 = gsk.ProblemSpec(coords=spec.coords, values=spec.values, grid_dims=spec.grid_dims, support=spec.support,
                              **dict(spec.params, estimator=2, uk_degree=0))
        m0, v0 = ctx.krige(uk0)
        assert np.array_equal(m0, mean, equal_nan=True) and np.array_equal(v0, var, equal_nan=True)
