"""Kriging of many value columns in one call (gsk_krige_columns) on the GPU.

Every column is checked against the extended-precision reference (oracle/extended_ref.py) run with that column as the
values, under the rule of tests/test_gpu_global_reference.py: |gpu − ref| ≤ 4(m + q)·u·B + 2u·|ref|. The local path
(the column-packed kernel's columns epilogue) also returns its Kriging weights λ and Lagrange multipliers ν, checked
against the reference's own solve of [C F; Fᵀ 0][λ; ν] = [c; f] at the first-order bound of that solve. The geometry
(neighbour counts and lists, the NaN pattern) must be gsk_krige's bit for bit, and the columns must not couple: a
column's mean does not depend on m, on its position or on the slab it is computed in."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_parity

import extended_ref as XR

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
KS = (1, 4, 20, 21, 32, 33, 64, 65, 96)
ESTS = ((0, 0), (1, 0), (2, 0), (2, 1), (2, 2))           # SK, OK, UK0, UK1, UK2
SUPPORTS = ("point", "block", "big")
GRID = {1: (300,), 2: (17, 13), 3: (8, 7, 6)}
NSAMP = {1: 300, 2: 520, 3: 800}
RANGE = {1: 30.0, 2: 11.0, 3: 7.0}


def _nterms(gsk, est, deg, dim):
    return 0 if est == 0 else (1 if est == 1 else len(gsk.uk_exponents(deg, dim)))


def _support(gsk, kind, dim, rng):
    if kind == "point":
        return None
    if kind == "block":
        return gsk.default_support_py([1.0] * dim, rng)
    side = {1: 130, 2: 12, 3: 6}[dim]                     # 130, 144, 216 points: more than the 125 staged in shared memory
    ax = (np.arange(side) + 0.5) / side - 0.5
    return [g.ravel() for g in np.meshgrid(*([ax] * dim), indexing="ij")]


def _local_cases():
    cases = []
    for i, k in enumerate(KS):
        for j, (est, deg) in enumerate(ESTS):
            dim = 3 if deg == 2 else (i + j) % 3 + 1
            c = 0 if est == 0 else (1 if est == 1 else {0: 1, 1: dim + 1, 2: 10}[deg])
            if k < c + 1:
                continue
            cases.append((dim, est, deg, k, (i + 2 * j) % 3, (0.0, 0.06)[(i + j) % 2], SUPPORTS[(i + j // 2) % 3]))
    return cases


LOCAL = _local_cases()


def local_spec(gsk, dim, est, deg, k, vk, nugget, sup, m=3):
    """A grid problem and m value columns (column 0 is the spec's own values); k % 8 == 0 adds a ball just inside
    the k-NN radius, so some lists are partly filled and some targets fall below min_neighbors."""
    grid, n, rng = GRID[dim], NSAMP[dim], RANGE[dim]
    coords, vals = gsk.synth.make_samples(800 + dim, n, grid, seed_extra=k + 7 * vk + 3 * est + deg)
    dens = n / np.prod(grid)
    knn_r = {1: k / (2 * dens), 2: np.sqrt(k / (np.pi * dens)), 3: (k / (4.18879 * dens)) ** (1 / 3)}[dim]
    c = _nterms(gsk, est, deg, dim)
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, support=_support(gsk, sup, dim, rng),
                           vario_kind=vk, vario_range=rng, vario_sill=1.2, vario_nugget=nugget, estimator=est,
                           uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=k,
                           min_neighbors=min(k, max(1, c + 2)),
                           ball_radius=0.95 * knn_r if k % 8 == 0 else float("nan"))
    r = np.random.default_rng(k * 31 + est)
    Z = np.column_stack([vals] + [vals * r.uniform(0.5, 2.0) + r.normal(0, 1, n) for _ in range(m - 1)])
    return spec, Z


def with_values(gsk, spec, z):
    import copy
    s = copy.copy(spec)
    s.values = np.ascontiguousarray(z, dtype=np.float64)
    return s


def check_columns(gsk, spec, Z, mean, var, rows, idx=None, nn=None, gram=False):
    """Every column at ``rows`` against the extended reference with that column as the values; returns the largest
    error / bound ratio of the means."""
    worst = 0.0
    for j in range(Z.shape[1]):
        ref = XR.reference(with_values(gsk, spec, Z[:, j]), rows, idx, nn, gram=gram)
        tm, tv = ref.tolerances(4)
        em = np.abs(mean[rows, j] - ref.mean)
        assert np.all(em <= tm), (j, float(np.max(em / tm)))
        if j == 0:
            ev = np.abs(var[rows] - ref.var)
            assert np.all(ev <= tv), float(np.max(ev / tv))
        worst = max(worst, float(np.max(em / tm)))
    return worst


def reference_rows(nn, k, ok, seed, count=16):
    rng = np.random.default_rng(seed)
    part, full = np.flatnonzero(ok & (nn < k)), np.flatnonzero(ok & (nn == k))
    part = rng.choice(part, min(count // 2, part.size), replace=False)
    return np.sort(np.concatenate([part, rng.choice(full, min(count - part.size, full.size), replace=False)]))


def solve_bounds(spec, rows, idx, nn):
    """λ, ν of the reference's long-double solve and their first-order bound c·u·|K⁻¹|(W_K|s| + W_R), c = 4(m + q)."""
    K, R, _, _, c, _, WK, WR = XR.assemble(spec, rows, idx, nn)
    fac, perm = XR.lu_factor(K)
    T, m = R.shape
    s = XR.lu_solve(fac, perm, R[:, :, None])[:, :, 0]
    Kinv = XR.lu_solve(fac, perm, np.broadcast_to(np.eye(m, dtype=XR.LD), (T, m, m)).copy())
    rhs = np.einsum("tij,tj->ti", WK, np.abs(s).astype(np.float64)) + WR
    q = spec.support[0].shape[0]
    bound = 4 * (nn[rows] + c + q)[:, None] * U * np.einsum("tij,tj->ti", np.abs(Kinv).astype(np.float64), rhs)
    return s, bound, c


@pytest.mark.parametrize("dim,est,deg,k,vk,nugget,sup", LOCAL,
                         ids=[f"d{c[0]}-e{c[1]}{c[2]}-k{c[3]}-v{c[4]}-g{c[5]}-{c[6]}" for c in LOCAL])
def test_local_columns_against_reference(gsk, ctx, dim, est, deg, k, vk, nugget, sup):
    spec, Z = local_spec(gsk, dim, est, deg, k, vk, nugget, sup)
    mean, var, nn, idx, w, lag = ctx.krige_columns(spec, Z, want_neighbors=True, want_weights=True)
    gm, gv, gnn, gidx = ctx.krige(spec, want_neighbors=True)
    # same geometry as gsk_krige: lists bit for bit, NaN rows identical, variance within the parity rule
    assert np.array_equal(nn, gnn) and np.array_equal(idx, gidx)
    miss = np.isnan(gm)
    assert np.array_equal(np.isnan(var), np.isnan(gv))
    assert all(np.array_equal(np.isnan(mean[:, j]), miss) for j in range(Z.shape[1]))
    loose = vk == 0 or deg == 2
    assert_parity(mean[:, 0], var, gm, gv, scale=max(1.0, np.abs(Z[:, 0]).max()), sill=1.2,
                  **(dict(atol_mean=2e-7, atol_var=2e-7) if loose else {}))
    if k % 8 == 0:
        assert (nn < k).any()
    rows = reference_rows(nn, k, ~miss, k + est)
    check_columns(gsk, spec, Z, mean, var, rows, idx, nn)
    # weights: zero past the list, the mean recomputed from them in long double, λ and ν against the reference's solve
    assert np.all(w[miss] == 0) and np.all(w[np.arange(k)[None, :] >= nn[:, None]] == 0)
    c = lag.shape[1]
    assert c == _nterms(gsk, est, deg, dim) and np.all(np.isnan(lag[miss]))
    s, bound, _ = solve_bounds(spec, rows, idx, nn)
    for r_i, t in enumerate(rows):
        kk = nn[t]
        assert np.all(np.abs(w[t, :kk] - s[r_i, :kk]) <= bound[r_i, :kk])
        assert np.all(np.abs(lag[t] - s[r_i, kk:kk + c]) <= bound[r_i, kk:kk + c])
        mu0 = XR.LD(spec.params["sk_mean"]) if est == 0 else XR.LD(0)
        for j in range(Z.shape[1]):
            mj = mu0 + np.sum(w[t, :kk].astype(XR.LD) * (Z[idx[t, :kk], j].astype(XR.LD) - mu0))
            ref = XR.reference(with_values(gsk, spec, Z[:, j]), rows[r_i:r_i + 1], idx, nn)
            assert abs(float(mj) - mean[t, j]) <= ref.tolerances(4)[0][0]
        if c:
            # the unbiasedness constraint Fᵀλ = f(x₀) (OK: Σλ = 1), to the bound the weights carry
            K, R, _, _, _, _, _, _ = XR.assemble(spec, rows[r_i:r_i + 1], idx, nn)
            F, f0 = K[0, :kk, kk:kk + c].astype(np.float64), R[0, kk:kk + c].astype(np.float64)
            resid = np.abs(F.T @ w[t, :kk] - f0)
            lim = np.abs(F).T @ bound[r_i, :kk] + 4 * kk * U * np.abs(F).T @ np.abs(w[t, :kk])
            assert np.all(resid <= lim), (resid, lim, U * np.linalg.norm(F) * np.linalg.norm(w[t, :kk]))


GLOBAL = [(n, *ESTS[j], (i + j) % 3 + 1, (i + 2 * j) % 3, (0.0, 0.06)[(i + j) % 2], SUPPORTS[(j + i // 2) % 3])
          for i, n in enumerate((63, 64, 65, 127, 128, 129)) for j in range(len(ESTS)) if (i + j) % 2 == 0]
GGRID = {1: (320,), 2: (12, 10), 3: (6, 5, 4)}
GRANGE = {0: {1: 4.0, 2: 3.0, 3: 2.0}, 1: {1: 12.0, 2: 6.0, 3: 4.0}, 2: {1: 12.0, 2: 6.0, 3: 4.0}}


def global_spec(gsk, n, est, deg, dim, vk, nugget, sup, m=3, grid=None):
    grid = GGRID[dim] if grid is None else grid
    rng = GRANGE[vk][dim]
    coords, vals = gsk.synth.make_samples(600 + dim, n, grid, seed_extra=n * 16 + 4 * est + deg)
    origin = None
    if dim == 1:   # lattice points: uniform draws on a line come near-singularly close (tests/test_gpu_global_reference.py)
        cells = np.random.default_rng(n).permutation(2 * n)[:n]
        coords = [(cells + 0.5) * (grid[0] / (2 * n)) - grid[0] / 2]
        origin = (-grid[0] / 2,)
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, grid_origin=origin,
                           support=_support(gsk, sup, dim, rng), vario_kind=vk, vario_range=rng, vario_sill=1.3,
                           vario_nugget=nugget, estimator=est, uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=0)
    r = np.random.default_rng(n + est)
    Z = np.column_stack([vals] + [r.normal(0, 2, n) + 3.0 for _ in range(m - 1)])
    return spec, Z


@pytest.mark.parametrize("n,est,deg,dim,vk,nugget,sup", GLOBAL,
                         ids=[f"n{c[0]}-e{c[1]}{c[2]}-d{c[3]}-v{c[4]}-g{c[5]}-{c[6]}" for c in GLOBAL])
def test_global_columns_against_reference(gsk, ctx, n, est, deg, dim, vk, nugget, sup):
    spec, Z = global_spec(gsk, n, est, deg, dim, vk, nugget, sup)
    mean, var, nn = ctx.krige_columns(spec, Z, want_nneigh=True)
    gm, gv, gnn = ctx.krige(spec, want_nneigh=True)
    assert np.array_equal(nn, gnn)
    rows = np.arange(spec.n_targets)
    check_columns(gsk, spec, Z, mean, var, rows, gram=True)
    assert np.array_equal(var, gv)   # the variance is gsk_krige's own computation


@pytest.mark.parametrize("path", ["local-4-lanes", "local-warp", "global"])
def test_columns_do_not_couple(gsk, ctx, path):
    """m = 257 against m = 1 per column and against a column permutation, bit for bit: the lanes of a target take the
    columns in strides of 4 (configuration B) or 32 (configuration D), and 257 leaves one column in a last stride. Slabs
    of the job computed separately equal the whole job's rows."""
    if path == "local-4-lanes":
        spec, Z = local_spec(gsk, 2, 0, 0, 20, 2, 0.06, "point", m=257)
    elif path == "local-warp":
        spec, Z = local_spec(gsk, 2, 1, 0, 40, 1, 0.0, "block", m=257)
    else:
        spec, Z = global_spec(gsk, 129, 2, 1, 2, 2, 0.06, "block", m=257)
    mean, var = ctx.krige_columns(spec, Z)
    assert mean.shape == (spec.n_targets, 257)
    for j in (0, 1, 7, 8, 31, 32, 100, 256):
        m1, v1 = ctx.krige_columns(spec, Z[:, j:j + 1])
        assert np.array_equal(m1[:, 0], mean[:, j], equal_nan=True), j
        assert np.array_equal(v1, var, equal_nan=True)
    perm = np.random.default_rng(5).permutation(257)
    mp, _ = ctx.krige_columns(spec, Z[:, perm])
    assert np.array_equal(mp, mean[:, perm], equal_nan=True)
    for a, b in ((0, 37), (37, 101), (101, spec.n_targets)):
        ms, vs = ctx.krige_columns(spec.with_slab(a, b - a), Z[:, :9])
        assert np.array_equal(ms, mean[a:b, :9], equal_nan=True) and np.array_equal(vs, var[a:b], equal_nan=True)


def test_target_order_slab_and_point_set(gsk, ctx):
    """A traversal order, a slab at an odd offset and an explicit point set (bin-sorted inside the library): rows land
    where gsk_krige puts them, and every column meets the reference."""
    import copy
    spec, Z = local_spec(gsk, 2, 2, 1, 33, 2, 0.06, "block")
    lin = ctx.krige_columns(spec, Z)
    order = np.random.default_rng(9).permutation(spec.n_targets)
    sp = copy.copy(spec)
    sp.target_order = order
    got = ctx.krige_columns(sp, Z)
    assert np.array_equal(got[0], lin[0][order], equal_nan=True) and np.array_equal(got[1], lin[1][order], equal_nan=True)
    slab = sp.with_slab(33, 101)
    ms, vs = ctx.krige_columns(slab, Z)
    assert np.array_equal(ms, got[0][33:134], equal_nan=True) and np.array_equal(vs, got[1][33:134], equal_nan=True)
    # point set: the samples' bounding box, random points
    r = np.random.default_rng(4)
    pts = [r.uniform(0, g, 700) for g in GRID[2]]
    ps = gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=pts,
                         **dict(spec.params, min_neighbors=1, ball_radius=float("nan")))
    mean, var, nn, idx = ctx.krige_columns(ps, Z, want_neighbors=True)
    gm, gv, gnn, gidx = ctx.krige(ps, want_neighbors=True)
    assert np.array_equal(nn, gnn) and np.array_equal(idx, gidx)
    assert_parity(mean[:, 0], var, gm, gv, scale=max(1.0, np.abs(Z[:, 0]).max()), sill=1.2)
    rows = np.sort(r.choice(700, 16, replace=False))
    check_columns(gsk, ps, Z, mean, var, rows, idx, nn)


def test_job_over_a_4m_chunk_edge(gsk, ctx):
    """4.41M targets: the local path processes chunks of about 4M targets (api.cu), so rows on both sides of the first
    chunk edge (4 200 000 on this grid) come from different launches."""
    grid = (2100, 2100)
    coords, vals = gsk.synth.make_samples(911, 20_000, grid, seed_extra=1)
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, vario_kind=1, vario_range=60.0, vario_sill=1.0,
                           estimator=1, max_neighbors=8)
    Z = np.column_stack([vals, 2.0 * vals - 1.0])
    mean, var, nn, idx = ctx.krige_columns(spec, Z, want_neighbors=True)
    gm, gv, gnn, gidx = ctx.krige(spec, want_neighbors=True)
    assert np.array_equal(nn, gnn) and np.array_equal(idx, gidx)
    assert_parity(mean[:, 0], var, gm, gv, scale=max(1.0, np.abs(vals).max()))
    rows = np.concatenate([np.arange(4_199_990, 4_200_010), [0, spec.n_targets - 1]])
    check_columns(gsk, spec, Z, mean, var, rows, idx, nn)


def _raw(ctx, spec, m, values, *, keep_values=False, mean=True, weights=False, lagrange=False):
    first, count = spec.slab
    ps = spec.c_struct()
    if not keep_values:
        ps.values = None
    out = np.empty((max(count, 1), max(m, 1)))
    var = np.empty(max(count, 1))
    w = np.empty((max(count, 1), max(spec.params["max_neighbors"], 1)))
    lg = np.empty((max(count, 1), 10))
    vals = values.ctypes.data if values is not None else None
    return ctx.lib.gsk_krige_columns(ctx._h, C.byref(ps), m, vals, out.ctypes.data if mean else None, var.ctypes.data,
                                     None, None, w.ctypes.data if weights else None,
                                     lg.ctypes.data if lagrange else None)


def test_rejections_and_context_state(gsk, ctx):
    spec, Z = local_spec(gsk, 2, 1, 0, 20, 1, 0.0, "block")
    gspec, gZ = global_spec(gsk, 64, 1, 0, 2, 1, 0.0, "point")
    assert _raw(ctx, spec, 3, Z, keep_values=True) == -1                  # prob->values must be NULL
    assert _raw(ctx, spec, 0, Z) == -1                                     # n_cols < 1
    assert _raw(ctx, spec, 3, None) == -1                                  # values NULL
    assert _raw(ctx, spec, 3, Z, mean=False) == -1                         # mean_out NULL
    reuse = gsk.ProblemSpec(coords=spec.coords, values=spec.values, grid_dims=spec.grid_dims, support=spec.support,
                            **dict(spec.params, flags=spec.params["flags"] | gsk.FLAG_REUSE_PLAN))
    assert _raw(ctx, reuse, 3, Z) == -1                                    # GSK_FLAG_REUSE_PLAN
    assert _raw(ctx, gspec, 3, gZ, weights=True) == -1                     # weights on the global path
    assert _raw(ctx, gspec, 3, gZ, lagrange=True) == -1                    # multipliers on the global path
    for solver in (gsk.SOLVER_IDW, gsk.SOLVER_LWR):
        s = gsk.ProblemSpec(coords=spec.coords, values=spec.values, grid_dims=spec.grid_dims,
                            **dict(spec.params, solver=solver))
        assert _raw(ctx, s, 3, Z) == -2
    # a refused neighbourhood is refused with gsk_krige's message
    big = gsk.ProblemSpec(coords=spec.coords, values=spec.values, grid_dims=spec.grid_dims,
                          **dict(spec.params, max_neighbors=97))
    with pytest.raises(gsk.GskError) as e1:
        ctx.krige(big)
    with pytest.raises(gsk.GskError) as e2:
        ctx.krige_columns(big, Z)
    assert e1.value.code == e2.value.code == -2 and str(e1.value) == str(e2.value)
    # the context holds no plan afterwards; a following gsk_krige equals one on a fresh context
    for sp, z in ((spec, Z), (gspec, gZ)):
        ctx.krige_columns(sp, z)
        dummy = C.c_void_p(64)
        assert ctx.lib.gsk_execute(ctx._h, 0, 1, dummy, dummy, None, None) == -5
        after = ctx.krige(sp)
        fresh = gsk.Context(0)
        try:
            ref = fresh.krige(sp)
        finally:
            fresh.close()
        assert np.array_equal(after[0], ref[0], equal_nan=True) and np.array_equal(after[1], ref[1], equal_nan=True)


def test_host_krige_columns_equals_solve(gsk, ctx):
    """Three variables with one missing set, Ordinary Kriging with a ball: `krige_columns` against `solve` per variable
    (units, masks, path order), and against the reference for a few targets."""
    r = np.random.default_rng(11)
    n = 400
    xy = np.column_stack([r.uniform(0, 40, n), r.uniform(0, 30, n)])
    a = np.sin(xy[:, 0] / 7) + r.normal(0, 0.1, n)
    miss = r.random(n) < 0.1
    cols = {"a": np.where(miss, np.nan, a), "b": np.where(miss, np.nan, 3 * a + 1), "c": np.where(miss, np.nan, a * a)}
    data = gsk.georef({k: np.ma.MaskedArray(v, mask=miss) for k, v in cols.items()}, [tuple(p) for p in xy])
    grid = gsk.CartesianGrid((40, 30))
    prob = gsk.EstimationProblem(data, grid, ("a", "b", "c"))
    p = dict(variogram=gsk.SphericalVariogram(range=12.0, sill=1.0), maxneighbors=24, neighborhood=gsk.MetricBall(6.0),
             minneighbors=4)
    solver = gsk.KrigingSolver(a=p, b=p, c=p)
    got = gsk.krige_columns(prob, solver, ctx=ctx)
    want = gsk.solve(prob, solver, ctx=ctx)
    assert got.names() == want.names()
    for name in want.names():
        g, w = got.table[name], want.table[name]
        assert np.array_equal(np.ma.getmaskarray(g), np.ma.getmaskarray(w))
        ok = ~np.ma.getmaskarray(w)
        np.testing.assert_allclose(np.ma.getdata(g)[ok], np.ma.getdata(w)[ok], rtol=1e-9, atol=1e-12)
