"""Leave-one-out cross-validation on the GPU (gsk_krige_loo): the local path against the oracle's independent
leave-one-out (brute-force kNN that skips the sample) and, bit for bit, against gsk_krige on the problem with the sample
deleted; the global path (Dubrule's closed form) against the extended-precision reference with every other sample as
the neighbourhood; the two paths against each other; argument checks and the context state afterwards."""
import numpy as np
import pytest

import _loo_oracle as LO

from conftest import assert_parity

import extended_ref as XR

pytestmark = pytest.mark.gpu

KS = (6, 20, 24, 32, 40, 64, 72, 96)                   # every local kernel: small, wpt2, wpt, A–E; 96 searches 97
ESTS = ((0, 0), (1, 0), (2, 1), (2, 2))                 # SK, OK, UK1, UK2
MATRIX = [(KS[i], *ESTS[j], (i + j) % 3 + 1, (i + 2 * j) % 3) for i in range(len(KS)) for j in range(len(ESTS))]
GRID = {1: (300,), 2: (24, 20), 3: (10, 9, 8)}
RANGE = {1: 12.0, 2: 9.0, 3: 6.0}
NSAMP = {1: 120, 2: 400, 3: 400}   # 1-D: spacing / range as in 2-D and 3-D (denser Gaussian UK2 systems reach cond ~1e10)


def local_spec(gsk, k, est, deg, dim, vk, n=None, **kw):
    n = NSAMP[dim] if n is None else n
    coords, vals = gsk.synth.make_samples(700 + dim, n, GRID[dim], seed_extra=k * 16 + 4 * est + deg)
    params = dict(vario_kind=vk, vario_range=RANGE[dim], vario_sill=1.3, vario_nugget=0.05, estimator=est, uk_degree=deg,
                  sk_mean=float(vals.mean()), max_neighbors=k)
    params.update(kw)
    return gsk.ProblemSpec(coords=coords, values=vals, points=coords, **params)


def _loose(vk, est, deg, k):
    return vk == 0 or deg == 2 or (est == 2 and k >= 40)   # Gaussian / drift monomials in raw coordinates: cond ≳ 1e6


def _parity(gsk, ctx, oracle, spec, loose):
    m, v, nn, idx = ctx.krige_loo(spec, want_neighbors=True)
    om, ov, onn, oidx = LO.krige_loo(oracle, spec, want_neighbors=True)
    assert np.array_equal(nn, onn)
    assert np.array_equal(idx, oidx)
    first = spec.target_first
    rows = first + np.arange(len(nn))
    assert not (idx == rows[:, None]).any()                 # never the row's own index
    tol = dict(atol_mean=2e-7, atol_var=2e-7) if loose else {}
    assert_parity(m, v, om, ov, scale=max(1.0, np.abs(spec.values).max()), sill=spec.params["vario_sill"], **tol)
    return m, v, nn, idx


@pytest.mark.parametrize("k,est,deg,dim,vk", MATRIX)
def test_local_loo_matches_oracle(gsk, ctx, oracle, k, est, deg, dim, vk):
    _parity(gsk, ctx, oracle, local_spec(gsk, k, est, deg, dim, vk), _loose(vk, est, deg, k))


def _deleted(gsk, spec, i):
    keep = np.arange(spec.n_samples) != i
    return gsk.ProblemSpec(coords=[c[keep] for c in spec.coords], values=spec.values[keep],
                           points=[c[i:i + 1] for c in spec.coords], **spec.params)


@pytest.mark.parametrize("k,est,deg,dim,vk", MATRIX)
def test_local_loo_bitwise_equals_krige_without_the_sample(gsk, ctx, k, est, deg, dim, vk):
    spec = local_spec(gsk, k, est, deg, dim, vk)
    m, v, nn, idx = ctx.krige_loo(spec, want_neighbors=True)
    for i in np.random.default_rng(k * 7 + est).choice(spec.n_samples, 16, replace=False):
        dm, dv, dnn, didx = ctx.krige(_deleted(gsk, spec, int(i)), want_neighbors=True)
        full = np.where(didx[0] >= i, didx[0] + 1, didx[0])
        assert nn[i] == dnn[0] and np.array_equal(idx[i], full)
        assert np.array_equal(m[i:i + 1], dm, equal_nan=True), (i, m[i], dm[0])
        assert np.array_equal(v[i:i + 1], dv, equal_nan=True), (i, v[i], dv[0])


def test_ball_and_min_neighbors_after_the_exclusion(gsk, ctx, oracle):
    spec = local_spec(gsk, 24, 1, 0, 2, 1, ball_radius=1.6, min_neighbors=5)
    m, v, nn, idx = _parity(gsk, ctx, oracle, spec, False)
    assert np.isnan(m).any() and (~np.isnan(m)).any()      # rows below min_neighbors after the exclusion
    assert np.array_equal(np.isnan(m), nn < 5)


@pytest.mark.parametrize("k", (8, 32, 64))
def test_twins_are_neighbours_at_distance_zero(gsk, ctx, oracle, k):
    spec = local_spec(gsk, k, 1, 0, 3, 2)
    for d in range(3):                                      # samples 10..19 sit on samples 0..9
        spec.coords[d][10:20] = spec.coords[d][0:10]
    m, v, nn, idx = ctx.krige_loo(spec, want_neighbors=True)
    om, ov, onn, oidx = LO.krige_loo(oracle, spec, want_neighbors=True)
    assert np.array_equal(nn, onn) and np.array_equal(idx, oidx)
    assert not (idx == np.arange(spec.n_samples)[:, None]).any()
    for i in range(10):                                     # each twin is the other's nearest neighbour
        assert idx[i, 0] == i + 10 and idx[i + 10, 0] == i
    # a list holding both members of a twin pair is a singular system (equal rows), in the reference as here: values are
    # compared on the other rows, the twins' own rows among them
    pair = np.zeros(len(nn), dtype=bool)
    for i in range(10):
        pair |= (idx == i).any(1) & (idx == i + 10).any(1)
    ok = ~pair
    assert ok[:20].any()
    assert_parity(m[ok], v[ok], om[ok], ov[ok], scale=max(1.0, np.abs(spec.values).max()), sill=1.3)


def test_slabs_concatenate_to_the_whole_call(gsk, ctx):
    for spec in (local_spec(gsk, 32, 1, 0, 3, 2), local_spec(gsk, 0, 1, 0, 2, 1, n=300)):
        m, v, nn = ctx.krige_loo(spec, want_nneigh=True)
        bounds = [0, 37, 128, 129, 300 if spec.n_samples == 300 else 250, spec.n_samples]
        parts = [ctx.krige_loo(spec.with_slab(a, b - a), want_nneigh=True) for a, b in zip(bounds[:-1], bounds[1:])]
        for j, full in enumerate((m, v, nn)):
            assert np.array_equal(np.concatenate([p[j] for p in parts]), full)


# ---- the global path: Dubrule's closed form against the long-double system of every other sample ----
NS = (63, 64, 65, 127, 128, 129, 255, 256, 257)
GESTS = ((0, 0), (1, 0), (2, 0), (2, 1), (2, 2))
GDESIGN = [(n, *GESTS[j], (i + j) % 3 + 1, (i + 2 * j) % 3, (0.0, 0.06)[(i + j) % 2])
           for i, n in enumerate(NS) for j in range(len(GESTS))]


def global_loo_spec(gsk, n, est, deg, dim, vk, nugget):
    from test_gpu_global_reference import global_spec
    g = global_spec(gsk, n, est, deg, dim, vk, nugget, "point")
    return gsk.ProblemSpec(coords=g.coords, values=g.values, points=g.coords, **g.params)


@pytest.mark.parametrize("n,est,deg,dim,vk,nugget", GDESIGN)
def test_global_loo_against_extended_reference(gsk, ctx, n, est, deg, dim, vk, nugget):
    spec = global_loo_spec(gsk, n, est, deg, dim, vk, nugget)
    m, v, nn = ctx.krige_loo(spec, want_nneigh=True)
    assert np.all(nn == n - 1)
    rows = np.random.default_rng(n + est).choice(n, 16, replace=False)
    others = np.array([[j for j in range(n) if j != i] for i in range(n)], dtype=np.int32)
    loc = gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=spec.coords,
                          **dict(spec.params, max_neighbors=n - 1))
    ref = XR.reference(loc, rows, others, np.full(n, n - 1))
    tol = 1e-6 if vk == 0 else 1e-9
    dm = np.abs(m[rows] - ref.mean) / np.maximum(1.0, np.abs(spec.values[rows]))
    dv = np.abs(v[rows] - ref.var) / spec.params["vario_sill"]
    assert dm.max() <= tol and dv.max() <= tol, (dm.max(), dv.max())


@pytest.mark.parametrize("n,est,deg,dim,vk", [(33, 1, 0, 2, 1), (64, 0, 0, 3, 2), (97, 2, 1, 2, 2), (64, 1, 0, 1, 1)])
def test_global_and_local_loo_agree(gsk, ctx, n, est, deg, dim, vk):
    g = global_loo_spec(gsk, n, est, deg, dim, vk, 0.06)
    mg, vg = ctx.krige_loo(g)
    loc = gsk.ProblemSpec(coords=g.coords, values=g.values, points=g.coords, **dict(g.params, max_neighbors=n - 1))
    ml, vl = ctx.krige_loo(loc)
    np.testing.assert_allclose(ml, mg, rtol=0, atol=1e-9 * max(1.0, np.abs(g.values).max()))
    np.testing.assert_allclose(vl, vg, rtol=0, atol=1e-9 * g.params["vario_sill"])


# ---- arguments and state ----
def _call(gsk, ctx, spec, **fields):
    from gskrige import _abi
    ps = _abi.loo_struct(spec)
    for f, val in fields.items():
        if f == "grid_dims0":
            ps.grid_dims[0] = val
        elif f == "points":
            ps.n_points = spec.n_samples
            for d in range(spec.dim):
                ps.point_coords[d] = _abi._ptr(spec.coords[d])
        else:
            setattr(ps, f, val)
    out = np.empty(max(spec.n_samples, 1))
    return ctx.lib.gsk_krige_loo(ctx._h, _abi.C.byref(ps), out.ctypes.data, out.ctypes.data, None, None)


def test_errors_and_state(gsk, ctx):
    spec = local_spec(gsk, 8, 1, 0, 2, 1, n=50)
    with pytest.raises(gsk.GskError) as e:
        ctx.krige_loo(gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=spec.coords, max_neighbors=8,
                                      solver=gsk.SOLVER_IDW))
    assert e.value.code == -2
    with pytest.raises(gsk.GskError) as e:
        ctx.krige_loo(gsk.ProblemSpec(coords=spec.coords, values=spec.values, points=spec.coords, max_neighbors=8,
                                      solver=gsk.SOLVER_LWR))
    assert e.value.code == -2
    assert _call(gsk, ctx, spec, grid_dims0=10) == -1
    assert _call(gsk, ctx, spec, points=True) == -1
    order = np.arange(50, dtype=np.int64)
    assert _call(gsk, ctx, spec, target_order=order.ctypes.data_as(gsk._abi._lp)) == -1
    assert _call(gsk, ctx, spec, n_support=2) == -1
    assert _call(gsk, ctx, spec, flags=gsk.FLAGS_DEFAULT | gsk.FLAG_REUSE_PLAN) == -1
    assert _call(gsk, ctx, spec, max_neighbors=50) == -1    # more than the fold's 49 samples
    one = gsk.ProblemSpec(coords=[c[:1] for c in spec.coords], values=spec.values[:1], points=[c[:1] for c in spec.coords])
    assert _call(gsk, ctx, one) == -1
    # a successful call leaves no plan behind
    ctx.krige_loo(spec)
    t = ctx.timing()
    assert t["targets"] == 50 and t["ms_plan"] > 0 and t["ms_total"] > 0
    import torch
    buf = torch.empty(2, dtype=torch.float64, device="cuda")
    with pytest.raises(gsk.GskError) as e:
        ctx.execute(0, 1, buf.data_ptr(), buf.data_ptr() + 8)
    assert e.value.code == -5


def test_leave_one_out_through_the_real_context(gsk, ctx):
    rng = np.random.default_rng(3)
    n = 120
    xy = rng.uniform(0, 20, size=(n, 2))
    t = list(10 + np.sin(xy[:, 0] / 4) + 0.1 * rng.standard_normal(n))
    for i in (5, 17, 60):
        t[i] = None
    u = np.ma.MaskedArray(np.cos(xy[:, 1] / 5), mask=np.isin(np.arange(n), [0, 99]))
    data = gsk.georef({"t": gsk.Quantities(t, gsk.degC), "u": u}, [tuple(p) for p in xy])
    solver = gsk.KrigingSolver(t=dict(variogram=gsk.SphericalVariogram(range=8.0), maxneighbors=16),
                               u=dict(variogram=gsk.ExponentialVariogram(range=10.0, nugget=0.01), degree=1))
    sol = gsk.leave_one_out(data, solver, ctx=ctx)
    tv = np.array([np.nan if x is None else x + 273.15 for x in t])
    keep = ~np.isnan(tv)
    st = gsk.ProblemSpec(coords=[xy[keep, 0], xy[keep, 1]], values=tv[keep], points=[xy[keep, 0], xy[keep, 1]],
                         vario_kind=gsk.VARIO_SPHERICAL, vario_range=8.0, estimator=gsk.EST_ORDINARY, max_neighbors=16)
    m, v = ctx.krige_loo(st)
    assert sol.t.unit == gsk.K
    assert np.array_equal(np.ma.getmaskarray(sol.t.values), ~keep)
    assert np.array_equal(sol.t.values.compressed(), m) and np.array_equal(sol.t_variance.values.compressed(), v)
    ku = ~np.ma.getmaskarray(u)
    su = gsk.ProblemSpec(coords=[xy[ku, 0], xy[ku, 1]], values=u.compressed(), points=[xy[ku, 0], xy[ku, 1]],
                         vario_kind=gsk.VARIO_EXPONENTIAL, vario_range=10.0, vario_nugget=0.01,
                         estimator=gsk.EST_UNIVERSAL, uk_degree=1)
    m, v = ctx.krige_loo(su)
    assert np.array_equal(np.ma.getmaskarray(sol.u), ~ku)
    assert np.array_equal(sol.u.compressed(), m) and np.array_equal(sol.u_variance.compressed(), v)
