"""Leave-one-out cross-validation without a GPU: what `leave_one_out` hands to the library (through a fake context),
and the tests' leave-one-out reference (tests/_loo_oracle.py: a brute-force scan that skips the sample, then the C
oracle's per-target solve) against n separate oracle solves with the sample deleted."""
import warnings

import numpy as np
import pytest

import _loo_oracle as LO


class FakeContext:
    """Records the spec of every krige_loo call and answers with recognisable rows."""

    def __init__(self, nneigh_fn=None):
        self.calls = []
        self.nneigh_fn = nneigh_fn

    def krige_loo(self, spec, want_nneigh=False, want_neighbors=False):
        self.calls.append(spec)
        n = spec.n_samples
        mean = spec.values + 0.5
        var = np.full(n, 0.25)
        nn = np.full(n, 7, dtype=np.int32) if self.nneigh_fn is None else self.nneigh_fn(spec)
        return (mean, var, nn) if want_nneigh else (mean, var)


def _table(gsk):
    xy = [(0.0, 0.0), (1.0, 0.0), (0.0, 2.0), (3.0, 1.0), (2.0, 2.0), (4.0, 4.0)]
    t = [10.0, None, 12.0, 13.0, None, 15.0]                     # °C, two missing
    u = np.ma.MaskedArray([1.0, 2.0, 3.0, 4.0, 5.0, 6.0], mask=[0, 0, 0, 0, 0, 1])
    return gsk.georef({"t": gsk.Quantities(t, gsk.degC), "u": u}, xy)


def test_leave_one_out_hands_samples_units_and_clamped_k(gsk):
    data = _table(gsk)
    ctx = FakeContext()
    solver = gsk.KrigingSolver(t=dict(variogram=gsk.SphericalVariogram(range=3.0, sill=2.0), maxneighbors=4,
                                      neighborhood=gsk.MetricBall(2.5), minneighbors=2),
                               u=dict(variogram=gsk.ExponentialVariogram(range=5.0), mean=3.0, maxneighbors=10))
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        sol = gsk.leave_one_out(data, solver, ctx=ctx)
    st, su = ctx.calls
    # t: the four non-missing samples in data order, °C → K, k = 4 clamped to the fold's 3 samples, ball radius
    assert st.n_samples == 4
    np.testing.assert_array_equal(st.values, np.array([10.0, 12.0, 13.0, 15.0]) + 273.15)
    np.testing.assert_array_equal(st.coords[0], [0.0, 0.0, 3.0, 4.0])
    np.testing.assert_array_equal(st.coords[1], [0.0, 2.0, 1.0, 4.0])
    assert st.params["max_neighbors"] == 3 and st.params["min_neighbors"] == 2
    assert st.params["ball_radius"] == 2.5
    assert st.params["estimator"] == gsk.EST_ORDINARY and st.params["vario_kind"] == gsk.VARIO_SPHERICAL
    assert st.params["vario_sill"] == 2.0
    # u: five samples, Simple Kriging, maxneighbors 10 → 5 by preprocess' clamp, then 4 by the fold's
    assert su.n_samples == 5 and su.params["max_neighbors"] == 4
    assert su.params["estimator"] == gsk.EST_SIMPLE and su.params["sk_mean"] == 3.0
    assert su.params["ball_radius"] != su.params["ball_radius"]  # NaN: KNearestSearch
    msgs = [str(x.message) for x in w]
    assert "Invalid maximum number of neighbors. Adjusting to 3..." in msgs
    assert "Invalid maximum number of neighbors. Adjusting to 4..." in msgs
    # the C struct of the call: no targets of its own, point support
    from gskrige import _abi
    ps = _abi.loo_struct(st)
    assert ps.grid_dims[0] == 0 and ps.n_points == 0 and ps.n_support == 1 and not ps.target_order
    # result: data domain and order, masked where missing, units K and K²
    assert sol.names() == ["t", "u", "t_variance", "u_variance"]
    assert sol.t.unit == gsk.K and repr(sol.t_variance.unit) == "K^2"
    tm = sol.t.values
    assert list(np.ma.getmaskarray(tm)) == [False, True, False, False, True, False]
    np.testing.assert_array_equal(tm.compressed(), np.array([10.0, 12.0, 13.0, 15.0]) + 273.15 + 0.5)
    np.testing.assert_array_equal(sol.t_variance.values.compressed(), [0.25] * 4)
    um = sol.u
    assert list(np.ma.getmaskarray(um)) == [False] * 5 + [True]
    np.testing.assert_array_equal(um.compressed(), [1.5, 2.5, 3.5, 4.5, 5.5])


def test_leave_one_out_global_and_min_neighbors_mask(gsk):
    data = gsk.georef({"z": [1.0, 2.0, 3.0, 4.0]}, [(0.0,), (1.0,), (2.0,), (5.0,)])
    ctx = FakeContext(nneigh_fn=lambda spec: np.array([2, 1, 2, 0], dtype=np.int32))
    sol = gsk.leave_one_out(data, gsk.KrigingSolver(z=dict(variogram=gsk.GaussianVariogram(range=2.0), degree=1)), ctx=ctx)
    (s,) = ctx.calls
    assert s.params["max_neighbors"] == 0                       # global: every other sample
    assert s.params["estimator"] == gsk.EST_UNIVERSAL and s.params["uk_degree"] == 1
    assert list(np.ma.getmaskarray(sol.z)) == [False, False, False, True]   # nneigh < max(minneighbors, 1)
    assert not isinstance(sol.z, gsk.Quantities)


@pytest.mark.parametrize("params", [dict(drifts=[lambda x: 1.0]), dict(degree=3),
                                    dict(maxneighbors=2, neighborhood="aniso")])
def test_leave_one_out_rejects_what_solve_rejects(gsk, params):
    if params.get("neighborhood") == "aniso":
        params = dict(params, neighborhood=gsk.MetricBall((1.0, 2.0)))
    data = gsk.georef({"z": [1.0, 2.0, 3.0, 4.0]}, [(0.0, 0.0), (1.0, 0.0), (2.0, 1.0), (5.0, 5.0)])
    with pytest.raises(gsk.UnsupportedOption):
        gsk.leave_one_out(data, gsk.KrigingSolver(z=params), ctx=FakeContext())
    with pytest.raises(gsk.UnsupportedOption):
        gsk.leave_one_out(data, gsk.IDWSolver(z=dict(maxneighbors=2)), ctx=FakeContext())


def _deleted(gsk, spec, i):
    keep = np.arange(spec.n_samples) != i
    return gsk.ProblemSpec(coords=[c[keep] for c in spec.coords], values=spec.values[keep],
                           points=[c[i:i + 1] for c in spec.coords], **spec.params)


@pytest.mark.parametrize("dim,k,est,deg,vk", [(2, 6, 1, 0, 1), (2, 0, 2, 1, 2), (3, 12, 0, 0, 2), (3, 0, 1, 0, 0),
                                              (3, 10, 2, 2, 1)])
def test_loo_reference_equals_deleted_solves(gsk, oracle, dim, k, est, deg, vk):
    n = 40
    grid = {2: (10, 8), 3: (5, 4, 4)}[dim]
    coords, vals = gsk.synth.make_samples(900 + dim, n, grid, seed_extra=k + est)
    coords = [c.copy() for c in coords]
    for d in range(dim):
        coords[d][7] = coords[d][3]                             # a twin: sample 7 sits on sample 3
    spec = gsk.ProblemSpec(coords=coords, values=vals, points=coords, vario_kind=vk, vario_range=4.0, vario_sill=1.2,
                           vario_nugget=0.05, estimator=est, uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=k)
    m, v, nn, idx = LO.krige_loo(oracle, spec, want_neighbors=True)
    assert np.all(nn == (k if k else n - 1))
    for i in range(n):
        dm, dv, dnn, didx = oracle.krige(_deleted(gsk, spec, i), search=oracle.SEARCH_BRUTE, want_neighbors=True)
        np.testing.assert_allclose(m[i], dm[0], rtol=1e-15, atol=0)
        np.testing.assert_allclose(v[i], dv[0], rtol=1e-15, atol=0)
        assert nn[i] == dnn[0]
        if k:
            full = np.where(didx[0] >= i, didx[0] + 1, didx[0])    # back to the indices of the full sample set
            assert np.array_equal(idx[i], full) and i not in idx[i]
    if k:
        assert 3 in idx[7] and 7 in idx[3]                      # the twin is a neighbour at distance zero
