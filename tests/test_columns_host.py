"""`krige_columns` without a GPU: how the host groups a problem's variables into one value matrix (through a fake
context), the differences it refuses, and the ctypes declaration of gsk_krige_columns against include/gskrige.h."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


class FakeContext:
    """Records (spec, Z) of every krige_columns call and answers with recognisable rows."""

    def __init__(self, nneigh=7):
        self.calls = []
        self.nneigh = nneigh

    def krige_columns(self, spec, Z, want_nneigh=False, want_neighbors=False, want_weights=False):
        self.calls.append((spec, Z))
        first, count = spec.slab
        mean = np.arange(count, dtype=np.float64)[:, None] * 10.0 + np.arange(Z.shape[1])[None, :]
        var = np.full(count, 0.25)
        nn = np.full(count, self.nneigh, dtype=np.int32)
        return (mean, var, nn) if want_nneigh else (mean, var)


def _table(gsk, c_missing=None):
    xy = [(0.0, 0.0), (1.0, 0.0), (0.0, 2.0), (3.0, 1.0), (2.0, 2.0)]
    t = [10.0, None, 12.0, 13.0, 14.0]                                     # °C, one missing
    u = np.ma.MaskedArray([1.0, 2.0, 3.0, 4.0, 5.0], mask=[0, 1, 0, 0, 0])
    c = np.ma.MaskedArray([5.0, 6.0, 7.0, 8.0, 9.0], mask=c_missing or [0, 1, 0, 0, 0])
    return gsk.georef({"t": gsk.Quantities(t, gsk.degC), "u": u, "c": c}, xy)


def test_columns_in_variable_order_with_units_and_masks(gsk):
    data = _table(gsk)
    grid = gsk.CartesianGrid((3, 2))
    prob = gsk.EstimationProblem(data, grid, ("t", "u", "c"))
    p = dict(variogram=gsk.SphericalVariogram(range=3.0, sill=2.0), maxneighbors=3, minneighbors=2)
    ctx = FakeContext(nneigh=1)
    sol = gsk.krige_columns(prob, gsk.KrigingSolver(t=p, u=p, c=p), ctx=ctx)
    (spec, Z), = ctx.calls
    assert Z.shape == (4, 3)
    np.testing.assert_array_equal(Z[:, 0], np.array([10.0, 12.0, 13.0, 14.0]) + 273.15)   # °C → K as solve does
    np.testing.assert_array_equal(Z[:, 1], [1.0, 3.0, 4.0, 5.0])
    np.testing.assert_array_equal(Z[:, 2], [5.0, 7.0, 8.0, 9.0])
    assert spec.n_samples == 4 and spec.params["max_neighbors"] == 3 and spec.params["min_neighbors"] == 2
    assert sol.names() == ["t", "u", "c", "t_variance", "u_variance", "c_variance"]
    assert sol.t.unit == gsk.K and repr(sol.t_variance.unit) == "K^2"
    assert np.ma.getmaskarray(sol.u).all()                                  # nneigh 1 < minneighbors 2
    ctx = FakeContext()
    sol = gsk.krige_columns(prob, gsk.KrigingSolver(t=p, u=p, c=p), ctx=ctx)
    np.testing.assert_array_equal(np.ma.getdata(sol.c), np.arange(6) * 10.0 + 2)


def test_global_problem_is_one_call(gsk):
    data = gsk.georef({"a": [1.0, 2.0, 3.0], "b": [3.0, 2.0, 1.0]}, [(0.0,), (1.0,), (2.0,)])
    prob = gsk.EstimationProblem(data, gsk.CartesianGrid((4,)), ("a", "b"))
    ctx = FakeContext()
    p = dict(variogram=gsk.GaussianVariogram(range=2.0), degree=1)
    sol = gsk.krige_columns(prob, gsk.KrigingSolver(a=p, b=p), ctx=ctx)
    (spec, Z), = ctx.calls
    assert spec.params["max_neighbors"] == 0 and spec.params["estimator"] == gsk.EST_UNIVERSAL
    assert Z.shape == (3, 2) and not np.ma.getmaskarray(sol.a).any()


def test_refuses_differing_missing_sets_and_parameters(gsk):
    data = _table(gsk, c_missing=[0, 0, 1, 0, 0])
    grid = gsk.CartesianGrid((3, 2))
    p = dict(variogram=gsk.SphericalVariogram(range=3.0), maxneighbors=3)
    with pytest.raises(ValueError, match="c and t have different non-missing samples"):
        gsk.krige_columns(gsk.EstimationProblem(data, grid, ("t", "u", "c")), gsk.KrigingSolver(t=p, u=p, c=p),
                          ctx=FakeContext())
    data = _table(gsk)
    prob = gsk.EstimationProblem(data, grid, ("t", "u"))
    for other, key in ((dict(p, maxneighbors=4), "maxneighbors"),
                       (dict(p, variogram=gsk.SphericalVariogram(range=3.5)), "variogram"),
                       (dict(p, mean=1.0), "mean")):
        with pytest.raises(ValueError, match=f"parameter `{key}` of u differs from t's"):
            gsk.krige_columns(prob, gsk.KrigingSolver(t=p, u=other), ctx=FakeContext())
    with pytest.raises(gsk.UnsupportedOption):
        gsk.krige_columns(prob, gsk.IDWSolver(t=dict(maxneighbors=2), u=dict(maxneighbors=2)), ctx=FakeContext())


def test_context_binding_checks_shapes(gsk):
    from gskrige import _abi
    ctx = _abi.Context.__new__(_abi.Context)   # no device: the checks run before any library call
    spec = gsk.ProblemSpec(coords=[np.arange(4.0)], values=np.arange(4.0), grid_dims=(3,), max_neighbors=2)
    with pytest.raises(ValueError, match="shape"):
        ctx.krige_columns(spec, np.zeros((3, 2)))
    with pytest.raises(ValueError, match="shape"):
        ctx.krige_columns(spec, np.zeros((4, 0)))
    gspec = gsk.ProblemSpec(coords=[np.arange(4.0)], values=np.arange(4.0), grid_dims=(3,), max_neighbors=0)
    with pytest.raises(ValueError, match="local path"):
        ctx.krige_columns(gspec, np.zeros((4, 2)), want_weights=True)


def test_ctypes_signature_matches_header(gsk):
    from gskrige import _abi
    hdr = (ROOT / "include" / "gskrige.h").read_text()
    decl = re.search(r"GSK_API int gsk_krige_columns\((.*?)\);", hdr, re.S).group(1)
    decl = re.sub(r"/\*.*?\*/", "", decl, flags=re.S)
    types = [re.sub(r"[\s*]*\w+$", "", a.strip()) + "*" * a.count("*") for a in decl.split(",")]
    assert types == ["gsk_ctx*", "const gsk_problem*", "int32_t", "const double*", "double*", "double*", "int32_t*",
                     "int32_t*", "double*", "double*"]
    lib = _abi.load_library()
    want = [C.c_void_p, C.POINTER(_abi.GskProblem), C.c_int32] + [C.c_void_p] * 7
    assert list(lib.gsk_krige_columns.argtypes) == want and lib.gsk_krige_columns.restype == C.c_int
    assert "gsk_krige_columns" in _abi.EXPORTED_SYMBOLS
