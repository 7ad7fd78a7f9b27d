"""Host-side mirror of the reference's Kriging solver interface.

Julia is not installed in the build or GPU images, so the host layer a Julia user would
keep (problem construction, units, missing values, per-variable loop, result table) is
mirrored here in Python with the reference's names, argument meaning and error behaviour;
julia/GSKrige.jl is the same logic as a Julia shim over the same C ABI.

Mirrors (reference file:line):
  IDWSolver / LWRSolver .............. src/estimation/idw.jl:50-148 / src/estimation/lwr.jl:53-152
  KrigingSolver + parameters ........ src/estimation/krig.jl:64-74
  preprocess ......................... src/estimation/krig.jl:76-128
  solve .............................. src/estimation/krig.jl:130-164
  exactsolve / approxsolve ........... src/estimation/krig.jl:166-186 / 188-234  → ONE ccall each (libgskrige.so)
  searcher_ui / kriging_ui ........... src/ui.jl:11-32 / 40-50
  elunit / uadjust ................... src/utils.jl:5-15

No numerics live here: the per-location loop of the reference is replaced by a single call
into the CUDA library. There is no CPU fallback.
"""
from __future__ import annotations

import dataclasses
import math
import warnings
from dataclasses import dataclass, field
from typing import Any, Callable, Optional, Sequence

import numpy as np

from . import _abi

# --------------------------------------------------------------------------------------
# units (stand-in for Unitful: only what utils.jl:5-15 needs)
# --------------------------------------------------------------------------------------


@dataclass(frozen=True)
class Unit:
    name: str
    affine_offset: float = 0.0        # value_abs = value + affine_offset   (°C → K: 273.15)
    absolute: Optional["Unit"] = None  # absoluteunit(U)

    @property
    def is_affine(self):
        return self.absolute is not None

    def __pow__(self, p):
        if self.name == "":
            return self
        return Unit(f"{self.name}^{p}")

    def __repr__(self):
        return self.name or "NoUnits"


NoUnits = Unit("")
K = Unit("K")
degC = Unit("°C", 273.15, K)
m = Unit("m")


class Quantities:
    """A column with a unit (``[1.0, 0.0, 1.0] * u"K"``); entries may be ``None``/masked (missing)."""

    def __init__(self, values, unit: Unit = NoUnits):
        self.values = values
        self.unit = unit

    def __rmul__(self, other):
        return Quantities(other, self.unit)

    def __repr__(self):
        return f"Quantities({self.values!r}, {self.unit!r})"


def _split_missing(col):
    """column → (float64 array with NaN at missing, bool mask of missing)"""
    if isinstance(col, np.ma.MaskedArray):
        mask = np.ma.getmaskarray(col).copy()
        vals = np.asarray(col.filled(np.nan), dtype=np.float64)
        return vals, mask
    arr = np.asarray(col, dtype=object) if not isinstance(col, np.ndarray) or col.dtype == object else col
    if arr.dtype == object:
        mask = np.array([v is None for v in arr], dtype=bool)
        vals = np.array([np.nan if v is None else float(v) for v in arr], dtype=np.float64)
        return vals, mask
    vals = np.asarray(arr, dtype=np.float64)
    return vals, np.zeros(vals.shape, dtype=bool)


def elunit(x) -> Unit:  # utils.jl:5
    return x.unit if isinstance(x, Quantities) else NoUnits


def uadjust(x):  # utils.jl:10-15
    """Affine units (°C) are converted to their absolute unit (K); everything else is unchanged."""
    u = elunit(x)
    if u.is_affine:
        vals, mask = _split_missing(x.values)
        out = np.ma.MaskedArray(vals + u.affine_offset, mask=mask)
        return Quantities(out, u.absolute)
    return x


# --------------------------------------------------------------------------------------
# domains (stand-in for the Meshes types the Kriging path touches)
# --------------------------------------------------------------------------------------


class PointSet:
    def __init__(self, coords):
        """dim×n matrix (Meshes' matrix constructor) or a list of n coordinate tuples."""
        if isinstance(coords, np.ndarray):
            a = np.asarray(coords, dtype=np.float64)
            if a.ndim == 1:
                a = a[None, :]
        else:
            coords = list(coords)
            if coords and isinstance(coords[0], (list, tuple, np.ndarray)):
                a = np.asarray(coords, dtype=np.float64).T
            else:
                a = np.asarray(coords, dtype=np.float64)[None, :]
        if a.ndim != 2 or not 1 <= a.shape[0] <= 3:
            raise ValueError("PointSet needs 1 to 3 coordinates per point")
        self.coords = np.ascontiguousarray(a)  # dim × n

    @property
    def dim(self):
        return self.coords.shape[0]

    def nelements(self):
        return self.coords.shape[1]

    def view(self, inds):
        return PointSet(self.coords[:, np.asarray(inds)])

    def centroids(self):
        return [np.ascontiguousarray(self.coords[d]) for d in range(self.dim)]


class CartesianGrid:
    """``CartesianGrid(100)``, ``CartesianGrid(100, 100)``, ``CartesianGrid((100,100), (0.5,0.5), (1.0,1.0))``
    (dims, origin, spacing) — ref test/estimation/krig.jl:7,26."""

    def __init__(self, *args):
        if len(args) >= 1 and isinstance(args[0], (tuple, list)):
            dims = tuple(int(d) for d in args[0])
            origin = tuple(float(x) for x in args[1]) if len(args) > 1 else (0.0,) * len(dims)
            spacing = tuple(float(x) for x in args[2]) if len(args) > 2 else (1.0,) * len(dims)
        else:
            dims = tuple(int(d) for d in args)
            origin = (0.0,) * len(dims)
            spacing = (1.0,) * len(dims)
        if not 1 <= len(dims) <= 3 or any(d < 1 for d in dims):
            raise ValueError("CartesianGrid needs 1 to 3 positive dimensions")
        self.dims, self.origin, self.spacing = dims, origin, spacing

    @property
    def dim(self):
        return len(self.dims)

    def nelements(self):
        return int(np.prod(self.dims, dtype=np.int64))

    def size(self):
        return self.dims

    def centroids(self):
        lin = np.arange(self.nelements(), dtype=np.int64)
        out, rem = [], lin
        for d in range(self.dim):
            i = rem % self.dims[d]
            rem = rem // self.dims[d]
            out.append(self.origin[d] + (i.astype(np.float64) + 0.5) * self.spacing[d])
        return out


def embeddim(domain):
    return domain.dim


def nelements(domain):
    return domain.nelements()


@dataclass
class MetricBall:
    """Isotropic ball (``MetricBall(100.0)``); anisotropic/rotated balls are outside the hot path."""
    radii: Any

    def __post_init__(self):
        if isinstance(self.radii, (tuple, list)):
            r = tuple(float(x) for x in self.radii)
            self.radii = r if len(set(r)) > 1 else r[0]
        else:
            self.radii = float(self.radii)

    @property
    def isotropic(self):
        return not isinstance(self.radii, tuple)

    def radius(self):
        if not self.isotropic:
            raise _unsupported("anisotropic MetricBall")
        return self.radii


class Euclidean:
    def __eq__(self, other):
        return isinstance(other, Euclidean)


class LinearPath:
    """Meshes' LinearPath: the domain's own order, 1:nelements."""


class MultiGridPath:
    """Meshes' MultiGridPath: coarse-to-fine traversal of a grid [3P-RECALLED, V10: restated as — for step sizes
    Δ = 2^L, 2^(L−1), …, 1 with 2^L >= the largest grid dimension, visit in column-major order every not yet visited
    cell whose (0-based) indices are all multiples of Δ]. The C ABI takes the order as an explicit array, so the Julia
    shim passes Meshes' own `traverse` result and does not depend on this restatement."""


class RandomPath:
    """Meshes' RandomPath: a random permutation (the reference draws it from Julia's RNG; here numpy's, seedable)."""

    def __init__(self, seed=None):
        self.seed = seed


def traverse(domain, path):
    """ref call sites src/estimation/krig.jl:179,204 — the visiting order as 0-based linear indices, or None for the
    domain's own order (LinearPath)."""
    if path is None or isinstance(path, LinearPath):
        return None
    n = domain.nelements()
    if isinstance(path, RandomPath):
        return np.random.default_rng(path.seed).permutation(n).astype(np.int64)
    if isinstance(path, MultiGridPath):
        if not isinstance(domain, CartesianGrid):
            raise _unsupported("MultiGridPath over a domain that is not a CartesianGrid")
        dims = domain.dims
        lin = np.arange(n, dtype=np.int64)
        idx, rem = [], lin
        for d in dims:
            idx.append(rem % d)
            rem = rem // d
        level = np.zeros(n, dtype=np.int64)          # the largest power of two dividing every index of the cell
        top = max(1, int(math.ceil(math.log2(max(dims)))) if max(dims) > 1 else 1)
        done = np.zeros(n, dtype=bool)
        order = []
        for lv in range(top, -1, -1):
            step = 1 << lv
            sel = np.ones(n, dtype=bool)
            for i in idx:
                sel &= (i % step) == 0
            sel &= ~done
            order.append(lin[sel])
            done |= sel
        del level
        return np.concatenate(order).astype(np.int64)
    raise _unsupported(f"path {type(path).__name__}")


# --------------------------------------------------------------------------------------
# geotables
# --------------------------------------------------------------------------------------


class GeoTable:
    def __init__(self, table: dict, domain):
        self.table = dict(table)
        self.domain = domain
        for name, col in self.table.items():
            vals = col.values if isinstance(col, Quantities) else col
            if len(vals) != domain.nelements():
                raise ValueError(f"column {name} has {len(vals)} rows, domain has {domain.nelements()} elements")

    def __getattr__(self, name):
        tbl = self.__dict__.get("table", {})
        if name in tbl:
            return tbl[name]
        raise AttributeError(name)

    def __getitem__(self, name):
        return self.table[name]

    def names(self):
        return list(self.table)


def georef(table: dict, domain_or_coords) -> GeoTable:
    dom = domain_or_coords
    if not isinstance(dom, (PointSet, CartesianGrid)):
        dom = PointSet(dom)
    return GeoTable(table, dom)


def asarray(sol: GeoTable, var: str) -> np.ndarray:
    """Column reshaped to the grid size, Julia (column-major) order: ``Z[i, j]`` with 0-based i, j."""
    col = sol.table[var]
    vals = col.values if isinstance(col, Quantities) else col
    return np.reshape(vals, sol.domain.size(), order="F")


# --------------------------------------------------------------------------------------
# variograms (parameters only — evaluation is in the CUDA library; formulas in DESIGN.md)
# --------------------------------------------------------------------------------------


class _Variogram:
    kind = -1

    def __init__(self, range=1.0, sill=1.0, nugget=0.0, **kw):
        if kw:
            raise _unsupported(f"variogram options {sorted(kw)} (anisotropy / custom distance)")
        self.range, self.sill, self.nugget = float(range), float(sill), float(nugget)


class GaussianVariogram(_Variogram):
    kind = _abi.VARIO_GAUSSIAN


class SphericalVariogram(_Variogram):
    kind = _abi.VARIO_SPHERICAL


class ExponentialVariogram(_Variogram):
    kind = _abi.VARIO_EXPONENTIAL


# --------------------------------------------------------------------------------------
# estimator / searcher descriptors returned by the *_ui helpers
# --------------------------------------------------------------------------------------


@dataclass
class OrdinaryKriging:
    variogram: Any


@dataclass
class SimpleKriging:
    variogram: Any
    mean: float


@dataclass
class UniversalKriging:
    variogram: Any
    degree: int
    dim: int


@dataclass
class ExternalDriftKriging:
    variogram: Any
    drifts: Any


@dataclass
class KNearestSearch:
    domain: Any
    k: int
    metric: Any = field(default_factory=Euclidean)


@dataclass
class KBallSearch:
    domain: Any
    k: int
    ball: MetricBall = None


def maxneighbors(method):
    return method.k


class UnsupportedOption(ValueError):
    """An option of the reference solver that is outside the accelerated hot path. Raised by the
    host layer (there is no CPU fallback to fall through to)."""


def _unsupported(what):
    return UnsupportedOption(f"{what} is not supported by the B200 Kriging path (no CPU fallback exists)")


def searcher_ui(domain, maxneighbors, metric, neighborhood):
    """ref src/ui.jl:11-32 — clamp k to the number of samples (with the reference's warning text),
    then kNN unless a neighbourhood is given."""
    nelem = nelements(domain)
    if maxneighbors is None:
        nmax = nelem
    elif maxneighbors < 1 or maxneighbors > nelem:
        warnings.warn(f"Invalid maximum number of neighbors. Adjusting to {nelem}...")
        nmax = nelem
    else:
        nmax = int(maxneighbors)
    if neighborhood is None:
        return KNearestSearch(domain, nmax, metric)
    return KBallSearch(domain, nmax, neighborhood)


def kriging_ui(domain, variogram, mean, degree, drifts):
    """ref src/ui.jl:40-50 — precedence drifts > degree > mean > ordinary."""
    if drifts is not None:
        return ExternalDriftKriging(variogram, drifts)
    if degree is not None:
        return UniversalKriging(variogram, int(degree), embeddim(domain))
    if mean is not None:
        return SimpleKriging(variogram, float(mean))
    return OrdinaryKriging(variogram)


# --------------------------------------------------------------------------------------
# problem + solver
# --------------------------------------------------------------------------------------


class EstimationProblem:
    """``EstimationProblem(geotable, domain, :z)`` (GeoStatsBase; ref test/estimation/krig.jl:8)."""

    def __init__(self, data: GeoTable, domain, vars):
        self._data, self._domain = data, domain
        self._vars = (vars,) if isinstance(vars, str) else tuple(vars)
        for v in self._vars:
            if v not in data.table:
                raise KeyError(f"variable {v} not found in the data")

    def data(self):
        return self._data

    def domain(self):
        return self._domain

    def variables(self):
        return self._vars


_DEFAULTS = dict(variogram=None, mean=None, degree=None, drifts=None, minneighbors=1, maxneighbors=None,
                 neighborhood=None, distance=None, path=None)


class KrigingSolver:
    """``KrigingSolver(z=dict(variogram=GaussianVariogram(range=35.), maxneighbors=3))`` or
    ``KrigingSolver(("z", {...}), ...)`` — the Python spelling of ``KrigingSolver(:z => (…))``.
    Parameters and defaults: ref src/estimation/krig.jl:64-74. Variables not listed get defaults."""

    def __init__(self, *pairs, **kwpairs):
        self.vparams = {}
        items = list(pairs) + list(kwpairs.items())
        for item in items:
            if isinstance(item, dict):
                sub = list(item.items())
            else:
                sub = [item]
            for var, params in sub:
                unknown = set(params) - set(_DEFAULTS)
                if unknown:
                    raise TypeError(f"unknown KrigingSolver parameter(s) {sorted(unknown)} for variable {var}")
                self.vparams[var] = dict(params)

    def params(self, var):
        p = dict(_DEFAULTS)
        p.update(self.vparams.get(var, {}))
        if p["variogram"] is None:
            p["variogram"] = GaussianVariogram()
        if p["distance"] is None:
            p["distance"] = Euclidean()
        if p["path"] is None:
            p["path"] = LinearPath()
        return p


Kriging = KrigingSolver  # north_star spells the solver `Kriging(...)` (older GeoStats releases)

_contexts: dict[int, _abi.Context] = {}


def default_context(device: int = 0) -> _abi.Context:
    if device not in _contexts:
        _contexts[device] = _abi.Context(device)
    return _contexts[device]


def preprocess(problem: EstimationProblem, solver: KrigingSolver) -> dict:
    """ref src/estimation/krig.jl:76-128"""
    pdata = problem.data()
    ddomain = pdata.domain
    pdomain = problem.domain()
    if not isinstance(ddomain, PointSet):
        raise _unsupported("sample domains that are not point sets")
    preproc = {}
    for var in problem.variables():
        varparams = solver.params(var)
        z = uadjust(pdata.table[var])                      # krig.jl:94
        unit = elunit(z)
        vals, missing = _split_missing(z.values if isinstance(z, Quantities) else z)
        inds = np.flatnonzero(~missing)                     # krig.jl:97
        if inds.size == 0:                                  # krig.jl:100-102
            raise AssertionError(f"all samples of {var} are missing, aborting...")
        vdomain = ddomain.view(inds)                        # krig.jl:106
        samples = GeoTable({var: vals[inds]}, vdomain)      # krig.jl:105-107
        estimator = kriging_ui(pdomain, varparams["variogram"], varparams["mean"], varparams["degree"],
                               varparams["drifts"])         # krig.jl:110
        searcher = searcher_ui(vdomain, varparams["maxneighbors"], varparams["distance"],
                               varparams["neighborhood"])   # krig.jl:117
        preproc[var] = dict(samples=samples, estimator=estimator, minneighbors=varparams["minneighbors"],
                            maxneighbors=varparams["maxneighbors"], searcher=searcher, path=varparams["path"],
                            unit=unit)
    return preproc


def _problem_spec(problem_samples: GeoTable, pdomain, var, pp, *, local: bool, order=None) -> _abi.ProblemSpec:
    est = pp["estimator"]
    searcher = pp["searcher"]
    gamma = est.variogram
    if isinstance(est, ExternalDriftKriging):
        raise _unsupported("ExternalDriftKriging (`drifts`, arbitrary host closures)")
    if not isinstance(gamma, _Variogram) or gamma.kind < 0:
        raise _unsupported(f"variogram {type(gamma).__name__}")
    if not isinstance(searcher.metric if isinstance(searcher, KNearestSearch) else Euclidean(), Euclidean):
        raise _unsupported("non-Euclidean `distance`")
    sdom = problem_samples.domain
    dim = sdom.dim
    if embeddim(pdomain) != dim:
        raise ValueError("sample and target domains have different embedding dimensions")
    kw = dict(coords=[sdom.coords[d] for d in range(dim)], values=problem_samples.table[var],
              vario_kind=gamma.kind, vario_range=gamma.range, vario_sill=gamma.sill, vario_nugget=gamma.nugget,
              target_order=order)
    if isinstance(pdomain, CartesianGrid):
        kw.update(grid_dims=pdomain.dims, grid_origin=pdomain.origin, grid_spacing=pdomain.spacing,
                  support=_abi.default_support(pdomain.spacing, gamma.range))
    elif isinstance(pdomain, PointSet):
        kw.update(points=pdomain.centroids())  # point support
    else:
        raise _unsupported(f"target domain {type(pdomain).__name__}")
    if isinstance(est, SimpleKriging):
        kw.update(estimator=_abi.EST_SIMPLE, sk_mean=est.mean)
    elif isinstance(est, UniversalKriging):
        if not 0 <= est.degree <= 2:
            raise _unsupported("UniversalKriging degree > 2")
        kw.update(estimator=_abi.EST_UNIVERSAL, uk_degree=est.degree)
    else:
        kw.update(estimator=_abi.EST_ORDINARY)
    if local:
        kw.update(max_neighbors=searcher.k, min_neighbors=int(pp["minneighbors"]))
        if isinstance(searcher, KBallSearch):
            kw.update(ball_radius=searcher.ball.radius())
        if searcher.k > _abi.GSK_MAX_NEIGHBORS:
            raise _unsupported(f"maxneighbors > {_abi.GSK_MAX_NEIGHBORS} on the local path")
    return _abi.ProblemSpec(**kw)


def _path_order(pdomain, path, path_order: bool):
    """The traversal order handed to the library: the reference maps over `traverse(pdomain, path)` and returns the
    predictions in VISITING order without permuting back (krig.jl:179-183, 204-231), so for a non-linear path row j of
    the result belongs to the j-th visited cell. `path_order=False` asks for domain order instead."""
    return traverse(pdomain, path) if path_order else None


def exactsolve(problem: EstimationProblem, var: str, preproc: dict, ctx: Optional[_abi.Context] = None, path_order=True):
    """ref src/estimation/krig.jl:166-186 — fit once on all samples, predict everywhere.
    One call into libgskrige.so (global system: one FP64 factorisation, batched triangular solves)."""
    pp = preproc[var]
    spec = _problem_spec(problem.data(), problem.domain(), var, pp, local=False,
                         order=_path_order(problem.domain(), pp["path"], path_order))
    mean, variance = (ctx or default_context()).krige(spec)
    return mean, variance


def approxsolve(problem: EstimationProblem, var: str, preproc: dict, ctx: Optional[_abi.Context] = None, path_order=True):
    """ref src/estimation/krig.jl:188-234 — per-location search → fit → predict, as ONE library call.
    Locations with fewer than `minneighbors` neighbours come back masked (the reference's `missing`). Only the
    neighbour COUNTS (4 B per target) come back with the two fields, never the index lists."""
    pp = preproc[var]
    spec = _problem_spec(problem.data(), problem.domain(), var, pp, local=True,
                         order=_path_order(problem.domain(), pp["path"], path_order))
    mean, variance, nneigh = (ctx or default_context()).krige(spec, want_nneigh=True)
    miss = nneigh < max(int(pp["minneighbors"]), 1)
    if miss.any():
        mean = np.ma.MaskedArray(mean, mask=miss)
        variance = np.ma.MaskedArray(variance, mask=miss)
    return mean, variance


def _solve_kriging(problem: EstimationProblem, solver: KrigingSolver, ctx, path_order) -> GeoTable:
    pdomain = problem.domain()
    preproc = preprocess(problem, solver)
    mus, sigmas = {}, {}
    for var in problem.variables():
        pp = preproc[var]
        prob = EstimationProblem(pp["samples"], pdomain, var)            # krig.jl:148
        if pp["maxneighbors"] is None:                                  # krig.jl:151
            varmu, varsigma = exactsolve(prob, var, preproc, ctx, path_order)
        else:
            varmu, varsigma = approxsolve(prob, var, preproc, ctx, path_order)
        unit = pp["unit"]
        if unit is not NoUnits:
            varmu, varsigma = Quantities(varmu, unit), Quantities(varsigma, unit ** 2)  # krig.jl:160
        mus[var] = varmu
        sigmas[f"{var}_variance"] = varsigma
    return georef({**mus, **sigmas}, pdomain)                           # krig.jl:163


def leave_one_out(data: GeoTable, solver: KrigingSolver, ctx: Optional[_abi.Context] = None) -> GeoTable:
    """Leave-one-out cross-validation (GeoStatsValidation's ``LeaveOneOut`` folds, each solved by ``solver``) as one
    library call per variable: row i of column `var` is sample i kriged at its own location from the other non-missing
    samples with the same parameters, `var_variance` its kriging variance (units u and u², as `solve` gives them).
    Every variable of the table is validated; rows whose value is missing come back masked, and so do rows with fewer
    than `minneighbors` neighbours. Each fold holds one sample less, so `maxneighbors` is clamped to n − 1 with the
    reference's warning. `path` does not apply (every sample is its own target)."""
    if not isinstance(solver, KrigingSolver):
        raise _unsupported(f"leave-one-out with {type(solver).__name__} (Kriging only)")
    ddomain = data.domain
    problem = EstimationProblem(data, ddomain, tuple(data.names()))
    preproc = preprocess(problem, solver)
    nrows = ddomain.nelements()
    mus, sigmas = {}, {}
    for var in problem.variables():
        pp = dict(preproc[var])
        samples = pp["samples"]
        n = samples.domain.nelements()
        if n < 2:
            raise AssertionError(f"leave-one-out of {var} needs at least two non-missing samples")
        local = pp["maxneighbors"] is not None
        if local and pp["searcher"].k > n - 1:                           # the fold's own searcher_ui clamp (ui.jl:16-23)
            warnings.warn(f"Invalid maximum number of neighbors. Adjusting to {n - 1}...")
            pp["searcher"] = dataclasses.replace(pp["searcher"], k=n - 1)
        spec = _problem_spec(samples, samples.domain, var, pp, local=local)
        mean, variance, nneigh = (ctx or default_context()).krige_loo(spec, want_nneigh=True)
        _, missing = _split_missing(uadjust(data.table[var]).values if isinstance(data.table[var], Quantities)
                                    else data.table[var])
        inds = np.flatnonzero(~missing)
        mask = np.ones(nrows, dtype=bool)
        mask[inds] = nneigh < max(int(pp["minneighbors"]), 1)
        mu = np.full(nrows, np.nan)
        sig = np.full(nrows, np.nan)
        mu[inds], sig[inds] = mean, variance
        if mask.any():
            mu, sig = np.ma.MaskedArray(mu, mask=mask), np.ma.MaskedArray(sig, mask=mask.copy())
        unit = pp["unit"]
        if unit is not NoUnits:
            mu, sig = Quantities(mu, unit), Quantities(sig, unit ** 2)
        mus[var] = mu
        sigmas[f"{var}_variance"] = sig
    return georef({**mus, **sigmas}, ddomain)


# --------------------------------------------------------------------------------------
# IDWSolver / LWRSolver: same searcher, traversal and centroid step, other per-location body (SURVEY §8f-1)
# --------------------------------------------------------------------------------------
_IDW_DEFAULTS = dict(minneighbors=1, maxneighbors=None, neighborhood=None, distance=None, exponent=1, path=None)
_LWR_DEFAULTS = dict(minneighbors=1, maxneighbors=None, neighborhood=None, distance=None, weightfun=None, path=None)


class _SimpleSolver:
    _defaults: dict = {}

    def __init__(self, *pairs, **kwpairs):
        self.vparams = {}
        for item in list(pairs) + list(kwpairs.items()):
            for var, params in (list(item.items()) if isinstance(item, dict) else [item]):
                unknown = set(params) - set(self._defaults)
                if unknown:
                    raise TypeError(f"unknown {type(self).__name__} parameter(s) {sorted(unknown)} for variable {var}")
                self.vparams[var] = dict(params)

    def params(self, var):
        p = dict(self._defaults)
        p.update(self.vparams.get(var, {}))
        if p["distance"] is None:
            p["distance"] = Euclidean()
        if p["path"] is None:
            p["path"] = LinearPath()
        return p


class IDWSolver(_SimpleSolver):
    """``IDWSolver(z=dict(maxneighbors=3))`` — parameters and defaults: ref src/estimation/idw.jl:50-57."""
    _defaults = _IDW_DEFAULTS


class LWRSolver(_SimpleSolver):
    """``LWRSolver(z=dict(maxneighbors=10))`` — parameters and defaults: ref src/estimation/lwr.jl:53-60. Only the
    default weight function h -> exp(-3 h^2) crosses the C ABI (`weightfun=None`)."""
    _defaults = _LWR_DEFAULTS


def _solve_simple(problem: EstimationProblem, solver: _SimpleSolver, ctx, path_order) -> GeoTable:
    """ref src/estimation/idw.jl:59-148 and src/estimation/lwr.jl:62-152 (host part; the estimation loop is one library call)."""
    pdata = problem.data()
    ddomain = pdata.domain
    pdomain = problem.domain()
    if not isinstance(ddomain, PointSet):
        raise _unsupported("sample domains that are not point sets")
    is_idw = isinstance(solver, IDWSolver)
    mus, sigmas = {}, {}
    for var in problem.variables():
        p = solver.params(var)
        vals, missing = _split_missing(pdata.table[var].values if isinstance(pdata.table[var], Quantities) else pdata.table[var])
        dinds = np.flatnonzero(~missing)                                   # idw.jl:78 / lwr.jl:81
        sdom = ddomain.view(dinds)
        n = sdom.nelements()
        nmin = int(p["minneighbors"])
        nmax = n if p["maxneighbors"] is None else min(int(p["maxneighbors"]), n)
        assert n > 0, "estimation requires data"                           # idw.jl:95 / lwr.jl:97
        if is_idw:
            assert p["exponent"] > 0, "exponent must be positive"          # idw.jl:96
        elif p["weightfun"] is not None:
            raise _unsupported("a custom LWR `weightfun` (an arbitrary closure)")
        assert nmin <= nmax, "invalid min/max number of neighbors"         # idw.jl:97 / lwr.jl:98
        if not isinstance(p["distance"], Euclidean):
            raise _unsupported("non-Euclidean `distance`")
        searcher = searcher_ui(sdom, p["maxneighbors"], p["distance"], p["neighborhood"])   # idw.jl:100 / lwr.jl:101
        z = uadjust(pdata.table[var])                                      # idw.jl:111 / lwr.jl:112
        unit = elunit(z)
        zvals, _ = _split_missing(z.values if isinstance(z, Quantities) else z)
        dim = sdom.dim
        if embeddim(pdomain) != dim:
            raise ValueError("sample and target domains have different embedding dimensions")
        k = 0 if p["maxneighbors"] is None else searcher.k
        if k > _abi.GSK_MAX_NEIGHBORS:
            raise _unsupported(f"maxneighbors > {_abi.GSK_MAX_NEIGHBORS} (omit it to use every sample)")
        kw = dict(coords=[sdom.coords[d] for d in range(dim)], values=zvals[dinds], max_neighbors=k, min_neighbors=nmin,
                  solver=_abi.SOLVER_IDW if is_idw else _abi.SOLVER_LWR, idw_exponent=float(p.get("exponent", 1.0)),
                  target_order=_path_order(pdomain, p["path"], path_order))
        if isinstance(pdomain, CartesianGrid):
            kw.update(grid_dims=pdomain.dims, grid_origin=pdomain.origin, grid_spacing=pdomain.spacing)
        elif isinstance(pdomain, PointSet):
            kw.update(points=pdomain.centroids())
        else:
            raise _unsupported(f"target domain {type(pdomain).__name__}")
        if k > 0 and isinstance(searcher, KBallSearch):
            kw.update(ball_radius=searcher.ball.radius())
        spec = _abi.ProblemSpec(**kw)
        mu, sig, nneigh = (ctx or default_context()).krige(spec, want_nneigh=True)
        miss = nneigh < max(nmin, 1)                                       # idw.jl:121-122 → (missing, missing)
        if miss.any():
            mu, sig = np.ma.MaskedArray(mu, mask=miss), np.ma.MaskedArray(sig, mask=miss)
        if is_idw:
            mus[var] = Quantities(mu, unit) if unit is not NoUnits else mu
            sigmas[f"{var}_distance"] = sig                                # idw.jl:146: no unit on the distance column
        else:
            mus[var] = Quantities(mu, unit) if unit is not NoUnits else mu
            sigmas[f"{var}_variance"] = Quantities(sig, unit ** 2) if unit is not NoUnits else sig   # lwr.jl:152
    return georef({**mus, **sigmas}, pdomain)


def solve(problem: EstimationProblem, solver, ctx: Optional[_abi.Context] = None, path_order: bool = True) -> GeoTable:
    """ref src/estimation/krig.jl:130-164 (KrigingSolver: columns `var`, `var_variance`, units u and u²),
    src/estimation/idw.jl:59-148 (IDWSolver: `var`, `var_distance`), src/estimation/lwr.jl:62-152 (LWRSolver: `var`,
    `var_variance`).

    Row order: for a non-linear `path` the reference returns its predictions in VISITING order (it maps over
    `traverse(pdomain, path)` and never permutes back), and so does this function by default; `path_order=False`
    returns domain (linear-index) order for every path — predictions do not depend on the visiting order."""
    if isinstance(solver, KrigingSolver):
        return _solve_kriging(problem, solver, ctx, path_order)
    if isinstance(solver, _SimpleSolver):
        return _solve_simple(problem, solver, ctx, path_order)
    from . import simulation as _sim
    if isinstance(solver, _sim.FFTGS):
        return _sim.solve_fftgs(problem, solver, ctx)
    if isinstance(solver, _sim.LUGS):
        return _sim.solve_lugs(problem, solver, ctx)
    if isinstance(solver, _sim.SGS):
        return _sim.solve_sgs(problem, solver, ctx)
    raise TypeError(f"solve: unsupported solver {type(solver).__name__}")
