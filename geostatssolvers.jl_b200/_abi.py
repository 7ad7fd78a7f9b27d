"""ctypes binding of include/gskrige.h (the C ABI of libgskrige.so).

This is the Python twin of the ``ccall`` layer in julia/GSKrige.jl: same struct, same
entry points. It carries no numerics. There is no CPU fallback — if libgskrige.so is
missing or no B200 is visible, compute calls raise.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
REPO_ROOT = PKG_DIR.parent
# GSKRIGE_LIB: development override (A/B of kernel variants built from other source states); not a fallback
LIB_PATH = Path(os.environ.get("GSKRIGE_LIB") or PKG_DIR / "csrc" / "libgskrige.so")

GSK_ABI_VERSION = 2
VARIO_GAUSSIAN, VARIO_SPHERICAL, VARIO_EXPONENTIAL = 0, 1, 2
EST_SIMPLE, EST_ORDINARY, EST_UNIVERSAL = 0, 1, 2
FLAG_CLAMP_VARIANCE, FLAG_SQRT_ROUNDTRIP, FLAG_REUSE_PLAN = 1, 2, 4
FLAGS_DEFAULT = 3
SOLVER_KRIGING, SOLVER_IDW, SOLVER_LWR = 0, 1, 2
LWR_WEIGHT_EXP3H2 = 0
GSK_MAX_NEIGHBORS = 96
GSK_MAX_SUPPORT = 125
GSK_MAX_SUPPORT_GLOBAL = 65536

ERRORS = {0: "ok", -1: "invalid argument", -2: "unsupported option", -3: "CUDA failure", -4: "out of memory",
          -5: "call-order violation"}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_int64)


class GskProblem(C.Structure):
    """Mirror of ``struct gsk_problem`` (include/gskrige.h)."""

    _fields_ = [
        ("abi_version", C.c_int32),
        ("dim", C.c_int32),
        ("n_samples", C.c_int64),
        ("coords", _dp * 3),
        ("values", _dp),
        ("grid_dims", C.c_int64 * 3),
        ("grid_origin", C.c_double * 3),
        ("grid_spacing", C.c_double * 3),
        ("n_points", C.c_int64),
        ("point_coords", _dp * 3),
        ("target_first", C.c_int64),
        ("target_count", C.c_int64),
        ("n_support", C.c_int32),
        ("support_offsets", _dp * 3),
        ("vario_kind", C.c_int32),
        ("vario_range", C.c_double),
        ("vario_sill", C.c_double),
        ("vario_nugget", C.c_double),
        ("gaussian_nugget_eps", C.c_double),
        ("estimator", C.c_int32),
        ("sk_mean", C.c_double),
        ("uk_degree", C.c_int32),
        ("min_neighbors", C.c_int32),
        ("max_neighbors", C.c_int32),
        ("ball_radius", C.c_double),
        ("flags", C.c_uint32),
        ("target_order", _lp),
        ("solver", C.c_int32),
        ("idw_exponent", C.c_double),
        ("lwr_weightfun", C.c_int32),
    ]


class GskTiming(C.Structure):
    _fields_ = [
        ("ms_plan", C.c_double),
        ("ms_search", C.c_double),
        ("ms_solve", C.c_double),
        ("ms_total", C.c_double),
        ("launches", C.c_int64),
        ("targets", C.c_int64),
    ]


def _as_f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _ptr(a):
    return a.ctypes.data_as(_dp)


class ProblemSpec:
    """Owns the numpy arrays behind a ``GskProblem`` (keeps them alive for the call)."""

    def __init__(self, *, coords, values, grid_dims=None, grid_origin=None, grid_spacing=None, points=None,
                 support=None, vario_kind=VARIO_GAUSSIAN, vario_range=1.0, vario_sill=1.0, vario_nugget=0.0,
                 gaussian_nugget_eps=1e-6, estimator=EST_ORDINARY, sk_mean=0.0, uk_degree=0, min_neighbors=1,
                 max_neighbors=0, ball_radius=float("nan"), flags=FLAGS_DEFAULT, target_first=0, target_count=-1,
                 target_order=None, solver=SOLVER_KRIGING, idw_exponent=1.0, lwr_weightfun=LWR_WEIGHT_EXP3H2):
        coords = [_as_f64(c) for c in coords]
        self.dim = len(coords)
        if not 1 <= self.dim <= 3:
            raise ValueError("dim must be 1, 2 or 3")
        self.coords = coords
        self.values = _as_f64(values)
        n = self.values.shape[0]
        if any(c.shape != (n,) for c in coords):
            raise ValueError("coords and values must have the same length")
        self.grid_dims = None
        self.points = None
        if grid_dims is not None:
            gd = [int(g) for g in grid_dims]
            if len(gd) != self.dim:
                raise ValueError("grid_dims must have `dim` entries")
            self.grid_dims = gd
            self.grid_origin = [float(x) for x in (grid_origin if grid_origin is not None else [0.0] * self.dim)]
            self.grid_spacing = [float(x) for x in (grid_spacing if grid_spacing is not None else [1.0] * self.dim)]
        else:
            if points is None:
                raise ValueError("either grid_dims or points is required")
            self.points = [_as_f64(p) for p in points]
            if len(self.points) != self.dim:
                raise ValueError("points must have `dim` coordinate arrays")
        if support is None:
            support = [np.zeros(1) for _ in range(self.dim)]
        self.support = [_as_f64(s) for s in support]
        self.params = dict(vario_kind=int(vario_kind), vario_range=float(vario_range), vario_sill=float(vario_sill),
                           vario_nugget=float(vario_nugget), gaussian_nugget_eps=float(gaussian_nugget_eps),
                           estimator=int(estimator), sk_mean=float(sk_mean), uk_degree=int(uk_degree),
                           min_neighbors=int(min_neighbors), max_neighbors=int(max_neighbors),
                           ball_radius=float(ball_radius), flags=int(flags), solver=int(solver),
                           idw_exponent=float(idw_exponent), lwr_weightfun=int(lwr_weightfun))
        self.target_first = int(target_first)
        self.target_count = int(target_count)
        self.target_order = None
        if target_order is not None:
            self.target_order = np.ascontiguousarray(np.asarray(target_order, dtype=np.int64))
            if self.target_order.shape != (self.n_targets,):
                raise ValueError("target_order must list every target once")

    # -- derived -------------------------------------------------------------------
    @property
    def n_samples(self):
        return int(self.values.shape[0])

    @property
    def n_targets(self):
        if self.grid_dims is not None:
            return int(np.prod(self.grid_dims, dtype=np.int64))
        return int(self.points[0].shape[0])

    @property
    def slab(self):
        first = self.target_first
        count = self.n_targets - first if self.target_count < 0 else self.target_count
        return first, count

    def with_slab(self, first, count):
        import copy
        other = copy.copy(self)
        other.target_first, other.target_count = int(first), int(count)
        return other

    def target_centers(self, first=None, count=None):
        """Centroids of targets [first, first+count) — origin + (i + 0.5)·spacing, x fastest."""
        if first is None:
            first, count = self.slab
        lin = np.arange(first, first + count, dtype=np.int64)
        if self.target_order is not None:
            lin = self.target_order[lin]
        if self.grid_dims is None:
            return [p[lin] for p in self.points]
        out, rem = [], lin
        for d in range(self.dim):
            i = rem % self.grid_dims[d]
            rem = rem // self.grid_dims[d]
            out.append(self.grid_origin[d] + (i.astype(np.float64) + 0.5) * self.grid_spacing[d])
        return out

    def c_struct(self):
        p = GskProblem()
        p.abi_version = GSK_ABI_VERSION
        p.dim = self.dim
        p.n_samples = self.n_samples
        for d in range(3):
            p.coords[d] = _ptr(self.coords[d]) if d < self.dim else None
            p.support_offsets[d] = _ptr(self.support[d]) if d < self.dim else None
            p.point_coords[d] = None
            p.grid_dims[d] = 1
            p.grid_origin[d] = 0.0
            p.grid_spacing[d] = 1.0
        p.values = _ptr(self.values)
        if self.grid_dims is not None:
            for d in range(self.dim):
                p.grid_dims[d] = self.grid_dims[d]
                p.grid_origin[d] = self.grid_origin[d]
                p.grid_spacing[d] = self.grid_spacing[d]
            p.n_points = 0
        else:
            p.grid_dims[0] = 0
            p.n_points = self.points[0].shape[0]
            for d in range(self.dim):
                p.point_coords[d] = _ptr(self.points[d])
        p.target_first = self.target_first
        p.target_count = self.target_count
        p.n_support = int(self.support[0].shape[0])
        for k, v in self.params.items():
            setattr(p, k, v)
        p.target_order = self.target_order.ctypes.data_as(_lp) if self.target_order is not None else None
        return p


def loo_struct(spec: ProblemSpec) -> GskProblem:
    """The ``GskProblem`` of a leave-one-out call: the spec's samples and parameters, no targets of its own (the
    samples are the targets), point support."""
    p = spec.c_struct()
    p.grid_dims[0] = 0
    p.n_points = 0
    p.n_support = 1
    for d in range(3):
        p.point_coords[d] = None
        p.support_offsets[d] = None
    p.target_order = None
    return p


# ------------------------------------------------------------------------------------
# library loading
# ------------------------------------------------------------------------------------
_lib = None


class GskError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libgskrige: {ERRORS.get(code, code)} ({code}): {message}")
        self.code = code


def load_library(path: os.PathLike | None = None):
    """dlopen libgskrige.so and declare every symbol of include/gskrige.h. Raises if absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else LIB_PATH
    if not p.exists():
        raise FileNotFoundError(
            f"{p} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the Kriging path)")
    lib = C.CDLL(str(p))
    ctx = C.c_void_p
    pp = C.POINTER(GskProblem)
    lib.gsk_create.argtypes = [C.POINTER(ctx), C.c_int]
    lib.gsk_create.restype = C.c_int
    lib.gsk_destroy.argtypes = [ctx]
    lib.gsk_destroy.restype = None
    lib.gsk_last_error.argtypes = [ctx]
    lib.gsk_last_error.restype = C.c_char_p
    lib.gsk_set_stream.argtypes = [ctx, C.c_void_p]
    lib.gsk_set_stream.restype = C.c_int
    lib.gsk_synchronize.argtypes = [ctx]
    lib.gsk_synchronize.restype = C.c_int
    lib.gsk_krige.argtypes = [ctx, pp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gsk_krige.restype = C.c_int
    lib.gsk_krige_loo.argtypes = [ctx, pp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gsk_krige_loo.restype = C.c_int
    lib.gsk_krige_columns.argtypes = [ctx, pp, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]
    lib.gsk_krige_columns.restype = C.c_int
    lib.gsk_krige_multi.argtypes = [_ip, C.c_int, pp, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
    lib.gsk_krige_multi.restype = C.c_int
    lib.gsk_krige_multi_release.argtypes = []
    lib.gsk_krige_multi_release.restype = None
    lib.gsk_plan.argtypes = [ctx, pp]
    lib.gsk_plan.restype = C.c_int
    lib.gsk_execute.argtypes = [ctx, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gsk_execute.restype = C.c_int
    lib.gsk_execute_peers.argtypes = [ctx, C.c_int64, C.c_int64, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                      C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
    lib.gsk_execute_peers.restype = C.c_int
    lib.gsk_update_values.argtypes = [ctx, _dp, C.c_int64]
    lib.gsk_update_values.restype = C.c_int
    lib.gsk_lu_plan.argtypes = [ctx, C.c_int, C.c_int64, C.c_int64, C.POINTER(_dp), _dp, C.c_int, C.c_double, C.c_double,
                                C.c_double, C.c_double]
    lib.gsk_lu_plan.restype = C.c_int
    lib.gsk_lu_sample.argtypes = [ctx, _dp, _dp]
    lib.gsk_lu_sample.restype = C.c_int
    lib.gsk_sgs_plan.argtypes = ([ctx, C.c_int, C.c_int64, C.POINTER(_dp), C.POINTER(C.c_int64), C.c_int] + [C.c_double] * 5
                                 + [C.c_int, C.c_int, C.c_double])
    lib.gsk_sgs_plan.restype = C.c_int
    lib.gsk_sgs_sample.argtypes = [ctx, C.c_int, _dp, _dp, _dp]
    lib.gsk_sgs_sample.restype = C.c_int
    lib.gsk_sgs_sample_device.argtypes = [ctx, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gsk_sgs_sample_device.restype = C.c_int
    lib.gsk_sgs_weights.argtypes = [ctx, _ip, _ip, _dp, _dp]
    lib.gsk_sgs_weights.restype = C.c_int
    lib.gsk_get_timing.argtypes = [ctx, C.POINTER(GskTiming)]
    lib.gsk_get_timing.restype = C.c_int
    lib.gsk_set_phase_timing.argtypes = [ctx, C.c_int]
    lib.gsk_set_phase_timing.restype = C.c_int
    lib.gsk_num_targets.argtypes = [pp]
    lib.gsk_num_targets.restype = C.c_int64
    lib.gsk_uk_exponents.argtypes = [C.c_int, C.c_int, _ip, C.c_int]
    lib.gsk_uk_exponents.restype = C.c_int
    lib.gsk_default_support.argtypes = [C.c_int, _dp, C.c_double, _dp, _dp, _dp, C.c_int]
    lib.gsk_default_support.restype = C.c_int
    lib.gsk_measure_fp64_peak.argtypes = [ctx, _dp, _dp]
    lib.gsk_measure_fp64_peak.restype = C.c_int
    lib.gsk_abi_version.argtypes = []
    lib.gsk_abi_version.restype = C.c_int
    if path is None:
        _lib = lib
    return lib


EXPORTED_SYMBOLS = [
    "gsk_create", "gsk_destroy", "gsk_last_error", "gsk_set_stream", "gsk_synchronize", "gsk_krige", "gsk_krige_loo", "gsk_krige_columns", "gsk_krige_multi", "gsk_krige_multi_release", "gsk_plan",
    "gsk_execute", "gsk_execute_peers", "gsk_update_values", "gsk_lu_plan", "gsk_lu_sample", "gsk_sgs_plan", "gsk_sgs_sample", "gsk_sgs_sample_device", "gsk_sgs_weights", "gsk_get_timing", "gsk_set_phase_timing", "gsk_num_targets", "gsk_uk_exponents", "gsk_default_support",
    "gsk_measure_fp64_peak", "gsk_abi_version",
]


class Context:
    """RAII wrapper of ``gsk_ctx`` (one CUDA device)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self._h = C.c_void_p()
        rc = self.lib.gsk_create(C.byref(self._h), int(device))
        if rc != 0:
            msg = self.lib.gsk_last_error(None)
            raise GskError(rc, msg.decode() if msg else "")
        self.device = device

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self.lib.gsk_destroy(h)
            self._h = None          # (module globals such as `C` may already be gone at interpreter shutdown)

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.gsk_last_error(self._h)
            raise GskError(rc, msg.decode() if msg else "")

    # -- one-shot, host buffers ------------------------------------------------------
    def krige(self, spec: ProblemSpec, want_neighbors: bool = False, want_nneigh: bool = False):
        """One-shot call. ``want_nneigh``: also return the neighbour COUNT per target (4 B per target — what the host
        needs to mark `missing`); ``want_neighbors``: also the count × k index lists (parity tests only)."""
        first, count = spec.slab
        mean = np.empty(count, dtype=np.float64)
        var = np.empty(count, dtype=np.float64)
        k = spec.params["max_neighbors"]
        nneigh = np.empty(count, dtype=np.int32) if (want_neighbors or want_nneigh) else None
        idx = np.empty((count, max(k, 1)), dtype=np.int32) if (want_neighbors and k > 0) else None
        ps = spec.c_struct()
        rc = self.lib.gsk_krige(self._h, C.byref(ps), mean.ctypes.data, var.ctypes.data,
                                nneigh.ctypes.data if nneigh is not None else None,
                                idx.ctypes.data if idx is not None else None)
        self._check(rc)
        if want_neighbors:
            return mean, var, nneigh, idx
        if want_nneigh:
            return mean, var, nneigh
        return mean, var

    def krige_loo(self, spec: ProblemSpec, want_nneigh: bool = False, want_neighbors: bool = False):
        """Leave-one-out cross-validation of the spec's samples (``gsk_krige_loo``): row i is sample i kriged at point
        support from the other samples. The spec's targets and support are not used (the samples are the targets);
        its slab (target_first, target_count) counts sample indices."""
        n = spec.n_samples
        first = spec.target_first
        count = n - first if spec.target_count < 0 else spec.target_count
        if not (0 <= first and 0 <= count and first + count <= n):
            raise ValueError("sample slab out of range")
        mean = np.empty(count, dtype=np.float64)
        var = np.empty(count, dtype=np.float64)
        k = spec.params["max_neighbors"]
        nneigh = np.empty(count, dtype=np.int32) if (want_neighbors or want_nneigh) else None
        idx = np.empty((count, max(k, 1)), dtype=np.int32) if (want_neighbors and k > 0) else None
        ps = loo_struct(spec)
        rc = self.lib.gsk_krige_loo(self._h, C.byref(ps), mean.ctypes.data, var.ctypes.data,
                                    nneigh.ctypes.data if nneigh is not None else None,
                                    idx.ctypes.data if idx is not None else None)
        self._check(rc)
        if want_neighbors:
            return mean, var, nneigh, idx
        if want_nneigh:
            return mean, var, nneigh
        return mean, var

    def krige_columns(self, spec: ProblemSpec, Z, want_nneigh: bool = False, want_neighbors: bool = False,
                      want_weights: bool = False):
        """Kriging of every column of ``Z`` (n_samples × m) over the spec's samples in one call (``gsk_krige_columns``):
        the search and the factorisations run once. The spec's own values are not used. Returns ``mean`` (count × m)
        and ``var`` (count), then — as requested — the neighbour counts, the count × k neighbour lists, and the
        count × k Kriging weights with the count × nterms Lagrange multipliers (local path only)."""
        Z = np.ascontiguousarray(Z, dtype=np.float64)
        if Z.ndim != 2 or Z.shape[0] != spec.n_samples or Z.shape[1] < 1:
            raise ValueError(f"Z must have shape (n_samples, m >= 1) = ({spec.n_samples}, m), got {Z.shape}")
        first, count = spec.slab
        m = Z.shape[1]
        k = spec.params["max_neighbors"]
        if want_weights and k == 0:
            raise ValueError("weights are returned by the local path only (max_neighbors > 0)")
        nterms = {EST_SIMPLE: 0, EST_ORDINARY: 1}.get(spec.params["estimator"])
        if nterms is None:
            nterms = len(uk_exponents(spec.params["uk_degree"], spec.dim))
        mean = np.empty((count, m), dtype=np.float64)
        var = np.empty(count, dtype=np.float64)
        nneigh = np.empty(count, dtype=np.int32) if (want_neighbors or want_nneigh) else None
        idx = np.empty((count, max(k, 1)), dtype=np.int32) if (want_neighbors and k > 0) else None
        w = np.empty((count, k), dtype=np.float64) if want_weights else None
        lag = np.empty((count, nterms), dtype=np.float64) if (want_weights and nterms > 0) else None
        ps = spec.c_struct()
        ps.values = None
        ptr = lambda a: a.ctypes.data if a is not None else None  # noqa: E731
        rc = self.lib.gsk_krige_columns(self._h, C.byref(ps), m, Z.ctypes.data, mean.ctypes.data, var.ctypes.data,
                                        ptr(nneigh), ptr(idx), ptr(w), ptr(lag))
        self._check(rc)
        out = [mean, var]
        if want_nneigh or want_neighbors:
            out.append(nneigh)
        if want_neighbors:
            out.append(idx)
        if want_weights:
            out += [w, lag if lag is not None else np.empty((count, 0))]
        return tuple(out)

    def krige_into(self, spec: ProblemSpec, mean: np.ndarray, var: np.ndarray):
        """Same as :meth:`krige` but writes into caller-provided (e.g. pinned) host arrays."""
        ps = spec.c_struct()
        self._check(self.lib.gsk_krige(self._h, C.byref(ps), mean.ctypes.data, var.ctypes.data, None, None))

    # -- resident two-step form ------------------------------------------------------
    def plan(self, spec: ProblemSpec):
        ps = spec.c_struct()
        self._check(self.lib.gsk_plan(self._h, C.byref(ps)))

    def update_values(self, values):
        """Values-only update of the planned problem (``gsk_update_values``): same coordinates, new sample values."""
        v = _as_f64(values)
        self._check(self.lib.gsk_update_values(self._h, _ptr(v), int(v.shape[0])))

    # -- LU Gaussian simulation --------------------------------------------------------
    def lu_plan(self, coords, n_data, data_values, *, vario_kind, vario_range, vario_sill=1.0, vario_nugget=0.0,
                gaussian_nugget_eps=1e-6):
        """coords: dim arrays of n_data + n_sim points, data locations first (``gsk_lu_plan``)."""
        cs = [_as_f64(c) for c in coords]
        n = cs[0].shape[0]
        arr = (_dp * 3)(*[_ptr(cs[d]) if d < len(cs) else None for d in range(3)])
        z = _as_f64(data_values) if n_data > 0 else None
        self._lu_n = n
        self._check(self.lib.gsk_lu_plan(self._h, len(cs), int(n_data), int(n - n_data), arr, _ptr(z) if z is not None else None,
                                         int(vario_kind), float(vario_range), float(vario_sill), float(vario_nugget),
                                         float(gaussian_nugget_eps)))

    def lu_sample(self, w):
        """one realisation for the standard normal draws ``w`` (length n_sim): the n_data + n_sim values"""
        w = _as_f64(w)
        y = np.empty(self._lu_n, dtype=np.float64)
        self._check(self.lib.gsk_lu_sample(self._h, _ptr(w), _ptr(y)))
        return y

    # -- sequential Gaussian simulation ------------------------------------------------
    def sgs_plan(self, coords, rank, *, vario_kind, vario_range, vario_sill=1.0, vario_nugget=0.0, gaussian_nugget_eps=1e-6,
                 mean=0.0, min_neighbors=1, max_neighbors=10, ball_radius=float("nan")):
        """coords: dim arrays with the n centroids of the domain; rank[i] = -1 where element i holds data, else its
        position in the simulation path among the other elements (``gsk_sgs_plan``)."""
        cs = [_as_f64(c) for c in coords]
        n = cs[0].shape[0]
        arr = (_dp * 3)(*[_ptr(cs[d]) if d < len(cs) else None for d in range(3)])
        rk = np.ascontiguousarray(rank, dtype=np.int64)
        if rk.shape != (n,):
            raise ValueError("rank must have one entry per element")
        self._sgs_n, self._sgs_k = n, min(int(max_neighbors), n)
        self._check(self.lib.gsk_sgs_plan(self._h, len(cs), n, arr, rk.ctypes.data_as(C.POINTER(C.c_int64)), int(vario_kind),
                                          float(vario_range), float(vario_sill), float(vario_nugget),
                                          float(gaussian_nugget_eps), float(mean), int(min_neighbors), int(max_neighbors),
                                          float(ball_radius)))

    def sgs_sample(self, z, values=None):
        """z: (nreal, n) or (n,) standard normal draws per element; values: (n,) read where rank < 0. Returns the
        realisations with the shape of z (``gsk_sgs_sample``)."""
        z = _as_f64(z)
        n = self._sgs_n
        if z.shape[-1] != n or z.ndim > 2:
            raise ValueError("z must be (n,) or (nreal, n)")
        nreal = 1 if z.ndim == 1 else z.shape[0]
        v = _as_f64(values) if values is not None else None
        if v is not None and v.shape != (n,):
            raise ValueError("values must have one entry per element")
        out = np.empty_like(z)
        self._check(self.lib.gsk_sgs_sample(self._h, nreal, _ptr(v) if v is not None else None, _ptr(z), _ptr(out)))
        return out

    def sgs_sample_device(self, nreal, d_values, d_z, d_out):
        """device pointers (ints; d_values may be 0 without data); asynchronous on the context stream"""
        self._check(self.lib.gsk_sgs_sample_device(self._h, int(nreal), C.c_void_p(d_values) if d_values else None,
                                                   C.c_void_p(d_z), C.c_void_p(d_out)))

    def sgs_weights(self):
        """(nneigh, idx, weights, sigma) of the resident plan (``gsk_sgs_weights``)."""
        n, k = self._sgs_n, self._sgs_k
        nn = np.empty(n, dtype=np.int32)
        idx = np.empty((n, k), dtype=np.int32)
        lam = np.empty((n, k))
        sig = np.empty(n)
        self._check(self.lib.gsk_sgs_weights(self._h, nn.ctypes.data_as(_ip), idx.ctypes.data_as(_ip), _ptr(lam), _ptr(sig)))
        return nn, idx, lam, sig

    def execute(self, first, count, d_mean, d_var, d_nneigh=0, d_idx=0):
        """Device pointers (ints). Asynchronous on the context stream."""
        self._check(self.lib.gsk_execute(self._h, int(first), int(count), C.c_void_p(d_mean), C.c_void_p(d_var),
                                         C.c_void_p(d_nneigh) if d_nneigh else None,
                                         C.c_void_p(d_idx) if d_idx else None))

    def execute_peers(self, first, count, mean_ptrs, var_ptrs, out_offset=0, multicast=False):
        """Like :meth:`execute`, but every result is stored into all peer-mapped buffers (fused gather)."""
        n = len(mean_ptrs)
        mp = (C.c_void_p * n)(*[C.c_void_p(int(p)) for p in mean_ptrs])
        vp = (C.c_void_p * n)(*[C.c_void_p(int(p)) for p in var_ptrs])
        self._check(self.lib.gsk_execute_peers(self._h, int(first), int(count), n, mp, vp, int(out_offset),
                                               int(bool(multicast)), None, None))

    def set_stream(self, cuda_stream: int):
        self._check(self.lib.gsk_set_stream(self._h, C.c_void_p(cuda_stream)))

    def set_phase_timing(self, on: bool):
        self._check(self.lib.gsk_set_phase_timing(self._h, int(bool(on))))

    def synchronize(self):
        self._check(self.lib.gsk_synchronize(self._h))

    def timing(self) -> dict:
        t = GskTiming()
        self._check(self.lib.gsk_get_timing(self._h, C.byref(t)))
        return {f: getattr(t, f) for f, _ in GskTiming._fields_}

    def measure_fp64_peak(self):
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.gsk_measure_fp64_peak(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value


def krige_multi(spec: ProblemSpec, device_ids, want_neighbors: bool = False, out=None):
    """Single-process multi-GPU call (``gsk_krige_multi``): the slab is split over ``device_ids``.
    ``out=(mean, var)``: caller-provided (e.g. page-locked) float64 arrays of the slab length."""
    lib = load_library()
    first, count = spec.slab
    mean, var = out if out is not None else (np.empty(count, dtype=np.float64), np.empty(count, dtype=np.float64))
    if mean.shape != (count,) or var.shape != (count,) or mean.dtype != np.float64 or var.dtype != np.float64:
        raise ValueError("out arrays must be float64 of the slab length")
    k = spec.params["max_neighbors"]
    nneigh = np.empty(count, dtype=np.int32) if want_neighbors else None
    idx = np.empty((count, max(k, 1)), dtype=np.int32) if (want_neighbors and k > 0) else None
    ids = np.asarray(list(device_ids), dtype=np.int32)
    err = C.create_string_buffer(512)
    ps = spec.c_struct()
    rc = lib.gsk_krige_multi(ids.ctypes.data_as(_ip), len(ids), C.byref(ps), mean.ctypes.data, var.ctypes.data,
                             nneigh.ctypes.data if nneigh is not None else None,
                             idx.ctypes.data if idx is not None else None, err, 512)
    if rc != 0:
        raise GskError(rc, err.value.decode())
    if want_neighbors:
        return mean, var, nneigh, idx
    return mean, var


# ------------------------------------------------------------------------------------
# host helpers (no device needed)
# ------------------------------------------------------------------------------------
def uk_exponents(degree: int, dim: int) -> np.ndarray:
    lib = load_library()
    out = np.zeros((16, dim), dtype=np.int32)
    n = lib.gsk_uk_exponents(degree, dim, out.ctypes.data_as(_ip), 16)
    if n < 0:
        raise GskError(n, "gsk_uk_exponents")
    return out[:n].copy()


def default_support(spacing, vario_range: float):
    """Block-support offsets of a grid cell (SURVEY §8a a15 / V1) via the library helper. Any size: the count is
    queried first (anisotropic cells or ranges shorter than the cell give far more than 27 points)."""
    lib = load_library()
    dim = len(spacing)
    sp = _as_f64(spacing)
    n = lib.gsk_default_support(dim, _ptr(sp), float(vario_range), None, None, None, 0)
    if n < 0:
        raise GskError(n, "gsk_default_support: the support of this cell size / range needs more than "
                          f"{GSK_MAX_SUPPORT_GLOBAL} points")
    bufs = [np.zeros(n) for _ in range(3)]
    m = lib.gsk_default_support(dim, _ptr(sp), float(vario_range), _ptr(bufs[0]), _ptr(bufs[1]), _ptr(bufs[2]), n)
    if m != n:
        raise GskError(m, "gsk_default_support")
    return [bufs[d] for d in range(dim)]


def default_support_py(spacing, vario_range: float):
    """Pure-Python statement of the same rule (used by the oracle-side tests, which must not
    depend on the CUDA library)."""
    sides = [float(s) for s in spacing]
    lmin = min(s for s in sides if s > 0)
    step = (min(vario_range, lmin) if vario_range > 0 else lmin) / 3.0
    axes = []
    for s in sides:
        n = max(1, int(math.ceil(s / step - 1e-12)))
        axes.append(np.array([(j / (n + 1) - 0.5) * s for j in range(1, n + 1)], dtype=np.float64))
    grids = np.meshgrid(*axes, indexing="ij")
    # x fastest
    return [np.ascontiguousarray(g.transpose(*reversed(range(len(axes)))).ravel()) for g in grids]
