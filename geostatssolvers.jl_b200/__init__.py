"""gskrige — B200-native Kriging estimation behind GeoStatsSolvers.jl's `solve(problem, KrigingSolver(...))`.

The directory is named ``geostatssolvers.jl_b200`` (not importable by that name because of the
dot); ``import gskrige`` (repo-root shim) loads it under the module name ``gskrige``.

Only the Kriging hot path exists here (SURVEY.md §8): the host mirror of the reference
interface (host.py), the ctypes binding of the C ABI (_abi.py), the build recipe (build.py)
and the CUDA sources (csrc/). No CPU fallback.
"""
from ._abi import (Context, GskError, ProblemSpec, krige_multi, default_support, default_support_py, load_library,  # noqa: F401
                   uk_exponents, EXPORTED_SYMBOLS, LIB_PATH,
                   VARIO_GAUSSIAN, VARIO_SPHERICAL, VARIO_EXPONENTIAL, EST_SIMPLE, EST_ORDINARY, EST_UNIVERSAL,
                   FLAG_CLAMP_VARIANCE, FLAG_SQRT_ROUNDTRIP, FLAG_REUSE_PLAN, FLAGS_DEFAULT, GSK_MAX_NEIGHBORS,
                   SOLVER_KRIGING, SOLVER_IDW, SOLVER_LWR)
from .host import (CartesianGrid, EstimationProblem, Euclidean, ExponentialVariogram, ExternalDriftKriging,  # noqa: F401
                   GaussianVariogram, GeoTable, IDWSolver, K, KBallSearch, KNearestSearch, Kriging, KrigingSolver, LWRSolver,
                   LinearPath, MetricBall, MultiGridPath, NoUnits, OrdinaryKriging, PointSet, Quantities, RandomPath,
                   SimpleKriging, SphericalVariogram, UniversalKriging, Unit, UnsupportedOption, approxsolve, asarray,
                   default_context, degC, elunit, embeddim, exactsolve, georef, krige_columns, kriging_ui, leave_one_out,
                   maxneighbors,
                   nelements,
                   preprocess, searcher_ui, solve, traverse, uadjust)
from . import sharding, simulation, synth  # noqa: F401
from .simulation import FFTGS, LUGS, SGS, SimulationProblem  # noqa: F401
from .sharding import gather_slabs, slab_bounds  # noqa: F401

__version__ = "0.1.0"
