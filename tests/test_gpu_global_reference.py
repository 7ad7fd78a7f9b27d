"""The global ("exact", max_neighbors == 0) path against the C oracle and against the extended-precision reference
(oracle/extended_ref.py) at a bound derived from each target's own system.

Rule: |gpu − ref| ≤ c·u·B + 2u·|ref| with u = 2⁻⁵³ and c = 4(m + q), m = n + c_drift the system size, q the support
points per target. B is the first-order change of the output when every entry of K, r and z moves by one unit roundoff
(Bμ for the mean, Bσ for the variance, see extended_ref.py). A backward-stable float64 solve perturbs the entries by
γ_m·|L||Lᵀ| ≈ m·u relatively; the right-hand side is a q-term average, so its entries carry up to q·u; the factor 4
covers the two triangular sweeps and the final dot products. The global variance is evaluated in Gram form through an
explicit L⁻¹, whose forward error is not backward stable: Bσ carries the derived term 2|ỹ|ᵀ|L⁻¹||L||L⁻¹|(|b| + |F||ν|)
(``gram=True``). The mean comes from dual weights refined against the assembled system and needs no extra term.

For spherical and exponential variograms the bound is asserted to be at most 1e-10 (relative to max(1, |z|) for the
mean and to the sill for the variance), so a bound that quietly grows fails instead of passing everything."""
import numpy as np
import pytest

from conftest import assert_parity

import extended_ref as XR

pytestmark = pytest.mark.gpu

C_FACTOR = 4
SILL = 1.3

# factor levels; the design below puts every level of each factor against every level of every other at least once
NS = (63, 64, 65, 127, 128, 129, 255, 256, 257)          # around the 64-row factor blocks and 128-row GEMM tiles
ESTS = ((0, 0), (1, 0), (2, 0), (2, 1), (2, 2))           # SK, OK, UK degree 0, 1, 2
DIMS, VARIOS, NUGGETS, SUPPORTS = (1, 2, 3), (0, 1, 2), (0.0, 0.06), ("point", "block", "big")
DESIGN = [(n, *ESTS[j], DIMS[(i + j) % 3], VARIOS[(i + 2 * j) % 3], NUGGETS[(i + j) % 2], SUPPORTS[(j + i // 3) % 3])
          for i, n in enumerate(NS) for j in range(len(ESTS))]

GRID = {1: (320,), 2: (12, 10), 3: (6, 5, 4)}
RANGE = {0: {1: 4.0, 2: 3.0, 3: 2.0}, 1: {1: 12.0, 2: 6.0, 3: 4.0}, 2: {1: 12.0, 2: 6.0, 3: 4.0}}


def _support(gsk, kind, dim, rng):
    if kind == "point":
        return None
    if kind == "block":
        return gsk.default_support_py([1.0] * dim, rng)
    side = {1: 130, 2: 12, 3: 6}[dim]                     # 130, 144, 216 points: more than the local path's 125
    ax = (np.arange(side) + 0.5) / side - 0.5
    return [g.ravel() for g in np.meshgrid(*([ax] * dim), indexing="ij")]


def global_spec(gsk, n, est, deg, dim, vk, nugget, sup, grid=None):
    grid = GRID[dim] if grid is None else grid
    rng = RANGE[vk][dim]
    coords, vals = gsk.synth.make_samples(500 + dim, n, grid, seed_extra=n * 16 + 4 * est + deg)
    origin = None
    if dim == 1:   # n of 2n lattice points: uniform draws on a line put pairs ~L/n² apart (near-singular without nugget);
        cells = np.random.default_rng(n).permutation(2 * n)[:n]   # centred on 0, where coordinates round least
        coords = [(cells + 0.5) * (grid[0] / (2 * n)) - grid[0] / 2]
        origin = (-grid[0] / 2,)
    return gsk.ProblemSpec(coords=coords, values=vals, grid_dims=grid, grid_origin=origin, support=_support(gsk, sup, dim, rng),
                           vario_kind=vk, vario_range=rng, vario_sill=SILL, vario_nugget=nugget, estimator=est,
                           uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=0)


def check_reference(spec, mean, var, rows, vacuity=True):
    """GPU outputs at ``rows`` of the slab against the extended reference; returns the largest error/bound ratios."""
    ref = XR.reference(spec, rows, gram=True)
    tm, tv = ref.tolerances(C_FACTOR)
    if vacuity and spec.params["vario_kind"] != XR.GAUSSIAN:
        assert tm.max() <= 1e-10 * max(1.0, np.abs(spec.values).max()), tm.max()
        assert tv.max() <= 1e-10 * spec.params["vario_sill"], tv.max()
    em, ev = np.abs(mean - ref.mean), np.abs(var - ref.var)
    bad = np.flatnonzero((em > tm) | (ev > tv))
    assert bad.size == 0, (f"{bad.size} targets off the bound, e.g. row {rows[bad[0]]}: mean {mean[bad[0]]!r} vs "
                           f"{ref.mean[bad[0]]!r} (tol {tm[bad[0]]:.2e}), var {var[bad[0]]!r} vs {ref.var[bad[0]]!r} "
                           f"(tol {tv[bad[0]]:.2e})")
    return float((em / tm).max()), float((ev / tv).max())


def _oracle_parity(spec, g, o):
    mean, var, nn, _ = g
    om, ov, onn, _ = o
    assert np.array_equal(nn, onn)
    loose = spec.params["vario_kind"] == XR.GAUSSIAN or spec.params["uk_degree"] == 2
    assert_parity(mean, var, om, ov, scale=max(1.0, np.abs(spec.values).max()), sill=spec.params["vario_sill"],
                  **(dict(atol_mean=2e-7, atol_var=2e-7) if loose else {}))


@pytest.mark.parametrize("n,est,deg,dim,vk,nugget,sup", DESIGN,
                         ids=[f"n{c[0]}-e{c[1]}{c[2]}-d{c[3]}-v{c[4]}-g{c[5]}-{c[6]}" for c in DESIGN])
def test_global_vs_oracle_and_extended_reference(gsk, ctx, oracle, n, est, deg, dim, vk, nugget, sup):
    spec = global_spec(gsk, n, est, deg, dim, vk, nugget, sup)
    g = ctx.krige(spec, want_neighbors=True)
    _oracle_parity(spec, g, oracle.krige(spec, want_neighbors=True))
    check_reference(spec, g[0], g[1], np.arange(spec.n_targets))


def test_global_uk_degree_0_is_ordinary_kriging(gsk, ctx):
    """UK with the constant monomial only is Ordinary Kriging: same system, same f₀ = 1, bit for bit."""
    for dim, vk, sup in ((1, 2, "point"), (2, 1, "block"), (3, 0, "big")):
        spec = global_spec(gsk, 129, 1, 0, dim, vk, 0.06, sup)
        ok = ctx.krige(spec)
        uk0 = ctx.krige(gsk.ProblemSpec(**_kw(spec, estimator=2, uk_degree=0)))
        assert np.array_equal(ok[0], uk0[0]) and np.array_equal(ok[1], uk0[1])


def _kw(spec, **over):
    p = dict(spec.params)
    p.update(over)
    return dict(coords=spec.coords, values=spec.values, grid_dims=spec.grid_dims, grid_origin=spec.grid_origin,
                grid_spacing=spec.grid_spacing, support=spec.support, **p)


@pytest.mark.parametrize("est", [0, 1])
@pytest.mark.parametrize("dim,vk", [(1, 2), (2, 1), (3, 2)])
def test_global_single_sample_known_answer(gsk, ctx, oracle, est, dim, vk):
    """n = 1: the factor is 1×1 and 127 padded identity rows (np = 128), the dual refinement runs its padded branch.
    Simple Kriging: mean μ + (b/sill)(z − μ), variance sill − b²/sill; Ordinary Kriging: mean z, variance 2(sill − b)
    before the clamp — with b the block-support average of the covariance, from the extended reference's assembly."""
    spec = global_spec(gsk, 1, est, 0, dim, vk, 0.06, "block")
    mean, var = ctx.krige(spec)
    rows = np.arange(spec.n_targets)
    K, R, ZT, _, _, _, _, _ = XR.assemble(spec, rows)
    b, z, mu, s = R[:, 0], XR.LD(spec.values[0]), XR.LD(spec.params["sk_mean"]), XR.LD(SILL)
    if est == 0:
        want_m, want_v = mu + (b / s) * (z - mu), s - b * b / s
    else:
        want_m, want_v = np.full(len(rows), z), 2 * (s - b)
    want_m, want_v = want_m.astype(np.float64), np.sqrt(np.maximum(want_v.astype(np.float64), 0.0)) ** 2
    ref = XR.reference(spec, rows, gram=True)
    tm, tv = ref.tolerances(C_FACTOR)
    assert np.all(np.abs(ref.mean - want_m) <= tm) and np.all(np.abs(ref.var - want_v) <= tv)
    assert np.all(np.abs(mean - want_m) <= tm) and np.all(np.abs(var - want_v) <= tv)
    om, ov = oracle.krige(spec)
    assert_parity(mean, var, om, ov, scale=max(1.0, abs(spec.values[0])), sill=SILL)


def _edge_rows(count, batch, rng):
    edges = [0] + list(range(batch, count, batch)) + [count]
    near = np.concatenate([np.arange(e - 4, e + 4) for e in edges])
    near = near[(near >= 0) & (near < count)]
    return np.unique(np.concatenate([near, rng.choice(count, 1000, replace=False)]))


@pytest.mark.parametrize("est,deg,n", [(0, 0, 129), (2, 1, 200), (2, 2, 257)])
def test_global_slab_over_three_batches(gsk, ctx, oracle, est, deg, n):
    """A slab of 80 001 targets starting at an odd offset: batch = 32 768 targets for np <= 7 680 (global.cu), so the
    GEMM loop runs three batches and the last is partial. Whole slab against the oracle; every target within 4 of a
    batch edge and 1 000 random ones against the extended reference; the same targets as separate smaller slabs (one
    batch each) bit for bit."""
    spec = global_spec(gsk, n, est, deg, 2, 2, 0.0, "block", grid=(300, 300))
    first, count, batch = 1001, 80_001, 32_768
    slab = spec.with_slab(first, count)
    g = ctx.krige(slab, want_neighbors=True)
    _oracle_parity(slab, g, oracle.krige(slab, want_neighbors=True))
    rows = _edge_rows(count, batch, np.random.default_rng(n))
    check_reference(slab, g[0][rows], g[1][rows], rows)
    cuts = [0, 9_999, 32_770, 60_001, count]
    for a, b in zip(cuts[:-1], cuts[1:]):
        m, v = ctx.krige(spec.with_slab(first + a, b - a))
        assert np.array_equal(m, g[0][a:b]) and np.array_equal(v, g[1][a:b])


def test_global_traversal_order_over_batches(gsk, ctx):
    """UK degree 1 through a traversal order of the 90 000-target grid (three batches): out[j] is the linear result at
    order[j], bit for bit."""
    spec = global_spec(gsk, 200, 2, 1, 2, 1, 0.06, "block", grid=(300, 300))
    lin = ctx.krige(spec)
    order = np.random.default_rng(3).permutation(spec.n_targets)
    import copy
    sp = copy.copy(spec)
    sp.target_order = order
    got = ctx.krige(sp)
    assert np.array_equal(got[0], lin[0][order]) and np.array_equal(got[1], lin[1][order])
