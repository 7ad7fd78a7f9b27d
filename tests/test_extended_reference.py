"""The extended-precision reference (oracle/extended_ref.py) itself, without a GPU: it agrees with the committed LAPACK
golden vectors within the bound it derives, with a 40-digit mpmath solve, and its bound measures something real."""
import numpy as np
import pytest

from _cases import CASES, GOLDEN, build_case

import extended_ref as XR


def test_long_double_is_wider_than_double():
    assert np.finfo(XR.LD).eps < np.finfo(np.float64).eps


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_reference_matches_lapack_golden_vectors(gsk, case):
    """The golden vectors come from dsytrf / dpotrf in float64 (numpy_twin.py), a backward-stable solve of the same
    systems: each must lie within c·u·B + 2u·|ref| of the reference, c = 4(m + q)."""
    name = case[0]
    spec = build_case(case)
    gm, gv, nn = GOLDEN[f"{name}/mean"], GOLDEN[f"{name}/var"], GOLDEN[f"{name}/nn"]
    rows = np.flatnonzero(~np.isnan(gm))
    idx = GOLDEN[f"{name}/idx"] if spec.params["max_neighbors"] > 0 else None
    ref = XR.reference(spec, rows, idx, nn if idx is not None else None)
    tm, tv = ref.tolerances(4)
    assert np.all(np.abs(gm[rows] - ref.mean) <= tm)
    assert np.all(np.abs(gv[rows] - ref.var) <= tv)


def test_reference_matches_mpmath_on_a_gaussian_global_system(gsk):
    """30 samples, global Ordinary Kriging with a Gaussian variogram (the worst-conditioned family): the same systems
    assembled and solved with mpmath at 40 digits; the long-double mean and variance agree to 1e-15 relative."""
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.dps = 40
    coords, vals = gsk.synth.make_samples(900, 30, (10, 10))
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(10, 10), support=gsk.default_support_py([1.0, 1.0], 4.0),
                           vario_kind=gsk.VARIO_GAUSSIAN, vario_range=4.0, vario_sill=1.3, max_neighbors=0)
    rows = np.arange(0, 100, 9)
    ref = XR.reference(spec, rows)
    mp = mpmath.mpf
    X = [[mp(float(c[i])) for c in coords] for i in range(30)]
    sill, a, nug = mp(1.3), mp(4.0), mp(1e-6)

    def cov(p, q):
        h2 = sum((pi - qi) ** 2 for pi, qi in zip(p, q))
        return sill if h2 == 0 else (sill - nug) * mpmath.exp(-3 * h2 / a ** 2)

    K = mpmath.matrix(31, 31)
    for i in range(30):
        for j in range(30):
            K[i, j] = cov(X[i], X[j])
        K[i, 30] = K[30, i] = 1
    ctr = np.stack(spec.target_centers(), 1)[rows]
    sup = np.stack(spec.support, 1)
    for t, c in enumerate(ctr):
        r = mpmath.matrix(31, 1)
        for i in range(30):
            r[i] = sum(cov([mp(float(c[d])) + mp(float(s[d])) for d in range(2)], X[i]) for s in sup) / len(sup)
        r[30] = 1
        lam = mpmath.lu_solve(K, r)
        mean = sum(lam[i] * mp(float(vals[i])) for i in range(30))
        var = sill - sum(lam[i] * r[i] for i in range(31))
        assert abs(ref.mean[t] - float(mean)) <= 1e-15 * abs(float(mean))
        assert abs(ref.var[t] - float(var)) <= 1e-15 * abs(float(var))


@pytest.mark.parametrize("vk,est,deg,k", [(1, 1, 0, 0), (2, 2, 1, 0), (0, 1, 0, 0), (2, 0, 0, 12), (1, 2, 2, 20)])
def test_bound_is_first_order_sensitivity(gsk, oracle, vk, est, deg, k):
    """Perturb every entry of K, r and z by ±u relatively (random signs, K kept symmetric) and re-solve in long
    double: the outputs move by less than u·B (first order: the bound is a bound) and by more than u·B/1000 (the bound
    is not vacuous)."""
    coords, vals = gsk.synth.make_samples(901 + vk, 60, (8, 8))
    spec = gsk.ProblemSpec(coords=coords, values=vals, grid_dims=(8, 8), support=gsk.default_support_py([1.0, 1.0], 5.0),
                           vario_kind=vk, vario_range=5.0, vario_sill=1.3, vario_nugget=0.05, estimator=est,
                           uk_degree=deg, sk_mean=float(vals.mean()), max_neighbors=k)
    rows = np.arange(0, 64, 5)
    nn = idx = None
    if k:
        _, _, nn, idx = oracle.krige(spec, want_neighbors=True)
    ref = XR.reference(spec, rows, idx, nn)
    K, R, ZT, nnr, c, mu0, _, _ = XR.assemble(spec, rows, idx, nn)
    rng = np.random.default_rng(vk + 10 * est + k)
    u = XR.LD(XR.U)

    def signs(shape):
        return rng.choice([-1.0, 1.0], size=shape).astype(XR.LD)

    S = signs(K.shape)
    S = np.triu(S) + np.swapaxes(np.triu(S, 1), -1, -2)
    Kp, Rp, Zp = K * (1 + u * S), R * (1 + u * signs(R.shape)), ZT * (1 + u * signs(ZT.shape))
    sill = XR.LD(spec.params["vario_sill"])

    def solve(K, R, ZT):
        fac, perm = XR.lu_factor(K)
        if nnr is None:
            lam = XR.lu_solve(fac, perm, R.T[None])[0].T
            ZT = np.broadcast_to(ZT, R.shape)
        else:
            lam = XR.lu_solve(fac, perm, R[:, :, None])[:, :, 0]
        return np.sum(lam * ZT, 1), sill - np.sum(lam * R, 1)

    m0, v0 = solve(K, R, ZT)
    m1, v1 = solve(Kp, Rp, Zp)
    dm, dv = np.abs(m1 - m0).astype(np.float64), np.abs(v1 - v0).astype(np.float64)
    assert np.all(dm <= XR.U * ref.bmu) and np.all(dv <= XR.U * ref.bsig)
    assert dm.max() >= XR.U * ref.bmu.max() / 1000 and dv.max() >= XR.U * ref.bsig.max() / 1000
