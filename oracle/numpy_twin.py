"""Second, independent CPU restatement of the Kriging path (numpy + LAPACK via scipy).

TEST INFRASTRUCTURE ONLY. Where gsk_oracle.c uses hand-written partial-pivot LU / Cholesky,
this twin calls the LAPACK routines Julia's LinearAlgebra dispatches to for the reference:
``bunchkaufman(Symmetric(LHS), check=false)`` → dsytrf/dsytrs (upper) for Ordinary/Universal
Kriging and ``cholesky(Symmetric(LHS), check=false)`` → dpotrf/dpotrs for Simple Kriging
(GeoStatsModels 0.2 [3P], SURVEY §8a a13/V3). It pins how much the factorisation choice moves
the result (tests/test_oracle_twin.py) and generates tests/golden/*.npz.

Follows ref src/estimation/krig.jl:166-234 for control flow. Pure brute-force search; small cases only.
"""
from __future__ import annotations

import numpy as np
from scipy.linalg import lapack

GAUSSIAN, SPHERICAL, EXPONENTIAL = 0, 1, 2
SIMPLE, ORDINARY, UNIVERSAL = 0, 1, 2


def variogram(kind, h, rng, sill, nugget, eps=1e-6):
    """γ(h) in the precision of h: float64, or np.longdouble for the extended reference (extended_ref.py). The model
    constants are converted first, so that sill − nugget − ε is formed in that precision too (in float64 it rounds,
    and the rounding would reach every covariance sill − γ as a constant offset)."""
    h = np.asarray(h)
    h = h.astype(np.result_type(h.dtype, np.float64), copy=False)
    f = h.dtype.type
    rng, sill, nugget, eps = f(rng), f(sill), f(nugget), f(eps)
    if kind == GAUSSIAN:
        n = nugget + eps
        g = (sill - n) * (1.0 - np.exp(-3.0 * (h / rng) ** 2))
    elif kind == SPHERICAL:
        n = nugget
        t = h / rng
        g = np.where(h < rng, (sill - n) * (1.5 * t - 0.5 * t ** 3), (sill - n))
    elif kind == EXPONENTIAL:
        n = nugget
        g = (sill - n) * (1.0 - np.exp(-3.0 * (h / rng)))
    else:
        raise ValueError(kind)
    return g + np.where(h > 0, n, 0.0)


def uk_exponents(degree, dim):
    """GeoStatsModels UKexps: multiexponents per degree, stable sort by descending max exponent."""
    def multiexp(m, d):  # descending lexicographic compositions of d into m parts
        if m == 1:
            return [[d]]
        out = []
        for a in range(d, -1, -1):
            out += [[a] + r for r in multiexp(m - 1, d - a)]
        return out
    cols = []
    for d in range(degree + 1):
        cols += multiexp(dim, d)
    mx = [max(c) for c in cols]
    order = sorted(range(len(cols)), key=lambda i: -mx[i])  # sorted() is stable
    return np.array([cols[i] for i in order], dtype=np.int64)


def knn(xyz, center, k):
    diff = center[None, :] - xyz
    d2 = diff[:, 0] * diff[:, 0]
    for d in range(1, xyz.shape[1]):
        d2 = d2 + diff[:, d] * diff[:, d]
    order = np.lexsort((np.arange(len(d2)), d2))[:k]
    return order, d2[order]


def _fit(xyz, est, vario, exps):
    k = xyz.shape[0]
    c = 0 if est == SIMPLE else (1 if est == ORDINARY else len(exps))
    m = k + c
    A = np.zeros((m, m))
    diff = xyz[:, None, :] - xyz[None, :, :]
    d2 = diff[..., 0] * diff[..., 0]
    for d in range(1, xyz.shape[1]):
        d2 = d2 + diff[..., d] * diff[..., d]
    A[:k, :k] = vario["sill"] - variogram(vario["kind"], np.sqrt(d2), vario["range"], vario["sill"], vario["nugget"],
                                          vario["eps"])
    if est == ORDINARY:
        A[k, :k] = 1.0
        A[:k, k] = 1.0
    elif est == UNIVERSAL:
        F = np.stack([np.prod(xyz ** e[None, :], axis=1) for e in exps], axis=1)
        A[:k, k:] = F
        A[k:, :k] = F.T
    if est == SIMPLE:
        fac, info = lapack.dpotrf(A, lower=0)
        return ("chol", fac, None, m, k)
    ldu, ipiv, info = lapack.dsytrf(A, lower=0)
    return ("bk", ldu, ipiv, m, k)


def _solve(fit, b):
    kind, fac, ipiv, m, k = fit
    if kind == "chol":
        x, info = lapack.dpotrs(fac, b, lower=0)
    else:
        x, info = lapack.dsytrs(fac, ipiv, b, lower=0)
    return x


def krige(coords, values, centers, *, support, vario, est, sk_mean=0.0, degree=0, k=0, radius=None,
          min_neighbors=1, clamp=True, roundtrip=True):
    """coords: (n,dim); centers: (T,dim); support: (q,dim) offsets. Returns mean, var, nneigh, idx."""
    coords = np.asarray(coords, dtype=np.float64)
    values = np.asarray(values, dtype=np.float64)
    centers = np.asarray(centers, dtype=np.float64)
    support = np.asarray(support, dtype=np.float64)
    n, dim = coords.shape
    T = centers.shape[0]
    exps = uk_exponents(degree, dim) if est == UNIVERSAL else None
    mean = np.full(T, np.nan)
    var = np.full(T, np.nan)
    kk = k if k > 0 else n
    nneigh = np.zeros(T, dtype=np.int32)
    idx = np.full((T, kk), -1, dtype=np.int32)
    gfit = _fit(coords, est, vario, exps) if k == 0 else None
    for t in range(T):
        ctr = centers[t]
        if k == 0:
            nb = np.arange(n)
        else:
            nb, d2 = knn(coords, ctr, k)
            if radius is not None:
                nb = nb[np.sqrt(d2) <= radius]
        nn = len(nb)
        nneigh[t] = nn
        idx[t, :nn] = nb
        if nn < min_neighbors or nn == 0:
            continue
        xyz = coords[nb]
        fit = gfit if k == 0 else _fit(xyz, est, vario, exps)
        m = fit[3]
        # RHS: mean of γ over the support points of the target geometry
        acc = np.zeros(nn)
        for s in range(support.shape[0]):
            u = ctr + support[s]
            diff = u[None, :] - xyz
            d2s = diff[:, 0] * diff[:, 0]
            for d in range(1, dim):
                d2s = d2s + diff[:, d] * diff[:, d]
            acc = acc + variogram(vario["kind"], np.sqrt(d2s), vario["range"], vario["sill"], vario["nugget"], vario["eps"])
        b = np.zeros(m)
        b[:nn] = vario["sill"] - acc / support.shape[0]
        if est == ORDINARY:
            b[nn] = 1.0
        elif est == UNIVERSAL:
            b[nn:] = [np.prod(ctr ** e) for e in exps]
        s = _solve(fit, b)
        lam = s[:nn]
        z = values[nb]
        if est == SIMPLE:
            mu = sk_mean + float(np.sum(lam * (z - sk_mean)))
        else:
            mu = float(np.sum(lam * z))
        s2 = vario["sill"] - (float(np.dot(b[:nn], lam)) + float(np.dot(b[nn:], s[nn:])))
        if clamp and not np.isnan(s2):
            s2 = max(0.0, s2)
        if roundtrip:
            s2 = np.sqrt(s2) ** 2
        mean[t], var[t] = mu, s2
    return mean, var, nneigh, idx
