"""Extended-precision reference of the Kriging prediction, with a first-order rounding bound per target.

TEST INFRASTRUCTURE ONLY. Every target's system is assembled in ``np.longdouble`` from the exact float64 inputs the
library receives (sample coordinates and values, support offsets, the target centres of ``ProblemSpec.target_centers``)
and solved by partial-pivot LU written in numpy (LAPACK has no long-double path). Neighbour lists are an input: they
come from the C oracle, which the suite pins bit-exact to the GPU's; this module does no search of its own.

For a target with neighbour set N (all samples on the global path), m = |N| + c rows (c drift terms):

    K = [[C, F], [Fᵀ, 0]]   C_ij = sill − γ(‖x_i − x_j‖),  F_it = f_t(x_i)
    r = [b; f₀]             b_i = sill − mean_s γ(‖t + δ_s − x_i‖),  f₀ = f(t)
    z̃ = [z − μ_SK or z; 0]
    λ̃ = K⁻¹ r,  w̃ = K⁻¹ z̃,  mean = z̃ᵀλ̃ (+ μ_SK),  var = sill − rᵀλ̃ (then the library's clamp / sqrt round trip)

Sensitivities (first-order change when every entry of K, r and z moves by at most one unit roundoff u, relatively):

    mean = z̃ᵀK⁻¹r:  d mean = dz̃ᵀλ̃ + w̃ᵀdr − w̃ᵀdK λ̃     →  Bμ = |λ|ᵀ|z̃| + |w̃|ᵀ(WR + WK|λ̃|)
    q = rᵀK⁻¹r:      dq = 2λ̃ᵀdr − λ̃ᵀdK λ̃                →  Bσ = 2|λ̃|ᵀWR + |λ̃|ᵀWK|λ̃|

The entries themselves are functions of coordinates, and forming a distance rounds too: a sample pair's d² carries
≲ (dim + 1)u relatively and the square root adds u/2, so h moves by ≲ a·u·h with a = (dim + 2)/2; a target's support point t + δ_s is rounded to float64 before the
difference, by e_s = ‖fl(t + δ_s) − (t + δ_s)‖ (computed exactly here; ≤ u‖t + δ_s‖, zero for point support), so h
moves by ≲ e_s + a·u·h. An entry C(h) then moves by u times

    WK_ij = |C_ij| + a·h_ij·|C'(h_ij)|,      WR_i = mean_s (|C(h_is)| + |C'(h_is)|·(e_s/u + a·h_is))

(|F|, |f₀| for the drift rows), and Bμ, Bσ use WK, WR where the plain form has |K|, |r|. The derivative term matters for
the Gaussian model: there h|C'|/C = 6(h/r)² grows with the distance, and ‖t‖/h is large where the coordinates are.

A backward-stable solver in float64 lands within a small multiple of (m + q)·u·B of the reference (q support points
per target: b is a q-term average). The tests state their constant next to the comparison.

The global path does not solve K: it forms y = L⁻¹b with an EXPLICIT inverse X = L⁻¹ of the Cholesky factor C = LLᵀ and
evaluates the variance in Gram form, var = sill − ‖ỹ‖² − 2f₀ᵀν with ỹ = y − Y_F ν = Lᵀλ, Y_F = X F, ν = λ̃[k:]. An
explicitly inverted triangle carries a forward error |δX| ≲ n·u·|X||L||X| (Higham, ASNA §14.2), so y and Y_F move by
|δy| ≲ n·u·M|b| and |δY_F| ≲ n·u·M|F| with M = |X||L||X|. The variance is stationary in everything but y and Y_F along
ỹ: dq = 2ỹᵀδy − 2ỹᵀδY_F ν, hence ``gram=True`` adds

    Bσ += 2|ỹ|ᵀ M (|b| + |F||ν|)            (for Simple Kriging: 2|y|ᵀ|L⁻¹||L||L⁻¹||b|).

The mean of the global path uses dual weights refined against the assembled system, so Bμ needs no such term.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from numpy_twin import EXPONENTIAL, GAUSSIAN, ORDINARY, SIMPLE, SPHERICAL, UNIVERSAL, uk_exponents, variogram

LD = np.longdouble
U = 2.0 ** -53
# 80-bit extended on x86-64, binary128 on aarch64; a platform whose long double is plain double would compare double
# to double and hide exactly the errors this reference is for
assert np.finfo(LD).nmant > np.finfo(np.float64).nmant, "np.longdouble is no wider than float64 on this platform"

__all__ = ["LD", "U", "Reference", "assemble", "reference", "lu_factor", "lu_solve", "GAUSSIAN", "SPHERICAL", "EXPONENTIAL",
           "SIMPLE", "ORDINARY", "UNIVERSAL"]


def lu_factor(A):
    """Partial-pivot LU of a stack of matrices A (B, m, m): returns (LU packed, row permutation (B, m))."""
    A = np.array(A, dtype=LD)
    nb, m, _ = A.shape
    perm = np.tile(np.arange(m), (nb, 1))
    bi = np.arange(nb)
    for j in range(m):
        p = j + np.argmax(np.abs(A[:, j:, j]), axis=1)
        row = A[bi, j].copy()
        A[bi, j] = A[bi, p]
        A[bi, p] = row
        pj = perm[bi, j].copy()
        perm[bi, j] = perm[bi, p]
        perm[bi, p] = pj
        A[:, j + 1:, j] /= A[:, j, j][:, None]
        A[:, j + 1:, j + 1:] -= A[:, j + 1:, j][:, :, None] * A[:, j, j + 1:][:, None, :]
    return A, perm


def lu_solve(F, perm, R):
    """Solve with the factor of :func:`lu_factor` for R (B, m, nrhs)."""
    X = np.array(R, dtype=LD)[np.arange(F.shape[0])[:, None], perm]
    m = F.shape[1]
    for j in range(m):
        X[:, j + 1:] -= F[:, j + 1:, j][:, :, None] * X[:, j][:, None, :]
    for j in range(m - 1, -1, -1):
        X[:, j] /= F[:, j, j][:, None]
        X[:, :j] -= F[:, :j, j][:, :, None] * X[:, j][:, None, :]
    return X


def _cholesky(C):
    """Lower Cholesky factor of one SPD matrix in long double."""
    C = np.array(C, dtype=LD)
    n = C.shape[0]
    L = np.zeros_like(C)
    for j in range(n):
        d = C[j, j] - np.dot(L[j, :j], L[j, :j])
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (C[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return L


def _tri_inv_lower(L):
    n = L.shape[0]
    X = np.zeros_like(L)
    eye = np.eye(n, dtype=LD)
    for i in range(n):
        X[i] = (eye[i] - L[i, :i] @ X[:i]) / L[i, i]
    return X


@dataclass
class Reference:
    mean: np.ndarray   # float64, rounded from the long-double solution
    var: np.ndarray    # float64, after the library's clamp / sqrt round trip (spec flags)
    bmu: np.ndarray    # Bμ per target (float64)
    bsig: np.ndarray   # Bσ per target (float64)
    m: np.ndarray      # system size per target
    q: int             # support points per target

    roundtrip: bool = True

    def tolerances(self, c_factor):
        """|gpu − ref| ≤ c·u·B + 2u·|ref| with c = c_factor·(m + q): the last term is the rounding of the reference
        itself to float64 and of the library's final add (μ_SK + …, sill − …). With the sqrt round trip each side's
        variance goes through fl(fl(√s)²) = s(1 + θ), |θ| ≤ 3u, once: 6u·|ref| more."""
        c = c_factor * (self.m + self.q)
        return (c * U * self.bmu + 2 * U * np.abs(self.mean),
                c * U * self.bsig + (8 if self.roundtrip else 2) * U * np.abs(self.var))


def _vario(p):
    return dict(kind=p["vario_kind"], rng=p["vario_range"], sill=p["vario_sill"], nugget=p["vario_nugget"],
                eps=p["gaussian_nugget_eps"])


def _cov(v, h):
    return v["sill"] - variogram(v["kind"], h, v["rng"], v["sill"], v["nugget"], v["eps"])


def _drift(p, dim):
    if p["estimator"] == SIMPLE:
        return np.zeros((0, dim), dtype=np.int64)
    if p["estimator"] == ORDINARY:
        return np.zeros((1, dim), dtype=np.int64)
    return uk_exponents(p["uk_degree"], dim)


def _monomials(exps, x):
    """x: (..., dim) long double → (..., c)"""
    out = np.ones(x.shape[:-1] + (len(exps),), dtype=LD)
    for t, e in enumerate(exps):
        for d, a in enumerate(e):
            for _ in range(int(a)):
                out[..., t] = out[..., t] * x[..., d]
    return out


def _dcov(v, h):
    """|dC/dh| for h > 0 (float64: it only scales the bound)."""
    h = np.asarray(h, dtype=np.float64)
    r = v["rng"]
    if v["kind"] == GAUSSIAN:
        cs = v["sill"] - v["nugget"] - v["eps"]
        return cs * 6.0 * h / (r * r) * np.exp(-3.0 * (h / r) ** 2)
    cs = v["sill"] - v["nugget"]
    if v["kind"] == SPHERICAL:
        t = h / r
        return np.where(t < 1.0, cs * 1.5 * (1.0 - t * t) / r, 0.0)
    return cs * 3.0 / r * np.exp(-3.0 * h / r)


def _rhs_b(v, X, T, S, a):
    """b (..., k) and its entry weight (module docstring): X (..., k, dim) sample coords, T (..., dim) target centres,
    S (q, dim) support offsets, a = (dim + 2)/2."""
    acc = np.zeros(X.shape[:-1], dtype=LD)
    wt = np.zeros(X.shape[:-1], dtype=np.float64)
    for s in S:
        u = T + s
        d = u[..., None, :] - X
        h = np.sqrt(np.sum(d * d, axis=-1))
        g = variogram(v["kind"], h, v["rng"], v["sill"], v["nugget"], v["eps"])
        acc = acc + g
        # the rounding of t + δ_s to float64, exactly: zero for point support and for sums that fit in 53 bits
        e = np.asarray(u.astype(np.float64).astype(LD) - u, dtype=np.float64)
        en = np.sqrt(np.sum(e * e, axis=-1))[..., None] / U
        wt = wt + np.abs(np.asarray(v["sill"] - g, dtype=np.float64)) + np.where(
            h > 0, _dcov(v, h) * (en + a * np.asarray(h, dtype=np.float64)), 0.0)
    return v["sill"] - acc / LD(len(S)), wt / len(S)


def assemble(spec, rows, idx=None, nneigh=None):
    """The long-double systems of the targets ``rows`` (positions within ``spec``'s slab): returns
    (K, R, ZT, nn, c, μ₀, WK, WR) with WK, WR the entry weights of the bound (float64, shapes of K and R).

    Global path (``max_neighbors == 0``): K is (1, m, m) with every sample, R (T, m), ZT (1, m). Local path: ``idx`` /
    ``nneigh`` are the C oracle's neighbour lists of the slab (``idx[j, :nneigh[j]]``); K is (T, m, m), R and ZT (T, m),
    each system padded with identity rows to the largest m (block diagonal: the padding leaves the solution, the
    sensitivities and the bound unchanged)."""
    p = spec.params
    v = _vario(p)
    rows = np.asarray(rows, dtype=np.int64)
    first, count = spec.slab
    ctr = np.stack(spec.target_centers(first, count), axis=1)[rows].astype(LD)
    S = np.stack(spec.support, axis=1).astype(LD)
    XS = np.stack(spec.coords, axis=1).astype(LD)
    Z = spec.values.astype(LD)
    exps = _drift(p, spec.dim)
    c = len(exps)
    mu0 = LD(p["sk_mean"]) if p["estimator"] == SIMPLE else LD(0)
    T = len(rows)
    a = (spec.dim + 2) / 2   # relative rounding of a distance, in units of u (module docstring)
    if p["max_neighbors"] == 0:
        n = XS.shape[0]
        m = n + c
        K = np.zeros((1, m, m), dtype=LD)
        dX = XS[:, None, :] - XS[None, :, :]
        h = np.sqrt(np.sum(dX * dX, axis=-1))
        K[0, :n, :n] = _cov(v, h)
        F = _monomials(exps, XS)
        K[0, :n, n:] = F
        K[0, n:, :n] = F.T
        R = np.zeros((T, m), dtype=LD)
        WR = np.zeros((T, m))
        R[:, :n], WR[:, :n] = _rhs_b(v, XS[None, :, :], ctr, S, a)
        R[:, n:] = _monomials(exps, ctr)
        WR[:, n:] = np.abs(R[:, n:]).astype(np.float64)
        WK = np.abs(K).astype(np.float64)
        WK[0, :n, :n] += np.where(h > 0, a * np.asarray(h, dtype=np.float64) * _dcov(v, h), 0.0)
        ZT = np.concatenate([Z - mu0, np.zeros(c, dtype=LD)])[None]
        return K, R, ZT, None, c, mu0, WK, WR
    nn = np.asarray(nneigh)[rows]
    assert np.all(nn > 0), "every target of the reference needs a neighbour"
    mmax = int(nn.max()) + c
    K = np.zeros((T, mmax, mmax), dtype=LD)
    R = np.zeros((T, mmax), dtype=LD)
    ZT = np.zeros((T, mmax), dtype=LD)
    WK = np.zeros((T, mmax, mmax))
    WR = np.zeros((T, mmax))
    for j in range(T):
        k = int(nn[j])
        nb = np.asarray(idx)[rows[j], :k]
        xs = XS[nb]
        d = xs[:, None, :] - xs[None, :, :]
        h = np.sqrt(np.sum(d * d, axis=-1))
        K[j, :k, :k] = _cov(v, h)
        WK[j, :k, :k] = np.where(h > 0, a * np.asarray(h, dtype=np.float64) * _dcov(v, h), 0.0)
        F = _monomials(exps, xs)
        K[j, :k, k:k + c] = F
        K[j, k:k + c, :k] = F.T
        for i in range(k + c, mmax):
            K[j, i, i] = 1
        R[j, :k], WR[j, :k] = _rhs_b(v, xs, ctr[j], S, a)
        R[j, k:k + c] = _monomials(exps, ctr[j])
        WR[j, k:k + c] = np.abs(R[j, k:k + c]).astype(np.float64)
        ZT[j, :k] = Z[nb] - mu0
    WK += np.abs(K).astype(np.float64)
    return K, R, ZT, nn, c, mu0, WK, WR


def reference(spec, rows, idx=None, nneigh=None, gram=False):
    """Long-double prediction and bounds for the targets ``rows`` (positions within ``spec``'s slab); arguments as
    :func:`assemble`. ``gram=True`` (global path) adds the variance term of the explicit-inverse Gram form."""
    K, R, ZT, nn, c, mu0, WK, WR = assemble(spec, rows, idx, nneigh)
    T, m = R.shape
    q = spec.support[0].shape[0]
    fac, perm = lu_factor(K)
    if nn is None:
        n = m - c
        sol = lu_solve(fac, perm, np.concatenate([R.T, ZT.T], axis=1)[None])[0]
        lam_t, w_t = sol[:, :T].T, np.broadcast_to(sol[:, T], (T, m))
        lam = lam_t[:, :n]
        ZT = np.broadcast_to(ZT, (T, m))
        K_abs_lam = np.abs(lam_t).astype(np.float64) @ WK[0].T
        sizes = np.full(T, m)
    else:
        sol = lu_solve(fac, perm, np.stack([R, ZT], axis=2))
        lam_t, w_t = sol[:, :, 0], sol[:, :, 1]
        lam = np.where(np.arange(m)[None, :] < nn[:, None], lam_t, 0)
        K_abs_lam = np.einsum("tij,tj->ti", WK, np.abs(lam_t).astype(np.float64))
        sizes = nn + c
    k = lam.shape[1]
    mean = np.sum(lam * ZT[:, :k], axis=1) + mu0
    qv = np.sum(R * lam_t, axis=1)
    aw, al = np.abs(w_t).astype(np.float64), np.abs(lam_t).astype(np.float64)
    bmu = (aw * (WR + K_abs_lam)).sum(1) + (np.abs(lam) * np.abs(ZT[:, :k])).sum(1).astype(np.float64)
    bsig = 2 * (al * WR).sum(1) + (al * K_abs_lam).sum(1)
    if gram:
        assert nn is None, "the Gram-form term belongs to the global path"
        n = m - c
        L = _cholesky(K[0, :n, :n])
        Xa = np.abs(_tri_inv_lower(L)).astype(np.float64)
        M = Xa @ (np.abs(L).astype(np.float64) @ Xa)                                # |L⁻¹||L||L⁻¹|
        ytil = np.abs(lam @ L).astype(np.float64)                                   # ỹ = Lᵀλ = L⁻¹(b − Fν)
        F = np.abs(K[0, :n, n:]).astype(np.float64)
        src = np.abs(R[:, :n]).astype(np.float64) + np.abs(lam_t[:, n:]).astype(np.float64) @ F.T   # |b| + |F||ν|
        bsig = bsig + 2 * np.sum(ytil * (src @ M.T), axis=1)
    var = np.asarray(LD(spec.params["vario_sill"]) - qv, dtype=np.float64)
    flags = spec.params["flags"]
    if flags & 1:                                                                   # GSK_FLAG_CLAMP_VARIANCE
        var = np.where((var > 0) | np.isnan(var), var, 0.0)
    if flags & 2:                                                                   # GSK_FLAG_SQRT_ROUNDTRIP
        var = np.sqrt(var) ** 2
    return Reference(np.asarray(mean, dtype=np.float64), var, np.asarray(bmu, dtype=np.float64),
                     np.asarray(bsig, dtype=np.float64), np.asarray(sizes), q, bool(flags & 2))
