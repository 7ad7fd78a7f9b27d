// local_solve.cuh — K3: per-target kriging system assembly + factorisation + solve + mean/variance,
// replacing `GeoStatsModels.fit(estimator, samples)` and `predictprob(krig, var, pdomain[ind])`
// inside approxsolve's loop (ref: src/estimation/krig.jl:217-226; SURVEY §8a a12-a16).
//
// Formulation (FP64 throughout). For k neighbours with covariance block C (k×k, SPD) and the
// "extra" rows E = [b; z; f_1 … f_c] (b = block-support RHS, z = values (− μ for SK), f = drift
// monomials: OK c=1 → ones, UK → UKexps order), one Cholesky sweep over the augmented matrix
//        [ C  ]           [ L ]
//        [ E  ]    →      [ Y ]      with  Y = E L^-T  (forward substitution comes for free),
// and the Schur complement  Gm = Y Yᵀ = E C⁻¹ Eᵀ  (e×e) holds every quantity kriging needs:
//   SK :  mean = μ + Gm[b,z]                     var = sill − Gm[b,b]
//   OK/UK:  ν = Gm[f,f]⁻¹ (Gm[f,b] − f₀)          (Lagrange multipliers; f₀ = drift at the target)
//           mean = Gm[b,z] − Gm[f,z]·ν            var = sill − (Gm[b,b] − Gm[f,b]·ν + f₀·ν)
// which is the reference's  s = LHS \ RHS;  μ̂ = Σλᵢzᵢ;  σ² = sill − RHS·s  solved by block
// elimination (C first, then the c×c Schur system) — no back substitution, no pivot search.
//
// Mapping: G lanes cooperate on one target (32/G targets per warp). Lane l owns rows l, l+G, …
// (R register slots, RT = R·G rows in total: KC neighbour rows padded to the panel width, then the
// extra rows, then zero padding). The factor lives column-packed in shared memory (column p keeps
// rows ≥ p rounded down to the panel alignment) and is built in place, W columns at a time:
// left-looking update from the finished columns (own entries + W broadcast entries per finished
// column → R·W independent DFMAs), then the W×W panel, whose pivots and row entries travel between
// the lanes of the group by warp shuffles. The panel loop is unrolled with static column offsets,
// so all shared-memory addressing is base + immediate.
#pragma once
#include <math.h>

#include "gsk_internal.cuh"

namespace gsk_local {

constexpr size_t GSK_SMEM_OPTIN_MAX = 232448;  // opt-in shared memory per CTA on sm_100 (227 KB)

template <int W>
__host__ __device__ constexpr int col_align() { return W >= 8 ? 8 : 4; }

// doubles stored before column p: Σ_{j<p} (RT − (j & ~(A−1)))
template <int RT, int A>
__host__ __device__ constexpr int col_off(int p) {
  return p * RT - A * A * ((p / A) * ((p / A) - 1) / 2) - A * (p / A) * (p % A);
}

// Leading dimension of the column-packed factor: column p holds rows [s_p, LD) of which [s_p, RS) are used.
// One warp per target (G = 32) updates its panels with the FP64 tensor instruction, whose operand fragments
// read 4 columns × 8 rows per half-warp: a stride ≡ 4 (mod 8) doubles spreads those over all banks. The
// 96-neighbour configuration (RS = 112) has no shared memory left for the padding.
template <int G, int RS>
__host__ __device__ constexpr int lead_dim() { return (G == 32 && RS <= 80) ? RS + 4 : RS; }

struct Layout {
  int KC;    // neighbour columns, padded to a multiple of W
  int e;     // live extra rows (2 + c)
  int EPr;   // e rounded up to a multiple of W
  int gsz;   // doubles of shared memory per target group
  int off_nb, off_gm;
};

template <int G, int R, int W, int RS, int DIM>
__host__ inline Layout make_layout(int k, int e) {
  constexpr int RT = RS, A = col_align<W>(), KCMAX = RT - W, LD = lead_dim<G, RS>();
  Layout L;
  L.KC = (k + W - 1) / W * W;
  L.e = e;
  L.EPr = (e + W - 1) / W * W;
  int o = col_off<LD, A>(KCMAX);  // factor storage (static maximum); multiple of 4 doubles
  L.off_nb = o;
  o += DIM * KCMAX;
  L.off_gm = o;
  o += L.EPr * L.EPr;
  while ((o & 15) != 4 && (o & 15) != 12) o += 4;  // spread the groups of a warp over the banks
  L.gsz = o;
  return L;
}

// 1/sqrt(d) to ~1 ulp: MUFU.RSQ64H seed (2^-22) + one cubically convergent step, 1/sqrt(d) = y(1 + e/2 + 3e²/8 + O(e³))
// with e = 1 − d·y² — a dependent chain of four FP64 operations (two Newton steps are six; the pivot of every panel
// column waits for this value)
__device__ __forceinline__ double gsk_rsqrt(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  const double e = fma(-(d * y), y, 1.0);
  return fma(y * e, fma(0.375, e, 0.5), y);
}

// sqrt(u) for u > 0 (u == 0 yields NaN, discarded by the callers' d2 > 0 select)
__device__ __forceinline__ double gsk_sqrt_pos(double u) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(u));
  // one cubically convergent step: sqrt(u) = t(1 + e/2 + 3e²/8 + O(e³)), t = u·y, e = 1 − u·y²  (|e| <= 2^-21)
  const double t = u * y;
  const double e = fma(-t, y, 1.0);
  const double q = e * fma(0.375, e, 0.5);
  return fma(t, q, t);
}

// sqrt(u) for u >= 0 with sqrt(0) = 0 and no select: the seed's high word is capped below infinity on the integer
// pipe (rsqrt(0) = +inf would give 0·inf), so u = 0 runs through the same arithmetic and yields t = 0·y = 0.
__device__ __forceinline__ double gsk_sqrt_nonneg(double u) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(u));
  y = __hiloint2double(min(__double2hiint(y), 0x7FE00000), 0);
  const double t = u * y;
  const double e = fma(-t, y, 1.0);
  const double q = e * fma(0.375, e, 0.5);
  return fma(t, q, t);
}

// exp(x) for x <= 0, branch-free (so that independent evaluations interleave): x = n·ln2 + f, |f| <= ln2/2,
// degree-12 Taylor/Horner on f (truncation 2e-17 relative), scaled by 2^n through the exponent field.
// Arguments below −700 are clamped (result ~1e-304, i.e. 0 at double precision for a covariance).
__device__ __forceinline__ double gsk_exp_neg(double x) {
  x = fmax(x, -700.0);
  const double t = fma(x, 1.4426950408889634, 6755399441055744.0);  // round(x·log2 e) in the low mantissa bits
  const int n = __double2loint(t);
  const double nd = t - 6755399441055744.0;
  double f = fma(nd, -6.93147180369123816490e-01, x);
  f = fma(nd, -1.90821492927058770002e-10, f);
  double p = 2.08767569878680989792e-09;           // 1/12!
  p = fma(p, f, 2.50521083854417187751e-08);       // 1/11!
  p = fma(p, f, 2.75573192239858906526e-07);       // 1/10!
  p = fma(p, f, 2.75573192239858906526e-06);       // 1/9!
  p = fma(p, f, 2.48015873015873015873e-05);       // 1/8!
  p = fma(p, f, 1.98412698412698412698e-04);       // 1/7!
  p = fma(p, f, 1.38888888888888888889e-03);       // 1/6!
  p = fma(p, f, 8.33333333333333333333e-03);       // 1/5!
  p = fma(p, f, 4.16666666666666666667e-02);       // 1/4!
  p = fma(p, f, 1.66666666666666666667e-01);       // 1/3!
  p = fma(p, f, 0.5);
  p = fma(p, f, 1.0);
  p = fma(p, f, 1.0);
  // scale by 2^n through the exponent field: n >= round(-700·log2 e) = -1010, so 2^n is a normal number
  return p * __hiloint2double((1023 + n) << 20, 0);
}

// D(16×8) = A(16×16, row) · B(16×8, col) + D on the FP64 tensor path (SASS DMMA). Fragment layout, g = lane/4,
// t = lane%4 (checked by scripts/dev/dmma_layout_test.cu): a[i] = A[g + 8(i&1)][t + 4(i>>1)], b[i] = B[t + 4i][g],
// d = {D[g][2t], D[g][2t+1], D[g+8][2t], D[g+8][2t+1]}.
__device__ __forceinline__ void gsk_dmma16816(double (&d)[4], const double (&a)[8], const double (&b)[4]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
      "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
      : "+d"(d[0]), "+d"(d[1]), "+d"(d[2]), "+d"(d[3])
      : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(a[4]), "d"(a[5]), "d"(a[6]), "d"(a[7]), "d"(b[0]), "d"(b[1]),
        "d"(b[2]), "d"(b[3]));
}

// D(8×8) += A(8×4, row) · B(4×8, col): the native FP64 tensor instruction (SASS DMMA.8x8x4; m16n8k16 is eight of
// them). Fragments, g = lane/4, t = lane%4: a = A[g][t], b = B[t][g], d = {D[g][2t], D[g][2t+1]}.
__device__ __forceinline__ void gsk_dmma884(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d[0]), "+d"(d[1])
               : "d"(a), "d"(b));
}

// Sign/magnitude tests on the high word run on the integer pipe instead of the FP64 pipe (DSETP), which is the
// pipe the kernels saturate. Valid for finite d >= 0; a subnormal d (distance below 1.5e-154) counts as zero —
// rsqrt.approx.ftz flushes it to zero anyway.
__device__ __forceinline__ bool gsk_is_pos(double d) { return __double2hiint(d) != 0; }
__device__ __forceinline__ bool gsk_lt_one(double d) { return __double2hiint(d) < 0x3FF00000; }

// covariance from the squared distance, fast-path math (same formulas as gsk_cov)
// UNIT: the coordinates were divided by the range beforehand, d2 is (h/r)² (spherical model only)
// NUG0: no nugget (sill == cs): C(0) then equals the model's own limit at h -> 0 and the d2 == 0 select goes away
// INR (spherical): the caller guarantees h < range, the range select is dropped
template <int VK, bool UNIT = false, bool NUG0 = false, bool INR = false>
__device__ __forceinline__ double cov_fast(const GskVario &v, double d2) {
  double c;
  if (VK == GSK_VARIO_GAUSSIAN) {
    c = v.cs * gsk_exp_neg(d2 * v.m3ir2);
  } else if (VK == GSK_VARIO_SPHERICAL) {
    const double u = UNIT ? d2 : d2 * v.inv_r2;
    const double t = NUG0 ? gsk_sqrt_nonneg(u) : gsk_sqrt_pos(u);
    c = fma(t, fma(v.hcs, u, v.m15cs), v.cs);  // cs(1 − 1.5t + 0.5t³)
    if (!INR) c = gsk_lt_one(u) ? c : 0.0;
  } else {
    const double h = NUG0 ? gsk_sqrt_nonneg(d2) : (gsk_is_pos(d2) ? gsk_sqrt_pos(d2) : 0.0);
    c = v.cs * gsk_exp_neg(v.m3ir * h);
  }
  if (NUG0) return c;
  return gsk_is_pos(d2) ? c : v.sill;
}

// Block-support right-hand side for the JM neighbours a lane owns:  bacc[jj] = Σ_q C(‖t + δ_q − x_jj‖).
// q is the outer loop so that the JM evaluations are independent chains. For the exponential model with a
// support that is small against the range (flag rhs_taylor, set on the host when 3·max|δ|/r <= 0.06) the
// identity exp(−3h/r) = exp(−3h₀/r)·exp(−3(h−h₀)/r), |h − h₀| <= |δ|, needs ONE exp per neighbour and a degree-8
// polynomial per support point (truncation <= 0.06⁹/9! = 3e-17 relative) instead of an exp per point.
template <int VK, int DIM, int JM, bool UNIT = false, bool NUG0 = false, bool INR = false>
__device__ __forceinline__ void rhs_block_support(const GskLocalArgs &a, const GskVario &vg, const double *sup,
                                                  const double (&tc)[3], const double (&nx)[JM], const double (&ny)[JM],
                                                  const double (&nz)[JM], double (&bacc)[JM]) {
  if (VK == GSK_VARIO_EXPONENTIAL && a.rhs_taylor) {
    double h0[JM], g[JM], zc[JM];
    const double sc = vg.m3ir;
#pragma unroll
    for (int jj = 0; jj < JM; ++jj) {
      const double dx = tc[0] - nx[jj], dy = tc[1] - ny[jj];
      double d2 = fma(dy, dy, dx * dx);
      if (DIM == 3) {
        const double dz = tc[2] - nz[jj];
        d2 = fma(dz, dz, d2);
      }
      h0[jj] = gsk_is_pos(d2) ? gsk_sqrt_pos(d2) : 0.0;
      g[jj] = 0.0;
      zc[jj] = 0.0;
    }
    for (int q = 0; q < a.nsup; ++q) {
      const double ux = tc[0] + sup[q], uy = tc[1] + sup[a.nsup + q];
      const double uz = (DIM == 3) ? tc[2] + sup[2 * a.nsup + q] : 0.0;
#pragma unroll
      for (int jj = 0; jj < JM; ++jj) {
        const double dx = ux - nx[jj], dy = uy - ny[jj];
        double d2 = fma(dy, dy, dx * dx);
        if (DIM == 3) {
          const double dz = uz - nz[jj];
          d2 = fma(dz, dz, d2);
        }
        const bool pos = gsk_is_pos(d2);
        const double h = pos ? gsk_sqrt_pos(d2) : 0.0;
        const double x = sc * (h - h0[jj]);
        double p = 2.48015873015873015873e-05;      // 1/8!
        p = fma(p, x, 1.98412698412698412698e-04);  // 1/7!
        p = fma(p, x, 1.38888888888888888889e-03);
        p = fma(p, x, 8.33333333333333333333e-03);
        p = fma(p, x, 4.16666666666666666667e-02);
        p = fma(p, x, 1.66666666666666666667e-01);
        p = fma(p, x, 0.5);
        p = fma(p, x, 1.0);
        p = fma(p, x, 1.0);
        g[jj] += pos ? p : 0.0;
        zc[jj] += pos ? 0.0 : 1.0;   // a support point exactly on the sample contributes C(0) = sill
      }
    }
#pragma unroll
    for (int jj = 0; jj < JM; ++jj) bacc[jj] = fma(vg.cs * gsk_exp_neg(sc * h0[jj]), g[jj], vg.sill * zc[jj]);
    return;
  }
#pragma unroll 3
  for (int q = 0; q < a.nsup; ++q) {
    const double ux = tc[0] + sup[q], uy = tc[1] + sup[a.nsup + q];
    const double uz = (DIM == 3) ? tc[2] + sup[2 * a.nsup + q] : 0.0;
#pragma unroll
    for (int jj = 0; jj < JM; ++jj) {  // branch-free: the JM chains interleave (invalid lanes compute on zeros)
      const double dx = ux - nx[jj], dy = uy - ny[jj];
      double d2 = fma(dy, dy, dx * dx);
      if (DIM == 3) {
        const double dz = uz - nz[jj];
        d2 = fma(dz, dz, d2);
      }
      bacc[jj] += cov_fast<VK, UNIT, NUG0, INR>(vg, d2);
    }
  }
}

// Block-support right-hand side when the support is a 3-per-axis tensor grid (GskLocalArgs::sup_tensor3): the squared
// distance from neighbour j to support point (kx, ky, kz) is sx[kx] + sy[ky] + sz[kz] with nine per-axis squares per
// neighbour, i.e. 1⅓ additions per support point instead of three subtractions and three multiply-adds. Summation
// order over q is the generic loop's (kx fastest). The Gaussian model separates completely:
// Σ_q exp(−3(sx+sy+sz)/r²) = (Σ e^{−3sx/r²})(Σ e^{−3sy/r²})(Σ e^{−3sz/r²}) — 3·DIM exponentials per neighbour.
// ax: the per-axis offsets (in range units when UNIT), tc: the target centroid (the origin when UNIT).
template <int VK, int DIM, int JM, bool UNIT = false>
__device__ __forceinline__ void rhs_tensor3(const GskLocalArgs &a, const GskVario &vg, const double (&ax)[3][3],
                                            const double (&tc)[3], const double (&nx)[JM], const double (&ny)[JM],
                                            const double (&nz)[JM], double (&bacc)[JM]) {
  const bool nug0 = (VK != GSK_VARIO_GAUSSIAN) && (vg.sill == vg.cs);  // uniform: no C(0) discontinuity to honour
#pragma unroll
  for (int jj = 0; jj < JM; ++jj) {
    double sx[3], sy[3], sz[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const double ex = (tc[0] + ax[0][i]) - nx[jj], ey = (tc[1] + ax[1][i]) - ny[jj];
      sx[i] = ex * ex;
      sy[i] = ey * ey;
      if (DIM == 3) {
        const double ez = (tc[2] + ax[2][i]) - nz[jj];
        sz[i] = ez * ez;
      } else {
        sz[i] = 0.0;
      }
    }
    if (VK == GSK_VARIO_GAUSSIAN) {
      double px = 0.0, py = 0.0, pz = 0.0;
      int zx = 0, zy = 0, zz = 0;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        px += gsk_exp_neg(sx[i] * vg.m3ir2);
        py += gsk_exp_neg(sy[i] * vg.m3ir2);
        if (DIM == 3) pz += gsk_exp_neg(sz[i] * vg.m3ir2);
        zx += gsk_is_pos(sx[i]) ? 0 : 1;
        zy += gsk_is_pos(sy[i]) ? 0 : 1;
        zz += gsk_is_pos(sz[i]) ? 0 : 1;
      }
      // support points that sit exactly on the sample contribute C(0) = sill instead of cs
      const int nzero = zx * zy * ((DIM == 3) ? zz : 1);
      const double prod = (DIM == 3) ? px * py * pz : px * py;
      bacc[jj] = fma(vg.cs, prod, (vg.sill - vg.cs) * (double)nzero);
      continue;
    }
    double h0 = 0.0;
    if (VK == GSK_VARIO_EXPONENTIAL && a.rhs_taylor) {
      const double dx = tc[0] - nx[jj], dy = tc[1] - ny[jj];
      double d2 = fma(dy, dy, dx * dx);
      if (DIM == 3) {
        const double dz = tc[2] - nz[jj];
        d2 = fma(dz, dz, d2);
      }
      h0 = gsk_is_pos(d2) ? gsk_sqrt_pos(d2) : 0.0;
    }
    double acc = 0.0, zc = 0.0;
#pragma unroll
    for (int kz = 0; kz < (DIM == 3 ? 3 : 1); ++kz) {
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const double syz = (DIM == 3) ? sy[ky] + sz[kz] : sy[ky];
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const double s = sx[kx] + syz;
          if (VK == GSK_VARIO_SPHERICAL) {
            const double u = UNIT ? s : s * vg.inv_r2;
            const double t = gsk_sqrt_nonneg(u);
            double c = fma(t, fma(vg.hcs, u, vg.m15cs), vg.cs);
            c = gsk_lt_one(u) ? c : 0.0;
            if (!nug0) c = gsk_is_pos(s) ? c : vg.sill;
            acc += c;
          } else if (a.rhs_taylor) {
            const bool pos = gsk_is_pos(s);
            const double h = gsk_sqrt_nonneg(s);
            const double x = vg.m3ir * (h - h0);
            double p = 2.48015873015873015873e-05;      // 1/8!
            p = fma(p, x, 1.98412698412698412698e-04);  // 1/7!
            p = fma(p, x, 1.38888888888888888889e-03);
            p = fma(p, x, 8.33333333333333333333e-03);
            p = fma(p, x, 4.16666666666666666667e-02);
            p = fma(p, x, 1.66666666666666666667e-01);
            p = fma(p, x, 0.5);
            p = fma(p, x, 1.0);
            p = fma(p, x, 1.0);
            acc += pos ? p : 0.0;
            zc += pos ? 0.0 : 1.0;
          } else {
            double c = vg.cs * gsk_exp_neg(vg.m3ir * gsk_sqrt_nonneg(s));
            if (!nug0) c = gsk_is_pos(s) ? c : vg.sill;
            acc += c;
          }
        }
      }
    }
    if (VK == GSK_VARIO_EXPONENTIAL && a.rhs_taylor) acc = fma(vg.cs * gsk_exp_neg(vg.m3ir * h0), acc, vg.sill * zc);
    bacc[jj] = acc;
  }
}

// G lanes per target, R register row slots (R·G >= RS), W panel width, RS rows stored per column,
// NT threads per CTA. COLS: the gsk_krige_columns epilogue (Kriging weights, then one mean per value column) follows
// phase 6; the instantiations without it compile to the same code as before it existed.
template <int G, int R, int W, int RS, int NT, int DIM, int VK, bool COLS = false>
__global__ void __launch_bounds__(NT) local_solve_kernel(const GskLocalArgs a, const Layout L, const GskColArgs ca) {
  static_assert(R * G >= RS && RS % W == 0, "register rows must cover the stored rows");
  constexpr int CTA_THREADS = NT;
  constexpr int RT = RS;
  constexpr int A = col_align<W>();
  constexpr int LD = lead_dim<G, RS>();  // column stride base (>= RT)
  constexpr int KCMAX = RT - W;
  constexpr bool USE_MMA = (G == 32 && W == 8 && A == 8);  // panel updates on the FP64 tensor path (DMMA)
  constexpr int TPW = 32 / G;
  constexpr int TPC = TPW * (CTA_THREADS / 32);
  constexpr bool UNROLL_P = (G == 4);  // small systems: unroll the left-looking loops completely
  // Rows are dealt to the register slots bottom-up: slot r holds rows ROW0(r) + l, ROW0(r) = RS − G·(r+1)
  // (the top slot may start below zero; those rows do not exist). For a panel starting at column c0 the live
  // rows [c0, RS) then fill ceil((RS − c0)/G) slots exactly — with a top-down deal and G = 32 most lanes of the
  // upper slots would be dead rows.
  // When RS is a multiple of G both deals are equivalent and the plain top-down one is kept.
  constexpr bool BOTTOM_UP = (RS % G) != 0;
#define ROW0(r) (BOTTOM_UP ? RS - G * ((r) + 1) : (r) * G)
#define GSK_ROW_OK(r) ((ROW0(r) >= 0) || (ROW0(r) + l >= 0))
#define SLOT_LIVE(r, c) (ROW0(r) + G - 1 >= (c))          /* slot r still holds rows >= c */
#define OWNER_SLOT(j) (BOTTOM_UP ? (RS - 1 - (j)) / G : (j) / G)
  // One warp per target: the neighbour coordinates used for the covariances are taken relative to the target
  // centroid and, for the spherical model, in units of the range (d² is then the polynomial's argument); the
  // covariance block is filled pair by pair (see phase 3)
  constexpr bool PAIRFILL = (G == 32);
  constexpr bool UNITG = PAIRFILL && (VK == GSK_VARIO_SPHERICAL);
  constexpr int CTAB = PAIRFILL ? ((KCMAX + 1) / 2 + 3) / 4 * 4 : 0;  // doubles holding the column-base table (ints)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *sm = reinterpret_cast<double *>(smem_raw);
  double *sup = sm;  // [3][nsup]
  const int nsup_pad = a.sup_smem ? ((3 * a.nsup + 3) & ~3) : 0;
  int *ctab = reinterpret_cast<int *>(sm + nsup_pad);  // element (row i, column c) of a packed factor sits at ctab[c] + i
  double *groups = sm + nsup_pad + CTAB;

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int l = lane % G;   // lane within the target group
  const int grp = tid / G;  // group within the CTA
  const int gbase = lane - l;  // first lane of my group in the warp
  const int KC = L.KC, e = L.e, EPr = L.EPr;

  const long long t = (long long)blockIdx.x * TPC + grp;  // slab-local target
  const bool live = t < a.count;
  // issue the neighbour-index loads and the dependent record loads first: their latency overlaps the
  // support staging, the barrier and the centroid arithmetic
  constexpr int JM = (KCMAX + G - 1) / G;
  int nidx[JM];
#pragma unroll
  for (int jj = 0; jj < JM; ++jj) {
    const int j = jj * G + l;
    nidx[jj] = (live && j < a.k) ? a.nbr[t * a.k + j] : -1;  // −1 padded beyond nn: no dependence on the nn load
  }
  double4 nrec[JM];
#pragma unroll
  for (int jj = 0; jj < JM; ++jj) {
    nrec[jj] = make_double4(0.0, 0.0, 0.0, 0.0);
    if (nidx[jj] >= 0) nrec[jj] = a.rec_orig[nidx[jj]];
  }

  const double cscale = UNITG ? a.vg.inv_r : 1.0;
  if (a.sup_smem)
    for (int i = tid; i < 3 * a.nsup; i += CTA_THREADS) sup[i] = UNITG ? a.sup[i] * cscale : a.sup[i];
  if (PAIRFILL)
    for (int c = tid; c < KCMAX; c += CTA_THREADS) ctab[c] = col_off<LD, A>(c) - (c & ~(A - 1));
  __syncthreads();

  double *S = groups + (size_t)grp * L.gsz;
  double *nbX = S + L.off_nb;
  double *nbY = nbX + KCMAX;
  double *nbZ = (DIM == 3) ? nbY + KCMAX : nbY;
  double *GM = S + L.off_gm;
  const GskVario vg = a.vg;

  // ---- target centroid ----
  double tc[3] = {0.0, 0.0, 0.0};
  int nn = 0;
  if (live) {
    const long long lin = a.first + t;
    if (a.tg.is_grid) {
      if (a.tg.gdim[0] * a.tg.gdim[1] * a.tg.gdim[2] < 0x7fffffffLL) {  // 32-bit index math (the common case)
        unsigned rem = (unsigned)lin;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          if (d < a.tg.dim) {
            const unsigned gd = (unsigned)a.tg.gdim[d];
            const unsigned qd = rem / gd;
            tc[d] = gsk_cell_center(a.tg.gorg[d], a.tg.gsp[d], (long long)(rem - qd * gd));
            rem = qd;
          }
        }
      } else {
        long long rem = lin;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          if (d < a.tg.dim) {
            long long c = rem % a.tg.gdim[d];
            rem /= a.tg.gdim[d];
            tc[d] = gsk_cell_center(a.tg.gorg[d], a.tg.gsp[d], c);
          }
        }
      }
    } else {
      for (int d = 0; d < a.tg.dim; ++d) tc[d] = a.tg.pts[d][lin];
    }
    nn = a.nn[t];
  }
  const bool estimate = live && nn >= a.min_neighbors && nn > 0;
  if (!estimate) nn = 0;

  // ---- phase 1+2: gather my neighbours (j = l, l+G, …) into registers; block-support RHS
  //      b_j = mean_q C(‖t + δ_q − x_j‖) with the q loop outermost so that the JM evaluations of a
  //      lane are independent (ILP); write the extra rows of column j ----
  double cx[JM], cy[JM], cz[JM];  // covariance coordinates of my neighbours (PAIRFILL keeps them for phase 3)
  {
    double nx[JM], ny[JM], nz[JM], nv[JM], bacc[JM];
#pragma unroll
    for (int jj = 0; jj < JM; ++jj) {
      const int j = jj * G + l;
      const double4 rc = nrec[jj];
      nx[jj] = rc.x; ny[jj] = rc.y; nz[jj] = rc.z; nv[jj] = rc.w;
      bacc[jj] = 0.0;
      // (relative to the centroid before scaling: scaling absolute coordinates would lose digits in the differences)
      cx[jj] = UNITG ? (rc.x - tc[0]) * cscale : rc.x;
      cy[jj] = UNITG ? (rc.y - tc[1]) * cscale : rc.y;
      cz[jj] = UNITG ? (rc.z - tc[2]) * cscale : rc.z;
      if (j < KC) {
        nbX[j] = cx[jj];
        nbY[j] = cy[jj];
        if (DIM == 3) nbZ[j] = cz[jj];
      }
    }
    {
      const double tcz[3] = {UNITG ? 0.0 : tc[0], UNITG ? 0.0 : tc[1], UNITG ? 0.0 : tc[2]};  // UNITG: the centroid is the origin
      if (PAIRFILL && a.sup_tensor3) {
        double axs[3][3];
#pragma unroll
        for (int d = 0; d < 3; ++d)
#pragma unroll
          for (int i = 0; i < 3; ++i) axs[d][i] = UNITG ? a.sup_ax[d][i] * cscale : a.sup_ax[d][i];
        rhs_tensor3<VK, DIM, JM, UNITG>(a, vg, axs, tcz, cx, cy, cz, bacc);
      } else if (a.sup_smem) {
        rhs_block_support<VK, DIM, JM, UNITG>(a, vg, sup, tcz, cx, cy, cz, bacc);
      } else {  // large support (or no shared memory left): every lane reads the same offset from global memory
        rhs_block_support<VK, DIM, JM, UNITG>(a, vg, UNITG ? a.sup_unit : a.sup, tcz, cx, cy, cz, bacc);
      }
    }
    const double inv_q = 1.0 / (double)a.nsup;
    const int nextra = RT - KC;
#pragma unroll
    for (int jj = 0; jj < JM; ++jj) {
      const int j = jj * G + l;
      if (j < KC) {
        const bool valid = j < nn;
        double *colj = S + col_off<LD, A>(j) - (j & ~(A - 1));
        colj[KC] = valid ? bacc[jj] * inv_q : 0.0;
        colj[KC + 1] = valid ? ((a.es.kind == GSK_EST_SIMPLE) ? nv[jj] - a.es.sk_mean : nv[jj]) : 0.0;
        for (int r2 = 2; r2 < nextra; ++r2) {
          double v = 0.0;
          if (valid && r2 < e) {
            if (a.es.kind == GSK_EST_ORDINARY) v = 1.0;
            else {
              const int *ex = a.es.exps[r2 - 2];
              v = gsk_ipow(nx[jj], ex[0]) * gsk_ipow(ny[jj], ex[1]);
              if (DIM == 3) v *= gsk_ipow(nz[jj], ex[2]);
            }
          }
          colj[KC + r2] = v;
        }
      }
    }
  }
  __syncwarp();

  // ---- phase 3: covariance block in place.
  if constexpr (PAIRFILL) {
    // One warp per target: every unordered pair of neighbours is evaluated exactly once by a round-robin pairing.
    // Lane l keeps rows i = l + 32·s (coordinates in registers, from phase 1); in round d it pairs each of them with
    // row j = (i + d) mod KC, whose coordinates come from shared memory (consecutive lanes read consecutive entries).
    // Rounds d = 1 … KC/2 − 1 cover the pairs at circular distance d from both sides, round KC/2 the antipodal pairs
    // once: KC(KC−1)/2 evaluations, all lanes busy — the column-by-column fill (below, for G < 32) keeps the lanes of
    // rows above the diagonal idle, 44 % of the work at KC = 64. Element (max, min) goes to ctab[min] + max.
    const int M = KC, H = KC >> 1;
#pragma unroll
    for (int s2 = 0; s2 < JM; ++s2) {
      const int i = l + 32 * s2;
      if (i < KC) {
        S[ctab[i] + i] = (i < nn) ? vg.sill : 1.0;                                 // diagonal (unused rows: identity)
        for (int r2 = i & ~(A - 1); r2 < i; ++r2) S[ctab[i] + r2] = 0.0;          // in-block entries above it
      }
    }
#pragma unroll 2
    for (int d = 1; d < H; ++d) {
#pragma unroll
      for (int s2 = 0; s2 < JM; ++s2) {
        const int i = l + 32 * s2;
        const bool act = i < M;
        int j = i + d;
        j = (j >= M) ? j - M : j;
        j = act ? j : 0;
        const double dx = cx[s2] - nbX[j], dy = cy[s2] - nbY[j];
        double d2 = fma(dy, dy, dx * dx);
        if (DIM == 3) {
          const double dz = cz[s2] - nbZ[j];
          d2 = fma(dz, dz, d2);
        }
        double v = cov_fast<VK, UNITG>(vg, d2);
        const int hi = max(i, j), lo = min(i, j);
        v = (hi < nn) ? v : 0.0;
        if (act) S[ctab[lo] + hi] = v;
      }
    }
#pragma unroll
    for (int s2 = 0; s2 < JM; ++s2) {
      const int i = l + 32 * s2;
      const bool act = i < H;
      const int j = act ? i + H : 0;
      const double dx = cx[s2] - nbX[j], dy = cy[s2] - nbY[j];
      double d2 = fma(dy, dy, dx * dx);
      if (DIM == 3) {
        const double dz = cz[s2] - nbZ[j];
        d2 = fma(dz, dz, d2);
      }
      double v = cov_fast<VK, UNITG>(vg, d2);
      v = (j < nn) ? v : 0.0;
      if (act) S[ctab[i] + j] = v;
    }
  } else {
    // Lane l owns rows i = r·G + l (coordinates in registers) and walks the columns p; the R evaluations per
    // column are independent ----
    constexpr int RS_S = R;  // every slot may hold neighbour rows
    double xi[RS_S], yi[RS_S], zi[RS_S];
#pragma unroll
    for (int r = 0; r < RS_S; ++r) {
      const int i = ROW0(r) + l;
      const bool ok = i >= 0 && i < KC;
      xi[r] = ok ? nbX[i] : 0.0;
      yi[r] = ok ? nbY[i] : 0.0;
      zi[r] = (DIM == 3 && ok) ? nbZ[i] : 0.0;
    }
    // columns in blocks of A share their first stored row sb, hence the set of active slots (static)
#pragma unroll
    for (int sb = 0; sb < KCMAX; sb += A) {
      if (sb < KC) {
        for (int pp = 0; pp < A; ++pp) {
          const int p = sb + pp;
          const bool valid_p = p < nn;
          const double xp = nbX[p], yp = nbY[p], zp = (DIM == 3) ? nbZ[p] : 0.0;
          double *col = S + col_off<LD, A>(sb) + pp * (LD - sb) - sb + l;
#pragma unroll
          for (int r = 0; r < RS_S; ++r) {
            if (SLOT_LIVE(r, sb) && ROW0(r) < KCMAX) {  // static after unrolling; slots of pure extra rows are skipped
              const int i = ROW0(r) + l;
              const double dx = xi[r] - xp, dy = yi[r] - yp;
              double d2 = fma(dy, dy, dx * dx);
              if (DIM == 3) {
                const double dz = zi[r] - zp;
                d2 = fma(dz, dz, d2);
              }
              double v = cov_fast<VK>(vg, d2);
              v = (i > p && i < nn) ? v : 0.0;
              v = (i == p) ? (valid_p ? vg.sill : 1.0) : v;
              if (i >= sb && i < KC) col[ROW0(r)] = v;
            }
          }
        }
      }
    }
  }
  __syncwarp();

  // ---- phase 4: blocked in-place Cholesky of the augmented matrix (panels unrolled, static offsets) ----
  double acc[R][W];
  double *Sl = S + l;  // element (i = r·G + l, column j) sits at Sl[col_off(j) − s_j + r·G]
#pragma unroll
  for (int c0 = 0; c0 < KCMAX; c0 += W) {
    if (c0 < KC) {
      if (USE_MMA && c0 > 0) {
        // Left-looking update of the panel, in place in shared memory, as one GEMM on the tensor path:
        //   P[c0:RT, c0:c0+8] −= L[c0:RT, 0:c0] · L[c0:c0+8, 0:c0]ᵀ
        // 16-row tiles × 16-column chunks of mma.m16n8k16; the tiles are independent chains. Rows past RT and
        // columns past c0 in the last tile/chunk are zero operands (decided statically).
        constexpr int MT_MAX = (RT - W + 15) / 16;
        const int g8 = lane >> 2, t4 = lane & 3;
        const int cpan = col_off<LD, A>(c0) - c0 + 2 * t4 * (LD - c0) + g8;  // element (row g8, column c0 + 2·t4)
        double cf[MT_MAX][4];
#pragma unroll
        for (int m = 0; m < MT_MAX; ++m) {
          if (c0 + 16 * m < RT) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const bool rows_ok = c0 + 16 * m + 8 * (c >> 1) < RT;
              cf[m][c] = rows_ok ? S[cpan + (c & 1) * (LD - c0) + c0 + 16 * m + 8 * (c >> 1)] : 0.0;
            }
          }
        }
#pragma unroll
        for (int p0 = 0; p0 < KCMAX; p0 += 16) {
          if (p0 < c0) {
            int cb[4];  // S index of (row g8, column p0 + 4i + t4)
            double bf[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int pc = p0 + 4 * i, sg = pc & ~(A - 1);
              cb[i] = col_off<LD, A>(sg) - sg + (pc - sg + t4) * (LD - sg) + g8;
              bf[i] = (pc < c0) ? -S[cb[i] + c0] : 0.0;
            }
#pragma unroll
            for (int m = 0; m < MT_MAX; ++m) {
              if (c0 + 16 * m < RT) {
                double af[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const bool ok = (p0 + 4 * (i >> 1) < c0) && (c0 + 16 * m + 8 * (i & 1) < RT);
                  af[i] = ok ? S[cb[i >> 1] + c0 + 16 * m + 8 * (i & 1)] : 0.0;
                }
                gsk_dmma16816(cf[m], af, bf);
              }
            }
          }
        }
#pragma unroll
        for (int m = 0; m < MT_MAX; ++m) {
          if (c0 + 16 * m < RT) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c0 + 16 * m + 8 * (c >> 1) < RT) S[cpan + (c & 1) * (LD - c0) + c0 + 16 * m + 8 * (c >> 1)] = cf[m][c];
            }
          }
        }
        __syncwarp();
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if (SLOT_LIVE(r, c0)) {
#pragma unroll
          for (int jj = 0; jj < W; ++jj) {
            const int j = c0 + jj;
            const int sj = j & ~(A - 1);
            const bool in = (ROW0(r) >= sj) || (ROW0(r) + l >= sj);
            acc[r][jj] = in ? Sl[col_off<LD, A>(j) - sj + ROW0(r)] : 0.0;
          }
        }
      }
      // left-looking update from the finished columns p < c0
      auto update = [&](int p) {
        const double *col = S + col_off<LD, A>(p) - (p & ~(A - 1));
        double piv[W];
#pragma unroll
        for (int jj = 0; jj < W; jj += 2) {
          const double2 t2 = *reinterpret_cast<const double2 *>(col + c0 + jj);
          piv[jj] = t2.x;
          piv[jj + 1] = t2.y;
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (SLOT_LIVE(r, c0)) {
            const double own = GSK_ROW_OK(r) ? col[ROW0(r) + l] : 0.0;
#pragma unroll
            for (int jj = 0; jj < W; ++jj) acc[r][jj] = fma(-own, piv[jj], acc[r][jj]);
          }
        }
      };
      if (USE_MMA) {
        // done above
      } else if (UNROLL_P) {
#pragma unroll
        for (int p = 0; p < c0; ++p) update(p);
      } else {
        // runtime loop with an incrementally advanced column pointer: colp[i] is element (row i, column p),
        // base(p+1) − base(p) = LD − s_{p+1}. (Unrolling whole column groups saves the mask arithmetic but costs
        // the 8-lane configuration registers: measured 5 % slower on C3b.)
        const double *colp = S;
#pragma unroll 2
        for (int p = 0; p < c0; ++p) {
          double piv[W];
#pragma unroll
          for (int jj = 0; jj < W; jj += 2) {
            const double2 t2 = *reinterpret_cast<const double2 *>(colp + c0 + jj);
            piv[jj] = t2.x;
            piv[jj + 1] = t2.y;
          }
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if (SLOT_LIVE(r, c0)) {
              const double own = GSK_ROW_OK(r) ? colp[ROW0(r) + l] : 0.0;
#pragma unroll
              for (int jj = 0; jj < W; ++jj) acc[r][jj] = fma(-own, piv[jj], acc[r][jj]);
            }
          }
          colp += LD - ((p + 1) & ~(A - 1));
        }
      }
      // the W×W panel: pivots and row entries are exchanged by shuffles inside the group
#pragma unroll
      for (int jj = 0; jj < W; ++jj) {
        const int j = c0 + jj;
        const int sj = j & ~(A - 1);
        const int ro = OWNER_SLOT(j), lo = j - ROW0(ro);  // owner of row j
        const double d = __shfl_sync(0xffffffffu, acc[ro][jj], gbase + lo);
        const double rinv = gsk_rsqrt(d);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (SLOT_LIVE(r, c0)) {
            acc[r][jj] *= rinv;
            if (ROW0(r) >= j || ROW0(r) + l >= j) Sl[col_off<LD, A>(j) - sj + ROW0(r)] = acc[r][jj];
          }
        }
#pragma unroll
        for (int j2 = jj + 1; j2 < W; ++j2) {
          const int r2 = OWNER_SLOT(c0 + j2), l2 = (c0 + j2) - ROW0(r2);  // owner of row c0 + j2
          const double lj = __shfl_sync(0xffffffffu, acc[r2][jj], gbase + l2);
#pragma unroll
          for (int r = 0; r < R; ++r)
            if (SLOT_LIVE(r, c0)) acc[r][j2] = fma(-acc[r][jj], lj, acc[r][j2]);
        }
      }
      __syncwarp();
    }
  }

  // ---- phase 5: Schur complement of the extra rows: Gm = Y Yᵀ (only the slots that hold extra rows work) ----
  if (USE_MMA) {
    // one 16-row tile holds all extra rows (EPr <= 16); Y Yᵀ needs the same fragment as A and as B
    const int g8 = lane >> 2, t4 = lane & 3;
    const bool two = EPr > 8;  // rows / columns 8..15 exist
    double d0[4] = {0.0, 0.0, 0.0, 0.0}, d1[4] = {0.0, 0.0, 0.0, 0.0};
    for (int p0 = 0; p0 < KC; p0 += 16) {
      double lo[4], hi[4];  // Y[g8][p0 + 4i + t4], Y[g8 + 8][·]
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int pc = p0 + 4 * i, sg = pc & ~(A - 1);
        const bool kin = pc < KC;  // KC is a multiple of 8: the last chunk may be half empty
        const int cb = col_off<LD, A>(sg) - sg + (pc - sg + t4) * (LD - sg) + g8 + KC;
        lo[i] = kin ? S[cb] : 0.0;
        hi[i] = (kin && two) ? S[cb + 8] : 0.0;
      }
      const double af[8] = {lo[0], hi[0], lo[1], hi[1], lo[2], hi[2], lo[3], hi[3]};
      gsk_dmma16816(d0, af, lo);
      if (two) gsk_dmma16816(d1, af, hi);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int row = g8 + 8 * (c >> 1), col = 2 * t4 + (c & 1);
      if (row < EPr) {
        GM[row * EPr + col] = d0[c];
        if (two) GM[row * EPr + 8 + col] = d1[c];
      }
    }
  }
  for (int cc = 0; cc < (USE_MMA ? 0 : EPr); cc += W) {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (ROW0(r) + G > KC && ROW0(r) < KC + EPr) {  // slot holds extra rows (warp-uniform)
        double g[W];
#pragma unroll
        for (int jj = 0; jj < W; ++jj) g[jj] = 0.0;
        const int i = ROW0(r) + l;
        const bool mine = i >= KC && i < KC + EPr;
        const double *col = S;  // col[i] = element (row i, column p)
#pragma unroll 4
        for (int p = 0; p < KC; ++p, col += LD - (p & ~(A - 1))) {
          const double own = mine ? col[i] : 0.0;
#pragma unroll
          for (int jj = 0; jj < W; jj += 2) {
            const double2 t2 = *reinterpret_cast<const double2 *>(col + KC + cc + jj);
            g[jj] = fma(own, t2.x, g[jj]);
            g[jj + 1] = fma(own, t2.y, g[jj + 1]);
          }
        }
        if (mine) {
#pragma unroll
          for (int jj = 0; jj < W; ++jj) GM[(i - KC) * EPr + cc + jj] = g[jj];
        }
      }
    }
  }
  __syncwarp();

  // ---- phase 6: e×e algebra, one lane per target ----
  if (l == 0 && live) {
    double mean = NAN, var = NAN;
    if (estimate) {
      const int c = a.es.nterms;
      const double gbb = GM[0], gbz = GM[1];
      if (c == 0) {
        mean = a.es.sk_mean + gbz;
        var = vg.sill - gbb;
      } else if (c == 1) {
        const double gff = GM[2 * EPr + 2], gfb = GM[2 * EPr], gfz = GM[2 * EPr + 1];
        const double f0 = 1.0;  // OK, or UK of degree 0
        const double nu = (gfb - f0) / gff;
        mean = gbz - gfz * nu;
        var = vg.sill - (gbb - gfb * nu + f0 * nu);
        if constexpr (COLS) GM[EPr] = nu;  // row 1 (the z row) is free: the columns epilogue reads ν from there
      } else {
        // solve Gff ν = gfb − f0 (c×c SPD) by Cholesky in place on GM
        double f0[GSK_MAX_DRIFT_TERMS], nu[GSK_MAX_DRIFT_TERMS];
        for (int t2 = 0; t2 < c; ++t2) {
          const int *ex = a.es.exps[t2];
          double m = gsk_ipow(tc[0], ex[0]) * gsk_ipow(tc[1], ex[1]);
          if (DIM == 3) m *= gsk_ipow(tc[2], ex[2]);
          f0[t2] = m;
        }
#define GFF(i, j) GM[(2 + (i)) * EPr + 2 + (j)]
        // Cholesky with reciprocal pivots (no FP64 divisions / sqrt sequences on the serial lane)
        double dinv[GSK_MAX_DRIFT_TERMS];
        for (int j = 0; j < c; ++j) {
          double d = GFF(j, j);
          for (int p = 0; p < j; ++p) d = fma(-GFF(j, p), GFF(j, p), d);
          const double ri = gsk_rsqrt(d);
          dinv[j] = ri;
          for (int i = j + 1; i < c; ++i) {
            double s = GFF(i, j);
            for (int p = 0; p < j; ++p) s = fma(-GFF(i, p), GFF(j, p), s);
            GFF(i, j) = s * ri;
          }
        }
        for (int j = 0; j < c; ++j) {
          double s = GM[(2 + j) * EPr + 0] - f0[j];
          for (int p = 0; p < j; ++p) s = fma(-GFF(j, p), nu[p], s);
          nu[j] = s * dinv[j];
        }
        for (int j = c - 1; j >= 0; --j) {
          double s = nu[j];
          for (int p = j + 1; p < c; ++p) s = fma(-GFF(p, j), nu[p], s);
          nu[j] = s * dinv[j];
        }
#undef GFF
        double mz = 0.0, mb = 0.0, mf = 0.0;
        for (int j = 0; j < c; ++j) {
          mz += GM[(2 + j) * EPr + 1] * nu[j];
          mb += GM[(2 + j) * EPr + 0] * nu[j];
          mf += f0[j] * nu[j];
        }
        mean = gbz - mz;
        var = vg.sill - (gbb - mb + mf);
        if constexpr (COLS)
          for (int j = 0; j < c; ++j) GM[EPr + j] = nu[j];
      }
      if (a.flags & GSK_FLAG_CLAMP_VARIANCE) var = (var > 0.0 || var != var) ? var : 0.0;
      if (a.flags & GSK_FLAG_SQRT_ROUNDTRIP) { double sd = sqrt(var); var = sd * sd; }
    }
    gsk_store_result(a.out, t, mean, var);
  }

  // ---- columns epilogue (gsk_krige_columns): λ from Lᵀλ = y_b − Y_F ν, then mean_j = Σ λ_i z[nbr_i, j] ----
  if constexpr (COLS) {
    __syncwarp();
    const int c = a.es.nterms;
    // lane l keeps w_i for rows i = l + G·s (column i of the packed factor starts at cb[s]); the extra rows of column
    // i hold y_b (row KC) and y_F (rows KC + 2 …). Rows past nn are identity with zero extra entries: w_i = λ_i = 0.
    double wv[JM];
    int cb[JM];
#pragma unroll
    for (int s = 0; s < JM; ++s) {
      const int i = s * G + l;
      cb[s] = col_off<LD, A>(i) - (i & ~(A - 1));
      double v = 0.0;
      if (i < KC && estimate) {
        v = S[cb[s] + KC];
        for (int q = 0; q < c; ++q) v = fma(-GM[EPr + q], S[cb[s] + KC + 2 + q], v);
      }
      wv[s] = v;
    }
    // backward substitution, column form: λ_j = w_j / L_jj is final, then w_i −= L[j][i]·λ_j for i < j (L[j][i] is
    // row j of packed column i). λ goes to nbX, free since phase 3.
    for (int j = KC - 1; j >= 0; --j) {
      const int sj = j / G, lj = j - sj * G;
      double wj = 0.0;
#pragma unroll
      for (int s = 0; s < JM; ++s) wj = (s == sj) ? wv[s] : wj;
      wj = __shfl_sync(0xffffffffu, wj, gbase + lj);
      const double lam = wj / S[col_off<LD, A>(j) - (j & ~(A - 1)) + j];
      if (l == lj) nbX[j] = lam;
#pragma unroll
      for (int s = 0; s < JM; ++s) {
        const int i = s * G + l;
        if (i < j) wv[s] = fma(-S[cb[s] + j], lam, wv[s]);
      }
    }
    int *nbi = reinterpret_cast<int *>(nbY);  // neighbour indices next to λ (nbY holds KCMAX doubles)
    for (int i = l; i < nn; i += G) nbi[i] = a.nbr[t * a.k + i];
    __syncwarp();
    if (live) {
      const long long row = ca.perm ? (long long)ca.perm[t] : t;
      const int m = ca.ncols;
      const bool sk = a.es.kind == GSK_EST_SIMPLE;
      const double mu = sk ? a.es.sk_mean : 0.0;
      // one column per lane: a neighbour's m values are contiguous, the lanes of a group read them together; the sum
      // runs over i in list order whatever the configuration, so a column's mean does not depend on m or its position
      for (int col = l; col < m; col += G) {
        double acc = 0.0;
        for (int i = 0; i < nn; ++i) acc = fma(nbX[i], ca.z[(size_t)nbi[i] * m + col] - mu, acc);
        ca.mean[row * m + col] = estimate ? mu + acc : NAN;
      }
      if (ca.w)
        for (int i = l; i < a.k; i += G) ca.w[row * a.k + i] = (estimate && i < nn) ? nbX[i] : 0.0;
      if (ca.lag)
        for (int q = l; q < c; q += G) ca.lag[row * c + q] = estimate ? GM[EPr + q] : NAN;
    }
  }
#undef GSK_ROW_OK
#undef ROW0
#undef SLOT_LIVE
#undef OWNER_SLOT
}

template <int G, int R, int W, int RS, int NT, int DIM, int VK, bool COLS>
inline cudaError_t launch_one(const GskLocalArgs &a, const GskColArgs &ca, int e, cudaStream_t st) {
  constexpr int CTA_THREADS = NT;
  constexpr int TPW = 32 / G;
  constexpr int TPC = TPW * (CTA_THREADS / 32);
  Layout L = make_layout<G, R, W, RS, DIM>(a.k, e);
  constexpr int KCMAX = RS - W;
  constexpr int CTAB = (G == 32) ? ((KCMAX + 1) / 2 + 3) / 4 * 4 : 0;  // column-base table of the pair fill (kernel: ctab)
  GskLocalArgs b = a;
  // the support offsets are staged in shared memory when they are few and there is room; otherwise the kernel
  // reads them from global memory (uniform addresses). The factor storage itself must fit.
  int nsup_pad = (3 * a.nsup + 3) & ~3;
  size_t smem = sizeof(double) * ((size_t)nsup_pad + CTAB + (size_t)TPC * L.gsz);
  b.sup_smem = (a.nsup <= GSK_MAX_SUPPORT && smem <= GSK_SMEM_OPTIN_MAX) ? 1 : 0;
  if (!b.sup_smem) smem = sizeof(double) * ((size_t)CTAB + (size_t)TPC * L.gsz);
  if (smem > GSK_SMEM_OPTIN_MAX) return cudaErrorInvalidConfiguration;  // reported as GSK_ERR_UNSUPPORTED by the caller
  auto kern = local_solve_kernel<G, R, W, RS, NT, DIM, VK, COLS>;
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) return err;
  unsigned grid = (unsigned)((a.count + TPC - 1) / TPC);
  kern<<<grid, CTA_THREADS, smem, st>>>(b, L, ca);
  return cudaGetLastError();
}

template <int G, int R, int W, int RS, int NT, bool COLS = false>
inline cudaError_t launch_cfg(const GskLocalArgs &a, const GskColArgs &ca, int e, cudaStream_t st) {
  const bool d3 = a.tg.dim == 3;
  switch (a.vg.kind) {
    case GSK_VARIO_GAUSSIAN:
      return d3 ? launch_one<G, R, W, RS, NT, 3, GSK_VARIO_GAUSSIAN, COLS>(a, ca, e, st) : launch_one<G, R, W, RS, NT, 2, GSK_VARIO_GAUSSIAN, COLS>(a, ca, e, st);
    case GSK_VARIO_SPHERICAL:
      return d3 ? launch_one<G, R, W, RS, NT, 3, GSK_VARIO_SPHERICAL, COLS>(a, ca, e, st) : launch_one<G, R, W, RS, NT, 2, GSK_VARIO_SPHERICAL, COLS>(a, ca, e, st);
    default:
      return d3 ? launch_one<G, R, W, RS, NT, 3, GSK_VARIO_EXPONENTIAL, COLS>(a, ca, e, st) : launch_one<G, R, W, RS, NT, 2, GSK_VARIO_EXPONENTIAL, COLS>(a, ca, e, st);
  }
}

}  // namespace gsk_local

// one translation unit per register/lanes configuration (compiled in parallel); cols: run the gsk_krige_columns epilogue
cudaError_t gsk_local_launch_A(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols = nullptr);  // G=4  R=3 W=4  12 rows, 128 thr
cudaError_t gsk_local_launch_B(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols = nullptr);  // G=4  R=6 W=4  24 rows, 128 thr
cudaError_t gsk_local_launch_C(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols = nullptr);  // G=8  R=5 W=8  40 rows,  64 thr
cudaError_t gsk_local_launch_D(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols = nullptr);  // G=32 R=3 W=8  72 rows, 128 thr
cudaError_t gsk_local_launch_E(const GskLocalArgs &a, int e, cudaStream_t st, const GskColArgs *cols = nullptr);  // G=32 R=4 W=8 112 rows, 128 thr
