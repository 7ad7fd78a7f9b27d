// global.cu — K4 + K5: the global ("exact") kriging system, replacing exactsolve's
// `fit(estimator, pdata)` once (ref: src/estimation/krig.jl:176) and `predictprob(krig, var, pdomain[ind])`
// for every target (krig.jl:180).
//
// Plan (once per GPU):  C = sill − Γ (n×n, FP64) is assembled on the device, factorised C = L Lᵀ by a
// blocked right-looking Cholesky, and L is inverted block row by block row (Linv). With
// E = [z (−μ) | f_1 … f_c] (drift columns: OK → ones, UK → monomials), Y_E = Linv·E and the constant
// Gram block G_EE = Y_EᵀY_E are kept resident.
// Execute (per batch of targets): the block-support right-hand sides B (n × batch) are assembled,
// then ONE triangular GEMM  Y = Linv·B  runs with a fused epilogue that never writes Y: per target it
// reduces ‖y‖² and Y_Eᵀy, i.e. the Gram entries Gm[b,b], Gm[E,b] of the same block elimination the
// local kernel uses (local_solve.cuh), from which ν, mean and variance follow:
//   ν = Gff⁻¹(Gfb − f₀),  mean = Gbz − Gfz·ν,  var = sill − (Gbb − Gfb·ν + f₀·ν)      (SK: μ + Gbz, sill − Gbb)
#include <math.h>
#include <string.h>

#include <cmath>

#include <algorithm>
#include <vector>

#include "gsk_internal.cuh"

namespace {

constexpr int NB = 64;   // block size of the factorisation and of the GEMM tiles
constexpr int BK = 16;

struct GArgs {
  const double4 *rec;  // samples {x,y,z,value}
  long long n, np;     // samples, padded to a multiple of NB
  GskVario vg;
  int dim;
};

// ---- C assembly (lower triangle + diagonal; padded rows/cols = identity) ----
template <int VK>
__global__ void assemble_kernel(GArgs g, double *__restrict__ A) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long j = blockIdx.y;
  if (i >= g.np || i < j) return;
  double v;
  if (i >= g.n || j >= g.n) v = (i == j) ? 1.0 : 0.0;
  else if (i == j) v = g.vg.sill;
  else {
    double4 a = g.rec[i], b = g.rec[j];
    double dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
    double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
    v = gsk_cov<VK>(g.vg, d2);
  }
  A[i + j * g.np] = v;
}

// ---- 64×64 tile product on the FP64 tensor path (DMMA): acc += A(64×K)·B(K×64), K a multiple of 16 ----
// A column-major (lda). B either column-major K×64 (TRANSB=false, element (k,n) at B[k + n·ldb])
// or given as 64×K column-major to be used transposed (TRANSB=true, element (k,n) at B[n + k·ldb]).
// 8 warps as 4 (M) × 2 (N); each warp owns a 16×32 sub-tile = 4 m16n8k16 accumulators: acc[n8][c] holds
// element (row, col) = (wm·16 + g + 8·(c>>1), wn·32 + n8·8 + 2t + (c&1)), g = lane>>2, t = lane&3.
constexpr int TLD = NB + 4;  // ≡ 4 (mod 16) doubles: conflict-free fragment loads
__device__ __forceinline__ void acc_coords(int n8, int c, int &row, int &col) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  row = (warp >> 1) * 16 + (lane >> 2) + 8 * (c >> 1);
  col = (warp & 1) * 32 + n8 * 8 + 2 * (lane & 3) + (c & 1);
}
template <bool TRANSB>
__device__ __forceinline__ void tile_mma(const double *__restrict__ A, long long lda, const double *__restrict__ B,
                                         long long ldb, int K, double (&acc)[4][4], double (*As)[TLD],
                                         double (*Bs)[TLD]) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 1, wn = warp & 1, g = lane >> 2, t = lane & 3;
  for (int k0 = 0; k0 < K; k0 += BK) {
    for (int e = tid; e < NB * BK; e += 256) {
      int m = e & 63, k = e >> 6;
      As[k][m] = A[m + (long long)(k0 + k) * lda];
    }
    if (TRANSB) {
      for (int e = tid; e < NB * BK; e += 256) {
        int nn = e & 63, k = e >> 6;
        Bs[k][nn] = B[nn + (long long)(k0 + k) * ldb];
      }
    } else {
      for (int e = tid; e < NB * BK; e += 256) {
        int k = e & 15, nn = e >> 4;
        Bs[k][nn] = B[(k0 + k) + (long long)nn * ldb];
      }
    }
    __syncthreads();
    double af[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) af[i] = As[t + 4 * (i >> 1)][wm * 16 + g + 8 * (i & 1)];
#pragma unroll
    for (int n8 = 0; n8 < 4; ++n8) {
      double bf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) bf[i] = Bs[t + 4 * i][wn * 32 + n8 * 8 + g];
      asm volatile(
          "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
          "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
          : "+d"(acc[n8][0]), "+d"(acc[n8][1]), "+d"(acc[n8][2]), "+d"(acc[n8][3])
          : "d"(af[0]), "d"(af[1]), "d"(af[2]), "d"(af[3]), "d"(af[4]), "d"(af[5]), "d"(af[6]), "d"(af[7]),
            "d"(bf[0]), "d"(bf[1]), "d"(bf[2]), "d"(bf[3]));
    }
    __syncthreads();
  }
}

// ---- pipelined variant for long K (Linv rows): 3-stage cp.async ring, NN operands ----
constexpr int LS = 3;
constexpr int LA_STAGE = BK * TLD;    // A stage: [k][m], m contiguous
constexpr int LB_LD = BK + 4;         // B stage: [n][k], k contiguous; ≡ 4 (mod 16) doubles
constexpr int LB_STAGE = NB * LB_LD;
constexpr size_t LINV_SMEM = sizeof(double) * (size_t)LS * (LA_STAGE + LB_STAGE);
__device__ __forceinline__ void cp16(void *dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src));
}
__device__ __forceinline__ void tile_mma_nn_async(const double *__restrict__ A, long long lda,
                                                  const double *__restrict__ B, long long ldb, int K,
                                                  double (&acc)[4][4], double *sm) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 1, wn = warp & 1, g = lane >> 2, t = lane & 3;
  const int nk = K / BK;
  auto load = [&](int s, int kt) {
    double *as = sm + (size_t)s * LA_STAGE;
    double *bs = sm + (size_t)LS * LA_STAGE + (size_t)s * LB_STAGE;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int c = tid + 256 * i;
      const int k = c >> 5, mc = c & 31;
      cp16(as + k * TLD + 2 * mc, A + 2 * mc + (long long)(kt * BK + k) * lda);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int c = tid + 256 * i;
      const int n = c >> 3, kc = c & 7;
      cp16(bs + n * LB_LD + 2 * kc, B + kt * BK + 2 * kc + (long long)n * ldb);
    }
  };
#pragma unroll
  for (int s = 0; s < LS - 1; ++s) {
    if (s < nk) load(s, s);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int kt = 0; kt < nk; ++kt) {
    asm volatile("cp.async.wait_group %0;" ::"n"(LS - 2) : "memory");
    __syncthreads();
    if (kt + LS - 1 < nk) load((kt + LS - 1) % LS, kt + LS - 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const double *as = sm + (size_t)(kt % LS) * LA_STAGE;
    const double *bs = sm + (size_t)LS * LA_STAGE + (size_t)(kt % LS) * LB_STAGE;
    double af[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) af[i] = as[(t + 4 * (i >> 1)) * TLD + wm * 16 + g + 8 * (i & 1)];
#pragma unroll
    for (int n8 = 0; n8 < 4; ++n8) {
      double bf[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) bf[i] = bs[(wn * 32 + n8 * 8 + g) * LB_LD + t + 4 * i];
      asm volatile(
          "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
          "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
          : "+d"(acc[n8][0]), "+d"(acc[n8][1]), "+d"(acc[n8][2]), "+d"(acc[n8][3])
          : "d"(af[0]), "d"(af[1]), "d"(af[2]), "d"(af[3]), "d"(af[4]), "d"(af[5]), "d"(af[6]), "d"(af[7]),
            "d"(bf[0]), "d"(bf[1]), "d"(bf[2]), "d"(bf[3]));
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
}

// ---- diagonal block: Cholesky of A[j0:j0+64, j0:j0+64] in place, and its inverse into Dinv ----
// 64 threads, thread i owns row i (left-looking by columns): s = a_ij − Σ_{p<j} l_ip·l_jp with row j broadcast from
// shared memory (row stride 65 doubles: the threads' own-row reads fall into distinct banks), the pivot's reciprocal
// square root from the owner of row j. Then thread c forward-substitutes column c of the inverse. (Round 1 ran the
// square roots on one thread of a 256-thread CTA with a right-looking update: 147 µs per block, 314 blocks in C4.)
__global__ void __launch_bounds__(64) potrf_diag_kernel(double *__restrict__ A, long long ld, long long j0,
                                                        double *__restrict__ Dinv) {
  __shared__ double L[NB][NB + 1];
  __shared__ double pivinv;
  const int i = threadIdx.x;
  double *blk = A + j0 + j0 * ld;
  for (int j = 0; j < NB; ++j) L[i][j] = (i >= j) ? blk[i + (long long)j * ld] : 0.0;
  __syncthreads();
  for (int j = 0; j < NB; ++j) {
    double s = L[i][j];
    for (int p = 0; p < j; ++p) s = fma(-L[i][p], L[j][p], s);
    if (i == j) {
      const double d = sqrt(s);
      L[j][j] = d;
      pivinv = 1.0 / d;
    }
    __syncthreads();
    if (i > j) L[i][j] = s * pivinv;
    __syncthreads();
  }
  for (int j = 0; j <= i; ++j) blk[i + (long long)j * ld] = L[i][j];
  // inverse of the lower-triangular block: thread c solves L x = e_c (column c of the inverse)
  {
    const int c = i;
    double *x = Dinv + c * NB;
    for (int r = 0; r < NB; ++r) {
      double s = (r == c) ? 1.0 : 0.0;
      for (int p = c; p < r; ++p) s -= L[r][p] * x[p];
      x[r] = (r >= c) ? s / L[r][r] : 0.0;
    }
  }
}

// ---- panel below the diagonal block: P = A[i-block, j-block] · Dinvᵀ, in place ----
__global__ void __launch_bounds__(256) trsm_panel_kernel(double *__restrict__ A, long long ld, long long j0,
                                                         const double *__restrict__ Dinv) {
  __shared__ double As[BK][TLD];
  __shared__ double Bs[BK][TLD];
  const long long i0 = j0 + NB + (long long)blockIdx.x * NB;
  double *blk = A + i0 + j0 * ld;
  double acc[4][4] = {};
  // the whole 64×64 source tile is consumed before anything is written back (same CTA owns it)
  tile_mma<true>(blk, ld, Dinv, NB, NB, acc, As, Bs);
  __syncthreads();
#pragma unroll
  for (int n8 = 0; n8 < 4; ++n8)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      int row, col;
      acc_coords(n8, c, row, col);
      blk[row + (long long)col * ld] = acc[n8][c];
    }
}

// ---- trailing update: A[bi, bj] −= P[bi]·P[bj]ᵀ for all tile pairs bi >= bj below the panel ----
__global__ void __launch_bounds__(256) syrk_kernel(double *__restrict__ A, long long ld, long long j0, int nrem) {
  __shared__ double As[BK][TLD];
  __shared__ double Bs[BK][TLD];
  // linear index over the lower-triangular tile pairs
  int t = blockIdx.x;
  int bi = (int)((sqrt(8.0 * t + 1.0) - 1.0) * 0.5);
  while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
  while (bi * (bi + 1) / 2 > t) --bi;
  int bj = t - bi * (bi + 1) / 2;
  if (bi >= nrem) return;
  const long long r0 = j0 + NB + (long long)bi * NB, c0 = j0 + NB + (long long)bj * NB;
  double acc[4][4] = {};
  tile_mma<true>(A + r0 + j0 * ld, ld, A + c0 + j0 * ld, ld, NB, acc, As, Bs);
  double *blk = A + r0 + c0 * ld;
#pragma unroll
  for (int n8 = 0; n8 < 4; ++n8)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      int row, col;
      acc_coords(n8, c, row, col);
      blk[row + (long long)col * ld] -= acc[n8][c];
    }
}

// ---- Linv block row i:  X[i, jb] = −Dinv_i · Σ_{m=jb}^{i−1} L[i, m]·X[m, jb]  (jb < i);  X[i,i] = Dinv_i ----
__global__ void __launch_bounds__(256) linv_row_kernel(const double *__restrict__ A, double *__restrict__ X,
                                                       long long ld, int bi, const double *__restrict__ Dinv_all) {
  // the stage ring is only live inside tile_mma_nn_async; T reuses the same shared memory afterwards
  extern __shared__ __align__(16) double lbuf[];
  static_assert(LINV_SMEM >= sizeof(double) * NB * (NB + 1), "T must fit in the stage ring");
  double (*T)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(lbuf);
  const int jb = blockIdx.x;
  const long long i0 = (long long)bi * NB, j0 = (long long)jb * NB;
  const double *Di = Dinv_all + (size_t)bi * NB * NB;
  const int tm = (threadIdx.x & 15) * 4, tn = (threadIdx.x >> 4) * 4;
  double *out = X + i0 + j0 * ld;
  if (jb == bi) {
    for (int e = threadIdx.x; e < NB * NB; e += 256) {
      int i = e & 63, j = e >> 6;
      out[i + (long long)j * ld] = Di[i + j * NB];
    }
    return;
  }
  double acc[4][4] = {};
  tile_mma_nn_async(A + i0 + j0 * ld, ld, X + j0 + j0 * ld, ld, (bi - jb) * NB, acc, lbuf);
#pragma unroll
  for (int n8 = 0; n8 < 4; ++n8)
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      int row, col;
      acc_coords(n8, c, row, col);
      T[row][col] = acc[n8][c];
    }
  __syncthreads();
  // out = −Di · T   (Di lower triangular 64×64)
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = tm + i, c = tn + j;
      double s = 0.0;
      for (int p = 0; p <= r; ++p) s = fma(Di[r + p * NB], T[p][c], s);
      out[r + (long long)c * ld] = -s;
    }
}

// ---- Y_E = Linv · E  (n × ne, tall-skinny): one warp per row ----
__global__ void linv_times_e_kernel(const double *__restrict__ X, long long ld, long long np,
                                    const double *__restrict__ E, int ne, double *__restrict__ YE) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= np) return;
  for (int c = 0; c < ne; ++c) {
    double s = 0.0;
    for (long long p = lane; p <= row; p += 32) s = fma(X[row + p * ld], E[p + c * np], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) YE[row + c * np] = s;
  }
}

// G_EE = Y_EᵀY_E, one CTA, deterministic
__global__ void gram_ee_kernel(const double *__restrict__ YE, long long np, int ne, double *__restrict__ GEE) {
  __shared__ double red[256];
  for (int a = 0; a < ne; ++a)
    for (int b = 0; b < ne; ++b) {
      double s = 0.0;
      for (long long i = threadIdx.x; i < np; i += 256) s = fma(YE[i + a * np], YE[i + b * np], s);
      red[threadIdx.x] = s;
      __syncthreads();
      for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
      }
      if (threadIdx.x == 0) GEE[a * ne + b] = red[0];
      __syncthreads();
    }
}

// E columns: z (− μ), then drift monomials of the samples; padded rows 0
__global__ void build_e_kernel(GArgs g, GskEstimator es, double *__restrict__ E) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= g.np) return;
  const int ne = 1 + es.nterms;
  if (i >= g.n) {
    for (int c = 0; c < ne; ++c) E[i + c * g.np] = 0.0;
    return;
  }
  double4 r = g.rec[i];
  E[i] = (es.kind == GSK_EST_SIMPLE) ? r.w - es.sk_mean : r.w;
  for (int t = 0; t < es.nterms; ++t) {
    double v = 1.0;
    if (es.kind == GSK_EST_UNIVERSAL)
      v = gsk_ipow(r.x, es.exps[t][0]) * gsk_ipow(r.y, es.exps[t][1]) * gsk_ipow(r.z, es.exps[t][2]);
    E[i + (1 + t) * g.np] = v;
  }
}

// ---- execute: right-hand sides of a batch, B[i + t·np] = mean_q C(‖c_t + δ_q − x_i‖) ----
template <int VK>
__global__ void rhs_kernel(GArgs g, GskTargets tg, const double *__restrict__ sup, int nsup, long long first,
                           int nbatch, double *__restrict__ Bm) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  int t = blockIdx.y;
  if (i >= g.np || t >= nbatch) return;
  double v = 0.0;
  if (i < g.n) {
    long long lin = first + t;
    double tc[3] = {0.0, 0.0, 0.0};
    if (tg.is_grid) {
      long long rem = lin;
      for (int d = 0; d < tg.dim; ++d) {
        long long c = rem % tg.gdim[d];
        rem /= tg.gdim[d];
        tc[d] = gsk_cell_center(tg.gorg[d], tg.gsp[d], c);
      }
    } else {
      for (int d = 0; d < tg.dim; ++d) tc[d] = tg.pts[d][lin];
    }
    double4 r = g.rec[i];
    double acc = 0.0;
    for (int q = 0; q < nsup; ++q) {
      double dx = (tc[0] + sup[q]) - r.x, dy = (tc[1] + sup[nsup + q]) - r.y, dz = (tc[2] + sup[2 * nsup + q]) - r.z;
      double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
      acc += gsk_cov<VK>(g.vg, d2);
    }
    v = acc / (double)nsup;
  }
  Bm[i + (long long)t * g.np] = v;
}

// ---- the hot kernel (K5): Y tile = Linv[mt, 0..mt]·B[0..mt, nt] on the FP64 tensor path ------------------
// 128×128 output tile per CTA, K stepped by 16 through a 3-stage cp.async pipeline, 8 warps each owning a
// 64×32 sub-tile computed with mma.sync.m16n8k16 f64 (SASS DMMA; tcgen05 has no FP64 kind). The epilogue
// never stores Y: per target column it reduces Σ y² and Σ y·Y_E[:,s] over the tile's 128 rows and writes
// 1+ne partial sums:  partial[(mt·(1+ne) + s)·nbpad + t].
constexpr int GT = 128;          // tile edge
constexpr int GKS = 16;          // k per pipeline stage
constexpr int GSTAGES = 3;
constexpr int AS_LD = GT + 4;    // A stage: [k][m], m contiguous; ≡ 4 (mod 16) doubles → conflict-free fragment loads
constexpr int BS_LD = GKS + 4;   // B stage: [n][k], k contiguous
constexpr int A_STAGE = GKS * AS_LD, B_STAGE = GT * BS_LD;
constexpr size_t YGEMM_SMEM = sizeof(double) * (size_t)GSTAGES * (A_STAGE + B_STAGE);

__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src));
}

__global__ void __launch_bounds__(256, 1) ygemm_dmma_kernel(const double *__restrict__ X, long long ld,
                                                            const double *__restrict__ Bm,
                                                            const double *__restrict__ YE, int ne, long long nbpad,
                                                            double *__restrict__ partial) {
  extern __shared__ __align__(16) double gsm[];
  double *As = gsm;                                  // [GSTAGES][GKS][AS_LD]
  double *Bs = gsm + (size_t)GSTAGES * A_STAGE;      // [GSTAGES][GT][BS_LD]
  __shared__ double red[2][GT];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
  const int nt = blockIdx.x, mt = gridDim.y - 1 - blockIdx.y;  // longest row tiles first
  const long long i0 = (long long)mt * GT, t0 = (long long)nt * GT;
  const int nk = (mt + 1) * (GT / GKS);

  auto load_stage = [&](int s, int kt) {
    double *as = As + (size_t)s * A_STAGE;
    double *bs = Bs + (size_t)s * B_STAGE;
    const long long k0 = (long long)kt * GKS;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = tid + 256 * i;
      const int k = c >> 6, mc = c & 63;
      cp_async16(as + k * AS_LD + 2 * mc, X + i0 + 2 * mc + (k0 + k) * ld);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = tid + 256 * i;
      const int n = c >> 3, kc = c & 7;
      cp_async16(bs + n * BS_LD + 2 * kc, Bm + (t0 + n) * ld + k0 + 2 * kc);
    }
  };

  double acc[4][4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.0;

#pragma unroll
  for (int s = 0; s < GSTAGES - 1; ++s) {
    if (s < nk) load_stage(s, s);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int kt = 0; kt < nk; ++kt) {
    asm volatile("cp.async.wait_group %0;" ::"n"(GSTAGES - 2) : "memory");
    __syncthreads();
    if (kt + GSTAGES - 1 < nk) load_stage((kt + GSTAGES - 1) % GSTAGES, kt + GSTAGES - 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    const double *as = As + (size_t)(kt % GSTAGES) * A_STAGE + wm * 64 + g;
    const double *bs = Bs + (size_t)(kt % GSTAGES) * B_STAGE + (wn * 32 + g) * BS_LD + t;
    double bf[4][4];
#pragma unroll
    for (int n8 = 0; n8 < 4; ++n8)
#pragma unroll
      for (int i = 0; i < 4; ++i) bf[n8][i] = bs[n8 * 8 * BS_LD + 4 * i];
#pragma unroll
    for (int m16 = 0; m16 < 4; ++m16) {
      double af[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) af[i] = as[(t + 4 * (i >> 1)) * AS_LD + m16 * 16 + 8 * (i & 1)];
#pragma unroll
      for (int n8 = 0; n8 < 4; ++n8) {
        asm volatile(
            "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
            "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
            : "+d"(acc[m16][n8][0]), "+d"(acc[m16][n8][1]), "+d"(acc[m16][n8][2]), "+d"(acc[m16][n8][3])
            : "d"(af[0]), "d"(af[1]), "d"(af[2]), "d"(af[3]), "d"(af[4]), "d"(af[5]), "d"(af[6]), "d"(af[7]),
              "d"(bf[n8][0]), "d"(bf[n8][1]), "d"(bf[n8][2]), "d"(bf[n8][3]));
      }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");

  // fused epilogue: c0,c1 → row g, cols 2t,2t+1; c2,c3 → row g+8 (of each 16×8 fragment)
  for (int s = 0; s <= ne; ++s) {
    double w[4][2];
#pragma unroll
    for (int m16 = 0; m16 < 4; ++m16)
#pragma unroll
      for (int h = 0; h < 2; ++h)
        w[m16][h] = (s == 0) ? 0.0 : YE[i0 + wm * 64 + m16 * 16 + g + 8 * h + (long long)(s - 1) * ld];
#pragma unroll
    for (int n8 = 0; n8 < 4; ++n8) {
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        double v = 0.0;
#pragma unroll
        for (int m16 = 0; m16 < 4; ++m16) {
          const double y0 = acc[m16][n8][cc], y1 = acc[m16][n8][cc + 2];
          v = fma(y0, (s == 0) ? y0 : w[m16][0], v);
          v = fma(y1, (s == 0) ? y1 : w[m16][1], v);
        }
        v += __shfl_xor_sync(0xffffffffu, v, 4);
        v += __shfl_xor_sync(0xffffffffu, v, 8);
        v += __shfl_xor_sync(0xffffffffu, v, 16);
        if (g == 0) red[wm][wn * 32 + n8 * 8 + 2 * t + cc] = v;
      }
    }
    __syncthreads();
    if (tid < GT) partial[((long long)mt * (1 + ne) + s) * nbpad + t0 + tid] = red[0][tid] + red[1][tid];
    __syncthreads();
  }
}

// ---- per-target epilogue: reduce the partials over the row tiles, then the e×e algebra ----
struct GDual {
  const double *dmean;  // w·b(t) per target of the batch
  double beta[GSK_MAX_DRIFT_TERMS];
};
__global__ void global_epilogue_kernel(const double *__restrict__ partial, int nmt, int ne, long long nbpad,
                                       int nbatch, const double *__restrict__ GEE, GskEstimator es, GskTargets tg,
                                       double sill, unsigned flags, long long first, GskOut out, GDual dual) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nbatch) return;
  double g[2 + GSK_MAX_DRIFT_TERMS];
  for (int s = 0; s <= ne; ++s) {
    double v = 0.0;
    for (int mt = 0; mt < nmt; ++mt) v += partial[((long long)mt * (1 + ne) + s) * nbpad + t];
    g[s] = v;
  }
  const double gbb = g[0], gbz = g[1];
  const int c = es.nterms;
  double mu, s2;
  (void)gbz;  // the Gram form of the mean (Gbz − Gfz·ν) is superseded by the refined dual weights
  if (c == 0) {
    mu = es.sk_mean + dual.dmean[t];
    s2 = sill - gbb;
  } else {
    double f0[GSK_MAX_DRIFT_TERMS], nu[GSK_MAX_DRIFT_TERMS], Lf[GSK_MAX_DRIFT_TERMS][GSK_MAX_DRIFT_TERMS];
    double tc[3] = {0.0, 0.0, 0.0};
    long long lin = first + t;
    if (tg.is_grid) {
      long long rem = lin;
      for (int d = 0; d < tg.dim; ++d) {
        long long cc = rem % tg.gdim[d];
        rem /= tg.gdim[d];
        tc[d] = gsk_cell_center(tg.gorg[d], tg.gsp[d], cc);
      }
    } else {
      for (int d = 0; d < tg.dim; ++d) tc[d] = tg.pts[d][lin];
    }
    for (int j = 0; j < c; ++j)
      f0[j] = (es.kind == GSK_EST_ORDINARY)
                  ? 1.0
                  : gsk_ipow(tc[0], es.exps[j][0]) * gsk_ipow(tc[1], es.exps[j][1]) * gsk_ipow(tc[2], es.exps[j][2]);
    // Gff = GEE[1+a][1+b], Gfz = GEE[1+a][0]
    for (int j = 0; j < c; ++j) {
      double d = GEE[(1 + j) * ne + 1 + j];
      for (int p = 0; p < j; ++p) d -= Lf[j][p] * Lf[j][p];
      d = sqrt(d);
      Lf[j][j] = d;
      for (int i = j + 1; i < c; ++i) {
        double s = GEE[(1 + i) * ne + 1 + j];
        for (int p = 0; p < j; ++p) s -= Lf[i][p] * Lf[j][p];
        Lf[i][j] = s / d;
      }
    }
    for (int j = 0; j < c; ++j) {
      double s = g[2 + j] - f0[j];
      for (int p = 0; p < j; ++p) s -= Lf[j][p] * nu[p];
      nu[j] = s / Lf[j][j];
    }
    for (int j = c - 1; j >= 0; --j) {
      double s = nu[j];
      for (int p = j + 1; p < c; ++p) s -= Lf[p][j] * nu[p];
      nu[j] = s / Lf[j][j];
    }
    double mb = 0.0, mf = 0.0, mbeta = 0.0;
    for (int j = 0; j < c; ++j) {
      mb += g[2 + j] * nu[j];
      mf += f0[j] * nu[j];
      mbeta += dual.beta[j] * f0[j];
    }
    mu = dual.dmean[t] + mbeta;  // w·b(t) + β·f₀(t)
    s2 = sill - (gbb - mb + mf);
  }
  if (flags & GSK_FLAG_CLAMP_VARIANCE) s2 = (s2 > 0.0 || s2 != s2) ? s2 : 0.0;
  if (flags & GSK_FLAG_SQRT_ROUNDTRIP) { double sd = sqrt(s2); s2 = sd * sd; }
  gsk_store_result(out, t, mu, s2);
}

// ---- dual weights of the mean (plan time) -------------------------------------------------------------------
// mean(t) = [z;0]ᵀ K⁻¹ [b(t); f₀(t)] = w·b(t) + β·f₀(t) with K [w; β] = [z; 0]: the mean needs only a dot product with the
// right-hand side once (w, β) are known. They are obtained from the factor and then REFINED with residuals accumulated
// in double-double arithmetic (error-free products and sums), which brings w to ~1 ulp of the solution of the assembled
// system — the Gram form Gbz − Gfz·ν of the same mean carries ~cond(C)·eps (2e-9 on the Gaussian C1 system, round 1).
__device__ __forceinline__ void dd_add_prod(double &hi, double &lo, double a, double b) {
  const double p = a * b, pe = fma(a, b, -p);  // a·b = p + pe exactly
  const double s = hi + p, bb = s - hi;
  const double se = (hi - (s - bb)) + (p - bb);  // hi + p = s + se exactly
  hi = s;
  lo += se + pe;
}

// out[j] = Σ_{i>=j} X[i, j]·v[i]  (Xᵀ v, X lower triangular, column-major): one warp per column
__global__ void xt_matvec_kernel(const double *__restrict__ X, long long ld, long long np, const double *__restrict__ v,
                                 double *__restrict__ out) {
  const long long j = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= np) return;
  double s = 0.0;
  for (long long i = j + lane; i < np; i += 32) s = fma(X[i + j * ld], v[i], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[j] = s;
}

// r[i] = z[i] − Σ_j C[i, j]·w[j] − Σ_t F[i, t]·β[t] in double-double, C re-evaluated exactly as assemble_kernel does
template <int VK>
__global__ void dual_residual_kernel(GArgs g, const double *__restrict__ E, int ne, const double *__restrict__ w,
                                     GskEstimator es, const double *__restrict__ beta, double *__restrict__ r) {
  const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= g.np) return;
  if (i >= g.n) {  // padded rows: identity block, zero right-hand side
    if (lane == 0) r[i] = -w[i];
    return;
  }
  const double4 a = g.rec[i];
  double hi = 0.0, lo = 0.0;
  for (long long j = lane; j < g.n; j += 32) {
    double c;
    if (j == i) c = g.vg.sill;
    else {
      const double4 b = g.rec[j];
      const double dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
      c = gsk_cov<VK>(g.vg, fma(dz, dz, fma(dy, dy, dx * dx)));
    }
    dd_add_prod(hi, lo, -c, w[j]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {  // combine the lanes' double-double partial sums
    const double oh = __shfl_xor_sync(0xffffffffu, hi, o), ol = __shfl_xor_sync(0xffffffffu, lo, o);
    const double s = hi + oh, bb = s - hi;
    lo += ((hi - (s - bb)) + (oh - bb)) + ol;
    hi = s;
  }
  if (lane == 0) {
    dd_add_prod(hi, lo, 1.0, E[i]);  // + z_i (E column 0 holds z − μ for Simple Kriging)
    for (int t = 0; t < es.nterms; ++t) dd_add_prod(hi, lo, -E[i + (long long)(1 + t) * g.np], beta[t]);
    r[i] = hi + lo;
  }
}

// out[t] = Σ_i A[i + t·ld]·v[i] in double-double (t < nt columns of length np): one CTA per column
__global__ void cols_dot_dd_kernel(const double *__restrict__ A, long long ld, long long np, const double *__restrict__ v,
                                   double *__restrict__ out) {
  __shared__ double sh[256], sl[256];
  const double *col = A + (long long)blockIdx.x * ld;
  double hi = 0.0, lo = 0.0;
  for (long long i = threadIdx.x; i < np; i += 256) dd_add_prod(hi, lo, col[i], v[i]);
  sh[threadIdx.x] = hi;
  sl[threadIdx.x] = lo;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      const double a = sh[threadIdx.x], b = sh[threadIdx.x + o];
      const double s = a + b, bb = s - a;
      sl[threadIdx.x] += ((a - (s - bb)) + (b - bb)) + sl[threadIdx.x + o];
      sh[threadIdx.x] = s;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sh[0] + sl[0];
}

// v[i] = y[i] − Σ_t YF[i, t]·d[t]   (YF = columns 1… of Y_E)
__global__ void sub_cols_kernel(const double *__restrict__ y, const double *__restrict__ YE, long long np, int nt,
                                const double *__restrict__ d, double *__restrict__ v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= np) return;
  double s = y[i];
  for (int t = 0; t < nt; ++t) s = fma(-YE[i + (long long)(1 + t) * np], d[t], s);
  v[i] = s;
}

__global__ void axpy_kernel(double *__restrict__ w, const double *__restrict__ d, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) w[i] += d[i];
}

// dmean[t] = Σ_i w[i]·B[i + t·np]: one warp per target column of the batch
__global__ void dual_mean_kernel(const double *__restrict__ Bm, long long np, int nbatch, const double *__restrict__ w,
                                 double *__restrict__ dmean) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= nbatch) return;
  const double *col = Bm + (long long)t * np;
  double s0 = 0.0, s1 = 0.0;
  for (long long i = lane; i < np; i += 64) {
    s0 = fma(col[i], w[i], s0);
    if (i + 32 < np) s1 = fma(col[i + 32], w[i + 32], s1);
  }
  double s = s0 + s1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) dmean[t] = s;
}

__global__ void fill_int_kernel(int *p, long long n, int v) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---- leave-one-out (Dubrule 1983) ------------------------------------------------------------------------------
// With Q the upper-left n×n block of K⁻¹, K = [C F; Fᵀ 0], sample i left out has the residual z_i − ẑ_{−i} = w_i / Q_ii
// and the kriging variance 1 / Q_ii, where (w, β) = K⁻¹[z; 0] are the resident dual weights. With C⁻¹ = XᵀX (X = L⁻¹,
// lower triangular) and Y_F = X F:  Q_ii = Σ_{r>=i} X[r,i]² − W_i G_FF⁻¹ W_iᵀ,  W_i = Σ_{r>=i} X[r,i] Y_F[r,:].
// Pass 1 reads the lower triangle of X once: CTA (column block of 64, row chunk of LOO_RCH rows) — every warp owns 8
// columns, each a contiguous stretch of X, read by its 32 lanes in 256-byte rows, four loads in flight per lane — and
// writes per-chunk partial sums; pass 2 reduces the chunks of a column in a fixed order (deterministic) and applies the
// e×e algebra and the variance flags.
constexpr int LOO_RCH = 1024;

__global__ void __launch_bounds__(256) loo_colsum_kernel(const double *__restrict__ X, long long np, long long n,
                                                         const double *__restrict__ YE, int c, long long cb0,
                                                         double *__restrict__ partial) {
  const long long jb = cb0 + blockIdx.x;
  const long long r0 = jb * NB + (long long)blockIdx.y * LOO_RCH;
  if (r0 >= n) return;
  const long long r1 = (r0 + LOO_RCH < n) ? r0 + LOO_RCH : n;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ns = 1 + c;
  for (int cc = 0; cc < 8; ++cc) {
    const long long i = jb * NB + warp * 8 + cc;
    if (i >= n) break;
    const double *col = X + i * np;
    double s = 0.0, wt[GSK_MAX_DRIFT_TERMS];
#pragma unroll
    for (int t = 0; t < GSK_MAX_DRIFT_TERMS; ++t) wt[t] = 0.0;
    long long r = ((r0 > i) ? r0 : i) + lane;
    for (; r + 96 < r1; r += 128) {
      const double x0 = col[r], x1 = col[r + 32], x2 = col[r + 64], x3 = col[r + 96];
      s = fma(x0, x0, s); s = fma(x1, x1, s); s = fma(x2, x2, s); s = fma(x3, x3, s);
#pragma unroll
      for (int t = 0; t < GSK_MAX_DRIFT_TERMS; ++t)
        if (t < c) {
          const double *yf = YE + (long long)(1 + t) * np + r;
          wt[t] = fma(x0, yf[0], wt[t]); wt[t] = fma(x1, yf[32], wt[t]);
          wt[t] = fma(x2, yf[64], wt[t]); wt[t] = fma(x3, yf[96], wt[t]);
        }
    }
    for (; r < r1; r += 32) {
      const double x = col[r];
      s = fma(x, x, s);
#pragma unroll
      for (int t = 0; t < GSK_MAX_DRIFT_TERMS; ++t)
        if (t < c) wt[t] = fma(x, YE[(long long)(1 + t) * np + r], wt[t]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
#pragma unroll
    for (int t = 0; t < GSK_MAX_DRIFT_TERMS; ++t)
      if (t < c)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wt[t] += __shfl_xor_sync(0xffffffffu, wt[t], o);
    if (lane == 0) {
      double *pp = partial + (long long)blockIdx.y * ns * np + i;
      pp[0] = s;
#pragma unroll
      for (int t = 0; t < GSK_MAX_DRIFT_TERMS; ++t)
        if (t < c) pp[(long long)(1 + t) * np] = wt[t];
    }
  }
}

__global__ void loo_epilogue_kernel(const double *__restrict__ partial, long long np, long long n, int c,
                                    const double *__restrict__ GEE, int ne, const double *__restrict__ w,
                                    const double4 *__restrict__ rec, long long first, long long count, unsigned flags,
                                    GskOut out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const long long i = first + t;
  const int nq = (int)((n - (i / NB) * NB + LOO_RCH - 1) / LOO_RCH);
  const int ns = 1 + c;
  double d = 0.0, y[GSK_MAX_DRIFT_TERMS];
  for (int j = 0; j < c; ++j) y[j] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double *pp = partial + (long long)q * ns * np + i;
    d += pp[0];
    for (int j = 0; j < c; ++j) y[j] += pp[(long long)(1 + j) * np];
  }
  // Q_ii = d − W G_FF⁻¹ Wᵀ = d − ‖L_F⁻¹ Wᵀ‖² with G_FF = L_F L_Fᵀ (rows/cols 1… of G_EE)
  double Lf[GSK_MAX_DRIFT_TERMS][GSK_MAX_DRIFT_TERMS];
  for (int j = 0; j < c; ++j) {
    double dd = GEE[(1 + j) * ne + 1 + j];
    for (int p = 0; p < j; ++p) dd -= Lf[j][p] * Lf[j][p];
    dd = sqrt(dd);
    Lf[j][j] = dd;
    for (int a = j + 1; a < c; ++a) {
      double s = GEE[(1 + a) * ne + 1 + j];
      for (int p = 0; p < j; ++p) s -= Lf[a][p] * Lf[j][p];
      Lf[a][j] = s / dd;
    }
  }
  double proj = 0.0;
  for (int j = 0; j < c; ++j) {
    double s = y[j];
    for (int p = 0; p < j; ++p) s -= Lf[j][p] * y[p];
    y[j] = s / Lf[j][j];
    proj = fma(y[j], y[j], proj);
  }
  const double Q = d - proj;
  const double mu = rec[i].w - w[i] / Q;
  double s2 = 1.0 / Q;
  if (flags & GSK_FLAG_CLAMP_VARIANCE) s2 = (s2 > 0.0 || s2 != s2) ? s2 : 0.0;
  if (flags & GSK_FLAG_SQRT_ROUNDTRIP) { double sd = sqrt(s2); s2 = sd * sd; }
  gsk_store_result(out, t, mu, s2);
}

// ---- gsk_krige_columns ---------------------------------------------------------------------------------------
// E's value column from column j of the n × m sample-major values (− μ for Simple Kriging); padded rows stay 0
__global__ void set_e_column_kernel(const double *__restrict__ Z, int m, int j, long long n, double shift,
                                    double *__restrict__ E) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) E[i] = Z[(size_t)i * m + j] - shift;
}

// Per-column means of a target batch from the dual weights: mean[t, j] = Σ_i B[i, t]·W[i, j] + β_j·f₀(t) (+ μ for
// Simple Kriging) — the same dual form as the single-column mean (dual_mean_kernel + global_epilogue_kernel), as one
// GEMM Bᵀ W on the FP64 tensor path. One warp per 16 targets × 8 columns, mma.m16n8k16 over the padded sample axis
// (np is a multiple of 16; the batch's padded target columns of B and the padded columns of W are zero). Every output
// element sees only its own row of Bᵀ and column of W, in the same k order, so a column's result does not depend on
// m or on its position.
__global__ void __launch_bounds__(128) cols_mean_kernel(const double *__restrict__ Bm, long long np, int nb,
                                                        const double *__restrict__ W, int m, int m8,
                                                        const double *__restrict__ beta, GskEstimator es, GskTargets tg,
                                                        long long first, double *__restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
  const long long t0 = (long long)blockIdx.x * 16;
  const int j0 = (blockIdx.y * 4 + warp) * 8;
  if (j0 >= m8) return;
  const double *a0 = Bm + (t0 + g) * np + t4, *a1 = a0 + 8 * np;
  const double *b0 = W + (long long)(j0 + g) * np + t4;
  double d[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long k0 = 0; k0 < np; k0 += 16) {
    const double af[8] = {a0[k0], a1[k0], a0[k0 + 4], a1[k0 + 4], a0[k0 + 8], a1[k0 + 8], a0[k0 + 12], a1[k0 + 12]};
    const double bf[4] = {b0[k0], b0[k0 + 4], b0[k0 + 8], b0[k0 + 12]};
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7,%8,%9,%10,%11}, "
        "{%12,%13,%14,%15}, {%0,%1,%2,%3};"
        : "+d"(d[0]), "+d"(d[1]), "+d"(d[2]), "+d"(d[3])
        : "d"(af[0]), "d"(af[1]), "d"(af[2]), "d"(af[3]), "d"(af[4]), "d"(af[5]), "d"(af[6]), "d"(af[7]), "d"(bf[0]),
          "d"(bf[1]), "d"(bf[2]), "d"(bf[3]));
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const long long t = t0 + g + 8 * h;
    if (t >= nb) continue;
    double f0[GSK_MAX_DRIFT_TERMS];
    if (es.nterms > 0) {
      double tc[3];
      gsk_target_center(tg, first + t, tc);
      for (int q = 0; q < es.nterms; ++q)
        f0[q] = (es.kind == GSK_EST_ORDINARY)
                    ? 1.0
                    : gsk_ipow(tc[0], es.exps[q][0]) * gsk_ipow(tc[1], es.exps[q][1]) * gsk_ipow(tc[2], es.exps[q][2]);
    }
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const int j = j0 + 2 * t4 + cc;
      if (j >= m) continue;
      double mu = d[2 * h + cc];
      if (es.kind == GSK_EST_SIMPLE) mu = es.sk_mean + mu;
      else {
        double mb = 0.0;
        for (int q = 0; q < es.nterms; ++q) mb += beta[j * GSK_MAX_DRIFT_TERMS + q] * f0[q];
        mu = mu + mb;
      }
      out[t * m + j] = mu;
    }
  }
}

}  // namespace

struct GlobalPlan {
  long long n = 0, np = 0;
  int ne = 0;
  double *A = nullptr;     // L (lower) after factorisation
  double *X = nullptr;     // Linv
  double *Dinv = nullptr;  // inverses of the diagonal blocks
  double *E = nullptr, *YE = nullptr, *GEE = nullptr;
  double *Bm = nullptr, *partial = nullptr;
  double *w = nullptr;       // dual weights of the mean (np)
  double *tmp = nullptr;     // 3·np + 32 scratch doubles of the refinement
  double *dmean = nullptr;   // w·b(t) of a batch
  double beta[GSK_MAX_DRIFT_TERMS] = {};
  long long batch = 0;
};

namespace {
// c×c SPD solve on the host in long double (c <= 10): G x = rhs
void host_spd_solve(int c, const double *G, int ldg, const long double *rhs, long double *x) {
  long double A[GSK_MAX_DRIFT_TERMS][GSK_MAX_DRIFT_TERMS + 1];
  for (int i = 0; i < c; ++i) {
    for (int j = 0; j < c; ++j) A[i][j] = G[i * ldg + j];
    A[i][c] = rhs[i];
  }
  for (int k = 0; k < c; ++k) {
    int piv = k;
    for (int i = k + 1; i < c; ++i)
      if (fabsl(A[i][k]) > fabsl(A[piv][k])) piv = i;
    for (int j = 0; j <= c; ++j) std::swap(A[k][j], A[piv][j]);
    for (int i = k + 1; i < c; ++i) {
      const long double f = A[i][k] / A[k][k];
      for (int j = k; j <= c; ++j) A[i][j] -= f * A[k][j];
    }
  }
  for (int i = c - 1; i >= 0; --i) {
    long double s = A[i][c];
    for (int j = i + 1; j < c; ++j) s -= A[i][j] * x[j];
    x[i] = s / A[i][i];
  }
}

// (w, β) = K⁻¹ [z; 0] from the factor, then two refinement steps with double-double residuals
int global_dual_weights(gsk_ctx *ctx) {
  GlobalPlan *g = ctx->gplan;
  cudaStream_t st = ctx->stream;
  const long long np = g->np;
  const int c = ctx->es.nterms, ne = g->ne;
  GArgs ga{ctx->d_rec_orig, g->n, np, ctx->vg, ctx->prob.dim};
  double *y = g->tmp, *v = g->tmp + np, *r = g->tmp + 2 * np, *small = g->tmp + 3 * np;  // small: 32 doubles
  const unsigned gw = (unsigned)((np + 7) / 8), gt = (unsigned)((np + 255) / 256);
  double hGEE[(1 + GSK_MAX_DRIFT_TERMS) * (1 + GSK_MAX_DRIFT_TERMS)];
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(hGEE, g->GEE, sizeof(double) * ne * ne, cudaMemcpyDeviceToHost, st));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  const double *Gff = hGEE + ne + 1;  // rows/cols 1… of G_EE
  long double beta[GSK_MAX_DRIFT_TERMS] = {}, rhs[GSK_MAX_DRIFT_TERMS], d[GSK_MAX_DRIFT_TERMS];
  double hb[GSK_MAX_DRIFT_TERMS] = {};
  // first solution: β = Gff⁻¹ Gfz,  w = L⁻ᵀ (Y_z − Y_F β)
  for (int j = 0; j < c; ++j) rhs[j] = hGEE[(1 + j) * ne];
  if (c > 0) host_spd_solve(c, Gff, ne, rhs, beta);
  for (int j = 0; j < c; ++j) hb[j] = (double)beta[j];
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(small, hb, sizeof(double) * GSK_MAX_DRIFT_TERMS, cudaMemcpyHostToDevice, st));
  sub_cols_kernel<<<gt, 256, 0, st>>>(g->YE, g->YE, np, c, small, v);
  xt_matvec_kernel<<<gw, 256, 0, st>>>(g->X, np, np, v, g->w);
  for (int it = 0; it < 2; ++it) {
    // residuals: r_w = z − C w − F β (double-double), r_β = −Fᵀ w
    switch (ctx->vg.kind) {
      case GSK_VARIO_GAUSSIAN: dual_residual_kernel<GSK_VARIO_GAUSSIAN><<<gw, 256, 0, st>>>(ga, g->E, ne, g->w, ctx->es, small, r); break;
      case GSK_VARIO_SPHERICAL: dual_residual_kernel<GSK_VARIO_SPHERICAL><<<gw, 256, 0, st>>>(ga, g->E, ne, g->w, ctx->es, small, r); break;
      default: dual_residual_kernel<GSK_VARIO_EXPONENTIAL><<<gw, 256, 0, st>>>(ga, g->E, ne, g->w, ctx->es, small, r); break;
    }
    double hrb[GSK_MAX_DRIFT_TERMS] = {}, ht[GSK_MAX_DRIFT_TERMS] = {};
    if (c > 0) {
      cols_dot_dd_kernel<<<c, 256, 0, st>>>(g->E + np, np, np, g->w, small + 16);  // Fᵀ w
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(hrb, small + 16, sizeof(double) * c, cudaMemcpyDeviceToHost, st));
    }
    // δ: y = L⁻¹ r_w;  δβ = Gff⁻¹ (Y_Fᵀ y + Fᵀw);  δw = L⁻ᵀ (y − Y_F δβ)
    linv_times_e_kernel<<<gw, 256, 0, st>>>(g->X, np, np, r, 1, y);
    if (c > 0) {
      cols_dot_dd_kernel<<<c, 256, 0, st>>>(g->YE + np, np, np, y, small + 16);
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ht, small + 16, sizeof(double) * c, cudaMemcpyDeviceToHost, st));
      GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
      for (int j = 0; j < c; ++j) rhs[j] = (long double)ht[j] + (long double)hrb[j];  // t − r_β with r_β = −Fᵀw
      host_spd_solve(c, Gff, ne, rhs, d);
      double hd[GSK_MAX_DRIFT_TERMS] = {};
      for (int j = 0; j < c; ++j) { hd[j] = (double)d[j]; beta[j] += d[j]; hb[j] = (double)beta[j]; }
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(small + 16, hd, sizeof(double) * GSK_MAX_DRIFT_TERMS, cudaMemcpyHostToDevice, st));
      sub_cols_kernel<<<gt, 256, 0, st>>>(y, g->YE, np, c, small + 16, v);
      xt_matvec_kernel<<<gw, 256, 0, st>>>(g->X, np, np, v, r);
      GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));  // hd leaves scope
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(small, hb, sizeof(double) * GSK_MAX_DRIFT_TERMS, cudaMemcpyHostToDevice, st));
    } else {
      xt_matvec_kernel<<<gw, 256, 0, st>>>(g->X, np, np, y, r);
    }
    axpy_kernel<<<gt, 256, 0, st>>>(g->w, r, np);
    GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  }
  for (int j = 0; j < GSK_MAX_DRIFT_TERMS; ++j) g->beta[j] = (j < c) ? (double)beta[j] : 0.0;
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return GSK_OK;
}
}  // namespace

void gsk_global_free(gsk_ctx *ctx) {
  GlobalPlan *g = ctx->gplan;
  if (!g) return;
  delete g;  // the device buffers are cached in the context (gsk_buf)
  ctx->gplan = nullptr;
}

int gsk_global_plan(gsk_ctx *ctx, const double *hx, const double *hy, const double *hz, const double *hv) {
  const long long n = ctx->prob.n_samples;
  const int dim = ctx->prob.dim;
  cudaStream_t st = ctx->stream;
  GlobalPlan *g = new GlobalPlan();
  ctx->gplan = g;
  g->n = n;
  g->np = (n + GT - 1) / GT * GT;  // multiple of the GEMM tile (and of the factorisation block)
  g->ne = 1 + ctx->es.nterms;
  const long long np = g->np;
  const int nblk = (int)(np / NB);

  // samples → {x,y,z,value} records
  std::vector<double4> rec((size_t)n);
  for (long long i = 0; i < n; ++i) {
    rec[(size_t)i] = make_double4(hx[i], dim > 1 ? hy[i] : 0.0, dim > 2 ? hz[i] : 0.0, hv[i]);
    if (!std::isfinite(rec[(size_t)i].x) || !std::isfinite(rec[(size_t)i].y) || !std::isfinite(rec[(size_t)i].z)) {
      ctx->err = "sample coordinates must be finite";
      return GSK_ERR_INVALID;
    }
  }
  int rc;
  if ((rc = gsk_buf(ctx, BUF_REC_ORIG, sizeof(double4) * (size_t)n, (void **)&ctx->d_rec_orig)) != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_rec_orig, rec.data(), sizeof(double4) * (size_t)n, cudaMemcpyHostToDevice, st));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));

  if ((rc = gsk_buf(ctx, BUF_G_A, sizeof(double) * (size_t)np * np, (void **)&g->A)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_X, sizeof(double) * (size_t)np * np, (void **)&g->X)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_DINV, sizeof(double) * (size_t)nblk * NB * NB, (void **)&g->Dinv)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_E, sizeof(double) * (size_t)np * g->ne, (void **)&g->E)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_YE, sizeof(double) * (size_t)np * g->ne, (void **)&g->YE)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_GEE, sizeof(double) * (size_t)g->ne * g->ne, (void **)&g->GEE)) != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaMemsetAsync(g->X, 0, sizeof(double) * (size_t)np * np, st));

  GArgs ga{ctx->d_rec_orig, n, np, ctx->vg, dim};
  {
    dim3 grid((unsigned)((np + 255) / 256), (unsigned)np);
    switch (ctx->vg.kind) {
      case GSK_VARIO_GAUSSIAN: assemble_kernel<GSK_VARIO_GAUSSIAN><<<grid, 256, 0, st>>>(ga, g->A); break;
      case GSK_VARIO_SPHERICAL: assemble_kernel<GSK_VARIO_SPHERICAL><<<grid, 256, 0, st>>>(ga, g->A); break;
      default: assemble_kernel<GSK_VARIO_EXPONENTIAL><<<grid, 256, 0, st>>>(ga, g->A); break;
    }
  }
  // blocked right-looking Cholesky
  for (int jb = 0; jb < nblk; ++jb) {
    const long long j0 = (long long)jb * NB;
    potrf_diag_kernel<<<1, 64, 0, st>>>(g->A, np, j0, g->Dinv + (size_t)jb * NB * NB);
    const int nrem = nblk - jb - 1;
    if (nrem > 0) {
      trsm_panel_kernel<<<nrem, 256, 0, st>>>(g->A, np, j0, g->Dinv + (size_t)jb * NB * NB);
      syrk_kernel<<<(unsigned)((long long)nrem * (nrem + 1) / 2), 256, 0, st>>>(g->A, np, j0, nrem);
    }
  }
  // Linv, block row by block row
  GSK_CUDA_CHECK(ctx, cudaFuncSetAttribute(linv_row_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LINV_SMEM));
  for (int bi = 0; bi < nblk; ++bi) linv_row_kernel<<<bi + 1, 256, LINV_SMEM, st>>>(g->A, g->X, np, bi, g->Dinv);
  // E, Y_E, G_EE
  build_e_kernel<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(ga, ctx->es, g->E);
  linv_times_e_kernel<<<(unsigned)((np + 7) / 8), 256, 0, st>>>(g->X, np, np, g->E, g->ne, g->YE);
  gram_ee_kernel<<<1, 256, 0, st>>>(g->YE, np, g->ne, g->GEE);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  if ((rc = gsk_buf(ctx, BUF_G_W, sizeof(double) * (size_t)np, (void **)&g->w)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_TMP, sizeof(double) * (size_t)(3 * np + 32), (void **)&g->tmp)) != GSK_OK) return rc;
  if ((rc = global_dual_weights(ctx)) != GSK_OK) return rc;

  // batch of targets per GEMM: bound B to ~2 GB (the buffers are sized in gsk_global_execute)
  long long batch = (long long)((2.0e9 / 8.0) / (double)np);
  batch = std::max<long long>(GT, std::min<long long>(batch, 32768) / GT * GT);
  g->batch = batch;
  GSK_CUDA_CHECK(ctx, cudaFuncSetAttribute(ygemm_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)YGEMM_SMEM));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  return GSK_OK;
}

// new sample values in rec_orig (gsk_update_values): only E's value column changes, hence Y_E = L⁻¹E and G_EE
int gsk_global_update_values(gsk_ctx *ctx) {
  GlobalPlan *g = ctx->gplan;
  if (!g) { ctx->err = "global plan missing"; return GSK_ERR_STATE; }
  cudaStream_t st = ctx->stream;
  const long long np = g->np;
  GArgs ga{ctx->d_rec_orig, g->n, np, ctx->vg, ctx->prob.dim};
  build_e_kernel<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(ga, ctx->es, g->E);
  linv_times_e_kernel<<<(unsigned)((np + 7) / 8), 256, 0, st>>>(g->X, np, np, g->E, g->ne, g->YE);
  gram_ee_kernel<<<1, 256, 0, st>>>(g->YE, np, g->ne, g->GEE);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return global_dual_weights(ctx);
}

int gsk_global_column_weights(gsk_ctx *ctx, const double *d_z, int m) {
  GlobalPlan *g = ctx->gplan;
  if (!g) { ctx->err = "global plan missing"; return GSK_ERR_STATE; }
  cudaStream_t st = ctx->stream;
  const long long np = g->np;
  const double shift = (ctx->es.kind == GSK_EST_SIMPLE) ? ctx->es.sk_mean : 0.0;
  const int m8 = (m + 7) / 8 * 8;
  int rc;
  if ((rc = gsk_buf(ctx, BUF_C_GW, sizeof(double) * (size_t)np * m8, (void **)&ctx->cols.gw)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_C_GBETA, sizeof(double) * (size_t)m * GSK_MAX_DRIFT_TERMS, (void **)&ctx->cols.gbeta)) != GSK_OK)
    return rc;
  if (m8 > m)  // padding columns of the column-mean GEMM
    GSK_CUDA_CHECK(ctx, cudaMemsetAsync(ctx->cols.gw + (size_t)m * np, 0, sizeof(double) * (size_t)(m8 - m) * np, st));
  std::vector<double> hbeta((size_t)m * GSK_MAX_DRIFT_TERMS);
  // column by column through the plan's own refinement (gsk_global_update_values without the record upload): only
  // E's value column, its row of Y_E and of G_EE change
  for (int j = 0; j < m; ++j) {
    set_e_column_kernel<<<(unsigned)((g->n + 255) / 256), 256, 0, st>>>(d_z, m, j, g->n, shift, g->E);
    linv_times_e_kernel<<<(unsigned)((np + 7) / 8), 256, 0, st>>>(g->X, np, np, g->E, 1, g->YE);
    gram_ee_kernel<<<1, 256, 0, st>>>(g->YE, np, g->ne, g->GEE);
    GSK_CUDA_CHECK(ctx, cudaGetLastError());
    if ((rc = global_dual_weights(ctx)) != GSK_OK) return rc;
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->cols.gw + (size_t)j * np, g->w, sizeof(double) * (size_t)np,
                                        cudaMemcpyDeviceToDevice, st));
    for (int q = 0; q < GSK_MAX_DRIFT_TERMS; ++q) hbeta[(size_t)j * GSK_MAX_DRIFT_TERMS + q] = g->beta[q];
  }
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->cols.gbeta, hbeta.data(), sizeof(double) * hbeta.size(), cudaMemcpyHostToDevice, st));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));  // hbeta leaves scope
  return GSK_OK;
}

int gsk_global_execute(gsk_ctx *ctx, long long first, long long count, int *d_nn, int *launches) {
  GlobalPlan *g = ctx->gplan;
  if (!g) { ctx->err = "global plan missing"; return GSK_ERR_STATE; }
  cudaStream_t st = ctx->stream;
  const long long np = g->np;
  const int nblk = (int)(np / NB);
  GArgs ga{ctx->d_rec_orig, g->n, np, ctx->vg, ctx->prob.dim};
  {
    const long long bmax = std::min<long long>(g->batch, (count + GT - 1) / GT * GT);
    int rc;
    if ((rc = gsk_buf(ctx, BUF_G_BM, sizeof(double) * (size_t)np * bmax, (void **)&g->Bm)) != GSK_OK) return rc;
    if ((rc = gsk_buf(ctx, BUF_G_PARTIAL, sizeof(double) * (size_t)(np / GT) * (1 + g->ne) * g->batch, (void **)&g->partial)) != GSK_OK) return rc;
    if ((rc = gsk_buf(ctx, BUF_G_DMEAN, sizeof(double) * (size_t)g->batch, (void **)&g->dmean)) != GSK_OK) return rc;
  }
  GDual dual{};
  dual.dmean = g->dmean;
  for (int j = 0; j < GSK_MAX_DRIFT_TERMS; ++j) dual.beta[j] = g->beta[j];
  for (long long off = 0; off < count; off += g->batch) {
    const int nb = (int)std::min<long long>(g->batch, count - off);
    const int nbp = (nb + GT - 1) / GT * GT;
    if (nbp > nb)  // zero the padded target columns so the GEMM reads defined data
      GSK_CUDA_CHECK(ctx, cudaMemsetAsync(g->Bm + (size_t)nb * np, 0, sizeof(double) * (size_t)(nbp - nb) * np, st));
    dim3 grid((unsigned)((np + 255) / 256), (unsigned)nb);
    switch (ctx->vg.kind) {
      case GSK_VARIO_GAUSSIAN:
        rhs_kernel<GSK_VARIO_GAUSSIAN><<<grid, 256, 0, st>>>(ga, ctx->tg, ctx->d_sup, ctx->prob.n_support, first + off, nb, g->Bm);
        break;
      case GSK_VARIO_SPHERICAL:
        rhs_kernel<GSK_VARIO_SPHERICAL><<<grid, 256, 0, st>>>(ga, ctx->tg, ctx->d_sup, ctx->prob.n_support, first + off, nb, g->Bm);
        break;
      default:
        rhs_kernel<GSK_VARIO_EXPONENTIAL><<<grid, 256, 0, st>>>(ga, ctx->tg, ctx->d_sup, ctx->prob.n_support, first + off, nb, g->Bm);
        break;
    }
    GskOut out_b = ctx->out;
    for (int p = 0; p < out_b.n; ++p) {
      out_b.mean[p] += off;
      out_b.var[p] += off;
    }
    dual_mean_kernel<<<(unsigned)((nb + 7) / 8), 256, 0, st>>>(g->Bm, np, nb, g->w, g->dmean);
    ygemm_dmma_kernel<<<dim3((unsigned)(nbp / GT), (unsigned)(np / GT)), 256, YGEMM_SMEM, st>>>(
        g->X, np, g->Bm, g->YE, g->ne, g->batch, g->partial);
    global_epilogue_kernel<<<(nb + 127) / 128, 128, 0, st>>>(g->partial, (int)(np / GT), g->ne, g->batch, nb, g->GEE, ctx->es,
                                                             ctx->tg, ctx->vg.sill, ctx->prob.flags, first + off,
                                                             out_b, dual);
    if (launches) *launches += 4;
    if (ctx->cols.active) {
      const int m = ctx->cols.m, m8 = (m + 7) / 8 * 8;
      cols_mean_kernel<<<dim3((unsigned)((nb + 15) / 16), (unsigned)((m8 / 8 + 3) / 4)), 128, 0, st>>>(
          g->Bm, np, nb, ctx->cols.gw, m, m8, ctx->cols.gbeta, ctx->es, ctx->tg, first + off, ctx->cols.mean + off * m);
      if (launches) *launches += 1;
    }
  }
  if (d_nn) {
    fill_int_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(d_nn, count, (int)g->n);
    if (launches) *launches += 1;
  }
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return GSK_OK;
}

int gsk_global_loo(gsk_ctx *ctx, long long first, long long count, int *d_nn, int *launches) {
  GlobalPlan *g = ctx->gplan;
  if (!g) { ctx->err = "global plan missing"; return GSK_ERR_STATE; }
  cudaStream_t st = ctx->stream;
  const long long np = g->np, n = g->n;
  const int c = ctx->es.nterms;
  const long long nq = (n + LOO_RCH - 1) / LOO_RCH;
  int rc;
  if ((rc = gsk_buf(ctx, BUF_G_PARTIAL, sizeof(double) * (size_t)nq * (1 + c) * np, (void **)&g->partial)) != GSK_OK)
    return rc;
  const long long cb0 = first / NB, cb1 = (first + count - 1) / NB;
  loo_colsum_kernel<<<dim3((unsigned)(cb1 - cb0 + 1), (unsigned)nq), 256, 0, st>>>(g->X, np, n, g->YE, c, cb0, g->partial);
  loo_epilogue_kernel<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(g->partial, np, n, c, g->GEE, g->ne, g->w,
                                                                       ctx->d_rec_orig, first, count, ctx->prob.flags,
                                                                       ctx->out);
  if (launches) *launches += 2;
  if (d_nn) {
    fill_int_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(d_nn, count, (int)(n - 1));
    if (launches) *launches += 1;
  }
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return GSK_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// LU Gaussian simulation (SURVEY §8f-4; ref src/simulation/lu.jl:75-160 preprocess, :198-224 lusim): the dense covariance
// of ALL points — data locations first, then simulation locations — is assembled and factorised once with the same
// blocked FP64 Cholesky as the global Kriging plan. With C = L Lᵀ, L = [L11 0; A21 L22], the reference's pieces are
// A21 = (L11⁻¹C12)ᵀ and L22 = chol(C22 − A21 A21ᵀ) (lu.jl:126-133), so one realisation d2 + L22 w2 with d2 = A21 L11⁻¹ z1
// (lu.jl:132,209) is the lower part of the single triangular product y = L·[L11⁻¹ z1; w2], whose upper part is z1 itself.
// ---------------------------------------------------------------------------------------------------------------
namespace {
// u = L11⁻¹ z (nd × nd leading block), one CTA: column-oriented forward substitution
__global__ void __launch_bounds__(256) lu_forward_kernel(const double *__restrict__ A, long long ld, int nd,
                                                         const double *__restrict__ z, double *__restrict__ u, double *__restrict__ r) {
  for (int i = threadIdx.x; i < nd; i += 256) r[i] = z[i];
  __syncthreads();
  for (int j = 0; j < nd; ++j) {
    const double uj = r[j] / A[j + (long long)j * ld];
    __syncthreads();
    if (threadIdx.x == 0) u[j] = uj;
    for (int i = j + 1 + threadIdx.x; i < nd; i += 256) r[i] = fma(-A[i + (long long)j * ld], uj, r[i]);
    __syncthreads();
  }
}
// y[i] = Σ_{j<=i} L[i, j]·v[j]: one warp per row
__global__ void lu_matvec_kernel(const double *__restrict__ A, long long ld, long long n, const double *__restrict__ v,
                                 double *__restrict__ y) {
  const long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  double s = 0.0;
  for (long long j = lane; j <= i; j += 32) s = fma(A[i + j * ld], v[j], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) y[i] = s;
}
}  // namespace

int gsk_lu_plan_impl(gsk_ctx *ctx, int dim, long long nd, long long ns, const double *const *coords, const double *z1,
                     const GskVario &vg) {
  cudaStream_t st = ctx->stream;
  const long long n = nd + ns, np = (n + GT - 1) / GT * GT;
  const int nblk = (int)(np / NB);
  std::vector<double4> rec((size_t)n);
  for (long long i = 0; i < n; ++i) {
    rec[(size_t)i] = make_double4(coords[0][i], dim > 1 ? coords[1][i] : 0.0, dim > 2 ? coords[2][i] : 0.0, 0.0);
    if (!std::isfinite(rec[(size_t)i].x) || !std::isfinite(rec[(size_t)i].y) || !std::isfinite(rec[(size_t)i].z)) {
      ctx->err = "point coordinates must be finite";
      return GSK_ERR_INVALID;
    }
  }
  int rc;
  double *A = nullptr, *Dinv = nullptr, *vec = nullptr;
  if ((rc = gsk_buf(ctx, BUF_REC_ORIG, sizeof(double4) * (size_t)n, (void **)&ctx->d_rec_orig)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_A, sizeof(double) * (size_t)np * np, (void **)&A)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_DINV, sizeof(double) * (size_t)nblk * NB * NB, (void **)&Dinv)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_G_TMP, sizeof(double) * (size_t)(3 * np + 32), (void **)&vec)) != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_rec_orig, rec.data(), sizeof(double4) * (size_t)n, cudaMemcpyHostToDevice, st));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  GArgs ga{ctx->d_rec_orig, n, np, vg, dim};
  {
    dim3 grid((unsigned)((np + 255) / 256), (unsigned)np);
    switch (vg.kind) {
      case GSK_VARIO_GAUSSIAN: assemble_kernel<GSK_VARIO_GAUSSIAN><<<grid, 256, 0, st>>>(ga, A); break;
      case GSK_VARIO_SPHERICAL: assemble_kernel<GSK_VARIO_SPHERICAL><<<grid, 256, 0, st>>>(ga, A); break;
      default: assemble_kernel<GSK_VARIO_EXPONENTIAL><<<grid, 256, 0, st>>>(ga, A); break;
    }
  }
  for (int jb = 0; jb < nblk; ++jb) {
    const long long j0 = (long long)jb * NB;
    potrf_diag_kernel<<<1, 64, 0, st>>>(A, np, j0, Dinv + (size_t)jb * NB * NB);
    const int nrem = nblk - jb - 1;
    if (nrem > 0) {
      trsm_panel_kernel<<<nrem, 256, 0, st>>>(A, np, j0, Dinv + (size_t)jb * NB * NB);
      syrk_kernel<<<(unsigned)((long long)nrem * (nrem + 1) / 2), 256, 0, st>>>(A, np, j0, nrem);
    }
  }
  // v = [L11⁻¹ z1; (w2 filled per realisation)], kept in vec[0:np); vec[np:2np) = y, vec[2np:3np) = scratch
  GSK_CUDA_CHECK(ctx, cudaMemsetAsync(vec, 0, sizeof(double) * (size_t)(3 * np + 32), st));
  if (nd > 0) {
    double *hz = nullptr;
    if ((rc = gsk_host_stage(ctx, sizeof(double) * (size_t)nd, (void **)&hz)) != GSK_OK) return rc;
    memcpy(hz, z1, sizeof(double) * (size_t)nd);
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(vec + 2 * np, hz, sizeof(double) * (size_t)nd, cudaMemcpyHostToDevice, st));
    lu_forward_kernel<<<1, 256, 0, st>>>(A, np, (int)nd, vec + 2 * np, vec, vec + np);
  }
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  ctx->lu_n = n;
  ctx->lu_nd = nd;
  ctx->lu_np = np;
  ctx->lu_A = A;
  ctx->lu_vec = vec;
  return GSK_OK;
}

int gsk_lu_sample_impl(gsk_ctx *ctx, const double *w, double *y_out) {
  cudaStream_t st = ctx->stream;
  const long long n = ctx->lu_n, nd = ctx->lu_nd, np = ctx->lu_np, ns = n - nd;
  double *vec = ctx->lu_vec;
  int rc;
  double *hs = nullptr;
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  if ((rc = gsk_host_stage(ctx, sizeof(double) * (size_t)n, (void **)&hs)) != GSK_OK) return rc;
  memcpy(hs, w, sizeof(double) * (size_t)ns);
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(vec + nd, hs, sizeof(double) * (size_t)ns, cudaMemcpyHostToDevice, st));
  lu_matvec_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(ctx->lu_A, np, n, vec, vec + np);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));  // the staging buffer is free again
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(hs, vec + np, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  memcpy(y_out, hs, sizeof(double) * (size_t)n);
  return GSK_OK;
}
