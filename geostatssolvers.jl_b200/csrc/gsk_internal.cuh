// gsk_internal.cuh — shared declarations of libgskrige.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/gskrige.h"

// Development tunables (bin occupancy, staging capacity, kernel selection) exist only in builds made with
// -DGSK_DEV_TUNABLES (scripts/dev A/B runs). The product library reads no environment variable.
#ifdef GSK_DEV_TUNABLES
#include <stdlib.h>
#define GSK_DEV_ENV(name) getenv(name)
#else
#define GSK_DEV_ENV(name) ((const char *)nullptr)
#endif

#define GSK_CUDA_CHECK(ctx, expr)                                                        \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                   \
      return GSK_ERR_CUDA;                                                               \
    }                                                                                    \
  } while (0)

// ---------------------------------------------------------------------------------------
// device-side problem description (passed by value to kernels)
// ---------------------------------------------------------------------------------------
struct GskVario {
  int kind;
  double sill;    // s
  double cs;      // s − n'   (n' = nugget [+ Gaussian epsilon])
  double range;   // r
  double inv_r2;  // 1/r²
  double inv_r;   // 1/r
  double hcs, m15cs;  // 0.5·cs, −1.5·cs (spherical polynomial with cs folded in)
  double m3ir2, m3ir; // −3/r², −3/r (exponent scales of the Gaussian and exponential models)
};

struct GskTargets {
  int is_grid;
  int dim;
  long long gdim[3];
  double gorg[3], gsp[3];
  const double *pts[3];  // explicit target points (device), original order
  long long npts;
};

struct GskBins {
  double lo[3], cell[3], inv[3];
  int nb[3];
  long long ncells;
  const double4 *rec;     // samples sorted by cell: {x, y, z, original index as double bits (int64)}
  const int *cell_start;  // ncells + 1
  double cell_max;        // largest cell side (slack scale)
};

struct GskEstimator {
  int kind;        // GSK_EST_*
  int nterms;      // c: Lagrange rows (SK 0, OK 1, UK C(d+deg,deg))
  double sk_mean;
  int exps[GSK_MAX_DRIFT_TERMS][3];
};

// Where results go. n == 1: one buffer (the caller's). n > 1: the same value is stored into every peer's
// buffer over NVLink (peer-mapped pointers, e.g. torch symmetric memory) — the result "gather" is fused
// into the epilogue of the compute kernel. multicast: out[0] is an NVLS multicast address and one
// multimem.st reaches all peers through the switch.
#define GSK_MAX_PEERS 8
struct GskOut {
  int n;
  int multicast;
  double *mean[GSK_MAX_PEERS];
  double *var[GSK_MAX_PEERS];
};

struct GskLocalArgs {
  GskTargets tg;
  GskVario vg;
  GskEstimator es;
  const double4 *rec_orig;  // samples in original order: {x, y, z, value}
  const double *sup;        // support offsets [3][nsup] (device)
  const double *sup_unit;   // the same in units of the variogram range
  int sup_smem;             // set by the launcher: the kernel stages the offsets in shared memory (else it reads them from
                            // global memory: supports above GSK_MAX_SUPPORT points, or no shared memory left for them)
  int nsup;
  double rhs_inr_lim2;      // spherical model: (1 − max|δ|/range)² (a bit less), or −1: a neighbour whose squared centroid distance in range units is below it has all its support points inside the range
  int sup_tensor3;          // the support is a tensor grid with 3 offsets per axis (the default for cells no larger than the range), x fastest
  double sup_ax[3][3];      // its per-axis offsets: support point q = (kx, ky, kz), q = kx + 3·ky + 9·kz, sits at (sup_ax[0][kx], sup_ax[1][ky], sup_ax[2][kz])
  int rhs_taylor;           // exponential model with 3·max|δ|/range <= 0.06: one exp per neighbour + polynomial per support point
  int k;                    // clamped max neighbours
  int min_neighbors;
  int use_ball;
  double radius;
  unsigned flags;
  long long first, count;   // slab
  const int *nn;            // neighbours per target (slab-local)
  const int *nbr;           // count × k original indices, −1 padded
  GskOut out;               // outputs, indexed by slab-local target (pointers already offset)
};

struct GskSearchArgs {
  GskTargets tg;
  GskBins bins;
  int k;
  int use_ball;
  double radius;
  long long first, count;
  // tile lattice (grid targets): tiles start at cell t0[d], ntile[d] tiles per axis
  long long t0[3];
  int ntile[3];
  int margin0[3];  // initial block margin in bins
  int scap;        // staged records per chunk
  int *nn;         // out: neighbours per target
  int *nbr;        // out: count × k original indices sorted by (d², idx), −1 padded
  const int *trank;  // ranked search (sgs.cu) only: rank + 1 of every target; records carry theirs in the high half of w
  // compact-key pass (search.cu): the low `keybits` bits of a list entry hold the sample index; tiles whose result
  // may depend on the dropped distance bits are appended to redo_list (redo_count of them) and searched again by
  // the exact-key variant, launched with redo_list set
  int keybits;
  int *redo_list;
  int *redo_count;
};

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
struct GlobalPlan;  // global.cu
struct SgsPlan;     // sgs.cu

// cached device buffers: grown on demand, never shrunk, released in gsk_destroy — so that repeated
// gsk_plan / gsk_krige calls do not pay cudaMalloc/cudaFree (which synchronise the device)
enum GskBufId {
  BUF_REC_ORIG, BUF_REC_SORTED, BUF_CELL_START, BUF_SUP, BUF_PTS0, BUF_PTS1, BUF_PTS2, BUF_CELL_OF, BUF_COUNTS,
  BUF_G_A, BUF_G_X, BUF_G_DINV, BUF_G_E, BUF_G_YE, BUF_G_GEE, BUF_G_BM, BUF_G_PARTIAL, BUF_G_W, BUF_G_TMP, BUF_G_DMEAN, BUF_PEAK,
  BUF_PT_CELL, BUF_PT_COUNTS, BUF_PT_PERM, BUF_PT_X, BUF_PT_Y, BUF_PT_Z, BUF_PT_MEAN, BUF_PT_VAR, BUF_PT_NN, BUF_PT_NBR, BUF_VALS, BUF_REDO, BUF_COUNT
};

struct gsk_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;   // main stream: solve kernels, copies (may be the caller's)
  bool own_stream = false;
  cudaStream_t stream2 = nullptr;  // side stream: the search of chunk c+1 overlaps the solve of chunk c
  cudaEvent_t ev_search[2] = {nullptr, nullptr}, ev_solve[2] = {nullptr, nullptr}, ev_fork = nullptr;
  std::string err;
  int sm_count = 148;

  // planned problem (host copy of scalars)
  bool planned = false;
  gsk_problem prob{};
  long long n_targets = 0;
  int nterms = 0;

  // resident device buffers
  double4 *d_rec_orig = nullptr;  // n
  double4 *d_rec_sorted = nullptr;
  int *d_cell_start = nullptr;
  double *d_sup = nullptr;
  double *d_pts[3] = {nullptr, nullptr, nullptr};
  GskBins bins{};
  GskTargets tg{};
  GskVario vg{};
  GskEstimator es{};
  int margin0[3] = {1, 1, 1};
  int rhs_taylor = 0;
  double sup_rmax = 0.0;  // max |δ_q| of the block support
  int sup_tensor3 = 0;    // see GskLocalArgs
  double sup_ax[3][3] = {};

  // scratch that grows on demand
  int *d_nn = nullptr;
  int *d_nbr = nullptr;
  size_t cap_nn = 0, cap_nbr = 0;
  double *d_mean = nullptr, *d_var = nullptr;
  size_t cap_out = 0;
  int *d_nn_out = nullptr, *d_nbr_out = nullptr;  // gsk_krige: neighbour counts / lists requested by the caller
  size_t cap_nn_out = 0, cap_nbr_out = 0;

  // neighbour lists kept from the last local gsk_execute (same plan, same target range): a values-only update
  // (gsk_update_values) then skips the search — and, for explicit points, the bin sort — of the next call
  bool nbr_cached = false;
  bool nbr_reuse = false;  // armed by gsk_update_values, cleared by gsk_plan
  bool loo = false;        // gsk_krige_loo is running: targets are the samples, each excluded from its own list
  long long nbr_first = -1, nbr_count = -1;
  int *pt_perm = nullptr;
  double *pt_sx = nullptr, *pt_sy = nullptr, *pt_sz = nullptr;

  // identity of the resident plan for gsk_krige's GSK_FLAG_REUSE_PLAN: the scalar fields and hashes of the arrays
  bool key_valid = false;
  gsk_problem key_prob{};
  unsigned long long key_geom = 0, key_vals = 0;

  GlobalPlan *gplan = nullptr;
  SgsPlan *sgs = nullptr;  // sequential Gaussian simulation plan (sgs.cu)

  // LU Gaussian simulation plan (global.cu: gsk_lu_plan_impl): factor of the joint covariance, [L11⁻¹z1; w2] and y
  long long lu_n = 0, lu_nd = 0, lu_np = 0;
  double *lu_A = nullptr, *lu_vec = nullptr;

  void *bufp[BUF_COUNT] = {};
  size_t bufcap[BUF_COUNT] = {};
  void *h_stage = nullptr;  // pinned host staging buffer
  size_t h_stage_cap = 0;
  void *h_out = nullptr;    // two pinned 8 MB buffers through which results reach pageable caller arrays
  size_t h_out_cap = 0;

  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  gsk_timing timing{};
  bool timing_pending = false;
  bool phase_timing = false;
  GskOut out{};  // destination of the running gsk_execute / gsk_execute_peers
};

// api.cu
int gsk_buf(gsk_ctx *ctx, GskBufId id, size_t bytes, void **out);
int gsk_host_stage(gsk_ctx *ctx, size_t bytes, void **out);
// bins.cu
// rank_in_w: hv[i] carries (rank + 1) << 32 as bits; the sorted records keep it in the high half of w (ranked search)
int gsk_build_bins(gsk_ctx *ctx, const double *hx, const double *hy, const double *hz, const double *hv, long long n,
                   int dim, int k, bool rank_in_w = false);
// search.cu
// k: list length (the planned max_neighbors, or one more for leave-one-out)
int gsk_launch_search(gsk_ctx *ctx, cudaStream_t st, long long first, long long count, int k, int *d_nn, int *d_nbr,
                      int *launches, const int *d_trank = nullptr);
// estim.cu: the IDW / LWR per-location bodies on the neighbour lists (or on all samples when k == 0)
int gsk_launch_simple_solver(gsk_ctx *ctx, cudaStream_t st, long long first, long long count, const int *d_nn,
                             const int *d_nbr, long long out_off, int *d_nn_out, int *launches);
// local_solve*.cu
int gsk_launch_local_solve(gsk_ctx *ctx, cudaStream_t st, long long first, long long count, const int *d_nn,
                           const int *d_nbr, long long out_off, int *launches);
// global.cu
int gsk_global_plan(gsk_ctx *ctx, const double *hx, const double *hy, const double *hz, const double *hv);
int gsk_global_execute(gsk_ctx *ctx, long long first, long long count, int *d_nn, int *launches);
void gsk_global_free(gsk_ctx *ctx);
int gsk_global_update_values(gsk_ctx *ctx);
// leave-one-out residuals and variances of samples [first, first+count) from the resident plan (Dubrule's identities)
int gsk_global_loo(gsk_ctx *ctx, long long first, long long count, int *d_nn, int *launches);
int gsk_lu_plan_impl(gsk_ctx *ctx, int dim, long long nd, long long ns, const double *const *coords, const double *z1,
                     const GskVario &vg);
int gsk_lu_sample_impl(gsk_ctx *ctx, const double *w, double *y_out);  // rec_orig carries new values: rebuild E, Y_E, G_EE (L, L⁻¹ stay)
// points.cu
int gsk_points_sort(gsk_ctx *ctx, long long first, long long count, int **perm, double **sx, double **sy, double **sz);
int gsk_points_unscatter(gsk_ctx *ctx, const int *perm, long long count, const double *ms, const double *vs,
                         const GskOut &out, const int *nn_s, int *nn_out, const int *nbr_s, int *nbr_out, int k);
// leave-one-out: drops each sorted target's own sample index (first + perm[s]) from its (k+1)-list and cuts it to k
int gsk_points_loo_compact(gsk_ctx *ctx, const int *perm, long long first, long long count, int k, const int *nn1,
                           const int *nbr1, int *nn_s, int *nbr_s);
// sgs.cu
int gsk_sgs_plan_impl(gsk_ctx *ctx, int dim, long long n, const double *const *coords, const long long *rank,
                      const GskVario &vg, double mean, int min_neighbors, int k, double ball_radius);
int gsk_sgs_sample_impl(gsk_ctx *ctx, int nreal, const double *values, const double *z, double *out, bool on_device);
int gsk_sgs_weights_impl(gsk_ctx *ctx, int *nn_out, int *nbr_out, double *lam_out, double *sig_out);
void gsk_sgs_free(gsk_ctx *ctx);
// peak.cu
int gsk_peak_measure(gsk_ctx *ctx, double *dfma, double *dmma);

// ---------------------------------------------------------------------------------------
// device helpers shared by kernels
// ---------------------------------------------------------------------------------------
#ifdef __CUDACC__
// target centroid: origin + (i + 0.5)·spacing, no FMA (bit-identical to the oracle)
__device__ __forceinline__ double gsk_cell_center(double org, double sp, long long i) {
  return __dadd_rn(org, __dmul_rn((double)i + 0.5, sp));
}

// centroid of target `lin` (grid: x-fastest linear index; explicit points otherwise)
__device__ __forceinline__ void gsk_target_center(const GskTargets &tg, long long lin, double (&tc)[3]) {
  tc[0] = tc[1] = tc[2] = 0.0;
  if (tg.is_grid) {
    long long rem = lin;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      if (d < tg.dim) {
        const long long c = rem % tg.gdim[d];
        rem /= tg.gdim[d];
        tc[d] = gsk_cell_center(tg.gorg[d], tg.gsp[d], c);
      }
    }
  } else {
#pragma unroll
    for (int d = 0; d < 3; ++d)
      if (d < tg.dim) tc[d] = tg.pts[d][lin];
  }
}

// squared Euclidean distance exactly as the search kernel and the oracle form it: ((dx·dx)+(dy·dy))+(dz·dz), no FMA
__device__ __forceinline__ double gsk_dist2_exact(int dim, const double (&tc)[3], const double4 &r) {
  const double dx = tc[0] - r.x;
  double d2 = __dmul_rn(dx, dx);
  if (dim > 1) {
    const double dy = tc[1] - r.y;
    d2 = __dadd_rn(d2, __dmul_rn(dy, dy));
  }
  if (dim > 2) {
    const double dz = tc[2] - r.z;
    d2 = __dadd_rn(d2, __dmul_rn(dz, dz));
  }
  return d2;
}

// covariance C(h) = sill − γ(h) from the squared distance (d2 == 0 → sill)
template <int VK>
__device__ __forceinline__ double gsk_cov(const GskVario &v, double d2) {
  double c;
  if (VK == GSK_VARIO_GAUSSIAN) {
    c = v.cs * exp(-3.0 * d2 * v.inv_r2);
  } else if (VK == GSK_VARIO_SPHERICAL) {
    double u = d2 * v.inv_r2;
    double t = sqrt(u);
    double g = fma(t, fma(0.5, u, -1.5), 1.0);  // 1 − 1.5t + 0.5t³
    c = (u < 1.0) ? v.cs * g : 0.0;
  } else {
    c = v.cs * exp(-3.0 * sqrt(d2) * v.inv_r);
  }
  return (d2 > 0.0) ? c : v.sill;
}

__device__ __forceinline__ double gsk_cov_rt(const GskVario &v, double d2) {
  switch (v.kind) {
    case GSK_VARIO_GAUSSIAN: return gsk_cov<GSK_VARIO_GAUSSIAN>(v, d2);
    case GSK_VARIO_SPHERICAL: return gsk_cov<GSK_VARIO_SPHERICAL>(v, d2);
    default: return gsk_cov<GSK_VARIO_EXPONENTIAL>(v, d2);
  }
}

// x^e for the drift monomials, e in {0, 1, 2} (Universal Kriging up to degree 2): branch-free
// store one target's result into every destination (see GskOut)
__device__ __forceinline__ void gsk_store_result(const GskOut &o, long long t, double m, double v) {
  if (o.multicast) {
    asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" ::"l"(o.mean[0] + t), "d"(m) : "memory");
    asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" ::"l"(o.var[0] + t), "d"(v) : "memory");
    return;
  }
#pragma unroll
  for (int p = 0; p < GSK_MAX_PEERS; ++p) {
    if (p < o.n) {
      o.mean[p][t] = m;
      o.var[p][t] = v;
    }
  }
}

// one field of one target (field 0: mean, 1: variance) — for kernels that stage a CTA's results in shared memory and
// write them with consecutive threads (coalesced 8-byte stores: thread i → target t0 + i)
__device__ __forceinline__ void gsk_store_field(const GskOut &o, int field, long long t, double x) {
  if (o.multicast) {
    asm volatile("multimem.st.relaxed.sys.global.f64 [%0], %1;" ::"l"((field ? o.var[0] : o.mean[0]) + t), "d"(x) : "memory");
    return;
  }
#pragma unroll
  for (int p = 0; p < GSK_MAX_PEERS; ++p)
    if (p < o.n) (field ? o.var[p] : o.mean[p])[t] = x;
}

__device__ __forceinline__ double gsk_ipow(double x, int e) {
  const double x1 = (e >= 1) ? x : 1.0;
  return (e >= 2) ? x1 * x : x1;
}
#endif
