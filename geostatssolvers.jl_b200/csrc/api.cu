// api.cu — the C ABI of libgskrige.so (include/gskrige.h): context, plan/execute orchestration, the
// one-shot host-buffer entry point that replaces exactsolve/approxsolve (ref: src/estimation/krig.jl:
// 166-186, 188-234), and the host helpers every binding shares. No CPU compute path exists here:
// without an sm_100 device gsk_create fails and nothing else can be called.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "gsk_internal.cuh"

static thread_local std::string g_static_err;

static int fail(gsk_ctx *ctx, int code, const std::string &msg) {
  if (ctx) ctx->err = msg;
  else g_static_err = msg;
  return code;
}

// ---------------------------------------------------------------------------------------------
// host helpers
// ---------------------------------------------------------------------------------------------
extern "C" GSK_API int gsk_abi_version(void) { return GSK_ABI_VERSION; }

extern "C" GSK_API int64_t gsk_num_targets(const gsk_problem *p) {
  if (!p) return -1;
  if (p->grid_dims[0] > 0) {
    int64_t t = 1;
    for (int d = 0; d < p->dim && d < 3; ++d) t *= p->grid_dims[d];
    return t;
  }
  return p->n_points;
}

// GeoStatsModels' UKexps [3P]: exponent vectors of total degree 0..degree (each degree in descending
// lexicographic order), stably sorted by descending max exponent → degree 1: x, y, (z), 1.
extern "C" GSK_API int gsk_uk_exponents(int degree, int dim, int32_t *out, int cap) {
  if (degree < 0 || degree > 2 || dim < 1 || dim > 3 || !out) return GSK_ERR_INVALID;
  int tmp[16][3];
  int n = 0;
  for (int deg = 0; deg <= degree; ++deg)
    for (int a = deg; a >= 0; --a)
      for (int b = deg - a; b >= 0; --b) {
        int c = deg - a - b;
        if (dim == 1 && (b != 0 || c != 0)) continue;
        if (dim == 2 && c != 0) continue;
        tmp[n][0] = a; tmp[n][1] = b; tmp[n][2] = c;
        ++n;
      }
  if (n > cap) return GSK_ERR_INVALID;
  int w = 0;
  for (int mx = degree; mx >= 0; --mx)
    for (int i = 0; i < n; ++i)
      if (std::max(tmp[i][0], std::max(tmp[i][1], tmp[i][2])) == mx) {
        for (int d = 0; d < dim; ++d) out[w * dim + d] = tmp[i][d];
        ++w;
      }
  return n;
}

// Variography's geometry sub-sampling for γ(cell, point) [3P, SURVEY V1]: per axis
// n = ceil(side / (min(range, min side)/3)) points at parametric positions j/(n+1), j = 1..n.
extern "C" GSK_API int gsk_default_support(int dim, const double *spacing, double vario_range, double *ox, double *oy,
                                   double *oz, int cap) {
  if (dim < 1 || dim > 3 || !spacing) return GSK_ERR_INVALID;
  double lmin = INFINITY;
  for (int d = 0; d < dim; ++d)
    if (spacing[d] > 0) lmin = std::min(lmin, spacing[d]);
  if (!(lmin < INFINITY)) return GSK_ERR_INVALID;
  double step = ((vario_range > 0) ? std::min(vario_range, lmin) : lmin) / 3.0;
  int n[3] = {1, 1, 1};
  long long tot = 1;
  for (int d = 0; d < dim; ++d) {
    n[d] = std::max(1, (int)ceil(spacing[d] / step - 1e-12));
    tot *= n[d];
  }
  if (tot > GSK_MAX_SUPPORT_GLOBAL) return GSK_ERR_UNSUPPORTED;
  if (!ox) return (int)tot;  // count only: the caller sizes its arrays with it
  if (tot > cap) return GSK_ERR_INVALID;
  double *o[3] = {ox, oy, oz};
  int w = 0;
  for (int kz = 0; kz < n[2]; ++kz)
    for (int ky = 0; ky < n[1]; ++ky)
      for (int kx = 0; kx < n[0]; ++kx) {
        int kk[3] = {kx, ky, kz};
        for (int d = 0; d < dim; ++d)
          if (o[d]) o[d][w] = ((double)(kk[d] + 1) / (double)(n[d] + 1) - 0.5) * spacing[d];
        ++w;
      }
  return (int)tot;
}

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
extern "C" GSK_API int gsk_create(gsk_ctx **out, int device_id) try {
  if (!out) return fail(nullptr, GSK_ERR_INVALID, "gsk_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, GSK_ERR_CUDA,
                std::string("no CUDA device visible (libgskrige has no CPU fallback): ") + cudaGetErrorString(e));
  if (device_id < 0 || device_id >= ndev) return fail(nullptr, GSK_ERR_INVALID, "gsk_create: device_id out of range");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device_id);
  if (e != cudaSuccess) return fail(nullptr, GSK_ERR_CUDA, cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, GSK_ERR_CUDA, "device is not sm_100 (libgskrige is built for B200 / sm_100a only)");
  gsk_ctx *ctx = new (std::nothrow) gsk_ctx();
  if (!ctx) return fail(nullptr, GSK_ERR_NOMEM, "gsk_create: out of host memory");
  ctx->device = device_id;
  ctx->sm_count = prop.multiProcessorCount;
  e = cudaSetDevice(device_id);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  ctx->own_stream = true;
  for (int i = 0; i < 6 && e == cudaSuccess; ++i) e = cudaEventCreate(&ctx->ev[i]);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking);
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&ctx->ev_search[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_solve[i], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    std::string m = cudaGetErrorString(e);
    delete ctx;
    return fail(nullptr, GSK_ERR_CUDA, m);
  }
  *out = ctx;
  return GSK_OK;
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(nullptr, GSK_ERR_NOMEM, "gsk_create: out of host memory");
} catch (const std::exception &e) {
  return fail(nullptr, GSK_ERR_STATE, std::string("gsk_create: ") + e.what());
}

int gsk_buf(gsk_ctx *ctx, GskBufId id, size_t bytes, void **out) {
  if (bytes == 0) bytes = 16;
  if (ctx->bufcap[id] < bytes) {
    cudaFree(ctx->bufp[id]);
    ctx->bufp[id] = nullptr;
    ctx->bufcap[id] = 0;
    cudaError_t e = cudaMalloc(&ctx->bufp[id], bytes);
    if (e != cudaSuccess) {
      ctx->err = std::string("device allocation failed: ") + cudaGetErrorString(e);
      return GSK_ERR_NOMEM;
    }
    ctx->bufcap[id] = bytes;
  }
  *out = ctx->bufp[id];
  return GSK_OK;
}

int gsk_host_stage(gsk_ctx *ctx, size_t bytes, void **out) {
  if (ctx->h_stage_cap < bytes) {
    if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
    ctx->h_stage = nullptr;
    ctx->h_stage_cap = 0;
    cudaError_t e = cudaHostAlloc(&ctx->h_stage, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) {
      ctx->err = std::string("pinned host allocation failed: ") + cudaGetErrorString(e);
      return GSK_ERR_NOMEM;
    }
    ctx->h_stage_cap = bytes;
  }
  *out = ctx->h_stage;
  return GSK_OK;
}

static void free_plan(gsk_ctx *ctx) {
  // device buffers stay cached in ctx->bufp; only the plan state is dropped
  ctx->d_rec_orig = ctx->d_rec_sorted = nullptr;
  ctx->d_cell_start = nullptr;
  ctx->d_sup = nullptr;
  for (int d = 0; d < 3; ++d) ctx->d_pts[d] = nullptr;
  gsk_global_free(ctx);
  gsk_sgs_free(ctx);
  ctx->planned = false;
  ctx->nbr_cached = false;
  ctx->nbr_reuse = false;
  ctx->key_valid = false;
  ctx->lu_n = 0;  // the LU simulation plan shares the buffers
}

extern "C" GSK_API void gsk_destroy(gsk_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  free_plan(ctx);
  for (int i = 0; i < BUF_COUNT; ++i) cudaFree(ctx->bufp[i]);
  if (ctx->h_stage) cudaFreeHost(ctx->h_stage);
  if (ctx->h_out) cudaFreeHost(ctx->h_out);
  cudaFree(ctx->d_nn);
  cudaFree(ctx->d_nbr);
  cudaFree(ctx->d_nn_out);
  cudaFree(ctx->d_nbr_out);
  cudaFree(ctx->d_mean);
  cudaFree(ctx->d_var);
  for (int i = 0; i < 6; ++i)
    if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->stream2) { cudaStreamSynchronize(ctx->stream2); cudaStreamDestroy(ctx->stream2); }
  for (int i = 0; i < 2; ++i) {
    if (ctx->ev_search[i]) cudaEventDestroy(ctx->ev_search[i]);
    if (ctx->ev_solve[i]) cudaEventDestroy(ctx->ev_solve[i]);
  }
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  delete ctx;
}

extern "C" GSK_API const char *gsk_last_error(const gsk_ctx *ctx) { return ctx ? ctx->err.c_str() : g_static_err.c_str(); }

extern "C" GSK_API int gsk_set_stream(gsk_ctx *ctx, void *cuda_stream) {
  if (!ctx) return GSK_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->own_stream = false;
  return GSK_OK;
}

extern "C" GSK_API int gsk_synchronize(gsk_ctx *ctx) {
  if (!ctx) return GSK_ERR_INVALID;
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  return GSK_OK;
}

// ---------------------------------------------------------------------------------------------
// plan
// ---------------------------------------------------------------------------------------------
static int validate(gsk_ctx *ctx, const gsk_problem *p) {
  if (!p) return fail(ctx, GSK_ERR_INVALID, "problem is NULL");
  if (p->abi_version != GSK_ABI_VERSION) return fail(ctx, GSK_ERR_INVALID, "gsk_problem.abi_version mismatch");
  if (p->dim < 1 || p->dim > 3) return fail(ctx, GSK_ERR_UNSUPPORTED, "dim must be 1, 2 or 3");
  if (p->n_samples < 1) return fail(ctx, GSK_ERR_INVALID, "n_samples must be >= 1");
  if (p->n_samples > 0x7fffffffLL) return fail(ctx, GSK_ERR_UNSUPPORTED, "n_samples must fit in int32");
  if (!p->values) return fail(ctx, GSK_ERR_INVALID, "values is NULL");
  for (int d = 0; d < p->dim; ++d)
    if (!p->coords[d]) return fail(ctx, GSK_ERR_INVALID, "coords[d] is NULL for d < dim");
  if (p->grid_dims[0] > 0) {
    for (int d = 0; d < p->dim; ++d) {
      if (p->grid_dims[d] < 1) return fail(ctx, GSK_ERR_INVALID, "grid_dims must be >= 1");
      if (!(p->grid_spacing[d] > 0.0) || !std::isfinite(p->grid_spacing[d]) || !std::isfinite(p->grid_origin[d]))
        return fail(ctx, GSK_ERR_INVALID, "grid_spacing must be finite and > 0, grid_origin finite");
    }
  } else {
    if (p->n_points < 0) return fail(ctx, GSK_ERR_INVALID, "n_points must be >= 0");
    for (int d = 0; d < p->dim; ++d)
      if (p->n_points > 0 && !p->point_coords[d]) return fail(ctx, GSK_ERR_INVALID, "point_coords[d] is NULL");
  }
  if (p->n_support < 1 || p->n_support > GSK_MAX_SUPPORT_GLOBAL)
    return fail(ctx, GSK_ERR_INVALID, "n_support must be in [1, GSK_MAX_SUPPORT_GLOBAL]");
  if (p->solver < GSK_SOLVER_KRIGING || p->solver > GSK_SOLVER_LWR) return fail(ctx, GSK_ERR_UNSUPPORTED, "unknown solver");
  if (p->solver != GSK_SOLVER_KRIGING) {
    // IDW / LWR: no variogram, estimator or block support; max_neighbors == 0 means every sample (idw.jl:93, lwr.jl:95)
    if (p->solver == GSK_SOLVER_IDW && !(p->idw_exponent > 0.0 && std::isfinite(p->idw_exponent)))
      return fail(ctx, GSK_ERR_INVALID, "exponent must be positive");  // idw.jl:96
    if (p->solver == GSK_SOLVER_LWR && p->lwr_weightfun != GSK_LWR_WEIGHT_EXP3H2)
      return fail(ctx, GSK_ERR_UNSUPPORTED, "only the default LWR weight function h -> exp(-3 h^2) crosses the C ABI");
    if (p->min_neighbors < 0 || p->max_neighbors < 0) return fail(ctx, GSK_ERR_INVALID, "min/max_neighbors must be >= 0");
    if (p->max_neighbors > GSK_MAX_NEIGHBORS)
      return fail(ctx, GSK_ERR_UNSUPPORTED, "max_neighbors exceeds GSK_MAX_NEIGHBORS (pass 0 to use every sample)");
    if (p->max_neighbors > p->n_samples)
      return fail(ctx, GSK_ERR_INVALID, "max_neighbors must be clamped to n_samples by the host (ui.jl:16-23)");
    if ((p->max_neighbors > 0 ? p->max_neighbors : p->n_samples) < p->min_neighbors)
      return fail(ctx, GSK_ERR_INVALID, "invalid min/max number of neighbors");  // idw.jl:97, lwr.jl:98
    if (p->max_neighbors > 0 && !(p->ball_radius != p->ball_radius) && !(p->ball_radius > 0.0))
      return fail(ctx, GSK_ERR_INVALID, "ball_radius must be > 0 or NaN");
    int64_t T = gsk_num_targets(p);
    int64_t first = p->target_first, count = p->target_count < 0 ? T - first : p->target_count;
    if (first < 0 || count < 0 || first + count > T) return fail(ctx, GSK_ERR_INVALID, "target slab out of range");
    return GSK_OK;
  }
  if (p->vario_kind < 0 || p->vario_kind > 2) return fail(ctx, GSK_ERR_UNSUPPORTED, "unknown variogram kind");
  if (!(p->vario_range > 0.0)) return fail(ctx, GSK_ERR_INVALID, "vario_range must be > 0");
  if (!(p->vario_sill > 0.0)) return fail(ctx, GSK_ERR_INVALID, "vario_sill must be > 0");
  if (!(p->vario_nugget >= 0.0) || !(p->gaussian_nugget_eps >= 0.0))
    return fail(ctx, GSK_ERR_INVALID, "vario_nugget and gaussian_nugget_eps must be >= 0");
  if (!(p->vario_sill - p->vario_nugget - (p->vario_kind == GSK_VARIO_GAUSSIAN ? p->gaussian_nugget_eps : 0.0) > 0.0) ||
      !std::isfinite(p->vario_sill) || !std::isfinite(p->vario_range))
    return fail(ctx, GSK_ERR_INVALID, "the nugget must be below a finite sill, the range finite");
  if (p->estimator == GSK_EST_SIMPLE && !std::isfinite(p->sk_mean))
    return fail(ctx, GSK_ERR_INVALID, "sk_mean must be finite");
  if (p->min_neighbors < 0) return fail(ctx, GSK_ERR_INVALID, "min_neighbors must be >= 0");
  if (p->estimator < 0 || p->estimator > 2) return fail(ctx, GSK_ERR_UNSUPPORTED, "unknown estimator");
  if (p->estimator == GSK_EST_UNIVERSAL && (p->uk_degree < 0 || p->uk_degree > 2))
    return fail(ctx, GSK_ERR_UNSUPPORTED, "uk_degree must be 0, 1 or 2");
  if (p->max_neighbors < 0) return fail(ctx, GSK_ERR_INVALID, "max_neighbors must be >= 0");
  if (p->max_neighbors > GSK_MAX_NEIGHBORS)
    return fail(ctx, GSK_ERR_UNSUPPORTED, "max_neighbors exceeds GSK_MAX_NEIGHBORS on the local path");
  if (p->max_neighbors > p->n_samples)
    return fail(ctx, GSK_ERR_INVALID, "max_neighbors must be clamped to n_samples by the host (ui.jl:16-23)");
  if (p->max_neighbors > 0 && !(p->ball_radius != p->ball_radius) && !(p->ball_radius > 0.0))
    return fail(ctx, GSK_ERR_INVALID, "ball_radius must be > 0 or NaN");
  int64_t T = gsk_num_targets(p);
  int64_t first = p->target_first, count = p->target_count < 0 ? T - first : p->target_count;
  if (first < 0 || count < 0 || first + count > T) return fail(ctx, GSK_ERR_INVALID, "target slab out of range");
  return GSK_OK;
}

static GskVario make_vario(int kind, double range, double sill, double nugget, double gaussian_eps) {
  GskVario v{};
  v.kind = kind;
  v.sill = sill;
  const double nug = nugget + (kind == GSK_VARIO_GAUSSIAN ? gaussian_eps : 0.0);
  v.cs = sill - nug;
  v.range = range;
  v.inv_r = 1.0 / range;
  v.inv_r2 = v.inv_r * v.inv_r;
  v.hcs = 0.5 * v.cs;
  v.m15cs = -1.5 * v.cs;
  v.m3ir2 = -3.0 * v.inv_r2;
  v.m3ir = -3.0 * v.inv_r;
  return v;
}

extern "C" GSK_API int gsk_plan(gsk_ctx *ctx, const gsk_problem *p) try {
  if (!ctx) return GSK_ERR_INVALID;
  int rc = validate(ctx, p);
  if (rc != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  free_plan(ctx);
  GSK_CUDA_CHECK(ctx, cudaEventRecord(ctx->ev[0], ctx->stream));
  ctx->prob = *p;
  ctx->n_targets = gsk_num_targets(p);
  const int dim = p->dim;

  // variogram constants
  ctx->vg = make_vario(p->vario_kind, p->vario_range, p->vario_sill, p->vario_nugget, p->gaussian_nugget_eps);

  // estimator
  GskEstimator &es = ctx->es;
  memset(&es, 0, sizeof(es));
  es.kind = p->estimator;
  es.sk_mean = p->sk_mean;
  es.nterms = 0;
  if (p->estimator == GSK_EST_ORDINARY) es.nterms = 1;
  if (p->estimator == GSK_EST_UNIVERSAL) {
    int32_t ex[3 * GSK_MAX_DRIFT_TERMS];
    int c = gsk_uk_exponents(p->uk_degree, dim, ex, GSK_MAX_DRIFT_TERMS);
    if (c < 0) return fail(ctx, GSK_ERR_UNSUPPORTED, "unsupported Universal Kriging degree");
    es.nterms = c;
    for (int t = 0; t < c; ++t)
      for (int d = 0; d < dim; ++d) es.exps[t][d] = ex[t * dim + d];
  }
  ctx->nterms = es.nterms;

  // targets
  GskTargets &tg = ctx->tg;
  memset(&tg, 0, sizeof(tg));
  tg.dim = dim;
  tg.is_grid = p->grid_dims[0] > 0;
  for (int d = 0; d < 3; ++d) {
    tg.gdim[d] = (tg.is_grid && d < dim) ? p->grid_dims[d] : 1;
    tg.gorg[d] = (d < dim) ? p->grid_origin[d] : 0.0;
    tg.gsp[d] = (d < dim) ? p->grid_spacing[d] : 1.0;
  }
  if (p->target_order) {
    // a traversal order (non-linear path): the targets become an explicit point list in VISITING order — the
    // centroid of target_order[j] with the library's own centroid arithmetic — so that out[j] is the j-th visited
    // target, as in the reference (krig.jl:179-183, 204-231). Block support still applies (grid cells).
    const int64_t T = ctx->n_targets;
    std::vector<double> pts[3];
    for (int d = 0; d < dim; ++d) pts[d].resize((size_t)std::max<int64_t>(1, T));
    for (int64_t j = 0; j < T; ++j) {
      const int64_t lin = p->target_order[j];
      if (lin < 0 || lin >= T) return fail(ctx, GSK_ERR_INVALID, "target_order entries must be in [0, gsk_num_targets)");
      if (tg.is_grid) {
        int64_t rem = lin;
        for (int d = 0; d < dim; ++d) {
          const int64_t c = rem % tg.gdim[d];
          rem /= tg.gdim[d];
          pts[d][(size_t)j] = tg.gorg[d] + ((double)c + 0.5) * tg.gsp[d];  // = gsk_cell_center (no contraction on the host)
        }
      } else {
        for (int d = 0; d < dim; ++d) pts[d][(size_t)j] = p->point_coords[d][lin];
      }
    }
    tg.is_grid = 0;
    tg.npts = T;
    for (int d = 0; d < dim; ++d) {
      rc = gsk_buf(ctx, (GskBufId)(BUF_PTS0 + d), sizeof(double) * (size_t)std::max<int64_t>(1, T), (void **)&ctx->d_pts[d]);
      if (rc != GSK_OK) return rc;
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_pts[d], pts[d].data(), sizeof(double) * (size_t)T, cudaMemcpyHostToDevice, ctx->stream));
      tg.pts[d] = ctx->d_pts[d];
    }
    GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));  // pts[] go out of scope
  } else if (!tg.is_grid) {
    tg.npts = p->n_points;
    for (int d = 0; d < dim; ++d) {
      rc = gsk_buf(ctx, (GskBufId)(BUF_PTS0 + d), sizeof(double) * (size_t)std::max<int64_t>(1, p->n_points), (void **)&ctx->d_pts[d]);
      if (rc != GSK_OK) return rc;
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_pts[d], p->point_coords[d], sizeof(double) * (size_t)p->n_points,
                                          cudaMemcpyHostToDevice, ctx->stream));
      tg.pts[d] = ctx->d_pts[d];
    }
  }

  // block support offsets, [3][nsup]
  {
    std::vector<double> sup(3 * (size_t)p->n_support, 0.0);
    for (int d = 0; d < dim; ++d)
      if (p->support_offsets[d])
        for (int q = 0; q < p->n_support; ++q) sup[(size_t)d * p->n_support + q] = p->support_offsets[d][q];
    // two copies: the offsets as given, and in units of the variogram range (the spherical kernels work in that frame
    // and read supports too large for shared memory straight from here)
    const size_t nq3 = sup.size();
    sup.resize(2 * nq3);
    for (size_t i = 0; i < nq3; ++i) sup[nq3 + i] = sup[i] * (1.0 / p->vario_range);
    rc = gsk_buf(ctx, BUF_SUP, sizeof(double) * sup.size(), (void **)&ctx->d_sup);
    if (rc != GSK_OK) return rc;
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_sup, sup.data(), sizeof(double) * sup.size(), cudaMemcpyHostToDevice,
                                        ctx->stream));
    // block-support RHS shortcut for the exponential model (local_solve.cuh: rhs_block_support)
    double dmax2 = 0.0;
    for (int q = 0; q < p->n_support; ++q) {
      double d2 = 0.0;
      for (int d = 0; d < 3; ++d) d2 += sup[(size_t)d * p->n_support + q] * sup[(size_t)d * p->n_support + q];
      dmax2 = std::max(dmax2, d2);
    }
    ctx->sup_rmax = sqrt(dmax2);
    // tensor-grid support with 3 offsets per axis, x fastest (what gsk_default_support produces for cells no larger
    // than the range): the solve kernels then form the squared distances to the support points from per-axis squares
    {
      const int q = p->n_support;
      int want = 1;
      for (int d = 0; d < dim; ++d) want *= 3;
      bool ok = (q == want) && dim >= 2;  // (1-D problems run the 2-D kernels with y = 0: their 3 offsets are not a 3×3 grid)
      for (int d = 0; d < 3 && ok; ++d) {
        const int stride = (d == 0) ? 1 : (d == 1 ? 3 : 9);
        for (int a = 0; a < 3; ++a) ctx->sup_ax[d][a] = (d < dim) ? sup[(size_t)d * q + (size_t)a * stride] : 0.0;
        for (int i = 0; i < q && ok; ++i) {
          const double expect = (d < dim) ? ctx->sup_ax[d][(i / stride) % 3] : 0.0;
          ok = (sup[(size_t)d * q + i] == expect);
        }
      }
      ctx->sup_tensor3 = ok ? 1 : 0;
    }
    ctx->rhs_taylor = (p->vario_kind == GSK_VARIO_EXPONENTIAL && p->n_support > 1 &&
                       3.0 * sqrt(dmax2) / p->vario_range <= 0.06 && !GSK_DEV_ENV("GSK_NO_RHS_TAYLOR")) ? 1 : 0;
    GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  }

  if (p->max_neighbors > 0) {
    rc = gsk_build_bins(ctx, p->coords[0], dim > 1 ? p->coords[1] : nullptr, dim > 2 ? p->coords[2] : nullptr,
                        p->values, p->n_samples, dim, p->max_neighbors);
  } else if (p->solver != GSK_SOLVER_KRIGING) {
    // IDW / LWR over every sample: only the {x, y, z, value} records are needed
    const long long n = p->n_samples;
    double4 *hrec = nullptr;
    if ((rc = gsk_buf(ctx, BUF_REC_ORIG, sizeof(double4) * (size_t)n, (void **)&ctx->d_rec_orig)) != GSK_OK) return rc;
    if ((rc = gsk_host_stage(ctx, sizeof(double4) * (size_t)n, (void **)&hrec)) != GSK_OK) return rc;
    for (long long i = 0; i < n; ++i) {
      hrec[i] = make_double4(p->coords[0][i], dim > 1 ? p->coords[1][i] : 0.0, dim > 2 ? p->coords[2][i] : 0.0, p->values[i]);
      if (!std::isfinite(hrec[i].x) || !std::isfinite(hrec[i].y) || !std::isfinite(hrec[i].z))
        return fail(ctx, GSK_ERR_INVALID, "sample coordinates must be finite");
    }
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_rec_orig, hrec, sizeof(double4) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  } else {
    rc = gsk_global_plan(ctx, p->coords[0], dim > 1 ? p->coords[1] : nullptr, dim > 2 ? p->coords[2] : nullptr,
                         p->values);
  }
  if (rc != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->timing = gsk_timing{};
  ctx->timing.ms_plan = ms;
  // the host pointers of the problem are not kept
  for (int d = 0; d < 3; ++d) { ctx->prob.coords[d] = nullptr; ctx->prob.point_coords[d] = nullptr; ctx->prob.support_offsets[d] = nullptr; }
  ctx->prob.values = nullptr;
  ctx->prob.target_order = nullptr;
  ctx->planned = true;
  return GSK_OK;
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_plan: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_plan: ") + e.what());
}

// ---------------------------------------------------------------------------------------------
// execute
// ---------------------------------------------------------------------------------------------
static int ensure(gsk_ctx *ctx, void **buf, size_t *cap, size_t bytes) {
  if (*cap >= bytes) return GSK_OK;
  cudaFree(*buf);
  *buf = nullptr;
  *cap = 0;
  cudaError_t e = cudaMalloc(buf, bytes);
  if (e != cudaSuccess) return fail(ctx, GSK_ERR_NOMEM, std::string("device allocation failed: ") + cudaGetErrorString(e));
  *cap = bytes;
  return GSK_OK;
}

static int execute_impl(gsk_ctx *ctx, int64_t first, int64_t count, int32_t *d_nneigh, int32_t *d_neigh_idx);

extern "C" GSK_API int gsk_execute(gsk_ctx *ctx, int64_t first, int64_t count, double *d_mean, double *d_var,
                           int32_t *d_nneigh, int32_t *d_neigh_idx) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!d_mean || !d_var) return fail(ctx, GSK_ERR_INVALID, "output buffers are NULL");
  ctx->out = GskOut{};
  ctx->out.n = 1;
  ctx->out.mean[0] = d_mean;
  ctx->out.var[0] = d_var;
  return execute_impl(ctx, first, count, d_nneigh, d_neigh_idx);
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_execute: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_execute: ") + e.what());
}

extern "C" GSK_API int gsk_execute_peers(gsk_ctx *ctx, int64_t first, int64_t count, int n_peers,
                                 double *const *d_mean_peers, double *const *d_var_peers, int64_t out_offset,
                                 int multicast, int32_t *d_nneigh, int32_t *d_neigh_idx) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (n_peers < 1 || n_peers > GSK_MAX_PEERS || !d_mean_peers || !d_var_peers)
    return fail(ctx, GSK_ERR_INVALID, "n_peers must be in [1, 8] with non-NULL pointer lists");
  if (multicast && n_peers != 1) return fail(ctx, GSK_ERR_INVALID, "multicast takes exactly one (multicast) address per field");
  ctx->out = GskOut{};
  ctx->out.n = n_peers;
  ctx->out.multicast = multicast ? 1 : 0;
  for (int p = 0; p < n_peers; ++p) {
    if (!d_mean_peers[p] || !d_var_peers[p]) return fail(ctx, GSK_ERR_INVALID, "peer output buffer is NULL");
    ctx->out.mean[p] = d_mean_peers[p] + out_offset;
    ctx->out.var[p] = d_var_peers[p] + out_offset;
  }
  return execute_impl(ctx, first, count, d_nneigh, d_neigh_idx);
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_execute_peers: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_execute_peers: ") + e.what());
}

static int execute_impl(gsk_ctx *ctx, int64_t first, int64_t count, int32_t *d_nneigh, int32_t *d_neigh_idx) {
  if (!ctx->planned) return fail(ctx, GSK_ERR_STATE, "gsk_execute called before gsk_plan");
  if (first < 0 || count < 0 || first + count > ctx->n_targets) return fail(ctx, GSK_ERR_INVALID, "target range out of bounds");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  const bool phase_timing = ctx->phase_timing;
  int launches = 0;
  double ms_search = 0.0, ms_solve = 0.0;
  GSK_CUDA_CHECK(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
  int rc = GSK_OK;
  const bool kriging = ctx->prob.solver == GSK_SOLVER_KRIGING;
  // the per-location body that follows the search: Kriging (assemble + factor + solve) or the IDW / LWR epilogue
  auto launch_body = [&](cudaStream_t st, long long f, long long c, const int *nn, const int *nbr, long long off) -> int {
    if (kriging) return gsk_launch_local_solve(ctx, st, f, c, nn, nbr, off, &launches);
    return gsk_launch_simple_solver(ctx, st, f, c, nn, nbr, off, nullptr, &launches);
  };
  if (ctx->prob.max_neighbors == 0) {
    if (ctx->loo) {
      if (phase_timing) cudaEventRecord(ctx->ev[4], ctx->stream);
      rc = gsk_global_loo(ctx, first, count, d_nneigh, &launches);
      if (rc == GSK_OK && phase_timing) {
        cudaEventRecord(ctx->ev[5], ctx->stream);
        cudaEventSynchronize(ctx->ev[5]);
        float b2 = 0.f;
        cudaEventElapsedTime(&b2, ctx->ev[4], ctx->ev[5]);
        ms_solve += b2;
      }
    } else if (kriging) {
      rc = gsk_global_execute(ctx, first, count, d_nneigh, &launches);
    } else {
      rc = gsk_launch_simple_solver(ctx, ctx->stream, first, count, nullptr, nullptr, 0, d_nneigh, &launches);
    }
    if (rc != GSK_OK) return rc;
  } else if (!ctx->tg.is_grid && count > 0) {
    // explicit points: process the slab in bin-sorted order (spatially coherent CTAs), then scatter back
    const int k = ctx->prob.max_neighbors;
    int *perm = nullptr, *nn_s = nullptr, *nbr_s = nullptr;
    double *sx = nullptr, *sy = nullptr, *sz = nullptr, *ms = nullptr, *vs = nullptr;
    // after a values-only update the bin order and the neighbour lists of the same range are still valid
    const bool reuse = !ctx->loo && ctx->nbr_reuse && ctx->nbr_cached && ctx->nbr_first == first && ctx->nbr_count == count &&
                       ctx->pt_perm;
    if (reuse) {
      perm = ctx->pt_perm; sx = ctx->pt_sx; sy = ctx->pt_sy; sz = ctx->pt_sz;
    } else {
      ctx->nbr_cached = false;
      if ((rc = gsk_points_sort(ctx, first, count, &perm, &sx, &sy, &sz)) != GSK_OK) return rc;
    }
    if ((rc = gsk_buf(ctx, BUF_PT_MEAN, sizeof(double) * (size_t)count, (void **)&ms)) != GSK_OK) return rc;
    if ((rc = gsk_buf(ctx, BUF_PT_VAR, sizeof(double) * (size_t)count, (void **)&vs)) != GSK_OK) return rc;
    if ((rc = gsk_buf(ctx, BUF_PT_NN, sizeof(int) * (size_t)count, (void **)&nn_s)) != GSK_OK) return rc;
    if ((rc = gsk_buf(ctx, BUF_PT_NBR, sizeof(int) * (size_t)count * k, (void **)&nbr_s)) != GSK_OK) return rc;
    const GskTargets tg_saved = ctx->tg;
    const GskOut out_saved = ctx->out;
    ctx->tg.pts[0] = sx; ctx->tg.pts[1] = sy; ctx->tg.pts[2] = sz;
    ctx->tg.npts = count;
    ctx->out = GskOut{};
    ctx->out.n = 1;
    ctx->out.mean[0] = ms;
    ctx->out.var[0] = vs;
    if (phase_timing) cudaEventRecord(ctx->ev[3], ctx->stream);
    if (ctx->loo) {
      // leave-one-out: the k+1 nearest in the exact (d², index) order contain the k nearest j != i, so search one more
      // and drop the target's own index (k + 1 <= n_samples: validate_loo)
      rc = ensure(ctx, (void **)&ctx->d_nn, &ctx->cap_nn, sizeof(int) * (size_t)count);
      if (rc == GSK_OK) rc = ensure(ctx, (void **)&ctx->d_nbr, &ctx->cap_nbr, sizeof(int) * (size_t)count * (k + 1));
      if (rc == GSK_OK) rc = gsk_launch_search(ctx, ctx->stream, 0, count, k + 1, ctx->d_nn, ctx->d_nbr, &launches);
      if (rc == GSK_OK) rc = gsk_points_loo_compact(ctx, perm, first, count, k, ctx->d_nn, ctx->d_nbr, nn_s, nbr_s);
      ++launches;
    } else if (!reuse) {
      rc = gsk_launch_search(ctx, ctx->stream, 0, count, k, nn_s, nbr_s, &launches);
    }
    if (phase_timing) cudaEventRecord(ctx->ev[4], ctx->stream);
    ctx->cols.perm = perm;  // the columns epilogue writes its rows in slab order itself
    if (rc == GSK_OK) rc = launch_body(ctx->stream, 0, count, nn_s, nbr_s, 0);
    ctx->cols.perm = nullptr;
    ctx->tg = tg_saved;
    ctx->out = out_saved;
    if (rc != GSK_OK) return rc;
    ctx->nbr_cached = !ctx->loo;  // leave-one-out lists belong to no problem a later gsk_execute could plan
    ctx->nbr_first = first; ctx->nbr_count = count;
    ctx->pt_perm = perm; ctx->pt_sx = sx; ctx->pt_sy = sy; ctx->pt_sz = sz;
    if (phase_timing) {
      cudaEventRecord(ctx->ev[5], ctx->stream);
      cudaEventSynchronize(ctx->ev[5]);
      float a = 0.f, b2 = 0.f;
      cudaEventElapsedTime(&a, ctx->ev[3], ctx->ev[4]);
      cudaEventElapsedTime(&b2, ctx->ev[4], ctx->ev[5]);
      ms_search += a;
      ms_solve += b2;
    }
    rc = gsk_points_unscatter(ctx, perm, count, ms, vs, ctx->out, nn_s, d_nneigh, nbr_s, d_neigh_idx, k);
    if (rc != GSK_OK) return rc;
    launches += 4;
  } else {
    const int k = ctx->prob.max_neighbors;
    // chunks of ~4M targets bound the neighbour-list scratch (4k+4 B per target: 1.1 GB at k = 64); chunk edges are aligned
    // to whole tile layers of the grid where that is cheap. 4M instead of 1M targets per launch: the search kernel's
    // 8 192 CTAs were 18.4 waves of the 444 resident ones, its last wave ran at half occupancy (C5 search 315 -> 308 ms
    // per 512^3 grid, C3a 13.6 -> 13.0 ms). (Running the search of chunk c+1 on a side stream while chunk c is solved
    // was measured on B200 in round 1: no gain — both kernels already fill the SMs.)
    static const int chunk_log2 = GSK_DEV_ENV("GSK_CHUNK_LOG2") ? atoi(GSK_DEV_ENV("GSK_CHUNK_LOG2")) : 22;  // development tunable
    long long chunk = 1ll << chunk_log2;
    if (ctx->tg.is_grid) {
      const int dim = ctx->tg.dim;
      long long unit = (dim == 3) ? ctx->tg.gdim[0] * ctx->tg.gdim[1] * 4 : (dim == 2 ? ctx->tg.gdim[0] * 8 : 128);
      if (unit <= (1ll << 21)) chunk = (chunk + unit - 1) / unit * unit;
    }
    chunk = std::min<long long>(chunk, std::max<long long>(count, 1));
    // Neighbour lists of the whole range are kept in the context's own scratch when they are at most 1 GiB: after a
    // values-only update (gsk_update_values arms `nbr_reuse`) the next execute of the same range skips the search.
    const bool keep = !d_nneigh && !d_neigh_idx && (size_t)count * (size_t)k * sizeof(int) <= ((size_t)1 << 30);
    const bool reuse = keep && ctx->nbr_reuse && ctx->nbr_cached && ctx->nbr_first == first && ctx->nbr_count == count &&
                       !ctx->pt_perm;
    if (!reuse) ctx->nbr_cached = false;
    const size_t scratch_targets = keep ? (size_t)count : (size_t)chunk;
    if (!d_nneigh) {
      rc = ensure(ctx, (void **)&ctx->d_nn, &ctx->cap_nn, sizeof(int) * scratch_targets);
      if (rc != GSK_OK) return rc;
    }
    if (!d_neigh_idx) {
      rc = ensure(ctx, (void **)&ctx->d_nbr, &ctx->cap_nbr, sizeof(int) * scratch_targets * k);
      if (rc != GSK_OK) return rc;
    }
    for (long long off = 0; off < count; off += chunk) {
      const long long cnt = std::min<long long>(chunk, count - off);
      int *nn = d_nneigh ? d_nneigh + off : ctx->d_nn + (keep ? (size_t)off : 0);
      int *nbr = d_neigh_idx ? d_neigh_idx + off * k : ctx->d_nbr + (keep ? (size_t)off * k : 0);
      if (phase_timing) cudaEventRecord(ctx->ev[3], ctx->stream);
      if (!reuse) {
        rc = gsk_launch_search(ctx, ctx->stream, first + off, cnt, k, nn, nbr, &launches);
        if (rc != GSK_OK) return rc;
      }
      if (phase_timing) cudaEventRecord(ctx->ev[4], ctx->stream);
      rc = launch_body(ctx->stream, first + off, cnt, nn, nbr, off);
      if (rc != GSK_OK) return rc;
      if (phase_timing) {
        cudaEventRecord(ctx->ev[5], ctx->stream);
        cudaEventSynchronize(ctx->ev[5]);
        float a = 0.f, b2 = 0.f;
        cudaEventElapsedTime(&a, ctx->ev[3], ctx->ev[4]);
        cudaEventElapsedTime(&b2, ctx->ev[4], ctx->ev[5]);
        ms_search += a;
        ms_solve += b2;
      }
    }
    if (keep && count > 0) {
      ctx->nbr_cached = true;
      ctx->nbr_first = first; ctx->nbr_count = count;
      ctx->pt_perm = nullptr;
    }
  }
  GSK_CUDA_CHECK(ctx, cudaEventRecord(ctx->ev[1], ctx->stream));
  ctx->timing.ms_search = ms_search;
  ctx->timing.ms_solve = ms_solve;
  ctx->timing.launches = launches;
  ctx->timing.targets = count;
  ctx->timing_pending = true;
  return GSK_OK;
}

extern "C" GSK_API int gsk_set_phase_timing(gsk_ctx *ctx, int on) {
  if (!ctx) return GSK_ERR_INVALID;
  ctx->phase_timing = on != 0;
  return GSK_OK;
}

extern "C" GSK_API int gsk_get_timing(const gsk_ctx *cctx, gsk_timing *out) {
  gsk_ctx *ctx = const_cast<gsk_ctx *>(cctx);
  if (!ctx || !out) return GSK_ERR_INVALID;
  if (ctx->timing_pending) {
    cudaSetDevice(ctx->device);
    if (cudaEventSynchronize(ctx->ev[1]) == cudaSuccess) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[1]) == cudaSuccess) ctx->timing.ms_total = ms;
    }
    ctx->timing_pending = false;
  }
  *out = ctx->timing;
  return GSK_OK;
}

// ---------------------------------------------------------------------------------------------
// values-only update and the identity of the resident plan
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void set_values_kernel(double4 *rec, const double *v, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) rec[i].w = v[i];
}

// 64-bit hash of an array of doubles (four interleaved FNV-style lanes; identity check, not cryptography)
unsigned long long hash_doubles(const double *p, long long n, unsigned long long seed) {
  unsigned long long h[4] = {seed ^ 0x9E3779B97F4A7C15ull, seed ^ 0xC2B2AE3D27D4EB4Full, seed ^ 0x165667B19E3779F9ull,
                             seed ^ 0x27D4EB2F165667C5ull};
  if (!p) return seed;
  long long i = 0;
  for (; i + 4 <= n; i += 4)
    for (int l = 0; l < 4; ++l) {
      unsigned long long b;
      memcpy(&b, p + i + l, 8);
      h[l] = (h[l] ^ b) * 0x100000001B3ull;
      h[l] ^= h[l] >> 32;
    }
  for (; i < n; ++i) {
    unsigned long long b;
    memcpy(&b, p + i, 8);
    h[0] = (h[0] ^ b) * 0x100000001B3ull;
    h[0] ^= h[0] >> 32;
  }
  return h[0] ^ (h[1] * 3) ^ (h[2] * 5) ^ (h[3] * 7) ^ (unsigned long long)n;
}

// everything of the problem except the sample VALUES and the slab: scalars (pointers zeroed) + array hashes
void problem_identity(const gsk_problem *p, gsk_problem *scalars, unsigned long long *geom, unsigned long long *vals) {
  *scalars = *p;
  for (int d = 0; d < 3; ++d) { scalars->coords[d] = nullptr; scalars->point_coords[d] = nullptr; scalars->support_offsets[d] = nullptr; }
  scalars->values = nullptr;
  scalars->target_order = nullptr;
  scalars->target_first = 0;
  scalars->target_count = 0;
  scalars->flags &= ~(uint32_t)GSK_FLAG_REUSE_PLAN;
  unsigned long long g = 0x51ED270B153A4D1Full;
  const int64_t T = gsk_num_targets(p);
  for (int d = 0; d < p->dim; ++d) {
    g = hash_doubles(p->coords[d], p->n_samples, g + d);
    g = hash_doubles(p->support_offsets[d], p->n_support, g + 8 + d);
    if (p->grid_dims[0] == 0) g = hash_doubles(p->point_coords[d], p->n_points, g + 16 + d);
  }
  if (p->target_order) g = hash_doubles(reinterpret_cast<const double *>(p->target_order), T, g + 32);  // 8-byte words
  else g ^= 0xABCDull;
  *geom = g;
  *vals = hash_doubles(p->values, p->n_samples, 0x7F4A7C15ull);
}
}  // namespace

extern "C" GSK_API int gsk_update_values(gsk_ctx *ctx, const double *values, int64_t n_values) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!ctx->planned) return fail(ctx, GSK_ERR_STATE, "gsk_update_values called before gsk_plan");
  if (!values || n_values != ctx->prob.n_samples)
    return fail(ctx, GSK_ERR_INVALID, "gsk_update_values: values must hold n_samples of the planned problem");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  const long long n = n_values;
  double *hst = nullptr, *dv = nullptr;
  int rc;
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));  // the staging buffer may still feed an earlier copy
  if ((rc = gsk_host_stage(ctx, sizeof(double) * (size_t)n, (void **)&hst)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_VALS, sizeof(double) * (size_t)n, (void **)&dv)) != GSK_OK) return rc;
  memcpy(hst, values, sizeof(double) * (size_t)n);
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(dv, hst, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  set_values_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_rec_orig, dv, n);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  if (ctx->prob.max_neighbors == 0 && ctx->prob.solver == GSK_SOLVER_KRIGING) {
    if ((rc = gsk_global_update_values(ctx)) != GSK_OK) return rc;
  }
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  ctx->nbr_reuse = true;  // the neighbour lists of the last execute stay valid: same coordinates
  if (ctx->key_valid) ctx->key_vals = hash_doubles(values, n, 0x7F4A7C15ull);
  return GSK_OK;
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_update_values: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_update_values: ") + e.what());
}

// ---------------------------------------------------------------------------------------------
// one-shot host-buffer call: plan + execute + copies
// ---------------------------------------------------------------------------------------------
static int krige_pieces(gsk_ctx *ctx, const gsk_problem *p, int64_t first, int64_t count, double *mean_out, double *var_out,
                        int32_t *nneigh_out, int32_t *neigh_idx_out) {
  const int k = p->max_neighbors;
  int rc = ensure(ctx, (void **)&ctx->d_mean, &ctx->cap_out, sizeof(double) * 2 * (size_t)count);
  if (rc != GSK_OK) return rc;
  double *d_mean = ctx->d_mean, *d_var = ctx->d_mean + count;
  int *d_nn = nullptr, *d_idx = nullptr;
  if (nneigh_out) {
    rc = ensure(ctx, (void **)&ctx->d_nn_out, &ctx->cap_nn_out, sizeof(int) * (size_t)count);
    if (rc != GSK_OK) return rc;
    d_nn = ctx->d_nn_out;
  }
  if (neigh_idx_out && k > 0) {
    rc = ensure(ctx, (void **)&ctx->d_nbr_out, &ctx->cap_nbr_out, sizeof(int) * (size_t)count * k);
    if (rc != GSK_OK) return rc;
    d_idx = ctx->d_nbr_out;
  }
  // The slab is computed in pieces of 40 / 30 / 20 / 10 %: the device→host copies of a finished piece run on the side
  // stream while the next piece is being computed (they overlap only when the host buffers are page-locked), and only
  // the last, smallest piece's copies are exposed after the compute has finished. A request for the neighbour lists
  // (parity tests) or explicit points runs as one piece.
  long long bounds[5] = {0, count, count, count, count};
  int npieces = 1;
  if (count >= (1ll << 19) && ctx->tg.is_grid && !d_idx) {
    const int dim = ctx->tg.dim;
    const long long unit = (dim == 3) ? ctx->tg.gdim[0] * ctx->tg.gdim[1] * 4 : (dim == 2 ? ctx->tg.gdim[0] * 8 : 128);
    const double cut[3] = {0.4, 0.7, 0.9};
    npieces = 4;
    for (int i = 0; i < 3; ++i) {
      long long b = (long long)(cut[i] * (double)count);
      if (unit <= count / 8) b = (b + unit - 1) / unit * unit;
      bounds[i + 1] = std::min<long long>(std::max<long long>(b, bounds[i]), count);
    }
    bounds[4] = count;
  }
  // from here on every error path drains both streams first: copies into the caller's (possibly page-locked) host
  // buffers may be in flight, and the caller is free to release them as soon as this function returns
  auto drain = [&](int code) {
    cudaStreamSynchronize(ctx->stream2);
    cudaStreamSynchronize(ctx->stream);
    return code;
  };
  // Are the caller's arrays page-locked? A plain Julia Vector / numpy array is not, and an asynchronous device→host
  // copy into pageable memory degenerates into a slow blocking one (measured: 8× the whole call on C5 slabs). Pageable
  // outputs are therefore filled through two page-locked 8 MB staging buffers: DMA into one while the host copies the
  // other out; piece i is drained while the kernels of piece i+1 — already enqueued — run.
  auto is_pinned = [](const void *ptr) {
    if (!ptr) return true;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
  };
  const bool pinned = is_pinned(mean_out) && is_pinned(var_out) && is_pinned(nneigh_out) && is_pinned(neigh_idx_out);
  constexpr size_t STG = (size_t)8 << 20;
  char *stg[2] = {nullptr, nullptr};
  if (!pinned) {
    if (ctx->h_out_cap < 2 * STG) {
      if (ctx->h_out) cudaFreeHost(ctx->h_out);
      ctx->h_out = nullptr;
      ctx->h_out_cap = 0;
      if (cudaHostAlloc(&ctx->h_out, 2 * STG, cudaHostAllocDefault) != cudaSuccess)
        return fail(ctx, GSK_ERR_NOMEM, "pinned staging allocation failed");
      ctx->h_out_cap = 2 * STG;
    }
    stg[0] = (char *)ctx->h_out;
    stg[1] = (char *)ctx->h_out + STG;
  }
  struct Pend { char *dst; size_t bytes; bool live; } pend[2] = {{nullptr, 0, false}, {nullptr, 0, false}};
  int tog = 0;
  cudaError_t ce = cudaSuccess;
  auto flush_slot = [&](int b) {
    if (!pend[b].live) return;
    if (ce == cudaSuccess) ce = cudaEventSynchronize(ctx->ev_solve[b]);
    if (ce == cudaSuccess) memcpy(pend[b].dst, stg[b], pend[b].bytes);
    pend[b].live = false;
  };
  auto staged_copy = [&](void *dst, const void *src, size_t bytes) {
    for (size_t o = 0; o < bytes && ce == cudaSuccess; o += STG) {
      const size_t nb = std::min(STG, bytes - o);
      flush_slot(tog);
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(stg[tog], (const char *)src + o, nb, cudaMemcpyDeviceToHost, ctx->stream2);
      if (ce == cudaSuccess) ce = cudaEventRecord(ctx->ev_solve[tog], ctx->stream2);
      pend[tog] = {(char *)dst + o, nb, true};
      tog ^= 1;
    }
  };
  auto copy_piece = [&](long long off, long long cnt) {  // stream2 already waits for the piece's kernels
    if (pinned) {
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(mean_out + off, d_mean + off, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost, ctx->stream2);
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(var_out + off, d_var + off, sizeof(double) * (size_t)cnt, cudaMemcpyDeviceToHost, ctx->stream2);
      if (ce == cudaSuccess && d_nn)
        ce = cudaMemcpyAsync(nneigh_out + off, d_nn + off, sizeof(int) * (size_t)cnt, cudaMemcpyDeviceToHost, ctx->stream2);
      if (ce == cudaSuccess && d_idx)
        ce = cudaMemcpyAsync(neigh_idx_out + off * k, d_idx + off * k, sizeof(int) * (size_t)cnt * k, cudaMemcpyDeviceToHost, ctx->stream2);
      return;
    }
    staged_copy(mean_out + off, d_mean + off, sizeof(double) * (size_t)cnt);
    staged_copy(var_out + off, d_var + off, sizeof(double) * (size_t)cnt);
    if (d_nn) staged_copy(nneigh_out + off, d_nn + off, sizeof(int) * (size_t)cnt);
    if (d_idx) staged_copy(neigh_idx_out + off * k, d_idx + off * k, sizeof(int) * (size_t)cnt * k);
  };
  long long prev_off = -1, prev_cnt = 0;
  for (int pi = 0; pi < npieces; ++pi) {
    const long long off = bounds[pi], cnt = bounds[pi + 1] - bounds[pi];
    if (cnt <= 0) continue;
    rc = gsk_execute(ctx, first + off, cnt, d_mean + off, d_var + off, d_nn ? d_nn + off : nullptr,
                     d_idx ? d_idx + off * k : nullptr);
    if (rc != GSK_OK) return drain(rc);
    const int eb = pi & 1;
    if (ce == cudaSuccess) ce = cudaEventRecord(ctx->ev_search[eb], ctx->stream);  // "piece done" marker
    if (pinned) {
      if (ce == cudaSuccess) ce = cudaStreamWaitEvent(ctx->stream2, ctx->ev_search[eb], 0);
      copy_piece(off, cnt);
    } else {
      // the previous piece's results leave while this piece's kernels run (its marker was recorded a round ago)
      if (prev_off >= 0) copy_piece(prev_off, prev_cnt);
      if (ce == cudaSuccess) ce = cudaStreamWaitEvent(ctx->stream2, ctx->ev_search[eb], 0);
      prev_off = off;
      prev_cnt = cnt;
    }
    if (ce != cudaSuccess) {
      ctx->err = std::string("gsk_krige: result copy failed: ") + cudaGetErrorString(ce);
      return drain(GSK_ERR_CUDA);
    }
  }
  if (!pinned) {
    if (prev_off >= 0) copy_piece(prev_off, prev_cnt);
    flush_slot(0);
    flush_slot(1);
    if (ce != cudaSuccess) {
      ctx->err = std::string("gsk_krige: result copy failed: ") + cudaGetErrorString(ce);
      return drain(GSK_ERR_CUDA);
    }
  }
  ctx->timing.targets = count;
  ce = cudaStreamSynchronize(ctx->stream2);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) {
    ctx->err = std::string("gsk_krige: ") + cudaGetErrorString(ce);
    return GSK_ERR_CUDA;
  }
  return GSK_OK;
}

extern "C" GSK_API int gsk_krige(gsk_ctx *ctx, const gsk_problem *p, double *mean_out, double *var_out, int32_t *nneigh_out,
                         int32_t *neigh_idx_out) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!mean_out || !var_out) return fail(ctx, GSK_ERR_INVALID, "mean_out / var_out are NULL");
  int rc = GSK_OK;
  if (p && (p->flags & GSK_FLAG_REUSE_PLAN) && p->abi_version == GSK_ABI_VERSION) {
    // same problem as the resident plan? then nothing is uploaded or rebuilt; same problem with other VALUES (the
    // conditional-simulation callers, fft.jl:184-188)? then only the values go up and bins / neighbour lists /
    // L and L⁻¹ stay. The flag is opt-in: without it the library never depends on what an earlier call was given.
    rc = validate(ctx, p);
    if (rc != GSK_OK) return rc;
    gsk_problem sc;
    unsigned long long geom = 0, vals = 0;
    problem_identity(p, &sc, &geom, &vals);
    if (ctx->planned && ctx->key_valid && geom == ctx->key_geom && memcmp(&sc, &ctx->key_prob, sizeof(sc)) == 0) {
      if (vals != ctx->key_vals) {
        rc = gsk_update_values(ctx, p->values, p->n_samples);
        if (rc != GSK_OK) return rc;
      } else {
        ctx->nbr_reuse = true;
      }
      ctx->timing.ms_plan = 0.0;
    } else {
      rc = gsk_plan(ctx, p);
      if (rc != GSK_OK) return rc;
      ctx->key_prob = sc;
      ctx->key_geom = geom;
      ctx->key_vals = vals;
      ctx->key_valid = true;
    }
  } else {
    rc = gsk_plan(ctx, p);
    if (rc != GSK_OK) return rc;
  }
  const int64_t T = ctx->n_targets;
  const int64_t first = p->target_first;
  const int64_t count = p->target_count < 0 ? T - first : p->target_count;
  if (count == 0) return GSK_OK;
  return krige_pieces(ctx, p, first, count, mean_out, var_out, nneigh_out, neigh_idx_out);
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  if (ctx) { cudaStreamSynchronize(ctx->stream2); cudaStreamSynchronize(ctx->stream); }
  return fail(ctx, GSK_ERR_NOMEM, "gsk_krige: out of host memory");
} catch (const std::exception &e) {
  if (ctx) { cudaStreamSynchronize(ctx->stream2); cudaStreamSynchronize(ctx->stream); }
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_krige: ") + e.what());
}

// ---------------------------------------------------------------------------------------------
// leave-one-out cross-validation: the samples are the targets, each kriged without itself
// ---------------------------------------------------------------------------------------------
static int validate_loo(gsk_ctx *ctx, const gsk_problem *p) {
  if (!p) return fail(ctx, GSK_ERR_INVALID, "problem is NULL");
  if (p->abi_version != GSK_ABI_VERSION) return fail(ctx, GSK_ERR_INVALID, "gsk_problem.abi_version mismatch");
  if (p->solver != GSK_SOLVER_KRIGING)
    return fail(ctx, GSK_ERR_UNSUPPORTED, "gsk_krige_loo: leave-one-out is implemented for the Kriging solver only");
  if (p->grid_dims[0] != 0 || p->n_points != 0 || p->target_order)
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: the targets are the samples (grid_dims[0] = 0, n_points = 0, "
                                      "target_order = NULL)");
  if (p->n_support != 1) return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: point support only (n_support = 1)");
  for (int d = 0; d < 3; ++d)
    if (p->support_offsets[d] && p->support_offsets[d][0] != 0.0)
      return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: the support offset must be zero");
  if (p->flags & GSK_FLAG_REUSE_PLAN)
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: GSK_FLAG_REUSE_PLAN does not apply (no plan is kept)");
  if (p->n_samples < 2) return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: n_samples must be >= 2");
  if (p->max_neighbors > p->n_samples - 1)
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: max_neighbors must be clamped to n_samples - 1 by the host (each "
                                      "fold holds n_samples - 1 samples)");
  const int64_t first = p->target_first, count = p->target_count < 0 ? p->n_samples - first : p->target_count;
  if (first < 0 || count < 0 || first + count > p->n_samples)
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_loo: sample slab out of range");
  return GSK_OK;
}

extern "C" GSK_API int gsk_krige_loo(gsk_ctx *ctx, const gsk_problem *p, double *mean_out, double *var_out,
                                     int32_t *nneigh_out, int32_t *neigh_idx_out) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!mean_out || !var_out) return fail(ctx, GSK_ERR_INVALID, "mean_out / var_out are NULL");
  int rc = validate_loo(ctx, p);
  if (rc != GSK_OK) return rc;
  // the explicit point list of the plan is the sample coordinates themselves: target t is sample t
  gsk_problem q = *p;
  q.n_points = p->n_samples;
  for (int d = 0; d < 3; ++d) q.point_coords[d] = p->coords[d];
  rc = gsk_plan(ctx, &q);
  if (rc == GSK_OK) {
    const int64_t first = p->target_first, count = p->target_count < 0 ? p->n_samples - first : p->target_count;
    ctx->loo = true;
    if (count > 0) rc = krige_pieces(ctx, &q, first, count, mean_out, var_out, nneigh_out, neigh_idx_out);
    ctx->loo = false;
  }
  // nothing of the leave-one-out plan (sample-target bins order, self-excluded lists) may serve a later gsk_execute
  cudaStreamSynchronize(ctx->stream);
  free_plan(ctx);
  return rc;
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  if (ctx) { ctx->loo = false; cudaStreamSynchronize(ctx->stream2); cudaStreamSynchronize(ctx->stream); free_plan(ctx); }
  return fail(ctx, GSK_ERR_NOMEM, "gsk_krige_loo: out of host memory");
} catch (const std::exception &e) {
  if (ctx) { ctx->loo = false; cudaStreamSynchronize(ctx->stream2); cudaStreamSynchronize(ctx->stream); free_plan(ctx); }
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_krige_loo: ") + e.what());
}

// ---------------------------------------------------------------------------------------------
// many value columns over one sample set: the geometry (search, factorisation) once, applied to every column
// ---------------------------------------------------------------------------------------------
extern "C" GSK_API int gsk_krige_columns(gsk_ctx *ctx, const gsk_problem *p, int32_t n_cols, const double *values,
                                         double *mean_out, double *var_out, int32_t *nneigh_out, int32_t *neigh_idx_out,
                                         double *weights_out, double *lagrange_out) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!mean_out || !var_out) return fail(ctx, GSK_ERR_INVALID, "mean_out / var_out are NULL");
  if (!p) return fail(ctx, GSK_ERR_INVALID, "problem is NULL");
  if (p->values)
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_columns: prob->values must be NULL (the values are the columns)");
  if (n_cols < 1 || !values) return fail(ctx, GSK_ERR_INVALID, "gsk_krige_columns: n_cols must be >= 1 and values non-NULL");
  if (p->flags & GSK_FLAG_REUSE_PLAN)
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_columns: GSK_FLAG_REUSE_PLAN does not apply (no plan is kept)");
  if (p->solver != GSK_SOLVER_KRIGING)
    return fail(ctx, GSK_ERR_UNSUPPORTED, "gsk_krige_columns: implemented for the Kriging solver only");
  if (p->max_neighbors == 0 && (weights_out || lagrange_out))
    return fail(ctx, GSK_ERR_INVALID, "gsk_krige_columns: weights_out / lagrange_out are for the local path only "
                                      "(max_neighbors > 0)");
  if (p->n_samples < 1) return fail(ctx, GSK_ERR_INVALID, "n_samples must be >= 1");
  const long long n = p->n_samples;
  const int m = n_cols;
  // the plan takes column 0 as its values (the kernels' own single-column mean is computed and discarded)
  std::vector<double> v0((size_t)n);
  for (long long i = 0; i < n; ++i) v0[(size_t)i] = values[(size_t)i * m];
  gsk_problem q = *p;
  q.values = v0.data();
  int rc = gsk_plan(ctx, &q);
  const int64_t first = p->target_first, count = rc == GSK_OK ? (p->target_count < 0 ? ctx->n_targets - first : p->target_count) : 0;
  const int k = p->max_neighbors, c = ctx->nterms;
  // pieces of the slab whose per-column means fit in 2 GiB of device memory
  const long long piece = std::max<long long>(1, std::min<long long>(count, (2ll << 30) / (8ll * m)));
  double *d_z = nullptr, *d_cm = nullptr, *d_mv = nullptr, *d_w = nullptr, *d_lag = nullptr;
  auto copy_out = [&](void *dst, const void *src, size_t bytes) -> int {
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return GSK_OK;
  };
  if (rc == GSK_OK && count > 0) rc = gsk_buf(ctx, BUF_C_Z, sizeof(double) * (size_t)n * m, (void **)&d_z);
  if (rc == GSK_OK && count > 0) rc = gsk_buf(ctx, BUF_C_MEAN, sizeof(double) * (size_t)piece * m, (void **)&d_cm);
  if (rc == GSK_OK && count > 0) rc = gsk_buf(ctx, BUF_C_MV, sizeof(double) * 2 * (size_t)piece, (void **)&d_mv);
  if (rc == GSK_OK && count > 0 && weights_out) rc = gsk_buf(ctx, BUF_C_W, sizeof(double) * (size_t)piece * k, (void **)&d_w);
  if (rc == GSK_OK && count > 0 && lagrange_out && c > 0)
    rc = gsk_buf(ctx, BUF_C_LAG, sizeof(double) * (size_t)piece * c, (void **)&d_lag);
  if (rc == GSK_OK && count > 0 && nneigh_out) rc = ensure(ctx, (void **)&ctx->d_nn_out, &ctx->cap_nn_out, sizeof(int) * (size_t)piece);
  if (rc == GSK_OK && count > 0 && neigh_idx_out && k > 0)
    rc = ensure(ctx, (void **)&ctx->d_nbr_out, &ctx->cap_nbr_out, sizeof(int) * (size_t)piece * k);
  if (rc == GSK_OK && count > 0) {
    if (cudaMemcpyAsync(d_z, values, sizeof(double) * (size_t)n * m, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
      rc = fail(ctx, GSK_ERR_CUDA, "gsk_krige_columns: value upload failed");
    ctx->cols = GskCols{};
    ctx->cols.active = true;
    ctx->cols.z = d_z;
    ctx->cols.m = m;
    ctx->cols.mean = d_cm;
    ctx->cols.w = d_w;
    ctx->cols.lag = d_lag;
    if (rc == GSK_OK && k == 0) rc = gsk_global_column_weights(ctx, d_z, m);
    for (long long off = 0; off < count && rc == GSK_OK; off += piece) {
      const long long cnt = std::min<long long>(piece, count - off);
      int *d_nn = nneigh_out ? ctx->d_nn_out : nullptr, *d_idx = (neigh_idx_out && k > 0) ? ctx->d_nbr_out : nullptr;
      rc = gsk_execute(ctx, first + off, cnt, d_mv, d_mv + piece, d_nn, d_idx);
      if (rc == GSK_OK) rc = copy_out(mean_out + off * m, d_cm, sizeof(double) * (size_t)cnt * m);
      if (rc == GSK_OK) rc = copy_out(var_out + off, d_mv + piece, sizeof(double) * (size_t)cnt);
      if (rc == GSK_OK && d_nn) rc = copy_out(nneigh_out + off, d_nn, sizeof(int) * (size_t)cnt);
      if (rc == GSK_OK && d_idx) rc = copy_out(neigh_idx_out + off * k, d_idx, sizeof(int) * (size_t)cnt * k);
      if (rc == GSK_OK && d_w) rc = copy_out(weights_out + off * k, d_w, sizeof(double) * (size_t)cnt * k);
      if (rc == GSK_OK && d_lag) rc = copy_out(lagrange_out + off * c, d_lag, sizeof(double) * (size_t)cnt * c);
      if (rc == GSK_OK) GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));  // the next piece reuses the buffers
    }
    ctx->timing.targets = count;
  }
  // like gsk_krige_loo: nothing of this call's plan serves a later gsk_execute
  cudaStreamSynchronize(ctx->stream);
  ctx->cols = GskCols{};
  free_plan(ctx);
  return rc;
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  if (ctx) { cudaStreamSynchronize(ctx->stream); ctx->cols = GskCols{}; free_plan(ctx); }
  return fail(ctx, GSK_ERR_NOMEM, "gsk_krige_columns: out of host memory");
} catch (const std::exception &e) {
  if (ctx) { cudaStreamSynchronize(ctx->stream); ctx->cols = GskCols{}; free_plan(ctx); }
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_krige_columns: ") + e.what());
}

// ---------------------------------------------------------------------------------------------
// LU Gaussian simulation (ref: src/simulation/lu.jl)
// ---------------------------------------------------------------------------------------------
extern "C" GSK_API int gsk_lu_plan(gsk_ctx *ctx, int dim, int64_t n_data, int64_t n_sim, const double *const *coords,
                                   const double *data_values, int vario_kind, double vario_range, double vario_sill,
                                   double vario_nugget, double gaussian_nugget_eps) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (dim < 1 || dim > 3 || n_data < 0 || n_sim < 1 || !coords || (n_data > 0 && !data_values))
    return fail(ctx, GSK_ERR_INVALID, "gsk_lu_plan: dim in 1..3, n_sim >= 1, coords and (for n_data > 0) data_values required");
  for (int d = 0; d < dim; ++d)
    if (!coords[d]) return fail(ctx, GSK_ERR_INVALID, "gsk_lu_plan: coords[d] is NULL for d < dim");
  if (vario_kind < 0 || vario_kind > 2) return fail(ctx, GSK_ERR_UNSUPPORTED, "unknown variogram kind");
  if (!(vario_range > 0.0) || !(vario_sill > 0.0) || !(vario_nugget >= 0.0) || !(gaussian_nugget_eps >= 0.0) ||
      !(vario_sill - vario_nugget - (vario_kind == GSK_VARIO_GAUSSIAN ? gaussian_nugget_eps : 0.0) > 0.0))
    return fail(ctx, GSK_ERR_INVALID, "range and sill must be > 0, the nugget below the sill");
  if (n_data + n_sim > 46000) return fail(ctx, GSK_ERR_UNSUPPORTED, "gsk_lu_plan: the dense factor of more than 46 000 points does not fit (lu.jl:60-62: small domains only)");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  free_plan(ctx);  // the buffers are shared with the Kriging plans
  ctx->lu_n = 0;
  const GskVario vg = make_vario(vario_kind, vario_range, vario_sill, vario_nugget, gaussian_nugget_eps);
  return gsk_lu_plan_impl(ctx, dim, n_data, n_sim, coords, data_values, vg);
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_lu_plan: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_lu_plan: ") + e.what());
}

extern "C" GSK_API int gsk_lu_sample(gsk_ctx *ctx, const double *w, double *y_out) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (ctx->lu_n <= 0) return fail(ctx, GSK_ERR_STATE, "gsk_lu_sample called before gsk_lu_plan");
  if (!w || !y_out) return fail(ctx, GSK_ERR_INVALID, "gsk_lu_sample: w / y_out are NULL");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  return gsk_lu_sample_impl(ctx, w, y_out);
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_lu_sample: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_lu_sample: ") + e.what());
}

#define GSK_SGS_MAX_NEIGHBORS 64
extern "C" GSK_API int gsk_sgs_plan(gsk_ctx *ctx, int dim, int64_t n, const double *const *coords, const int64_t *rank,
                                    int vario_kind, double vario_range, double vario_sill, double vario_nugget,
                                    double gaussian_nugget_eps, double mean, int min_neighbors, int max_neighbors,
                                    double ball_radius) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (dim < 1 || dim > 3 || n < 1 || !coords || !rank)
    return fail(ctx, GSK_ERR_INVALID, "gsk_sgs_plan: dim in 1..3, n >= 1, coords and rank required");
  for (int d = 0; d < dim; ++d)
    if (!coords[d]) return fail(ctx, GSK_ERR_INVALID, "gsk_sgs_plan: coords[d] is NULL for d < dim");
  if (n > 0x7fffffffll) return fail(ctx, GSK_ERR_UNSUPPORTED, "gsk_sgs_plan: more than 2^31-1 locations");
  if (vario_kind < 0 || vario_kind > 2) return fail(ctx, GSK_ERR_UNSUPPORTED, "unknown variogram kind");
  if (!(vario_range > 0.0) || !(vario_sill > 0.0) || !(vario_nugget >= 0.0) || !(gaussian_nugget_eps >= 0.0) ||
      !(vario_sill - vario_nugget - (vario_kind == GSK_VARIO_GAUSSIAN ? gaussian_nugget_eps : 0.0) > 0.0))
    return fail(ctx, GSK_ERR_INVALID, "range and sill must be > 0, the nugget below the sill");
  if (max_neighbors < 1 || min_neighbors < 0 || !std::isfinite(mean))
    return fail(ctx, GSK_ERR_INVALID, "gsk_sgs_plan: max_neighbors >= 1, min_neighbors >= 0, finite mean");
  if (max_neighbors > GSK_SGS_MAX_NEIGHBORS)
    return fail(ctx, GSK_ERR_UNSUPPORTED, "gsk_sgs_plan: max_neighbors above 64");
  if (!(ball_radius != ball_radius) && !(ball_radius > 0.0))
    return fail(ctx, GSK_ERR_INVALID, "gsk_sgs_plan: ball_radius must be > 0 (or NaN for none)");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  free_plan(ctx);  // the buffers are shared with the Kriging plans
  const GskVario vg = make_vario(vario_kind, vario_range, vario_sill, vario_nugget, gaussian_nugget_eps);
  const int k = (int)std::min<int64_t>(max_neighbors, n);
  int rc = gsk_sgs_plan_impl(ctx, dim, n, coords, (const long long *)rank, vg, mean, min_neighbors, k, ball_radius);
  if (rc != GSK_OK) {
    cudaStreamSynchronize(ctx->stream);
    free_plan(ctx);
  }
  return rc;
} catch (const std::bad_alloc &) {  // no exception may cross the C ABI
  return fail(ctx, GSK_ERR_NOMEM, "gsk_sgs_plan: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_sgs_plan: ") + e.what());
}

extern "C" GSK_API int gsk_sgs_sample(gsk_ctx *ctx, int n_realizations, const double *values, const double *z,
                                      double *out) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!ctx->sgs) return fail(ctx, GSK_ERR_STATE, "gsk_sgs_sample called before gsk_sgs_plan");
  if (n_realizations < 1 || !z || !out) return fail(ctx, GSK_ERR_INVALID, "gsk_sgs_sample: n_realizations >= 1, z and out required");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  return gsk_sgs_sample_impl(ctx, n_realizations, values, z, out, false);
} catch (const std::bad_alloc &) {
  return fail(ctx, GSK_ERR_NOMEM, "gsk_sgs_sample: out of host memory");
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_sgs_sample: ") + e.what());
}

extern "C" GSK_API int gsk_sgs_sample_device(gsk_ctx *ctx, int n_realizations, const double *d_values, const double *d_z,
                                             double *d_out) try {
  if (!ctx) return GSK_ERR_INVALID;
  if (!ctx->sgs) return fail(ctx, GSK_ERR_STATE, "gsk_sgs_sample_device called before gsk_sgs_plan");
  if (n_realizations < 1 || !d_z || !d_out)
    return fail(ctx, GSK_ERR_INVALID, "gsk_sgs_sample_device: n_realizations >= 1, d_z and d_out required");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  return gsk_sgs_sample_impl(ctx, n_realizations, d_values, d_z, d_out, true);
} catch (const std::exception &e) {
  return fail(ctx, GSK_ERR_STATE, std::string("gsk_sgs_sample_device: ") + e.what());
}

extern "C" GSK_API int gsk_sgs_weights(gsk_ctx *ctx, int32_t *nneigh_out, int32_t *neigh_idx_out, double *weights_out,
                                       double *sigma_out) {
  if (!ctx) return GSK_ERR_INVALID;
  if (!ctx->sgs) return fail(ctx, GSK_ERR_STATE, "gsk_sgs_weights called before gsk_sgs_plan");
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  return gsk_sgs_weights_impl(ctx, nneigh_out, neigh_idx_out, weights_out, sigma_out);
}

extern "C" GSK_API int gsk_measure_fp64_peak(gsk_ctx *ctx, double *dfma_tflops, double *dmma_tflops) {
  if (!ctx || !dfma_tflops || !dmma_tflops) return GSK_ERR_INVALID;
  GSK_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
  return gsk_peak_measure(ctx, dfma_tflops, dmma_tflops);
}

// ---------------------------------------------------------------------------------------------
// single-process multi-GPU: one host thread + one cached context per piece
// ---------------------------------------------------------------------------------------------
namespace {
std::mutex g_multi_mutex;
std::vector<gsk_ctx *> g_multi_ctx;   // slot i serves piece i (re-created if the device id changes)
}  // namespace

// destroys the contexts gsk_krige_multi keeps between calls (device buffers, streams); the next call re-creates them
extern "C" GSK_API void gsk_krige_multi_release(void) {
  std::lock_guard<std::mutex> lock(g_multi_mutex);
  for (gsk_ctx *&c : g_multi_ctx) {
    if (c) gsk_destroy(c);
    c = nullptr;
  }
  g_multi_ctx.clear();
}

extern "C" GSK_API int gsk_krige_multi(const int *device_ids, int n_devices, const gsk_problem *p, double *mean_out,
                                       double *var_out, int32_t *nneigh_out, int32_t *neigh_idx_out, char *errbuf,
                                       int errbuf_len) try {
  auto set_err = [&](const std::string &m) {
    if (errbuf && errbuf_len > 0) {
      strncpy(errbuf, m.c_str(), (size_t)errbuf_len - 1);
      errbuf[errbuf_len - 1] = 0;
    }
  };
  if (!device_ids || n_devices < 1 || n_devices > 64 || !p || !mean_out || !var_out) {
    set_err("gsk_krige_multi: invalid arguments");
    return GSK_ERR_INVALID;
  }
  std::lock_guard<std::mutex> lock(g_multi_mutex);  // one multi-GPU call at a time per process
  if ((int)g_multi_ctx.size() < n_devices) g_multi_ctx.resize(n_devices, nullptr);
  for (int i = 0; i < n_devices; ++i) {
    if (g_multi_ctx[i] && g_multi_ctx[i]->device != device_ids[i]) {
      gsk_destroy(g_multi_ctx[i]);
      g_multi_ctx[i] = nullptr;
    }
    if (!g_multi_ctx[i]) {
      int rc = gsk_create(&g_multi_ctx[i], device_ids[i]);
      if (rc != GSK_OK) {
        set_err(gsk_last_error(nullptr));
        return rc;
      }
    }
  }
  const int64_t T = gsk_num_targets(p);
  const int64_t first = p->target_first;
  const int64_t count = p->target_count < 0 ? T - first : p->target_count;
  if (first < 0 || count < 0 || first + count > T) {
    set_err("gsk_krige_multi: target slab out of range");
    return GSK_ERR_INVALID;
  }
  const int k = p->max_neighbors;
  std::vector<int> rcs(n_devices, GSK_OK);
  std::vector<std::thread> workers;
  workers.reserve((size_t)n_devices);
  bool spawn_failed = false;
  for (int i = 0; i < n_devices && !spawn_failed; ++i) {
    try {
      workers.emplace_back([&, i]() {
        const int64_t lo = count * i / n_devices, hi = count * (i + 1) / n_devices;
        gsk_problem pi = *p;
        pi.target_first = first + lo;
        pi.target_count = hi - lo;
        rcs[i] = gsk_krige(g_multi_ctx[i], &pi, mean_out + lo, var_out + lo, nneigh_out ? nneigh_out + lo : nullptr,
                           (neigh_idx_out && k > 0) ? neigh_idx_out + lo * k : nullptr);
      });
    } catch (const std::exception &) {
      spawn_failed = true;  // joinable threads must be joined before anything else (std::terminate otherwise)
    }
  }
  for (auto &w : workers) w.join();
  if (spawn_failed) {
    set_err("gsk_krige_multi: could not start a worker thread");
    return GSK_ERR_NOMEM;
  }
  for (int i = 0; i < n_devices; ++i)
    if (rcs[i] != GSK_OK) {
      set_err(gsk_last_error(g_multi_ctx[i]));
      return rcs[i];
    }
  return GSK_OK;
} catch (const std::exception &e) {  // no exception may cross the C ABI (std::thread, allocations)
  if (errbuf && errbuf_len > 0) {
    strncpy(errbuf, e.what(), (size_t)errbuf_len - 1);
    errbuf[errbuf_len - 1] = 0;
  }
  return GSK_ERR_NOMEM;
}
