// local_solve.cu — picks the lanes/registers configuration of K3 for (k, extra rows) and launches it.
#include <stdlib.h>

#include "local_solve_small.cuh"
#include "local_solve_wpt.cuh"

int gsk_launch_local_solve(gsk_ctx *ctx, cudaStream_t st, long long first, long long count, const int *d_nn,
                           const int *d_nbr, long long out_off, int *launches) {
  GskLocalArgs a{};
  a.tg = ctx->tg;
  a.vg = ctx->vg;
  a.es = ctx->es;
  a.rec_orig = ctx->d_rec_orig;
  a.sup = ctx->d_sup;
  a.sup_unit = ctx->d_sup + 3 * (size_t)ctx->prob.n_support;
  a.nsup = ctx->prob.n_support;
  a.rhs_taylor = ctx->rhs_taylor;
  a.sup_tensor3 = ctx->sup_tensor3;
  for (int d = 0; d < 3; ++d)
    for (int i = 0; i < 3; ++i) a.sup_ax[d][i] = ctx->sup_ax[d][i];
  {
    const double ds = ctx->sup_rmax / ctx->vg.range;
    a.rhs_inr_lim2 = (ds < 1.0) ? (1.0 - ds) * (1.0 - ds) * (1.0 - 1e-12) : -1.0;
  }
  a.k = ctx->prob.max_neighbors;
  a.min_neighbors = ctx->prob.min_neighbors;
  a.use_ball = !(ctx->prob.ball_radius != ctx->prob.ball_radius);
  a.radius = ctx->prob.ball_radius;
  a.flags = ctx->prob.flags;
  a.first = first;
  a.count = count;
  a.nn = d_nn;
  a.nbr = d_nbr;
  a.out = ctx->out;
  for (int p = 0; p < a.out.n; ++p) {
    a.out.mean[p] += out_off;
    a.out.var[p] += out_off;
  }
  const bool cols = ctx->cols.active;
  GskColArgs ca{};
  if (cols) {
    ca.z = ctx->cols.z;
    ca.ncols = ctx->cols.m;
    ca.perm = ctx->cols.perm;
    ca.mean = ctx->cols.mean + out_off * ctx->cols.m;
    ca.w = ctx->cols.w ? ctx->cols.w + out_off * a.k : nullptr;
    ca.lag = ctx->cols.lag ? ctx->cols.lag + out_off * ctx->es.nterms : nullptr;
  }
  // Which kernel: k <= 20 with Simple / Ordinary Kriging → the small kernel (4 lanes per target, everything static);
  // 20 < k <= 64 with at most 6 drift terms → the block-pool kernels (local_solve_wpt.cuh: two targets per warp up to
  // k = 32, one warp per target above); everything else (Universal Kriging with k <= 20, more than 6 drift terms,
  // 64 < k <= 96) → the column-packed kernel in the smallest configuration that holds k + extra rows.
  // gsk_krige_columns runs every k on the column-packed kernel: only it carries the columns epilogue.
  // extra rows: b, z, then the c drift rows
  const int e = 2 + ctx->es.nterms;
  auto rows = [&](int W) { return (a.k + W - 1) / W * W + (e + W - 1) / W * W; };
  cudaError_t err;
  static const bool no_small = GSK_DEV_ENV("GSK_NO_SMALL_KERNEL") != nullptr;  // development switch
  static const int wpt2_min_k = GSK_DEV_ENV("GSK_WPT2_MIN_K") ? atoi(GSK_DEV_ENV("GSK_WPT2_MIN_K")) : 21;  // development switch
  if (cols) {
    if (rows(4) <= 12) err = gsk_local_launch_A(a, e, st, &ca);
    else if (rows(4) <= 24) err = gsk_local_launch_B(a, e, st, &ca);
    else if (rows(8) <= 40) err = gsk_local_launch_C(a, e, st, &ca);
    else if (rows(8) <= 72) err = gsk_local_launch_D(a, e, st, &ca);
    else if (rows(8) <= 112) err = gsk_local_launch_E(a, e, st, &ca);
    else {
      ctx->err = "max_neighbors too large for the local kernels";
      return GSK_ERR_UNSUPPORTED;
    }
  } else if (!no_small && a.k <= gsk_local::SK_KMAX && (ctx->es.kind == GSK_EST_SIMPLE || ctx->es.nterms == 1))
    err = gsk_local_launch_small(a, st);
  else if (a.k > 32 && a.k <= 64 && e <= 8) err = gsk_local_launch_wpt(a, e, st);          // block-pool kernel, one warp per target (C5)
  else if (a.k >= wpt2_min_k && a.k <= 32 && e <= 8) err = gsk_local_launch_wpt2(a, e, st);  // … two targets per warp (C3)
  else if (rows(4) <= 12) err = gsk_local_launch_A(a, e, st);
  else if (rows(4) <= 24) err = gsk_local_launch_B(a, e, st);
  else if (rows(8) <= 40) err = gsk_local_launch_C(a, e, st);
  else if (rows(8) <= 72) err = gsk_local_launch_D(a, e, st);
  else if (rows(8) <= 112) err = gsk_local_launch_E(a, e, st);
  else {
    ctx->err = "max_neighbors too large for the local kernels";
    return GSK_ERR_UNSUPPORTED;
  }
  if (err == cudaErrorInvalidConfiguration) {
    (void)cudaGetLastError();
    ctx->err = "this combination of max_neighbors, drift terms and n_support needs more shared memory per CTA than sm_100 "
               "offers (227 KB): reduce n_support below 64, max_neighbors below 89 or the Universal Kriging degree";
    return GSK_ERR_UNSUPPORTED;
  }
  GSK_CUDA_CHECK(ctx, err);
  if (launches) *launches += 1;
  return GSK_OK;
}
