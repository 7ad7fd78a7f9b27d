// sgs.cu — sequential Gaussian simulation (ref: src/simulation/sgs.jl:56-89 sets the Simple Kriging estimator and the
// Normal(mean, √sill) marginal; src/simulation/seq.jl:102-135 is the loop: for every location of the path, search the
// neighbours among the already simulated locations, fit, draw from the conditional Normal).
//
// What the reference does one location at a time splits into a part that does not depend on the simulated VALUES and a
// part that does:
//   * which locations are the k nearest already-simulated ones of location i, their Simple Kriging weights λ_i and
//     the conditional standard deviation σ_i depend on the geometry, the variogram and the path only. gsk_sgs_plan
//     computes them for ALL locations at once: a rank-masked search (search.cu, RANKED: a record is a candidate only
//     if its rank in the path is lower than the target's; data locations have the lowest rank) and one small SPD
//     solve per location (sgs_weights_kernel, one thread per location).
//   * the values follow the recurrence v_i = μ + Σ_j λ_ij (v_n(i,j) − μ) + σ_i z_i. The neighbour lists make it a DAG
//     over the locations; its levels (level = 1 + the deepest simulated neighbour) are computed once with the plan,
//     and a realisation is evaluated level by level: every location of a level is independent of the others
//     (sgs_level_kernel, one thread per location and realisation; runs of small levels share one launch,
//     sgs_run_kernel). Only when the DAG is nearly a chain (a linear path on a line) the path is walked by one warp
//     per realisation instead (sgs_recurrence_kernel). The results do not depend on the schedule.
// The draws z come from the caller's generator (rand(rng, Normal(μ, σ)) = μ + σ·randn(rng), one per location in path
// order), so the library holds no random state.
#include <math.h>

#include <algorithm>
#include <chrono>
#include <cstring>
#include <vector>

#include "gsk_internal.cuh"

struct SgsPlan {
  long long n = 0, m = 0;  // locations, of which m are simulated (rank >= 0)
  int k = 0, dim = 0;
  double mean = 0.0, sd_marginal = 1.0;
  int *nn = nullptr;      // n: neighbours of location i (0: draw from the marginal)
  int *nbr = nullptr;     // n × k location indices
  double *lam = nullptr;  // n × k Simple Kriging weights
  double *sig = nullptr;  // n conditional standard deviations
  int *order = nullptr;   // m: location visited at path position p
  int *isdata = nullptr;  // n: 1 where the value is given
  double *vals = nullptr, *z = nullptr, *out = nullptr;  // sample buffers (grown on demand)
  size_t cap_real = 0;
  // level schedule (depth == 0: not used, the path is walked by sgs_recurrence_kernel)
  int depth = 0;
  int *lv_start = nullptr;  // depth + 1: positions of level l are [lv_start[l], lv_start[l + 1])
  int *lv_loc = nullptr;    // m: location at position pos (positions are sorted by level)
  int *lv_nn = nullptr;     // m
  int *lv_nbr = nullptr;    // k × m, neighbour j of position pos at [j · m + pos]
  double *lv_lam = nullptr; // k × m
  double *lv_sig = nullptr; // m
  struct Seg { int l0, l1, wide; };  // launch schedule: one wide level, or a run [l0, l1) of small levels
  std::vector<Seg> segs;
  std::vector<int> h_lv_start;
};

namespace {

__global__ void sgs_trank_kernel(const int *__restrict__ perm, const int *__restrict__ rankp1, long long n,
                                 int *__restrict__ trank) {
  long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n) trank[s] = rankp1[perm[s]];
}

// One thread per location (bin-sorted order s, results stored at the location's own index). The k×k covariance
// matrix of the neighbours is held as a packed lower triangle in `work` with element-major layout
// work[e · stride + thread] (shared memory: stride = blockDim.x, bank-conflict free; global scratch for large k).
__global__ void sgs_weights_kernel(GskTargets tg, GskVario vg, const double4 *__restrict__ rec, const int *__restrict__ perm,
                                   const int *__restrict__ nn_s, const int *__restrict__ nbr_s, long long n, int k,
                                   int min_neighbors, double sd_marginal, double *__restrict__ gwork, int *__restrict__ nn_out,
                                   int *__restrict__ nbr_out, double *__restrict__ lam_out, double *__restrict__ sig_out) {
  extern __shared__ double swork[];
  double *work;
  long long stride;
  if (gwork) {
    stride = (long long)gridDim.x * blockDim.x;
    work = gwork + ((long long)blockIdx.x * blockDim.x + threadIdx.x);
  } else {
    stride = blockDim.x;
    work = swork + threadIdx.x;
  }
  const int ntri = k * (k + 1) / 2;
  double *A = work;                      // packed lower triangle, row i starts at i(i+1)/2
  double *b = work + (size_t)ntri * stride;  // right-hand side, then the weights
#define AT(i, j) A[(size_t)((i) * ((i) + 1) / 2 + (j)) * stride]
#define BV(i) b[(size_t)(i) * stride]
  for (long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (long long)gridDim.x * blockDim.x) {
    const long long o = perm[s];
    int nn = nn_s[s];
    const int *nb = nbr_s + s * k;
    double sig = sd_marginal;
    bool ok = nn >= min_neighbors && nn >= 1;
    if (ok) {
      double tc[3] = {tg.pts[0][s], tg.dim > 1 ? tg.pts[1][s] : 0.0, tg.dim > 2 ? tg.pts[2][s] : 0.0};
      // covariances among the neighbours and to the location (point support: the domain's centroids, seq.jl:91)
      for (int i = 0; i < nn; ++i) {
        const double4 ri = rec[nb[i]];
        const double ci[3] = {ri.x, ri.y, ri.z};
        for (int j = 0; j < i; ++j) AT(i, j) = gsk_cov_rt(vg, gsk_dist2_exact(tg.dim, ci, rec[nb[j]]));
        AT(i, i) = vg.sill;
        BV(i) = gsk_cov_rt(vg, gsk_dist2_exact(tg.dim, tc, ri));
      }
      // Cholesky (status(fitted) is the success of this factorisation, seq.jl:123)
      for (int j = 0; j < nn && ok; ++j) {
        double d = AT(j, j);
        for (int p = 0; p < j; ++p) { const double l = AT(j, p); d = fma(-l, l, d); }
        if (!(d > 0.0)) { ok = false; break; }
        const double ld = sqrt(d), inv = 1.0 / ld;
        AT(j, j) = ld;
        for (int i = j + 1; i < nn; ++i) {
          double v = AT(i, j);
          for (int p = 0; p < j; ++p) v = fma(-AT(i, p), AT(j, p), v);
          AT(i, j) = v * inv;
        }
      }
    }
    if (ok) {
      // σ² = sill − bᵀC⁻¹b = sill − ‖L⁻¹b‖² ; λ = L⁻ᵀ L⁻¹ b
      double q = 0.0;
      for (int i = 0; i < nn; ++i) {
        double v = BV(i);
        for (int p = 0; p < i; ++p) v = fma(-AT(i, p), BV(p), v);
        v /= AT(i, i);
        BV(i) = v;
        q = fma(v, v, q);
      }
      for (int i = nn - 1; i >= 0; --i) {
        double v = BV(i);
        for (int p = i + 1; p < nn; ++p) v = fma(-AT(p, i), BV(p), v);
        BV(i) = v / AT(i, i);
      }
      double s2 = vg.sill - q;
      s2 = (s2 > 0.0) ? s2 : 0.0;  // predictvar clamps at zero
      sig = sqrt(s2);
      for (int i = 0; i < k; ++i) {
        nbr_out[o * k + i] = (i < nn) ? nb[i] : -1;
        lam_out[o * k + i] = (i < nn) ? BV(i) : 0.0;
      }
    } else {
      nn = 0;  // fewer than min_neighbors, or the factorisation failed: the marginal (seq.jl:108-110,126-128)
      for (int i = 0; i < k; ++i) { nbr_out[o * k + i] = -1; lam_out[o * k + i] = 0.0; }
    }
    nn_out[o] = nn;
    sig_out[o] = sig;
  }
#undef AT
#undef BV
}

__global__ void sgs_init_kernel(const double *__restrict__ vals, const int *__restrict__ isdata, long long n, int nreal,
                                double *__restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * nreal) return;
  const long long loc = i % n;
  out[i] = isdata[loc] ? (vals ? vals[loc] : 0.0) : nan("");
}

// One warp per realisation walks the path. The neighbour lists, weights, σ and the draw of position p + 1 are loaded
// while position p is reduced (they do not depend on simulated values); the only dependent chain per location is
// {load the k neighbour values from L2, 5 shuffles, store}. Values are read and written past L1 (ld.cg / st.cg): a
// location simulated a few iterations ago by lane 0 must be seen by the other lanes.
__global__ void __launch_bounds__(32) sgs_recurrence_kernel(const int *__restrict__ order, long long m, long long n, int k,
                                                            const int *__restrict__ nnv, const int *__restrict__ nbr,
                                                            const double *__restrict__ lam, const double *__restrict__ sig,
                                                            const double *__restrict__ z, double mean, double *__restrict__ out) {
  const int lane = threadIdx.x;
  const long long r = blockIdx.x;
  const double *zr = z + r * n;
  double *vr = out + r * n;
  struct Slot { int loc, nn, i0, i1; double l0, l1, sg, zz; };
  auto fetch = [&](long long p, Slot &s) {
    s.loc = -1; s.nn = 0; s.i0 = s.i1 = -1; s.l0 = s.l1 = 0.0; s.sg = 0.0; s.zz = 0.0;
    if (p >= m) return;
    const int loc = order[p];
    s.loc = loc;
    s.nn = nnv[loc];
    const long long base = (long long)loc * k;
    if (lane < s.nn) { s.i0 = nbr[base + lane]; s.l0 = lam[base + lane]; }
    if (lane + 32 < s.nn) { s.i1 = nbr[base + lane + 32]; s.l1 = lam[base + lane + 32]; }
    s.sg = sig[loc];
    s.zz = zr[loc];
  };
  Slot cur, nxt;
  fetch(0, cur);
  for (long long p = 0; p < m; ++p) {
    fetch(p + 1, nxt);
    double acc = 0.0;
    if (cur.i0 >= 0) acc = cur.l0 * (__ldcg(vr + cur.i0) - mean);
    if (cur.i1 >= 0) acc = fma(cur.l1, __ldcg(vr + cur.i1) - mean, acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) __stcg(vr + cur.loc, (mean + acc) + cur.sg * cur.zz);
    __syncwarp();
    cur = nxt;
  }
}

// plan arrays re-ordered by level position, neighbour-major (coalesced for one thread per position)
__global__ void sgs_to_levels_kernel(const int *__restrict__ lv_loc, long long m, int k, const int *__restrict__ nn,
                                     const int *__restrict__ nbr, const double *__restrict__ lam, const double *__restrict__ sig,
                                     int *__restrict__ lv_nn, int *__restrict__ lv_nbr, double *__restrict__ lv_lam,
                                     double *__restrict__ lv_sig) {
  long long pos = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= m) return;
  const long long loc = lv_loc[pos];
  lv_nn[pos] = nn[loc];
  lv_sig[pos] = sig[loc];
  for (int j = 0; j < k; ++j) {
    lv_nbr[(long long)j * m + pos] = nbr[loc * k + j];
    lv_lam[(long long)j * m + pos] = lam[loc * k + j];
  }
}

template <bool SAME_SM>
__device__ __forceinline__ void sgs_eval_position(long long pos, long long m, long long n, const int *__restrict__ lv_loc,
                                                  const int *__restrict__ lv_nn, const int *__restrict__ lv_nbr,
                                                  const double *__restrict__ lv_lam, const double *__restrict__ lv_sig,
                                                  const double *__restrict__ zr, double mean, double *vr) {
  const int nn = lv_nn[pos];
  double acc = 0.0;
  // eight neighbours at a time: their indices and weights first, then the eight values (independent loads in flight
  // together — inside a run of levels the latency of this chain is the cost of a level), then the sum in list order
  for (int j0 = 0; j0 < nn; j0 += 8) {
    int idx[8];
    double lm[8], v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const bool in = j0 + u < nn;
      idx[u] = in ? lv_nbr[(long long)(j0 + u) * m + pos] : -1;
      lm[u] = in ? lv_lam[(long long)(j0 + u) * m + pos] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      // inside a run of levels the value may have been written by another thread of this CTA a moment ago: read past L1
      v[u] = (idx[u] >= 0) ? (SAME_SM ? __ldcg(vr + idx[u]) : vr[idx[u]]) : mean;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) acc = fma(lm[u], v[u] - mean, acc);
  }
  const int loc = lv_loc[pos];
  const double x = (mean + acc) + lv_sig[pos] * zr[loc];
  if (SAME_SM) __stcg(vr + loc, x); else vr[loc] = x;
}

// one level: thread per (position, realisation)
__global__ void sgs_level_kernel(int pos0, int cnt, long long m, long long n, const int *__restrict__ lv_loc,
                                 const int *__restrict__ lv_nn, const int *__restrict__ lv_nbr, const double *__restrict__ lv_lam,
                                 const double *__restrict__ lv_sig, const double *__restrict__ z, double mean,
                                 double *out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= cnt) return;
  const long long r = blockIdx.y;
  sgs_eval_position<false>(pos0 + t, m, n, lv_loc, lv_nn, lv_nbr, lv_lam, lv_sig, z + r * n, mean, out + r * n);
}

// a run of consecutive small levels: one CTA per realisation, a CTA-wide barrier between levels
__global__ void sgs_run_kernel(int l0, int l1, const int *__restrict__ lv_start, long long m, long long n,
                               const int *__restrict__ lv_loc, const int *__restrict__ lv_nn, const int *__restrict__ lv_nbr,
                               const double *__restrict__ lv_lam, const double *__restrict__ lv_sig, const double *__restrict__ z,
                               double mean, double *out) {
  const long long r = blockIdx.x;
  const double *zr = z + r * n;
  double *vr = out + r * n;
  int a = lv_start[l0];
  for (int l = l0; l < l1; ++l) {
    const int b = lv_start[l + 1];
    for (int pos = a + threadIdx.x; pos < b; pos += blockDim.x)
      sgs_eval_position<true>(pos, m, n, lv_loc, lv_nn, lv_nbr, lv_lam, lv_sig, zr, mean, vr);
    __syncthreads();
    a = b;
  }
}

}  // namespace

void gsk_sgs_free(gsk_ctx *ctx) {
  SgsPlan *s = ctx->sgs;
  if (!s) return;
  cudaFree(s->nn); cudaFree(s->nbr); cudaFree(s->lam); cudaFree(s->sig); cudaFree(s->order); cudaFree(s->isdata);
  cudaFree(s->vals); cudaFree(s->z); cudaFree(s->out);
  cudaFree(s->lv_start); cudaFree(s->lv_loc); cudaFree(s->lv_nn); cudaFree(s->lv_nbr); cudaFree(s->lv_lam); cudaFree(s->lv_sig);
  delete s;
  ctx->sgs = nullptr;
}

int gsk_sgs_plan_impl(gsk_ctx *ctx, int dim, long long n, const double *const *coords, const long long *rank,
                      const GskVario &vg, double mean, int min_neighbors, int k, double ball_radius) {
  cudaStream_t st = ctx->stream;
  using clk = std::chrono::steady_clock;
  auto ms_since = [](clk::time_point t) { return std::chrono::duration<double, std::milli>(clk::now() - t).count(); };
  const clk::time_point t_begin = clk::now();
  // ---- the path: order[p] = location of rank p; ranks must be a permutation of 0..m−1 over the locations without data
  long long m = 0;
  for (long long i = 0; i < n; ++i) if (rank[i] >= 0) ++m;
  if (m == 0) { ctx->err = "gsk_sgs_plan: every location holds data, nothing to simulate"; return GSK_ERR_INVALID; }
  std::vector<int> order((size_t)m, -1), rankp1((size_t)n), isdata((size_t)n);
  for (long long i = 0; i < n; ++i) {
    const long long r = rank[i];
    if (r >= m || (r >= 0 && order[(size_t)r] != -1)) {
      ctx->err = "gsk_sgs_plan: rank must be -1 (data) or a permutation of 0..m-1 over the other locations";
      return GSK_ERR_INVALID;
    }
    if (r >= 0) order[(size_t)r] = (int)i;
    rankp1[(size_t)i] = (r >= 0) ? (int)r + 1 : 0;
    isdata[(size_t)i] = r < 0;
  }
  // ---- bins over all locations; the record's w carries (rank + 1) << 32 | index ----
  {
    std::vector<double> hv((size_t)n);
    for (long long i = 0; i < n; ++i) {
      const long long bits = (long long)rankp1[(size_t)i] << 32;
      memcpy(&hv[(size_t)i], &bits, sizeof(double));
    }
    int rc = gsk_build_bins(ctx, coords[0], dim > 1 ? coords[1] : nullptr, dim > 2 ? coords[2] : nullptr, hv.data(), n, dim,
                            k, true);
    if (rc != GSK_OK) return rc;
  }
  // ---- the locations as explicit targets ----
  GskTargets &tg = ctx->tg;
  memset(&tg, 0, sizeof(tg));
  tg.is_grid = 0;
  tg.dim = dim;
  tg.npts = n;
  int rc;
  {
    double *hp = nullptr;
    if ((rc = gsk_host_stage(ctx, sizeof(double) * (size_t)n * 3, (void **)&hp)) != GSK_OK) return rc;
    for (int d = 0; d < dim; ++d) {
      if ((rc = gsk_buf(ctx, (GskBufId)(BUF_PTS0 + d), sizeof(double) * (size_t)n, (void **)&ctx->d_pts[d])) != GSK_OK) return rc;
      memcpy(hp + (size_t)d * n, coords[d], sizeof(double) * (size_t)n);
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->d_pts[d], hp + (size_t)d * n, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
      tg.pts[d] = ctx->d_pts[d];
    }
  }
  ctx->prob = gsk_problem{};
  ctx->prob.dim = dim;
  ctx->prob.n_samples = n;
  ctx->prob.max_neighbors = k;
  ctx->prob.min_neighbors = min_neighbors;
  ctx->prob.ball_radius = ball_radius;
  ctx->vg = vg;

  SgsPlan *s = new SgsPlan();
  ctx->sgs = s;
  s->n = n; s->m = m; s->k = k; s->dim = dim; s->mean = mean; s->sd_marginal = sqrt(vg.sill);
  GSK_CUDA_CHECK(ctx, cudaMalloc(&s->nn, sizeof(int) * (size_t)n));
  GSK_CUDA_CHECK(ctx, cudaMalloc(&s->nbr, sizeof(int) * (size_t)n * k));
  GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lam, sizeof(double) * (size_t)n * k));
  GSK_CUDA_CHECK(ctx, cudaMalloc(&s->sig, sizeof(double) * (size_t)n));
  GSK_CUDA_CHECK(ctx, cudaMalloc(&s->order, sizeof(int) * (size_t)m));
  GSK_CUDA_CHECK(ctx, cudaMalloc(&s->isdata, sizeof(int) * (size_t)n));
  int *d_rankp1 = nullptr, *d_trank = nullptr;
  if ((rc = gsk_buf(ctx, BUF_PT_MEAN, sizeof(int) * (size_t)n, (void **)&d_rankp1)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_VAR, sizeof(int) * (size_t)n, (void **)&d_trank)) != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(s->order, order.data(), sizeof(int) * (size_t)m, cudaMemcpyHostToDevice, st));
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(s->isdata, isdata.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(d_rankp1, rankp1.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));

  ctx->timing = gsk_timing{};
  ctx->timing_pending = false;
  ctx->timing.ms_plan = ms_since(t_begin);  // path checks, bins, uploads
  // ---- bin-sort the locations, search with the rank mask, solve ----
  clk::time_point t_phase = clk::now();
  int *perm = nullptr, *nn_s = nullptr, *nbr_s = nullptr;
  double *sx = nullptr, *sy = nullptr, *sz = nullptr;
  if ((rc = gsk_points_sort(ctx, 0, n, &perm, &sx, &sy, &sz)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_NN, sizeof(int) * (size_t)n, (void **)&nn_s)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_NBR, sizeof(int) * (size_t)n * k, (void **)&nbr_s)) != GSK_OK) return rc;
  const unsigned g = (unsigned)((n + 255) / 256);
  sgs_trank_kernel<<<g, 256, 0, st>>>(perm, d_rankp1, n, d_trank);
  GskTargets tgs = tg;
  tgs.pts[0] = sx; tgs.pts[1] = sy; tgs.pts[2] = sz;
  const GskTargets tg_saved = ctx->tg;
  ctx->tg = tgs;
  int launches = 0;
  rc = gsk_launch_search(ctx, st, 0, n, k, nn_s, nbr_s, &launches, d_trank);
  ctx->tg = tg_saved;
  if (rc != GSK_OK) return rc;
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  ctx->timing.ms_search = ms_since(t_phase);
  t_phase = clk::now();

  const size_t per_thread = sizeof(double) * (size_t)(k * (k + 1) / 2 + k);
  int tpb = 128;
  while (tpb > 32 && per_thread * tpb > (size_t)96 * 1024) tpb >>= 1;
  double *gwork = nullptr;
  size_t smem = per_thread * tpb;
  unsigned grid = (unsigned)((n + tpb - 1) / tpb);
  if (smem > (size_t)200 * 1024) {  // large k: the triangles live in global scratch (L2-resident, coalesced by thread)
    tpb = 128;
    grid = (unsigned)std::min<long long>((n + tpb - 1) / tpb, (long long)ctx->sm_count * 8);
    if ((rc = gsk_buf(ctx, BUF_G_TMP, per_thread * (size_t)grid * tpb, (void **)&gwork)) != GSK_OK) return rc;
    smem = 0;
  } else {
    GSK_CUDA_CHECK(ctx, cudaFuncSetAttribute(sgs_weights_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  sgs_weights_kernel<<<grid, tpb, smem, st>>>(tgs, vg, ctx->d_rec_orig, perm, nn_s, nbr_s, n, k, min_neighbors,
                                             s->sd_marginal, gwork, s->nn, s->nbr, s->lam, s->sig);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  ctx->timing.ms_solve = ms_since(t_phase);
  ctx->timing.launches = launches + 6 + 4 + 2;
  ctx->timing.targets = m;

  // ---- level schedule of the recurrence: level(i) = 1 + max level of i's simulated neighbours (data: level 0) ----
  {
    std::vector<int> h_nn((size_t)n), h_nbr((size_t)n * k), level((size_t)n, 0);
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(h_nn.data(), s->nn, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(h_nbr.data(), s->nbr, sizeof(int) * (size_t)n * k, cudaMemcpyDeviceToHost, st));
    GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
    int depth = 0;
    for (long long p = 0; p < m; ++p) {
      const size_t i = (size_t)order[(size_t)p];
      int lv = 0;
      const int *nb = &h_nbr[i * k];
      for (int j = 0; j < h_nn[i]; ++j) lv = std::max(lv, level[(size_t)nb[j]]);
      level[i] = lv + 1;
      depth = std::max(depth, lv + 1);
    }
    // a nearly sequential DAG gains nothing from levels: one warp per realisation walks the path instead
    if ((long long)depth * 8 <= m || m < 4096) {
      std::vector<int> start((size_t)depth + 1, 0), lv_loc((size_t)m);
      for (long long p = 0; p < m; ++p) ++start[(size_t)level[(size_t)order[(size_t)p]]];  // start[l] = size of level l (1-based)
      int run = 0;
      for (int l = 1; l <= depth; ++l) { const int c = start[(size_t)l]; start[(size_t)l - 1] = run; run += c; }
      start[(size_t)depth] = run;  // start[l-1] = first position of level l  → 0-based levels from here on
      {
        std::vector<int> cursor(start.begin(), start.end() - 1);
        for (long long p = 0; p < m; ++p) {  // path order inside a level
          const int i = order[(size_t)p];
          lv_loc[(size_t)cursor[(size_t)level[(size_t)i] - 1]++] = i;
        }
      }
      s->depth = depth;
      s->h_lv_start = start;
      GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lv_start, sizeof(int) * ((size_t)depth + 1)));
      GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lv_loc, sizeof(int) * (size_t)m));
      GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lv_nn, sizeof(int) * (size_t)m));
      GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lv_nbr, sizeof(int) * (size_t)m * k));
      GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lv_lam, sizeof(double) * (size_t)m * k));
      GSK_CUDA_CHECK(ctx, cudaMalloc(&s->lv_sig, sizeof(double) * (size_t)m));
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(s->lv_start, start.data(), sizeof(int) * ((size_t)depth + 1), cudaMemcpyHostToDevice, st));
      GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(s->lv_loc, lv_loc.data(), sizeof(int) * (size_t)m, cudaMemcpyHostToDevice, st));
      sgs_to_levels_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(s->lv_loc, m, k, s->nn, s->nbr, s->lam, s->sig, s->lv_nn,
                                                                      s->lv_nbr, s->lv_lam, s->lv_sig);
      GSK_CUDA_CHECK(ctx, cudaGetLastError());
      // launch schedule: consecutive levels of at most SGS_SMALL positions share one launch
      const int SGS_SMALL = 1024;
      for (int l = 0; l < depth;) {
        if (start[(size_t)l + 1] - start[(size_t)l] > SGS_SMALL) { s->segs.push_back({l, l + 1, 1}); ++l; continue; }
        int e = l;
        while (e < depth && start[(size_t)e + 1] - start[(size_t)e] <= SGS_SMALL) ++e;
        s->segs.push_back({l, e, 0});
        l = e;
      }
      GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
      ctx->timing.launches += 1;
    }
  }
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));  // host vectors above go out of scope
  ctx->timing.ms_total = ms_since(t_begin);          // the rest: level schedule (host) and its upload
  return GSK_OK;
}

// the kernels of one gsk_sgs_sample call on device buffers (vals may be nullptr when the plan has no data locations)
static int sgs_launch(gsk_ctx *ctx, int nreal, const double *d_vals, const double *d_z, double *d_out, int *launches_out) {
  SgsPlan *s = ctx->sgs;
  cudaStream_t st = ctx->stream;
  const size_t n = (size_t)s->n;
  const long long tot = (long long)n * nreal;
  sgs_init_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d_vals, s->isdata, s->n, nreal, d_out);
  int launches = 1;
  if (s->depth > 0) {
    for (const SgsPlan::Seg &g : s->segs) {
      if (g.wide) {
        const int pos0 = s->h_lv_start[(size_t)g.l0], cnt = s->h_lv_start[(size_t)g.l1] - pos0;
        // realisations in chunks of 65535 (gridDim.y)
        for (int r0 = 0; r0 < nreal; r0 += 65535) {
          const dim3 grid((unsigned)((cnt + 127) / 128), (unsigned)std::min(nreal - r0, 65535));
          sgs_level_kernel<<<grid, 128, 0, st>>>(pos0, cnt, s->m, s->n, s->lv_loc, s->lv_nn, s->lv_nbr, s->lv_lam, s->lv_sig,
                                                 d_z + (size_t)r0 * n, s->mean, d_out + (size_t)r0 * n);
          ++launches;
        }
      } else {
        sgs_run_kernel<<<(unsigned)nreal, 256, 0, st>>>(g.l0, g.l1, s->lv_start, s->m, s->n, s->lv_loc, s->lv_nn, s->lv_nbr,
                                                        s->lv_lam, s->lv_sig, d_z, s->mean, d_out);
        ++launches;
      }
    }
  } else {
    sgs_recurrence_kernel<<<(unsigned)nreal, 32, 0, st>>>(s->order, s->m, s->n, s->k, s->nn, s->nbr, s->lam, s->sig, d_z,
                                                          s->mean, d_out);
    ++launches;
  }
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  *launches_out = launches;
  return GSK_OK;
}

int gsk_sgs_sample_impl(gsk_ctx *ctx, int nreal, const double *values, const double *z, double *out, bool on_device) {
  SgsPlan *s = ctx->sgs;
  cudaStream_t st = ctx->stream;
  const std::chrono::steady_clock::time_point t_begin = std::chrono::steady_clock::now();
  const size_t n = (size_t)s->n;
  int launches = 0, rc;
  if (on_device) {  // the caller's device buffers, asynchronous on the context stream (as gsk_execute)
    if (!values && s->m < s->n) { ctx->err = "gsk_sgs_sample_device: the plan has data locations, d_values is required"; return GSK_ERR_INVALID; }
    if ((rc = sgs_launch(ctx, nreal, values, z, out, &launches)) != GSK_OK) return rc;
    ctx->timing = gsk_timing{};
    ctx->timing_pending = false;
    ctx->timing.targets = (long long)s->m * nreal;
    ctx->timing.launches = launches;
    return GSK_OK;
  }
  if (s->cap_real < (size_t)nreal) {
    cudaFree(s->z); cudaFree(s->out); cudaFree(s->vals);
    s->z = s->out = s->vals = nullptr;
    s->cap_real = 0;
    GSK_CUDA_CHECK(ctx, cudaMalloc(&s->vals, sizeof(double) * n));
    GSK_CUDA_CHECK(ctx, cudaMalloc(&s->z, sizeof(double) * n * nreal));
    GSK_CUDA_CHECK(ctx, cudaMalloc(&s->out, sizeof(double) * n * nreal));
    s->cap_real = (size_t)nreal;
  }
  if (values) GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(s->vals, values, sizeof(double) * n, cudaMemcpyHostToDevice, st));
  else GSK_CUDA_CHECK(ctx, cudaMemsetAsync(s->vals, 0, sizeof(double) * n, st));
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(s->z, z, sizeof(double) * n * nreal, cudaMemcpyHostToDevice, st));
  cudaEventRecord(ctx->ev[3], st);
  if ((rc = sgs_launch(ctx, nreal, s->vals, s->z, s->out, &launches)) != GSK_OK) return rc;
  cudaEventRecord(ctx->ev[4], st);
  GSK_CUDA_CHECK(ctx, cudaMemcpyAsync(out, s->out, sizeof(double) * n * nreal, cudaMemcpyDeviceToHost, st));
  GSK_CUDA_CHECK(ctx, cudaStreamSynchronize(st));
  ctx->timing = gsk_timing{};
  ctx->timing_pending = false;
  float ms_k = 0.f;
  if (cudaEventElapsedTime(&ms_k, ctx->ev[3], ctx->ev[4]) == cudaSuccess) ctx->timing.ms_solve = ms_k;  // the kernels alone
  ctx->timing.ms_total = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
  ctx->timing.targets = (long long)s->m * nreal;
  ctx->timing.launches = launches;
  return GSK_OK;
}

int gsk_sgs_weights_impl(gsk_ctx *ctx, int *nn_out, int *nbr_out, double *lam_out, double *sig_out) {
  SgsPlan *s = ctx->sgs;
  const size_t n = (size_t)s->n, k = (size_t)s->k;
  if (nn_out) GSK_CUDA_CHECK(ctx, cudaMemcpy(nn_out, s->nn, sizeof(int) * n, cudaMemcpyDeviceToHost));
  if (nbr_out) GSK_CUDA_CHECK(ctx, cudaMemcpy(nbr_out, s->nbr, sizeof(int) * n * k, cudaMemcpyDeviceToHost));
  if (lam_out) GSK_CUDA_CHECK(ctx, cudaMemcpy(lam_out, s->lam, sizeof(double) * n * k, cudaMemcpyDeviceToHost));
  if (sig_out) GSK_CUDA_CHECK(ctx, cudaMemcpy(sig_out, s->sig, sizeof(double) * n, cudaMemcpyDeviceToHost));
  return GSK_OK;
}
