/*
 * gskrige.h — C ABI of libgskrige.so: B200-native Kriging estimation.
 *
 * This is the drop-in boundary for ONE hot path of juliohm/GeoStatsSolvers.jl:
 * the two internal functions
 *
 *     exactsolve(problem, var, preproc)   -> (varμ, varσ)   ref: src/estimation/krig.jl:166-186
 *     approxsolve(problem, var, preproc)  -> (varμ, varσ)   ref: src/estimation/krig.jl:188-234
 *
 * called from solve(problem, ::KrigingSolver) at ref: src/estimation/krig.jl:151-157.
 * Everything above these two calls (problem construction, units, missing-value
 * filtering, per-variable loop, georef of the result) stays host code (Julia shim in
 * julia/GSKrige.jl, Python mirror in geostatssolvers.jl_b200/). Everything below —
 * neighbour search, variogram evaluation, kriging-system assembly, factorisation,
 * weight solve, mean/variance — runs in hand-written sm_100a CUDA kernels.
 *
 * The reference has no FFI of its own; the entry points below are what a `ccall`
 * from the Julia shim binds (see INTEGRATION.md). Plain pointers and sizes only,
 * no C++/torch types. All arrays are caller-owned; the library never keeps a host
 * pointer after a call returns. There is NO CPU fallback: every compute entry point
 * fails with GSK_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef GSKRIGE_H
#define GSKRIGE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSK_ABI_VERSION 2

#if defined(__GNUC__)
#define GSK_API __attribute__((visibility("default")))
#else
#define GSK_API
#endif

/* ---- enumerations (values are ABI) ------------------------------------------------ */

/* variogram family — ref call site: test/estimation/krig.jl:10 (GaussianVariogram(range=35.0, nugget=0.0));
 * formulas are Variography 0.22's (ref: Project.toml:42), restated in oracle/gsk_oracle.c */
enum { GSK_VARIO_GAUSSIAN = 0, GSK_VARIO_SPHERICAL = 1, GSK_VARIO_EXPONENTIAL = 2 };

/* estimator — selection precedence is host logic, ref: src/ui.jl:40-50 (kriging_ui) */
enum { GSK_EST_SIMPLE = 0, GSK_EST_ORDINARY = 1, GSK_EST_UNIVERSAL = 2 };

/* estimation solver whose per-location loop runs. All three share searcher_ui (ref: src/ui.jl:11-32), the traversal
 * and the centroid/search step; they differ in what is computed from the neighbours:
 *   KRIGING  ref: src/estimation/krig.jl:166-234   outputs: mean, variance
 *   IDW      ref: src/estimation/idw.jl:112-142    outputs: Σ w z / Σ w with w = 1/d^exponent (a zero distance returns that
 *                                                   sample's value), and the distance to the nearest neighbour (`var_distance`)
 *   LWR      ref: src/estimation/lwr.jl:113-146    outputs: weighted-least-squares plane evaluated at the target and
 *                                                   ‖W X (XᵀWX)⁻¹ x₀‖ (`var_variance`), weights weightfun(d / max d) */
enum { GSK_SOLVER_KRIGING = 0, GSK_SOLVER_IDW = 1, GSK_SOLVER_LWR = 2 };

/* LWR weight functions (lwr.jl:58: the default is h -> exp(-3 h^2); arbitrary Julia closures cannot cross the ABI) */
enum { GSK_LWR_WEIGHT_EXP3H2 = 0 };

/* flags */
enum {
  GSK_FLAG_CLAMP_VARIANCE = 1u << 0, /* σ² = max(0, σ²)  (GeoStatsModels predictvar)            */
  GSK_FLAG_SQRT_ROUNDTRIP = 1u << 1, /* σ² -> (sqrt σ²)²  (Normal(μ,√σ²) then var(), krig.jl:183,231) */
  /* gsk_krige only: when the samples, support and parameters are byte-identical to those of the plan already resident
   * in the context, skip the upload and the bin build / factorisation (the repeated solve(prob, krig) calls of the
   * conditional-simulation callers, ref: src/simulation/fft.jl:112-126,184-188). Off by default: the library then
   * never depends on what an earlier call was given. */
  GSK_FLAG_REUSE_PLAN = 1u << 2,
  GSK_FLAGS_DEFAULT = (1u << 0) | (1u << 1)
};

/* return codes */
enum {
  GSK_OK = 0,
  GSK_ERR_INVALID = -1,     /* bad argument (message says which)                              */
  GSK_ERR_UNSUPPORTED = -2, /* option outside the hot path (drifts, non-Euclidean metric, …)  */
  GSK_ERR_CUDA = -3,        /* CUDA runtime failure / no sm_100 device                        */
  GSK_ERR_NOMEM = -4,       /* host or device allocation failed                               */
  GSK_ERR_STATE = -5        /* call order violation (execute before plan, …)                  */
};

/* limits of the local (maxneighbors) kernels */
#define GSK_MAX_NEIGHBORS 96
#define GSK_MAX_SUPPORT 125 /* block-support points per cell kept in shared memory; larger supports (anisotropic cells,
                              short ranges: up to GSK_MAX_SUPPORT_GLOBAL) are streamed from global memory */
#define GSK_MAX_SUPPORT_GLOBAL 65536
#define GSK_MAX_DRIFT_TERMS 10 /* C(3+2,2): universal kriging up to degree 2 in 3-D */

/* ---- the problem description ------------------------------------------------------ */

typedef struct gsk_problem {
  int32_t abi_version; /* = GSK_ABI_VERSION */
  int32_t dim;         /* 1, 2 or 3 (embeddim of sample and target domains) */

  /* samples: the NON-MISSING subset the host built at krig.jl:97-107, SoA, units stripped
   * (utils.jl:10-15). Neighbour indices reported back refer to this subset (0-based). */
  int64_t n_samples;
  const double *coords[3]; /* each length n_samples; unused dims may be NULL */
  const double *values;    /* length n_samples */

  /* targets: a CartesianGrid (column-major / x-fastest linear index, pinned by
   * ref test/estimation/krig.jl:34-37,69-72) when grid_dims[0] > 0 … */
  int64_t grid_dims[3]; /* unused dims = 1 */
  double grid_origin[3];
  double grid_spacing[3];
  /* … or an explicit point list (PointSet domains, ref: src/simulation/fft.jl:113-114) when grid_dims[0] == 0 */
  int64_t n_points;
  const double *point_coords[3];

  /* slab of the linear target range this call computes (multi-GPU sharding, SURVEY §8e).
   * target_count < 0 means "through the end". Output arrays are slab-local. */
  int64_t target_first;
  int64_t target_count;

  /* block support of a target (Variography's geometry sub-sampling, SURVEY §8a a15):
   * n_support offsets relative to the target centroid; n_support = 1 with a zero offset
   * is point support. */
  int32_t n_support;
  const double *support_offsets[3]; /* each length n_support; unused dims may be NULL */

  /* variogram */
  int32_t vario_kind;
  double vario_range, vario_sill, vario_nugget;
  double gaussian_nugget_eps; /* Variography adds 1e-6 to a Gaussian nugget; 0 switches it off */

  /* estimator */
  int32_t estimator;
  double sk_mean;    /* Simple Kriging mean */
  int32_t uk_degree; /* Universal Kriging polynomial degree (0..2) */

  /* neighbourhood — ref: src/ui.jl:11-32 (searcher_ui), krig.jl:113-117,213 */
  int32_t min_neighbors; /* targets with fewer neighbours -> NaN (the host maps to `missing`) */
  int32_t max_neighbors; /* 0 -> global system (maxneighbors === nothing, krig.jl:151), else the CLAMPED k */
  double ball_radius;    /* NaN -> KNearestSearch; else KBallSearch: kNN then dist <= radius */

  uint32_t flags;

  /* ---- ABI version 2 ---- */
  /* Traversal order (ref: traverse(pdomain, path), krig.jl:179,204; idw.jl:111; lwr.jl:112). NULL = LinearPath.
   * Otherwise target_order[j] (j < gsk_num_targets) is the 0-based linear index of the j-th visited target and the
   * outputs are written in VISITING order, as the reference does (it maps over the path and never permutes back,
   * krig.jl:179-183,204-231): out[j] belongs to target target_order[j]. The slab [target_first, +target_count)
   * then counts positions of the path. */
  const int64_t *target_order;
  int32_t solver;        /* GSK_SOLVER_* (0 = Kriging) */
  double idw_exponent;   /* IDW: `exponent` (> 0; idw.jl:56,96) */
  int32_t lwr_weightfun; /* LWR: GSK_LWR_WEIGHT_* */
} gsk_problem;

typedef struct gsk_ctx gsk_ctx; /* opaque: one CUDA device, its stream, resident buffers */

/* per-phase device times (CUDA events on the context stream) of the last gsk_execute/gsk_krige/gsk_krige_loo/
 * gsk_krige_columns (columns: ms_solve includes the per-column epilogue; leave-one-out: ms_search includes the removal of each row's own index; on the global path ms_solve is the
 * pass over L⁻¹ that yields every row's leave-one-out residual and variance) */
typedef struct gsk_timing {
  double ms_plan;    /* H2D of samples + bin build, or global assembly + factorisation */
  double ms_search;  /* local: neighbour-search kernel(s) */
  double ms_solve;   /* local: assemble+factor+solve kernel; global: RHS + triangular-solve kernels */
  double ms_total;   /* first launch -> last result byte in the device output buffers */
  int64_t launches;  /* kernels launched by the last gsk_execute */
  int64_t targets;   /* targets computed by the last gsk_execute */
} gsk_timing;

/* ---- context ---------------------------------------------------------------------- */
GSK_API int gsk_create(gsk_ctx **out, int device_id);
GSK_API void gsk_destroy(gsk_ctx *ctx);
/* NUL-terminated, owned by ctx (or static when ctx == NULL), valid until the next call on ctx */
GSK_API const char *gsk_last_error(const gsk_ctx *ctx);
/* run all work of this context on the caller's CUDA stream (cudaStream_t passed as void*) */
GSK_API int gsk_set_stream(gsk_ctx *ctx, void *cuda_stream);
GSK_API int gsk_synchronize(gsk_ctx *ctx);

/* ---- one-shot, host buffers: replaces exactsolve / approxsolve (krig.jl:166,188) --- */
GSK_API int gsk_krige(gsk_ctx *ctx, const gsk_problem *prob,
              double *mean_out, double *var_out, /* length = slab target count */
              int32_t *nneigh_out,               /* optional: neighbours used per target (global: n_samples) */
              int32_t *neigh_idx_out);           /* optional: count × max_neighbors, 0-based, sorted by (d², idx), −1 padded */

/* Leave-one-out cross-validation of the Kriging problem's samples: row i is sample i kriged from the other
 * samples at point support (local: its k nearest j != i; global: all j != i). Targets are the samples, so
 * grid_dims[0] = 0, n_points = 0, n_support = 1 (zero offset), target_order = NULL; target_first/target_count
 * select a slab of SAMPLE indices (callers shard with it). solver must be GSK_SOLVER_KRIGING; n_samples >= 2;
 * max_neighbors <= n_samples - 1 (the fold's own clamp); GSK_FLAG_REUSE_PLAN is rejected. nneigh_out /
 * neigh_idx_out (optional, count × max_neighbors, -1 padded, never containing the row's own index) as in
 * gsk_krige. The context holds no plan afterwards. */
GSK_API int gsk_krige_loo(gsk_ctx *ctx, const gsk_problem *prob, double *mean_out, double *var_out,
                          int32_t *nneigh_out, int32_t *neigh_idx_out);

/* Kriging of m value columns over one sample set: the search and the factorisation of every target's system run
 * once and are applied to each column. Everything but the values behaves as in gsk_krige (domain, slab,
 * target_order, support, estimator, neighbourhood, min_neighbors, flags, local/global switch); column j of
 * mean_out is what gsk_krige computes with prob->values = column j, up to rounding (Simple Kriging:
 * μ + Σ λᵢ (z_ij − μ)). Rows below min_neighbors are NaN in every column. prob->values must be NULL, n_cols >= 1,
 * values non-NULL; GSK_FLAG_REUSE_PLAN is rejected, IDW / LWR are GSK_ERR_UNSUPPORTED. The local path solves
 * [C F; Fᵀ 0][λ; ν] = [c; f] for the weights λ and Lagrange multipliers ν (rows below min_neighbors: λ = 0,
 * ν = NaN); the global path applies the dual weights of each column. The context holds no plan afterwards. */
GSK_API int gsk_krige_columns(gsk_ctx *ctx, const gsk_problem *prob,
                              int32_t n_cols, const double *values,  /* n_samples × n_cols, row-major: values[i*n_cols + j] */
                              double *mean_out,                      /* count × n_cols, row-major: mean_out[t*n_cols + j] */
                              double *var_out,                       /* count (the variance does not depend on the values) */
                              int32_t *nneigh_out, int32_t *neigh_idx_out,  /* optional, exactly as gsk_krige */
                              double *weights_out,   /* optional, local path only: count × max_neighbors, 0-padded */
                              double *lagrange_out); /* optional, local path only: count × nterms (OK 1, UK C(d+deg,deg), SK none) */

/* ---- single-process multi-GPU convenience (a Julia host drives all GPUs of a box from one process):
 * the slab [target_first, target_first+target_count) is split into n_devices contiguous pieces, one host
 * thread and one cached context per listed device computes its piece (samples replicated) and copies it
 * straight into the caller's host arrays — no collective is needed when results return to host memory.
 * device_ids may repeat (two pieces on one GPU). Returns the first failing piece's code; its message goes
 * to errbuf (NUL-terminated, may be NULL). */
GSK_API int gsk_krige_multi(const int *device_ids, int n_devices, const gsk_problem *prob, double *mean_out,
                            double *var_out, int32_t *nneigh_out, int32_t *neigh_idx_out, char *errbuf,
                            int errbuf_len);

/* The per-device contexts of gsk_krige_multi (buffers, streams) are cached in the process between calls — one call at a
 * time per process; gsk_krige_multi_release destroys them (call it before unloading the library or to give the memory back). */
GSK_API void gsk_krige_multi_release(void);

/* ---- resident two-step form: replaces preprocess' searcher/estimator construction
 *      (krig.jl:110,117; fit at krig.jl:176) and then the per-target loops ------------- */
/* uploads samples, builds the bin structure (local) or assembles + factorises the
 * global system (max_neighbors == 0); keeps everything resident in HBM */
GSK_API int gsk_plan(gsk_ctx *ctx, const gsk_problem *prob);
/* computes targets [first, first+count) of the planned problem into DEVICE buffers;
 * asynchronous on the context stream */
GSK_API int gsk_execute(gsk_ctx *ctx, int64_t first, int64_t count,
                double *d_mean, double *d_var, int32_t *d_nneigh, int32_t *d_neigh_idx);
/* same, with the result gather fused into the compute kernels: every target's mean/variance is stored
 * into n_peers peer-mapped buffers (NVLink P2P pointers valid in this process, e.g. from CUDA IPC / torch
 * symmetric memory) at index out_offset + (target - first). multicast != 0: n_peers must be 1 and the
 * pointers are NVLS multicast addresses (one multimem.st per value reaches every peer through NVSwitch). */
GSK_API int gsk_execute_peers(gsk_ctx *ctx, int64_t first, int64_t count, int n_peers,
                              double *const *d_mean_peers, double *const *d_var_peers, int64_t out_offset,
                              int multicast, int32_t *d_nneigh, int32_t *d_neigh_idx);
/* Values-only update of the planned problem: same sample coordinates, same parameters, new `values` (length
 * n_samples of the plan). This is what the conditional-simulation callers need between realisations (ref:
 * src/simulation/fft.jl:184-188 solves the same EstimationProblem again with the unconditional realisation's values
 * at the data locations). Bins, the neighbour lists of the last gsk_execute range (local path) and the factor
 * L, L⁻¹ (global path; only Y_E's value column and G_EE are recomputed) stay resident. */
GSK_API int gsk_update_values(gsk_ctx *ctx, const double *values, int64_t n_values);
GSK_API int gsk_get_timing(const gsk_ctx *ctx, gsk_timing *out);
/* when on, gsk_execute brackets every search / solve launch with CUDA events (and synchronises on them)
 * so that gsk_timing.ms_search / ms_solve are filled; off by default (no synchronisation in gsk_execute) */
GSK_API int gsk_set_phase_timing(gsk_ctx *ctx, int on);

/* ---- LU Gaussian simulation: replaces the dense factorisation of preprocess (ref: src/simulation/lu.jl:118-139) and
 *      lusim (lu.jl:198-224) -------------------------------------------------------------------------------------
 * coords[d] hold n_data + n_sim points, the DATA locations first (their values in data_values), then the simulation
 * locations. The joint covariance sill − γ(h) is assembled and factorised on the GPU (blocked FP64 Cholesky, the same
 * kernels as the global Kriging plan) and stays resident. */
GSK_API int gsk_lu_plan(gsk_ctx *ctx, int dim, int64_t n_data, int64_t n_sim, const double *const *coords,
                        const double *data_values, int vario_kind, double vario_range, double vario_sill,
                        double vario_nugget, double gaussian_nugget_eps);
/* one realisation: w = n_sim standard normal draws (the caller's RNG; for two correlated variables the caller passes
 * ρ·w₁ + √(1−ρ²)·w₂, lu.jl:213). y_out (n_data + n_sim): the data values, then d₂ + L₂₂·w (lu.jl:209-219) */
GSK_API int gsk_lu_sample(gsk_ctx *ctx, const double *w, double *y_out);

/* ---- sequential Gaussian simulation: replaces the simulation loop of SeqSim (ref: src/simulation/seq.jl:102-135) with
 *      the Simple Kriging estimator and the Normal(mean, √sill) marginal SGS gives it (ref: src/simulation/sgs.jl:62-84) --
 * coords[d] hold the centroids of the domain's n elements (seq.jl:91). rank[i] = -1: element i holds data (the buffer
 * NearestInit filled, seq.jl:88; its value is passed with every sample call); otherwise rank[i] is the 0-based position
 * of element i in traverse(pdomain, path) among the elements without data (a permutation of 0..m-1).
 * What the loop computes for element i before it draws — the max_neighbors nearest elements among the data and the
 * elements of lower rank (search! with mask = simulated, seq.jl:105; ball_radius NaN: KNearestSearch, else KBallSearch),
 * their Simple Kriging weights and the conditional standard deviation — depends on the geometry and the path only, so
 * the plan computes it for ALL elements in parallel and keeps it resident. max_neighbors <= 64. */
GSK_API int gsk_sgs_plan(gsk_ctx *ctx, int dim, int64_t n, const double *const *coords, const int64_t *rank,
                         int vario_kind, double vario_range, double vario_sill, double vario_nugget,
                         double gaussian_nugget_eps, double mean, int min_neighbors, int max_neighbors,
                         double ball_radius);
/* n_realizations realisations at once (one warp each). values (n, may be NULL when there is no data): read where
 * rank < 0. z (n_realizations × n): the standard normal draw of every element (the caller's RNG; seq.jl:110,130:
 * rand(rng, Normal(μ, σ)) = μ + σ·randn(rng), so the draw made at path position p goes to z[r·n + order[p]]).
 * out (n_realizations × n): the data values, and for the others mean + Σ_j λ_ij (out[n_ij] − mean) + σ_i z_i — or
 * mean + √sill·z_i where fewer than min_neighbors were found or the factorisation failed (seq.jl:108-110,126-128). */
GSK_API int gsk_sgs_sample(gsk_ctx *ctx, int n_realizations, const double *values, const double *z, double *out);
/* the same on DEVICE buffers (d_values may be NULL when no element holds data), asynchronous on the context stream like
 * gsk_execute: for callers that draw on the GPU, nothing crosses PCIe */
GSK_API int gsk_sgs_sample_device(gsk_ctx *ctx, int n_realizations, const double *d_values, const double *d_z,
                                  double *d_out);
/* the plan's per-element neighbour counts (n), neighbour indices (n × k, -1 padded; k = min(max_neighbors, n)),
 * weights (n × k) and conditional standard deviations (n); any pointer may be NULL */
GSK_API int gsk_sgs_weights(gsk_ctx *ctx, int32_t *nneigh_out, int32_t *neigh_idx_out, double *weights_out,
                            double *sigma_out);

/* ---- host helpers shared by every binding ------------------------------------------ */
/* number of targets of the problem's domain (grid product or n_points) */
GSK_API int64_t gsk_num_targets(const gsk_problem *prob);
/* Universal-Kriging monomial exponents in the reference's order (GeoStatsModels UKexps:
 * descending max exponent, stable, constant term last). out: dim × nterms, term-major
 * (out[t*dim + d]); returns nterms or a negative error */
GSK_API int gsk_uk_exponents(int degree, int dim, int32_t *out, int out_capacity_terms);
/* default block support of a grid cell (SURVEY §8a a15, V1): per axis
 * n = ceil(side / (min(range, min side)/3)), offsets (j/(n+1) − 1/2)·side, j = 1..n.
 * Writes x-fastest tensor-product offsets; returns n_support or a negative error. With off_x == NULL nothing is
 * written and the count is returned (size the arrays with it: anisotropic cells or ranges shorter than the cell
 * give more than 27 points; counts above GSK_MAX_SUPPORT_GLOBAL are GSK_ERR_UNSUPPORTED) */
GSK_API int gsk_default_support(int dim, const double *spacing, double vario_range,
                        double *off_x, double *off_y, double *off_z, int capacity);
/* measured FP64 peaks of the context's device (roofline denominators): a dependent-free
 * DFMA loop and an mma.sync m16n8k16 f64 (DMMA) loop, TFLOP/s */
GSK_API int gsk_measure_fp64_peak(gsk_ctx *ctx, double *dfma_tflops, double *dmma_tflops);
GSK_API int gsk_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GSKRIGE_H */
