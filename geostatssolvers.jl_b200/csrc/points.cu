// points.cu — explicit target points (PointSet domains, ref: src/simulation/fft.jl:113-114 calls the Kriging
// solver on a PointSet of centroids). The search kernel wants spatially coherent CTAs, so a slab of points is
// first counting-sorted by the bin of the sample lattice it falls into (count → scan → scatter, as K1 does for
// the samples), processed in that order, and the results are scattered back to the caller's order.
#include "gsk_internal.cuh"

namespace {

__device__ __forceinline__ int pbin(double x, double lo, double inv, int nb) {
  double f = floor((x - lo) * inv);
  return (f < 0.0) ? 0 : ((f >= (double)nb) ? nb - 1 : (int)f);
}

__global__ void pt_count_kernel(GskTargets tg, GskBins bins, long long first, long long count, int *__restrict__ cell_of,
                                int *__restrict__ counts) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  int b[3] = {0, 0, 0};
  for (int d = 0; d < tg.dim; ++d) b[d] = pbin(tg.pts[d][first + i], bins.lo[d], bins.inv[d], bins.nb[d]);
  int c = (b[2] * bins.nb[1] + b[1]) * bins.nb[0] + b[0];
  cell_of[i] = c;
  atomicAdd(&counts[c], 1);
}

__global__ void pt_scan_kernel(const int *__restrict__ counts, long long ncells, int *__restrict__ start) {
  __shared__ int warp_sums[32];
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (long long base = 0; base < ncells; base += blockDim.x) {
    long long i = base + tid;
    int v = (i < ncells) ? counts[i] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int w = (lane < (int)(blockDim.x >> 5)) ? warp_sums[lane] : 0;
      int wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += t;
      }
      warp_sums[lane] = wi - w;
    }
    __syncthreads();
    int excl = carry + warp_sums[wid] + incl - v;
    if (i < ncells) start[i] = excl;
    __syncthreads();
    if (tid == blockDim.x - 1) carry = excl + v;
    __syncthreads();
  }
}

__global__ void pt_scatter_kernel(GskTargets tg, long long first, long long count, const int *__restrict__ cell_of,
                                  const int *__restrict__ start, int *__restrict__ cursor, int *__restrict__ perm,
                                  double *__restrict__ sx, double *__restrict__ sy, double *__restrict__ sz) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  int c = cell_of[i];
  int s = start[c] + atomicAdd(&cursor[c], 1);
  perm[s] = (int)i;
  sx[s] = tg.pts[0][first + i];
  if (tg.dim > 1) sy[s] = tg.pts[1][first + i];
  if (tg.dim > 2) sz[s] = tg.pts[2][first + i];
}

__global__ void pt_unscatter_kernel(const int *__restrict__ perm, long long count, const double *__restrict__ ms,
                                    const double *__restrict__ vs, GskOut out, const int *__restrict__ nn_s,
                                    int *__restrict__ nn_out, const int *__restrict__ nbr_s, int *__restrict__ nbr_out,
                                    int k) {
  long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= count) return;
  const long long o = perm[s];
  gsk_store_result(out, o, ms[s], vs[s]);
  if (nn_out) nn_out[o] = nn_s[s];
  if (nbr_out)
    for (int j = 0; j < k; ++j) nbr_out[o * k + j] = nbr_s[s * k + j];
}

// Leave-one-out: sorted target s is sample first + perm[s]. Its (k+1)-list (exact (d², index) order, −1 padded beyond
// nn1[s]) holds the k nearest samples j != i once i itself is dropped — by index, never by distance: a twin at the same
// location stays — and the rest is cut to k. One thread per target; the k-stride lists feed the ordinary solve kernels.
__global__ void pt_loo_compact_kernel(const int *__restrict__ perm, long long first, long long count, int k,
                                      const int *__restrict__ nn1, const int *__restrict__ nbr1, int *__restrict__ nn_s,
                                      int *__restrict__ nbr_s) {
  const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= count) return;
  const int self = (int)(first + perm[s]);
  const int n1 = nn1[s];
  const int *in = nbr1 + s * (k + 1);
  int *out = nbr_s + s * k;
  int j = 0;
  for (int i = 0; i < n1 && j < k; ++i) {
    const int v = in[i];
    if (v != self) out[j++] = v;
  }
  nn_s[s] = j;
  for (int i = j; i < k; ++i) out[i] = -1;
}

}  // namespace

int gsk_points_loo_compact(gsk_ctx *ctx, const int *perm, long long first, long long count, int k, const int *nn1,
                           const int *nbr1, int *nn_s, int *nbr_s) {
  pt_loo_compact_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(perm, first, count, k, nn1, nbr1, nn_s,
                                                                                 nbr_s);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return GSK_OK;
}

// Sorts the points [first, first+count) by sample-lattice bin. Outputs (cached context buffers): perm[s] = slab-local
// original index of the s-th point in sorted order, and the sorted coordinates.
int gsk_points_sort(gsk_ctx *ctx, long long first, long long count, int **perm, double **sx, double **sy, double **sz) {
  cudaStream_t st = ctx->stream;
  const long long ncells = ctx->bins.ncells;
  int *cell_of = nullptr, *counts = nullptr;
  int rc;
  if ((rc = gsk_buf(ctx, BUF_PT_CELL, sizeof(int) * (size_t)count, (void **)&cell_of)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_COUNTS, sizeof(int) * (size_t)(2 * ncells + 1), (void **)&counts)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_PERM, sizeof(int) * (size_t)count, (void **)perm)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_X, sizeof(double) * (size_t)count, (void **)sx)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_Y, sizeof(double) * (size_t)count, (void **)sy)) != GSK_OK) return rc;
  if ((rc = gsk_buf(ctx, BUF_PT_Z, sizeof(double) * (size_t)count, (void **)sz)) != GSK_OK) return rc;
  int *start = counts + ncells;  // ncells entries (the scan's total is not needed)
  GSK_CUDA_CHECK(ctx, cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)ncells, st));
  const unsigned g = (unsigned)((count + 255) / 256);
  pt_count_kernel<<<g, 256, 0, st>>>(ctx->tg, ctx->bins, first, count, cell_of, counts);
  pt_scan_kernel<<<1, 1024, 0, st>>>(counts, ncells, start);
  GSK_CUDA_CHECK(ctx, cudaMemsetAsync(counts, 0, sizeof(int) * (size_t)ncells, st));  // reuse as the scatter cursor
  pt_scatter_kernel<<<g, 256, 0, st>>>(ctx->tg, first, count, cell_of, start, counts, *perm, *sx, *sy, *sz);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return GSK_OK;
}

int gsk_points_unscatter(gsk_ctx *ctx, const int *perm, long long count, const double *ms, const double *vs,
                         const GskOut &out, const int *nn_s, int *nn_out, const int *nbr_s, int *nbr_out, int k) {
  pt_unscatter_kernel<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(perm, count, ms, vs, out, nn_s, nn_out,
                                                                               nbr_s, nbr_out, k);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  return GSK_OK;
}
