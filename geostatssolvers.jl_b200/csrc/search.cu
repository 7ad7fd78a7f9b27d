// search.cu — K2: exact k-nearest / k-ball neighbour search on the bin lattice, replacing
// `search!(neighbors, center, searcher)` (ref: src/estimation/krig.jl:210; Meshes KNearestSearch /
// KBallSearch over a NearestNeighbors KD-tree [3P]).
//
// One CTA owns a tile of spatially adjacent targets (one target per thread). The CTA grows a block
// of bins around the tile shell by shell; each shell's samples (contiguous 32-byte records per bin
// row) are staged into shared memory with 1-D TMA bulk copies (cp.async.bulk → SASS UBLKCP) that
// complete on an mbarrier, and every thread scans the staged records (broadcast LDS.128) keeping
// its own top-k list in shared memory ([slot][thread] layout, conflict-free): one 64-bit key per
// entry (distance bits + sample index, template parameter CK) or, for ball and ranked searches,
// exact (d², index) pairs. The CTA stops when every thread's k-th distance is strictly inside the
// scanned block (or, for ball search, the block covers the ball), so the result is the exact kNN
// set; tiles whose compact-key result could depend on the dropped distance bits are searched again
// with exact keys (redo pass).
//
// Ordering key is (d², original sample index): d² is evaluated as ((dx·dx)+(dy·dy))+(dz·dz) with
// round-to-nearest mul/add and no FMA — the oracle's chain — so neighbour sets are bit-identical
// and ties fall to the lower sample index (north_star).
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "gsk_internal.cuh"

namespace {

constexpr int NT = 128;       // targets (threads) per CTA
constexpr int CB = 4;         // candidates whose loads and distances are issued together
constexpr int SCAP_MAX = 1024;  // upper bound of staged records per chunk (32 KB)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk copy global → shared, completion signalled on the mbarrier (bytes % 16 == 0, 16-B aligned)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ int bin_clamp(double x, double lo, double inv, int nb) {
  double f = floor((x - lo) * inv);
  return (f < 0.0) ? 0 : ((f >= (double)nb) ? nb - 1 : (int)f);
}

// block-wide exclusive scan of one int per thread (NT threads); returns exclusive prefix, total in *total
__device__ __forceinline__ int block_excl_scan(int v, int *warp_buf, int *total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_buf[wid] = incl;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < NT / 32; ++w) {
    int s = warp_buf[w];
    if (w < wid) base += s;
    tot += s;
  }
  __syncthreads();
  *total = tot;
  return base + incl - v;
}

// HEAP selects how a thread keeps its k best candidates: an ascending list with insertion (cheap for small k,
// O(k) per accepted candidate) or a binary max-heap (O(log k) per accepted candidate, heap-sorted once at the
// end) for large k.
// RANKED (sequential simulation, sgs.cu): records carry a rank in the high 32 bits of w next to the index, the target
// its own rank, and only records of LOWER rank are candidates — the `mask = simulated` of the reference's sequential
// loop (ref: src/simulation/seq.jl:105), evaluated for every location of the path at once.
//
// CK (compact keys): a list entry is ONE 64-bit word — the bits of d² with the low `keybits` mantissa bits replaced by
// the sample index (n <= 2^keybits) — so the (d², index) order is a single unsigned compare, the list takes 8 instead
// of 12 bytes per entry (more resident CTAs: the kernel is latency-bound) and tied distances still fall to the lower
// index. Two candidates whose d² differ only in the dropped bits would be ordered by index instead: a thread that
// meets such a pair where it matters (inside its final list, or between its k-th best and a rejected/evicted
// candidate) flags its tile, and the tile is searched again by the exact-key variant (redo list, same stream), so the
// result is the exact (d², index) order in every case. Distances whose dropped bits are all zero (lattice data) lose
// nothing and never flag.
// Launch bounds: the heap variants are asked for six CTAs per SM (<= 80 registers): left alone the compiler picks 56
// registers and spills into the hot loop (C5 search 4.60 -> 4.49 ms per 2M targets without the spills); the insertion
// compact-key variants stay at 72 registers (seven CTAs; at 80 the C2 search goes from 0.271 to 0.291 ms); the exact-key
// variants (ball and ranked searches, the redo pass) take up to 80 as well.
template <int TX, int TY, int TZ, int DIM, bool HEAP, bool RANKED = false, bool CK = false>
__global__ void __launch_bounds__(NT, (CK && !HEAP) ? 7 : 6) search_kernel(const GskSearchArgs a) {
  static_assert(TX * TY * TZ == NT, "tile must hold NT targets");
  static_assert(!(CK && RANKED), "ranked search keeps exact keys");
  typedef unsigned long long u64;
  // redo pass (exact keys): CTA i searches the i-th tile flagged by the compact-key pass
  int tile_id = blockIdx.x;
  if (!CK && a.redo_list) {
    if (blockIdx.x >= (unsigned)*a.redo_count) return;
    tile_id = a.redo_list[blockIdx.x];
  }
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = a.k;
  const int SCAP = a.scap;
  double4 *stage = reinterpret_cast<double4 *>(smem_raw);                 // SCAP records
  double *topd = reinterpret_cast<double *>(smem_raw + sizeof(double4) * SCAP);  // [K][NT]
  int *topi = reinterpret_cast<int *>(topd + (size_t)K * NT);             // [K][NT]
  u64 *topk = reinterpret_cast<u64 *>(topd);                               // CK: [K][NT] keys instead
  const u64 LOWMASK = CK ? ((1ull << a.keybits) - 1ull) : 0ull;
  __shared__ uint64_t bar;
  __shared__ int warp_buf[NT / 32];
  __shared__ int sh_bb[6];

  const int tid = threadIdx.x;
  const GskTargets &tg = a.tg;
  const GskBins &bn = a.bins;
  const int dim = tg.dim;

  // ---- my target ----
  double tc[3] = {0.0, 0.0, 0.0};
  long long lin = -1;
  bool active = false;
  int my_rank = 0;  // RANKED only
  int b0[3] = {0, 0, 0}, b1[3] = {0, 0, 0};  // bins overlapped by the tile's targets
  if (tg.is_grid) {
    int tile = tile_id;
    int tix = tile % a.ntile[0];
    int tiy = (tile / a.ntile[0]) % a.ntile[1];
    int tiz = tile / (a.ntile[0] * a.ntile[1]);
    int ix = tid % TX, iy = (tid / TX) % TY, iz = tid / (TX * TY);
    long long c[3] = {a.t0[0] + (long long)tix * TX + ix, a.t0[1] + (long long)tiy * TY + iy,
                      a.t0[2] + (long long)tiz * TZ + iz};
    bool inside = c[0] < tg.gdim[0] && c[1] < tg.gdim[1] && c[2] < tg.gdim[2];
    if (inside) {
      lin = (c[2] * tg.gdim[1] + c[1]) * tg.gdim[0] + c[0];
      active = lin >= a.first && lin < a.first + a.count;
    }
    long long cmin[3] = {a.t0[0] + (long long)tix * TX, a.t0[1] + (long long)tiy * TY, a.t0[2] + (long long)tiz * TZ};
    const int tdim[3] = {TX, TY, TZ};
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      if (d < dim) {
        tc[d] = gsk_cell_center(tg.gorg[d], tg.gsp[d], c[d]);
        long long cmax = cmin[d] + tdim[d] - 1;
        if (cmax > tg.gdim[d] - 1) cmax = tg.gdim[d] - 1;
        double lo = gsk_cell_center(tg.gorg[d], tg.gsp[d], cmin[d]);
        double hi = gsk_cell_center(tg.gorg[d], tg.gsp[d], cmax);
        if (hi < lo) { double t = lo; lo = hi; hi = t; }
        b0[d] = bin_clamp(lo, bn.lo[d], bn.inv[d], bn.nb[d]);
        b1[d] = bin_clamp(hi, bn.lo[d], bn.inv[d], bn.nb[d]);
      }
    }
  } else {
    long long t = (long long)tile_id * NT + tid;
    active = t < a.count;
    lin = a.first + t;
    int mb[3] = {0, 0, 0};
    if (active) {
      for (int d = 0; d < dim; ++d) {
        tc[d] = tg.pts[d][lin];
        mb[d] = bin_clamp(tc[d], bn.lo[d], bn.inv[d], bn.nb[d]);
      }
      if (RANKED) my_rank = a.trank[lin];
    }
    if (tid < 6) sh_bb[tid] = (tid < 3) ? 0x7fffffff : -1;
    __syncthreads();
    if (active) {
      for (int d = 0; d < 3; ++d) {
        atomicMin(&sh_bb[d], mb[d]);
        atomicMax(&sh_bb[3 + d], mb[d]);
      }
    }
    __syncthreads();
    for (int d = 0; d < 3; ++d) { b0[d] = sh_bb[d]; b1[d] = sh_bb[3 + d]; }
    if (b1[0] < 0) return;  // no active target in this CTA
  }
  // a tile with no active target exits early (uniform for the CTA)
  if (__syncthreads_or(active ? 1 : 0) == 0) return;

  if (tid == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  uint32_t parity = 0;

  int cnt = 0;
  double worst = INFINITY;  // k-th best d² once the list is full (CK: the largest d² that shares its key's distance bits)
  int worst_i = 0x7fffffff;
  u64 wkey = ~0ull;         // CK: key of the k-th best
  u64 lowbits = 0ull;       // CK: OR of the d² bits of every candidate that was not rejected on distance alone
  u64 amb = ~0ull;          // CK: distance bits at which the last candidate tied with the k-th best was left out
  const double r2 = a.use_ball ? a.radius * a.radius : INFINITY;
  // slack that keeps the "strictly inside the scanned block" test conservative against the
  // rounding of the bin assignment
  const double slack = 1e-9 * bn.cell_max;

  int ob0[3] = {1, 1, 1}, ob1[3] = {0, 0, 0};  // previously scanned block (empty)
  // The block grows one bin per level from the tile's own bins out to the density-based margin
  // (centre-out order keeps the top-k insertions short: near samples arrive first), and by ×1.5
  // per level after that. The stop test only runs once the density-based margin is reached.
  int mg[3] = {0, 0, 0};
  bool have_old = false;
  bool reached = a.margin0[0] == 0 && a.margin0[1] == 0 && a.margin0[2] == 0;

  for (;;) {
    int nb0[3], nb1[3];
    bool whole = true;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      nb0[d] = max(0, b0[d] - mg[d]);
      nb1[d] = min(bn.nb[d] - 1, b1[d] + mg[d]);
      whole = whole && nb0[d] == 0 && nb1[d] == bn.nb[d] - 1;
    }
    const int nyr = nb1[1] - nb0[1] + 1, nzr = nb1[2] - nb0[2] + 1;
    const int nrows = nyr * nzr;

    // ---- scan the shell new \ old, NT bin rows at a time ----
    for (int rbase = 0; rbase < nrows; rbase += NT) {
      int r = rbase + tid;
      int sA = 0, lA = 0, sB = 0, lB = 0;  // two record ranges (start, length)
      if (r < nrows) {
        int by = nb0[1] + r % nyr, bz = nb0[2] + r / nyr;
        long long rowbase = ((long long)bz * bn.nb[1] + by) * bn.nb[0];
        bool in_old = have_old && by >= ob0[1] && by <= ob1[1] && bz >= ob0[2] && bz <= ob1[2];
        if (!in_old) {
          sA = bn.cell_start[rowbase + nb0[0]];
          lA = bn.cell_start[rowbase + nb1[0] + 1] - sA;
        } else {
          if (nb0[0] < ob0[0]) {
            sA = bn.cell_start[rowbase + nb0[0]];
            lA = bn.cell_start[rowbase + ob0[0]] - sA;
          }
          if (nb1[0] > ob1[0]) {
            sB = bn.cell_start[rowbase + ob1[0] + 1];
            lB = bn.cell_start[rowbase + nb1[0] + 1] - sB;
          }
        }
      }
      int total;
      int off = block_excl_scan(lA + lB, warp_buf, &total);
      for (int lo = 0; lo < total; lo += SCAP) {
        const int hi = min(total, lo + SCAP);
        // TMA: every thread bulk-copies the part of its ranges that falls into [lo, hi)
        if (tid == 0) mbar_expect_tx(&bar, (uint32_t)(hi - lo) * (uint32_t)sizeof(double4));
        {
          int s0 = max(off, lo), e0 = min(off + lA, hi);
          if (e0 > s0) bulk_g2s(stage + (s0 - lo), bn.rec + sA + (s0 - off), (uint32_t)(e0 - s0) * 32u, &bar);
          int offB = off + lA;
          int s1 = max(offB, lo), e1 = min(offB + lB, hi);
          if (e1 > s1) bulk_g2s(stage + (s1 - lo), bn.rec + sB + (s1 - offB), (uint32_t)(e1 - s1) * 32u, &bar);
        }
        mbar_wait(&bar, parity);
        parity ^= 1u;
        if (active) {
          const int ns = hi - lo;
          // squared distance with round-to-nearest mul/add and no FMA: bit-identical to the oracle
          auto dist2 = [&](const double4 &rc) {
            double dx = tc[0] - rc.x;
            double d2 = __dmul_rn(dx, dx);
            if (DIM > 1) {
              double dy = tc[1] - rc.y;
              d2 = __dadd_rn(d2, __dmul_rn(dy, dy));
            }
            if (DIM > 2) {
              double dz = tc[2] - rc.z;
              d2 = __dadd_rn(d2, __dmul_rn(dz, dz));
            }
            return d2;
          };
#define TD(sl) topd[(size_t)(sl) * NT + tid]
#define TI(sl) topi[(size_t)(sl) * NT + tid]
#define TK(sl) topk[(size_t)(sl) * NT + tid]
          // CK max-heap: put `key` into the hole at slot i of a heap of n keys, moving larger children up
          auto ck_sift_down = [&](int i, const int n, const u64 key) {
            for (;;) {
              int c = 2 * i + 1;
              if (c >= n) break;
              u64 kch = TK(c);
              if (c + 1 < n) {
                const u64 kr = TK(c + 1);
                if (kr > kch) { kch = kr; ++c; }
              }
              if (kch > key) {
                TK(i) = kch;
                i = c;
              } else {
                break;
              }
            }
            TK(i) = key;
          };
          auto consider = [&](const double d2, const double w) {
            if (d2 > worst) return;
            const long long wl = __double_as_longlong(w);
            if (RANKED && (int)(wl >> 32) >= my_rank) return;
            const int oi = (int)wl;
            if (CK) {
              const u64 bits = (u64)__double_as_longlong(d2);
              const u64 kc = (bits & ~LOWMASK) | (u64)(unsigned)oi;
              lowbits |= bits;
              if (cnt == K) {
                if (kc > wkey) {  // same distance bits as the k-th best (it passed the distance test), sorted behind it
                  amb = wkey & ~LOWMASK;
                  return;
                }
              }
              if (!HEAP) {
                // ascending list, sorted insertion from the tail; a full list drops its last entry
                const int p0 = (cnt < K) ? cnt : K - 1;
                u64 *pk = &TK(p0);
                u64 *const pk_first = &TK(0);
                while (pk != pk_first) {
                  const u64 kp = pk[-NT];
                  if (kc > kp) break;
                  pk[0] = kp;
                  pk -= NT;
                }
                pk[0] = kc;
                if (cnt < K) {
                  if (++cnt == K) {
                    wkey = TK(K - 1);
                    worst = __longlong_as_double((long long)(wkey | LOWMASK));
                  }
                } else {
                  const u64 nw = TK(K - 1);
                  if (((nw ^ wkey) & ~LOWMASK) == 0ull) amb = nw & ~LOWMASK;  // the dropped entry ties with the new k-th
                  wkey = nw;
                  worst = __longlong_as_double((long long)(wkey | LOWMASK));
                }
              } else {
                if (cnt < K) {
                  // The first K candidates are only appended; the heap is built once the list is full (Floyd: at most
                  // K level steps in total). Candidates arrive roughly nearest first, so sifting each one up a
                  // max-heap would climb to the root every time (log2(cnt) levels each).
                  TK(cnt) = kc;
                  if (++cnt == K) {
                    for (int i = K / 2 - 1; i >= 0; --i) ck_sift_down(i, K, TK(i));
                    wkey = TK(0);
                    worst = __longlong_as_double((long long)(wkey | LOWMASK));
                  }
                } else {  // replace the root (the current k-th best)
                  ck_sift_down(0, K, kc);
                  const u64 nw = TK(0);
                  if (((nw ^ wkey) & ~LOWMASK) == 0ull) amb = nw & ~LOWMASK;  // the evicted entry ties with the new k-th
                  wkey = nw;
                  worst = __longlong_as_double((long long)(wkey | LOWMASK));
                }
              }
              return;
            }
            if (d2 == worst && oi > worst_i) return;
            if (!HEAP) {
              // sorted insertion with running pointers (slot stride NT is a compile-time constant, so the
              // neighbouring slot is an immediate offset) and a branch-free (d², index) comparison
              const int p0 = (cnt < K) ? cnt : K - 1;
              double *pd = &TD(p0);
              int *pi = &TI(p0);
              double *const pd_first = &TD(0);
              while (pd != pd_first) {
                const double dp = pd[-NT];
                const int ip = pi[-NT];
                const bool before = (d2 < dp) | ((d2 == dp) & (oi < ip));
                if (!before) break;
                pd[0] = dp;
                pi[0] = ip;
                pd -= NT;
                pi -= NT;
              }
              pd[0] = d2;
              pi[0] = oi;
              if (cnt < K) ++cnt;
              if (cnt == K) {
                worst = TD(K - 1);
                worst_i = TI(K - 1);
              }
            } else {
              int i;
              if (cnt < K) {  // sift up
                i = cnt++;
                while (i > 0) {
                  const int par = (i - 1) >> 1;
                  const double dp = TD(par);
                  const int ip = TI(par);
                  if (d2 > dp || (d2 == dp && oi > ip)) {
                    TD(i) = dp;
                    TI(i) = ip;
                    i = par;
                  } else {
                    break;
                  }
                }
              } else {  // replace the root (the current k-th best), sift down
                i = 0;
                for (;;) {
                  int c = 2 * i + 1;
                  if (c >= K) break;
                  double dc = TD(c);
                  int ic = TI(c);
                  if (c + 1 < K) {
                    const double dr = TD(c + 1);
                    const int ir = TI(c + 1);
                    if (dr > dc || (dr == dc && ir > ic)) { dc = dr; ic = ir; ++c; }
                  }
                  if (dc > d2 || (dc == d2 && ic > oi)) {
                    TD(i) = dc;
                    TI(i) = ic;
                    i = c;
                  } else {
                    break;
                  }
                }
              }
              TD(i) = d2;
              TI(i) = oi;
              if (cnt == K) {
                worst = TD(0);
                worst_i = TI(0);
              }
            }
          };
          // candidates in batches of CB: their broadcast loads and distance arithmetic are issued together (the
          // loads cannot move above the previous candidate's shared-memory stores by themselves), the top-k
          // updates then run in order
          int s = 0;
          for (; s + CB <= ns; s += CB) {
            double4 rc[CB];
            double dd[CB];
#pragma unroll
            for (int u = 0; u < CB; ++u) rc[u] = stage[s + u];
#pragma unroll
            for (int u = 0; u < CB; ++u) dd[u] = dist2(rc[u]);
#pragma unroll
            for (int u = 0; u < CB; ++u) consider(dd[u], rc[u].w);
          }
          for (; s < ns; ++s) {
            const double4 rc = stage[s];
            consider(dist2(rc), rc.w);
          }
        }
        __syncthreads();  // stage is overwritten by the next chunk
      }
    }

    // ---- can this thread stop? distance from the target to the nearest open face of the block ----
    bool done = true;
    if (active && !whole) {
      double margin = INFINITY;
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        if (d < dim) {
          if (nb0[d] > 0) margin = fmin(margin, tc[d] - (bn.lo[d] + nb0[d] * bn.cell[d]));
          if (nb1[d] < bn.nb[d] - 1) margin = fmin(margin, (bn.lo[d] + (nb1[d] + 1) * bn.cell[d]) - tc[d]);
        }
      }
      margin -= slack;
      double safe2 = (margin > 0.0) ? margin * margin : 0.0;
      done = (cnt == K && worst < safe2) || (safe2 > r2);
    }
    if (whole) break;
    if (reached && __syncthreads_and(done ? 1 : 0)) break;
    bool next_reached = true;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      ob0[d] = nb0[d];
      ob1[d] = nb1[d];
      if (!reached) {
        if (mg[d] < a.margin0[d]) ++mg[d];
        next_reached = next_reached && mg[d] >= a.margin0[d];
      } else {
        mg[d] += max(1, mg[d] / 2);
      }
    }
    reached = reached || next_reached;
    have_old = true;
  }

  // ---- emit: ascending (d², idx); ball search keeps sqrt(d²) <= radius (inclusive) ----
  if (CK) {
    bool flag = false;
    if (active) {
      if (HEAP) {  // heap sort in place on the keys (a list that never filled up is still unordered: build its heap first)
        auto sift_down = [&](int i, const int n, const u64 key) {
          for (;;) {
            int c = 2 * i + 1;
            if (c >= n) break;
            u64 kch = TK(c);
            if (c + 1 < n) {
              const u64 kr = TK(c + 1);
              if (kr > kch) { kch = kr; ++c; }
            }
            if (kch > key) {
              TK(i) = kch;
              i = c;
            } else {
              break;
            }
          }
          TK(i) = key;
        };
        if (cnt < K)
          for (int i = cnt / 2 - 1; i >= 0; --i) sift_down(i, cnt, TK(i));
        for (int end = cnt - 1; end > 0; --end) {
          const u64 kk = TK(end);
          TK(end) = TK(0);
          sift_down(0, end, kk);
        }
      }
      const long long t = lin - a.first;
      a.nn[t] = cnt;
      int *out = a.nbr + t * K;
      u64 prev = ~0ull;
      bool tie = false;
      for (int i = 0; i < K; ++i) {
        const u64 kk = (i < cnt) ? TK(i) : ~0ull;
        tie = tie || (((kk ^ prev) & ~LOWMASK) == 0ull && i < cnt);
        prev = kk;
        out[i] = (i < cnt) ? (int)(kk & LOWMASK) : -1;
      }
      // dropped distance bits only matter when some candidate had any
      if ((lowbits & LOWMASK) != 0ull) flag = tie || (cnt == K && amb == (wkey & ~LOWMASK));
    }
    if (__syncthreads_or(flag ? 1 : 0) && tid == 0) a.redo_list[atomicAdd(a.redo_count, 1)] = tile_id;
    return;
  }
  if (active) {
    if (HEAP) {  // heap sort in place: repeatedly move the maximum behind the shrinking heap
      for (int end = cnt - 1; end > 0; --end) {
        const double kd = TD(end);
        const int ki = TI(end);
        TD(end) = TD(0);
        TI(end) = TI(0);
        int i = 0;
        for (;;) {
          int c = 2 * i + 1;
          if (c >= end) break;
          double dc = TD(c);
          int ic = TI(c);
          if (c + 1 < end) {
            const double dr = TD(c + 1);
            const int ir = TI(c + 1);
            if (dr > dc || (dr == dc && ir > ic)) { dc = dr; ic = ir; ++c; }
          }
          if (dc > kd || (dc == kd && ic > ki)) {
            TD(i) = dc;
            TI(i) = ic;
            i = c;
          } else {
            break;
          }
        }
        TD(i) = kd;
        TI(i) = ki;
      }
    }
    int nn = cnt;
    if (a.use_ball) {
      nn = 0;
      while (nn < cnt && sqrt(topd[(size_t)nn * NT + tid]) <= a.radius) ++nn;
    }
    const long long t = lin - a.first;
    a.nn[t] = nn;
    int *out = a.nbr + t * K;
    for (int i = 0; i < K; ++i) out[i] = (i < nn) ? topi[(size_t)i * NT + tid] : -1;
  }
#undef TD
#undef TI
#undef TK
}

}  // namespace

int gsk_launch_search(gsk_ctx *ctx, cudaStream_t st, long long first, long long count, int k, int *d_nn, int *d_nbr,
                      int *launches, const int *d_trank) {
  GskSearchArgs a{};
  a.trank = d_trank;
  a.tg = ctx->tg;
  a.bins = ctx->bins;
  a.k = k;
  a.use_ball = !(ctx->prob.ball_radius != ctx->prob.ball_radius);
  a.radius = a.use_ball ? ctx->prob.ball_radius : 0.0;
  a.first = first;
  a.count = count;
  a.nn = d_nn;
  a.nbr = d_nbr;
  for (int d = 0; d < 3; ++d) a.margin0[d] = ctx->margin0[d];
  static const int scap_env = GSK_DEV_ENV("GSK_SCAP") ? atoi(GSK_DEV_ENV("GSK_SCAP")) : 0;
  {
    // staging capacity: just enough for the block a tile is expected to scan (smaller shared-memory footprint
    // → more resident CTAs, which is what the latency-bound insertion loop needs); larger blocks are simply
    // processed in several chunks. GSK_SCAP overrides (development tunable).
    double expect = 512.0;
    const int dim = ctx->tg.dim;
    if (ctx->tg.is_grid && ctx->bins.ncells > 0) {
      const int tdim[3] = {dim == 1 ? NT : (dim == 2 ? 16 : 8), dim == 1 ? 1 : (dim == 2 ? 8 : 4), dim == 3 ? 4 : 1};
      double nb = 1.0;
      for (int d = 0; d < dim; ++d)
        nb *= std::min((double)ctx->bins.nb[d],
                       tdim[d] * fabs(ctx->tg.gsp[d]) / ctx->bins.cell[d] + 1.0 + 2.0 * ctx->margin0[d]);
      expect = nb * (double)ctx->prob.n_samples / (double)ctx->bins.ncells;
    }
    int sc = 128;
    while (sc < SCAP_MAX && sc < 1.25 * expect) sc *= 2;
    a.scap = scap_env > 0 ? std::min(scap_env, SCAP_MAX) : sc;
  }
  const int dim = ctx->tg.dim;
  unsigned nblocks;
  int tile[3] = {NT, 1, 1};
  if (dim == 2) { tile[0] = 16; tile[1] = 8; }
  if (dim == 3) { tile[0] = 8; tile[1] = 4; tile[2] = 4; }
  if (ctx->tg.is_grid) {
    // bounding box of the slab in cell coordinates: whole rows/planes except along the slowest axis
    long long gd[3] = {ctx->tg.gdim[0], ctx->tg.gdim[1], ctx->tg.gdim[2]};
    long long last = first + count - 1;
    long long lo[3] = {0, 0, 0}, hi[3] = {gd[0] - 1, gd[1] - 1, gd[2] - 1};
    int slow = dim - 1;
    long long stride = 1;
    for (int d = 0; d < slow; ++d) stride *= gd[d];
    lo[slow] = first / stride;
    hi[slow] = last / stride;
    if (lo[slow] == hi[slow] && slow > 0) {  // slab inside one plane/row: tighten the next axis too
      long long s2 = stride / gd[slow - 1];
      lo[slow - 1] = (first % stride) / s2;
      hi[slow - 1] = (last % stride) / s2;
    }
    long long nt = 1;
    for (int d = 0; d < 3; ++d) {
      a.t0[d] = lo[d];
      a.ntile[d] = (int)((hi[d] - lo[d] + tile[d]) / tile[d]);
      nt *= a.ntile[d];
    }
    nblocks = (unsigned)nt;
  } else {
    nblocks = (unsigned)((count + NT - 1) / NT);
  }
  // compact keys (8 bytes per list entry) whenever the sample index fits beside >= 28 bits of the distance's mantissa;
  // ball searches (which need sqrt of the exact d²) and ranked searches keep exact keys
  int keybits = 1;
  while (keybits < 31 && (1ll << keybits) < ctx->prob.n_samples) ++keybits;
  static const int no_ck = GSK_DEV_ENV("GSK_NO_COMPACT_KEYS") ? atoi(GSK_DEV_ENV("GSK_NO_COMPACT_KEYS")) : 0;  // development tunable
  const bool ck = !d_trank && !a.use_ball && keybits <= 24 && !no_ck;
  a.keybits = keybits;
  if (ck) {
    void *p = nullptr;
    int rc = gsk_buf(ctx, BUF_REDO, sizeof(int) * ((size_t)nblocks + 1), &p);
    if (rc != GSK_OK) return rc;
    a.redo_count = reinterpret_cast<int *>(p);
    a.redo_list = a.redo_count + 1;
    GSK_CUDA_CHECK(ctx, cudaMemsetAsync(a.redo_count, 0, sizeof(int), st));
    if (scap_env <= 0) {
      // the smaller list leaves room for more CTAs: shrink the stage while that adds another resident CTA (measured,
      // C3a k = 32: 512 records 2.07 ms, 256 1.81 ms, 128 1.66 ms per 2M targets; C5 k = 64: 512 6.36 ms, 256 = 128 4.7 ms)
      auto ctas = [&](int sc) { return (int)(232448 / (sizeof(double4) * sc + (size_t)a.k * NT * 8 + 1024 + 64)); };
      while (a.scap > 128 && ctas(a.scap / 2) > ctas(a.scap)) a.scap /= 2;
    }
  }
  const size_t smem_exact = sizeof(double4) * a.scap + (size_t)a.k * NT * (sizeof(double) + sizeof(int));
  const size_t smem = ck ? sizeof(double4) * a.scap + (size_t)a.k * NT * sizeof(unsigned long long) : smem_exact;
  cudaError_t e;
  static const int heap_min_k = GSK_DEV_ENV("GSK_HEAP_MIN_K") ? atoi(GSK_DEV_ENV("GSK_HEAP_MIN_K")) : 24;  // development tunable
  const bool heap = a.k >= heap_min_k;
#define GSK_LAUNCH_SEARCH(TX, TY, TZ, D, H)                                                                        \
  do {                                                                                                             \
    if (ck) {                                                                                                      \
      e = cudaFuncSetAttribute(search_kernel<TX, TY, TZ, D, H, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
      if (e == cudaSuccess) search_kernel<TX, TY, TZ, D, H, false, true><<<nblocks, NT, smem, st>>>(a);            \
      if (e == cudaSuccess) e = cudaGetLastError();                                                                \
    } else {                                                                                                       \
      a.redo_list = nullptr;                                                                                       \
      a.redo_count = nullptr;                                                                                      \
      e = cudaSuccess;                                                                                             \
    }                                                                                                              \
    if (e == cudaSuccess)                                                                                          \
      e = cudaFuncSetAttribute(search_kernel<TX, TY, TZ, D, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_exact); \
    if (e == cudaSuccess) search_kernel<TX, TY, TZ, D, H><<<nblocks, NT, smem_exact, st>>>(a);                     \
  } while (0)
#define GSK_LAUNCH_RANKED(D, H)                                                                                    \
  do {                                                                                                             \
    e = cudaFuncSetAttribute(search_kernel<NT, 1, 1, D, H, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    if (e == cudaSuccess) search_kernel<NT, 1, 1, D, H, true><<<nblocks, NT, smem, st>>>(a);                       \
  } while (0)
  if (d_trank) {  // explicit points only (the tile shape is unused on that branch)
    if (ctx->tg.is_grid) { ctx->err = "ranked search needs explicit points"; return GSK_ERR_STATE; }
    if (dim == 1) { if (heap) GSK_LAUNCH_RANKED(1, true); else GSK_LAUNCH_RANKED(1, false); }
    else if (dim == 2) { if (heap) GSK_LAUNCH_RANKED(2, true); else GSK_LAUNCH_RANKED(2, false); }
    else { if (heap) GSK_LAUNCH_RANKED(3, true); else GSK_LAUNCH_RANKED(3, false); }
  } else if (dim == 1) {
    if (heap) GSK_LAUNCH_SEARCH(NT, 1, 1, 1, true); else GSK_LAUNCH_SEARCH(NT, 1, 1, 1, false);
  } else if (dim == 2) {
    if (heap) GSK_LAUNCH_SEARCH(16, 8, 1, 2, true); else GSK_LAUNCH_SEARCH(16, 8, 1, 2, false);
  } else {
    if (heap) GSK_LAUNCH_SEARCH(8, 4, 4, 3, true); else GSK_LAUNCH_SEARCH(8, 4, 4, 3, false);
  }
#undef GSK_LAUNCH_SEARCH
#undef GSK_LAUNCH_RANKED
  GSK_CUDA_CHECK(ctx, e);
  GSK_CUDA_CHECK(ctx, cudaGetLastError());
  if (launches) *launches += ck ? 2 : 1;
  return GSK_OK;
}
