// ranging_kernel.cuh -- k_ranging: sensitivity ranges of optimal LPs from their final tableaus (a post-pass over
// tableaus already in device memory; yalps_b200/sensitivity.py ranges_from_tableau is the specification).
//
// Per variable id v, packed like pos_out, with b+_r = max(M[r,0], +0), g_c = min(M[0,c], +0) and a cell counting
// when |cell| > precision:
//   structural j non-basic at column c   (-inf, -g_c)                                              O(1)
//   structural j basic at row r          max / min of g_c / M[r,c] over c = 1..W-1                 row reduction
//   slack of row k                       max / min of -b+_r / d[r] over r = 1..H-1,                 column reduction,
//                                        d = dir(W+k) - dir(W+pair)  (dir: column M[:,pos] or unit)  O(1) if all unit
// Ids 0 and W, and every id of a non-optimal LP: NaN.
//
// Column view of the reductions: the slack s that is non-basic at column c owns column c (task T1, d = M[:,c] -
// dir(pair)); its pair p, when basic at row rp, is ranged on the same column (task T2, d = e_rp - M[:,c]).  A thread
// that owns column c therefore walks down the rows once and serves both, plus its share of every row reduction.
//
// Every candidate is one IEEE division with its zero normalised to +0.0, so lo candidates lie in [-inf, +0] and hi
// candidates in [+0, +inf].  On those two intervals the order of doubles is the order of their bit patterns read as
// unsigned integers (reversed for lo): max(lo) and min(hi) are both the minimum of the bits.  Partial results of a
// warp, a CTA or several CTAs combine with one unsigned min (__reduce_min_sync, atomicMin), which gives the same bits
// whatever the tiling or the launch order.
//
// Two decompositions, chosen by the host from the launch's caps:
//   warp mode (kRngWarp, small tableaus such as config 2's 33x65): one warp per LP, columns in 32-wide chunks, all
//     rows per chunk; the inverse of pos and the row reductions live in the warp's shared memory; no atomics.
//   tile mode (KC/KG/K4 sizes, up to 4097x8193): kRngInit writes the O(1) results, the empty value of every
//     reduction and the inverse of pos (scratch `var`); kRngTiles then runs one CTA per (LP, kRngTileRows rows,
//     kRngTileCols columns) tile and combines its partials with atomicMin on the output bits.
// Each cell of a final tableau is read once (coalesced along its row), except the column of a pair partner that is
// non-basic as well: an optimal basis never has both slacks of one key non-basic (their rows would make the basis
// singular), so that read only happens on synthetic input.
#pragma once

#include "simplex_device.cuh"

namespace yalps {

enum : int { kRngWarp = 0, kRngInit = 1, kRngTiles = 2 };

constexpr int kRngWarps = 4;        // warp mode: LPs (warps) per CTA
constexpr int kRngTileCols = 256;   // tile mode: threads per CTA, one column each
constexpr int kRngTileRows = 128;   // tile mode: rows per tile
constexpr int kRngBatch = 4;        // rows whose loads are issued together

// The LPs a post-pass over final tableaus visits (k_ranging, k_certificate): uniform or ragged, optionally through the
// `index` of a ragged group, packed like the solve's outputs.
struct PostArgs {
  long long n;
  int H, W;                                       // uniform shape (heights == nullptr)
  int Hcap, Wcap;                                 // largest LP of the launch (warp or CTA decomposition)
  const double *M;                                // final tableaus, packed like mat_out
  const int *heights, *widths;                    // ragged (nullable)
  const long long *mat_off, *rhs_off, *pos_off;
  const int *index;                               // launch-local LP -> LP id (nullable)
  const int *pos;                                 // positionOfVariable, packed like pos_out
  const int *status;                              // nullable (k_ranging: every LP is optimal)
};

// one warp per LP for tableaus up to 256 x 128, else a wider decomposition
inline bool post_warp_mode(const PostArgs &a) { return a.Wcap <= 128 && a.Hcap <= 256; }

// LP i of a post-pass launch: its id, shape and the offsets of its tableau, rows and variable ids
struct PostLP {
  long long id, mo, ro, po;
  int H, W;
};

__device__ __forceinline__ PostLP post_lp(const PostArgs &a, long long i) {
  PostLP P;
  P.id = a.index ? a.index[i] : i;
  const bool ragged = a.heights != nullptr;
  P.H = ragged ? a.heights[P.id] : a.H;
  P.W = ragged ? a.widths[P.id] : a.W;
  P.mo = ragged ? a.mat_off[P.id] : P.id * (long long)a.H * a.W;
  P.ro = ragged ? a.rhs_off[P.id] : P.id * (long long)a.H;
  P.po = ragged ? a.pos_off[P.id] : P.id * (long long)(a.H + a.W);
  return P;
}

struct RangingArgs : PostArgs {
  const int *pairs;                               // nullable: per row, the other row of its key or -1 (like rhs_out)
  double precision;
  double *lo, *hi;                                // outputs, packed like pos_out
  int *var;                                       // tile mode: inverse of pos, packed like pos (scratch)
  int tiles_r, tiles_c;                           // tile mode: row tiles and column tiles per LP (from the caps)
  size_t warp_smem;                               // warp mode: shared-memory bytes per warp
};

struct RngLP {
  const double *M;
  const int *pos, *pairs;
  double *lo, *hi;
  int *var;
  int H, W;
  bool optimal;
};

__device__ __forceinline__ RngLP rng_lp(const RangingArgs &a, long long i) {
  const PostLP P = post_lp(a, i);
  RngLP L;
  L.H = P.H;
  L.W = P.W;
  L.M = a.M + P.mo;
  L.pos = a.pos + P.po;
  L.pairs = a.pairs ? a.pairs + P.ro : nullptr;
  L.lo = a.lo + P.po;
  L.hi = a.hi + P.po;
  L.var = a.var ? a.var + P.po : nullptr;
  L.optimal = !a.status || a.status[P.id] == ST_OPTIMAL;
  return L;
}

constexpr unsigned long long kRngLoEmpty = 0xfff0000000000000ULL;  // bits of -inf
constexpr unsigned long long kRngHiEmpty = 0x7ff0000000000000ULL;  // bits of +inf

__device__ __forceinline__ unsigned long long rng_bits(double x) { return (unsigned long long)__double_as_longlong(x); }
__device__ __forceinline__ double rng_val(unsigned long long b) { return __longlong_as_double((long long)b); }

// one candidate: num / den (div_rn: the bits of __ddiv_rn) with -0.0 turned into +0.0
__device__ __forceinline__ double rng_q(double num, double den) { return __dadd_rn(div_rn(num, den), 0.0); }

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long x) {
  const unsigned h = (unsigned)(x >> 32), l = (unsigned)x;
  const unsigned wh = __reduce_min_sync(0xffffffffu, h);
  const unsigned wl = __reduce_min_sync(0xffffffffu, h == wh ? l : 0xffffffffu);
  return ((unsigned long long)wh << 32) | wl;
}

// the pair of slack row k, or -1 (an out-of-range entry counts as none)
__device__ __forceinline__ int rng_pair(const RngLP &L, int k) {
  if (!L.pairs) return -1;
  const int p = L.pairs[k];
  return (p >= 1 && p < L.H && p != k) ? p : -1;
}

// The O(1) part of id v: writes the final value of an id that needs no reduction, and the empty interval of one
// that does (row or column reductions then lower / raise it).
__device__ __forceinline__ void rng_o1(const RngLP &L, int v, double prec) {
  const int W = L.W, H = L.H;
  const double nan = d_nan(), inf = d_inf();
  double lo = -inf, hi = inf;
  if (v == 0 || v == W) {
    lo = hi = nan;
  } else if (v < W) {
    const int p = L.pos[v];
    if (p >= 1 && p < W) hi = __dadd_rn(-fmin(L.M[p], 0.0), 0.0);
  } else {
    const int k = v - W, p = L.pos[v], q = rng_pair(L, k);
    const int pq = q >= 0 ? L.pos[W + q] : -1;
    const bool k_nb = p >= 1 && p < W, q_nb = pq >= 1 && pq < W;
    if (!k_nb && !q_nb && fabs(1.0) > prec) {  // d is e_r1 [- e_r2]: one cell per unit vector
      const int r1 = p - W, r2 = q >= 0 ? pq - W : -1;
      if (r1 >= 1 && r1 < H) lo = rng_q(-fmax(L.M[(long long)r1 * W], 0.0), 1.0);
      if (r2 >= 1 && r2 < H) hi = rng_q(-fmax(L.M[(long long)r2 * W], 0.0), -1.0);
    }
  }
  L.lo[v] = lo;
  L.hi[v] = hi;
}

// Column c's tasks: T1 = the slack that is non-basic at c (id1), T2 = its pair when basic (id2, at row rp); c2 = the
// pair's column when it is non-basic too.
struct RngCol {
  int id1 = -1, id2 = -1, rp = -1, c2 = -1;
  double g = 0.0;
  double lo1, hi1, lo2, hi2;
};

__device__ __forceinline__ void rng_col_setup(const RngLP &L, int c, int var_c, RngCol &t) {
  t.lo1 = t.lo2 = -d_inf();
  t.hi1 = t.hi2 = d_inf();
  if (c < 1 || c >= L.W) return;
  t.g = fmin(L.M[c], 0.0);
  if (var_c <= L.W || var_c >= L.W + L.H) return;
  t.id1 = var_c;
  const int q = rng_pair(L, var_c - L.W);
  if (q < 0) return;
  const int pq = L.pos[L.W + q];
  if (pq >= 1 && pq < L.W) {
    t.c2 = pq;
  } else {
    t.rp = pq - L.W;
    t.id2 = L.W + q;
  }
}

// row r of column c: a = M[r,c], nb = -b+_r, a2 = M[r,c2] (when c2 >= 0)
__device__ __forceinline__ void rng_col_row(RngCol &t, int r, double a, double nb, double a2, double prec) {
  if (t.id1 < 0) return;
  const double u = r == t.rp ? 1.0 : 0.0;
  const double d1 = __dsub_rn(a, t.c2 >= 0 ? a2 : u);
  if (fabs(d1) > prec) {
    const double q = rng_q(nb, d1);
    if (d1 > 0.0) t.lo1 = fmax(t.lo1, q);
    else t.hi1 = fmin(t.hi1, q);
  }
  if (t.id2 >= 0) {
    const double d2 = __dsub_rn(u, a);
    if (fabs(d2) > prec) {
      const double q = rng_q(nb, d2);
      if (d2 > 0.0) t.lo2 = fmax(t.lo2, q);
      else t.hi2 = fmin(t.hi2, q);
    }
  }
}

// a row reduction's candidates from column c (a = M[r,c], g = g_c), as bits
__device__ __forceinline__ void rng_row_cand(bool col_ok, double a, double g, double prec, unsigned long long &lo,
                                             unsigned long long &hi) {
  lo = kRngLoEmpty;
  hi = kRngHiEmpty;
  if (col_ok && fabs(a) > prec) {
    const unsigned long long b = rng_bits(rng_q(g, a));
    if (a > 0.0) lo = b;
    else hi = b;
  }
}

// ---- warp mode: one warp per LP -------------------------------------------------------------------------------------
__device__ __forceinline__ void rng_warp(const RangingArgs &a, char *smem) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * kRngWarps;
  char *base = smem + (threadIdx.x >> 5) * a.warp_smem;
  const double prec = a.precision;
  for (long long i = (long long)blockIdx.x * kRngWarps + (threadIdx.x >> 5); i < a.n; i += warps) {
    const RngLP L = rng_lp(a, i);
    const int H = L.H, W = L.W;
    if (!L.optimal) {
      for (int v = lane; v < W + H; v += 32) L.lo[v] = L.hi[v] = d_nan();
      continue;
    }
    int *var = (int *)base;                                                          // W + H
    unsigned long long *rk = (unsigned long long *)(base + (((size_t)(W + H) * 4 + 15) & ~(size_t)15));  // 2 per row
    for (int v = lane; v < W + H; v += 32) {
      const int p = L.pos[v];
      if (p >= 0 && p < W + H) var[p] = v;
      rng_o1(L, v, prec);
    }
    for (int r = lane; r < H; r += 32) {
      rk[2 * r] = kRngLoEmpty;
      rk[2 * r + 1] = kRngHiEmpty;
    }
    __syncwarp();
    for (int c0 = 0; c0 < W; c0 += 32) {
      const int c = c0 + lane;
      RngCol t;
      rng_col_setup(L, c, c < W ? var[c] : -1, t);
      const bool col_ok = c >= 1 && c < W;
      for (int rb = 1; rb < H; rb += kRngBatch) {  // the loads of kRngBatch rows in flight together
        double av[kRngBatch], nb[kRngBatch], a2[kRngBatch];
#pragma unroll
        for (int u = 0; u < kRngBatch; u++) {
          const double *row = L.M + (long long)min(rb + u, H - 1) * W;
          av[u] = col_ok ? row[c] : 0.0;
          nb[u] = -fmax(row[0], 0.0);
          a2[u] = t.c2 >= 0 ? row[t.c2] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < kRngBatch; u++) {
          const int r = rb + u;
          if (r >= H) continue;
          rng_col_row(t, r, av[u], nb[u], a2[u], prec);
          const int rv = var[W + r];
          if (rv >= 1 && rv < W) {  // basic structural: warp-uniform branch
            unsigned long long lo, hi;
            rng_row_cand(col_ok, av[u], t.g, prec, lo, hi);
            lo = warp_min_u64(lo);
            hi = warp_min_u64(hi);
            if (lane == 0) {
              rk[2 * r] = min(rk[2 * r], lo);
              rk[2 * r + 1] = min(rk[2 * r + 1], hi);
            }
          }
        }
      }
      if (t.id1 >= 0) {
        L.lo[t.id1] = t.lo1;
        L.hi[t.id1] = t.hi1;
      }
      if (t.id2 >= 0) {
        L.lo[t.id2] = t.lo2;
        L.hi[t.id2] = t.hi2;
      }
    }
    __syncwarp();
    for (int r = 1 + lane; r < H; r += 32) {
      const int rv = var[W + r];
      if (rv >= 1 && rv < W) {
        L.lo[rv] = rng_val(rk[2 * r]);
        L.hi[rv] = rng_val(rk[2 * r + 1]);
      }
    }
    __syncwarp();
  }
}

// ---- tile mode --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void rng_init(const RangingArgs &a) {
  for (long long i = blockIdx.x; i < a.n; i += gridDim.x) {
    const RngLP L = rng_lp(a, i);
    for (int v = threadIdx.x; v < L.W + L.H; v += blockDim.x) {
      if (!L.optimal) {
        L.lo[v] = L.hi[v] = d_nan();
        continue;
      }
      const int p = L.pos[v];
      if (p >= 0 && p < L.W + L.H) L.var[p] = v;
      rng_o1(L, v, a.precision);
    }
  }
}

__device__ __forceinline__ void rng_tiles(const RangingArgs &a) {
  __shared__ double s_nb[kRngTileRows];
  __shared__ int s_rv[kRngTileRows];
  __shared__ unsigned long long s_rk[2 * kRngTileRows];
  const int tid = threadIdx.x, lane = tid & 31;
  const long long per_lp = (long long)a.tiles_r * a.tiles_c;
  const double prec = a.precision;
  for (long long b = blockIdx.x; b < a.n * per_lp; b += gridDim.x) {
    const RngLP L = rng_lp(a, b / per_lp);
    const int tr = (int)((b % per_lp) / a.tiles_c), tc = (int)(b % a.tiles_c);
    const int H = L.H, W = L.W;
    const int r0 = 1 + tr * kRngTileRows, r1 = min(H, r0 + kRngTileRows), c0 = tc * kRngTileCols;
    if (!L.optimal || r0 >= H || c0 >= W) continue;  // block-uniform
    if (tid < r1 - r0) {
      const int r = r0 + tid;
      s_nb[tid] = -fmax(L.M[(long long)r * W], 0.0);
      const int rv = L.var[W + r];
      s_rv[tid] = (rv >= 1 && rv < W) ? rv : -1;
      s_rk[2 * tid] = kRngLoEmpty;
      s_rk[2 * tid + 1] = kRngHiEmpty;
    }
    const int c = c0 + tid;
    const bool col_ok = c >= 1 && c < W;
    RngCol t;
    rng_col_setup(L, c, c < W ? L.var[c] : -1, t);
    __syncthreads();
    for (int rb = r0; rb < r1; rb += kRngBatch) {
      double av[kRngBatch], a2[kRngBatch];
#pragma unroll
      for (int u = 0; u < kRngBatch; u++) {
        const double *row = L.M + (long long)min(rb + u, r1 - 1) * W;
        av[u] = col_ok ? row[c] : 0.0;
        a2[u] = t.c2 >= 0 ? row[t.c2] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < kRngBatch; u++) {
        const int r = rb + u;
        if (r >= r1) continue;
        rng_col_row(t, r, av[u], s_nb[r - r0], a2[u], prec);
        if (s_rv[r - r0] >= 0) {  // block-uniform
          unsigned long long lo, hi;
          rng_row_cand(col_ok, av[u], t.g, prec, lo, hi);
          lo = warp_min_u64(lo);
          hi = warp_min_u64(hi);
          if (lane == 0) {
            if (lo != kRngLoEmpty) atomicMin(&s_rk[2 * (r - r0)], lo);
            if (hi != kRngHiEmpty) atomicMin(&s_rk[2 * (r - r0) + 1], hi);
          }
        }
      }
    }
    __syncthreads();
    if (tid < r1 - r0 && s_rv[tid] >= 0) {
      if (s_rk[2 * tid] != kRngLoEmpty) atomicMin((unsigned long long *)(L.lo + s_rv[tid]), s_rk[2 * tid]);
      if (s_rk[2 * tid + 1] != kRngHiEmpty) atomicMin((unsigned long long *)(L.hi + s_rv[tid]), s_rk[2 * tid + 1]);
    }
    if (t.id1 >= 0) {
      if (rng_bits(t.lo1) != kRngLoEmpty) atomicMin((unsigned long long *)(L.lo + t.id1), rng_bits(t.lo1));
      if (rng_bits(t.hi1) != kRngHiEmpty) atomicMin((unsigned long long *)(L.hi + t.id1), rng_bits(t.hi1));
    }
    if (t.id2 >= 0) {
      if (rng_bits(t.lo2) != kRngLoEmpty) atomicMin((unsigned long long *)(L.lo + t.id2), rng_bits(t.lo2));
      if (rng_bits(t.hi2) != kRngHiEmpty) atomicMin((unsigned long long *)(L.hi + t.id2), rng_bits(t.hi2));
    }
    __syncthreads();  // the shared arrays are refilled by the next tile
  }
}

__global__ void __launch_bounds__(kRngTileCols) k_ranging(RangingArgs a, int mode) {
  extern __shared__ __align__(16) char rng_smem[];
  if (mode == kRngWarp)
    rng_warp(a, rng_smem);
  else if (mode == kRngInit)
    rng_init(a);
  else
    rng_tiles(a);
}

}  // namespace yalps
