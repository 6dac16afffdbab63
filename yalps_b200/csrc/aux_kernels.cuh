// aux_kernels.cuh -- non-template kernels (compiled once, in yalps_b200.cu): standalone node assembly (K3),
// input generators (K5), density probe, roundToPrecision probe, shared-memory stream benchmark.
#pragma once

#include "fastdiv.cuh"
#include "kernels.cuh"

namespace yalps {

// K3 standalone: applyCuts (src/branchAndCut.ts:22-61) for a wave of nodes into HBM working copies
// (row stride W, node stride Hcap*W) -- used in front of the grid kernel; K1/K2 fuse the same assembly.
__global__ void k_assemble_nodes(long long n, int rootH, int W, int Hcap, const double *root, const int *root_pos,
                                 const int *cut_off, const double *cut_sign, const int *cut_var, const double *cut_val,
                                 double *work) {
  const size_t root_cells = (size_t)rootH * W;
  for (long long node = blockIdx.y; node < n; node += gridDim.y) {
    double *dst = work + (size_t)node * Hcap * W;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < root_cells; k += (size_t)gridDim.x * blockDim.x)
      dst[k] = root[k];
    const int cbeg = cut_off[node], ncuts = cut_off[node + 1] - cbeg;
    for (int i = blockIdx.x; i < ncuts; i += gridDim.x) {
      const double sign = cut_sign[cbeg + i], value = cut_val[cbeg + i];
      const int p = root_pos[cut_var[cbeg + i]];
      double *dr = dst + (size_t)(rootH + i) * W;
      if (p < W) {
        for (int c = threadIdx.x; c < W; c += blockDim.x) dr[c] = (c == 0) ? __dmul_rn(sign, value) : (c == p ? sign : 0.0);
      } else {
        const double *sr = root + (size_t)(p - W) * W;
        for (int c = threadIdx.x; c < W; c += blockDim.x)
          dr[c] = (c == 0) ? __dmul_rn(sign, __dsub_rn(value, sr[0])) : __dmul_rn(-sign, sr[c]);
      }
    }
  }
}

// ---- K5: generators -------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t prospector_hash(uint32_t x) {  // tests/helpers/util.ts:20-29
  x ^= x >> 16;
  x *= 0x21f0aaadu;
  x ^= x >> 15;
  x *= 0xd35a2d97u;
  x ^= x >> 15;
  return x;
}

// draw d (0-based) of newRand(seed0): state after d+1 increments (tests/helpers/util.ts:38-41)
__host__ __device__ __forceinline__ double rand_draw(uint32_t seed0, uint32_t d) {
  return (double)prospector_hash(seed0 + (d + 1u) * 0x9e3779b9u) / 4294967296.0;
}

// Dense synthetic LPs (SURVEY 8(d) config 2 / 5).  Draw order: c_1..c_n, then per row a_k1..a_kn, b_k.
__global__ void k_generate_synthetic(long long first, long long n, int m, int nvars, int neg_rows, uint32_t salt,
                                     double *out) {
  const int W = nvars + 1, H = m + 1;
  const size_t cells = (size_t)W * H;
  const size_t total = (size_t)n * cells;
  for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
    const long long i = (long long)(g / cells);
    const int cell = (int)(g % cells);
    const int r = cell / W, c = cell % W;
    const uint32_t seed0 = prospector_hash((uint32_t)(first + i) ^ salt);
    double v;
    if (r == 0) {
      v = (c == 0) ? 0.0 : rand_draw(seed0, (uint32_t)(c - 1));
    } else {
      const uint32_t base = (uint32_t)nvars + (uint32_t)(r - 1) * (uint32_t)(nvars + 1);
      if (c == 0) {
        const double u = rand_draw(seed0, base + (uint32_t)nvars);
        v = (r <= neg_rows) ? -(0.5 + u) : (double)nvars * (0.25 + 0.5 * u);
      } else {
        v = rand_draw(seed0, base + (uint32_t)(c - 1));
        if (r <= neg_rows) v = -v;
      }
    }
    out[g] = v;
  }
}

// RHS-perturbed replicas of one base tableau (SURVEY 8(d) config 3).
__global__ void k_generate_replicas(long long first, long long n, int H, int W, const double *base, const int *group,
                                    double eps, uint32_t salt, double *out) {
  const size_t cells = (size_t)W * H;
  const size_t total = (size_t)n * cells;
  for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
    const long long i = (long long)(g / cells);
    const int cell = (int)(g % cells);
    const int r = cell / W, c = cell % W;
    double v = base[cell];
    if (c == 0 && group[r] >= 0) {
      const uint32_t seed0 = prospector_hash((uint32_t)(first + i) ^ salt);
      const double u = rand_draw(seed0, (uint32_t)group[r]);
      v = __dmul_rn(v, __dadd_rn(1.0, __dmul_rn(eps, __dsub_rn(__dmul_rn(2.0, u), 1.0))));
    }
    out[g] = v;
  }
}

// Replicas of one base tableau that differ only in the RHS column (yalps_solve_replicas): the caller ships the base
// once and n*H right-hand sides; the working copies are assembled here, in HBM, at copy bandwidth.
__global__ void k_expand_replicas(long long n, int H, int W, const double *base, const double *rhs, double *out) {
  const size_t cells = (size_t)W * H;
  const size_t total = (size_t)n * cells;
  for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
    const size_t i = g / cells;
    const int cell = (int)(g - i * cells);
    const int r = cell / W, c = cell - r * W;
    out[g] = c == 0 ? rhs[i * (size_t)H + r] : base[cell];
  }
}

// Row subsets of one base tableau (yalps_solve_row_subsets): LP i is `base` with every row r >= 1 whose bit is clear in
// keep[i*words + r/32] set to +0.0 in every cell, column 0 included.  The simplex then follows the trajectory of the
// model without those rows (DESIGN §3), so the caller ships the base once and H/8 bytes of mask per LP.  Write-bound:
// one warp per (LP, row), whose keep word lane 0 reads once; a zeroed row does not read the base; a row is stored as
// 16-byte pairs from its first 16-byte aligned cell (consecutive tableaus, and the rows of an odd width, are only
// 8-byte aligned).  Cells move as 64-bit integers, so NaN payloads and signed zeros keep their bits.
__global__ void k_expand_subsets(long long n, int H, int W, int words, const double *base, const unsigned *keep,
                                 double *out) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  const long long *src0 = reinterpret_cast<const long long *>(base);
  for (long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); item < n * H; item += warps) {
    const long long i = item / H;
    const int r = (int)(item - i * H);
    unsigned w = 0;
    if (lane == 0) w = keep[i * words + (r >> 5)];
    w = __shfl_sync(0xffffffffu, w, 0);
    const bool kept = r == 0 || ((w >> (r & 31)) & 1u);
    long long *dst = reinterpret_cast<long long *>(out) + item * W;
    const long long *src = src0 + (size_t)r * W;
    const int head = min((int)((reinterpret_cast<uintptr_t>(dst) >> 3) & 1), W);  // 1: dst is 8 mod 16
    const int pairs = (W - head) >> 1;
    if (lane == 0 && head) dst[0] = kept ? src[0] : 0;
    longlong2 *d2 = reinterpret_cast<longlong2 *>(dst + head);
    for (int k = lane; k < pairs; k += 32)
      d2[k] = kept ? make_longlong2(src[head + 2 * k], src[head + 2 * k + 1]) : make_longlong2(0, 0);
    if (lane == 0 && head + 2 * pairs < W) dst[W - 1] = kept ? src[W - 1] : 0;
  }
}

// ---- replica path sharing (yalps_solve_replicas) -----------------------------------------------------------------
// n replicas of one tableau differ only in column 0.  Everything else of the tableau -- objective row, pivot rows and
// columns, the basis bookkeeping -- evolves identically for every replica that makes the same pivot choices, and those
// choices depend on a replica's own data only through its RHS column: the leaving row of phase 1 (most negative RHS),
// the ratio test of phase 2, and the moment phase 1 ends.  So ONE replica (the leader: the base tableau itself) is
// solved with a trace -- per pivot the choice, the pivot element and the raw pivot column, plus tableau snapshots --
// and every other replica FOLLOWS it carrying only its RHS column (one warp per replica, H doubles in shared memory):
// per pivot it re-derives its own choice from the trace and its RHS, applies the pivot to its RHS with the reference's
// operations (src/simplex.ts:16-36 restricted to column 0), and stops following at the first step where its choice
// differs from the leader's.  From there it continues alone: its tableau is the leader's snapshot of that step with its
// own column 0, handed to the ordinary kernels together with (phase, pivot counters) to resume.  Results are those of
// solving every replica on its own, bit for bit; the coefficient updates of a shared path are simply not repeated.
struct FollowArgs {
  long long n;
  int H, W, Hp;
  const double *rhs_in;   // [n][H]
  const int *steps;       // [K + 1][4]: phase, row, col, terminal flag
  const double *q;        // [K]
  const double *colraw;   // [K][Hp]
  const int *leader_var;  // variableAtPosition of the leader's final tableau
  int K;                  // pivots recorded
  int leader_done;        // the trace ends with the leader's own termination (not with a full trace buffer)
  int leader_status;
  double precision, max_pivots;
  int *status;
  double *value;
  long long *pivots;
  double *rhs_out;        // [n][H]: final RHS of a replica that finished on the path, its RHS at the fork otherwise
  int *pos_out, *var_out; // [n][W + H] (nullable)
  int *fork_count;        // number of replicas that left the path
  int *fork_ids;          // [n] their indices, in arrival order
  int *fork_step;         // [n] (indexed by replica) the step at which it left
  long long *fork_resume; // [n][3] (indexed by replica) phase and pivot counters at that step
  // optional reduced costs [n][W + H] (BatchArgs::red_out): a replica that finishes on the path has the leader's final
  // row 0 in columns 1..W-1 (column 0 never feeds the others) and its basis, so it copies the leader's vector
  double *red_out;
  const double *leader_red;
};

constexpr int kFollowWarps = 8;

__global__ void __launch_bounds__(kFollowWarps * 32) k_replica_follow(const FollowArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int H = a.H, W = a.W;
  double *b = reinterpret_cast<double *>(smem_raw) + (size_t)warp * a.Hp;
  const double precision = a.precision, INF = d_inf();
  const long long budget =
      !(a.max_pivots > 0.0) ? 0LL : (a.max_pivots >= 9.0e18 ? 0x7fffffffffffffffLL : (long long)ceil(a.max_pivots));
  const int end_phase = a.steps[4 * a.K], end_row = a.steps[4 * a.K + 1], end_col = a.steps[4 * a.K + 2];
  for (long long i = (long long)blockIdx.x * kFollowWarps + warp; i < a.n; i += (long long)gridDim.x * kFollowWarps) {
    for (int r = lane; r < H; r += 32) b[r] = a.rhs_in[(size_t)i * H + r];
    __syncwarp();
    int phase = 1, k = 0, status = ST_CYCLED;
    long long p1 = 0, p2 = 0, iter = 0;
    double value = d_nan();
    bool forked = false;
    for (;;) {
      if (iter >= budget) break;  // "cycled" (:102,:141): on the shared path the leader ends the same way
      int row = kNone;
      if (phase == 1) {
        double bv = INF;
        int bi = kNone;
        for (int r = 1 + lane; r < H; r += 32) {  // (:111-119)
          const double v = b[r];
          if (v < -precision && v < bv) {
            bv = v;
            bi = r;
          }
        }
        const unsigned long long key = bi == kNone ? no_key<false>() : order_key(bv);
        row = warp_best<false>((unsigned)(key >> 32), (unsigned)key, bi).idx;
        if (row == kNone) {  // (:120)
          phase = 2;
          iter = 0;
          continue;
        }
        if (k == a.K) {  // the leader stopped here: same verdict only if it had chosen the same row and found no column
          if (a.leader_done && end_phase == 1 && a.leader_status == ST_INFEASIBLE && end_row == row)
            status = ST_INFEASIBLE;
          else
            forked = true;
          break;
        }
        if (a.steps[4 * k] != 1 || a.steps[4 * k + 1] != row) {  // (the column follows from the row and shared data)
          forked = true;
          break;
        }
      } else {
        if (k == a.K) {  // entering column and candidate rows depend on shared data only
          if (a.leader_done && end_phase == 2 && a.leader_status == ST_OPTIMAL) {
            status = ST_OPTIMAL;
            value = round_to_precision(b[0], precision);
          } else if (a.leader_done && end_phase == 2 && a.leader_status == ST_UNBOUNDED) {
            status = ST_UNBOUNDED;
            value = (double)end_col;
          } else {
            forked = true;
          }
          break;
        }
        if (a.steps[4 * k] != 2) {
          forked = true;
          break;
        }
        const double *colk = a.colraw + (size_t)k * a.Hp;
        double bv = INF;
        int bi = kNone;
        for (int r = 1 + lane; r < H; r += 32) {  // ratio test (:83-95)
          const double v = colk[r];
          if (v > precision) {
            const double ratio = div_rn(b[r], v);
            if (ratio < INF) {
              const double kk = (ratio <= precision) ? -INF : ratio;
              if (bi == kNone || kk < bv) {
                bv = kk;
                bi = r;
              }
            }
          }
        }
        const unsigned long long key = bi == kNone ? no_key<false>() : order_key(bv);
        row = warp_best<false>((unsigned)(key >> 32), (unsigned)key, bi).idx;
        if (row != a.steps[4 * k + 1]) {  // (kNone included: the ordinary kernel gives the verdict)
          forked = true;
          break;
        }
      }
      // ---- pivot k applied to column 0 (:16-36): b[row] = |b[row]| > 1e-16 ? b[row] / q : 0, and for every other row
      // with |coef| > 1e-16, b[r] -= coef * b[row] when column 0 is among the pivot row's non-zero cells
      {
        const double *colk = a.colraw + (size_t)k * a.Hp;
        const double braw = b[row];
        const bool nz0 = fabs(braw) > kTiny;
        const double p0 = nz0 ? __ddiv_rn(braw, a.q[k]) : 0.0;
        __syncwarp();
        for (int r = lane; r < H; r += 32) {
          if (r == row) {
            b[r] = p0;
          } else if (nz0) {
            const double coef = colk[r];
            if (fabs(coef) > kTiny) b[r] = __dsub_rn(b[r], __dmul_rn(coef, p0));
          }
        }
        __syncwarp();
      }
      if (phase == 1)
        p1++;
      else
        p2++;
      iter++;
      k++;
    }
    for (int r = lane; r < H; r += 32) a.rhs_out[(size_t)i * H + r] = b[r];
    if (forked) {
      if (lane == 0) {
        a.fork_step[i] = k;
        a.fork_resume[3 * i] = phase;
        a.fork_resume[3 * i + 1] = p1;
        a.fork_resume[3 * i + 2] = p2;
        a.fork_ids[atomicAdd(a.fork_count, 1)] = (int)i;
      }
    } else {
      if (lane == 0) {
        if (a.status) a.status[i] = status;
        if (a.value) a.value[i] = value;
        if (a.pivots) {
          a.pivots[2 * i] = p1;
          a.pivots[2 * i + 1] = p2;
        }
      }
      for (int p = lane; p < W + H; p += 32) {
        const int v = a.leader_var[p];
        if (a.var_out) a.var_out[(size_t)i * (W + H) + p] = v;
        if (a.pos_out) a.pos_out[(size_t)i * (W + H) + v] = p;
        if (a.red_out) a.red_out[(size_t)i * (W + H) + p] = a.leader_red[p];
      }
    }
    __syncwarp();
  }
}

// Forked replicas [first, first + m) of the fork list: private tableau = leader snapshot of the fork step with the
// replica's own column 0; variableAtPosition of that step; resume state.
__global__ void k_replica_materialise(int first, int m, int H, int W, const int *fork_ids, const int *fork_step,
                                      const long long *fork_resume, const double *rhs_state, const double *snap,
                                      const int *snap_var, double *work, int *var_in, long long *resume) {
  const size_t cells = (size_t)H * W;
  for (int f = blockIdx.y; f < m; f += gridDim.y) {
    const int i = fork_ids[first + f], k = fork_step[i];
    const double *src = snap + (size_t)k * cells;
    double *dst = work + (size_t)f * cells;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < cells; e += (size_t)gridDim.x * blockDim.x) {
      const int r = (int)(e / W), c = (int)(e - (size_t)r * W);
      dst[e] = c == 0 ? rhs_state[(size_t)i * H + r] : src[e];
    }
    if (blockIdx.x == 0) {
      for (int p = threadIdx.x; p < W + H; p += blockDim.x) var_in[(size_t)f * (W + H) + p] = snap_var[(size_t)k * (W + H) + p];
      if (threadIdx.x < 3) resume[3 * f + threadIdx.x] = fork_resume[3 * i + threadIdx.x];
    }
  }
}

// Results of the forked replicas [first, first + m) (compact, as solved) back to their replica slots.
__global__ void k_replica_scatter(int first, int m, int H, int W, const int *fork_ids, const int *c_status,
                                  const double *c_value, const long long *c_pivots, const double *c_rhs, const int *c_pos,
                                  const int *c_var, const double *c_red, int *status, double *value, long long *pivots,
                                  double *rhs_out, int *pos_out, int *var_out, double *red_out) {
  for (int f = blockIdx.x; f < m; f += gridDim.x) {
    const size_t i = (size_t)fork_ids[first + f];
    if (threadIdx.x == 0) {
      if (status) status[i] = c_status[f];
      if (value) value[i] = c_value[f];
      if (pivots) {
        pivots[2 * i] = c_pivots[2 * f];
        pivots[2 * i + 1] = c_pivots[2 * f + 1];
      }
    }
    for (int r = threadIdx.x; r < H; r += blockDim.x) rhs_out[i * H + r] = c_rhs[(size_t)f * H + r];
    for (int p = threadIdx.x; p < W + H; p += blockDim.x) {
      if (pos_out) pos_out[i * (W + H) + p] = c_pos[(size_t)f * (W + H) + p];
      if (var_out) var_out[i * (W + H) + p] = c_var[(size_t)f * (W + H) + p];
      if (red_out) red_out[i * (W + H) + p] = c_red[(size_t)f * (W + H) + p];
    }
  }
}

// Incumbent min-allreduce, the part inside one GPU: the logical ranks that share this GPU are reduced by ONE kernel
// over all their slots (never by launches that wait for one another); slot[k] then goes through ncclAllReduce(min)
// across the distinct GPUs and is broadcast back to the rank slots.
__global__ void k_incumbent_reduce(double *slots, int k) {
  double m = slots[0];
  for (int i = 1; i < k; i++) m = slots[i] < m ? slots[i] : m;
  slots[k] = m;
}
__global__ void k_incumbent_broadcast(double *slots, int k) {
  const double m = slots[k];
  for (int i = 0; i < k; i++) slots[i] = m;
}

// Sparse producer boundary (yalps_solve_sparse): the initial tableau arrives as (cell, value) pairs over a zeroed
// matrix -- what tableauModel (src/tableau.ts:88-134) writes into its zero-filled Float64Array, without the zeros.
__global__ void k_scatter_cells(long long nnz, const int *__restrict__ cell, const double *__restrict__ val, double *M) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x)
    M[cell[i]] = val[i];
}

// The reference's stores happen in order (a later duplicate of a cell wins, src/tableau.ts:100-117); the scatter above
// is unordered.  Duplicates with different bits are the only case where that shows: then some pair does not find its
// own value in the matrix, and the host repeats the call with the duplicates resolved.
__global__ void k_verify_cells(long long nnz, const int *__restrict__ cell, const double *__restrict__ val,
                               const double *__restrict__ M, int *mismatch) {
  bool bad = false;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x)
    bad |= __double_as_longlong(M[cell[i]]) != __double_as_longlong(val[i]);
  if (bad) *mismatch = 1;
}

// Non-zero count of a sample of one tableau (kernel-path policy: sparse batches go to the HBM/L2-resident kernel).
__global__ void k_sample_density(const double *m, long long cells, long long step, int *out /* [2]: seen, nz */) {
  int seen = 0, nz = 0;
  for (long long k = (long long)threadIdx.x * step; k < cells; k += (long long)blockDim.x * step) {
    seen++;
    nz += m[k] != 0.0;
  }
  atomicAdd(out, seen);
  atomicAdd(out + 1, nz);
}

// fastdiv.cuh against __ddiv_rn on hash-generated operand pairs; counts bit mismatches.
//   mode 0: random bit patterns (all exponents, NaN/inf included)   mode 1: tableau-like magnitudes
//   mode 2: special numerators (0, -0, inf, NaN, denormals, huge)     mode 3: exact quotients and small integers
//   mode 4: exponents near the denormal / overflow boundaries
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
  x += 0x9e3779b97f4a7c15ULL;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ULL;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebULL;
  return x ^ (x >> 31);
}

__global__ void k_probe_division(long long n, unsigned long long seed, int mode, unsigned long long *out /* [4] */) {
  unsigned long long bad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const unsigned long long a = splitmix64(seed + 2 * (unsigned long long)i), b = splitmix64(seed + 2 * (unsigned long long)i + 1);
    double x = __longlong_as_double((long long)a), y = __longlong_as_double((long long)b);
    if (mode == 1) {
      x = ((double)(a >> 11) / 9007199254740992.0 - 0.5) * (double)(1 + (a & 1023));
      y = ((double)(b >> 11) / 9007199254740992.0 - 0.5) * (double)(1 + (b & 255));
      if ((a & 0x7000) == 0) x = 0.0;
      if ((a & 0x7000) == 0x1000) x = -0.0;
    } else if (mode == 2) {
      const double sp[12] = {0.0, -0.0, d_inf(), -d_inf(), d_nan(), 4.9e-324, -4.9e-324, 2.2250738585072014e-308,
                             1.7976931348623157e308, -1.7976931348623157e308, 1e-16, 1.0};
      x = sp[a % 12];
      if ((b & 15) == 0) y = sp[(b >> 4) % 12];
    } else if (mode == 3) {
      const double k = (double)((long long)(a & 0xffff) - 32768);
      y = (double)((long long)(b & 0xfffff) - 524288) * 0.125;
      x = (a & 0x10000) ? __dmul_rn(k, y) : k;
    } else if (mode == 4) {
      const unsigned long long ex = (a & 1) ? (unsigned long long)(a >> 1 & 63) : (unsigned long long)(0x7fe - (a >> 1 & 63));
      const unsigned long long ey = (b & 1) ? (unsigned long long)(b >> 1 & 63) : (unsigned long long)(0x7fe - (b >> 1 & 63));
      x = __longlong_as_double((long long)((a & 0x800fffffffffffffULL) | (ex << 52)));
      y = __longlong_as_double((long long)((b & 0x800fffffffffffffULL) | (ey << 52)));
    }
    const Recip rc(y);
    const double q1 = rc.quot(x), q2 = rc.quot(y), q3 = div_rn(1.0, y);
    const double r1 = __ddiv_rn(x, y), r2 = __ddiv_rn(y, y), r3 = __ddiv_rn(1.0, y);
    // the branch-free batch form (K1t): accepted quotients must already be exact, rejected ones go out of line
    RecipBatch rb(y);
    double b1 = rb.quot(x), b2 = rb.quot(y), b3 = rb.quot(1.0);
    (void)rb.quot(__longlong_as_double((long long)(a ^ b)), false);  // an unused quotient must not change the verdict
    if (!rb.ok) {
      b1 = div_rn_slow(x, y);
      b2 = div_rn_slow(y, y);
      b3 = div_rn_slow(1.0, y);
    }
    if (__double_as_longlong(q1) != __double_as_longlong(r1) || __double_as_longlong(q2) != __double_as_longlong(r2) ||
        __double_as_longlong(q3) != __double_as_longlong(r3) || __double_as_longlong(b1) != __double_as_longlong(r1) ||
        __double_as_longlong(b2) != __double_as_longlong(r2) || __double_as_longlong(b3) != __double_as_longlong(r3)) {
      bad++;
      if (atomicAdd(out + 1, 1ULL) == 0) {
        out[2] = (unsigned long long)__double_as_longlong(x);
        out[3] = (unsigned long long)__double_as_longlong(y);
      }
    }
  }
  if (bad) atomicAdd(out, bad);
}

__global__ void k_round_to_precision(long long n, const double *x, double precision, double *out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = round_to_precision(x[i], precision);
}

// L2 stream: every thread reads and rewrites 16-byte cells of a buffer that fits L2, `iters` times over
// (the ld - mul - sub - st pattern of the rank-1 update on an L2-resident working copy).  bytes = words*8 * iters * 2.
__global__ void k_l2_stream(double2 *buf, size_t n2, int iters, double coef) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (int it = 0; it < iters; it++)
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n2; k += stride) {
      double2 x = __ldcg(buf + k);
      x.x = __dsub_rn(x.x, __dmul_rn(coef, 1e-9));
      x.y = __dsub_rn(x.y, __dmul_rn(coef, 2e-9));
      __stcg(buf + k, x);
    }
}

// Shared-memory stream: every thread reads and rewrites 8-byte cells of a CTA-private buffer.
// bytes = grid * iters * words * 16.
__global__ void k_smem_stream(int words, int iters, double *sink) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double *buf = reinterpret_cast<double *>(smem_raw);
  for (int k = threadIdx.x; k < words; k += blockDim.x) buf[k] = (double)k;
  __syncthreads();
  double acc = 0.0;
  for (int it = 0; it < iters; it++) {
#pragma unroll 4
    for (int k = threadIdx.x; k < words; k += blockDim.x) {
      const double x = buf[k];
      buf[k] = x + 1.0;
      acc += x;
    }
    __syncthreads();
  }
  if (acc == -1.0) sink[0] = acc;
}

}  // namespace yalps
