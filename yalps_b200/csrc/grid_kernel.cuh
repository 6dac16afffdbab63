// grid_kernel.cuh -- K4: ONE large LP spread over the whole GPU (cooperative persistent launch).
//
// Same algorithm and rounding sequence as simplex_device.cuh (src/simplex.ts:5-142), different work split:
//   * the tableau stays in HBM/L2 in the reference layout (row stride W, column 0 = RHS), updated in place;
//   * every CTA recomputes the pivot choice redundantly from the (L2-resident) objective row / RHS column /
//     pivot column, so all CTAs agree on (row, col) without exchanging partial results;
//   * every CTA keeps private shared-memory copies of the objective row and of the RHS column and applies the
//     same rank-1 update to them as the owners of those cells apply in HBM (same operands, same operations, so
//     the copies stay bit-identical): the first selection of every pivot reads shared memory only, and a pivot
//     costs two dependent trips to L2/HBM (pivot row, pivot column) instead of four or five;
//   * every CTA stages the normalised pivot row (and its non-zero flags) in its own shared memory;
//   * every CTA also stages the old pivot column (0 for rows the update must skip), so the update never waits on
//     a dependent global load and a row can be split between warps without a read/write hazard on its
//     pivot-column cell;
//   * the update is dealt to the warps of the whole grid as (row, 256-column segment) items, round-robin:
//     coalesced 8-byte accesses, 8 loads in flight per lane, skipped rows cost one shared-memory read;
//   * two grid barriers per pivot: one after every CTA has finished reading (pivot choice + staging of the old
//     pivot row) and one after the update, so that no CTA ever selects from a half-updated tableau.
#pragma once

#include "simplex_device.cuh"

namespace yalps {

// Grid-wide barrier for a cooperative launch (all CTAs co-resident): monotonically increasing arrival counter,
// release on arrival / acquire on the spin so that every CTA's tableau writes are visible to every other CTA.
__device__ __forceinline__ void grid_barrier(unsigned long long *counter, unsigned long long &epoch) {
  __syncthreads();
  epoch++;
  if (threadIdx.x == 0) {
    const unsigned long long goal = epoch * gridDim.x;
    __threadfence();
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(counter) : "memory");
    unsigned long long seen;
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(counter) : "memory");
    } while (seen < goal);
    __threadfence();
  }
  __syncthreads();
}

struct GridArgs {
  double *M;  // H x W, reference layout, updated in place
  int H, W;
  int *var;   // variableAtPosition[W+H] (global), maintained by CTA 0
  const int *init_var;  // node mode: root variableAtPosition (first init_n entries), identity beyond
  int init_n;
  int *pos_out;
  double *rhs_out;
  int *status;
  double *value;
  long long *pivots;
  double precision, max_pivots;
  int check_cycles;
  int *hist;
  int hist_cap;
  int *flags;                  // [2] cycle / history-overflow verdict of CTA 0, by iteration parity
  unsigned long long *barrier; // grid barrier arrival counter, zeroed before the launch
  unsigned long long *rows_out; // optional: rows rewritten by the updates are ADDED here (roofline diagnostics)
  double *red_out;  // optional reduced costs [W+H] (BatchArgs::red_out), from the CTAs' identical objective-row copies
};

constexpr int kGridThreads = 1024;
constexpr int kGridWarps = kGridThreads / 32;

// shared memory: prow[W], row0[W] (objective row copy), colbuf[H], bcol[H] (RHS column copy), nz bitmask, scratch
struct GridSmem {
  size_t off_prow, off_row0, off_col, off_b, off_nz, off_red, total;
  __host__ __device__ GridSmem(int H, int W) {
    size_t o = 0;
    off_prow = o;
    o += (size_t)((W + 1) & ~1) * 8;
    off_row0 = o;
    o += (size_t)((W + 1) & ~1) * 8;
    off_col = o;
    o += (size_t)((H + 1) & ~1) * 8;
    off_b = o;
    o += (size_t)((H + 1) & ~1) * 8;
    o = (o + 15) & ~(size_t)15;
    off_nz = o;
    o += (size_t)(((W + 31) / 32 + 8 + 7) & ~7) * 4;
    o = (o + 15) & ~(size_t)15;
    off_red = o;
    o += 192 * 4;
    total = (o + 15) & ~(size_t)15;
  }
};

constexpr int kSegCols = 256;  // columns per update item: 8 loads in flight per lane

__global__ void __launch_bounds__(kGridThreads, 1) k_simplex_grid(const GridArgs a) {
  constexpr int NT = kGridThreads, NW = kGridWarps;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long epoch = 0;
  const GridSmem L(a.H, a.W);
  double *prow = reinterpret_cast<double *>(smem_raw + L.off_prow);
  double *row0 = reinterpret_cast<double *>(smem_raw + L.off_row0);
  double *colbuf = reinterpret_cast<double *>(smem_raw + L.off_col);
  double *bcol = reinterpret_cast<double *>(smem_raw + L.off_b);
  unsigned *nzmask = reinterpret_cast<unsigned *>(smem_raw + L.off_nz);
  unsigned *red = reinterpret_cast<unsigned *>(smem_raw + L.off_red);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int H = a.H, W = a.W;
  double *__restrict__ M = a.M;
  const double precision = a.precision, INF = d_inf();
  const int gwarp = blockIdx.x * NW + warp, gwarps = gridDim.x * NW;

  for (int k = blockIdx.x * NT + tid; k < W + H; k += gridDim.x * NT)
    a.var[k] = (a.init_var && k < a.init_n) ? a.init_var[k] : k;
  for (int c = tid; c < W; c += NT) row0[c] = M[c];
  for (int r = tid; r < H; r += NT) bcol[r] = M[(size_t)r * W];
  grid_barrier(a.barrier, epoch);

  int status = ST_CYCLED;
  double value = d_nan();
  long long p1 = 0, p2 = 0, iter = 0;
  unsigned long long rows_mine = 0;
  int phase = 1, parity = 0, hist_len = 0;
  // this thread's candidates for the next first selection, collected by the fused stage of the previous pivot
  bool have_carry = false;
  double carry_cv = -INF, carry_rv = INF;
  int carry_ci = kNone, carry_ri = kNone;

  for (;;) {
    if (!((double)iter < a.max_pivots)) break;
    int row, col;
    if (phase == 1) {
      // leaving row from the private RHS copy (:111-119)
      double bv = INF;
      int bi = kNone;
      if (have_carry) {  // collected while the previous pivot was applied to the private RHS copy
        bv = carry_rv;
        bi = carry_ri;
      } else {
        for (int r = 1 + tid; r < H; r += NT) {
          const double v = bcol[r];
          if (v < -precision && v < bv) {
            bv = v;
            bi = r;
          }
        }
      }
      row = block_best<false, NW>(bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity);
      if (row == kNone) {
        phase = 2;
        iter = 0;
        hist_len = 0;
        continue;
      }
      // trip 1: the pivot row (raw) into shared memory, entering column from it and the private objective row
      bv = -INF;
      bi = kNone;
      for (int c = tid; c < W; c += NT) {
        const double coef = M[(size_t)row * W + c];
        prow[c] = coef;
        if (c >= 1 && coef < -precision) {
          const double ratio = __ddiv_rn(-row0[c], coef);
          if (ratio > bv) {
            bv = ratio;
            bi = c;
          }
        }
      }
      col = block_best<true, NW>(bi == kNone ? no_key<true>() : order_key(bv), bi, red, parity);
      if (col == kNone) {
        status = ST_INFEASIBLE;
        break;
      }
      // trip 2: the pivot column (raw)
      for (int r = tid; r < H; r += NT) colbuf[r] = M[(size_t)r * W + col];
    } else {
      // entering column from the private objective row (:71-79)
      double bv = -INF;
      int bi = kNone;
      if (have_carry) {  // collected while the previous pivot was applied to the private objective row
        bv = carry_cv;
        bi = carry_ci;
      } else {
        for (int c = 1 + tid; c < W; c += NT) {
          const double v = row0[c];
          if (v > precision && v > bv) {
            bv = v;
            bi = c;
          }
        }
      }
      col = block_best<true, NW>(bi == kNone ? no_key<true>() : order_key(bv), bi, red, parity);
      if (col == kNone) {
        status = ST_OPTIMAL;
        value = round_to_precision(row0[0], precision);
        break;
      }
      // trip 1: the pivot column (raw) into shared memory, ratio test against the private RHS copy (:83-95)
      bv = INF;
      bi = kNone;
      for (int r = tid; r < H; r += NT) {
        const double v = M[(size_t)r * W + col];
        colbuf[r] = v;
        if (r >= 1 && v > precision) {
          const double ratio = __ddiv_rn(bcol[r], v);
          if (ratio < INF) {
            const double key = (ratio <= precision) ? -INF : ratio;
            if (bi == kNone || key < bv) {
              bv = key;
              bi = r;
            }
          }
        }
      }
      row = block_best<false, NW>(bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity);
      if (row == kNone) {
        status = ST_UNBOUNDED;
        value = (double)col;
        break;
      }
      // trip 2: the pivot row (raw)
      for (int c = tid; c < W; c += NT) prow[c] = M[(size_t)row * W + c];
    }
    __syncthreads();  // raw pivot row and column are complete in shared memory

    if (a.check_cycles) {  // CTA 0 keeps the history; its verdict reaches the other CTAs through a grid barrier
      if (blockIdx.x == 0) {
        int verdict = 0;
        if (hist_len >= a.hist_cap) {
          verdict = 2;
        } else {
          if (tid == 0) {
            a.hist[2 * hist_len] = a.var[W + row];
            a.hist[2 * hist_len + 1] = a.var[col];
          }
          __syncthreads();
          if (history_has_cycle<NT>(a.hist, hist_len + 1)) verdict = 1;
        }
        if (tid == 0) a.flags[iter & 1] = verdict;
        __threadfence();
      }
      hist_len++;
      grid_barrier(a.barrier, epoch);
      const int verdict = *reinterpret_cast<volatile int *>(a.flags + (iter & 1));
      if (verdict == 2) status = ST_ERR_HISTORY;
      if (verdict) break;
    }

    // ---- ONE fused stage over the staged pivot row and column (every cell is handled by exactly one thread, so no
    // barrier is needed between its parts): normalise the row in place (src/simplex.ts:16-25) and collect its non-zero
    // flags; apply the pivot to the private objective-row copy; reduce the pivot column to "0 = row left alone"
    // (:29,:31); apply the pivot to the private RHS copy; and carry this thread's candidates for the NEXT pivot's
    // first selection (largest reduced cost above precision / most negative RHS), which saves that scan.
    const double q = prow[col];
    const double coef0 = colbuf[0];  // objective-row cell of the pivot column, before colbuf is rewritten
    const double braw = prow[0];     // RHS cell of the pivot row (column 0 is never the pivot column)
    __syncthreads();
    {
      const bool act0 = fabs(coef0) > kTiny;  // row 0 is never the pivot row
      const bool nz0 = fabs(braw) > kTiny;
      const double p0 = nz0 ? __ddiv_rn(braw, q) : 0.0;  // every thread for itself: the same division, the same bits
      carry_cv = -INF;
      carry_ci = kNone;
      for (int cbase = warp * 32; cbase < W; cbase += NT) {
        const int c = cbase + lane;
        bool nz = false;
        if (c < W) {
          const double v = (c == col) ? 1.0 : prow[c];
          nz = fabs(v) > kTiny;
          const double pn = nz ? __ddiv_rn(v, q) : 0.0;
          prow[c] = pn;
          if (c == col) nz = false;  // the pivot column gets -coef/q instead (:36)
          double o = row0[c];
          if (act0) {
            if (nz)
              o = __dsub_rn(o, __dmul_rn(coef0, pn));
            else if (c == col)
              o = __ddiv_rn(-coef0, q);
            row0[c] = o;
          }
          if (c == 0) bcol[0] = o;  // the corner cell belongs to both copies
          if (c >= 1 && o > precision && o > carry_cv) {  // (:71-79), ascending c per thread: strict > keeps the first
            carry_cv = o;
            carry_ci = c;
          }
        }
        const unsigned m = __ballot_sync(0xffffffffu, nz);
        if (lane == 0) nzmask[cbase >> 5] = m;
      }
      carry_rv = INF;
      carry_ri = kNone;
      for (int r = tid; r < H; r += NT) {
        const double coef = colbuf[r];
        const bool on = r != row && fabs(coef) > kTiny;
        colbuf[r] = on ? coef : 0.0;
        rows_mine += on;  // every CTA builds the whole column: CTA 0 reports the count
        if (r >= 1) {
          double bnew = bcol[r];
          if (r == row) {
            bnew = p0;
            bcol[r] = bnew;
          } else if (on && nz0) {
            bnew = __dsub_rn(bnew, __dmul_rn(coef, p0));
            bcol[r] = bnew;
          }
          if (bnew < -precision && bnew < carry_rv) {  // (:111-119)
            carry_rv = bnew;
            carry_ri = r;
          }
        }
      }
      have_carry = true;
    }
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) {  // basis bookkeeping (:7-12)
      const int leaving = a.var[W + row];
      a.var[W + row] = a.var[col];
      a.var[col] = leaving;
    }
    grid_barrier(a.barrier, epoch);  // every CTA has made its choice and staged the old pivot row: the tableau may change now

    // ---- rank-1 update (:28-38): (row, column segment) items dealt round-robin to the warps of the grid.
    // Item decomposition is incremental 32-bit arithmetic; a full segment runs without bounds checks, with the
    // eight non-zero flags of the lane gathered from two 16-byte shared-memory loads.
    {
      const int nseg = (W + kSegCols - 1) / kSegCols;
      const int step_r = gwarps / nseg, step_s = gwarps - step_r * nseg;
      int r = gwarp / nseg, seg = gwarp - r * nseg;
      while (r < H) {
        const int c0 = seg * kSegCols + lane;
        double *__restrict__ Mr = M + (size_t)r * W + c0;
        const double coef = colbuf[r];
        const bool full_seg = (seg + 1) * kSegCols <= W;
        if (r == row) {
#pragma unroll
          for (int u = 0; u < 8; u++)
            if (full_seg || c0 + 32 * u < W) Mr[32 * u] = prow[c0 + 32 * u];
        } else if (coef != 0.0) {  // else: row skip (:31)
          // nz flags of my 8 columns: words seg*8 .. seg*8+7 (the mask array is padded to a multiple of 8 words)
          const uint4 w0 = *reinterpret_cast<const uint4 *>(nzmask + seg * 8);
          const uint4 w1 = *reinterpret_cast<const uint4 *>(nzmask + seg * 8 + 4);
          const unsigned bits = ((w0.x >> lane) & 1u) | (((w0.y >> lane) & 1u) << 1) | (((w0.z >> lane) & 1u) << 2) |
                                (((w0.w >> lane) & 1u) << 3) | (((w1.x >> lane) & 1u) << 4) |
                                (((w1.y >> lane) & 1u) << 5) | (((w1.z >> lane) & 1u) << 6) |
                                (((w1.w >> lane) & 1u) << 7);
          double x[8];
          if (full_seg) {
#pragma unroll
            for (int u = 0; u < 8; u++) x[u] = Mr[32 * u];
#pragma unroll
            for (int u = 0; u < 8; u++)
              if ((bits >> u) & 1u) Mr[32 * u] = __dsub_rn(x[u], __dmul_rn(coef, prow[c0 + 32 * u]));
          } else {
#pragma unroll
            for (int u = 0; u < 8; u++)
              if (c0 + 32 * u < W) x[u] = Mr[32 * u];
#pragma unroll
            for (int u = 0; u < 8; u++)
              if (c0 + 32 * u < W && ((bits >> u) & 1u)) Mr[32 * u] = __dsub_rn(x[u], __dmul_rn(coef, prow[c0 + 32 * u]));
          }
          // the pivot-column cell of this row (:36), by the lane that owns it
          if (col >= seg * kSegCols && col < (seg + 1) * kSegCols && ((col - lane) & 31) == 0)
            M[(size_t)r * W + col] = __ddiv_rn(-coef, q);
        }
        r += step_r;
        seg += step_s;
        if (seg >= nseg) {
          seg -= nseg;
          r++;
        }
      }
    }
    grid_barrier(a.barrier, epoch);

    if (phase == 1)
      p1++;
    else
      p2++;
    iter++;
  }

  // ---- outputs (all CTAs leave the loop in the same iteration with the same verdict)
  if (blockIdx.x == 0 && tid == 0) {
    if (a.status) a.status[0] = status;
    if (a.value) a.value[0] = value;
    if (a.pivots) {
      a.pivots[0] = p1;
      a.pivots[1] = p2;
    }
  }
  if (a.rows_out && blockIdx.x == 0 && rows_mine != 0) atomicAdd(a.rows_out, rows_mine);
  if (a.rhs_out)
    for (int r = blockIdx.x * NT + tid; r < H; r += gridDim.x * NT) a.rhs_out[r] = M[(size_t)r * W];
  if (a.pos_out)
    for (int k = blockIdx.x * NT + tid; k < W + H; k += gridDim.x * NT) a.pos_out[a.var[k]] = k;
  if (a.red_out)
    for (int k = blockIdx.x * NT + tid; k < W + H; k += gridDim.x * NT) a.red_out[a.var[k]] = (k >= 1 && k < W) ? row0[k] : 0.0;
}

}  // namespace yalps
