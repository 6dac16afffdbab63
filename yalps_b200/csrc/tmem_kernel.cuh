// tmem_kernel.cuh -- K1t: one small LP per warp with the tableau resident in TENSOR MEMORY.
//
// K1 (kernels.cuh) keeps a tableau in shared memory and is bound by the shared-memory data pipe: every cell goes
// through it twice per pivot (128 B/clk/SM).  Blackwell's tensor memory (256 KB per SM, 128 lanes x 512 32-bit
// columns) is normally the accumulator store of tcgen05.mma, but `tcgen05.ld/st.32x32b` make it a lane-private
// scratchpad: lane i of warp w reads/writes TMEM lane 32*(w%4)+i.  scripts/micro/tmem_stream.cu measures 800 GB/s
// per SM (read + write) for the ld - mul - sub - st pattern of the rank-1 update against 243 GB/s through shared
// memory, so the simplex pivot (src/simplex.ts:5-39) of a tableau whose columns are OWNED by lanes never has to
// touch shared memory for the tableau body:
//
//   * lane l owns the coefficient columns 2l+1, 2l+2 (two fp64 = four 32-bit TMEM columns per row).  Rows 1..H-1
//     live in TMEM in blocks of eight rows = 32 TMEM columns, element-major inside a block:
//         row r, k = r-1:  my first cell  at columns 32*(k/8)      + 2*(k%8), +1
//                          my second cell at columns 32*(k/8) + 16 + 2*(k%8), +1
//     so that ONE tcgen05.ld/st.x32 moves a block for the rank-1 update and ONE tcgen05.ld.x16 reads one tableau
//     column of eight rows (the entering column, below);
//   * row 0 (objective row) lives in registers (two cells per lane), the RHS column in registers (lane l owns row
//     l+1), M[0,0] redundantly in every lane;
//   * only the pivot column crosses lanes, through shared memory: after the entering column is chosen its owner
//     lane reads its cells of all rows (four tcgen05.ld.x16) and stores them (colx), every lane reads back "its"
//     row; the new pivot-column cells (-coef/q, lane-distributed after the division) return to their owner lane
//     as {coef, -coef/q} broadcast loads in the row pass.
//
// A CTA is four warps = the four lane quarters of a 128-column allocation; each warp solves its own LPs (no CTA
// barrier in the loop) and four CTAs share an SM: 16 LPs per SM in flight (tableaus of 34..65 rows: 256-column
// allocations, two RHS cells per lane, 8 LPs per SM -- template parameter HR).  Limits: H <= 65, W <= 65, no
// checkCycles, no node mode.  Same selection rules, skip rules and rounding sequence as simplex_device.cuh, and
// bit-identical results (tests/test_gpu_simplex.py).
#pragma once

#include "kernels.cuh"

namespace yalps {

// Template parameter HR = RHS cells per lane: HR = 1 holds tableaus of up to 33 rows (128 TMEM columns per CTA, four
// CTAs = 16 LPs per SM), HR = 2 up to 65 rows (256 columns per CTA, two CTAs = 8 LPs per SM; lane l owns the RHS
// cells of rows l+1 and l+33).
constexpr int kTmemMaxCols = 65;   // 64 coefficient columns = 32 lanes x 2
constexpr int kTmemWarps = 4;
template <int HR>
struct TmemShape {
  static constexpr int kMaxRows = 32 * HR + 1;   // rows 1..32*HR <-> (lane, slot) for the RHS column
  static constexpr int kColumns = 128 * HR;      // TMEM columns per CTA (power of two): 4 columns per row
  static constexpr int kCtasPerSm = 512 / kColumns;
  static_assert(HR == 1 || HR == 2, "supported shapes");
};
constexpr int kTmemMaxRows = TmemShape<2>::kMaxRows;  // tallest tableau of any shape
constexpr int kTmemColumns = TmemShape<1>::kColumns;  // (k_tmem_stream uses the HR = 1 shape)
constexpr int kTmemCtasPerSm = TmemShape<1>::kCtasPerSm;

// shared memory per warp
template <int HR>
struct TmemWarpSmem {
  double2 cb[TmemShape<HR>::kMaxRows + 7];  // [r] = {pivot-column coefficient or 0 (row left alone), new pivot-column cell}
  double colx_store[TmemShape<HR>::kMaxRows + 9];  // colx = colx_store + 1: entering column M[r, col]; &colx[1] is 16-byte aligned
  int var[kTmemMaxCols + TmemShape<HR>::kMaxRows + 2];
};

// ---- tcgen05 wrappers ---------------------------------------------------------------------------------------
// (the consumers of a tcgen05.ld go through tm_wait_ld*, which takes the registers as operands so that no use of
// them can be scheduled in front of the wait)
__device__ __forceinline__ void tm_ld2(unsigned taddr, unsigned &a, unsigned &b) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "r"(taddr));
}
__device__ __forceinline__ void tm_st2(unsigned taddr, unsigned a, unsigned b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_wait_ld4(unsigned &a, unsigned &b, unsigned &c, unsigned &d) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(a), "+r"(b), "+r"(c), "+r"(d)::"memory");
}
__device__ __forceinline__ void tm_ld16(unsigned taddr, unsigned *v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tm_ld32(unsigned taddr, unsigned (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tm_st32(unsigned taddr, const unsigned (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
template <int N>
__device__ __forceinline__ void tm_wait_ld(unsigned (&v)[N]) {
  static_assert(N % 8 == 0, "whole groups of eight registers");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; i += 8)
    asm volatile("" : "+r"(v[i]), "+r"(v[i + 1]), "+r"(v[i + 2]), "+r"(v[i + 3]), "+r"(v[i + 4]), "+r"(v[i + 5]),
                      "+r"(v[i + 6]), "+r"(v[i + 7])::"memory");
}

// first TMEM column (relative to the warp's base) of cell e (0/1) of row r >= 1
__device__ __forceinline__ unsigned tm_cell(int r, int e) {
  const unsigned k = (unsigned)(r - 1);
  return 32u * (k >> 3) + 16u * (unsigned)e + 2u * (k & 7u);
}
__device__ __forceinline__ void tm_load_row(unsigned tbase, int r, double &x0, double &x1) {
  unsigned a, b, c, d;
  tm_ld2(tbase + tm_cell(r, 0), a, b);
  tm_ld2(tbase + tm_cell(r, 1), c, d);
  tm_wait_ld4(a, b, c, d);
  x0 = __hiloint2double((int)b, (int)a);
  x1 = __hiloint2double((int)d, (int)c);
}
__device__ __forceinline__ void tm_store_row(unsigned tbase, int r, double x0, double x1) {
  tm_st2(tbase + tm_cell(r, 0), (unsigned)__double2loint(x0), (unsigned)__double2hiint(x0));
  tm_st2(tbase + tm_cell(r, 1), (unsigned)__double2loint(x1), (unsigned)__double2hiint(x1));
}

// Per-pivot lane state of the rank-1 pass.
struct TmemPivot {
  double pn0, pn1;   // normalised pivot-row cells of my two columns (0.0 where the old cell was flushed)
  bool st0, st1;     // the rank-1 pass rewrites my first / second cell
  bool own0, own1;   // my first / second column is the pivot column: its cells become cb[r].y
};

// Eight rows r0..r0+7 (one TMEM block) of the rank-1 update.  cc[i] = {coef, cn}: coef == 0 leaves the row alone
// (:31); cn is the new value of the row's pivot-column cell (the old one for rows that are left alone).
// Fast form: every lane rewrites both cells of every row (dense pivot row, eight active rows), EC = which of my
// two columns can be the pivot column.
template <int EC>
__device__ __forceinline__ void tmem_block_fast(unsigned tblk, const double2 *cbr, const TmemPivot &p) {
  unsigned v[32];
  tm_ld32(tblk, v);
  double2 cc[8];
#pragma unroll
  for (int i = 0; i < 8; i++) cc[i] = cbr[i];
  tm_wait_ld(v);
  const bool own = EC ? p.own1 : p.own0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    double x0 = __hiloint2double((int)v[2 * i + 1], (int)v[2 * i]), x1 = __hiloint2double((int)v[16 + 2 * i + 1], (int)v[16 + 2 * i]);
    x0 = __dsub_rn(x0, __dmul_rn(cc[i].x, p.pn0));
    x1 = __dsub_rn(x1, __dmul_rn(cc[i].x, p.pn1));
    if (EC == 0 && own) x0 = cc[i].y;
    if (EC == 1 && own) x1 = cc[i].y;
    v[2 * i] = (unsigned)__double2loint(x0);
    v[2 * i + 1] = (unsigned)__double2hiint(x0);
    v[16 + 2 * i] = (unsigned)__double2loint(x1);
    v[16 + 2 * i + 1] = (unsigned)__double2hiint(x1);
  }
  tm_st32(tblk, v);
}

// General form: per-cell predicates, rows with coef == 0 untouched.  Flat predicates (row active AND cell rewritten)
// instead of a branch per row: the block stays one straight-line sequence.
template <int EC>
__device__ __forceinline__ void tmem_block_general(unsigned tblk, const double2 *cbr, const TmemPivot &p) {
  unsigned v[32];
  tm_ld32(tblk, v);
  double2 cc[8];
#pragma unroll
  for (int i = 0; i < 8; i++) cc[i] = cbr[i];
  tm_wait_ld(v);
  const bool own = EC ? p.own1 : p.own0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    double x0 = __hiloint2double((int)v[2 * i + 1], (int)v[2 * i]), x1 = __hiloint2double((int)v[16 + 2 * i + 1], (int)v[16 + 2 * i]);
    const bool on = cc[i].x != 0.0;
    const bool a0 = on && p.st0, a1 = on && p.st1;
    const double t0 = __dsub_rn(x0, __dmul_rn(cc[i].x, p.pn0)), t1 = __dsub_rn(x1, __dmul_rn(cc[i].x, p.pn1));
    x0 = a0 ? t0 : x0;  // (selects, not branches: the arithmetic of an untouched cell is computed and dropped)
    x1 = a1 ? t1 : x1;
    if (EC == 0 && own) x0 = cc[i].y;
    if (EC == 1 && own) x1 = cc[i].y;
    v[2 * i] = (unsigned)__double2loint(x0);
    v[2 * i + 1] = (unsigned)__double2hiint(x0);
    v[16 + 2 * i] = (unsigned)__double2loint(x1);
    v[16 + 2 * i + 1] = (unsigned)__double2hiint(x1);
  }
  tm_st32(tblk, v);
}

// Sparse pivot column: only the rows with a non-zero coefficient are touched (bit l of `mask` <-> row first_row + l),
// four rows per TMEM round trip -- the one-warp counterpart of the row-split kernels' active-row compaction.
__device__ __forceinline__ void tmem_rows_sparse(unsigned tbase, unsigned mask, int first_row, const double2 *cb,
                                                 const TmemPivot &p) {
  while (mask) {
    int r[4];
    unsigned v[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      r[i] = -1;
      if (mask) {
        r[i] = first_row + __ffs((int)mask) - 1;
        mask &= mask - 1;
      }
#pragma unroll
      for (int k = 0; k < 4; k++) v[i][k] = 0u;
    }
#pragma unroll
    for (int i = 0; i < 4; i++)
      if (r[i] >= 0) {  // (warp-uniform)
        tm_ld2(tbase + tm_cell(r[i], 0), v[i][0], v[i][1]);
        tm_ld2(tbase + tm_cell(r[i], 1), v[i][2], v[i][3]);
      }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 4; i++) asm volatile("" : "+r"(v[i][0]), "+r"(v[i][1]), "+r"(v[i][2]), "+r"(v[i][3])::"memory");
#pragma unroll
    for (int i = 0; i < 4; i++)
      if (r[i] >= 0) {
        const double2 cc = cb[r[i]];
        double x0 = __hiloint2double((int)v[i][1], (int)v[i][0]), x1 = __hiloint2double((int)v[i][3], (int)v[i][2]);
        if (p.st0) x0 = __dsub_rn(x0, __dmul_rn(cc.x, p.pn0));
        if (p.st1) x1 = __dsub_rn(x1, __dmul_rn(cc.x, p.pn1));
        if (p.own0) x0 = cc.y;
        if (p.own1) x1 = cc.y;
        tm_st2(tbase + tm_cell(r[i], 0), (unsigned)__double2loint(x0), (unsigned)__double2hiint(x0));
        tm_st2(tbase + tm_cell(r[i], 1), (unsigned)__double2loint(x1), (unsigned)__double2hiint(x1));
      }
  }
}

// kCount: a second instantiation that also counts the rows every pivot rewrites (roofline diagnostics, launched only
// when a row counter is set); the production instantiation carries no trace of it.
// kCycles: the instantiation with the checkCycles history (src/simplex.ts:44-63: one buffer of (leaving, entering)
// variable pairs per warp in HBM, tested after every push by the 32 lanes); launched only for checkCycles: true.
template <int HR, bool kCount = false, bool kCycles = false>
__global__ void __launch_bounds__(kTmemWarps * 32, TmemShape<HR>::kCtasPerSm) k_simplex_tmem(const BatchArgs a) {
  using S = TmemShape<HR>;
  __shared__ __align__(16) TmemWarpSmem<HR> s_warp[kTmemWarps];
  __shared__ unsigned s_tmem_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double precision = a.precision, INF = d_inf();

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (unsigned)__cvta_generic_to_shared(&s_tmem_base)),
                 "n"(S::kColumns)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const unsigned tbase = s_tmem_base + ((unsigned)(warp & 3) * 32u << 16);  // this warp's lane quarter

  double2 *cb = s_warp[warp].cb;
  double *colx = s_warp[warp].colx_store + 1;
  int *var = s_warp[warp].var;
  const long long nwarps = (long long)gridDim.x * kTmemWarps;
  // per-phase pivot budget as an integer: (double)iter < maxPivots  <=>  iter < ceil(maxPivots)  (:69,:109)
  long long budget = 0;
  if (a.max_pivots > 0.0) budget = a.max_pivots >= 9.0e18 ? 0x7fffffffffffffffLL : (long long)ceil(a.max_pivots);

  // static assignment (few LPs): LP i -> CTA i % grid, warp i / grid, so that a small batch spreads over the SMs
  // (reading the queue one LP ahead, to prefetch the next tableau into L2 while the current one is solved, was measured
  // 3.5 % SLOWER: the last LPs sit reserved by busy warps while others idle)
  for (long long static_lp = (long long)warp * gridDim.x + blockIdx.x;; static_lp += nwarps) {
    long long lp = static_lp;
    if (a.counter) {
      unsigned long long got = 0;
      if (lane == 0) got = atomicAdd(a.counter, 1ULL);
      lp = (long long)__shfl_sync(0xffffffffu, got, 0);
    }
    if (lp >= a.n) break;
    if (a.index) lp = a.index[lp];
    int H, W;
    size_t moff, roff, poff;
    if (a.heights) {
      H = a.heights[lp];
      W = a.widths[lp];
      moff = (size_t)a.mat_off[lp];
      roff = (size_t)a.rhs_off[lp];
      poff = (size_t)a.pos_off[lp];
    } else {
      H = a.H;
      W = a.W;
      moff = (size_t)lp * H * W;
      roff = (size_t)lp * H;
      poff = (size_t)lp * (W + H);
    }
    const int Wm1 = W - 1;
    const int j0 = 2 * lane;
    const bool v0 = j0 < Wm1, v1 = j0 + 1 < Wm1;  // my two columns exist
    bool has_b[HR];                                // I own the RHS cell of row lane+1+32h
#pragma unroll
    for (int h = 0; h < HR; h++) has_b[h] = lane + 1 + 32 * h < H;
    const int nblocks = (H - 1 + 7) >> 3;          // TMEM blocks of eight rows

    // ---- load: global -> registers -> TMEM (16 bytes per lane per row, 8 rows in flight)
    const double *src = a.in + moff;
    double o0 = v0 ? src[1 + j0] : 0.0, o1 = v1 ? src[2 + j0] : 0.0;
    double bv[HR];
#pragma unroll
    for (int h = 0; h < HR; h++) bv[h] = has_b[h] ? src[(size_t)(lane + 1 + 32 * h) * W] : 0.0;
    double b0 = src[0];
    for (int blk = 0; blk < nblocks; blk += 2) {  // two blocks (32 loads per lane) in flight; a block past H-1 gets zeros
      double x[2][8][2];
#pragma unroll
      for (int b = 0; b < 2; b++) {
        const int r0 = 1 + 8 * (blk + b);
        const double *rp = src + (size_t)r0 * W + 1 + j0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
          x[b][i][0] = (r0 + i < H && v0) ? rp[0] : 0.0;
          x[b][i][1] = (r0 + i < H && v1) ? rp[1] : 0.0;
          rp += W;
        }
      }
#pragma unroll
      for (int b = 0; b < 2; b++) {
        unsigned v[32];
#pragma unroll
        for (int i = 0; i < 8; i++) {
          v[2 * i] = (unsigned)__double2loint(x[b][i][0]);
          v[2 * i + 1] = (unsigned)__double2hiint(x[b][i][0]);
          v[16 + 2 * i] = (unsigned)__double2loint(x[b][i][1]);
          v[16 + 2 * i + 1] = (unsigned)__double2hiint(x[b][i][1]);
        }
        tm_st32(tbase + 32u * (unsigned)(blk + b), v);
      }
    }
    for (int k = lane; k < W + H; k += 32) var[k] = a.var_in ? a.var_in[poff + k] : k;
    // rows past H-1 in the last block of eight: zeros in TMEM, never read; a non-zero coefficient keeps the block on
    // the straight-line path
    for (int k = H + lane; k < S::kMaxRows + 7; k += 32) cb[k] = make_double2(1.0, 0.0);
    tm_wait_st();
    __syncwarp();

    int status = ST_CYCLED;
    double value = d_nan();
    unsigned long long rows_rewritten = 0;
    long long p1 = 0, iter = 0;
    int phase = 1;
    int hist_len = 0;
    int *hist = kCycles ? a.hist + ((size_t)blockIdx.x * kTmemWarps + warp) * 2 * (size_t)a.hist_cap : nullptr;

    // read-only pass: cells of column c in rows 0..H-1 -> colx (its owner lane reads them, one tcgen05.ld per block)
    auto extract_column = [&](int c) {
      const int l = (c - 1) >> 1, e = (c - 1) & 1;
      if (lane == l) colx[0] = e ? o1 : o0;
      tm_wait_st();  // the pivot-row store of the previous pivot
      for (int blk = 0; blk < nblocks; blk += 2) {  // (blocks past H-1 are allocated, zero and never read)
        unsigned u[32];
#pragma unroll
        for (int b = 0; b < 2; b++) tm_ld16(tbase + 32u * (unsigned)(blk + b) + 16u * (unsigned)e, u + 16 * b);
        tm_wait_ld(u);
        if (lane == l) {
          uint4 *dst = reinterpret_cast<uint4 *>(colx + 1 + 8 * blk);
#pragma unroll
          for (int i = 0; i < 8; i++) dst[i] = make_uint4(u[4 * i], u[4 * i + 1], u[4 * i + 2], u[4 * i + 3]);
        }
      }
      __syncwarp();
    };

    for (;;) {
      if (iter >= budget) break;  // per-phase budget exhausted -> "cycled" (:102,:141)
      int row, col;
      double pr0, pr1;   // old pivot row cells of my two columns
      double cmine[HR];  // pivot-column cells of my RHS rows
      double rcp_q;      // refined reciprocal of the pivot element: the selection's own division already computed it in one lane
      if (phase == 1) {
        // leaving row: first index of the most negative RHS below -precision (:111-119)
        {
          double best = INF;
          int bi = kNone;
#pragma unroll
          for (int h = 0; h < HR; h++)
            if (has_b[h] && bv[h] < -precision && bv[h] < best) {  // ascending rows: strict < keeps the first
              best = bv[h];
              bi = lane + 1 + 32 * h;
            }
          const unsigned long long key = bi == kNone ? no_key<false>() : order_key(best);
          row = warp_best<false>((unsigned)(key >> 32), (unsigned)key, bi).idx;
        }
        if (row == kNone) {  // feasible: phase 2 with a fresh counter (:120, :67-69)
          phase = 2;
          hist_len = 0;  // a fresh history per phase (:67-69)
          p1 = iter;
          iter = 0;
          continue;
        }
        // entering column: first index of max -M[0,c]/M[row,c] over M[row,c] < -precision (:123-134)
        tm_wait_st();  // the pivot-row store of the previous pivot
        tm_load_row(tbase, row, pr0, pr1);
        double best = -INF;
        int bi = kNone;
        double rcp0, rcp1;
        {
          const bool c0 = v0 && pr0 < -precision, c1 = v1 && pr1 < -precision;
          RecipBatch d0(pr0, c0), d1(pr1, c1);
          rcp0 = d0.r;
          rcp1 = d1.r;
          double ratio0 = d0.quot(-o0, c0), ratio1 = d1.quot(-o1, c1);
          if (!(d0.ok && d1.ok)) {  // rare: exact division out of line
            ratio0 = div_rn_slow(-o0, pr0);
            ratio1 = div_rn_slow(-o1, pr1);
          }
          if (c0 && ratio0 > best) {  // best starts at -inf: -inf and NaN ratios never win, as in the reference
            best = ratio0;
            bi = j0 + 1;
          }
          if (c1 && ratio1 > best) {
            best = ratio1;
            bi = j0 + 2;
          }
        }
        const unsigned long long key = bi == kNone ? no_key<true>() : order_key(best);
        col = warp_best<true>((unsigned)(key >> 32), (unsigned)key, bi).idx;
        if (col == kNone) {
          status = ST_INFEASIBLE;
          break;
        }
        rcp_q = __shfl_sync(0xffffffffu, ((col - 1) & 1) ? rcp1 : rcp0, (col - 1) >> 1);  // q = M[row, col]: that lane's divisor
        extract_column(col);
#pragma unroll
        for (int h = 0; h < HR; h++) cmine[h] = has_b[h] ? colx[lane + 1 + 32 * h] : 0.0;
      } else {
        // entering column: first index of the largest reduced cost above precision (:71-79)
        {
          double best = -INF;
          int bi = kNone;
          if (v0 && o0 > precision) {
            best = o0;
            bi = j0 + 1;
          }
          if (v1 && o1 > precision && o1 > best) {
            best = o1;
            bi = j0 + 2;
          }
          const unsigned long long key = bi == kNone ? no_key<true>() : order_key(best);
          col = warp_best<true>((unsigned)(key >> 32), (unsigned)key, bi).idx;
        }
        if (col == kNone) {
          status = ST_OPTIMAL;
          value = round_to_precision(b0, precision);
          break;
        }
        extract_column(col);
#pragma unroll
        for (int h = 0; h < HR; h++) cmine[h] = has_b[h] ? colx[lane + 1 + 32 * h] : 0.0;
        // leaving row: ratio test with the reference's early break (:83-95) == lowest r whose ratio is <= precision
        // if any, else first index of the minimum ratio
        {
          double keyv = INF;
          int bi = kNone;
          double rcp[HR];
#pragma unroll
          for (int h = 0; h < HR; h++) {
            bool cand = has_b[h] && cmine[h] > precision;
            RecipBatch dr(cmine[h], cand);
            rcp[h] = dr.r;
            double ratio = dr.quot(bv[h], cand);
            if (!dr.ok) ratio = div_rn_slow(bv[h], cmine[h]);  // rare (e.g. a zero RHS): exact division out of line
            cand = cand && ratio < INF;                        // +inf and NaN never win
            const double k = (ratio <= precision) ? -INF : ratio;
            if (cand && (bi == kNone || k < keyv)) {  // ascending rows: strict < keeps the first
              keyv = k;
              bi = lane + 1 + 32 * h;
            }
          }
          const unsigned long long key = bi == kNone ? no_key<false>() : order_key(keyv);
          row = warp_best<false>((unsigned)(key >> 32), (unsigned)key, bi).idx;
          rcp_q = __shfl_sync(0xffffffffu, (HR > 1 && row > 32) ? rcp[HR - 1] : rcp[0], (row - 1) & 31);  // q = M[row, col]
        }
        if (row == kNone) {
          status = ST_UNBOUNDED;
          value = (double)col;
          break;
        }
        tm_load_row(tbase, row, pr0, pr1);
      }

      if (kCycles) {  // (:98, :137): push (leaving, entering), then look for two identical runs of length 6..len/2
        if (hist_len >= a.hist_cap) {
          status = ST_ERR_HISTORY;
          break;
        }
        if (lane == 0) {
          hist[2 * hist_len] = var[W + row];
          hist[2 * hist_len + 1] = var[col];
        }
        hist_len++;
        __syncwarp();
        bool found = false;
        for (int Lc = 6 + lane; Lc <= hist_len / 2 && !found; Lc += 32) {
          bool cyc = true;
          for (int i = 0; i < Lc; i++) {
            const int item = hist_len - 1 - i;
            if (hist[2 * item] != hist[2 * (item - Lc)] || hist[2 * item + 1] != hist[2 * (item - Lc) + 1]) {
              cyc = false;
              break;
            }
          }
          found = cyc;
        }
        if (__any_sync(0xffffffffu, found)) break;  // "cycled", NaN
      }
      // ---- pivot(row, col) (:5-39)
      const int jc = col - 1, lc = jc >> 1, ec = jc & 1;
      const double q = colx[row];
      const double c0raw = colx[0];
      RecipBatch rq(q, rcp_q);  // one acceptance branch for the four quotients of this lane; the reciprocal is the selection's
      // normalised pivot row cells of my columns; the pivot cell itself becomes 1/q
      const bool own0 = lane == lc && ec == 0, own1 = lane == lc && ec == 1;
      const double x0 = own0 ? 1.0 : pr0, x1 = own1 ? 1.0 : pr1;
      const bool n0 = v0 && fabs(x0) > kTiny, n1 = v1 && fabs(x1) > kTiny;
      // rows 1..H-1: one (lane, slot) each (the owner of the pivot row normalises the RHS cell instead)
      bool is_prow[HR], nzq[HR];
      double num[HR], quo[HR];
#pragma unroll
      for (int h = 0; h < HR; h++) {
        is_prow[h] = lane + 1 + 32 * h == row;
        num[h] = is_prow[h] ? bv[h] : -cmine[h];
        nzq[h] = has_b[h] && fabs(num[h]) > kTiny;  // false for NaN, as in the reference
      }
      const bool act0 = fabs(c0raw) > kTiny;       // row 0 (objective row): every lane redundantly
      double pn0 = rq.quot(x0, n0), pn1 = rq.quot(x1, n1);
#pragma unroll
      for (int h = 0; h < HR; h++) quo[h] = rq.quot(num[h], nzq[h]);
      double cn0 = rq.quot(-c0raw, act0);
      if (!rq.ok) {  // rare: exact divisions out of line
        pn0 = div_rn_slow(x0, q);
        pn1 = div_rn_slow(x1, q);
#pragma unroll
        for (int h = 0; h < HR; h++) quo[h] = div_rn_slow(num[h], q);
        cn0 = div_rn_slow(-c0raw, q);
      }
      pn0 = n0 ? pn0 : 0.0;
      pn1 = n1 ? pn1 : 0.0;
      cn0 = act0 ? cn0 : 0.0;
      const bool st0 = n0 && !own0, st1 = n1 && !own1;  // cells the rank-1 pass rewrites
      double coef_mine[HR];
      bool rows_on = true;  // my rows take the fast form of the row pass
#pragma unroll
      for (int h = 0; h < HR; h++) {
        quo[h] = nzq[h] ? quo[h] : 0.0;
        coef_mine[h] = (nzq[h] && !is_prow[h]) ? cmine[h] : 0.0;  // 0 = my row is skipped (:31) or is the pivot row
        // the pivot row takes part in the row pass with a throw-away coefficient (it is rewritten afterwards)
        const double cbx = is_prow[h] ? 1.0 : coef_mine[h];
        if (has_b[h]) cb[lane + 1 + 32 * h] = make_double2(cbx, coef_mine[h] != 0.0 ? quo[h] : cmine[h]);
        rows_on = rows_on && (!has_b[h] || cbx != 0.0);
      }
      const unsigned on_mask = __ballot_sync(0xffffffffu, rows_on);  // all ones: every row takes the fast form
      // normalised RHS of the pivot row and whether it was above 1e-16, from its owner: lane (row-1)%32, slot (row-1)/32
      const bool pslot = HR > 1 && row > 32;
      const double p0 = __shfl_sync(0xffffffffu, pslot ? quo[HR - 1] : quo[0], (row - 1) & 31);
      const bool nz0 = __shfl_sync(0xffffffffu, (pslot ? nzq[HR - 1] : nzq[0]) ? 1 : 0, (row - 1) & 31);
      if (lane == 0) {  // basis bookkeeping (:7-12)
        const int leaving = var[W + row];
        var[W + row] = var[col];
        var[col] = leaving;
      }
      __syncwarp();  // cb complete; every lane has read q, c0raw and its colx cell

      // objective row and RHS column in registers
      if (act0) {
        if (st0) o0 = __dsub_rn(o0, __dmul_rn(c0raw, pn0));
        if (st1) o1 = __dsub_rn(o1, __dmul_rn(c0raw, pn1));
        if (own0) o0 = cn0;
        if (own1) o1 = cn0;
        if (nz0) b0 = __dsub_rn(b0, __dmul_rn(c0raw, p0));
      }
#pragma unroll
      for (int h = 0; h < HR; h++) {
        if (is_prow[h])
          bv[h] = quo[h];
        else if (coef_mine[h] != 0.0 && nz0)
          bv[h] = __dsub_rn(bv[h], __dmul_rn(coef_mine[h], p0));
      }

      // rank-1 pass over the TMEM blocks; a lane's padding cells (zeros, never read) count as rewritable
      {
        const bool dense = __all_sync(0xffffffffu, (st0 || own0 || !v0) && (st1 || own1 || !v1));
        const TmemPivot pv{pn0, pn1, st0, st1, own0, own1};
        if (dense && on_mask == 0xffffffffu) {  // the common case of a dense LP: every block takes the fast form
          if (kCount) rows_rewritten += (unsigned)(H - 2 + (act0 ? 1 : 0));  // every row but the pivot row
          if (ec == 0) {
            for (int blk = 0; blk < nblocks; blk++) tmem_block_fast<0>(tbase + 32u * (unsigned)blk, cb + 1 + 8 * blk, pv);
          } else {
            for (int blk = 0; blk < nblocks; blk++) tmem_block_fast<1>(tbase + 32u * (unsigned)blk, cb + 1 + 8 * blk, pv);
          }
        } else {
          unsigned act[HR];  // rows the update rewrites (:31): not skipped, not the pivot row
          int nact = 0;
#pragma unroll
          for (int h = 0; h < HR; h++) {
            act[h] = __ballot_sync(0xffffffffu, coef_mine[h] != 0.0);
            nact += __popc(act[h]);
          }
          if (kCount) rows_rewritten += (unsigned)(nact + (act0 ? 1 : 0));
          if (4 * nact <= H - 1) {  // sparse pivot column: touch the active rows only
#pragma unroll
            for (int h = 0; h < HR; h++) tmem_rows_sparse(tbase, act[h], 1 + 32 * h, cb, pv);
          } else {
            if (ec == 0) {
              for (int blk = 0; blk < nblocks; blk++) tmem_block_general<0>(tbase + 32u * (unsigned)blk, cb + 1 + 8 * blk, pv);
            } else {
              for (int blk = 0; blk < nblocks; blk++) tmem_block_general<1>(tbase + 32u * (unsigned)blk, cb + 1 + 8 * blk, pv);
            }
          }
        }
      }
      tm_wait_st();  // the row pass stored a throw-away value in the pivot row: order the real one behind it
      tm_store_row(tbase, row, pn0, pn1);  // (:19,22,25); waited for in front of the next TMEM read
      iter++;
    }
    long long p2 = 0;
    if (phase == 1)
      p1 = iter;
    else
      p2 = iter;

    // ---- outputs
    if (lane == 0) {
      if (a.status) a.status[lp] = status;
      if (a.value) a.value[lp] = value;
      if (a.pivots) {
        a.pivots[2 * lp] = p1;
        a.pivots[2 * lp + 1] = p2;
      }
      if (a.rhs_out) a.rhs_out[roff] = b0;
      if (kCount && a.rows_out) atomicAdd(a.rows_out + (a.rows_per_lp ? lp : 0), rows_rewritten);
    }
#pragma unroll
    for (int h = 0; h < HR; h++)
      if (a.rhs_out && has_b[h]) a.rhs_out[roff + lane + 1 + 32 * h] = bv[h];
    if (a.pos_out)
      for (int k = lane; k < W + H; k += 32) a.pos_out[poff + var[k]] = k;
    if (a.var_out)
      for (int k = lane; k < W + H; k += 32) a.var_out[poff + k] = var[k];
    if (a.red_out) {  // row 0 is in registers: lane l holds columns 2l+1 (o0) and 2l+2 (o1)
      if (v0) a.red_out[poff + var[1 + j0]] = o0;
      if (v1) a.red_out[poff + var[2 + j0]] = o1;
      for (int k = lane; k < H + 1; k += 32) a.red_out[poff + var[k == 0 ? 0 : W - 1 + k]] = 0.0;
    }
    tm_wait_st();
    if (a.mat_out) {
      double *dst = a.mat_out + moff;
      if (lane == 0) dst[0] = b0;
#pragma unroll
      for (int h = 0; h < HR; h++)
        if (has_b[h]) dst[(size_t)(lane + 1 + 32 * h) * W] = bv[h];
      if (v0) dst[1 + j0] = o0;
      if (v1) dst[2 + j0] = o1;
      for (int r = 1; r < H; r++) {
        double y0, y1;
        tm_load_row(tbase, r, y0, y1);
        if (v0) dst[(size_t)r * W + 1 + j0] = y0;
        if (v1) dst[(size_t)r * W + 2 + j0] = y1;
      }
    }
    __syncwarp();
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_tmem_base), "n"(S::kColumns) : "memory");
}

}  // namespace yalps
