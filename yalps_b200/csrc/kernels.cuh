// kernels.cuh -- batch kernels built on simplex_device.cuh.
//
//  K1  k_simplex<NW,KC,true >  one tableau per CTA resident in shared memory (persistent CTAs, atomic LP queue)
//  K2  k_simplex<NW,KC,false>  tableau in HBM/L2 (working copy), pivot row / column staged in shared memory
//  K3  node assembly (applyCuts, src/branchAndCut.ts:22-61) fused as the prologue of K1/K2 (mode == kModeNodes)
//  K5  generators and the other non-template kernels live in aux_kernels.cuh
#pragma once

#include "simplex_device.cuh"
#include "simplex_split.cuh"

namespace yalps {

enum : int { kModeBatch = 0, kModeNodes = 1 };

struct BatchArgs {
  long long n;
  int mode;
  int H, W;       // uniform LP shape (kModeBatch, heights == nullptr) or root shape (kModeNodes)
  int Hcap;       // tallest LP of the launch (shared-memory carve-up, output stride in node mode)
  int Wcap;       // widest LP of the launch (shared-memory carve-up)
  const double *in;   // input tableaus (kModeBatch)
  double *work;       // K2 working copies (may alias `in`); unused by K1
  double *mat_out;    // optional final tableaus
  const int *heights, *widths;          // ragged batch (nullable)
  const long long *mat_off, *rhs_off, *pos_off;
  const int *index;                     // ragged groups: launch-local LP -> LP id within the chunk (nullable)
  int *status;
  double *value;
  long long *pivots;
  double *rhs_out;
  int *pos_out, *var_out;
  // optional diagnostics for the roofline (SURVEY 8d): rows rewritten by the rank-1 updates, summed over the pivots of
  // an LP, ADDED (atomically) to rows_out[rows_per_lp ? lp : 0]; the host zeroes the buffer
  unsigned long long *rows_out;
  int rows_per_lp;
  // optional per-LP resume state, 3 long long per LP: [phase, pivots done in phase 1, in phase 2] (replica path sharing)
  const long long *resume;
  // optional trace of ONE LP (n == 1): see SplitScratch (simplex_split.cuh); only the row-split kernels record it
  int *tr_steps;
  double *tr_q, *tr_col, *tr_snap;
  int *tr_var;
  int tr_hp, tr_cap;
  const int *var_in;  // optional initial variableAtPosition, packed like var_out (null: the identity, src/tableau.ts:95-98)
  // node mode
  const double *root;
  const int *root_pos, *root_var;
  int assembled;  // node mode: a.work already holds root + cut rows (k_assemble_nodes ran first)
  const int *cut_off;
  const double *cut_sign;
  const int *cut_var;
  const double *cut_val;
  // options
  double precision, max_pivots;
  int check_cycles;
  int *hist;        // gridDim.x * 2 * hist_cap
  int hist_cap;
  unsigned long long *counter;
  double *cl_scratch;  // cluster kernel: per cluster 2 * C * ldA doubles (published candidate pivot rows)
  int tma_mode;        // cluster kernel: how the winner's row is staged (0 ld.global.cg, 1 cp.async.bulk, 2 multicast)
  uint4 *gx_slots;     // grid-resident kernel (KG): [2][gridDim.x][gridDim.x] selection records (inbox per CTA); `counter` is its grid barrier
  // optional reduced costs, packed like pos_out: red_out[v] = M[0, pos[v]] for a non-basic structural or slack
  // variable (1 <= pos[v] < W), +0.0 for the basic ones and for ids 0 and W (row 0 re-indexed, written for every status)
  double *red_out;
};

// Shared-memory carve-up, identical on host and device.
// Resident layout: every tableau row is  [ A(0..W-2) | pad | b | -coef/q ]  with an even row stride ldA
// (16-byte aligned rows -> v2.f64 accesses) whose half is odd (strided column reads spread over the banks);
// the RHS cell and the per-pivot -coef/q scratch cell of a row live in its last two slots.
// Split kernels (row groups, simplex_split.cuh) replace colbuf/colnew by the compacted active-row list.
struct SmemLayout {
  size_t off_A, off_colbuf, off_colnew, off_misc, off_red, off_var, off_cc, off_list, off_cnt, off_bcol, total;
  int ldA;
  __host__ __device__ static int ld_for(int W) {
    int ld = (W - 1 + 2 + 1) & ~1;
    if (((ld >> 1) & 1) == 0) ld += 2;
    return ld;
  }
  __host__ __device__ SmemLayout(int Hcap, int Wcap, bool resident, int nw, bool split = false) {
    size_t o = 0;
    ldA = ld_for(Wcap);
    off_A = o;
    if (resident) o += (size_t)Hcap * ldA * 8;
    off_colbuf = off_colnew = off_cc = off_list = off_cnt = o;
    if (split) {
      off_cc = o;
      o += (size_t)(Hcap + 8) * 16;
      off_list = o;
      o += (size_t)((Hcap + 3) & ~3) * 4;
      off_cnt = o;
      o += 16;
    } else {
      off_colbuf = o;
      o += (size_t)((Hcap + 7) & ~7) * 8;
      off_colnew = o;
      if (!resident) o += (size_t)((Hcap + 1) & ~1) * 8;
    }
    off_misc = o;
    o += 16;
    off_red = o;
    if (nw > 1) o += 192 * 4;
    off_var = o;
    if (resident || split) o += (size_t)(Wcap + Hcap) * 4;  // (split kernels: variableAtPosition on chip in either layout)
    // HBM/L2-resident split kernels keep the RHS column of their tableau in shared memory (see k_simplex)
    o = (o + 15) & ~(size_t)15;
    off_bcol = o;
    if (!resident && split) o += (size_t)((Hcap + 1) & ~1) * 8;
    total = (o + 15) & ~(size_t)15;
  }
};

__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// min CTAs/SM in the launch bounds caps the register count so that shared memory, not registers, limits residency
// (one-warp CTAs: 12 per SM -> <= 168 registers per thread).
// NWR > 1: split kernel, NWC column warps x NWR row groups, registers capped at 128 per thread.
constexpr int min_ctas_per_sm(int nwc, int nwr) {
  return nwr == 1 ? (nwc == 1 ? 12 : (nwc == 2 ? 6 : (nwc == 4 ? 3 : (nwc == 8 ? 2 : 1))))
                  : (nwc * nwr >= 16 ? 1 : 16 / (nwc * nwr));
}

template <int NWC, int KC, bool kResident, int NWR = 1>
__global__ void __launch_bounds__(NWC *NWR * 32, min_ctas_per_sm(NWC, NWR)) k_simplex(const BatchArgs a) {
  constexpr int NW = NWC * NWR;
  constexpr int NT = NW * 32;
  constexpr bool kSplit = NWR > 1;
  constexpr int VW = kResident ? 2 : 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ long long s_lp;
  const int tid = threadIdx.x;

  for (long long static_lp = blockIdx.x;; static_lp += gridDim.x) {
    long long lp = static_lp;  // small launches (node waves): LPs dealt statically, no queue to reset
    if (a.counter) {           // big batches: persistent CTAs pull the next LP from an atomic queue
      if (tid == 0) s_lp = (long long)atomicAdd(a.counter, 1ULL);
      __syncthreads();
      lp = s_lp;
      __syncthreads();
    }
    if (lp >= a.n) break;
    if (a.index) lp = a.index[lp];

    int H, W, ncuts = 0;
    size_t moff, roff, poff;
    if (a.mode == kModeNodes) {
      ncuts = a.cut_off[lp + 1] - a.cut_off[lp];
      H = a.H + ncuts;
      W = a.W;
      moff = (size_t)lp * a.Hcap * W;
      roff = (size_t)lp * a.Hcap;
      poff = (size_t)lp * (W + a.Hcap);
    } else if (a.heights) {
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

    const SmemLayout L(a.Hcap, a.Wcap, kResident, NW, kSplit);
    LpView t;
    t.H = H;
    t.W = W;
    Scratch s;
    SplitScratch ss;
    if (kResident) {
      t.A = reinterpret_cast<double *>(smem_raw + L.off_A);
      t.ldA = t.ldb = SmemLayout::ld_for(W);
      t.b = t.A + (t.ldA - 2);
      s.colnew = t.A + (t.ldA - 1);
      s.ldc = t.ldA;
      t.var = reinterpret_cast<int *>(smem_raw + L.off_var);
    } else {
      s.colnew = reinterpret_cast<double *>(smem_raw + L.off_colnew);
      s.ldc = 1;
      t.A = a.work + moff + 1;
      t.b = a.work + moff;
      t.ldA = t.ldb = W;
      t.var = kSplit ? reinterpret_cast<int *>(smem_raw + L.off_var) : a.var_out + poff;
    }
    s.colbuf = reinterpret_cast<double *>(smem_raw + L.off_colbuf);
    s.misc = reinterpret_cast<double *>(smem_raw + L.off_misc);
    s.red = reinterpret_cast<unsigned *>(smem_raw + L.off_red);
    s.hist = a.hist ? a.hist + (size_t)blockIdx.x * 2 * a.hist_cap : nullptr;
    s.hist_cap = a.hist_cap;
    ss.cc = reinterpret_cast<double *>(smem_raw + L.off_cc);
    ss.list = reinterpret_cast<int *>(smem_raw + L.off_list);
    ss.cnt = reinterpret_cast<int *>(smem_raw + L.off_cnt);
    ss.misc = s.misc;
    ss.red = s.red;
    ss.hist = s.hist;
    ss.hist_cap = s.hist_cap;
    s.resume = ss.resume = a.resume ? a.resume + 3 * lp : nullptr;
    ss.tr_steps = a.tr_steps;
    ss.tr_q = a.tr_q;
    ss.tr_col = a.tr_col;
    ss.tr_snap = a.tr_snap;
    ss.tr_var = a.tr_var;
    ss.tr_hp = a.tr_hp;
    ss.tr_cap = a.tr_cap;
    if (kSplit && tid == 0) *ss.cnt = 0;
#ifdef YALPS_TIMING
    long long yt_local[16];
    for (int k = 0; k < 16; k++) yt_local[k] = 0;
    yt_local[15] = clock64();
    ss.yt = yt_local;
#endif

    // ---- load / assemble the tableau (reference layout, row stride W) into the (A, b) view
    const int ldA = t.ldA, ldb = t.ldb;
    const int rootH = a.mode == kModeNodes ? a.H : H;
    const double *src = a.mode == kModeNodes ? a.root : a.in + moff;
    if (kResident) {
      // asynchronous 8-byte copies (LDGSTS) straight into the (A, b) layout: every copy of the tableau is in
      // flight before the first one is waited for, so the load costs one memory latency, not one per row
      // (addresses advance incrementally: one 32-bit shared address and one global pointer per lane)
      {
        const int lane = tid & 31;
        const unsigned sA0 = (unsigned)__cvta_generic_to_shared(t.A) + 8u * (unsigned)lane;  // A[r][lane]
        const unsigned sB0 = (unsigned)__cvta_generic_to_shared(t.b);
        const unsigned row_bytes = 8u * (unsigned)ldA;
        const int full = (W - 1) / 32, tail = (W - 1) - 32 * full;  // coefficient columns per lane
        unsigned sA = sA0 + row_bytes * (unsigned)(tid >> 5), sB = sB0 + 8u * (unsigned)ldb * (unsigned)(tid >> 5);
        const double *g = src + (size_t)(tid >> 5) * W;
        for (int r = tid >> 5; r < rootH; r += NW) {
          if (lane == 0) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sB), "l"(g) : "memory");
          const double *gc = g + 1 + lane;
          unsigned d = sA;
          for (int k = 0; k < full; k++) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gc) : "memory");
            gc += 32;
            d += 256u;
          }
          if (lane < tail) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gc) : "memory");
          g += (size_t)NW * W;
          sA += row_bytes * NW;
          sB += 8u * (unsigned)ldb * NW;
        }
      }
    } else if (src != a.work + moff && !(a.mode == kModeNodes && a.assembled)) {
      const size_t cells = (size_t)rootH * W;
      double *dst = a.work + moff;
      for (size_t k = tid; k < cells; k += NT) dst[k] = src[k];
    }
    if (a.mode == kModeNodes) {
      // applyCuts (src/branchAndCut.ts:22-61): one row per cut below the root rows
      const int cbeg = a.cut_off[lp];
      for (int i = 0; i < (a.assembled ? 0 : ncuts); i++) {
        const double sign = a.cut_sign[cbeg + i], value = a.cut_val[cbeg + i];
        const int p = a.root_pos[a.cut_var[cbeg + i]];
        const int r = rootH + i;
        double *dA = t.A + (size_t)r * ldA - 1;
        if (p < W) {
          for (int c = tid; c < W; c += NT) {
            if (c == 0)
              t.b[(size_t)r * ldb] = __dmul_rn(sign, value);
            else
              dA[c] = (c == p) ? sign : 0.0;
          }
        } else {
          const double *sr = a.root + (size_t)(p - W) * W;
          for (int c = tid; c < W; c += NT) {
            if (c == 0)
              t.b[(size_t)r * ldb] = __dmul_rn(sign, __dsub_rn(value, sr[0]));
            else
              dA[c] = __dmul_rn(-sign, sr[c]);
          }
        }
      }
      const int nroot = W + rootH;
      for (int k = tid; k < W + H; k += NT) t.var[k] = k < nroot ? a.root_var[k] : k;
    } else if (a.var_in) {  // caller-supplied basis (src/branchAndCut.ts:127 calls simplex on applyCuts' permutation)
      for (int k = tid; k < W + H; k += NT) t.var[k] = a.var_in[poff + k];
    } else {
      for (int k = tid; k < W + H; k += NT) t.var[k] = k;
    }
    if (kResident) {  // zero the padding columns so that vector loads past W-1 read defined values
      const int pad = ldA - 2 - (W - 1);
      for (int k = tid; k < H * pad; k += NT) t.A[(size_t)(k / pad) * ldA + (W - 1) + (k % pad)] = 0.0;
    }
    if (kResident) cp_async_wait_all();
    __syncthreads();
    // HBM/L2-resident split kernels: the RHS column moves into shared memory for the whole solve.  It is the one
    // strided column every pivot reads (leaving row of phase 1, ratio test of phase 2) and rewrites, and with it in
    // shared memory the first selection of a phase-1 pivot -- all a branch-and-cut node LP consists of -- costs no trip
    // to L2.  Same values, same operations; the column is written back behind the solve.
    constexpr bool kBcolShared = !kResident && kSplit;
    if (kBcolShared) {
      double *bcol = reinterpret_cast<double *>(smem_raw + L.off_bcol);
      for (int r = tid; r < H; r += NT) bcol[r] = t.b[(size_t)r * ldb];
      __syncthreads();
      t.b = bcol;
      t.ldb = 1;
    }

    LpResult res;
    if constexpr (kSplit)
      res = simplex_cta_split<NWC, KC, NWR, VW>(t, ss, a.precision, a.max_pivots, a.check_cycles);
    else
      res = simplex_cta<NW, KC, VW>(t, s, a.precision, a.max_pivots, a.check_cycles);
    __syncthreads();
    if (tid == 0) {
      if (a.status) a.status[lp] = res.status;
      if (a.value) a.value[lp] = res.value;
      if (a.pivots) {
        a.pivots[2 * lp] = res.p1;
        a.pivots[2 * lp + 1] = res.p2;
      }
    }
    if (a.rows_out && res.rows != 0 && (!kSplit || tid == 0)) atomicAdd(a.rows_out + (a.rows_per_lp ? lp : 0), res.rows);
    if (a.rhs_out)
      for (int r = tid; r < H; r += NT) a.rhs_out[roff + r] = t.b[(size_t)r * t.ldb];
    if (kBcolShared)  // column 0 of the working copy: whoever reads the final tableau finds it complete
      for (int r = tid; r < H; r += NT) a.work[moff + (size_t)r * W] = t.b[r];
#ifdef YALPS_TIMING
    __syncthreads();
    if (kSplit && a.rhs_out && (tid == 0 || tid == NT - 1 || tid == 32)) {
      // debug builds only: phase cycle counters of three threads overwrite the RHS output (needs H >= 27)
      double *o = a.rhs_out + roff + (tid == 0 ? 0 : (tid == 32 ? 9 : 18));
      for (int k = 0; k < 8; k++) o[k] = (double)yt_local[k];
      o[8] = (double)(res.p1 + res.p2);
    }
#endif
    if (a.pos_out)  // positionOfVariable is the inverse permutation of variableAtPosition
      for (int k = tid; k < W + H; k += NT) a.pos_out[poff + t.var[k]] = k;
    if ((kResident || kSplit) && a.var_out)
      for (int k = tid; k < W + H; k += NT) a.var_out[poff + k] = t.var[k];
    if (a.red_out)  // row 0, column k >= 1, is t.A[k - 1]
      for (int k = tid; k < W + H; k += NT) a.red_out[poff + t.var[k]] = (k >= 1 && k < W) ? t.A[k - 1] : 0.0;
    if (a.mat_out) {
      double *dst = a.mat_out + moff;
      if (kResident || dst != a.work + moff) {
        for (int r = tid >> 5; r < H; r += NW) {
          const double *sA = t.A + (size_t)r * ldA - 1;
          double *dr = dst + (size_t)r * W;
          for (int c = tid & 31; c < W; c += 32) dr[c] = (c == 0) ? t.b[(size_t)r * t.ldb] : sA[c];
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace yalps
