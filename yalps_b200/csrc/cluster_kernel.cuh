// cluster_kernel.cuh -- KC: one LP per thread-block cluster, tableau resident in the cluster's shared memory.
//
// For tableaus that do not fit the 227 KB of one SM but fit the 1.8-3.6 MB of a cluster of 8-16 CTAs: Netlib-size
// models solved one at a time, branch-and-cut roots, mid-size batches (BASELINE.json north_star (b)).  Same
// algorithm, arithmetic and tie-breaking as simplex_split.cuh (src/simplex.ts:5-142), different placement:
//   * rows 1..H-1 are dealt round-robin to the C CTAs of the cluster (row r lives in CTA (r-1) % C at local index
//     (r-1) / C), in the padded layout [ A | pad | b | s ] of the resident kernels; pivot-column cells, ratio
//     tests, RHS scans and the rank-1 update of a row are therefore local to its CTA;
//   * every CTA keeps a private copy of the objective row (row 0) and applies the pivot to it with the same
//     operands and operations as every other CTA, so the copies stay bit-identical and the entering-column scan
//     of phase 2 needs no communication;
//   * a row selection is a CTA-local arg-reduction, one 16-byte DSMEM store per peer (st.shared::cluster into the
//     peer's exchange slots) and ONE cluster barrier per pivot.  DSMEM moves only ~20 B/clk per SM (measured: a
//     first version in which every thread read the pivot row out of its owner's shared memory spent 4-16 k cycles
//     per pivot there), so the pivot row itself travels through L2: before that barrier every CTA publishes the
//     row of its own candidate (W cells, st.global.cg) to a per-cluster scratch buffer, after it every CTA stages
//     the winner's row from L2 into its shared memory once (ld.global.cg) and all its row groups read it there;
//   * the pivot row is normalised redundantly in registers by every thread that needs its cells (one shared
//     reciprocal, fastdiv.cuh); the owner writes the normalised row back into its shared memory.
// Per pivot: one cluster barrier and four CTA barriers, against two full grid barriers for K4.
//
// KG (kGrid = true): the same kernel with the "cluster" widened to the WHOLE GRID of a cooperative launch -- up to one
// CTA per SM, the tableau resident in their 148 x 227 KB of shared memory (tableaus up to ~25 MB: 1025 x 2049,
// Netlib 25FV47), so the rank-1 update never leaves the SMs.  The cluster barrier becomes a grid barrier (one per
// pivot, release/acquire on an L2 counter) and the 16-byte selection records travel through an L2 slot array instead
// of DSMEM; candidate rows go through the L2 scratch exactly as in KC.  K4 pays two grid barriers, two dependent L2
// trips and an L2-bound update per pivot for such tableaus.
#pragma once

#include <cooperative_groups.h>

#include "kernels.cuh"

namespace yalps {

namespace cg = cooperative_groups;

constexpr int kMaxCluster = 16;
constexpr int kGiveUp = -2;  // grid_select: a record never arrived

struct ClusterSmem {
  size_t off_A, off_obj, off_prow, off_cc, off_list, off_cnt, off_misc, off_red, off_xch, off_var, total;
  int ldA, Hloc;
  __host__ __device__ ClusterSmem(int Hcap, int Wcap, int C) {
    ldA = SmemLayout::ld_for(Wcap);
    Hloc = (Hcap - 1 + C - 1) / C;
    size_t o = 0;
    off_A = o;
    o += (size_t)Hloc * ldA * 8;
    off_obj = o;
    o += (size_t)ldA * 8;
    off_prow = o;  // staged copy of the (raw) pivot row
    o += (size_t)ldA * 8;
    off_cc = o;
    o += (size_t)(Hloc + 8) * 16;
    off_list = o;
    o += (size_t)((Hloc + 3) & ~3) * 4;
    off_cnt = o;
    o += 16;
    off_misc = o;
    o += 32;
    off_red = o;
    o += 192 * 4;
    off_xch = o;
    o += 2 * kMaxCluster * 16;
    off_var = o;
    o += (size_t)(Wcap + Hcap) * 4;
    total = (o + 15) & ~(size_t)15;
  }
};

// CTA-wide winner with its key (block_best of simplex_device.cuh returns only the index).
template <bool kMax, int NW>
__device__ __forceinline__ Best block_best_full(unsigned long long key, int idx, unsigned *red, int &parity) {
  Best w = warp_best<kMax>((unsigned)(key >> 32), (unsigned)key, idx);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned *r = red + parity * 96;
  parity ^= 1;
  if (lane == 0) {
    r[warp] = w.hi;
    r[32 + warp] = w.lo;
    r[64 + warp] = (unsigned)w.idx;
  }
  __syncthreads();
  const unsigned long long nk = no_key<kMax>();
  const unsigned hi = lane < NW ? r[lane] : (unsigned)(nk >> 32);
  const unsigned lo = lane < NW ? r[32 + lane] : (unsigned)nk;
  const int id = lane < NW ? (int)r[64 + lane] : kNone;
  return warp_best<kMax>(hi, lo, id);
}

// ---- TMA (bulk asynchronous copy) staging of the winner's row, selectable at run time for the A/B of north_star (b):
//   mode 0  every thread loads 16-byte chunks from the L2 scratch (ld.global.cg) and stores them to shared memory
//   mode 1  one thread per CTA issues ONE cp.async.bulk global -> shared of the whole row, completion on an mbarrier
//   mode 2  the winner's owner issues ONE cp.async.bulk ... .multicast::cluster that lands the row in the shared
//           memory of every CTA of the cluster (each CTA's own mbarrier counts the bytes)
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_g2s_multicast(void *dst_smem, const void *src_gmem, unsigned bytes, unsigned long long *bar,
                                                   unsigned short cta_mask) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
      : "memory");
}

// Cluster-wide winning row.  Every CTA posts its local winner into slot [rank] of every CTA's exchange buffer and
// publishes that candidate's row (padded layout, ldA cells) to scratch[xpar][rank]; after the barrier every CTA
// stages the winner's row into prow_s.  Returns kNone (nothing staged) when no CTA had a candidate.
template <bool kMax, int NW>
__device__ __forceinline__ int cluster_select(cg::cluster_group &cluster, int C, int rank, unsigned long long key, int idx,
                                              unsigned *red, int &parity, uint4 *xch, int &xpar, const double *A, int ldA,
                                              double *scratch, double *prow_s, int tma_mode = 0,
                                              unsigned long long *mbar = nullptr, unsigned *mphase = nullptr) {
  constexpr int NT = NW * 32;
  const Best w = block_best_full<kMax, NW>(key, idx, red, parity);
  uint4 *slots = xch + xpar * kMaxCluster;
  double *pub = scratch + (size_t)xpar * C * ldA;
  xpar ^= 1;
  if (w.idx != kNone) {  // publish my candidate row (16-byte chunks; ldA is even and rows are 16-byte aligned)
    const double2 *src = reinterpret_cast<const double2 *>(A + (size_t)((w.idx - 1) / C) * ldA);
    double2 *dst = reinterpret_cast<double2 *>(pub + (size_t)rank * ldA);
    for (int c = threadIdx.x; c < ldA / 2; c += NT) __stcg(dst + c, src[c]);
    if (tma_mode) asm volatile("fence.proxy.async;" ::: "memory");  // generic-proxy stores before async-proxy (TMA) reads
  }
  if ((int)threadIdx.x < C) {
    uint4 *dst = cluster.map_shared_rank(slots + rank, threadIdx.x);
    *dst = make_uint4(w.hi, w.lo, (unsigned)w.idx, 0u);
  }
  cluster.sync();
  const int lane = threadIdx.x & 31;
  const unsigned long long nk = no_key<kMax>();
  uint4 e = make_uint4((unsigned)(nk >> 32), (unsigned)nk, (unsigned)kNone, 0u);
  if (lane < C) e = slots[lane];
  const int row = warp_best<kMax>(e.x, e.y, (int)e.z).idx;
  if (row != kNone) {
    const int owner = (row - 1) % C;
    const double2 *src = reinterpret_cast<const double2 *>(pub + (size_t)owner * ldA);
    if (tma_mode == 0) {
      double2 *dst = reinterpret_cast<double2 *>(prow_s);
      for (int c = threadIdx.x; c < ldA / 2; c += NT) dst[c] = __ldcg(src + c);
      __syncthreads();
    } else {
      const unsigned bytes = (unsigned)ldA * 8u;  // ldA is even: a multiple of 16 bytes, rows are 16-byte aligned
      if (threadIdx.x == 0) {
        mbar_expect_tx(mbar, bytes);  // every CTA arms its own barrier
        if (tma_mode == 1)
          bulk_g2s(prow_s, src, bytes, mbar);
        else if (rank == owner)
          bulk_g2s_multicast(prow_s, src, bytes, mbar, (unsigned short)((1u << C) - 1u));
      }
      mbar_wait(mbar, *mphase);
      *mphase ^= 1u;
    }
  }
  return row;
}

// Grid-wide barrier of a cooperative launch: one release reduction and an acquire spin by thread 0 between two CTA
// barriers (the CTA barrier makes the other threads' writes part of what the release publishes).
__device__ __forceinline__ void grid_sync_lean(unsigned long long *counter, unsigned long long &epoch) {
  __syncthreads();
  epoch++;
  if (threadIdx.x == 0) {
    const unsigned long long goal = epoch * gridDim.x;
    asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(counter) : "memory");
    unsigned long long seen;
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(counter) : "memory");
    } while (seen < goal);
  }
  __syncthreads();
}

// cluster_select for the grid-wide kernel, WITHOUT a barrier: a selection record is one 16-byte slot
//   A = key[63:16] << 16 | seq,   B = key[15:0] << 48 | idx << 16 | seq
// whose 8-byte halves each carry the 16-bit sequence number of the exchange (flag in data, as NCCL's LL protocol: a half
// is valid the moment its sequence matches), written by thread 0 after a fence that orders the CTA's published
// candidate row before it.  Warp 0 of every CTA polls all C slots (lane j takes j, j + 32, ...), picks the winner
// (best key, lowest index on ties, as warp_best), fences and hands the row index to the CTA; the winner's row is then
// staged from the L2 scratch.  Slots and scratch are double-buffered by exchange parity: a CTA can only be one exchange
// ahead of the slowest one, because it needs that CTA's next record, which is written after that CTA has finished
// reading the current buffers.  (First version: counter barrier + sequential record reads, 10,000 cycles per
// selection on 25FV47; see profiles/.)
template <bool kMax, int NW, int kRowU>
__device__ __forceinline__ int grid_select(int C, int rank, unsigned long long key, int idx, unsigned *red, int &parity,
                                           uint4 *gslots, unsigned &xcount, const double *A, int ldA, double *scratch,
                                           double *prow_s, int *s_row, long long *yt = nullptr, long long *yt_last = nullptr) {
  constexpr int NT = NW * 32;
  // (timing builds: yt[6] = candidate row published + records pushed (warp 0), yt[7] += winner's row staged; the wait in between
  // lands in the caller's selection slot)
#define GS_MARK(k) do { if (yt) { const long long now_ = clock64(); yt[k] += now_ - *yt_last; *yt_last = now_; } } while (0)
  constexpr int kMaxPerLane = 5;  // C <= 160
  const Best w = block_best_full<kMax, NW>(key, idx, red, parity);
  xcount++;
  const int xpar = (int)(xcount & 1u);
  const unsigned long long seq = (unsigned long long)(xcount % 65535u) + 1ULL;  // never 0 (the cleared state)
  // inbox[xpar][receiver][sender]: every CTA polls lines nobody else polls (a first version had all CTAs poll one
  // shared array of C records: 148 x 148 reads of the same 19 lines per round, 6,000 cycles of waiting per selection)
  ulonglong2 *inbox = reinterpret_cast<ulonglong2 *>(gslots) + (size_t)xpar * C * C;
  ulonglong2 *slots = inbox + (size_t)rank * C;
  // candidate rows travel as flag-in-data slots too: one 16-byte {low word, sequence, high word, sequence} per cell
  // (the 32-bit exchange counter), so neither the publisher nor the readers need a fence and the records can leave
  // BEFORE the row is written (a version with plain row stores + fence + records spent 2,700 cycles publishing)
  uint4 *pub = reinterpret_cast<uint4 *>(scratch) + (size_t)xpar * C * ldA;
  const unsigned rseq = xcount;
  if (threadIdx.x < 32) {  // records first
    const int lane = threadIdx.x;
    const unsigned long long k = ((unsigned long long)w.hi << 32) | w.lo;
    const unsigned long long ra = (k & ~0xffffULL) | seq;
    const unsigned long long rb = ((k & 0xffffULL) << 48) | ((unsigned long long)(unsigned)w.idx << 16) | seq;
#pragma unroll
    for (int u = 0; u < kMaxPerLane; u++)
      if (lane + 32 * u < C)
        asm volatile("st.volatile.global.v2.u64 [%0], {%1, %2};" ::"l"(inbox + (size_t)(lane + 32 * u) * C + rank), "l"(ra), "l"(rb)
                     : "memory");
  }
  if (w.idx != kNone) {
    const double *src = A + (size_t)((w.idx - 1) / C) * ldA;
    uint4 *dst = pub + (size_t)rank * ldA;
    for (int c = threadIdx.x; c < ldA; c += NT) {
      const double v = src[c];
      asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst + c), "r"((unsigned)__double2loint(v)), "r"(rseq),
                   "r"((unsigned)__double2hiint(v)), "r"(rseq)
                   : "memory");
    }
  }
  if (threadIdx.x < 32) {
    const int lane = threadIdx.x;
    GS_MARK(6);
    const unsigned long long nk = no_key<kMax>();
    unsigned long long bk = nk;
    int bi = kNone;
    unsigned pending = 0, spins = 0;
#pragma unroll
    for (int u = 0; u < kMaxPerLane; u++)
      if (lane + 32 * u < C) pending |= 1u << u;
    while (pending) {
      if (++spins > (1u << 22)) {  // seconds: a CTA of the grid is gone (cannot happen in a cooperative launch)
        bi = kGiveUp;
        break;
      }
      unsigned long long ra[kMaxPerLane], rb[kMaxPerLane];
#pragma unroll
      for (int u = 0; u < kMaxPerLane; u++)
        if ((pending >> u) & 1u)
          asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(ra[u]), "=l"(rb[u]) : "l"(slots + lane + 32 * u) : "memory");
#pragma unroll
      for (int u = 0; u < kMaxPerLane; u++)
        if (((pending >> u) & 1u) && (ra[u] & 0xffffULL) == seq && (rb[u] & 0xffffULL) == seq) {
          pending &= ~(1u << u);
          const unsigned long long k = (ra[u] & ~0xffffULL) | (rb[u] >> 48);
          const int i = (int)(unsigned)(rb[u] >> 16);
          if (i != kNone && (bi == kNone || (kMax ? k > bk : k < bk) || (k == bk && i < bi))) {
            bk = k;
            bi = i;
          }
        }
    }
    const bool gave_up = __any_sync(0xffffffffu, bi == kGiveUp);
    if (bi == kNone || gave_up) bk = nk;
    const int row = gave_up ? kGiveUp : warp_best<kMax>((unsigned)(bk >> 32), (unsigned)bk, gave_up ? kNone : bi).idx;
    if (lane == 0) *s_row = row;
  }
  __syncthreads();
  int row = *s_row;
  if (yt) {  // the wait belongs to the caller's slot: restart the clock for the staging part
    const long long now_ = clock64();
    yt[8] += now_ - *yt_last;
    *yt_last = now_;
  }
  bool bad = false;
  if (row != kNone && row != kGiveUp) {  // the winner's row: every thread polls the slots of its own cells
    const int owner = (row - 1) % C;
    const uint4 *src = pub + (size_t)owner * ldA;
    // (kRowU = the most slots a thread of this instantiation can own: all of them in ONE flight -- 2049 columns / 256
    // threads are 8.02 slots per thread, and a second pass for the last four cells was a second round trip to L2 per pivot)
    for (int c0 = 0; c0 < ldA; c0 += kRowU * NT) {
      unsigned pend = 0, spins = 0;
#pragma unroll
      for (int u = 0; u < kRowU; u++)
        if (c0 + u * NT + (int)threadIdx.x < ldA) pend |= 1u << u;
      while (pend) {
        if (++spins > (1u << 22)) {
          bad = true;
          break;
        }
        uint4 v[kRowU];
#pragma unroll
        for (int u = 0; u < kRowU; u++)
          if ((pend >> u) & 1u)
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(v[u].x), "=r"(v[u].y), "=r"(v[u].z), "=r"(v[u].w)
                         : "l"(src + c0 + u * NT + threadIdx.x)
                         : "memory");
#pragma unroll
        for (int u = 0; u < kRowU; u++)
          if (((pend >> u) & 1u) && v[u].y == rseq && v[u].w == rseq) {
            pend &= ~(1u << u);
            prow_s[c0 + u * NT + threadIdx.x] = __hiloint2double((int)v[u].z, (int)v[u].x);
          }
      }
    }
  }
  if (__syncthreads_or(bad)) row = kGiveUp;
  GS_MARK(7);
#undef GS_MARK
  return row;
}

template <int NWC, int KC, int NWR, bool kGrid = false>
__global__ void __launch_bounds__(NWC *NWR * 32, 1) k_simplex_cluster(const BatchArgs a) {
  constexpr int NTC = NWC * 32, NW = NWC * NWR, NT = NW * 32, VW = 2;
  constexpr int RU = KC >= 4 ? 1 : 4 / KC;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  cg::cluster_group cluster = cg::this_cluster();
  const int C = kGrid ? (int)gridDim.x : (int)cluster.num_blocks();
  const int rank = kGrid ? (int)blockIdx.x : (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, ctid = tid % NTC, rg = tid / NTC;
  const long long cid = kGrid ? 0 : blockIdx.x / C, ncl = kGrid ? 1 : gridDim.x / C;  // KG: the LPs one after the other
  unsigned long long epoch = 0;
  unsigned xcount = 0;  // KG: selections so far in this launch (sequence numbers of the record slots)
  __shared__ int s_row;
  auto scope_sync = [&]() {
    if (kGrid)
      grid_sync_lean(a.counter, epoch);
    else
      cluster.sync();
  };
  const double INF = d_inf();

  for (long long lp0 = cid; lp0 < a.n; lp0 += ncl) {
    const long long lp = a.index ? a.index[lp0] : lp0;
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
    const ClusterSmem L(a.Hcap, a.Wcap, C);
    double *__restrict__ A = reinterpret_cast<double *>(smem_raw + L.off_A);
    double *__restrict__ obj = reinterpret_cast<double *>(smem_raw + L.off_obj);
    double *prow_s = reinterpret_cast<double *>(smem_raw + L.off_prow);
    double *cc = reinterpret_cast<double *>(smem_raw + L.off_cc);
    int *list = reinterpret_cast<int *>(smem_raw + L.off_list);
    int *cnt = reinterpret_cast<int *>(smem_raw + L.off_cnt);
    unsigned *red = reinterpret_cast<unsigned *>(smem_raw + L.off_red);
    uint4 *xch = reinterpret_cast<uint4 *>(smem_raw + L.off_xch);
    int *var = reinterpret_cast<int *>(smem_raw + L.off_var);
    const int ldA = SmemLayout::ld_for(W), Wm1 = W - 1;
    const int bslot = ldA - 2;                                          // RHS cell of a row
    const int nloc = (H - 1 > rank) ? (H - 1 - rank + C - 1) / C : 0;   // local rows: r = 1 + rank + l*C
    int *hist = a.hist ? a.hist + (size_t)blockIdx.x * 2 * a.hist_cap : nullptr;
    double *scratch = a.cl_scratch + (size_t)cid * 2 * C * L.ldA;  // [2][C][ldA] published candidate rows

    // ---- load: local rows and the private objective-row copy, reference layout -> [ A | pad | b | s ]
    {
      const double *src = a.in + moff;
      const int warp = tid >> 5;
      for (int l = warp; l <= nloc; l += NW) {  // l == nloc: the objective row
        const int r = l < nloc ? 1 + rank + l * C : 0;
        double *drow = l < nloc ? A + (size_t)l * ldA : obj;
        const double *g = src + (size_t)r * W;
        if (lane == 0) cp_async8(drow + bslot, g);
        for (int c = lane; c < Wm1; c += 32) cp_async8(drow + c, g + 1 + c);
        for (int c = Wm1 + lane; c < bslot; c += 32) drow[c] = 0.0;  // padding cells
      }
      for (int k = tid; k < W + H; k += NT) var[k] = a.var_in ? a.var_in[poff + k] : k;
      if (tid == 0) *cnt = 0;
      cp_async_wait_all();
    }
    __shared__ __align__(8) unsigned long long s_mbar;
    unsigned mphase = 0;
    const int tma_mode = kGrid ? 0 : a.tma_mode;
    if (tma_mode && tid == 0) mbar_init(&s_mbar, 1);
    __syncthreads();
    scope_sync();

    LpResult res;
    res.status = ST_CYCLED;
    res.value = d_nan();
    res.p1 = res.p2 = 0;
    res.rows = 0;  // this CTA's share of the rewritten rows (CTA 0 also counts the objective row)
    int phase = 1, parity = 0, xpar = 0, hist_len = 0;
    long long iter = 0;
    const double precision = a.precision;
    const long long budget = !(a.max_pivots > 0.0) ? 0LL
                                                    : (a.max_pivots >= 9.0e18 ? 0x7fffffffffffffffLL : (long long)ceil(a.max_pivots));

#ifdef YALPS_TIMING
    long long yt[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, yt_last = clock64();
#define CT_MARK(k) do { const long long now_ = clock64(); yt[k] += now_ - yt_last; yt_last = now_; } while (0)
#define GS_TIMING_ARGS , yt, &yt_last
#else
#define CT_MARK(k)
#define GS_TIMING_ARGS
#endif
    for (;;) {
      if (iter >= budget) break;  // per-phase budget exhausted -> "cycled" (:102,:141)
      int row, col;
      if (phase == 1) {
        // leaving row: first index of the most negative RHS below -precision (:111-119)
        double bv = INF;
        int bi = kNone;
        for (int l = tid; l < nloc; l += NT) {
          const double v = A[(size_t)l * ldA + bslot];
          if (v < -precision && v < bv) {
            bv = v;
            bi = 1 + rank + l * C;
          }
        }
        if (kGrid)
          row = grid_select<false, NW, (2 * KC * NTC + 4 + NT - 1) / NT>(C, rank, bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity, a.gx_slots, xcount,
                                       A, ldA, scratch, prow_s, &s_row GS_TIMING_ARGS);
        else
          row = cluster_select<false, NW>(cluster, C, rank, bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity, xch,
                                          xpar, A, ldA, scratch, prow_s, tma_mode, &s_mbar, &mphase);
        CT_MARK(0);
        if (kGrid && row == kGiveUp) {
          res.status = ST_ERR_PEER;
          break;
        }
        if (row == kNone) {  // feasible: phase 2 with a fresh counter and history (:120, :67-69)
          phase = 2;
          iter = 0;
          hist_len = 0;
          continue;
        }
        // entering column: first index of max -M[0,c]/M[row,c] over M[row,c] < -precision (:123-134); every CTA
        // scans all columns of the staged pivot row itself
        bv = -INF;
        bi = kNone;
        {
          // (KC blocks of NT column pairs cover the row: NT >= NTC.  Branch-free batch form of the divisions, fastdiv.cuh:
          // the quotients of a thread overlap and share one acceptance test; the exact division runs out of line)
          const double *prow = prow_s;
          double ratio[KC][VW], coefs[KC][VW], nums[KC][VW];
          unsigned use = 0;
          bool ok = true;
#pragma unroll
          for (int k = 0; k < KC; k++) {
            const int j0 = VW * (tid + NT * k);
            double2 cf = make_double2(0.0, 0.0), ob = make_double2(0.0, 0.0);
            if (j0 < Wm1) {
              cf = *reinterpret_cast<const double2 *>(prow + j0);
              ob = *reinterpret_cast<const double2 *>(obj + j0);
            }
#pragma unroll
            for (int e = 0; e < VW; e++) {
              coefs[k][e] = e ? cf.y : cf.x;
              nums[k][e] = -(e ? ob.y : ob.x);
              const bool u = j0 + e < Wm1 && coefs[k][e] < -precision;
              RecipBatch d(coefs[k][e], u);
              ratio[k][e] = d.quot(nums[k][e], u);
              ok = ok && d.ok;
              use |= (u ? 1u : 0u) << (k * VW + e);
            }
          }
          if (!ok) {  // rare
#pragma unroll
            for (int k = 0; k < KC; k++)
#pragma unroll
              for (int e = 0; e < VW; e++)
                if ((use >> (k * VW + e)) & 1u) ratio[k][e] = div_rn_slow(nums[k][e], coefs[k][e]);
          }
#pragma unroll
          for (int k = 0; k < KC; k++)
#pragma unroll
            for (int e = 0; e < VW; e++)
              if (((use >> (k * VW + e)) & 1u) && ratio[k][e] > bv) {  // bv starts at -inf: -inf and NaN ratios never win, as in the reference
                bv = ratio[k][e];
                bi = VW * (tid + NT * k) + e + 1;
              }
        }
        col = block_best<true, NW>(bi == kNone ? no_key<true>() : order_key(bv), bi, red, parity);
        CT_MARK(1);
        if (col == kNone) {
          res.status = ST_INFEASIBLE;
          break;
        }
      } else {
        // entering column: first index of the largest reduced cost above precision (:71-79), private objective copy
        double bv = -INF;
        int bi = kNone;
#pragma unroll
        for (int k = 0; k < KC; k++) {
          const int j0 = VW * (ctid + NTC * k);
          if (j0 < Wm1) {
            const double2 ob = *reinterpret_cast<const double2 *>(obj + j0);
#pragma unroll
            for (int e = 0; e < VW; e++) {
              const double v = e ? ob.y : ob.x;
              if (j0 + e < Wm1 && v > precision && v > bv) {
                bv = v;
                bi = j0 + e + 1;
              }
            }
          }
        }
        {
          const unsigned long long key = bi == kNone ? no_key<true>() : order_key(bv);
          if (NWC == 1)
            col = warp_best<true>((unsigned)(key >> 32), (unsigned)key, bi).idx;
          else
            col = block_best<true, NW>(key, bi, red, parity);
        }
        CT_MARK(0);
        if (col == kNone) {
          res.status = ST_OPTIMAL;
          res.value = round_to_precision(obj[bslot], precision);
          break;
        }
        // leaving row: ratio test with the reference's early break (:83-95) == lowest r whose ratio is
        // <= precision if any, else first index of the minimum ratio.  Ratios <= precision get key -inf.
        bv = INF;
        bi = kNone;
        for (int l = tid; l < nloc; l += NT) {
          const double v = A[(size_t)l * ldA + (col - 1)];
          if (v > precision) {
            const double ratio = div_rn(A[(size_t)l * ldA + bslot], v);
            if (ratio < INF) {  // +inf and NaN never win (`ratio < minRatio` with minRatio = Infinity)
              const double key = (ratio <= precision) ? -INF : ratio;
              if (bi == kNone || key < bv) {
                bv = key;
                bi = 1 + rank + l * C;
              }
            }
          }
        }
        if (kGrid)
          row = grid_select<false, NW, (2 * KC * NTC + 4 + NT - 1) / NT>(C, rank, bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity, a.gx_slots, xcount,
                                       A, ldA, scratch, prow_s, &s_row GS_TIMING_ARGS);
        else
          row = cluster_select<false, NW>(cluster, C, rank, bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity, xch,
                                          xpar, A, ldA, scratch, prow_s, tma_mode, &s_mbar, &mphase);
        CT_MARK(1);
        if (kGrid && row == kGiveUp) {
          res.status = ST_ERR_PEER;
          break;
        }
        if (row == kNone) {
          res.status = ST_UNBOUNDED;
          res.value = (double)col;
          break;
        }
      }

      if (a.check_cycles) {  // (:98, :137); every CTA keeps its own (identical) history
        if (hist_len >= a.hist_cap) {
          res.status = ST_ERR_HISTORY;
          break;
        }
        if (tid == 0) {
          hist[2 * hist_len] = var[W + row];
          hist[2 * hist_len + 1] = var[col];
        }
        hist_len++;
        __syncthreads();
        if (history_has_cycle<NT>(hist, hist_len)) break;  // "cycled", NaN
      }

      // ================= pivot (src/simplex.ts:5-39) =================
      {
        const int jc = col - 1;
        const int owner = (row - 1) % C, lrow = (row - 1) / C;
        const double *prow = prow_s;
        // every load of this phase first: pivot element, pivot row cells and its RHS (staged copy), local column cell
        const double q = prow[jc];
        const double braw = prow[bslot];
        double2 v[KC];
#pragma unroll
        for (int k = 0; k < KC; k++)
          if (VW * (ctid + NTC * k) < Wm1) v[k] = *reinterpret_cast<const double2 *>(prow + VW * (ctid + NTC * k));
        const double coef0 = obj[jc];
        double cell0 = 0.0;
        if (tid < nloc) cell0 = A[(size_t)tid * ldA + jc];
        const Recip rq(q);

        // (branch-free batch form of the divisions, fastdiv.cuh: the quotients of a thread overlap and share ONE acceptance
        // test -- a test-and-branch per quotient made this stage ~2,000 cycles of every CTA's critical path)
        RecipBatch rb(q, rq.r);
        double p[KC][VW];
        unsigned st = 0, full = 0, valid = 0, partial = 0, live = 0;
        int jc_off = -1;
#pragma unroll
        for (int k = 0; k < KC; k++) {
          const int j0 = VW * (ctid + NTC * k);
#pragma unroll
          for (int e = 0; e < VW; e++) {
            const int j = j0 + e;
            const double x = (j == jc) ? 1.0 : (e ? v[k].y : v[k].x);
            const bool use = j < Wm1 && fabs(x) > kTiny;
            p[k][e] = rb.quot(x, use);
            live |= (use ? 1u : 0u) << (k * VW + e);
            if (j < Wm1) {
              valid |= 1u << (k * VW + e);
              if (j == jc) jc_off = VW * NTC * k + e;
            }
          }
        }
        const bool nz0 = fabs(braw) > kTiny;
        double p0 = rb.quot(braw, nz0);  // normalised RHS of the pivot row (:19 for c = 0)
        if (!rb.ok) {  // rare: exact divisions out of line
#pragma unroll
          for (int k = 0; k < KC; k++)
#pragma unroll
            for (int e = 0; e < VW; e++)
              if ((live >> (k * VW + e)) & 1u)
                p[k][e] = div_rn_slow((VW * (ctid + NTC * k) + e == jc) ? 1.0 : (e ? v[k].y : v[k].x), q);
          if (nz0) p0 = div_rn_slow(braw, q);
        }
        if (!nz0) p0 = 0.0;
#pragma unroll
        for (int k = 0; k < KC; k++) {
          const int j0 = VW * (ctid + NTC * k);
#pragma unroll
          for (int e = 0; e < VW; e++) {
            if (!((live >> (k * VW + e)) & 1u)) p[k][e] = 0.0;
            if ((live >> (k * VW + e)) & 1u)
              st |= 1u << (k * VW + e);
            else if (j0 + e >= Wm1 && j0 < Wm1)
              st |= 1u << (k * VW + e);  // padding cell next to the last column: rewriting it is harmless
          }
          const unsigned m = (st >> (k * VW)) & 3u;
          if (m == 3u)
            full |= 1u << k;
          else if (m)
            partial = 1u;
        }
        CT_MARK(2);

        // ---- local pivot-column cells: -coef/q (:36) and the compacted list of local rows to rewrite (:31)
        for (int l0 = 0; l0 < nloc; l0 += NT) {
          const int l = l0 + tid;
          bool act = false;
          double cell = 0.0, quo = 0.0;
          if (l < nloc && !(owner == rank && l == lrow)) {
            cell = l0 == 0 ? cell0 : A[(size_t)l * ldA + jc];
            const double num = -cell;
            act = fabs(num) > kTiny;  // also false for NaN, as in the reference
            quo = act ? rq.quot(num) : 0.0;
          }
          const unsigned m = __ballot_sync(0xffffffffu, act);
          if (m) {
            int base = 0;
            if (lane == 0) base = atomicAdd(cnt, __popc(m));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (act) {
              const int k = base + __popc(m & ((1u << lane) - 1u));
              list[k] = l;
              *reinterpret_cast<double2 *>(cc + 2 * k) = make_double2(cell, quo);
            }
          }
        }
        if (tid == 0) {  // basis bookkeeping (:7-12), every CTA for itself
          const int leaving = var[W + row];
          var[W + row] = var[col];
          var[col] = leaving;
        }
        __syncthreads();
        const int R = *cnt;
        const bool any_partial = __any_sync(0xffffffffu, partial);
        res.rows += (unsigned)(R + ((rank == 0 && fabs(coef0) > kTiny) ? 1 : 0));
        CT_MARK(3);

        if (rg == NWR - 1) {
          // RHS cells of the local active rows (:34 for c = 0)
          if (nz0) {
            for (int i = ctid; i < R; i += NTC) {
              const int l = list[i];
              const double x = A[(size_t)l * ldA + bslot];
              A[(size_t)l * ldA + bslot] = __dsub_rn(x, __dmul_rn(cc[2 * i], p0));
            }
          }
          // private objective row: the same update every CTA applies to its copy
          if (fabs(coef0) > kTiny) {
            const double cnew0 = rq.quot(-coef0);
            double *orow = obj + VW * ctid;
#pragma unroll
            for (int k = 0; k < KC; k++) {
              const unsigned m = (st >> (k * VW)) & 3u;
              if (m) {
                double *dst = orow + (size_t)VW * NTC * k;
                const double2 x = *reinterpret_cast<const double2 *>(dst);
                double t0 = __dsub_rn(x.x, __dmul_rn(coef0, p[k][0]));
                double t1 = __dsub_rn(x.y, __dmul_rn(coef0, p[k][1]));
                if (jc_off == VW * NTC * k) t0 = cnew0;
                if (jc_off == VW * NTC * k + 1) t1 = cnew0;
                if (m & 1u) dst[0] = t0;
                if (m & 2u) dst[1] = t1;
              }
            }
            if (ctid == NTC - 1 && nz0) obj[bslot] = __dsub_rn(obj[bslot], __dmul_rn(coef0, p0));
          }
        }
        CT_MARK(4);
        // ---- rank-1 update of the local active rows, pivot-column cell included
        if (any_partial)
          update_split<NTC, KC, VW, RU, NWR, true>(A + VW * ctid, ldA, R, rg, list, cc, p, st, full, jc_off);
        else
          update_split<NTC, KC, VW, RU, NWR, false>(A + VW * ctid, ldA, R, rg, list, cc, p, st, full, jc_off);
        CT_MARK(5);
        // ---- the owner writes the normalised pivot row back (:19,22,25); peers only ever read the published copy
        if (owner == rank && rg == 0) {
          double *Arow = A + (size_t)lrow * ldA + VW * ctid;
#pragma unroll
          for (int k = 0; k < KC; k++)
            if ((valid >> (k * VW)) & 1u) *reinterpret_cast<double2 *>(Arow + (size_t)VW * NTC * k) = make_double2(p[k][0], p[k][1]);
          if (ctid == 0) A[(size_t)lrow * ldA + bslot] = p0;
        }
        __syncthreads();
        if (tid == 0) *cnt = 0;
        CT_MARK(7);
      }
      if (phase == 1)
        res.p1++;
      else
        res.p2++;
      iter++;
    }

    // ---- outputs (every CTA its own rows; CTA 0 the scalars, the objective row and the basis)
    scope_sync();
    if (a.rows_out && tid == 0 && res.rows != 0) atomicAdd(a.rows_out + (a.rows_per_lp ? lp : 0), res.rows);
    if (rank == 0) {
      if (tid == 0) {
        if (a.status) a.status[lp] = res.status;
        if (a.value) a.value[lp] = res.value;
        if (a.pivots) {
          a.pivots[2 * lp] = res.p1;
          a.pivots[2 * lp + 1] = res.p2;
        }
        if (a.rhs_out) a.rhs_out[roff] = obj[bslot];
      }
      if (a.pos_out)
        for (int k = tid; k < W + H; k += NT) a.pos_out[poff + var[k]] = k;
      if (a.var_out)
        for (int k = tid; k < W + H; k += NT) a.var_out[poff + k] = var[k];
      if (a.red_out)  // the private objective row: column k >= 1 is obj[k - 1]
        for (int k = tid; k < W + H; k += NT) a.red_out[poff + var[k]] = (k >= 1 && k < W) ? obj[k - 1] : 0.0;
      if (a.mat_out)
        for (int c = tid; c < W; c += NT) a.mat_out[moff + c] = (c == 0) ? obj[bslot] : obj[c - 1];
    }
    if (a.rhs_out)
      for (int l = tid; l < nloc; l += NT) a.rhs_out[roff + 1 + rank + l * C] = A[(size_t)l * ldA + bslot];
#ifdef YALPS_TIMING
    __syncthreads();
    if (a.rhs_out && rank == 0 && (tid == 0 || tid == NT - 1)) {  // debug builds only: overwrite the RHS output (H >= 20)
      double *o = a.rhs_out + roff + (tid == 0 ? 0 : 10);
      for (int k = 0; k < 8; k++) o[k] = (double)yt[k];
      o[8] = (double)(res.p1 + res.p2);
      o[9] = (double)yt[8];  // KG: wait for the selection records
    }
#endif
    if (a.mat_out) {
      for (int l = tid >> 5; l < nloc; l += NW) {
        const double *sA = A + (size_t)l * ldA;
        double *dr = a.mat_out + moff + (size_t)(1 + rank + l * C) * W;
        for (int c = lane; c < W; c += 32) dr[c] = (c == 0) ? sA[bslot] : sA[c - 1];
      }
    }
    scope_sync();  // nobody may start overwriting its shared memory while a peer is still in this LP
  }
}

}  // namespace yalps
