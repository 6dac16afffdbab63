// certificate_kernel.cuh -- k_certificate: Farkas certificates of infeasible LPs and unbounded rays of unbounded LPs
// from their final tableaus (a post-pass over tableaus already in device memory; yalps_b200/sensitivity.py
// certificate_from_tableau is the specification).
//
// Per variable id v, packed like pos_out:
//   infeasible (status 1): r = the row phase 1 chose, the lowest r in 1..H-1 whose M[r,0] is the minimum over the rows
//     with M[r,0] < -precision (NaN never qualifies, -inf does).  Phase 1 ends `infeasible` on that row without
//     pivoting, so the final tableau is the tableau of that choice.
//       cert[0] = M[r,0], cert[W] = +0, cert[v] = M[r,pos[v]] (1 <= pos[v] < W), 1 (pos[v] == W+r), +0 otherwise
//   unbounded (status 2): c = (int)value, the entering column phase 2 found no leaving row for.
//       cert[0] = M[0,c], cert[W] = +0, cert[v] = 1 (pos[v] == c), -M[pos[v]-W, c] (W < pos[v] < W+H), +0 otherwise
//   every other status, an infeasible LP without a qualifying row, c outside 1..W-1: NaN.
// The row choice is the simplex kernels' arg-reduction on order_key, so ties, NaN and +-inf resolve as in the
// reference's strict-< scan.  Cells are moved as 64-bit integers (negated by flipping the sign bit), never as doubles:
// a floating-point negation or select may be emitted as an FP add, which would turn every NaN into the canonical one.
//
// One warp per LP up to k_ranging's warp-mode bound, one CTA per LP above it.  A thread group reads column 0 (an
// infeasible LP only), pos, then row r or column c of its LP once, and writes cert by id; no atomics.
#pragma once

#include "ranging_kernel.cuh"

namespace yalps {

constexpr int kCertThreads = 256;

struct CertArgs : PostArgs {
  const double *value;  // per LP, as the solve reports it (the entering column of an unbounded LP)
  double precision;
  double *cert;         // output, packed like pos_out
};

constexpr long long kCertOne = 0x3ff0000000000000LL;  // bits of 1.0
constexpr long long kCertNaN = 0x7ff8000000000000LL;  // bits of the NaN fill
constexpr long long kCertSign = (long long)0x8000000000000000ULL;

// LP i on NW warps (NW == 1: one warp); t = the thread's index among them
template <int NW>
__device__ __forceinline__ void cert_lp(const CertArgs &a, long long i, int t, unsigned *red, int &parity) {
  constexpr int NT = NW * 32;
  const PostLP P = post_lp(a, i);
  const int H = P.H, W = P.W;
  const double *M = a.M + P.mo;
  const int *pos = a.pos + P.po;
  long long *cert = reinterpret_cast<long long *>(a.cert + P.po);
  const int st = a.status[P.id];  // uniform over the group, like everything that decides r and c
  int r = kNone, c = kNone;
  if (st == ST_INFEASIBLE) {
    // src/simplex.ts:111-119: first index of the most negative RHS below -precision
    double bv = d_inf();
    int bi = kNone;
    for (int k = 1 + t; k < H; k += NT) {
      const double v = M[(long long)k * W];
      if (v < -a.precision && v < bv) {
        bv = v;
        bi = k;
      }
    }
    r = block_best<false, NW>(bi == kNone ? no_key<false>() : order_key(bv), bi, red, parity);
  } else if (st == ST_UNBOUNDED) {
    const double x = a.value[P.id];
    if (x >= 1.0 && x < (double)W) c = (int)x;  // NaN fails both tests
  }
  const long long *Mb = reinterpret_cast<const long long *>(M);
  const long long *row = Mb + (long long)(r == kNone ? 0 : r) * W;
  for (int v = t; v < W + H; v += NT) {
    long long y = kCertNaN;
    if (r != kNone) {
      const int p = pos[v];
      y = v == 0 ? row[0] : v == W ? 0 : (p >= 1 && p < W) ? row[p] : p == W + r ? kCertOne : 0;
    } else if (c != kNone) {
      const int p = pos[v];
      y = v == 0                 ? Mb[c]
          : v == W               ? 0
          : p == c               ? kCertOne
          : p > W && p < W + H   ? Mb[(long long)(p - W) * W + c] ^ kCertSign
                                 : 0;
    }
    cert[v] = y;
  }
}

__global__ void __launch_bounds__(kCertThreads) k_certificate(CertArgs a, int warp_mode) {
  __shared__ unsigned red[192];  // block_best's cross-warp scratch (CTA mode)
  int parity = 0;
  if (warp_mode) {
    constexpr int kWarps = kCertThreads / 32;
    const long long warps = (long long)gridDim.x * kWarps;
    for (long long i = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5); i < a.n; i += warps)
      cert_lp<1>(a, i, threadIdx.x & 31, red, parity);
  } else {
    for (long long i = blockIdx.x; i < a.n; i += gridDim.x) cert_lp<kCertThreads / 32>(a, i, threadIdx.x, red, parity);
  }
}

// The rows a Farkas certificate uses (yalps_solve_row_subsets, the IIS search): bit r of support[i*words + r/32] is
// set when LP i is infeasible and cert[i*(W+H) + W + r] > +0.0, rows 1..H-1 (the raw value: NaN and both zeros do not
// count, noise above zero does); count[i] is the number of bits set.  Every other LP gets zero words.  Uniform batches
// only.  One warp per LP: lane l reads row 32k + l, the ballot is word k.
__global__ void k_cert_support(long long n, int H, int W, int words, const int *status, const double *cert,
                               unsigned *support, int *count) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long i = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
    const bool inf = status[i] == ST_INFEASIBLE;
    const double *y = cert + i * (long long)(W + H) + W;
    int total = 0;
    for (int k = 0; k < words; k++) {
      const int r = 32 * k + lane;
      const unsigned m = __ballot_sync(0xffffffffu, inf && r >= 1 && r < H && y[r] > 0.0);
      if (lane == 0) support[i * words + k] = m;
      total += __popc(m);
    }
    if (lane == 0) count[i] = total;
  }
}

}  // namespace yalps
