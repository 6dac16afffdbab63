// yalps_b200.cu -- C ABI (include/yalps_b200.h) over the sm_100a kernels.
//
// Host runtime: context, device buffer pool, double-buffered chunked H2D -> kernel -> D2H pipeline,
// kernel-path selection, and the branch-and-cut driver (speculative node waves replayed in the
// reference's pop order, src/branchAndCut.ts:89-176).
#include "../../include/yalps_b200.h"

#include <cuda_runtime.h>

#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only: libnccl.so.2 is opened at run time (multi.inl)

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <condition_variable>
#include <functional>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "kernel_table.h"
#include "aux_kernels.cuh"
#include "cluster_kernel.cuh"
#include "grid_kernel.cuh"
#include "multigrid_kernel.cuh"
#include "certificate_kernel.cuh"
#include "ranging_kernel.cuh"
#include "tmem_launch.h"
#include "bnb_launch.h"

using namespace yalps;

namespace {

thread_local std::string g_create_error;

// cudaFuncAttributeMaxDynamicSharedMemorySize is a property of the function on the device, shared by every ctx of
// the process: it is only ever raised, under a lock (several contexts may run on different host threads).
std::mutex g_attr_mutex;
std::unordered_map<std::string, int> g_smem_attr;

cudaError_t raise_smem_limit(int device, const void *fn, int bytes) {
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  int &cur = g_smem_attr[std::to_string(device) + ":" + std::to_string((size_t)fn)];
  if (bytes <= cur) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}

// The dynamic shared memory a launch of fn can have: the per-block opt-in limit less fn's static shared memory
// (k_simplex and the cluster kernels: 16 bytes).  A carve-up is checked against this, not the opt-in limit itself --
// at the tallest tableau of a kernel the difference decides between a launch and a failing cudaFuncSetAttribute.
size_t dynamic_smem_limit(int device, int optin, const void *fn) {
  std::lock_guard<std::mutex> lock(g_attr_mutex);
  static std::unordered_map<std::string, int> static_bytes;
  const std::string key = std::to_string(device) + ":" + std::to_string((size_t)fn);
  auto it = static_bytes.find(key);
  if (it == static_bytes.end()) {
    cudaFuncAttributes a{};
    const int s = cudaFuncGetAttributes(&a, fn) == cudaSuccess ? (int)a.sharedSizeBytes : 0;
    it = static_bytes.emplace(key, s).first;
  }
  return (size_t)std::max(0, optin - it->second);
}

struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct Root {
  bool valid = false;
  int H = 0, W = 0, max_extra = 0;
  double density = 1.0;  // fraction of non-zero cells of (a sample of) the root-optimal tableau
  DevBuf m, pos, var;
  std::vector<double> h_m;  // host copy of column 0 is enough for the driver, but keep rhs + pos + var
  std::vector<double> h_rhs;
  std::vector<int32_t> h_pos, h_var;
};

}  // namespace

struct yalps_ctx {
  int device = 0;
  cudaDeviceProp prop{};
  int smem_optin = 0;
  std::string error;
  cudaStream_t streams[2]{};
  cudaEvent_t events[2]{};
  int64_t launches = 0;
  int tune_path = 0, tune_threads = 0, tune_rows = 0;
  std::vector<cudaStream_t> aux_streams;  // concurrent K4 launches of one node wave
  std::vector<cudaEvent_t> aux_events;
  cudaEvent_t fork_event = nullptr;
  // YALPS_BNB_DEBUG: where the host spends a node wave (ns): before the first CUDA call, enqueueing, waiting, copying out
  int64_t wave_ns[4] = {0, 0, 0, 0};
  int wave = 256;  // upper bound of the adaptive look-ahead of the branch-and-cut driver
  int kc_tma = 0;    // KC: staging of the winner's pivot row (YALPS_KC_TMA: 0 ld.global.cg, 1 cp.async.bulk, 2 multicast)
  int bnb_mode = 0;  // 0: device-resident search when it fits, else host waves; 1: host waves only; 2: device only
  int bnb_workers = 0;  // device-resident search: worker CTAs (0 = one per SM beside the scheduler; yalps_multi_solve_many
                        // shares the SMs between its concurrent searches)
  int64_t replica_forks = -1;  // last yalps_solve_replicas call: replicas that left the shared path (-1: sharing not used)
  int replica_sharing = 1;  // yalps_solve_replicas: follow the base tableau's pivot path while a replica makes the same choices
  unsigned long long *d_rows = nullptr;  // roofline diagnostics: device counter(s) of rewritten rows (yalps_set_row_counter)
  int rows_per_lp = 0;
  // pooled device buffers (index = purpose * 2 + pipeline slot)
  std::unordered_map<std::string, DevBuf> pool;
  std::unordered_map<std::string, DevBuf> pinned;
  std::unordered_map<std::string, int> occ_cache;
  std::unordered_map<std::string, double> density_cache;
  Root root;
};

namespace {

int fail(yalps_ctx *ctx, int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx)
    ctx->error = buf;
  else
    g_create_error = buf;
  return code;
}

#define CU(ctx, call)                                                                                   \
  do {                                                                                                  \
    cudaError_t e_ = (call);                                                                            \
    if (e_ != cudaSuccess)                                                                              \
      return fail(ctx, YALPS_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

int dev_ensure(yalps_ctx *ctx, const std::string &name, size_t bytes, void **out) {
  DevBuf &b = ctx->pool[name];
  if (b.cap < bytes) {
    if (b.p) CU(ctx, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = std::max(bytes, (size_t)256);
    CU(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
  }
  *out = b.p;
  return 0;
}

int pin_ensure(yalps_ctx *ctx, const std::string &name, size_t bytes, void **out) {
  DevBuf &b = ctx->pinned[name];
  if (b.cap < bytes) {
    if (b.p) CU(ctx, cudaFreeHost(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = std::max(bytes * 2, (size_t)4096);
    CU(ctx, cudaHostAlloc(&b.p, want, cudaHostAllocMapped | cudaHostAllocPortable));
    b.cap = want;
  }
  *out = b.p;
  return 0;
}

// Device-side alias of a buffer from pin_ensure (zero-copy access over PCIe for latency-bound small launches).
int pin_device_ptr(yalps_ctx *ctx, void *host, void **dev) {
  CU(ctx, cudaHostGetDevicePointer(dev, host, 0));
  return 0;
}

// ---- kernel table -------------------------------------------------------------------------------------
// All k_simplex instantiations (kernel_table.h), gathered once.
const std::vector<KernelEntry> &all_kernels() {
  static const std::vector<KernelEntry> table = [] {
    std::vector<KernelEntry> v;
    int n = 0;
    const KernelEntry *t;
    t = kernel_table_base(&n);
    v.insert(v.end(), t, t + n);
    t = kernel_table_split_a(&n);
    v.insert(v.end(), t, t + n);
    t = kernel_table_split_b(&n);
    v.insert(v.end(), t, t + n);
    t = kernel_table_split_c(&n);
    v.insert(v.end(), t, t + n);
    return v;
  }();
  return table;
}

// Thread (row group, t) keeps the pivot-row cells of vector-columns t, t+NTC, ... in registers:
// 32*NWC*KC*VW >= W-1 is required.  Among the kernels with `nwr` row groups: smallest NWC >= nwc_want whose
// widest KC covers the row (else the largest NWC), then the smallest covering KC.
const KernelEntry *pick_kernel(int nwc_want, int nwr, int W, bool resident) {
  const int vw = resident ? 2 : 1;
  const int wm1 = std::max(W - 1, 1);
  const KernelEntry *best = nullptr;
  for (const auto &k : all_kernels()) {
    if (k.nwr != nwr) continue;
    if ((long long)k.nw * 32 * k.kc * vw < wm1) continue;
    if (!best) {
      best = &k;
      continue;
    }
    const bool k_ok = k.nw >= nwc_want, b_ok = best->nw >= nwc_want;
    if (k_ok != b_ok) {
      if (k_ok) best = &k;
      continue;
    }
    if (k_ok) {  // both at least as wide as wanted: prefer the narrower CTA, then the smaller KC
      if (k.nw < best->nw || (k.nw == best->nw && k.kc < best->kc)) best = &k;
    } else {     // both narrower than wanted: prefer the wider CTA, then the smaller KC
      if (k.nw > best->nw || (k.nw == best->nw && k.kc < best->kc)) best = &k;
    }
  }
  return best;
}

// CTA width by tableau size, from scripts/sweep_paths.py on B200 (profiles/r01_sweep_paths.jsonl).
int default_warps(long long cells, bool resident) {
  if (resident) {
    if (cells < 3000) return 1;
    if (cells < 12000) return 2;
    if (cells < 40000) return 4;
    if (cells < 120000) return 8;
    return 16;
  }
  if (cells < 3000) return 1;
  if (cells < 6000) return 2;
  if (cells < 25000) return 4;
  if (cells < 50000) return 8;
  if (cells < 400000) return 16;
  return 32;
}

// ---- kernel path: which kernels a launch takes (choose_route) and how they are enqueued (launch_route) --------------
enum RouteKind {
  ROUTE_K1T,       // K1t: tableau in tensor memory, one LP per warp (tmem_kernel.cuh)
  ROUTE_SIMPLEX,   // k_simplex table: K1/K1s (tableau in shared memory) or K2/K2s (HBM/L2), one LP per CTA
  ROUTE_CLUSTER,   // KC: one LP per thread-block cluster (cluster_kernel.cuh)
  ROUTE_GRID_RES,  // KG: one LP over the cooperative grid, tableau in the SMs' shared memory
  ROUTE_GRID,      // K4: one LP over the cooperative grid, tableau in HBM/L2, the LPs one after another
};

struct Route {
  RouteKind kind = ROUTE_GRID;
  const KernelEntry *k = nullptr;  // SIMPLEX, CLUSTER, GRID_RES
  bool resident = false;   // K1t, K1/K1s; under GRID what the k_simplex plan said (node waves stage their I/O by it)
  bool assembled = false;  // node waves: K3 assembles the nodes before the row-split kernel runs (big, very sparse nodes)
  size_t smem = 0;
  int grid = 0;            // K1T, SIMPLEX: CTAs
  int C = 0;               // CLUSTER: CTAs per cluster; GRID_RES: CTAs
  int clusters = 0;        // CLUSTER: co-resident clusters
};

struct RouteRequest {
  long long n;
  int Hcap, Wcap;
  // fraction of non-zero cells of a sample of the input (< 0 = unknown).  Sparse tableaus skip most of the rank-1
  // update, their pivots are latency-bound, and the HBM/L2-resident kernel wins because it needs no shared memory for
  // the tableau and therefore runs many more LPs per SM (profiles/r01_sweep_paths.jsonl).
  double density = -1.0;
  bool check_cycles = false;
  bool allow_k1t = false;
  // replica leader and forks: the k_simplex kernel as planned, never KC, KG or K4 in its place (GRID only when no
  // kernel of the table is wide enough).  The forks resume mid-solve, which only k_simplex can.
  bool table_only = false;
  // node waves: KC and KG have no node mode (a forced KC path plans as AUTO, a forced KG path as a forced k_simplex
  // one); root_density is that of the root optimum (big-sparse-node rule)
  bool nodes = false;
  double root_density = 1.0;
};

int plan_cluster(yalps_ctx *ctx, int Hcap, int Wcap, Route *r);
int plan_gridres(yalps_ctx *ctx, int Hcap, int Wcap, Route *r);

// The kernel path of one launch of q.n LPs of at most q.Hcap x q.Wcap: the tuning of yalps_set_tuning /
// yalps_set_row_groups, the YALPS_* switches, and otherwise the rules measured on B200 (comments below).  A forced path
// that cannot take the tableau fails with YALPS_ERR_TOO_LARGE.
int choose_route(yalps_ctx *ctx, const RouteRequest &q, Route *r) {
  *r = Route{};
  const long long n = q.n;
  const int Hcap = q.Hcap, Wcap = q.Wcap;
  const int path = ctx->tune_path;
  if (!q.nodes && !q.table_only && path == YALPS_PATH_CLUSTER) {
    if (int rc = plan_cluster(ctx, Hcap, Wcap, r)) return rc;
    if (!r->k)
      return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d does not fit the shared memory of a %d-CTA cluster", Hcap, Wcap, kMaxCluster);
    return 0;
  }
  if (!q.nodes && !q.table_only && path == YALPS_PATH_GRID_RESIDENT) {
    if (int rc = plan_gridres(ctx, Hcap, Wcap, r)) return rc;
    if (!r->k)
      return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d does not fit the shared memory of the grid (or is wider than 2049)", Hcap, Wcap);
    return 0;
  }
  // ---- the k_simplex table (and K1t)
  const int tune_path = (path == YALPS_PATH_CLUSTER || path == YALPS_PATH_GRID_RESIDENT) ? (int)YALPS_PATH_AUTO : path;
  SmemLayout Lr(Hcap, Wcap, true, 32), Lg(Hcap, Wcap, false, 32);
  bool resident = Lr.total <= (size_t)ctx->smem_optin;
  // (throughput mode only: with at most two LPs per SM the shared-memory row-split kernels are 3x faster than K2 on
  // sparse Netlib models -- AFIRO, 148 LPs: 46 vs 155 us)
  if (resident && tune_path == YALPS_PATH_AUTO && q.density >= 0.0 && q.density < 0.35 &&
      n > std::max(64LL, 2LL * ctx->prop.multiProcessorCount))
    resident = false;
  if (tune_path == YALPS_PATH_SMEM) {
    if (!resident) return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d does not fit in shared memory", Hcap, Wcap);
  } else if (tune_path == YALPS_PATH_GMEM) {
    resident = false;
  }
  const bool grid_ok = tune_path == YALPS_PATH_GRID || (tune_path == YALPS_PATH_AUTO && n <= 16);
  // K1t (tensor-memory resident, one LP per warp, no CTA barrier in the pivot loop): every batch whose tableaus fit
  // it, whatever its size and density.  Measured against the previous choices on B200: 1.47-1.68x K1 on big dense
  // batches of every shape from 9x17 to 33x65 (scripts/tmem_vs_smem.py); 1.5-2.3x K2 on big batches with 70-90 % zeros
  // (scripts/tmem_sparse_batches.py); 8-33 % faster than the row-split latency kernels for 1..296 LPs, dense or sparse
  // (scripts/tmem_small_batches.py).
  // Tableaus of 34..65 rows take the 256-column shape (8 LPs per SM, scripts/tmem_tall_crossover.py): 1.4-1.85x K1 on
  // big batches, dense or sparse; 10-20 % faster than K1s for 1..296 DENSE LPs, but 26-40 % slower on sparse Netlib
  // models (AFIRO, KLEIN1: the row-split kernels compact the few active rows, one warp walks all blocks) -- so in
  // latency mode the tall shape needs a density probe that says "dense".
  const bool latency_mode = n <= 2LL * ctx->prop.multiProcessorCount;
  // The short shape wins or ties everywhere, very sparse tableaus included (its sparse row pass touches only the
  // active rows: 90 % zeros, 33x65, one LP: 18.8 vs 18.9 us for K1s; scripts/tmem_small_batches.py).
  const bool tmem_auto = tune_path == YALPS_PATH_AUTO && ctx->tune_threads <= 0 && ctx->tune_rows <= 0 &&
                         (!tmem_kernel_is_tall(Hcap) ||
                          (latency_mode ? q.density >= 0.5
                                        // throughput mode (scripts/policy_mid_batches.py): KLEIN1 55x55 (density 0.24) 2.2-2.6x
                                        // the HBM-resident K2; very sparse AFIRO 36x33 (0.1) only while one wave of
                                        // 8 LPs per SM covers the batch, beyond that K2 is 20-30 % faster
                                        : (q.density < 0.0 || q.density >= 0.15 || n <= 8LL * ctx->prop.multiProcessorCount)));
  if (q.allow_k1t && tmem_kernel_fits(Hcap, Wcap) && (tune_path == YALPS_PATH_TMEM || tmem_auto)) {
    r->kind = ROUTE_K1T;
    r->resident = true;
    r->smem = tmem_kernel_dynamic_smem(Hcap);
    CU(ctx, raise_smem_limit(ctx->device, tmem_kernel_fn(Hcap, false, q.check_cycles), (int)r->smem));
    if (ctx->d_rows) CU(ctx, raise_smem_limit(ctx->device, tmem_kernel_fn(Hcap, true, q.check_cycles), (int)r->smem));
    // checkCycles: one history buffer per warp, so one CTA per SM bounds the memory (4 warps x 2 x hist_cap ints each)
    const long long ctas = (long long)(q.check_cycles ? 1 : tmem_kernel_ctas_per_sm(Hcap)) * ctx->prop.multiProcessorCount;
    r->grid = (int)std::max(1LL, std::min(ctas, n));  // few LPs: one per CTA (the kernel deals LP i to CTA i % grid)
    return 0;
  }
  if (tune_path == YALPS_PATH_TMEM)
    return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d does not fit the tensor-memory kernel (max %dx%d, no node mode)",
                Hcap, Wcap, 65, 65);
  r->resident = resident;
  // pivot row/column staging beyond shared memory: only the grid kernel (K4) can take the tableau
  const bool staged = resident || Lg.total <= (size_t)ctx->smem_optin;
  if (!staged && !grid_ok)
    return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d: pivot row/column staging exceeds shared memory", Hcap, Wcap);
  // CTA shape.  Explicit tuning wins; otherwise (scripts/single_lp_latency.py, scripts/sweep_config3.py on B200):
  //  * latency mode (every LP can have an SM to itself): row-split CTAs, sized by the tableau;
  //  * throughput mode: one row group and many CTAs per SM for tableaus in shared memory, a small row split for
  //    the HBM/L2-resident kernel on mid-size tableaus.
  const long long cells = (long long)Hcap * Wcap;
  int want_threads = ctx->tune_threads, want_rows = ctx->tune_rows;
  if (want_threads <= 0 && want_rows <= 0) {
    if (latency_mode) {
      // latency mode wants the row-split layout (compacted row list next to the tableau): a tableau that only fits
      // shared memory without it is better off on the cluster / HBM-resident split kernels than on one-row-group K1
      if (resident && tune_path == YALPS_PATH_AUTO && SmemLayout(Hcap, Wcap, true, 16, true).total > (size_t)ctx->smem_optin)
        resident = false;
      if (!resident) {
        want_threads = 512, want_rows = 4;
      } else if (cells < 2500) {
        want_threads = 128, want_rows = 4;
      } else if (cells < 4000) {
        want_threads = 256, want_rows = 8;
      } else if (cells < 12000) {
        want_threads = 256, want_rows = 4;
      } else {
        want_threads = 512, want_rows = 8;
      }
    } else if (!resident) {
      // (with the RHS column and the basis in shared memory a pivot of the split kernel waits on L2 less often, and one
      // column warp per row group -- twice the cells per thread and row -- beats two: SC105 78.5 -> 81.8, ADLITTLE
      // 139.8 -> 151.1 M pivots/s, profiles/r02u_sweep_config3.jsonl)
      if (cells >= 5000) want_threads = Wcap <= 129 ? 64 : 128, want_rows = 2;
    }
  }
  const bool small_for_grid = !resident && cells < 40000;  // few LPs outside shared memory, yet one row-split CTA beats K4
  const int nw = want_threads > 0 ? std::max(1, want_threads / 32) : default_warps(cells, resident);
  int nwr = want_rows > 0 ? want_rows : 1;
  const KernelEntry *k = nullptr;
  if (staged && nwr > 1) {
    k = pick_kernel(std::max(1, nw / nwr), nwr, Wcap, resident);
    if (k && SmemLayout(Hcap, Wcap, resident, k->nw * k->nwr, true).total >
                 dynamic_smem_limit(ctx->device, ctx->smem_optin, (const void *)(resident ? k->resident : k->global)))
      k = nullptr;
  }
  if (staged && !k) {
    nwr = 1;
    k = pick_kernel(nw, 1, Wcap, resident);
    // (the staging checks above use the 32-warp carve-up; the kernel's own static shared memory comes on top)
    if (k && SmemLayout(Hcap, Wcap, resident, k->nw, false).total >
                 dynamic_smem_limit(ctx->device, ctx->smem_optin, (const void *)(resident ? k->resident : k->global))) {
      if (!grid_ok) return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d does not fit in shared memory", Hcap, Wcap);
      k = nullptr;
    }
  }
  if (!k && !grid_ok) return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau width %d exceeds the widest kernel", Wcap);
  if (k) {
    SimplexKernel fn = resident ? k->resident : k->global;
    const size_t smem = SmemLayout(Hcap, Wcap, resident, k->nw * k->nwr, k->nwr > 1).total;
    CU(ctx, raise_smem_limit(ctx->device, (const void *)fn, (int)smem));
    // the occupancy query costs microseconds: remember it per (kernel, shared memory size)
    const std::string key = std::to_string((size_t)(void *)fn) + ":" + std::to_string(smem);
    auto it = ctx->occ_cache.find(key);
    int occ = 0;
    if (it != ctx->occ_cache.end()) {
      occ = it->second;
    } else {
      CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, k->nw * k->nwr * 32, smem));
      if (occ < 1) return fail(ctx, YALPS_ERR_TOO_LARGE, "kernel does not fit on an SM (smem %zu)", smem);
      ctx->occ_cache[key] = occ;
    }
    if (q.check_cycles) occ = std::min(occ, 4);  // bounds the history buffer
    if (const char *env = getenv("YALPS_CTAS_PER_SM")) occ = std::max(1, std::min(occ, atoi(env)));  // experiments
    r->k = k;
    r->resident = resident;
    r->smem = smem;
    r->grid = (int)std::max(1LL, std::min((long long)occ * ctx->prop.multiProcessorCount, n));
  }
  // K4 (whole grid per LP, LPs one after another) beats K2 (one CTA per LP) when the tableaus do not fit in
  // shared memory and there are too few of them to give every SM its own LP.
  const bool k4 = !r->k || (!q.table_only && (path == YALPS_PATH_GRID ||
                                               ((path == YALPS_PATH_AUTO || path == YALPS_PATH_CLUSTER) && !r->resident &&
                                                n <= 16 && !small_for_grid)));
  if (path == YALPS_PATH_AUTO && !r->resident && !q.nodes && !q.table_only) {
    // few LPs that do not fit one SM's shared memory: KC when they fit a cluster's
    Route c;
    if (int rc = plan_cluster(ctx, Hcap, Wcap, &c)) return rc;
    if (c.k && n <= 2LL * std::max(1, c.clusters)) {
      *r = c;
      return 0;
    }
    // the batches K4 would take (beyond one cluster's shared memory too) go to KG when the tableau fits the grid's
    if (k4 && !getenv("YALPS_NO_KG")) {
      if (int rc = plan_gridres(ctx, Hcap, Wcap, &c)) return rc;
      if (c.k) {
        *r = c;
        return 0;
      }
    }
  }
  // Big, very sparse nodes (Monster-class models: ~1 % non-zeros, ~10 rows rewritten per pivot): the row-split HBM/L2
  // kernel with one CTA per node compacts the few active rows and needs no grid barrier -- 5.8 us per pivot for every
  // node of the wave at once, against 9.5 us per pivot and node on K4 (scripts/big_sparse_paths.py).  Denser nodes
  // (Vendor Selection: 28 % non-zeros at the root optimum) stay on K4.
  if (q.nodes && k4 && !r->resident && path == YALPS_PATH_AUTO && ctx->tune_threads <= 0 && ctx->tune_rows <= 0 &&
      q.root_density < 0.03) {
    int split_nwc = 8, split_nwr = 2;
    if (const char *env = getenv("YALPS_NODE_SPLIT")) sscanf(env, "%d,%d", &split_nwc, &split_nwr);  // experiments: "column warps,row groups"
    if (const KernelEntry *k = pick_kernel(split_nwc, split_nwr, Wcap, false)) {
      if (k->nwr == split_nwr) {
        const size_t smem_k = SmemLayout(Hcap, Wcap, false, k->nw * k->nwr, true).total;
        if (smem_k <= dynamic_smem_limit(ctx->device, ctx->smem_optin, (const void *)k->global)) {
          CU(ctx, raise_smem_limit(ctx->device, (const void *)k->global, (int)smem_k));
          int occ = 0;
          CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k->global, k->nw * k->nwr * 32, smem_k));
          if (occ >= 1) {
            r->kind = ROUTE_SIMPLEX;
            r->k = k;
            r->smem = smem_k;
            r->grid = (int)std::max<long long>(1, std::min<long long>((long long)occ * ctx->prop.multiProcessorCount, n));
            r->assembled = true;
            return 0;
          }
        }
      }
    }
  }
  r->kind = k4 ? ROUTE_GRID : ROUTE_SIMPLEX;
  return 0;
}

int hist_capacity(const yalps_options *opt) {
  if (!opt->check_cycles) return 0;
  double cap = opt->max_pivots;
  if (!(cap < 262144.0)) cap = 262144.0;
  if (cap < 1.0) cap = 1.0;
  return (int)cap;
}

// K1t, K1/K1s, K2/K2s: one launch.
int launch_simplex(yalps_ctx *ctx, const Route &r, BatchArgs &args, const std::string &slot, cudaStream_t stream) {
  const bool tmem = r.kind == ROUTE_K1T;
  if (!args.rows_out && ctx->d_rows && !ctx->rows_per_lp) args.rows_out = ctx->d_rows;  // total mode: every launch of the ctx
  args.counter = nullptr;
  const long long solvers = tmem ? (long long)r.grid * tmem_kernel_warps() : r.grid;  // K1t: one LP per warp
  if (args.n > solvers) {  // more LPs than CTAs: dynamic queue (pivot counts vary per LP)
    void *counter = nullptr;
    if (int rc = dev_ensure(ctx, "counter" + slot, 8, &counter)) return rc;
    CU(ctx, cudaMemsetAsync(counter, 0, 8, stream));
    args.counter = (unsigned long long *)counter;
  }
  if (args.check_cycles) {
    void *hist = nullptr;
    const size_t per_cta = (size_t)(tmem ? tmem_kernel_warps() : 1) * 2 * args.hist_cap * sizeof(int);  // K1t: per warp
    if (int rc = dev_ensure(ctx, "hist" + slot, (size_t)r.grid * per_cta, &hist)) return rc;
    args.hist = (int *)hist;
  } else {
    args.hist = nullptr;
  }
  if (tmem) {
    CU(ctx, launch_simplex_tmem(args, r.grid, stream));
    ctx->launches++;
    return 0;
  }
  SimplexKernel fn = r.resident ? r.k->resident : r.k->global;
  fn<<<r.grid, r.k->nw * r.k->nwr * 32, r.smem, stream>>>(args);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  return 0;
}

// ---- KC: one LP per thread-block cluster (cluster_kernel.cuh) -------------------------------------------
// Smallest cluster (2, 4, 8, 16 CTAs) whose shared memory holds the tableau, and the kernel covering its width.
// r->k stays null when the tableau does not fit or the device cannot co-schedule such a cluster.
int plan_cluster(yalps_ctx *ctx, int Hcap, int Wcap, Route *r) {
  r->k = nullptr;
  int count = 0;
  const KernelEntry *tab = kernel_table_cluster(&count);
  const KernelEntry *k = nullptr;
  for (int i = 0; i < count && !k; i++)
    if (tab[i].resident && (long long)tab[i].nw * 32 * tab[i].kc * 2 >= std::max(Wcap - 1, 1)) k = &tab[i];
  if (!k) return 0;
  for (int C = 2; C <= kMaxCluster; C *= 2) {
    const ClusterSmem L(Hcap, Wcap, C);
    if (L.total > dynamic_smem_limit(ctx->device, ctx->smem_optin, (const void *)k->resident)) continue;
    // more CTAs than the capacity needs when a CTA would otherwise own many rows (dense updates are row-parallel)
    if (L.Hloc > 40 && C < kMaxCluster) continue;
    const std::string key = "cl:" + std::to_string((size_t)(void *)k->resident) + ":" + std::to_string(C) + ":" + std::to_string(L.total);
    int ncl = 0;
    auto it = ctx->occ_cache.find(key);
    if (it != ctx->occ_cache.end()) {
      ncl = it->second;
    } else {
      CU(ctx, raise_smem_limit(ctx->device, (const void *)k->resident, (int)L.total));
      if (C > 8) CU(ctx, cudaFuncSetAttribute((const void *)k->resident, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3((unsigned)C * 64);
      cfg.blockDim = dim3((unsigned)(k->nw * k->nwr * 32));
      cfg.dynamicSmemBytes = L.total;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = (unsigned)C;
      attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      if (cudaOccupancyMaxActiveClusters(&ncl, (const void *)k->resident, &cfg) != cudaSuccess) {
        cudaGetLastError();
        ncl = 0;
      }
      ctx->occ_cache[key] = ncl;
    }
    if (ncl < 1) continue;
    CU(ctx, raise_smem_limit(ctx->device, (const void *)k->resident, (int)L.total));
    r->kind = ROUTE_CLUSTER;
    r->k = k;
    r->C = C;
    r->smem = L.total;
    r->clusters = ncl;
    return 0;
  }
  return 0;
}

// KC: one LP per thread-block cluster.
int launch_cluster(yalps_ctx *ctx, const Route &r, BatchArgs &args, const std::string &slot, cudaStream_t stream) {
  const int ncl = (int)std::max<long long>(1, std::min<long long>(r.clusters, args.n));
  if (!args.rows_out && ctx->d_rows && !ctx->rows_per_lp) args.rows_out = ctx->d_rows;
  args.counter = nullptr;
  args.hist = nullptr;
  if (args.check_cycles) {
    void *hist = nullptr;
    if (int rc = dev_ensure(ctx, "hist_cl" + slot, (size_t)ncl * r.C * 2 * args.hist_cap * sizeof(int), &hist)) return rc;
    args.hist = (int *)hist;
  }
  {
    void *scr = nullptr;
    const size_t per_cluster = (size_t)2 * r.C * SmemLayout::ld_for(args.Wcap) * sizeof(double);
    if (int rc = dev_ensure(ctx, "cl_scratch" + slot, per_cluster * ncl, &scr)) return rc;
    args.cl_scratch = (double *)scr;
  }
  args.tma_mode = ctx->kc_tma;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(ncl * r.C));
  cfg.blockDim = dim3((unsigned)(r.k->nw * r.k->nwr * 32));
  cfg.dynamicSmemBytes = r.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)r.C;
  attr[0].val.clusterDim.y = attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CU(ctx, cudaLaunchKernelEx(&cfg, r.k->resident, (const BatchArgs)args));
  ctx->launches++;
  return 0;
}

// ---- KG: the cluster kernel with the whole cooperative grid as its "cluster" (tableau resident in the SMs' shared memory)
// KG: the cluster kernel with the whole cooperative grid as its "cluster".  r->k stays null when the tableau does not
// fit the shared memory of the grid.
int plan_gridres(yalps_ctx *ctx, int Hcap, int Wcap, Route *r) {
  r->k = nullptr;
  int count = 0, coop = 0;
  const KernelEntry *tab = kernel_table_cluster(&count);
  const KernelEntry *k = nullptr;
  // narrowest kernel that covers the width; among those the one with the most threads (YALPS_KG_THREADS caps them)
  int max_threads = 512;
  if (const char *env = getenv("YALPS_KG_THREADS")) max_threads = atoi(env);
  for (int i = 0; i < count; i++) {
    const long long cap = (long long)tab[i].nw * 32 * tab[i].kc * 2;
    const int threads = tab[i].nw * tab[i].nwr * 32;
    if (!tab[i].global || cap < std::max(Wcap - 1, 1) || threads > max_threads) continue;
    const long long kcap = k ? (long long)k->nw * 32 * k->kc * 2 : 0;
    if (!k || cap < kcap || (cap == kcap && threads > k->nw * k->nwr * 32)) k = &tab[i];
  }
  if (!k) return 0;
  CU(ctx, cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device));
  if (!coop) return 0;
  int C = std::max(1, std::min(std::min(ctx->prop.multiProcessorCount, 160), Hcap - 1));  // (grid_select: 5 slots per lane)
  if (const char *env = getenv("YALPS_KG_CTAS")) C = std::max(1, std::min(C, atoi(env)));
  const ClusterSmem L(Hcap, Wcap, C);
  if (L.total > dynamic_smem_limit(ctx->device, ctx->smem_optin, (const void *)k->global)) return 0;
  CU(ctx, raise_smem_limit(ctx->device, (const void *)k->global, (int)L.total));
  const std::string key = "kg:" + std::to_string((size_t)(void *)k->global) + ":" + std::to_string(L.total);
  int occ = 0;
  auto it = ctx->occ_cache.find(key);
  if (it != ctx->occ_cache.end()) {
    occ = it->second;
  } else {
    CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void *)k->global, k->nw * k->nwr * 32, L.total));
    ctx->occ_cache[key] = occ;
  }
  if ((long long)occ * ctx->prop.multiProcessorCount < C) return 0;
  r->kind = ROUTE_GRID_RES;
  r->k = k;
  r->C = C;
  r->smem = L.total;
  return 0;
}

// KG: one LP over the cooperative grid, tableau resident in the SMs' shared memory.
int launch_gridres(yalps_ctx *ctx, const Route &r, BatchArgs &args, const std::string &slot, cudaStream_t stream) {
  if (!args.rows_out && ctx->d_rows && !ctx->rows_per_lp) args.rows_out = ctx->d_rows;
  args.hist = nullptr;
  if (args.check_cycles) {
    void *hist = nullptr;
    if (int rc = dev_ensure(ctx, "hist_kg" + slot, (size_t)r.C * 2 * args.hist_cap * sizeof(int), &hist)) return rc;
    args.hist = (int *)hist;
  }
  void *p = nullptr;
  const size_t ldA = (size_t)SmemLayout::ld_for(args.Wcap);
  // candidate rows as 16-byte flag-in-data slots {low word, sequence, high word, sequence}: [2][C][ldA]
  const size_t pub_bytes = (size_t)2 * r.C * ldA * sizeof(uint4);
  if (int rc = dev_ensure(ctx, "kg_scratch" + slot, pub_bytes, &p)) return rc;
  args.cl_scratch = (double *)p;
  CU(ctx, cudaMemsetAsync(p, 0, pub_bytes, stream));  // sequence numbers of an earlier launch must not look current
  const size_t inbox_bytes = (size_t)2 * r.C * r.C * sizeof(uint4);  // [2][receiver][sender] selection records
  if (int rc = dev_ensure(ctx, "kg_slots" + slot, inbox_bytes + 64, &p)) return rc;
  args.gx_slots = (uint4 *)p;
  args.counter = (unsigned long long *)((char *)p + inbox_bytes);
  // slots: sequence numbers of an earlier launch must not look current; counter: the grid barrier's arrival count
  CU(ctx, cudaMemsetAsync(p, 0, inbox_bytes + 64, stream));
  args.tma_mode = 0;
  void *params[] = {&args};
  CU(ctx, cudaLaunchCooperativeKernel((const void *)r.k->global, dim3((unsigned)r.C),
                                      dim3((unsigned)(r.k->nw * r.k->nwr * 32)), params, r.smem, stream));
  ctx->launches++;
  return 0;
}

// K4: one LP over the whole grid.  d_M (H*W doubles, reference layout) is solved in place; the options come from `o`
// (fill_options).
int launch_grid(yalps_ctx *ctx, int H, int W, double *d_M, const BatchArgs &o, int *d_status, double *d_value,
                long long *d_pivots, double *d_rhs, int *d_pos, int *d_var, cudaStream_t stream, const int *d_init_var,
                int init_n, int max_ctas, const std::string &slot, unsigned long long *d_rows, double *d_red = nullptr) {
  const GridSmem L(H, W);
  if (L.total > (size_t)ctx->smem_optin)
    return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau %dx%d: pivot row/column staging exceeds shared memory", H, W);
  int coop = 0;
  CU(ctx, cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device));
  if (!coop) return fail(ctx, YALPS_ERR_CUDA, "device does not support cooperative launches");
  CU(ctx, raise_smem_limit(ctx->device, (const void *)k_simplex_grid, (int)L.total));
  int occ = 0;
  CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_simplex_grid, kGridThreads, L.total));
  if (occ < 1) return fail(ctx, YALPS_ERR_TOO_LARGE, "grid kernel does not fit on an SM");
  // at most ~2 update items (row x 256-column segment) per warp, never more CTAs than can be co-resident
  int grid = ctx->prop.multiProcessorCount;
  {
    const long long items = (long long)H * ((W + kSegCols - 1) / kSegCols);
    grid = (int)std::min<long long>(grid, std::max(1LL, (items + 2 * kGridWarps - 1) / (2 * kGridWarps)));
  }
  if (const char *env = getenv("YALPS_GRID_CTAS")) grid = std::max(1, std::min(atoi(env), ctx->prop.multiProcessorCount * occ));
  if (max_ctas > 0) grid = std::max(1, std::min(grid, max_ctas));  // several K4 launches sharing the GPU (node waves)
  GridArgs a{};
  a.M = d_M;
  a.H = H;
  a.W = W;
  a.status = d_status;
  a.value = d_value;
  a.pivots = d_pivots;
  a.rhs_out = d_rhs;
  a.pos_out = d_pos;
  a.red_out = d_red;
  a.precision = o.precision;
  a.max_pivots = o.max_pivots;
  a.check_cycles = o.check_cycles;
  a.hist_cap = o.hist_cap;
  void *p = nullptr;
  if (!d_var) {
    if (int rc = dev_ensure(ctx, "grid_var" + slot, (size_t)(W + H) * 4, &p)) return rc;
    d_var = (int *)p;
  }
  a.var = d_var;
  a.init_var = d_init_var;
  a.init_n = init_n;
  a.rows_out = d_rows ? d_rows : ((ctx->d_rows && !ctx->rows_per_lp) ? ctx->d_rows : nullptr);
  if (int rc = dev_ensure(ctx, "grid_flags" + slot, 64, &p)) return rc;
  a.flags = (int *)p;
  a.barrier = (unsigned long long *)((char *)p + 32);
  CU(ctx, cudaMemsetAsync(p, 0, 64, stream));
  if (a.check_cycles) {
    if (int rc = dev_ensure(ctx, "grid_hist" + slot, (size_t)2 * a.hist_cap * sizeof(int), &p)) return rc;
    a.hist = (int *)p;
  }
  void *params[] = {&a};
  CU(ctx, cudaLaunchCooperativeKernel((void *)k_simplex_grid, dim3(grid), dim3(kGridThreads), params, L.total, stream));
  ctx->launches++;
  return 0;
}

// Enqueue route `r` for the LPs of `args` (device pointers filled in by the caller).  K4 solves them one after another
// in args.work, LP i being LP args.index[i] of the launch; a ragged batch's shapes, offsets and index are read from
// `host`, host-side copies of those fields of `args`.  Final tableaus under K4: one bulk copy in and one out for a
// uniform batch whose work buffer is not its input / output, one copy per LP into mat_out for a ragged batch.
int launch_route(yalps_ctx *ctx, const Route &r, BatchArgs &args, const std::string &slot, cudaStream_t stream,
                 const BatchArgs *host = nullptr) {
  if (r.kind == ROUTE_CLUSTER) return launch_cluster(ctx, r, args, slot, stream);
  if (r.kind == ROUTE_GRID_RES) return launch_gridres(ctx, r, args, slot, stream);
  if (r.kind != ROUTE_GRID) return launch_simplex(ctx, r, args, slot, stream);
  const bool ragged = args.heights != nullptr;
  const BatchArgs &h = ragged ? *host : args;
  const long long cells = (long long)args.H * args.W;
  if (!ragged && args.work != args.in)
    CU(ctx, cudaMemcpyAsync(args.work, args.in, (size_t)(args.n * cells) * 8, cudaMemcpyDeviceToDevice, stream));
  for (long long i = 0; i < args.n; i++) {
    const long long id = h.index ? h.index[i] : i;
    const int H = ragged ? h.heights[id] : args.H, W = ragged ? h.widths[id] : args.W;
    const long long mo = ragged ? h.mat_off[id] : id * cells, ro = ragged ? h.rhs_off[id] : id * args.H,
                    po = ragged ? h.pos_off[id] : id * (args.H + args.W);
    if (int rc = launch_grid(ctx, H, W, args.work + mo, args, args.status ? args.status + id : nullptr,
                             args.value ? args.value + id : nullptr, args.pivots ? args.pivots + 2 * id : nullptr,
                             args.rhs_out ? args.rhs_out + ro : nullptr, args.pos_out ? args.pos_out + po : nullptr,
                             args.var_out ? args.var_out + po : nullptr, stream,
                             args.var_in ? args.var_in + po : nullptr, args.var_in ? W + H : 0, 0, slot,
                             args.rows_out ? args.rows_out + (args.rows_per_lp ? id : 0) : nullptr,
                             args.red_out ? args.red_out + po : nullptr))
      return rc;
    if (ragged && args.mat_out)
      CU(ctx, cudaMemcpyAsync(args.mat_out + mo, args.work + mo, (size_t)H * W * 8, cudaMemcpyDeviceToDevice, stream));
  }
  if (!ragged && args.mat_out && args.mat_out != args.work)
    CU(ctx, cudaMemcpyAsync(args.mat_out, args.work, (size_t)(args.n * cells) * 8, cudaMemcpyDeviceToDevice, stream));
  return 0;
}

void fill_options(BatchArgs &a, const yalps_options *opt) {
  a.rows_out = nullptr;
  a.rows_per_lp = 0;
  a.precision = opt->precision;
  a.max_pivots = opt->max_pivots;
  a.check_cycles = opt->check_cycles ? 1 : 0;
  a.hist_cap = hist_capacity(opt);
}

int check_device_status(yalps_ctx *ctx, const int32_t *status, long long n) {
  if (!status) return 0;
  for (long long i = 0; i < n; i++)
    if (status[i] == ST_ERR_HISTORY)
      return fail(ctx, YALPS_ERR_HISTORY, "checkCycles history exhausted for LP %lld (more than 262144 pivots in a phase)", i);
    else if (status[i] == ST_ERR_PEER)
      return fail(ctx, YALPS_ERR_CUDA, "LP %lld: an in-kernel exchange between the CTAs of the grid timed out", i);
  return 0;
}

// k_ranging over the LPs of `a` (device pointers, shape or ragged fields and caps filled in by the caller).  Small
// tableaus take warp mode (one launch), the others tile mode (two launches; the inverse of pos goes to per-slot scratch
// of pv_total ints, the size of the pos layout the launch's offsets index into).
int launch_ranging(yalps_ctx *ctx, RangingArgs a, size_t pv_total, const std::string &slot, cudaStream_t stream) {
  if (a.n <= 0) return 0;
  const long long sms = ctx->prop.multiProcessorCount;
  if (post_warp_mode(a)) {
    a.warp_smem = (((size_t)(a.Hcap + a.Wcap) * 4 + 15) & ~(size_t)15) + (size_t)16 * a.Hcap;
    const long long blocks = std::min<long long>((a.n + kRngWarps - 1) / kRngWarps, sms * 64);
    k_ranging<<<(unsigned)blocks, kRngWarps * 32, kRngWarps * a.warp_smem, stream>>>(a, kRngWarp);
    CU(ctx, cudaGetLastError());
    ctx->launches++;
    return 0;
  }
  void *p;
  if (int rc = dev_ensure(ctx, "rng_var" + slot, pv_total * 4, &p)) return rc;
  a.var = (int *)p;
  a.tiles_r = std::max(1, (a.Hcap - 1 + kRngTileRows - 1) / kRngTileRows);
  a.tiles_c = (a.Wcap + kRngTileCols - 1) / kRngTileCols;
  k_ranging<<<(unsigned)std::min<long long>(a.n, sms * 16), kRngTileCols, 0, stream>>>(a, kRngInit);
  CU(ctx, cudaGetLastError());
  const long long tiles = a.n * a.tiles_r * a.tiles_c;
  k_ranging<<<(unsigned)std::min<long long>(tiles, sms * 64), kRngTileCols, 0, stream>>>(a, kRngTiles);
  CU(ctx, cudaGetLastError());
  ctx->launches += 2;
  return 0;
}

// k_certificate over the LPs of `a`: one warp per LP when post_warp_mode allows it, else one CTA per LP.
int launch_certificate(yalps_ctx *ctx, const CertArgs &a, cudaStream_t stream) {
  if (a.n <= 0) return 0;
  const bool warp = post_warp_mode(a);
  const long long per_block = warp ? kCertThreads / 32 : 1;
  const long long blocks = std::min<long long>((a.n + per_block - 1) / per_block, ctx->prop.multiProcessorCount * 64LL);
  k_certificate<<<(unsigned)blocks, kCertThreads, 0, stream>>>(a, warp ? 1 : 0);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  return 0;
}

// pairs (packed like rhs_out, one LP after another): pairs[0] = -1, every other entry -1 or another row 1..H-1 of the
// same LP that points back
int check_pairs(yalps_ctx *ctx, const int32_t *pairs, long long n, int32_t height, const int32_t *heights) {
  if (!pairs) return 0;
  long long ro = 0;
  for (long long i = 0; i < n; i++) {
    const int H = heights ? heights[i] : height;
    const int32_t *pr = pairs + ro;
    if (pr[0] != -1) return fail(ctx, YALPS_ERR_ARGUMENT, "LP %lld: pairs[0] must be -1 (row 0 is the objective)", i);
    for (int r = 1; r < H; r++) {
      const int q = pr[r];
      if (q == -1) continue;
      if (q < 1 || q >= H || q == r || pr[q] != r)
        return fail(ctx, YALPS_ERR_ARGUMENT, "LP %lld: pairs[%d] = %d is not a symmetric pair of two rows 1..%d", i, r,
                    q, H - 1);
    }
    ro += H;
  }
  return 0;
}

}  // namespace

// =========================================================================================================
extern "C" {

void yalps_default_options(yalps_options *opt) {
  opt->precision = 1e-8;
  opt->max_pivots = 8192;
  opt->tolerance = 0;
  opt->timeout_ms = std::numeric_limits<double>::infinity();
  opt->max_iterations = 32768;
  opt->check_cycles = 0;
  opt->reserved = 0;
}

int yalps_create(int device, yalps_ctx **out) {
  if (!out) return fail(nullptr, YALPS_ERR_ARGUMENT, "out is null");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(nullptr, YALPS_ERR_CUDA, "no CUDA device available (%s); yalps_b200 has no CPU fallback",
                e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
  if (device < 0 || device >= count) return fail(nullptr, YALPS_ERR_ARGUMENT, "device %d out of range [0,%d)", device, count);
  std::unique_ptr<yalps_ctx> ctx(new yalps_ctx);
  ctx->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(nullptr, YALPS_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
  if ((e = cudaGetDeviceProperties(&ctx->prop, device)) != cudaSuccess)
    return fail(nullptr, YALPS_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (ctx->prop.major < 10)
    return fail(nullptr, YALPS_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                ctx->prop.major, ctx->prop.minor);
  ctx->smem_optin = (int)ctx->prop.sharedMemPerBlockOptin;
  if (const char *env = getenv("YALPS_KC_TMA")) ctx->kc_tma = std::max(0, std::min(2, atoi(env)));
  for (int i = 0; i < 2; i++) {
    if ((e = cudaStreamCreateWithFlags(&ctx->streams[i], cudaStreamNonBlocking)) != cudaSuccess)
      return fail(nullptr, YALPS_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    if ((e = cudaEventCreateWithFlags(&ctx->events[i], cudaEventDisableTiming)) != cudaSuccess)
      return fail(nullptr, YALPS_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e));
  }
  *out = ctx.release();
  return 0;
}

void yalps_destroy(yalps_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (auto &kv : ctx->pool)
    if (kv.second.p) cudaFree(kv.second.p);
  for (auto &kv : ctx->pinned)
    if (kv.second.p) cudaFreeHost(kv.second.p);
  for (DevBuf *b : {&ctx->root.m, &ctx->root.pos, &ctx->root.var})
    if (b->p) cudaFree(b->p);
  for (int i = 0; i < 2; i++) {
    if (ctx->streams[i]) cudaStreamDestroy(ctx->streams[i]);
    if (ctx->events[i]) cudaEventDestroy(ctx->events[i]);
  }
  for (cudaStream_t st : ctx->aux_streams) cudaStreamDestroy(st);
  for (cudaEvent_t ev : ctx->aux_events) cudaEventDestroy(ev);
  if (ctx->fork_event) cudaEventDestroy(ctx->fork_event);
  delete ctx;
}

const char *yalps_last_error(const yalps_ctx *ctx) { return ctx ? ctx->error.c_str() : g_create_error.c_str(); }

int yalps_device_info(const yalps_ctx *ctx, int32_t *sm_count, int32_t *smem_per_block_optin, int32_t *cc_major,
                      int32_t *cc_minor) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (sm_count) *sm_count = ctx->prop.multiProcessorCount;
  if (smem_per_block_optin) *smem_per_block_optin = ctx->smem_optin;
  if (cc_major) *cc_major = ctx->prop.major;
  if (cc_minor) *cc_minor = ctx->prop.minor;
  return 0;
}

int yalps_set_tuning(yalps_ctx *ctx, int32_t path, int32_t threads_per_lp) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (path < 0 || path > YALPS_PATH_GRID_RESIDENT || path == 4) return fail(ctx, YALPS_ERR_ARGUMENT, "bad path %d", path);
  ctx->tune_path = path;
  ctx->tune_threads = threads_per_lp;
  return 0;
}

int yalps_set_row_groups(yalps_ctx *ctx, int32_t row_groups) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (row_groups < 0 || row_groups > 16 || (row_groups & (row_groups - 1)))
    return fail(ctx, YALPS_ERR_ARGUMENT, "row_groups must be 0 (automatic), 1, 2, 4, 8 or 16");
  ctx->tune_rows = row_groups;
  return 0;
}

int64_t yalps_launch_count(const yalps_ctx *ctx) { return ctx ? ctx->launches : 0; }

int yalps_set_row_counter(yalps_ctx *ctx, uint64_t *d_rows, int32_t per_lp) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  ctx->d_rows = (unsigned long long *)d_rows;
  ctx->rows_per_lp = per_lp ? 1 : 0;
  return 0;
}

int yalps_host_alloc(yalps_ctx *ctx, uint64_t bytes, void **out) {
  if (!ctx || !out) return YALPS_ERR_ARGUMENT;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaMallocHost(out, bytes ? bytes : 1));
  return 0;
}

int yalps_host_free(yalps_ctx *ctx, void *ptr) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (ptr) CU(ctx, cudaFreeHost(ptr));
  return 0;
}

// ---------------------------------------------------------------------------------------------------------
// `a` holds the shape (n, H, W), the input, the work buffer, the final-tableau output and the outputs, all in device
// memory; the rest is filled in here.  `slot` names the pooled scratch (LP queue counter, cycle history, cluster
// scratch) of this launch: calls that may be in flight at the same time on different streams of one ctx must use
// different slots.
static int solve_batch_device_impl(yalps_ctx *ctx, BatchArgs a, const yalps_options *opt, const std::string &slot,
                                   cudaStream_t stream, int64_t rows_base = 0) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  const long long n = a.n;
  const int height = a.H, width = a.W;
  if (n < 0 || height < 1 || width < 1 || !opt || (n > 0 && !a.in))
    return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments (n=%lld, %dx%d)", n, height, width);
  if ((long long)height * width >= (1LL << 31)) return fail(ctx, YALPS_ERR_TOO_LARGE, "height*width must be < 2^31");
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  // density probe for the path policy, once per (buffer, shape): synchronises `stream` the first time only
  double density = -1.0;
  if (ctx->tune_path == YALPS_PATH_AUTO && n > 64 && a.work) {
    const std::string key = std::to_string((size_t)a.in) + ":" + std::to_string(height) + "x" + std::to_string(width);
    auto it = ctx->density_cache.find(key);
    if (it == ctx->density_cache.end()) {
      void *hp, *dp;
      if (int rc = pin_ensure(ctx, "density_probe", 64, &hp)) return rc;
      if (int rc = pin_device_ptr(ctx, hp, &dp)) return rc;
      ((int *)hp)[0] = ((int *)hp)[1] = 0;
      const long long cells = (long long)height * width;
      k_sample_density<<<1, 256, 0, stream>>>(a.in, cells, std::max(1LL, cells / 4096), (int *)dp);
      CU(ctx, cudaGetLastError());
      CU(ctx, cudaStreamSynchronize(stream));
      ctx->launches++;
      const int seen = ((int *)hp)[0], nz = ((int *)hp)[1];
      density = seen ? (double)nz / seen : 1.0;
      if (ctx->density_cache.size() > 64) ctx->density_cache.clear();
      ctx->density_cache[key] = density;
    } else {
      density = it->second;
    }
  }
  a.mode = kModeBatch;
  a.Hcap = height;
  a.Wcap = width;
  fill_options(a, opt);
  a.rows_out = ctx->d_rows ? ctx->d_rows + (ctx->rows_per_lp ? rows_base : 0) : nullptr;
  a.rows_per_lp = ctx->rows_per_lp;
  Route route;
  if (int rc = choose_route(ctx, {n, height, width, density, opt->check_cycles != 0, true}, &route)) return rc;
  if (route.kind == ROUTE_GRID && !a.work) return fail(ctx, YALPS_ERR_ARGUMENT, "d_work is required for the grid path");
  if (route.kind == ROUTE_SIMPLEX && !route.resident) {
    if (!a.work) return fail(ctx, YALPS_ERR_ARGUMENT, "d_work is required for the HBM-resident path");
    if (!a.pos_out || !a.var_out) {
      void *p = nullptr;
      if (int rc = dev_ensure(ctx, "posvar_scratch" + slot, (size_t)n * (width + height) * 2 * sizeof(int), &p)) return rc;
      if (!a.pos_out) a.pos_out = (int *)p;
      if (!a.var_out) a.var_out = (int *)p + (size_t)n * (width + height);
    }
  }
  return launch_route(ctx, route, a, slot, stream);
}

int yalps_solve_batch_device(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                             double *d_work, const yalps_options *opt, int32_t *d_status, double *d_value,
                             int64_t *d_pivots, double *d_rhs_out, int32_t *d_pos_out, int32_t *d_var_out,
                             double *d_matrices_out, void *stream) {
  return yalps_solve_batch_device_duals(ctx, n, height, width, d_matrices, d_work, opt, d_status, d_value, d_pivots,
                                        d_rhs_out, d_pos_out, d_var_out, d_matrices_out, stream, nullptr);
}

int yalps_solve_batch_device_duals(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                                   double *d_work, const yalps_options *opt, int32_t *d_status, double *d_value,
                                   int64_t *d_pivots, double *d_rhs_out, int32_t *d_pos_out, int32_t *d_var_out,
                                   double *d_matrices_out, void *stream, double *d_reduced_out) {
  BatchArgs a{};
  a.n = n;
  a.H = height;
  a.W = width;
  a.in = d_matrices;
  a.work = d_work;
  a.mat_out = d_matrices_out;
  a.status = d_status;
  a.value = d_value;
  a.pivots = (long long *)d_pivots;
  a.rhs_out = d_rhs_out;
  a.pos_out = d_pos_out;
  a.var_out = d_var_out;
  a.red_out = d_reduced_out;
  return solve_batch_device_impl(ctx, a, opt, "dev", (cudaStream_t)stream);
}

int yalps_ranging_device(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                         const int32_t *d_pos, const int32_t *d_status, const int32_t *d_pairs, double precision,
                         double *d_range_lo, double *d_range_hi, void *stream) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (n < 0 || height < 1 || width < 1 || (n > 0 && (!d_matrices || !d_pos || !d_range_lo || !d_range_hi)))
    return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments (n=%lld, %dx%d)", (long long)n, height, width);
  if ((long long)height * width >= (1LL << 31)) return fail(ctx, YALPS_ERR_TOO_LARGE, "height*width must be < 2^31");
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  RangingArgs a{};
  a.n = n;
  a.H = a.Hcap = height;
  a.W = a.Wcap = width;
  a.M = d_matrices;
  a.pos = d_pos;
  a.status = d_status;
  a.pairs = d_pairs;
  a.precision = precision;
  a.lo = d_range_lo;
  a.hi = d_range_hi;
  return launch_ranging(ctx, a, (size_t)n * (width + height), "dev", (cudaStream_t)stream);
}

int yalps_certificate_device(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                             const int32_t *d_pos, const int32_t *d_status, const double *d_value, double precision,
                             double *d_cert_out, void *stream) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (n < 0 || height < 1 || width < 1 ||
      (n > 0 && (!d_matrices || !d_pos || !d_status || !d_value || !d_cert_out)))
    return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments (n=%lld, %dx%d)", (long long)n, height, width);
  if ((long long)height * width >= (1LL << 31)) return fail(ctx, YALPS_ERR_TOO_LARGE, "height*width must be < 2^31");
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  CertArgs a{};
  a.n = n;
  a.H = a.Hcap = height;
  a.W = a.Wcap = width;
  a.M = d_matrices;
  a.pos = d_pos;
  a.status = d_status;
  a.value = d_value;
  a.precision = precision;
  a.cert = d_cert_out;
  return launch_certificate(ctx, a, (cudaStream_t)stream);
}

}  // extern "C"

// ---- host batches --------------------------------------------------------------------------------------------------
namespace {

// One host batch solve: the shape, where the tableaus come from, the optional inputs and every output (null: not
// wanted).  The yalps_solve_{batch,ragged}_certificate entries, yalps_solve's root LP, the sparse entries, the replica
// entries and the row-subset entries fill one in.
struct HostBatch {
  int64_t n = 0;
  int32_t height = 0, width = 0;                        // a uniform batch, or
  const int32_t *heights = nullptr, *widths = nullptr;  // a ragged one (heights given)
  const int64_t *mat_offsets = nullptr;
  const double *matrices = nullptr;  // dense host tableaus, or (n == 1, uniform, nnz >= 0) the (cell, value) stores
  const int32_t *cell = nullptr;     // into a zero tableau, scattered on the device (yalps_solve_sparse)
  const double *val = nullptr;
  int64_t nnz = -1;
  const double *d_base = nullptr;  // or (uniform) LPs derived on the device from this base tableau in device memory
  const double *rhs_in = nullptr;  // by their own column 0 (n x height values: replicas), or
  const uint32_t *keep = nullptr;  // by their own row mask (n x words, words = (height + 31) / 32: row subsets)
  const int32_t *pos_in = nullptr, *var_in = nullptr;  // the basis the tableaus arrive with (both null: the identity)
  const int32_t *pairs = nullptr;                       // ranging: the other row of each row's key
  const yalps_options *opt = nullptr;
  int32_t *status = nullptr;
  double *value = nullptr;
  int64_t *pivots = nullptr;
  double *rhs_out = nullptr;
  int32_t *pos_out = nullptr, *var_out = nullptr;
  double *matrices_out = nullptr, *reduced_out = nullptr, *range_lo = nullptr, *range_hi = nullptr;
  double *cert_out = nullptr;
  uint32_t *support_out = nullptr;  // the rows each certificate uses (a mask, packed like keep) and their number
  int32_t *count_out = nullptr;
  bool keep_final = false;  // (n == 1, uniform) leave the final tableau on the device, no D2H copy of it
  // results
  double *kept_final = nullptr;  // keep_final: where the final tableau is (valid until the next batch call on the ctx)
  int32_t dup_cells = 0;         // nnz >= 0: the device found duplicate cells with different values
  // the supports are read from the certificates, wanted or not
  bool want_support() const { return support_out != nullptr || count_out != nullptr; }
  // a post-pass (k_ranging, k_certificate) reads the final tableaus, which therefore stay in device memory
  bool post_pass() const { return range_lo != nullptr || cert_out != nullptr || want_support(); }
};

// The per-LP outputs of a host batch, described once: pool name, host array (null: not wanted), element size and
// packing.  The kernels write the first six whether they are wanted or not, so those always get a device buffer;
// k_cert_support reads the certificates and writes both support and count when either is wanted.
enum OutPack { PER_LP, PER_ROW, PER_VAR };  // per LP (times k), per row like rhs_out, per variable id like pos_out
struct OutSpec {
  const char *name;
  void *host;
  size_t elem;
  OutPack pack;
  int k;
  bool always;
  bool used() const { return always || host; }
  // bytes for `lps` LPs of `rows` rows and `pvs` variable ids in all
  size_t bytes(long long lps, long long rows, long long pvs) const {
    return elem * (size_t)(pack == PER_LP ? lps * k : pack == PER_ROW ? rows : pvs);
  }
};
enum { O_STATUS, O_VALUE, O_PIVOTS, O_RHS, O_POS, O_VAR, O_RED, O_RLO, O_RHI, O_CERT, O_SUP, O_CNT, O_COUNT };
struct Outputs {
  OutSpec t[O_COUNT];
  explicit Outputs(const HostBatch &b)
      : t{{"status", b.status, 4, PER_LP, 1, true},     {"value", b.value, 8, PER_LP, 1, true},
          {"pivots", b.pivots, 8, PER_LP, 2, true},     {"rhs", b.rhs_out, 8, PER_ROW, 1, true},
          {"pos", b.pos_out, 4, PER_VAR, 1, true},      {"var", b.var_out, 4, PER_VAR, 1, true},
          {"red", b.reduced_out, 8, PER_VAR, 1, false}, {"rlo", b.range_lo, 8, PER_VAR, 1, false},
          {"rhi", b.range_hi, 8, PER_VAR, 1, false},    {"cert", b.cert_out, 8, PER_VAR, 1, b.want_support()},
          {"support", b.support_out, 4, PER_LP, (b.height + 31) / 32, b.want_support()},
          {"count", b.count_out, 4, PER_LP, 1, b.want_support()}} {}

  // device buffers "<name><slot>" for a chunk of `lps` LPs (`rows` rows, `pvs` variable ids); null where not used
  int ensure(yalps_ctx *ctx, const std::string &slot, long long lps, long long rows, long long pvs, void **dev) const {
    for (int i = 0; i < O_COUNT; i++) {
      dev[i] = nullptr;
      if (t[i].used())
        if (int rc = dev_ensure(ctx, t[i].name + slot, t[i].bytes(lps, rows, pvs), &dev[i])) return rc;
    }
    return 0;
  }
  // D2H copies of the wanted outputs of a chunk that starts after lp0 LPs (row0 rows, pv0 variable ids)
  int copy_out(yalps_ctx *ctx, void *const *dev, long long lp0, long long row0, long long pv0, long long lps,
               long long rows, long long pvs, cudaStream_t st) const {
    for (const OutSpec &o : t)
      if (o.host)
        CU(ctx, cudaMemcpyAsync((char *)o.host + o.bytes(lp0, row0, pv0), dev[&o - t], o.bytes(lps, rows, pvs),
                                cudaMemcpyDeviceToHost, st));
    return 0;
  }
};

// The LPs [lo, hi) of request b, after row0 rows and pv0 variable ids.  A uniform batch moves its tableaus by cells; a
// ragged one moves its shapes and offsets by LPs and keeps matrices and matrices_out, which those offsets index
// absolutely.  The basis moves by variable ids, the pairs and right-hand sides by rows, the row masks by LPs, the
// outputs as the Outputs table packs them.
HostBatch slice_request(const HostBatch &b, int64_t lo, int64_t hi, long long row0, long long pv0) {
  HostBatch s = b;
  s.n = hi - lo;
  if (b.heights) {
    s.heights += lo;
    s.widths += lo;
    s.mat_offsets += lo;
  } else {
    const size_t cells = (size_t)lo * b.height * b.width;
    if (s.matrices) s.matrices += cells;
    if (s.matrices_out) s.matrices_out += cells;
  }
  if (s.pos_in) s.pos_in += pv0;
  if (s.var_in) s.var_in += pv0;
  if (s.pairs) s.pairs += row0;
  if (s.rhs_in) s.rhs_in += row0;
  if (s.keep) s.keep += lo * ((b.height + 31) / 32);
  const Outputs o(b);
  auto at = [&](int i) -> void * { return o.t[i].host ? (char *)o.t[i].host + o.t[i].bytes(lo, row0, pv0) : nullptr; };
  s.status = (int32_t *)at(O_STATUS);
  s.value = (double *)at(O_VALUE);
  s.pivots = (int64_t *)at(O_PIVOTS);
  s.rhs_out = (double *)at(O_RHS);
  s.pos_out = (int32_t *)at(O_POS);
  s.var_out = (int32_t *)at(O_VAR);
  s.reduced_out = (double *)at(O_RED);
  s.range_lo = (double *)at(O_RLO);
  s.range_hi = (double *)at(O_RHI);
  s.cert_out = (double *)at(O_CERT);
  s.support_out = (uint32_t *)at(O_SUP);
  s.count_out = (int32_t *)at(O_CNT);
  return s;
}

void set_outputs(BatchArgs &a, void *const *dev) {
  a.status = (int *)dev[O_STATUS];
  a.value = (double *)dev[O_VALUE];
  a.pivots = (long long *)dev[O_PIVOTS];
  a.rhs_out = (double *)dev[O_RHS];
  a.pos_out = (int *)dev[O_POS];
  a.var_out = (int *)dev[O_VAR];
  a.red_out = (double *)dev[O_RED];
}

// The post-passes `b` wants (k_ranging, then k_certificate) over the final tableaus M of the LPs `a` solved (all LPs
// of a launch, or one ragged group through a.index), on the solve's stream before the copies back.  pairs: device
// copy of the request's pairs, or null; pv_total: the variable ids of the layout a's offsets index into.
int post_passes(yalps_ctx *ctx, const HostBatch &b, const BatchArgs &a, const double *M, const int *pairs,
                void *const *dev, size_t pv_total, const std::string &slot, cudaStream_t st) {
  PostArgs p{};
  p.n = a.n;
  p.H = a.H;
  p.W = a.W;
  p.Hcap = a.Hcap;
  p.Wcap = a.Wcap;
  p.M = M;
  p.heights = a.heights;
  p.widths = a.widths;
  p.mat_off = a.mat_off;
  p.rhs_off = a.rhs_off;
  p.pos_off = a.pos_off;
  p.index = a.index;
  p.pos = a.pos_out;
  p.status = a.status;
  if (b.range_lo) {
    RangingArgs g{};
    static_cast<PostArgs &>(g) = p;
    g.pairs = pairs;
    g.precision = b.opt->precision;
    g.lo = (double *)dev[O_RLO];
    g.hi = (double *)dev[O_RHI];
    if (int rc = launch_ranging(ctx, g, pv_total, slot, st)) return rc;
  }
  if (b.cert_out || b.want_support()) {
    CertArgs g{};
    static_cast<PostArgs &>(g) = p;
    g.value = a.value;
    g.precision = b.opt->precision;
    g.cert = (double *)dev[O_CERT];
    if (int rc = launch_certificate(ctx, g, st)) return rc;
  }
  return 0;
}

// What solve_host derives from a valid request: the caps and the per-LP prefix counts of cells, rows and variable ids.
struct BatchLayout {
  bool ragged = false;
  int32_t height = 0, width = 0, Hcap = 0, Wcap = 0;
  std::vector<long long> moff, roff, poff;  // ragged only
  const int32_t *pairs = nullptr;           // the request's pairs when ranges are wanted, else null
  long long cells_upto(int64_t i) const { return ragged ? moff[i] : (long long)i * height * width; }
  long long rows_upto(int64_t i) const { return ragged ? roff[i] : (long long)i * height; }
  long long pv_upto(int64_t i) const { return ragged ? poff[i] : (long long)i * (height + width); }
};

// Validates a request and lays it out (nothing more when b.n == 0).
int batch_layout(yalps_ctx *ctx, const HostBatch &b, BatchLayout *L) {
  const int64_t n = b.n;
  if (n < 0 || !b.opt || (n > 0 && !b.matrices && b.nnz < 0)) return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments");
  if ((b.pos_in == nullptr) != (b.var_in == nullptr))
    return fail(ctx, YALPS_ERR_ARGUMENT, "pos_in and var_in must be given together (or both null for the identity)");
  if ((b.range_lo == nullptr) != (b.range_hi == nullptr))
    return fail(ctx, YALPS_ERR_ARGUMENT, "range_lo and range_hi must be given together (or both null)");
  if (n == 0) return 0;
  L->ragged = b.heights != nullptr;
  L->height = L->Hcap = b.height;
  L->width = L->Wcap = b.width;
  L->pairs = b.range_lo ? b.pairs : nullptr;
  if (L->ragged) {
    if (!b.widths || !b.mat_offsets) return fail(ctx, YALPS_ERR_ARGUMENT, "ragged batch needs widths and mat_offsets");
    L->moff.resize(n + 1);
    L->roff.resize(n + 1);
    L->poff.resize(n + 1);
    long long r = 0, p = 0, m = 0;
    L->Hcap = L->Wcap = 1;
    for (int64_t i = 0; i < n; i++) {
      const int32_t h = b.heights[i], w = b.widths[i];
      if (h < 1 || w < 1) return fail(ctx, YALPS_ERR_ARGUMENT, "LP %lld has empty shape", (long long)i);
      if ((long long)h * w >= (1LL << 31)) return fail(ctx, YALPS_ERR_TOO_LARGE, "height*width must be < 2^31");
      L->moff[i] = m;
      L->roff[i] = r;
      L->poff[i] = p;
      m += (long long)h * w;
      r += h;
      p += h + w;
      L->Hcap = std::max(L->Hcap, h);
      L->Wcap = std::max(L->Wcap, w);
    }
    L->moff[n] = m;
    L->roff[n] = r;
    L->poff[n] = p;
  } else {
    if (b.height < 1 || b.width < 1) return fail(ctx, YALPS_ERR_ARGUMENT, "bad shape %dx%d", b.height, b.width);
    if ((long long)b.height * b.width >= (1LL << 31)) return fail(ctx, YALPS_ERR_TOO_LARGE, "height*width must be < 2^31");
  }
  if (int rc = check_pairs(ctx, L->pairs, n, b.height, b.heights)) return rc;
  // caller-supplied basis: the two arrays must be inverse permutations of 0..W+H-1 (src/tableau.ts:9-15); the kernels
  // carry variableAtPosition and rebuild positionOfVariable on output, so an inconsistent pair would silently
  // change meaning instead of behaving like the reference
  if (b.var_in) {
    for (int64_t i = 0; i < n; i++) {
      const long long o = L->pv_upto(i), len = L->pv_upto(i + 1) - o;
      for (long long k = 0; k < len; k++) {
        const int32_t v = b.var_in[o + k];
        if (v < 0 || v >= len || b.pos_in[o + v] != (int32_t)k)
          return fail(ctx, YALPS_ERR_ARGUMENT, "LP %lld: pos_in/var_in are not inverse permutations at position %lld",
                      (long long)i, k);
      }
    }
  }
  return 0;
}

// density of (a sample of) the first tableau: the path policy distinguishes dense from very sparse LPs
double first_density(const HostBatch &b) {
  const bool ragged = b.heights != nullptr;
  const double *m0 = b.matrices + (ragged ? b.mat_offsets[0] : 0);
  const long long c0 = ragged ? (long long)b.heights[0] * b.widths[0] : (long long)b.height * b.width;
  const long long step = std::max(1LL, c0 / 4096);
  long long seen = 0, nz = 0;
  for (long long k = 0; k < c0; k += step, seen++) nz += m0[k] != 0.0;
  return seen ? (double)nz / (double)seen : 1.0;
}

// Small calls (a single LP, a handful of models) are latency-bound.  Stage through one mapped pinned buffer, let the
// kernel read the tableaus and write the results zero-copy: launch + synchronise, no memcpy calls.  *taken is false
// (and nothing was done) when the batch does not qualify.
int solve_small(yalps_ctx *ctx, const HostBatch &b, const BatchLayout &L, bool *taken) {
  *taken = false;
  const int64_t n = b.n;
  const bool ragged = L.ragged, post = b.post_pass();
  const long long rows = L.rows_upto(n), pvs = L.pv_upto(n);
  const size_t in_b = (size_t)L.cells_upto(n) * 8, rows_b = (size_t)rows * 8, pv_b = (size_t)pvs * 4;
  const size_t red_b = b.reduced_out ? 2 * pv_b : 0;  // doubles, packed like pos_out
  const size_t rng_b = b.range_lo ? 2 * pv_b : 0;     // range_lo, range_hi: doubles, packed like pos_out
  const size_t cert_b = b.cert_out ? 2 * pv_b : 0;    // doubles, packed like pos_out
  const size_t pair_b = L.pairs ? rows_b / 2 : 0;     // int32, packed like rhs_out
  const size_t out_b = (size_t)n * 32 + rows_b + 2 * pv_b + 64 + (b.matrices_out ? in_b : 0) + (red_b ? red_b + 16 : 0) +
                       (rng_b ? 2 * rng_b + 32 : 0) + (cert_b ? cert_b + 16 : 0);
  const size_t desc_b = (ragged ? (size_t)n * 32 + 64 : 0) + (b.var_in ? pv_b + 16 : 0) + (pair_b ? pair_b + 16 : 0);
  Route route;
  if (b.keep_final || b.nnz >= 0 || in_b + out_b + desc_b > ((size_t)768 << 10) ||
      choose_route(ctx, {n, L.Hcap, L.Wcap, first_density(b), b.opt->check_cycles != 0, true}, &route) != 0 ||
      !(route.kind == ROUTE_K1T || (route.kind == ROUTE_SIMPLEX && route.resident)))
    return 0;
  *taken = true;
  const Outputs outs(b);
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  size_t o = 0;
  const size_t o_in = o; o += up16(in_b);
  const size_t o_h = o; o += ragged ? up16((size_t)n * 4) : 0;
  const size_t o_w = o; o += ragged ? up16((size_t)n * 4) : 0;
  const size_t o_mo = o; o += ragged ? up16((size_t)n * 8) : 0;
  const size_t o_ro = o; o += ragged ? up16((size_t)n * 8) : 0;
  const size_t o_po = o; o += ragged ? up16((size_t)n * 8) : 0;
  const size_t o_vin = o; o += b.var_in ? up16(pv_b) : 0;
  size_t o_out[O_COUNT];
  for (int i = 0; i < O_COUNT; i++) {
    o_out[i] = o;
    o += outs.t[i].used() ? up16(outs.t[i].bytes(n, rows, pvs)) : 0;
  }
  const size_t o_mat = o; o += b.matrices_out ? up16(in_b) : 0;
  const size_t o_pair = o; o += up16(pair_b);
  void *hb, *db;
  int rc;
  if ((rc = pin_ensure(ctx, "small_io", o + 16, &hb))) return rc;
  if ((rc = pin_device_ptr(ctx, hb, &db))) return rc;
  char *h = (char *)hb, *d = (char *)db;
  // the post-passes read the final tableaus from device scratch, not over PCIe from the mapped buffer
  void *d_fin = nullptr;
  if (post && (rc = dev_ensure(ctx, "small_final", in_b, &d_fin))) return rc;
  if (L.pairs) std::memcpy(h + o_pair, L.pairs, pair_b);
  if (ragged) {
    for (int64_t i = 0; i < n; i++)
      std::memcpy(h + o_in + (size_t)L.moff[i] * 8, b.matrices + b.mat_offsets[i], (size_t)b.heights[i] * b.widths[i] * 8);
    std::memcpy(h + o_h, b.heights, (size_t)n * 4);
    std::memcpy(h + o_w, b.widths, (size_t)n * 4);
    std::memcpy(h + o_mo, L.moff.data(), (size_t)n * 8);
    std::memcpy(h + o_ro, L.roff.data(), (size_t)n * 8);
    std::memcpy(h + o_po, L.poff.data(), (size_t)n * 8);
  } else {
    std::memcpy(h + o_in, b.matrices, in_b);
  }
  if (b.var_in) std::memcpy(h + o_vin, b.var_in, pv_b);
  void *dev[O_COUNT];
  for (int i = 0; i < O_COUNT; i++) dev[i] = outs.t[i].used() ? d + o_out[i] : nullptr;
  BatchArgs a{};
  a.n = n;
  a.mode = kModeBatch;
  a.H = L.height;
  a.W = L.width;
  a.Hcap = L.Hcap;
  a.Wcap = L.Wcap;
  a.in = (const double *)(d + o_in);
  a.work = nullptr;
  a.mat_out = post ? (double *)d_fin : b.matrices_out ? (double *)(d + o_mat) : nullptr;
  set_outputs(a, dev);
  a.var_in = b.var_in ? (const int *)(d + o_vin) : nullptr;
  if (ragged) {
    a.heights = (const int *)(d + o_h);
    a.widths = (const int *)(d + o_w);
    a.mat_off = (const long long *)(d + o_mo);
    a.rhs_off = (const long long *)(d + o_ro);
    a.pos_off = (const long long *)(d + o_po);
  }
  fill_options(a, b.opt);
  cudaStream_t st = ctx->streams[0];
  if ((rc = launch_route(ctx, route, a, "small", st))) return rc;
  if (post) {
    const int *pairs = L.pairs ? (const int *)(d + o_pair) : nullptr;
    if ((rc = post_passes(ctx, b, a, (const double *)d_fin, pairs, dev, (size_t)pvs, "small", st))) return rc;
    if (b.matrices_out) CU(ctx, cudaMemcpyAsync(h + o_mat, d_fin, in_b, cudaMemcpyDeviceToHost, st));
  }
  CU(ctx, cudaStreamSynchronize(st));
  for (int i = 0; i < O_COUNT; i++)
    if (outs.t[i].host) std::memcpy(outs.t[i].host, h + o_out[i], outs.t[i].bytes(n, rows, pvs));
  if (b.matrices_out) {
    if (ragged)
      for (int64_t i = 0; i < n; i++)
        std::memcpy(b.matrices_out + b.mat_offsets[i], h + o_mat + (size_t)L.moff[i] * 8,
                    (size_t)b.heights[i] * b.widths[i] * 8);
    else
      std::memcpy(b.matrices_out, h + o_mat, in_b);
  }
  return check_device_status(ctx, b.status, n);
}

// The (cell, value) stores of request b (b.nnz >= 0) into the tableau d_M of `cells` cells, on stream st: the pairs
// cross PCIe, the zeros are written by the device.  b.dup_cells is valid once st has reached this point.
int scatter_cells(yalps_ctx *ctx, HostBatch &b, double *d_M, size_t cells, cudaStream_t st) {
  const size_t nnz = (size_t)b.nnz, val_off = (nnz * 4 + 15) & ~(size_t)15;
  void *h_coo, *d_coo, *d_flag;
  int rc;
  if ((rc = pin_ensure(ctx, "coo", val_off + nnz * 8 + 16, &h_coo))) return rc;
  if ((rc = dev_ensure(ctx, "coo", val_off + nnz * 8 + 16, &d_coo))) return rc;
  if ((rc = dev_ensure(ctx, "coo_flag", 4, &d_flag))) return rc;
  if (nnz) {
    std::memcpy(h_coo, b.cell, nnz * 4);
    std::memcpy((char *)h_coo + val_off, b.val, nnz * 8);
    CU(ctx, cudaMemcpyAsync(d_coo, h_coo, val_off + nnz * 8, cudaMemcpyHostToDevice, st));
  }
  CU(ctx, cudaMemsetAsync(d_M, 0, cells * 8, st));
  CU(ctx, cudaMemsetAsync(d_flag, 0, 4, st));
  if (nnz) {
    const int blocks = (int)std::min<size_t>((nnz + 255) / 256, (size_t)ctx->prop.multiProcessorCount * 8);
    const int *d_cell = (const int *)d_coo;
    const double *d_val = (const double *)((char *)d_coo + val_off);
    k_scatter_cells<<<blocks, 256, 0, st>>>((long long)nnz, d_cell, d_val, d_M);
    k_verify_cells<<<blocks, 256, 0, st>>>((long long)nnz, d_cell, d_val, (const double *)d_M, (int *)d_flag);
    ctx->launches += 2;
    CU(ctx, cudaGetLastError());
  }
  CU(ctx, cudaMemcpyAsync(&b.dup_cells, d_flag, 4, cudaMemcpyDeviceToHost, st));
  return 0;
}

// The pipelined path: two slots; a large batch is cut into ~8 chunks (64 MiB .. 1.5 GiB each) so that the H2D copy of
// chunk k+1 overlaps the kernel and the D2H copies of chunk k.
int solve_chunks(yalps_ctx *ctx, HostBatch &b, const BatchLayout &L) {
  const int64_t n = b.n;
  const bool ragged = L.ragged;
  const yalps_options *opt = b.opt;
  const Outputs outs(b);
  const size_t total_bytes = (size_t)L.cells_upto(n) * 8;
  const size_t kSlotBytes = std::min((size_t)1536 << 20, std::max((size_t)64 << 20, total_bytes / 8 + 4096));

  int64_t begin = 0;
  int slot = 0;
  int rc = 0;
  double density = -1.0;
  bool used[2] = {false, false};
  while (begin < n) {
    int64_t end = begin + 1;
    while (end < n && (size_t)(L.cells_upto(end + 1) - L.cells_upto(begin)) * 8 <= kSlotBytes) end++;
    const int64_t cn = end - begin;
    const size_t ccells = (size_t)(L.cells_upto(end) - L.cells_upto(begin));
    const size_t crows = (size_t)(L.rows_upto(end) - L.rows_upto(begin));
    const size_t cpv = (size_t)(L.pv_upto(end) - L.pv_upto(begin));
    const std::string s = std::to_string(slot);
    cudaStream_t st = ctx->streams[slot];
    if (used[slot]) CU(ctx, cudaEventSynchronize(ctx->events[slot]));

    int chcap = L.Hcap, cwcap = L.Wcap;
    if (ragged) {
      chcap = cwcap = 1;
      for (int64_t i = begin; i < end; i++) {
        chcap = std::max(chcap, b.heights[i]);
        cwcap = std::max(cwcap, b.widths[i]);
      }
    }
    const bool from_cells = b.nnz >= 0;
    if (from_cells) density = (double)b.nnz / (double)((long long)b.height * b.width);
    if (density < 0.0) density = first_density(b);  // sampled once
    // a uniform chunk is one launch, routed before its buffers are set up (the route decides where its final tableaus
    // go); a ragged chunk is routed group by group below
    Route route;
    if (!ragged && (rc = choose_route(ctx, {cn, chcap, cwcap, density, opt->check_cycles != 0, true}, &route))) return rc;

    void *d_in, *dev[O_COUNT];
    if ((rc = dev_ensure(ctx, "in" + s, ccells * 8, &d_in))) return rc;
    if ((rc = outs.ensure(ctx, s, cn, crows, cpv, dev))) return rc;
    void *d_pairs = nullptr;
    if (L.pairs) {
      if ((rc = dev_ensure(ctx, "pairs" + s, crows * 4, &d_pairs))) return rc;
      CU(ctx, cudaMemcpyAsync(d_pairs, L.pairs + L.rows_upto(begin), crows * 4, cudaMemcpyHostToDevice, st));
    }
    void *d_vin = nullptr;
    if (b.var_in) {
      if ((rc = dev_ensure(ctx, "varin" + s, cpv * 4, &d_vin))) return rc;
      CU(ctx, cudaMemcpyAsync(d_vin, b.var_in + L.pv_upto(begin), cpv * 4, cudaMemcpyHostToDevice, st));
    }
    void *d_out = nullptr;
    const bool want_mat = b.matrices_out != nullptr || b.post_pass() || b.keep_final;
    // K1t and K1/K1s write the final tableaus apart; the others leave them in the working copy d_in
    const bool out_apart = ragged || (route.resident && route.kind != ROUTE_GRID);
    if (want_mat && out_apart)
      if ((rc = dev_ensure(ctx, "matout" + s, ccells * 8, &d_out))) return rc;

    const double *src = b.matrices + (ragged ? b.mat_offsets[begin] : L.cells_upto(begin));
    if (ragged) {
      // caller offsets may be non-contiguous: copy LP by LP when they are
      bool contiguous = true;
      for (int64_t i = begin; i < end && contiguous; i++)
        contiguous = (b.mat_offsets[i] - b.mat_offsets[begin]) == (L.moff[i] - L.moff[begin]);
      if (contiguous) {
        CU(ctx, cudaMemcpyAsync(d_in, src, ccells * 8, cudaMemcpyHostToDevice, st));
      } else {
        for (int64_t i = begin; i < end; i++)
          CU(ctx, cudaMemcpyAsync((double *)d_in + (L.moff[i] - L.moff[begin]), b.matrices + b.mat_offsets[i],
                                  (size_t)b.heights[i] * b.widths[i] * 8, cudaMemcpyHostToDevice, st));
      }
    } else if (from_cells) {
      if ((rc = scatter_cells(ctx, b, (double *)d_in, ccells, st))) return rc;
    } else {
      CU(ctx, cudaMemcpyAsync(d_in, src, ccells * 8, cudaMemcpyHostToDevice, st));
    }

    BatchArgs a{};
    a.n = cn;
    a.mode = kModeBatch;
    a.H = L.height;
    a.W = L.width;
    a.Hcap = chcap;
    a.Wcap = cwcap;
    a.in = (const double *)d_in;
    a.work = (double *)d_in;  // K2 works in place on the device copy
    a.mat_out = want_mat ? (out_apart ? (double *)d_out : (double *)d_in) : nullptr;
    set_outputs(a, dev);
    a.var_in = (const int *)d_vin;
    std::vector<long long> lm, lr, lpv;  // chunk-local offsets of a ragged chunk
    if (ragged) {
      void *d_h, *d_w, *d_mo, *d_ro, *d_po;
      lm.resize(cn), lr.resize(cn), lpv.resize(cn);
      for (int64_t i = 0; i < cn; i++) {
        lm[i] = L.moff[begin + i] - L.moff[begin];
        lr[i] = L.roff[begin + i] - L.roff[begin];
        lpv[i] = L.poff[begin + i] - L.poff[begin];
      }
      if ((rc = dev_ensure(ctx, "rg_h" + s, (size_t)cn * 4, &d_h))) return rc;
      if ((rc = dev_ensure(ctx, "rg_w" + s, (size_t)cn * 4, &d_w))) return rc;
      if ((rc = dev_ensure(ctx, "rg_mo" + s, (size_t)cn * 8, &d_mo))) return rc;
      if ((rc = dev_ensure(ctx, "rg_ro" + s, (size_t)cn * 8, &d_ro))) return rc;
      if ((rc = dev_ensure(ctx, "rg_po" + s, (size_t)cn * 8, &d_po))) return rc;
      CU(ctx, cudaMemcpyAsync(d_h, b.heights + begin, (size_t)cn * 4, cudaMemcpyHostToDevice, st));
      CU(ctx, cudaMemcpyAsync(d_w, b.widths + begin, (size_t)cn * 4, cudaMemcpyHostToDevice, st));
      CU(ctx, cudaMemcpyAsync(d_mo, lm.data(), (size_t)cn * 8, cudaMemcpyHostToDevice, st));
      CU(ctx, cudaMemcpyAsync(d_ro, lr.data(), (size_t)cn * 8, cudaMemcpyHostToDevice, st));
      CU(ctx, cudaMemcpyAsync(d_po, lpv.data(), (size_t)cn * 8, cudaMemcpyHostToDevice, st));
      CU(ctx, cudaStreamSynchronize(st));  // the staging vectors die at the end of the chunk
      a.heights = (const int *)d_h;
      a.widths = (const int *)d_w;
      a.mat_off = (const long long *)d_mo;
      a.rhs_off = (const long long *)d_ro;
      a.pos_off = (const long long *)d_po;
    }
    fill_options(a, opt);
    if (!ragged) {
      if ((rc = launch_route(ctx, route, a, s, st))) return rc;
      if (b.post_pass() && (rc = post_passes(ctx, b, a, a.mat_out, (const int *)d_pairs, dev, cpv, s, st))) return rc;
    } else {
      // Ragged chunk: LPs of very different sizes must not share one launch configuration (one large model would
      // push a thousand small ones onto the HBM-resident kernel).  Group by (fits in shared memory, CTA width) and
      // route each group on its own through an index indirection.
      std::vector<std::vector<int>> groups;
      std::vector<std::pair<int, int>> caps;  // (Hcap, Wcap) per group
      std::unordered_map<int, int> group_of;
      for (int64_t i = 0; i < cn; i++) {
        const int hi = b.heights[begin + i], wi = b.widths[begin + i];
        const bool res = SmemLayout(hi, wi, true, 32).total <= (size_t)ctx->smem_optin;
        const int key = (res ? 0 : 64) + default_warps((long long)hi * wi, res);
        auto it = group_of.find(key);
        if (it == group_of.end()) {
          it = group_of.emplace(key, (int)groups.size()).first;
          groups.emplace_back();
          caps.emplace_back(1, 1);
        }
        groups[it->second].push_back((int)i);
        caps[it->second].first = std::max(caps[it->second].first, hi);
        caps[it->second].second = std::max(caps[it->second].second, wi);
      }
      std::vector<int> flat;
      for (auto &g : groups) flat.insert(flat.end(), g.begin(), g.end());
      void *d_index;
      if ((rc = dev_ensure(ctx, "rg_index" + s, flat.size() * 4, &d_index))) return rc;
      CU(ctx, cudaMemcpyAsync(d_index, flat.data(), flat.size() * 4, cudaMemcpyHostToDevice, st));
      CU(ctx, cudaStreamSynchronize(st));
      BatchArgs h{};  // host-side copies of the shape, offset and index arrays (K4 reads them on the host)
      h.heights = b.heights + begin;
      h.widths = b.widths + begin;
      h.mat_off = lm.data();
      h.rhs_off = lr.data();
      h.pos_off = lpv.data();
      size_t at = 0;
      for (size_t g = 0; g < groups.size(); g++) {
        BatchArgs ga = a;
        ga.n = (long long)groups[g].size();
        ga.Hcap = caps[g].first;
        ga.Wcap = caps[g].second;
        ga.index = (const int *)d_index + at;
        h.index = flat.data() + at;
        if ((rc = choose_route(ctx, {ga.n, ga.Hcap, ga.Wcap, groups.size() == 1 ? density : -1.0, opt->check_cycles != 0, true},
                               &route)))
          return rc;
        if ((rc = launch_route(ctx, route, ga, s, st, &h))) return rc;
        if (b.post_pass() && (rc = post_passes(ctx, b, ga, a.mat_out, (const int *)d_pairs, dev, cpv, s, st))) return rc;
        at += groups[g].size();
      }
    }

    if ((rc = outs.copy_out(ctx, dev, begin, L.rows_upto(begin), L.pv_upto(begin), cn, crows, cpv, st))) return rc;
    if (b.keep_final) b.kept_final = a.mat_out;
    if (b.matrices_out) {
      if (ragged) {
        for (int64_t i = begin; i < end; i++)
          CU(ctx, cudaMemcpyAsync(b.matrices_out + b.mat_offsets[i], (double *)a.mat_out + (L.moff[i] - L.moff[begin]),
                                  (size_t)b.heights[i] * b.widths[i] * 8, cudaMemcpyDeviceToHost, st));
      } else {
        CU(ctx, cudaMemcpyAsync(b.matrices_out + L.cells_upto(begin), a.mat_out, ccells * 8, cudaMemcpyDeviceToHost, st));
      }
    }
    CU(ctx, cudaEventRecord(ctx->events[slot], st));
    used[slot] = true;
    slot ^= 1;
    begin = end;
  }
  for (int i = 0; i < 2; i++)
    if (used[i]) CU(ctx, cudaStreamSynchronize(ctx->streams[i]));
  return check_device_status(ctx, b.status, n);
}

// Shared host-side solve of uniform and ragged batches: the zero-copy small call when the batch qualifies, else the
// pipelined chunks.
int solve_host(yalps_ctx *ctx, HostBatch &b) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  BatchLayout L;
  if (int rc = batch_layout(ctx, b, &L)) return rc;
  if (b.n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  bool taken;
  if (int rc = solve_small(ctx, b, L, &taken)) return rc;
  return taken ? 0 : solve_chunks(ctx, b, L);
}

// The request of a yalps_solve_{batch,ragged}_certificate call (heights null: a uniform batch of height x width).
HostBatch batch_request(int64_t n, int32_t height, int32_t width, const int32_t *heights, const int32_t *widths,
                        const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                        const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                        int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out, double *matrices_out,
                        double *reduced_out, const int32_t *pairs, double *range_lo, double *range_hi,
                        double *cert_out) {
  HostBatch b;
  b.n = n;
  b.height = height;
  b.width = width;
  b.heights = heights;
  b.widths = widths;
  b.mat_offsets = mat_offsets;
  b.matrices = matrices;
  b.pos_in = pos_in;
  b.var_in = var_in;
  b.pairs = pairs;
  b.opt = opt;
  b.status = status;
  b.value = value;
  b.pivots = pivots;
  b.rhs_out = rhs_out;
  b.pos_out = pos_out;
  b.var_out = var_out;
  b.matrices_out = matrices_out;
  b.reduced_out = reduced_out;
  b.range_lo = range_lo;
  b.range_hi = range_hi;
  b.cert_out = cert_out;
  return b;
}

}  // namespace

extern "C" {

int yalps_solve_batch(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                      const yalps_options *opt, int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                      int32_t *pos_out, int32_t *var_out, double *matrices_out) {
  return yalps_solve_batch_ranging(ctx, n, height, width, matrices, nullptr, nullptr, opt, status, value, pivots, rhs_out,
                                   pos_out, var_out, matrices_out, nullptr, nullptr, nullptr, nullptr);
}

int yalps_solve_ragged(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                       const int64_t *mat_offsets, const double *matrices, const yalps_options *opt, int32_t *status,
                       double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                       double *matrices_out) {
  return yalps_solve_ragged_ranging(ctx, n, heights, widths, mat_offsets, matrices, nullptr, nullptr, opt, status, value,
                                    pivots, rhs_out, pos_out, var_out, matrices_out, nullptr, nullptr, nullptr, nullptr);
}

int yalps_solve_batch_basis(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                            const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                            double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                            double *matrices_out) {
  return yalps_solve_batch_ranging(ctx, n, height, width, matrices, pos_in, var_in, opt, status, value, pivots, rhs_out,
                                   pos_out, var_out, matrices_out, nullptr, nullptr, nullptr, nullptr);
}

int yalps_solve_ragged_basis(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                             const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                             const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                             int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                             double *matrices_out) {
  return yalps_solve_ragged_ranging(ctx, n, heights, widths, mat_offsets, matrices, pos_in, var_in, opt, status, value,
                                    pivots, rhs_out, pos_out, var_out, matrices_out, nullptr, nullptr, nullptr, nullptr);
}

int yalps_solve_batch_duals(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                            const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                            double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                            double *matrices_out, double *reduced_out) {
  return yalps_solve_batch_ranging(ctx, n, height, width, matrices, pos_in, var_in, opt, status, value, pivots, rhs_out,
                                   pos_out, var_out, matrices_out, reduced_out, nullptr, nullptr, nullptr);
}

int yalps_solve_ragged_duals(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                             const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                             const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                             int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                             double *matrices_out, double *reduced_out) {
  return yalps_solve_ragged_ranging(ctx, n, heights, widths, mat_offsets, matrices, pos_in, var_in, opt, status, value,
                                    pivots, rhs_out, pos_out, var_out, matrices_out, reduced_out, nullptr, nullptr,
                                    nullptr);
}

int yalps_solve_batch_ranging(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                              const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                              double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                              double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                              double *range_hi) {
  return yalps_solve_batch_certificate(ctx, n, height, width, matrices, pos_in, var_in, opt, status, value, pivots,
                                       rhs_out, pos_out, var_out, matrices_out, reduced_out, pairs, range_lo, range_hi,
                                       nullptr);
}

int yalps_solve_ragged_ranging(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                               const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                               const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                               int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                               double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                               double *range_hi) {
  return yalps_solve_ragged_certificate(ctx, n, heights, widths, mat_offsets, matrices, pos_in, var_in, opt, status,
                                        value, pivots, rhs_out, pos_out, var_out, matrices_out, reduced_out, pairs,
                                        range_lo, range_hi, nullptr);
}

int yalps_solve_batch_certificate(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                                  const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt,
                                  int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                                  int32_t *var_out, double *matrices_out, double *reduced_out, const int32_t *pairs,
                                  double *range_lo, double *range_hi, double *cert_out) {
  HostBatch b = batch_request(n, height, width, nullptr, nullptr, nullptr, matrices, pos_in, var_in, opt, status, value,
                              pivots, rhs_out, pos_out, var_out, matrices_out, reduced_out, pairs, range_lo, range_hi,
                              cert_out);
  return solve_host(ctx, b);
}

int yalps_solve_ragged_certificate(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                                   const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                                   const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                                   int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                                   double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                                   double *range_hi, double *cert_out) {
  if (!heights) return fail(ctx, YALPS_ERR_ARGUMENT, "heights is null");
  HostBatch b = batch_request(n, 0, 0, heights, widths, mat_offsets, matrices, pos_in, var_in, opt, status, value,
                              pivots, rhs_out, pos_out, var_out, matrices_out, reduced_out, pairs, range_lo, range_hi,
                              cert_out);
  return solve_host(ctx, b);
}

// ---- replica path sharing (aux_kernels.cuh: k_replica_follow) ------------------------------------------------------
// The leader (the base tableau itself) is solved once by a row-split kernel that records its trace; see the comment
// above FollowArgs for why following it gives every replica its own result, bit for bit.
struct ReplicaTrace {
  bool ok = false;
  int K = 0, Hp = 0, cap = 0, leader_done = 0, leader_status = 0;
  int *steps = nullptr, *var = nullptr;
  double *q = nullptr, *col = nullptr, *snap = nullptr;
  double *red = nullptr;  // the leader's final reduced costs (when the caller asked for them)
  double density = -1.0;
};

static int replica_leader_trace(yalps_ctx *ctx, int H, int W, const double *base_host, const double *d_base,
                                const yalps_options *opt, cudaStream_t st, ReplicaTrace *tr, bool want_red) {
  tr->ok = false;
  if (!ctx->replica_sharing || opt->check_cycles || getenv("YALPS_NO_REPLICA_SHARING")) return 0;
  if (ctx->tune_path != YALPS_PATH_AUTO) return 0;  // a forced kernel path means "measure that kernel"
  const size_t cells = (size_t)H * W, pv = (size_t)H + W;
  const SmemLayout Lg(H, W, false, 32);
  if (Lg.total > (size_t)ctx->smem_optin) return 0;  // the forks need a one-CTA-per-LP kernel
  // trace capacity: both phases of the budget, bounded by 512 MiB of snapshots
  const double budget = !(opt->max_pivots > 0.0) ? 0.0 : std::min(opt->max_pivots, 1.0e6);
  long long cap = (long long)std::min(2.0 * std::ceil(budget), 4096.0);
  cap = std::min<long long>(cap, (long long)(((size_t)512 << 20) / (cells * 8)) - 1);
  if (cap < 8) return 0;
  Route route;
  RouteRequest q{1, H, W};
  q.table_only = true;
  if (int rc = choose_route(ctx, q, &route)) return rc;
  if (route.kind != ROUTE_SIMPLEX || route.k->nwr < 2) return 0;  // only the row-split kernels record a trace
  size_t nz = 0;
  for (size_t i = 0; i < cells; i++) nz += base_host[i] != 0.0;
  tr->density = (double)nz / (double)cells;
  tr->Hp = (H + 1) & ~1;
  tr->cap = (int)cap;
  void *p;
  int rc;
  if ((rc = dev_ensure(ctx, "rs_steps", (size_t)(cap + 1) * 4 * sizeof(int), &p))) return rc;
  tr->steps = (int *)p;
  if ((rc = dev_ensure(ctx, "rs_q", (size_t)cap * 8, &p))) return rc;
  tr->q = (double *)p;
  if ((rc = dev_ensure(ctx, "rs_col", (size_t)cap * tr->Hp * 8, &p))) return rc;
  tr->col = (double *)p;
  if ((rc = dev_ensure(ctx, "rs_snap", (size_t)(cap + 1) * cells * 8, &p))) return rc;
  tr->snap = (double *)p;
  if ((rc = dev_ensure(ctx, "rs_var", (size_t)(cap + 1) * pv * sizeof(int), &p))) return rc;
  tr->var = (int *)p;
  void *d_lwork, *d_lres, *d_lpv;
  if ((rc = dev_ensure(ctx, "rs_lwork", cells * 8, &d_lwork))) return rc;
  if ((rc = dev_ensure(ctx, "rs_lres", 64, &d_lres))) return rc;
  if ((rc = dev_ensure(ctx, "rs_lpv", 2 * pv * sizeof(int), &d_lpv))) return rc;
  tr->red = nullptr;
  if (want_red) {
    if ((rc = dev_ensure(ctx, "rs_lred", pv * 8, &p))) return rc;
    tr->red = (double *)p;
  }
  BatchArgs a{};
  a.n = 1;
  a.mode = kModeBatch;
  a.H = a.Hcap = H;
  a.W = a.Wcap = W;
  a.in = d_base;
  a.work = (double *)d_lwork;
  a.status = (int *)d_lres;
  a.value = (double *)((char *)d_lres + 8);
  a.pivots = (long long *)((char *)d_lres + 16);
  a.pos_out = (int *)d_lpv;
  a.var_out = (int *)d_lpv + pv;
  a.red_out = tr->red;
  fill_options(a, opt);
  a.tr_steps = tr->steps;
  a.tr_q = tr->q;
  a.tr_col = tr->col;
  a.tr_snap = tr->snap;
  a.tr_var = tr->var;
  a.tr_hp = tr->Hp;
  a.tr_cap = tr->cap;
  if ((rc = launch_route(ctx, route, a, "rs_lead", st))) return rc;
  struct {
    int status, pad;
    double value;
    long long p1, p2;
  } res;
  CU(ctx, cudaMemcpyAsync(&res, d_lres, sizeof res, cudaMemcpyDeviceToHost, st));
  CU(ctx, cudaStreamSynchronize(st));
  if (res.status == ST_ERR_HISTORY) return 0;
  const long long K = res.p1 + res.p2;
  // a trace that did not fit ends one step early: snapshots exist for the states BEFORE pivots 0 .. cap - 1 only
  tr->leader_done = K <= cap;
  tr->K = (int)(K <= cap ? K : cap - 1);
  tr->leader_status = res.status;
  tr->ok = true;
  return 0;
}

// One chunk of replicas whose right-hand sides are in d_rin, results into the chunk's outputs dev (outs.ensure):
// followers first, then the replicas that left the path (tableau = the leader's snapshot of the fork step + their own
// column 0) through the ordinary batch kernels, into compact outputs of their own scattered back into dev.
static int replica_chunk_shared(yalps_ctx *ctx, const ReplicaTrace &tr, const Outputs &outs, int64_t cn, int H, int W,
                                const double *d_rin, double *d_work, const yalps_options *opt, void *const *dev,
                                cudaStream_t st, const std::string &s, int64_t *forks_out) {
  const size_t cells = (size_t)H * W, pv = (size_t)H + W;
  void *p, *hp;
  int rc;
  if ((rc = dev_ensure(ctx, "rs_fcount" + s, 64, &p))) return rc;
  int *d_fcount = (int *)p;
  if ((rc = dev_ensure(ctx, "rs_fids" + s, (size_t)cn * 4, &p))) return rc;
  int *d_fids = (int *)p;
  if ((rc = dev_ensure(ctx, "rs_fstep" + s, (size_t)cn * 4, &p))) return rc;
  int *d_fstep = (int *)p;
  if ((rc = dev_ensure(ctx, "rs_fres" + s, (size_t)cn * 24, &p))) return rc;
  long long *d_fres = (long long *)p;
  if ((rc = pin_ensure(ctx, "rs_fcount_h" + s, 64, &hp))) return rc;
  CU(ctx, cudaMemsetAsync(d_fcount, 0, 4, st));
  BatchArgs d{};  // the chunk's outputs, typed
  set_outputs(d, dev);
  FollowArgs fa{};
  fa.n = cn;
  fa.H = H;
  fa.W = W;
  fa.Hp = tr.Hp;
  fa.rhs_in = d_rin;
  fa.steps = tr.steps;
  fa.q = tr.q;
  fa.colraw = tr.col;
  fa.leader_var = tr.var + (size_t)tr.K * pv;
  fa.K = tr.K;
  fa.leader_done = tr.leader_done;
  fa.leader_status = tr.leader_status;
  fa.precision = opt->precision;
  fa.max_pivots = opt->max_pivots;
  fa.status = d.status;
  fa.value = d.value;
  fa.pivots = d.pivots;
  fa.rhs_out = d.rhs_out;
  fa.pos_out = d.pos_out;
  fa.var_out = d.var_out;
  fa.fork_count = d_fcount;
  fa.fork_ids = d_fids;
  fa.fork_step = d_fstep;
  fa.fork_resume = d_fres;
  fa.red_out = d.red_out;
  fa.leader_red = tr.red;
  const int grid = (int)std::min<int64_t>((cn + kFollowWarps - 1) / kFollowWarps, (int64_t)ctx->prop.multiProcessorCount * 8);
  k_replica_follow<<<grid, kFollowWarps * 32, (size_t)kFollowWarps * tr.Hp * 8, st>>>(fa);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  CU(ctx, cudaMemcpyAsync(hp, d_fcount, 4, cudaMemcpyDeviceToHost, st));
  CU(ctx, cudaStreamSynchronize(st));
  const int nf = *(int *)hp;
  if (forks_out) *forks_out += nf;
  if (nf == 0) return 0;
  // compact buffers of the forked replicas: their resume state and basis in, their outputs
  if ((rc = dev_ensure(ctx, "rs_cvin" + s, (size_t)nf * pv * 4, &p))) return rc;
  int *c_vin = (int *)p;
  if ((rc = dev_ensure(ctx, "rs_cres" + s, (size_t)nf * 24, &p))) return rc;
  long long *c_resume = (long long *)p;
  const std::string fs = "rs_fork" + s;
  void *cdev[O_COUNT];
  if ((rc = outs.ensure(ctx, fs, nf, (long long)nf * H, (long long)nf * pv, cdev))) return rc;
  {
    const dim3 g((unsigned)std::min<size_t>((cells + 255) / 256, 64), (unsigned)std::min(nf, 32768));
    k_replica_materialise<<<g, 256, 0, st>>>(0, nf, H, W, d_fids, d_fstep, d_fres, d.rhs_out, tr.snap, tr.var, d_work,
                                             c_vin, c_resume);
    CU(ctx, cudaGetLastError());
    ctx->launches++;
  }
  // one CTA per fork, also where K4 would take a batch of this size: a plan that K4 would replace is already the
  // HBM-resident kernel
  Route route;
  RouteRequest q{nf, H, W, tr.density};
  q.table_only = true;
  if ((rc = choose_route(ctx, q, &route))) return rc;
  if (route.kind != ROUTE_SIMPLEX) return fail(ctx, YALPS_ERR_TOO_LARGE, "tableau width %d exceeds the widest kernel", W);
  BatchArgs a{};
  a.n = nf;
  a.mode = kModeBatch;
  a.H = a.Hcap = H;
  a.W = a.Wcap = W;
  a.in = d_work;
  a.work = d_work;
  set_outputs(a, cdev);
  a.var_in = c_vin;
  a.resume = c_resume;
  fill_options(a, opt);
  if ((rc = launch_route(ctx, route, a, fs, st))) return rc;
  k_replica_scatter<<<(unsigned)std::min(nf, ctx->prop.multiProcessorCount * 8), 128, 0, st>>>(
      0, nf, H, W, d_fids, a.status, a.value, a.pivots, a.rhs_out, a.pos_out, a.var_out, a.red_out, d.status, d.value,
      d.pivots, d.rhs_out, d.pos_out, d.var_out, d.red_out);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  return 0;
}

// The LPs of a request derived from b.d_base (replicas: b.rhs_in, row subsets: b.keep), in chunks of at most ~1.5 GiB
// of working copies over two pipeline slots: the H2D of chunk k+1's inputs and the D2H of chunk k-1's results overlap
// the solve of chunk k.  Per chunk, on its slot's stream: the per-LP inputs in; the replicas' shared path when `trace`
// is usable, else the expand kernel and the solve in place; the post-passes, k_cert_support, the results out.
// Returns once every copy has landed.
static int solve_from_base(yalps_ctx *ctx, HostBatch &b, const ReplicaTrace *trace) {
  const int64_t n = b.n;
  const int H = b.height, W = b.width, words = (H + 31) / 32;
  const size_t cells = (size_t)H * W, pv = (size_t)H + W, in_lp = b.keep ? (size_t)words * 4 : (size_t)H * 8;
  const long long sms = ctx->prop.multiProcessorCount;
  const int64_t per_chunk = std::max<int64_t>(1, std::min<int64_t>((n + 1) / 2 > 4096 ? (n + 7) / 8 : n,
                                                                  (int64_t)(((size_t)1536 << 20) / (cells * 8))));
  const Outputs outs(b);
  bool used[2] = {false, false};
  int slot = 0, rc;
  for (int64_t begin = 0; begin < n; begin += per_chunk, slot ^= 1) {
    const int64_t cn = std::min(per_chunk, n - begin);
    const std::string s = (b.keep ? "ss" : "rp") + std::to_string(slot);
    cudaStream_t st = ctx->streams[slot];
    if (used[slot]) CU(ctx, cudaEventSynchronize(ctx->events[slot]));
    void *d_in, *d_work, *dev[O_COUNT];
    if ((rc = dev_ensure(ctx, (b.keep ? "keep" : "rin") + s, cn * in_lp, &d_in))) return rc;
    if ((rc = dev_ensure(ctx, "work" + s, (size_t)cn * cells * 8, &d_work))) return rc;
    if ((rc = outs.ensure(ctx, s, cn, cn * H, cn * (long long)pv, dev))) return rc;
    const char *in = b.keep ? (const char *)b.keep : (const char *)b.rhs_in;
    CU(ctx, cudaMemcpyAsync(d_in, in + begin * in_lp, cn * in_lp, cudaMemcpyHostToDevice, st));
    BatchArgs a{};
    a.n = cn;
    a.H = a.Hcap = H;
    a.W = a.Wcap = W;
    a.work = (double *)d_work;
    a.in = a.work;
    // in place: every route reads an LP's tableau before it writes that LP's final one
    a.mat_out = b.post_pass() ? a.work : nullptr;
    set_outputs(a, dev);
    if (trace && trace->ok) {
      if ((rc = replica_chunk_shared(ctx, *trace, outs, cn, H, W, (const double *)d_in, a.work, b.opt, dev, st, s,
                                     &ctx->replica_forks)))
        return rc;
    } else {
      if (b.keep) {
        const int grid = (int)std::min<long long>((cn * H + 7) / 8, sms * 16);
        k_expand_subsets<<<grid, 256, 0, st>>>(cn, H, W, words, b.d_base, (const unsigned *)d_in, a.work);
      } else {
        const int grid = (int)std::min<long long>((cn * (long long)cells + 255) / 256, sms * 16);
        k_expand_replicas<<<grid, 256, 0, st>>>(cn, H, W, b.d_base, (const double *)d_in, a.work);
      }
      CU(ctx, cudaGetLastError());
      ctx->launches++;
      // The route's density probe is cached per (buffer, shape), so later calls on this pooled buffer -- the later
      // rounds of an IIS search -- reuse the first call's route choice.  That decides speed only, never a result bit.
      if ((rc = solve_batch_device_impl(ctx, a, b.opt, s, st, begin))) return rc;
    }
    if ((rc = post_passes(ctx, b, a, a.work, nullptr, dev, cn * pv, s, st))) return rc;
    if (b.want_support()) {
      const int grid = (int)std::min<long long>((cn + 7) / 8, sms * 16);
      k_cert_support<<<grid, 256, 0, st>>>(cn, H, W, words, a.status, (const double *)dev[O_CERT],
                                           (unsigned *)dev[O_SUP], (int *)dev[O_CNT]);
      CU(ctx, cudaGetLastError());
      ctx->launches++;
    }
    if ((rc = outs.copy_out(ctx, dev, begin, begin * H, begin * (long long)pv, cn, cn * H, cn * (long long)pv, st)))
      return rc;
    CU(ctx, cudaEventRecord(ctx->events[slot], st));
    used[slot] = true;
  }
  for (int i = 0; i < 2; i++)
    if (used[i]) CU(ctx, cudaStreamSynchronize(ctx->streams[i]));
  return check_device_status(ctx, b.status, n);
}

// The replicas of request b (b.rhs_in) of the host base tableau `base`: the base crosses PCIe once, the leader's trace
// is recorded when path sharing applies, then solve_from_base.  Every rank of a multi-GPU call runs its slice here.
static int solve_replicas(yalps_ctx *ctx, const double *base, HostBatch &b) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  const int64_t n = b.n;
  const int32_t height = b.height, width = b.width;
  if (n < 0 || height < 1 || width < 1 || !b.opt || (n > 0 && (!base || !b.rhs_in)))
    return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments (n=%lld, %dx%d)", (long long)n, height, width);
  if ((long long)height * width >= (1LL << 31)) return fail(ctx, YALPS_ERR_TOO_LARGE, "height*width must be < 2^31");
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  const size_t cells = (size_t)height * width;
  void *d_base;
  int rc;
  if ((rc = dev_ensure(ctx, "rep_base", cells * 8, &d_base))) return rc;
  CU(ctx, cudaMemcpy(d_base, base, cells * 8, cudaMemcpyHostToDevice));
  b.d_base = (const double *)d_base;
  ReplicaTrace trace;
  if ((rc = replica_leader_trace(ctx, height, width, base, b.d_base, b.opt, ctx->streams[0], &trace,
                                 b.reduced_out != nullptr)))
    return rc;
  ctx->replica_forks = trace.ok ? 0 : -1;
  return solve_from_base(ctx, b, &trace);
}

int yalps_solve_replicas_duals(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *base,
                               const double *rhs, const yalps_options *opt, int32_t *status, double *value,
                               int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                               double *reduced_out) {
  HostBatch b = batch_request(n, height, width, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, opt, status, value,
                              pivots, rhs_out, pos_out, var_out, nullptr, reduced_out, nullptr, nullptr, nullptr,
                              nullptr);
  b.rhs_in = rhs;
  return solve_replicas(ctx, base, b);
}

int yalps_solve_replicas(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *base,
                         const double *rhs, const yalps_options *opt, int32_t *status, double *value, int64_t *pivots,
                         double *rhs_out, int32_t *pos_out, int32_t *var_out) {
  return yalps_solve_replicas_duals(ctx, n, height, width, base, rhs, opt, status, value, pivots, rhs_out, pos_out,
                                    var_out, nullptr);
}

int yalps_set_replica_sharing(yalps_ctx *ctx, int32_t on) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  ctx->replica_sharing = on ? 1 : 0;
  return 0;
}

int64_t yalps_replica_forks(const yalps_ctx *ctx) { return ctx ? ctx->replica_forks : -1; }

int yalps_generate_synthetic_device(yalps_ctx *ctx, int64_t first, int64_t n, int32_t m, int32_t nvars,
                                    int32_t neg_rows, uint32_t salt, double *d_out, void *stream) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (n < 0 || m < 0 || nvars < 0 || !d_out) return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments");
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  const size_t total = (size_t)n * (m + 1) * (nvars + 1);
  const int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)ctx->prop.multiProcessorCount * 16);
  k_generate_synthetic<<<grid, 256, 0, (cudaStream_t)stream>>>(first, n, m, nvars, neg_rows, salt, d_out);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  return 0;
}

int yalps_generate_replicas_device(yalps_ctx *ctx, int64_t first, int64_t n, int32_t height, int32_t width,
                                   const double *base_host, const int32_t *group_host, int32_t ngroups, double eps,
                                   uint32_t salt, double *d_out, void *stream) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (n < 0 || height < 1 || width < 1 || !base_host || !group_host || !d_out)
    return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments");
  (void)ngroups;
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  void *d_base, *d_group;
  const size_t cells = (size_t)height * width;
  if (int rc = dev_ensure(ctx, "rep_base", cells * 8, &d_base)) return rc;
  if (int rc = dev_ensure(ctx, "rep_group", (size_t)height * 4, &d_group)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CU(ctx, cudaMemcpyAsync(d_base, base_host, cells * 8, cudaMemcpyHostToDevice, st));
  CU(ctx, cudaMemcpyAsync(d_group, group_host, (size_t)height * 4, cudaMemcpyHostToDevice, st));
  const size_t total = (size_t)n * cells;
  const int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)ctx->prop.multiProcessorCount * 16);
  k_generate_replicas<<<grid, 256, 0, st>>>(first, n, height, width, (const double *)d_base, (const int *)d_group, eps,
                                            salt, d_out);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaStreamSynchronize(st));  // base_host / group_host may be pageable
  ctx->launches++;
  return 0;
}

int yalps_round_to_precision(yalps_ctx *ctx, int64_t n, const double *x, double precision, double *out) {
  if (!ctx) return YALPS_ERR_ARGUMENT;
  if (n < 0 || (n > 0 && (!x || !out))) return fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments");
  if (n == 0) return 0;
  CU(ctx, cudaSetDevice(ctx->device));
  void *d_x, *d_o;
  if (int rc = dev_ensure(ctx, "round_x", (size_t)n * 8, &d_x)) return rc;
  if (int rc = dev_ensure(ctx, "round_o", (size_t)n * 8, &d_o)) return rc;
  cudaStream_t st = ctx->streams[0];
  CU(ctx, cudaMemcpyAsync(d_x, x, (size_t)n * 8, cudaMemcpyHostToDevice, st));
  k_round_to_precision<<<(int)((n + 255) / 256), 256, 0, st>>>(n, (const double *)d_x, precision, (double *)d_o);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  CU(ctx, cudaMemcpyAsync(out, d_o, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
  CU(ctx, cudaStreamSynchronize(st));
  return 0;
}

int yalps_probe_division(yalps_ctx *ctx, int64_t n, uint64_t seed, int32_t mode, uint64_t *mismatches,
                         uint64_t *first_bad_bits) {
  if (!ctx || !mismatches || n < 0 || mode < 0 || mode > 4) return YALPS_ERR_ARGUMENT;
  CU(ctx, cudaSetDevice(ctx->device));
  void *d;
  if (int rc = dev_ensure(ctx, "probe_div", 32, &d)) return rc;
  cudaStream_t st = ctx->streams[0];
  CU(ctx, cudaMemsetAsync(d, 0, 32, st));
  k_probe_division<<<ctx->prop.multiProcessorCount * 8, 256, 0, st>>>(n, seed, mode, (unsigned long long *)d);
  CU(ctx, cudaGetLastError());
  ctx->launches++;
  unsigned long long h[4];
  CU(ctx, cudaMemcpyAsync(h, d, 32, cudaMemcpyDeviceToHost, st));
  CU(ctx, cudaStreamSynchronize(st));
  *mismatches = h[0];
  if (first_bad_bits) {
    first_bad_bits[0] = h[2];
    first_bad_bits[1] = h[3];
  }
  return 0;
}

int yalps_measure_smem_bandwidth(yalps_ctx *ctx, double *gbs, double *sm_clock_mhz) {
  if (!ctx || !gbs) return YALPS_ERR_ARGUMENT;
  CU(ctx, cudaSetDevice(ctx->device));
  const int words = 24 * 1024 / 8 * 4;  // 96 KiB per CTA, 2 CTAs per SM
  const int threads = 512, iters = 2000;
  const size_t smem = (size_t)words * 8;
  CU(ctx, raise_smem_limit(ctx->device, (const void *)k_smem_stream, (int)smem));
  void *sink;
  if (int rc = dev_ensure(ctx, "sink", 64, &sink)) return rc;
  const int grid = ctx->prop.multiProcessorCount * 2;
  cudaStream_t st = ctx->streams[0];
  cudaEvent_t e0, e1;
  CU(ctx, cudaEventCreate(&e0));
  CU(ctx, cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    CU(ctx, cudaEventRecord(e0, st));
    k_smem_stream<<<grid, threads, smem, st>>>(words, iters, (double *)sink);
    CU(ctx, cudaEventRecord(e1, st));
    CU(ctx, cudaEventSynchronize(e1));
    CU(ctx, cudaGetLastError());
    ctx->launches++;
    float ms = 0;
    CU(ctx, cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0) best = std::min(best, ms);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  const double bytes = (double)grid * iters * words * 16.0;
  *gbs = bytes / (best * 1e-3) / 1e9;
  if (sm_clock_mhz) {
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
    *sm_clock_mhz = khz / 1000.0;
  }
  return 0;
}

int yalps_measure_l2_bandwidth(yalps_ctx *ctx, uint64_t bytes, double *gbs) {
  if (!ctx || !gbs || bytes < 4096) return YALPS_ERR_ARGUMENT;
  CU(ctx, cudaSetDevice(ctx->device));
  void *d;
  if (int rc = dev_ensure(ctx, "l2_probe", bytes, &d)) return rc;
  cudaStream_t st = ctx->streams[0];
  CU(ctx, cudaMemsetAsync(d, 0, bytes, st));
  const int iters = 50, grid = ctx->prop.multiProcessorCount * 8;
  cudaEvent_t e0, e1;
  CU(ctx, cudaEventCreate(&e0));
  CU(ctx, cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 4; rep++) {
    CU(ctx, cudaEventRecord(e0, st));
    k_l2_stream<<<grid, 256, 0, st>>>((double2 *)d, bytes / 16, iters, 0.5);
    CU(ctx, cudaEventRecord(e1, st));
    CU(ctx, cudaEventSynchronize(e1));
    CU(ctx, cudaGetLastError());
    ctx->launches++;
    float ms = 0;
    CU(ctx, cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0) best = std::min(best, ms);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *gbs = (double)(bytes / 16 * 16) * iters * 2.0 / (best * 1e-3) / 1e9;
  return 0;
}

int yalps_measure_h2d_bandwidth(yalps_ctx *ctx, const void *pinned_host, uint64_t bytes, int32_t reps, int32_t nstreams,
                                double *seconds) {
  if (!ctx || !pinned_host || !seconds || bytes == 0 || reps < 1 || nstreams < 1 || nstreams > 2)
    return ctx ? fail(ctx, YALPS_ERR_ARGUMENT, "bad arguments") : YALPS_ERR_ARGUMENT;
  CU(ctx, cudaSetDevice(ctx->device));
  void *d;
  if (int rc = dev_ensure(ctx, "h2d_probe", bytes, &d)) return rc;
  const size_t part = ((bytes / nstreams) + 255) & ~(size_t)255;
  CU(ctx, cudaDeviceSynchronize());
  const auto t0 = std::chrono::steady_clock::now();
  for (int r = 0; r < reps; r++)
    for (int k = 0; k < nstreams; k++) {
      const size_t off = (size_t)k * part;
      if (off >= bytes) break;
      const size_t len = std::min(part, (size_t)bytes - off);
      CU(ctx, cudaMemcpyAsync((char *)d + off, (const char *)pinned_host + off, len, cudaMemcpyHostToDevice, ctx->streams[k]));
    }
  for (int k = 0; k < nstreams; k++) CU(ctx, cudaStreamSynchronize(ctx->streams[k]));
  *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / reps;
  return 0;
}

int yalps_measure_tmem_bandwidth(yalps_ctx *ctx, double *gbs, double *sm_clock_mhz) {
  if (!ctx || !gbs) return YALPS_ERR_ARGUMENT;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, raise_smem_limit(ctx->device, tmem_stream_fn(), (int)tmem_stream_dynamic_smem()));
  void *sink;
  if (int rc = dev_ensure(ctx, "sink", 64, &sink)) return rc;
  const int grid = ctx->prop.multiProcessorCount * tmem_stream_ctas_per_sm();
  cudaStream_t st = ctx->streams[0];
  cudaEvent_t e0, e1;
  CU(ctx, cudaEventCreate(&e0));
  CU(ctx, cudaEventCreate(&e1));
  float best = 1e30f;
  double bytes = 0.0;
  for (int rep = 0; rep < 5; rep++) {
    CU(ctx, cudaEventRecord(e0, st));
    CU(ctx, launch_tmem_stream(grid, 4000, (double *)sink, st, &bytes));
    CU(ctx, cudaEventRecord(e1, st));
    CU(ctx, cudaEventSynchronize(e1));
    ctx->launches++;
    float ms = 0;
    CU(ctx, cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0) best = std::min(best, ms);
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *gbs = bytes / (best * 1e-3) / 1e9;
  if (sm_clock_mhz) {
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
    *sm_clock_mhz = khz / 1000.0;
  }
  return 0;
}

}  // extern "C"

#include "bnb.inl"
#include "multi.inl"
#include "iis.inl"
