/*
 * yalps_b200.h -- C ABI of libyalps_b200.so: the B200-native replacement for
 * the YALPS simplex / node-LP hot path.
 *
 * The reference (Ivordir/YALPS, TypeScript) has no FFI; the seam this library
 * replaces is the module-internal call
 *     simplex(tableau, options) -> [status, number]      src/simplex.ts:144
 * made from src/YALPS.ts:79 (root LP) and src/branchAndCut.ts:127 (node LPs),
 * plus applyCuts (src/branchAndCut.ts:22-61) and the branch-and-cut loop
 * (src/branchAndCut.ts:89-176) that issues the node LPs.  A Node N-API addon
 * (bindings/node/, see INTEGRATION.md) binds exactly these entry points.
 *
 * Conventions
 *  - Tableau layout is the reference's (src/tableau.ts:9-21): row-major fp64,
 *    `matrix[row*width + col]`, row 0 = objective row, column 0 = RHS;
 *    positionOfVariable / variableAtPosition are int32[width+height] and start
 *    as the identity (src/tableau.ts:95-98), so the batch entry points create
 *    them on the device instead of taking them as inputs.
 *  - All pointers are plain host pointers unless the name says `_device`.
 *    The caller owns every buffer; nothing is retained past the call except
 *    through the ctx (root tableau of a branch-and-cut session).
 *  - Every function returns 0 on success and a negative yalps_error on
 *    failure; yalps_last_error() gives the message.  Nothing throws across
 *    the ABI.  There is no CPU fallback: without a CUDA device every compute
 *    entry point fails with YALPS_ERR_CUDA.
 *  - Arithmetic is IEEE-754 binary64 with the reference's operation order
 *    (no FMA contraction, true divisions); statuses, pivot counts, bases and
 *    values are bit-identical to the reference loop on the same input.
 *  - A ctx is not thread-safe; use one per host thread (the reference is
 *    synchronous on the JS main thread, so `solve` blocks).
 */
#ifndef YALPS_B200_H
#define YALPS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct yalps_ctx yalps_ctx;

/* SolutionStatus, src/types.ts:154 (same spelling order as STATUS_NAMES in the host layer). */
enum yalps_status {
  YALPS_OPTIMAL = 0,
  YALPS_INFEASIBLE = 1,
  YALPS_UNBOUNDED = 2,
  YALPS_TIMEDOUT = 3, /* branch-and-cut only, src/branchAndCut.ts:171 */
  YALPS_CYCLED = 4
};

enum yalps_error {
  YALPS_OK = 0,
  YALPS_ERR_CUDA = -1,     /* CUDA runtime failure or no device */
  YALPS_ERR_ARGUMENT = -2, /* bad sizes / null pointers */
  YALPS_ERR_TOO_LARGE = -3,/* tableau exceeds what any kernel path supports */
  YALPS_ERR_HISTORY = -4   /* checkCycles history buffer exhausted (see max_pivots) */
};

/* Required<Options>, src/types.ts:203-265, defaults src/YALPS.ts:52-60.
 * max_pivots, timeout_ms and max_iterations may be +infinity
 * (benchmarks/runners.ts:10 passes maxPivots: Infinity). */
typedef struct yalps_options {
  double precision;      /* 1e-8 */
  double max_pivots;     /* 8192, per phase (src/simplex.ts:69,109) */
  double tolerance;      /* 0 */
  double timeout_ms;     /* +inf */
  double max_iterations; /* 32768 */
  int32_t check_cycles;  /* 0 */
  int32_t reserved;
} yalps_options;

void yalps_default_options(yalps_options *opt);

/* Kernel path selection for the batch entry points (diagnostics / benchmarks). */
enum yalps_path {
  YALPS_PATH_AUTO = 0,
  YALPS_PATH_SMEM = 1, /* K1: one tableau per CTA resident in shared memory */
  YALPS_PATH_GMEM = 2, /* K2: tableau in HBM/L2, CTA per LP, pivot row/column staged in shared memory */
  YALPS_PATH_GRID = 3, /* K4: one LP across the whole grid (cooperative launch) */
  YALPS_PATH_CLUSTER = 5, /* KC: one LP per thread-block cluster, tableau distributed over the cluster's shared
                             memory; candidate pivot rows are published to an L2-resident scratch and the winner's row
                             is staged from there, DSMEM carries only the 16-byte selection records
                             (csrc/cluster_kernel.cuh) */
  YALPS_PATH_TMEM = 6, /* K1t: one LP per warp, tableau resident in tensor memory (tcgen05.ld/st as a lane-private
                          scratchpad; at most 65 x 65), csrc/tmem_kernel.cuh */
  YALPS_PATH_GRID_RESIDENT = 7, /* KG: one LP across the whole grid with the tableau resident in the SMs' shared memory
                                   (up to ~25 MB: 148 x 227 KB), one grid barrier per pivot; the automatic choice for the
                                   tableaus K4 used to take that fit (csrc/cluster_kernel.cuh, kGrid) */
  /* 4 is retired (a register-resident experiment that never beat K1) and rejected by yalps_set_tuning */
};

/* ---- context ------------------------------------------------------------ */
int yalps_create(int device, yalps_ctx **out);
void yalps_destroy(yalps_ctx *ctx);
const char *yalps_last_error(const yalps_ctx *ctx); /* ctx may be NULL: error of the last failed yalps_create */
int yalps_device_info(const yalps_ctx *ctx, int32_t *sm_count, int32_t *smem_per_block_optin, int32_t *cc_major,
                      int32_t *cc_minor);
/* Force a path / CTA width for subsequent batch calls (0 = auto). */
int yalps_set_tuning(yalps_ctx *ctx, int32_t path, int32_t threads_per_lp);
/* Row groups per CTA for the shared-memory / HBM paths: > 1 selects the row-split latency kernels
 * (csrc/simplex_split.cuh: threads_per_lp / row_groups column threads x row_groups), 0 = automatic. */
int yalps_set_row_groups(yalps_ctx *ctx, int32_t row_groups);
/* Experiment switches read from the environment (results never depend on them, only the launch configuration):
 * YALPS_CTAS_PER_SM=n caps the resident CTAs per SM of the k_simplex kernels; YALPS_NODE_SPLIT="w,r" sets column warps
 * and row groups of the one-CTA-per-node kernel of big sparse node waves; YALPS_KC_TMA=0|1|2 the pivot-row staging of the
 * cluster kernel; YALPS_KG_CTAS / YALPS_KG_THREADS / YALPS_NO_KG the grid-resident kernel; YALPS_GRID_CTAS the grid of K4;
 * YALPS_LARGE_ROW_PARTS the row split of yalps_multi_solve_large; YALPS_NO_REPLICA_SHARING the replica path sharing. */
/* Number of kernels launched by this ctx since creation (bench.py's gpu_launches). */
int64_t yalps_launch_count(const yalps_ctx *ctx);

/*
 * Roofline diagnostics (SURVEY 8d): algorithmic bytes of a pivot are 16*W*(1+R) + 8*(2(H-1)+2(W-1)) with R = the rows
 * the rank-1 update rewrites (|coef| > 1e-16, src/simplex.ts:31).  While a counter is set, every kernel ADDS the R
 * of each pivot to d_rows[per_lp ? LP index within the call : 0] (device memory, uint64, zeroed by the caller):
 * yalps_solve_batch_device and yalps_solve_replicas per LP or in total, branch-and-cut node waves in total only.
 * The tensor-memory kernel runs a counting instantiation while the counter is set, so set it for a measuring pass,
 * not for the timed one.  NULL switches the counter off.
 */
int yalps_set_row_counter(yalps_ctx *ctx, uint64_t *d_rows, int32_t per_lp);

/* Pinned host memory for callers that want zero-staging transfers. */
int yalps_host_alloc(yalps_ctx *ctx, uint64_t bytes, void **out);
int yalps_host_free(yalps_ctx *ctx, void *ptr);

/* ---- simplex(tableau, options), batched: replaces src/simplex.ts:144 ----- */
/*
 * n tableaus of identical shape height x width, contiguous in `matrices`
 * (n*height*width doubles, not modified).  Outputs (any may be NULL):
 *   status[n]            yalps_status
 *   value[n]             rounded objective M[0,0] (optimal) / entering column (unbounded) / NaN
 *   pivots[2n]           phase-1 and phase-2 pivot counts
 *   rhs_out[n*height]    column 0 of the final tableau
 *   pos_out/var_out[n*(width+height)]  final positionOfVariable / variableAtPosition
 *   matrices_out[n*height*width]       final tableau (the in-place result of the reference)
 * This is what solve() needs to build a Solution (src/YALPS.ts:8-50).
 */
int yalps_solve_batch(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                      const yalps_options *opt, int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                      int32_t *pos_out, int32_t *var_out, double *matrices_out);

/*
 * simplex(tableau, options) on tableaus that carry their own basis bookkeeping: pos_in / var_in
 * (int32[n*(width+height)], mutually inverse permutations) are the positionOfVariable / variableAtPosition
 * the tableaus arrive with.  This is the drop-in for the SECOND caller of the seam, src/branchAndCut.ts:127,
 * where simplex runs on applyCuts' output whose permutation is the root's final one (:46-52), not the identity.
 * Every output may alias the corresponding input (matrices_out == matrices etc.) for the reference's in-place
 * contract.  pos_in == var_in == NULL is yalps_solve_batch.
 */
int yalps_solve_batch_basis(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                            const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                            double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                            double *matrices_out);
int yalps_solve_ragged_basis(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                             const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                             const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                             int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                             double *matrices_out);

/*
 * n replicas of ONE base tableau that differ only in column 0 (BASELINE config 3: perturbed right-hand sides):
 * the caller ships base (height*width doubles) once and rhs (n*height doubles, replica-major; rhs[i*height + 0] is
 * replica i's M[0,0]) -- 8*height bytes per LP over PCIe instead of 8*height*width.  The working copies are
 * assembled on the device.  Outputs as yalps_solve_batch.
 */
int yalps_solve_replicas(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *base,
                         const double *rhs, const yalps_options *opt, int32_t *status, double *value, int64_t *pivots,
                         double *rhs_out, int32_t *pos_out, int32_t *var_out);

/* Replica path sharing (default on).  The replicas of yalps_solve_replicas differ only in column 0, and a pivot choice
 * depends on a replica's own data only through that column (most negative RHS in phase 1, ratio test in phase 2): the
 * base tableau is solved once with a recorded trace, every replica follows it carrying just its RHS column (one warp,
 * H doubles) while it makes the same choices, and continues alone -- from the leader's tableau of that step with its own
 * column 0, same phase, same pivot counters -- the moment it would choose differently.  Every output bit is that of
 * solving the replica on its own (src/simplex.ts:99-142); the coefficient updates of the shared stretch are simply not
 * repeated.  Not used with checkCycles or a forced kernel path.  yalps_replica_forks: how many replicas of the last
 * call left the shared path (-1: sharing was not used). */
int yalps_set_replica_sharing(yalps_ctx *ctx, int32_t on);
int64_t yalps_replica_forks(const yalps_ctx *ctx);


/* Ragged batch: LP i is heights[i] x widths[i] at matrices[mat_offsets[i]];
 * rhs_out is packed by cumulative heights, pos_out/var_out by cumulative (width+height). */
int yalps_solve_ragged(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                       const int64_t *mat_offsets, const double *matrices, const yalps_options *opt, int32_t *status,
                       double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                       double *matrices_out);

/* Same as yalps_solve_batch with every buffer already in device memory and the
 * work enqueued on `stream` (a cudaStream_t, NULL = default stream); returns
 * without synchronising.  d_work (n*height*width doubles) is only required when
 * the HBM-resident path is taken and may alias d_matrices for an in-place solve.  When d_work is given the
 * first call for a (buffer, shape) samples the density of the first tableau to choose the kernel path, which
 * synchronises `stream` once. */
int yalps_solve_batch_device(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                             double *d_work, const yalps_options *opt, int32_t *d_status, double *d_value,
                             int64_t *d_pivots, double *d_rhs_out, int32_t *d_pos_out, int32_t *d_var_out,
                             double *d_matrices_out, void *stream);

/* Synthetic dense LP batch of SURVEY 8(d) (configs 2 and 5) generated on the device:
 * LP `first+i` -> (m+1) x (nvars+1) tableau, integer-hash PRNG of tests/helpers/util.ts:20-41. */
int yalps_generate_synthetic_device(yalps_ctx *ctx, int64_t first, int64_t n, int32_t m, int32_t nvars,
                                    int32_t neg_rows, uint32_t salt, double *d_out, void *stream);

/* Config 3: n replicas of one base tableau whose RHS column is perturbed per replica,
 * rhs_i[r] = base[r,0] * (1 + eps*(2U-1)), U drawn per `group[r]` (rows of one constraint key share a
 * draw; group < 0 = unperturbed) from newRand(prospectorHash((first+i) ^ salt)). */
int yalps_generate_replicas_device(yalps_ctx *ctx, int64_t first, int64_t n, int32_t height, int32_t width,
                                   const double *base_host, const int32_t *group_host, int32_t ngroups, double eps,
                                   uint32_t salt, double *d_out, void *stream);

/* ---- branch and cut: replaces src/branchAndCut.ts ------------------------ */
/*
 * Root session: uploads the root-optimal tableau once (applyCuts needs the full
 * matrix, src/branchAndCut.ts:28,38-42).  max_extra_rows = 2*|integers| (:108).
 */
int yalps_bnb_set_root(yalps_ctx *ctx, int32_t height, int32_t width, const double *matrix, const int32_t *pos,
                       const int32_t *var, int32_t max_extra_rows);
/*
 * Node wave: node j carries cuts [cut_offsets[j], cut_offsets[j+1]) as
 * (sign, variable, value) triples (Cut, src/branchAndCut.ts:18).  The device
 * assembles root + cut rows (applyCuts) and runs simplex.  Outputs are strided
 * by the wave's tallest node: stride_h = height + max_j ncuts_j:
 *   rhs_out[n*stride_h], pos_out/var_out[n*(width+stride_h)], matrices_out[n*stride_h*width] (optional).
 */
int yalps_bnb_solve_nodes(yalps_ctx *ctx, int64_t n, const int32_t *cut_offsets, const double *cut_sign,
                          const int32_t *cut_var, const double *cut_value, const yalps_options *opt, int32_t *status,
                          double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                          double *matrices_out);
/*
 * The whole branchAndCut(tabmod, initResult, options) of src/branchAndCut.ts:89-176
 * on the current root: best-first search with the reference's heap order, node LPs
 * evaluated in speculative waves on the device and consumed in the reference's
 * pop order.  ints = TableauModel.integers (variable ids), sign = TableauModel.sign.
 * Outputs describe the best tableau (src/branchAndCut.ts:175): out_height rows,
 * rhs_out[out_height], pos_out/var_out[width+out_height] (buffers sized for
 * height+max_extra_rows).  stats[8] (optional): nodes evaluated by the replay, node pivots,
 * max cuts, max heap, waves, nodes solved on device (incl. unused speculation),
 * microseconds spent in device waves, microseconds total.
 * When the node tableaus fit one CTA's shared memory the whole search runs inside one
 * persistent kernel (csrc/bnb_kernel.cuh: scheduler CTA + worker CTAs that expand
 * optimal fractional nodes speculatively); the result is the same search node for node.
 * Tuning / diagnostics through the environment, read per search: YALPS_BNB_SPEC
 * (generations of speculation, default 2, 0 = none), YALPS_BNB_WORKERS (worker CTAs,
 * default one per SM beside the scheduler), YALPS_BNB_DEBUG=1 (scheduler and worker stage
 * cycles and pool usage on stderr; for the wave driver: host microseconds per wave spent
 * enqueueing, waiting for the device, copying out and replaying).
 */
int yalps_branch_and_cut(yalps_ctx *ctx, const int32_t *ints, int32_t nints, double sign, double init_result,
                         const yalps_options *opt, int32_t *status, double *result, int32_t *out_height,
                         double *rhs_out, int32_t *pos_out, int32_t *var_out, int64_t *stats);
/* Where the search loop runs: 0 (default) = inside one persistent kernel (csrc/bnb_kernel.cuh: a scheduler CTA replays
 * the reference's loop, the other CTAs evaluate node LPs) when the node tableaus fit one CTA's shared memory, otherwise
 * -- and whenever a device pool overflows -- the host wave driver; 1 = host wave driver only; 2 = device kernel only
 * (YALPS_ERR_TOO_LARGE when the search does not fit).  Both produce the reference's search node for node. */
int yalps_bnb_set_mode(yalps_ctx *ctx, int32_t mode);
/* Upper bound of the speculative look-ahead per wave (default 256; the driver adapts the actual width, starting at
 * 16, to how much of each wave the replay consumes). */
int yalps_bnb_set_wave(yalps_ctx *ctx, int32_t wave);

/*
 * One call for solve()'s numeric part (src/YALPS.ts:77-91): root simplex on the
 * given initial tableau and, if it is optimal and nints > 0, branch and cut.
 * Buffers sized for height + 2*nints rows.  root_status/root_value/root_pivots[2]
 * report the root LP (optional).
 */
int yalps_solve(yalps_ctx *ctx, int32_t height, int32_t width, const double *matrix, const int32_t *ints,
                int32_t nints, double sign, const yalps_options *opt, int32_t *status, double *result,
                int32_t *out_height, double *rhs_out, int32_t *pos_out, int32_t *var_out, int32_t *root_status,
                double *root_value, int64_t *root_pivots, int64_t *stats);

/*
 * yalps_solve with the initial tableau given as (cell, value) pairs over a zero matrix: exactly the stores tableauModel
 * makes into its zero-filled Float64Array (src/tableau.ts:88-134: objective row, constraint rows, RHS cells, binary
 * rows), cell = row*width + col, applied in order (a later pair for the same cell wins, :100-117).  Model tableaus
 * are very sparse (Vendor Selection: 1722x1641 = 22.6 MB with < 0.3 % non-zeros), so the host neither fills nor ships
 * the zeros: the pairs cross PCIe, the device zeroes the matrix and scatters them.  Results are bit-identical to
 * yalps_solve on the dense image (negative zeros included).  Tableaus under 768 KB are densified on the host and
 * take yalps_solve's zero-copy path.
 */
int yalps_solve_sparse(yalps_ctx *ctx, int32_t height, int32_t width, int64_t nnz, const int32_t *cell, const double *val,
                       const int32_t *ints, int32_t nints, double sign, const yalps_options *opt, int32_t *status,
                       double *result, int32_t *out_height, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                       int32_t *root_status, double *root_value, int64_t *root_pivots, int64_t *stats);

/* ---- dual values: shadow prices and reduced costs ------------------------------------------------------------
 * Each *_duals entry point takes the arguments of its sibling plus a trailing reduced_out (NULL: the sibling exactly).
 * reduced_out holds one double per variable id and is packed like pos_out (width + height per LP):
 *     reduced_out[v] = M[0, pos[v]]   if 1 <= pos[v] < width  (v non-basic: its column's row-0 cell, bits as they are)
 *     reduced_out[v] = +0.0           otherwise                (basic variables, and ids 0 and width)
 * where M, pos are the final tableau and positionOfVariable the call reports.  Ids 1..width-1 are the structural
 * columns, id width + r is the slack of row r.  It is written for every status (it is row 0 re-indexed) and costs
 * 8*(width+height) bytes of device-to-host copy per LP.  With the reference's conventions (entering column = positive
 * row-0 cell, result = -sign * M[0,0]) these are the partial derivatives of result:
 *     d result / d x_j   =  sign * reduced_out[j]           (structural variable j)
 *     d result / d rhs_r = -sign * reduced_out[width + r]   (right-hand side of row r)
 * e.g. max 3x s.t. x <= 4 ends with row 0 = [-12, -3]: sign = 1, the shadow price of the row is 3.
 * How far each of these values holds is what the *_ranging entry points below report ("sensitivity ranging").
 */
/* yalps_solve_batch_basis + reduced_out (pos_in = var_in = NULL: yalps_solve_batch) */
int yalps_solve_batch_duals(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                            const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                            double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                            double *matrices_out, double *reduced_out);
/* yalps_solve_ragged_basis + reduced_out (packed by cumulative width + height, like pos_out) */
int yalps_solve_ragged_duals(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                             const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                             const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                             int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                             double *matrices_out, double *reduced_out);
int yalps_solve_replicas_duals(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *base,
                               const double *rhs, const yalps_options *opt, int32_t *status, double *value,
                               int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                               double *reduced_out);
/* d_reduced_out is device memory, like every other buffer of yalps_solve_batch_device */
int yalps_solve_batch_device_duals(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                                   double *d_work, const yalps_options *opt, int32_t *d_status, double *d_value,
                                   int64_t *d_pivots, double *d_rhs_out, int32_t *d_pos_out, int32_t *d_var_out,
                                   double *d_matrices_out, void *stream, double *d_reduced_out);
/* The root LP of yalps_solve_sparse (no branch and cut): status, value (as yalps_solve_batch), pivots[2], rhs_out[height],
 * pos_out/var_out[width+height], reduced_out[width+height]. */
int yalps_solve_sparse_duals(yalps_ctx *ctx, int32_t height, int32_t width, int64_t nnz, const int32_t *cell,
                             const double *val, const yalps_options *opt, int32_t *status, double *value, int64_t *pivots,
                             double *rhs_out, int32_t *pos_out, int32_t *var_out, double *reduced_out);

/* ---- sensitivity ranging: how far the optimal basis holds ---------------------------------------------------
 * A shadow price or reduced cost is valid while the optimal basis stays the same.  Ranging reports, per variable id
 * (packed like pos_out, width + height doubles per LP), the interval [range_lo, range_hi] of shifts over which it does:
 *   structural j (1 <= j < width):  shifts of the initial objective cell M0[0,j] (= sign * c_j) that keep the final
 *                                   basis optimal;
 *   slack of row k (id width + k):  shifts of row k's initial right-hand side that keep it primal feasible.
 * With b+_r = max(M[r,0], +0), g_c = min(M[0,c], +0) and a cell counting when |cell| > opt->precision:
 *   structural j non-basic at column c:  (-inf, -g_c)
 *   structural j basic at row r:         (max g_c / M[r,c] over counting M[r,c] > 0, min over M[r,c] < 0), c >= 1
 *   slack of row k:                      (max -b+_r / d[r] over counting d[r] > 0, min over d[r] < 0), r >= 1
 * where d is dir(width + k), or dir(width + k) - dir(width + pairs[k]) when the row has a pair, and dir(u) is the final
 * tableau's column pos[u] when u is non-basic, else the unit vector of u's basic row.  A pair is the other row of the
 * same constraint (the lower row of a key whose upper row is k, or the other way round): its right-hand side moves by
 * -t when row k's moves by +t, which is how a key with two finite bounds (a range or an equality) shifts as one;
 * ranging its rows one by one would give the wrong interval.  pairs is packed like rhs_out: pairs[0] = -1, every
 * other entry -1 (none) or a row 1..height-1 whose entry points back (YALPS_ERR_ARGUMENT otherwise).
 * An empty max is -inf, an empty min +inf, zeros are +0.0 and lo <= 0 <= hi.  Ids 0 and width, and every id of an LP
 * that is not optimal, are NaN.  Every value is one IEEE division followed by a max or min: bit-exact, whatever the
 * kernel path.  e.g. max 3x s.t. x <= 4: the row ranges over [-4, inf), the objective cell of x over [-3, inf).
 * k_ranging computes the ranges on the device from the final tableaus after the solve; the tableaus are copied to the
 * host only when matrices_out is given, and the ranges cost 16*(width+height) bytes of device-to-host copy per LP.
 *
 * yalps_solve_{batch,ragged}_ranging: the *_duals sibling's arguments plus pairs (NULL: no pairs), range_lo and
 * range_hi (both NULL: the *_duals call exactly; one without the other is YALPS_ERR_ARGUMENT).
 */
int yalps_solve_batch_ranging(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                              const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                              double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                              double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                              double *range_hi);
int yalps_solve_ragged_ranging(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                               const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                               const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                               int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                               double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                               double *range_hi);
/* yalps_solve_sparse_duals + pairs, range_lo, range_hi */
int yalps_solve_sparse_ranging(yalps_ctx *ctx, int32_t height, int32_t width, int64_t nnz, const int32_t *cell,
                               const double *val, const yalps_options *opt, int32_t *status, double *value,
                               int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out, double *reduced_out,
                               const int32_t *pairs, double *range_lo, double *range_hi);
/* Ranges of n final tableaus already in device memory (e.g. d_matrices_out of yalps_solve_batch_device_duals), with
 * their positionOfVariable d_pos and status d_status (NULL: every LP is optimal); d_pairs NULL: no pairs.  Every pointer
 * is device memory; the kernel is enqueued on `stream`.  d_pairs is not validated here. */
int yalps_ranging_device(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                         const int32_t *d_pos, const int32_t *d_status, const int32_t *d_pairs, double precision,
                         double *d_range_lo, double *d_range_hi, void *stream);

/* ---- certificates: why an LP is infeasible or unbounded ----------------------------------------------------
 * One double per variable id (packed like pos_out, width + height per LP), read from the final tableau M, its
 * positionOfVariable pos, and the status and value the call reports:
 *   infeasible (status 1), a Farkas certificate.  r is the row phase 1 chose: the lowest r in 1..height-1 whose
 *     M[r,0] is the minimum over the rows with M[r,0] < -opt->precision (NaN never qualifies, -inf does).  Phase 1
 *     stops there without a pivot, so the final tableau is the tableau of that choice.
 *       cert[0] = M[r,0], cert[width] = +0.0, and for every other id v:
 *       cert[v] = M[r, pos[v]] if 1 <= pos[v] < width (bits as they are), 1.0 if pos[v] == width + r, +0.0 otherwise.
 *     cert[width + k] is the multiplier y_k >= -precision of original row k (a_k.x <= b_k); the structural entries
 *     equal sum_k y_k a_kj >= -precision and cert[0] = sum_k y_k b_k < 0, so no x >= 0 satisfies every row.
 *   unbounded (status 2), a ray.  c = (int)value is the entering column.
 *       cert[0] = M[0,c] (d result / dt = sign * cert[0], the convention of reduced_out), cert[width] = +0.0, and
 *       cert[v] = 1.0 if pos[v] == c, -M[pos[v] - width, c] if width < pos[v] < width + height (the sign bit
 *       flipped), +0.0 otherwise.
 *     Moving every variable by t * cert[v] keeps every row feasible and improves the objective without bound.
 *   Every other status, an infeasible LP with no qualifying row and an unbounded LP with c outside 1..width-1: NaN.
 * The values are raw tableau cells (nothing below precision is cleaned), bit-exact whatever the kernel path.
 * k_certificate computes them on the device from the final tableaus after the solve, like k_ranging; they cost
 * 8*(width+height) bytes of device-to-host copy per LP.  e.g. max p with c: x <= -1 and p = x: infeasible,
 * cert = [-1, 1, +0, 1].
 *
 * Each *_certificate entry takes its *_ranging sibling's arguments plus a trailing cert_out (NULL: the sibling
 * exactly).
 */
int yalps_solve_batch_certificate(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *matrices,
                                  const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt,
                                  int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                                  int32_t *var_out, double *matrices_out, double *reduced_out, const int32_t *pairs,
                                  double *range_lo, double *range_hi, double *cert_out);
int yalps_solve_ragged_certificate(yalps_ctx *ctx, int64_t n, const int32_t *heights, const int32_t *widths,
                                   const int64_t *mat_offsets, const double *matrices, const int32_t *pos_in,
                                   const int32_t *var_in, const yalps_options *opt, int32_t *status, double *value,
                                   int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                                   double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                                   double *range_hi, double *cert_out);
int yalps_solve_sparse_certificate(yalps_ctx *ctx, int32_t height, int32_t width, int64_t nnz, const int32_t *cell,
                                   const double *val, const yalps_options *opt, int32_t *status, double *value,
                                   int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                                   double *reduced_out, const int32_t *pairs, double *range_lo, double *range_hi,
                                   double *cert_out);
/* Certificates of n final tableaus already in device memory, with their positionOfVariable d_pos, status d_status and
 * value d_value as a solve reported them.  Every pointer is device memory; the kernel is enqueued on `stream`. */
int yalps_certificate_device(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *d_matrices,
                             const int32_t *d_pos, const int32_t *d_status, const double *d_value, double precision,
                             double *d_cert_out, void *stream);

/* ---- irreducible infeasible subsets: which constraints conflict ------------------------------------------------
 * For a row set S of 1..height-1, T_S is the tableau with every row outside S set to +0.0 (column 0 included); row 0,
 * the objective, always stays.  With precision >= 0 the simplex never picks a zero row in phase 1 (its RHS is not
 * < -precision), never in the ratio test (its cell is not > precision) and never changes it in a pivot (its cells are
 * not above 1e-16): status, value, pivot counts and every other row are those of the model without the removed rows,
 * bit for bit.  Variables keep their implicit x >= 0 in every subset.
 * supp(cert) of an infeasible LP is the set of rows k with cert[width + k] > +0.0 (the raw value: NaN and both zeros
 * do not count), the rows its Farkas certificate combines.  Words of a row mask: words = (height + 31) / 32, bit r of
 * word r / 32 is row r.
 *
 * n LPs = base restricted to row subsets (keep: n*words uint32, bit r = row r; row 0 always kept, bit 0 ignored, bits
 * >= height must be clear), expanded on the device; outputs as yalps_solve_batch plus cert_out[n*(width+height)] and
 * support_out[n*words] (zero words unless infeasible), each may be NULL.  A negative or NaN precision is
 * YALPS_ERR_ARGUMENT. */
int yalps_solve_row_subsets(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *base,
                            const uint32_t *keep, const yalps_options *opt, int32_t *status, double *value,
                            int64_t *pivots, double *cert_out, uint32_t *support_out);
/* An IIS: a row set S whose T_S the solver finds infeasible while every T_{S \ {r}} it finds optimal or unbounded, by
 * deletion rounds on the GPU.  Round 0 solves the whole tableau; if it is not infeasible that status is returned with
 * *count = 0.  Otherwise S = supp(cert), and each round solves T_S and every T_{S \ {u}}, u in S, as one batch: when
 * T_S is not infeasible S falls back to the last set solved infeasible; when no T_{S \ {u}} is infeasible S is the
 * result; else S becomes the support of the infeasible T_{S \ {u}} with the smallest support (lowest u on ties).
 * S strictly shrinks, so there are at most height rounds.  opt->max_pivots and check_cycles apply to every subset LP;
 * opt->timeout_ms (+inf: none) is checked between rounds and returns the last set solved infeasible.
 * status = the model's own status, rows_out[height] ascending, *count rows; stats[5] (may be NULL): rounds (round 0
 * included), LPs solved, their pivots (both phases), undecided rows (u whose T_{S \ {u}} ended `cycled` in the final
 * round), timed out (0/1).  S is irreducible when the last two are 0.  A negative or NaN precision is
 * YALPS_ERR_ARGUMENT. */
int yalps_iis(yalps_ctx *ctx, int32_t height, int32_t width, const double *matrix, const yalps_options *opt,
              int32_t *status, int32_t *rows_out, int32_t *count, int64_t *stats);
/* yalps_iis with the tableau given as (cell, value) stores into a zero matrix, as yalps_solve_sparse */
int yalps_iis_sparse(yalps_ctx *ctx, int32_t height, int32_t width, int64_t nnz, const int32_t *cell,
                     const double *val, const yalps_options *opt, int32_t *status, int32_t *rows_out,
                     int32_t *count, int64_t *stats);

/* ---- warm starts: variants of one LP re-optimised from its final basis ------------------------------------------
 * A variant of the base LP keeps its constraint coefficients and has its own column 0 b' (rhs + i*height: height
 * values, b'[0] is the new M0[0,0]) and/or its own row 0 c' (obj + i*width: width values, c'[0] ignored); rhs or obj
 * NULL: that part is the base's.  Its start tableau T keeps the base's final basis (pos / var) and is derived on the
 * device from the base's initial tableau M0 and final tableau F (any status) by:
 *   dir(v): for a non-basic id (1 <= pos[v] < width) the column F[:, pos[v]], row 0 included; for a basic id the unit
 *     vector of row pos[v] - width; for id width + 0 the unit vector of row 0 (the direction ranging uses).
 *   1. column pass: T = F.  delta_k = b'[k] - M0[k,0] (rounded once; skipped when == 0.0).  For every row r and every
 *      changed k in ascending order: T[r,0] = T[r,0] + delta_k * dir(width+k)[r], product and sum rounded apart (no
 *      FMA).
 *   2. row pass, on the result of 1.  delta_j = c'[j] - M0[0,j], j = 1..width-1 (skipped when == 0.0).  For every
 *      column c and every changed j in ascending order: x_j non-basic: T[0,c] = T[0,c] + delta_j when c == pos[j];
 *      x_j basic at row q = pos[j] - width: T[0,c] = T[0,c] - delta_j * T[q,c].
 * With no change T is F bit for bit.  In exact arithmetic column 0 becomes B^-1 b' and row 0 the reduced costs and
 * objective value of the same basis under c' (yalps_b200/warm.py has the derivation).  Each variant is then the
 * reference's loop on T from that basis: after RHS changes phase 1 is the dual simplex from a dual-feasible basis, after
 * objective changes phase 2 continues from the old vertex.
 * Caveat: the results are bit-exact against the reference's loop run on T, NOT against a cold solve of the changed
 * model: the pivot path differs.  Statuses agree and optimal values agree within the precision, but with alternative
 * optima the reported vertex can differ.
 *
 * base: M0 (height*width).  final / final_pos / final_var: F and its basis (all three or none; the basis must be a pair
 * of inverse permutations).  With none the library solves the base first with opt, keeps its final tableau on the
 * device (it never crosses PCIe) and reports its status, value and pivots[2] in base_status / base_value /
 * base_pivots (each may be NULL; untouched when final is given).  Per variant the outputs of
 * yalps_solve_batch_certificate: status, value, pivots, rhs_out, pos_out, var_out, matrices_out (the final tableaus),
 * reduced_out, pairs (n*height, packed like rhs_out) with range_lo / range_hi, and cert_out, each may be NULL.  n < 0,
 * a bad shape, a negative or NaN precision, and rhs and obj both NULL with n > 0 are YALPS_ERR_ARGUMENT. */
int yalps_solve_warm(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, const double *base,
                     const double *final_m, const int32_t *final_pos, const int32_t *final_var, const double *rhs,
                     const double *obj, const yalps_options *opt, int32_t *base_status, double *base_value,
                     int64_t *base_pivots, int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                     int32_t *pos_out, int32_t *var_out, double *matrices_out, double *reduced_out,
                     const int32_t *pairs, double *range_lo, double *range_hi, double *cert_out);
/* yalps_solve_warm with the base's initial tableau given as (cell, value) stores into a zero matrix, as
 * yalps_solve_sparse: it is built on the device and never exists densely on the host */
int yalps_solve_warm_sparse(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, int64_t nnz,
                            const int32_t *cell, const double *val, const double *final_m, const int32_t *final_pos,
                            const int32_t *final_var, const double *rhs, const double *obj, const yalps_options *opt,
                            int32_t *base_status, double *base_value, int64_t *base_pivots, int32_t *status,
                            double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                            double *matrices_out, double *reduced_out, const int32_t *pairs, double *range_lo,
                            double *range_hi, double *cert_out);
/* Warm starts that also add constraints and variables.  Every variant adds K = add_rows rows and M = add_cols
 * columns to the base (H = height, W = width): rows_in + i*K*(W+M) holds its K rows in initial-tableau form over the
 * W+M columns (cell 0 the RHS, then the W-1 base structurals, then the M added ones; an upper row a.x <= max, a lower
 * row -a.x <= -min), cols_in + i*M*H its M columns in initial-tableau form over the H base rows (cell 0 sign * cost,
 * then the coefficient in each base row).  The start tableau has (H+K) x (W+M) cells; in base ids and positions:
 *   1. column pass as above (step 1).
 *   2. added columns: T[r, W+j] = sum over k ascending of g_j[k] * dir(W+k)[r], from +0.0, skipping g_j[k] == 0.0,
 *      product and sum rounded apart (dir read from F, row 0 included; dir(W+0) is the unit vector of row 0).
 *   3. row pass as above (step 2), over all W+M columns.
 *   4. added rows, on the result of 3: row i starts as (a[0], +0.0, ...); for every structural v with a[v] != 0.0,
 *      base ids then added ids ascending: v non-basic: t[pos(v)] += a[v]; v basic at row q: t[c] -= a[v] * T[q,c] for
 *      every c, column 0 included.  Added variables are non-basic at column W+j.
 *   5. the basis, relabelled: base structural v < W keeps v; added structural j is W+j, non-basic at column W+j; base
 *      slack W+k becomes W+M+k; added row i's slack is W+M+H+i, basic at row H+i.
 * In exact arithmetic an added column is B^-1 times the column with its reduced cost under the current costs, and an
 * added row is the constraint with the basic variables substituted out (for a one-variable cut it equals the
 * applyCuts row of branch and cut); it starts primal infeasible and dual feasible, so phase 1 runs the dual simplex.
 * With K = M = 0 this is yalps_solve_warm bit for bit.  Outputs are per LP at the extended shape, packed as for a
 * batch of (H+K) x (W+M) LPs; pairs covers the H+K rows.  rhs and obj keep the base's sizes (H and W values) and may
 * both be NULL when K or M is positive.  K < 0, M < 0, rows_in NULL with K > 0 and cols_in NULL with M > 0 are
 * YALPS_ERR_ARGUMENT; an extended shape of 2^31 cells or more is YALPS_ERR_TOO_LARGE. */
int yalps_solve_warm_extend(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, int32_t add_rows,
                            int32_t add_cols, const double *base, const double *final_m, const int32_t *final_pos,
                            const int32_t *final_var, const double *rhs, const double *obj, const double *rows_in,
                            const double *cols_in, const yalps_options *opt, int32_t *base_status, double *base_value,
                            int64_t *base_pivots, int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                            int32_t *pos_out, int32_t *var_out, double *matrices_out, double *reduced_out,
                            const int32_t *pairs, double *range_lo, double *range_hi, double *cert_out);
/* yalps_solve_warm_extend with the base's initial tableau given as (cell, value) stores, as yalps_solve_warm_sparse */
int yalps_solve_warm_extend_sparse(yalps_ctx *ctx, int64_t n, int32_t height, int32_t width, int32_t add_rows,
                                   int32_t add_cols, int64_t nnz, const int32_t *cell, const double *val,
                                   const double *final_m, const int32_t *final_pos, const int32_t *final_var,
                                   const double *rhs, const double *obj, const double *rows_in, const double *cols_in,
                                   const yalps_options *opt, int32_t *base_status, double *base_value,
                                   int64_t *base_pivots, int32_t *status, double *value, int64_t *pivots,
                                   double *rhs_out, int32_t *pos_out, int32_t *var_out, double *matrices_out,
                                   double *reduced_out, const int32_t *pairs, double *range_lo, double *range_hi,
                                   double *cert_out);

/* ---- one process, several GPUs (SURVEY 8b/8e) ------------------------------------------------------------
 * The reference is single-process and synchronous (src/YALPS.ts:73-92); a Node addon cannot use torchrun.  A
 * yalps_multi owns one ctx (plus worker ctxs for concurrent branch-and-cut searches) per entry of `devices` and one
 * host thread per ctx.  Independent LPs shard as contiguous ranges, LP i -> rank floor(i*ndev/n), with no collective
 * on the data path; results land in the caller's arrays exactly as from the single-GPU entry points.  An entry may
 * repeat a device (several logical ranks on one GPU: how a 1-GPU box exercises the multi-rank code).
 */
typedef struct yalps_multi yalps_multi;
int yalps_create_multi(const int32_t *devices, int32_t ndev, yalps_multi **out);
void yalps_destroy_multi(yalps_multi *m);
const char *yalps_multi_last_error(const yalps_multi *m); /* m may be NULL: error of the last failed create */
int32_t yalps_multi_size(const yalps_multi *m);
yalps_ctx *yalps_multi_ctx(yalps_multi *m, int32_t rank); /* rank's ctx (tuning, launch counts); owned by m */
int64_t yalps_multi_launch_count(const yalps_multi *m);   /* kernels launched by all ctxs of m */
int yalps_multi_solve_batch(yalps_multi *m, int64_t n, int32_t height, int32_t width, const double *matrices,
                            const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt, int32_t *status,
                            double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                            double *matrices_out);
int yalps_multi_solve_ragged(yalps_multi *m, int64_t n, const int32_t *heights, const int32_t *widths,
                             const int64_t *mat_offsets, const double *matrices, const yalps_options *opt,
                             int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                             int32_t *var_out, double *matrices_out);
int yalps_multi_solve_replicas(yalps_multi *m, int64_t n, int32_t height, int32_t width, const double *base,
                               const double *rhs, const yalps_options *opt, int32_t *status, double *value,
                               int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out);
/* the three above + reduced_out (see "dual values"), sharded like pos_out */
int yalps_multi_solve_batch_duals(yalps_multi *m, int64_t n, int32_t height, int32_t width, const double *matrices,
                                  const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt,
                                  int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                                  int32_t *var_out, double *matrices_out, double *reduced_out);
int yalps_multi_solve_ragged_duals(yalps_multi *m, int64_t n, const int32_t *heights, const int32_t *widths,
                                   const int64_t *mat_offsets, const double *matrices, const yalps_options *opt,
                                   int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                                   int32_t *var_out, double *matrices_out, double *reduced_out);
int yalps_multi_solve_replicas_duals(yalps_multi *m, int64_t n, int32_t height, int32_t width, const double *base,
                                     const double *rhs, const yalps_options *opt, int32_t *status, double *value,
                                     int64_t *pivots, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                                     double *reduced_out);
/* yalps_solve_warm with the variants sharded as contiguous ranges; every rank solves (or uploads) the base on its own
 * GPU, rank 0 reports it in base_status / base_value / base_pivots */
int yalps_multi_solve_warm(yalps_multi *m, int64_t n, int32_t height, int32_t width, const double *base,
                           const double *final_m, const int32_t *final_pos, const int32_t *final_var, const double *rhs,
                           const double *obj, const yalps_options *opt, int32_t *base_status, double *base_value,
                           int64_t *base_pivots, int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                           int32_t *pos_out, int32_t *var_out, double *matrices_out, double *reduced_out,
                           const int32_t *pairs, double *range_lo, double *range_hi, double *cert_out);
/* yalps_solve_warm_extend with the variants sharded as yalps_multi_solve_warm shards them */
int yalps_multi_solve_warm_extend(yalps_multi *m, int64_t n, int32_t height, int32_t width, int32_t add_rows,
                                  int32_t add_cols, const double *base, const double *final_m,
                                  const int32_t *final_pos, const int32_t *final_var, const double *rhs,
                                  const double *obj, const double *rows_in, const double *cols_in,
                                  const yalps_options *opt, int32_t *base_status, double *base_value,
                                  int64_t *base_pivots, int32_t *status, double *value, int64_t *pivots,
                                  double *rhs_out, int32_t *pos_out, int32_t *var_out, double *matrices_out,
                                  double *reduced_out, const int32_t *pairs, double *range_lo, double *range_hi,
                                  double *cert_out);
/* the batch and ragged *_duals entries + pairs, range_lo, range_hi (see "sensitivity ranging"), sharded like rhs_out
 * and pos_out */
int yalps_multi_solve_batch_ranging(yalps_multi *m, int64_t n, int32_t height, int32_t width, const double *matrices,
                                    const int32_t *pos_in, const int32_t *var_in, const yalps_options *opt,
                                    int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                                    int32_t *var_out, double *matrices_out, double *reduced_out, const int32_t *pairs,
                                    double *range_lo, double *range_hi);
int yalps_multi_solve_ragged_ranging(yalps_multi *m, int64_t n, const int32_t *heights, const int32_t *widths,
                                     const int64_t *mat_offsets, const double *matrices, const yalps_options *opt,
                                     int32_t *status, double *value, int64_t *pivots, double *rhs_out, int32_t *pos_out,
                                     int32_t *var_out, double *matrices_out, double *reduced_out, const int32_t *pairs,
                                     double *range_lo, double *range_hi);
/* the two above + cert_out (see "certificates"), sharded like pos_out */
int yalps_multi_solve_batch_certificate(yalps_multi *m, int64_t n, int32_t height, int32_t width,
                                        const double *matrices, const int32_t *pos_in, const int32_t *var_in,
                                        const yalps_options *opt, int32_t *status, double *value, int64_t *pivots,
                                        double *rhs_out, int32_t *pos_out, int32_t *var_out, double *matrices_out,
                                        double *reduced_out, const int32_t *pairs, double *range_lo, double *range_hi,
                                        double *cert_out);
int yalps_multi_solve_ragged_certificate(yalps_multi *m, int64_t n, const int32_t *heights, const int32_t *widths,
                                         const int64_t *mat_offsets, const double *matrices, const yalps_options *opt,
                                         int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                                         int32_t *pos_out, int32_t *var_out, double *matrices_out, double *reduced_out,
                                         const int32_t *pairs, double *range_lo, double *range_hi, double *cert_out);
/*
 * incumbent_allreduce (SURVEY 8b, north_star): min-allreduce of one fp64 per rank -- the incumbent objective of a
 * branch-and-bound search, lower is better internally (src/branchAndCut.ts:124,130).  local[ndev] in, agreed[ndev]
 * out (all equal).  Ranks that share a GPU are reduced by one kernel; the distinct GPUs go through
 * ncclAllReduce(ncclMin) on communicators from ncclCommInitAll (libnccl.so.2 is opened on first use; without it the
 * call fails with YALPS_ERR_CUDA -- there is no host-side substitute).
 */
int yalps_incumbent_allreduce(yalps_multi *m, const double *local, double *agreed);
/*
 * solve()'s numeric part (yalps_solve) with the branch-and-bound frontier sharded over the ranks (north_star,
 * BASELINE config 4): root LP on rank 0, final root tableau replicated on every rank, the nodes of each speculative
 * wave dealt over the ranks as contiguous ranges when a wave is worth splitting (nodes too big for one SM's shared
 * memory, or many small ones), the incumbent min-allreduced every `allreduce_every` waves; the replay stays the
 * reference's sequential loop, so nodes, pivots and the result are those of yalps_solve.  stats[8] as
 * yalps_branch_and_cut, plus stats[8] = waves that were sharded, stats[9] = allreduces (stats has 10 entries).
 */
int yalps_multi_solve(yalps_multi *m, int32_t height, int32_t width, const double *matrix, const int32_t *ints,
                      int32_t nints, double sign, const yalps_options *opt, int32_t allreduce_every, int32_t *status,
                      double *result, int32_t *out_height, double *rhs_out, int32_t *pos_out, int32_t *var_out,
                      int32_t *root_status, double *root_value, int64_t *root_pivots, int64_t *stats);
/*
 * solveMany(models, options): n_models tableaus (ragged, as yalps_solve_ragged) with their integer-variable lists
 * ints[ints_offsets[i] .. ints_offsets[i+1]) and signs[i].  All root LPs run as one ragged batch sharded over the
 * ranks; the models whose root is optimal and fractional then run branch and cut, MANY SEARCHES IN PARALLEL (each
 * search is a chain of latency-bound waves): they are dealt to ndev * searches_per_device worker contexts.
 * Outputs per model i: status, result, out_height; rhs_out packed by cumulative (heights[i] + 2*nints_i),
 * pos_out/var_out by cumulative (widths[i] + heights[i] + 2*nints_i).  Results equal yalps_solve per model.
 */
int yalps_multi_solve_many(yalps_multi *m, int64_t n_models, const int32_t *heights, const int32_t *widths,
                           const int64_t *mat_offsets, const double *matrices, const int64_t *ints_offsets,
                           const int32_t *ints, const double *signs, const yalps_options *opt,
                           int32_t searches_per_device, int32_t *status, double *result, int32_t *out_height,
                           double *rhs_out, int32_t *pos_out, int32_t *var_out);

/*
 * ONE large LP over all the ranks of m (SURVEY 8(f)-3; north_star (c) widened from the grid of one GPU to the GPUs of
 * one box): simplex() of src/simplex.ts:99-142 on one height x width tableau whose rows are dealt round robin to the
 * ranks (row r -> rank r % ndev), so ndev GPUs hold -- and update -- a tableau ndev times the size one could.  One
 * persistent cooperative kernel per rank; per pivot the pivot column is all-gathered and the raw pivot row broadcast by
 * stores into the peers' memory (NVLink / NVSwitch peer access, cudaDeviceEnablePeerAccess) from inside those kernels,
 * published with system-scope release flags: no host round trip and no collective call per pivot.  Every rank makes the
 * same pivot choice from private copies of the objective row and RHS column, so the trajectory -- and every output bit
 * -- is that of yalps_solve_batch(n = 1).  matrix is a HOST array (reference layout); outputs as yalps_solve_batch for
 * n = 1, matrix_out (nullable) receives the final tableau; kernel_ms (nullable) the device time of the slowest rank's
 * kernel (CUDA events).  Fails with YALPS_ERR_CUDA when two GPUs of m have no peer path or the ranks' kernels could not
 * run at the same time (every in-kernel wait has a ~2 s budget, so a missing peer cannot hang a GPU).
 */
int yalps_multi_solve_large(yalps_multi *m, int32_t height, int32_t width, const double *matrix,
                            const yalps_options *opt, int32_t *status, double *value, int64_t *pivots, double *rhs_out,
                            int32_t *pos_out, int32_t *var_out, double *matrix_out, double *kernel_ms);

/* roundToPrecision (src/util.ts:1-4) evaluated on the device for n values (parity probe). */
int yalps_round_to_precision(yalps_ctx *ctx, int64_t n, const double *x, double precision, double *out);

/* Probe: the shared-reciprocal division of csrc/fastdiv.cuh against __ddiv_rn on n hash-generated operand pairs
 * (mode 0..4: random bit patterns, tableau-like values, special values, exact quotients, exponent extremes).
 * The kernels must divide exactly like the reference's JS `/` (src/simplex.ts:19,25,36,89,128). */
int yalps_probe_division(yalps_ctx *ctx, int64_t n, uint64_t seed, int32_t mode, uint64_t *mismatches,
                         uint64_t *first_bad_bits /* [2]: numerator, divisor; may be NULL */);
/* Shared-memory stream microbenchmark: bytes moved per second by ld/st.shared.f64 on all SMs
 * (the measured denominator of the K1 roofline).  Returns GB/s in *gbs. */
int yalps_measure_smem_bandwidth(yalps_ctx *ctx, double *gbs, double *sm_clock_mhz);
/* L2 stream microbenchmark: read + write GB/s of the rank-1 update's ld-mul-sub-st pattern over a `bytes`-sized buffer
 * that stays in L2 (the denominator for working copies that are L2-resident while their CTA works on them). */
int yalps_measure_l2_bandwidth(yalps_ctx *ctx, uint64_t bytes, double *gbs);
/* Bare host-to-device copy of `bytes` from a PINNED host buffer into a device scratch buffer, `reps` times over
 * `nstreams` (1 or 2) streams: seconds per repetition.  bench.py runs it on all ranks at once to print the ceiling
 * the box's PCIe / host-memory fabric puts on the end-to-end rate (e2e.h2d_ceiling_gbs). */
int yalps_measure_h2d_bandwidth(yalps_ctx *ctx, const void *pinned_host, uint64_t bytes, int32_t reps, int32_t nstreams,
                                double *seconds);
/* Tensor-memory stream microbenchmark: bytes read + written per second by tcgen05.ld/st.32x32b.x32 with the
 * multiply-subtract of the rank-1 update in between, 16 warps per SM (what bounds K1t's row pass). */
int yalps_measure_tmem_bandwidth(yalps_ctx *ctx, double *gbs, double *sm_clock_mhz);

#ifdef __cplusplus
}
#endif
#endif /* YALPS_B200_H */
