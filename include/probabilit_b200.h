/* probabilit_b200 -- C ABI of the B200-native sampling hot path of tommyod/probabilit.
 *
 * The reference is pure Python; its "plugin seam" is duck-typed (SURVEY.md section 8b):
 *   correlator protocol   Correlator.set_target(C) -> self ; correlator(X) -> X'
 *                         (reference src/probabilit/correlation.py:162-179, :368-425;
 *                          called from src/probabilit/modeling.py:577-581)
 * Each entry point below names the reference interface it replaces.  All functions return a
 * pbl_status; pbl_last_error() gives the message of the last failure on the calling thread.
 * Pointers named *_dev are device pointers on the current CUDA device, everything else is host
 * memory.  Matrices are (n rows = observations, k columns = variables), fp64, addressed as
 * base[row * row_stride + col * col_stride] with strides in ELEMENTS (NumPy F-order: row_stride 1,
 * col_stride n; C-order: row_stride k, col_stride 1).  No call takes ownership of caller memory;
 * inputs are never modified (the reference writes into np.empty_like(X), correlation.py:418).
 */
#ifndef PROBABILIT_B200_H
#define PROBABILIT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBL_API __attribute__((visibility("default")))

typedef enum pbl_status {
  PBL_OK = 0,
  PBL_NOT_POSITIVE_DEFINITE = 1, /* ValueError "Rank data correlation not positive definite." correlation.py:399-403 */
  PBL_NON_FINITE = 2,            /* ValueError "array must not contain infs or NaNs" (scipy check_finite at :409) */
  PBL_BAD_SHAPE = 3,             /* ValueError from Correlator._validate_X, correlation.py:181-202 */
  PBL_CUDA_ERROR = 4,
  PBL_INTERNAL = 5,
  PBL_RETRY = 6, /* stage API only (pbl_ic_stage_status): the data are too dense for the 32-bit sort window;
                   the plan has switched to the exact 64-bit sort, repeat from pbl_ic_stage_begin.
                   pbl_ic_plan_run / pbl_iman_conover_f64 handle this internally. */
  PBL_OUT_OF_TABLE = 7 /* pbl_stats_histogram: a bin index left the edge table, where np.histogram's indexing raises
                          (int64 data beyond 2^53 cast outside the float edges); bad_row[] names the first row */
} pbl_status;

/* ---- library ---- */
PBL_API int pbl_version(void);
PBL_API const char* pbl_last_error(void);
PBL_API int pbl_device_count(void);
PBL_API int pbl_set_device(int device);
/* the calling thread's current CUDA device (so that a caller can restore it after pbl_set_device) */
PBL_API int pbl_get_device(int* device);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
PBL_API int64_t pbl_kernel_launches(void);

/* CUDA-event timing of the radix-sort digit passes (the dominant kernel), for bench.py's
 * roofline leg: enable, run, then read (#launches, their total ms, keys moved) and reset. */
PBL_API int pbl_sort_profile_enable(int on);
PBL_API int pbl_sort_profile_read(int64_t* launches, double* total_ms, int64_t* keys);

/* ---- memory helpers (so that a host language without a CUDA binding can stage data) ---- */
PBL_API int pbl_device_malloc(void** ptr_dev, uint64_t bytes);
PBL_API int pbl_device_free(void* ptr_dev);
PBL_API int pbl_host_malloc_pinned(void** ptr, uint64_t bytes);
PBL_API int pbl_host_free_pinned(void* ptr);
PBL_API int pbl_memcpy_h2d(void* dst_dev, const void* src, uint64_t bytes, void* stream);
PBL_API int pbl_memcpy_d2h(void* dst, const void* src_dev, uint64_t bytes, void* stream);
PBL_API int pbl_stream_synchronize(void* stream);

/* ---- peer memory (one process per GPU, NVLink): the multi-GPU Iman-Conover moves its row <-> column
 * transposes with the copy engines straight into / out of the peers' buffers.  The reference is
 * single-process (no counterpart).  export: 64-byte CUDA IPC handle of a buffer that is the BASE of a
 * device allocation made by this library (pbl_device_malloc, pbl_ic_plan_buffer 0/1); open: map a
 * peer's buffer into this process (peer access is enabled on first use); copy_many: `count`
 * device-to-device copies (local or peer pointers) issued on a pool of side streams, ordered after
 * the work already in `stream`, which resumes when all of them have finished. ---- */
PBL_API int pbl_ipc_export(const void* ptr_dev, void* handle64);
PBL_API int pbl_ipc_open(const void* handle64, void** ptr_dev);
PBL_API int pbl_ipc_close(void* ptr_dev);
PBL_API int pbl_peer_copy_streams(int32_t n); /* side streams used by copy_many: 1..8, default 4 */
PBL_API int pbl_peer_copy_many(int32_t count, void* const* dst_dev, const void* const* src_dev,
                               const uint64_t* bytes, void* stream);

/* ---- Iman-Conover correlator: ImanConover().set_target(C)(X), correlation.py:288-425 ---- */
typedef struct pbl_ic_plan pbl_ic_plan;

/* Workspace for (n, k) problems on the current device.  col_batch <= 0: choose automatically
 * (columns sorted per launch batch; bounds the sort workspace). */
PBL_API int pbl_ic_plan_create(int64_t n, int32_t k, int32_t col_batch, pbl_ic_plan** plan);
/* flags bit 0 (PBL_IC_ROWS_ONLY): no sort workspace -- the plan serves the Gram / solve / transform
 * stages of a row shard in the multi-GPU driver (the sorts run in a second, column-shard plan). */
#define PBL_IC_ROWS_ONLY 1
PBL_API int pbl_ic_plan_create_ex(int64_t n, int32_t k, int32_t col_batch, int32_t flags, pbl_ic_plan** plan);
PBL_API int pbl_ic_plan_destroy(pbl_ic_plan* plan);
PBL_API uint64_t pbl_ic_plan_bytes(const pbl_ic_plan* plan);

/* Correlator.set_target (correlation.py:162-179): the k x k validation and P = cholesky(C) stay
 * on the host (NumPy); P_lower is that lower-triangular factor, row-major k*k doubles. */
PBL_API int pbl_ic_plan_set_target(pbl_ic_plan* plan, const double* P_lower);

/* ImanConover.__call__ (correlation.py:368-425) on device-resident X -> Y.  Synchronous: returns
 * after the stream has drained, with the status the reference would have raised. */
PBL_API int pbl_ic_plan_run(pbl_ic_plan* plan, const double* X_dev, int64_t x_row_stride,
                    int64_t x_col_stride, double* Y_dev, int64_t y_row_stride,
                    int64_t y_col_stride, void* stream);

/* Cholesky().set_target(C)(X), reference correlation.py:205-285, on device-resident X -> Y with a
 * plan whose target has been set (a PBL_IC_ROWS_ONLY plan is enough: no sorts).  Synchronous.
 * PBL_NOT_POSITIVE_DEFINITE = numpy.linalg.LinAlgError from cholesky(cov) (:271). */
PBL_API int pbl_cholesky_plan_run(pbl_ic_plan* plan, const double* X_dev, int64_t x_row_stride,
                                  int64_t x_col_stride, double* Y_dev, int64_t y_row_stride,
                                  int64_t y_col_stride, void* stream);

/* ---- PermutationCorrelator, reference correlation.py:473-703 with CorrelationMatrix :757-921 ----
 * begin : Y <- X (column-major [k][n], caller-owned), CorrelationMatrix.__init__ (:819-853) on it
 *         (spearman != 0: on rankdata(X), needs a plan with sort workspace).  target / weights are
 *         HOST k*k row-major (weights already normalised to sum 1, :592-593).
 *         PBL_NOT_POSITIVE_DEFINITE here means "X has one or several constant columns" (:847-848).
 * steps : run n_steps hill-climbing steps in ONE launch.  Step t works on column step_col[t] with the
 *         swap lists i = swaps[2*step_off[t] .. +step_cnt[t]), j = the next step_cnt[t] entries -- the
 *         host draws them exactly like SwapIndexGenerator (:428-470) so the accept/reject sequence is
 *         the reference's.  After every step on column 0 the weighted RMSE (:597-601) is compared with
 *         tol (:689-697); errors[0] = error before the first step, errors[1..] = after each check.
 * corr  : the running correlation matrix (k*k, host), for tests. */
PBL_API int pbl_permcorr_begin(pbl_ic_plan* plan, const double* X_dev, int64_t x_row_stride,
                               int64_t x_col_stride, double* Y_dev, int32_t spearman, const double* target,
                               const double* weights, void* stream);
PBL_API int pbl_permcorr_steps(pbl_ic_plan* plan, double* Y_dev, const int32_t* step_col,
                               const int32_t* step_off, const int32_t* step_cnt, const int64_t* swaps,
                               int64_t n_swaps_total, int64_t n_steps, double tol, int64_t* steps_done,
                               int32_t* converged, double* errors, int64_t errors_cap, int64_t* n_errors,
                               void* stream);
PBL_API int pbl_permcorr_corr(pbl_ic_plan* plan, double* corr);

/* dst[r * d_row_stride + c * d_col_stride] = src[r * s_row_stride + c * s_col_stride] for an (n, k) fp64 matrix on
 * the device (element strides; the buffers must not overlap).  Layout conversion around the correlators that
 * work column-major inside: `X.copy()` keeps the caller's C order in the reference (correlation.py:830-831), so
 * the result of PermutationCorrelator goes back row-major without a host-side transpose.  Asynchronous. */
PBL_API int pbl_copy_strided_f64(const double* src_dev, int64_t s_row_stride, int64_t s_col_stride, double* dst_dev,
                                 int64_t d_row_stride, int64_t d_col_stride, int64_t n, int32_t k, void* stream);

/* Verification helper: np.corrcoef(X, rowvar=False) (spearman == 0) or the Spearman matrix
 * (Pearson correlation of scipy.stats.rankdata's average ranks; the Spearman mode of CorrelationMatrix,
 * correlation.py:835-837) of device-resident X into HOST out[k*k].  Spearman needs a plan with sort
 * workspace.  Synchronous. */
PBL_API int pbl_corrcoef_f64(pbl_ic_plan* plan, const double* X_dev, int64_t x_row_stride, int64_t x_col_stride,
                             int32_t spearman, double* out, void* stream);

/* ImanConover.__call__ with HOST buffers on a reusable plan: X / Y contiguous in C or F order, the
 * caller provides device staging for n*k doubles each.  For column-major data the host<->device
 * copies are pipelined with the per-column sorts (page-locked host memory makes them asynchronous). */
PBL_API int pbl_ic_plan_run_host(pbl_ic_plan* plan, const double* X, int64_t x_row_stride, int64_t x_col_stride,
                                 double* Y, int64_t y_row_stride, int64_t y_col_stride, double* X_staging_dev,
                                 double* Y_staging_dev, void* stream);

/* Same call with HOST buffers (what a NumPy caller holds): copies X to the device, runs, copies Y
 * back.  X and Y must each be one contiguous block in C or F order. */
PBL_API int pbl_iman_conover_f64(const double* X, int64_t n, int32_t k, int64_t x_row_stride,
                         int64_t x_col_stride, const double* P_lower, double* Y,
                         int64_t y_row_stride, int64_t y_col_stride);

/* Stage-level entry points (asynchronous on `stream`): used by the parity tests and by the
 * multi-GPU host driver, which places its collectives between them.
 *   rank_scores : correlation.py:394-395 (+ np.sort of :423) for columns [col0, col0+ncols)
 *   gram        : the reduction inside np.corrcoef, :398
 *   solve       : corrcoef normalisation, cholesky, T = Q^-T P^T, :398-414 (n_total = global rows)
 *   transform   : :409-414 applied to the rows
 *   rank_gather : :419-423 for columns [col0, col0+ncols)
 *   status      : synchronise and report (PBL_OK / NOT_POSITIVE_DEFINITE / NON_FINITE / ...)  */
PBL_API int pbl_ic_stage_begin(pbl_ic_plan* plan, void* stream);
PBL_API int pbl_ic_stage_rank_scores(pbl_ic_plan* plan, const double* X_dev, int64_t row_stride,
                             int64_t col_stride, int32_t col0, int32_t ncols, void* stream);
PBL_API int pbl_ic_stage_gram(pbl_ic_plan* plan, void* stream);
PBL_API int pbl_ic_stage_solve(pbl_ic_plan* plan, int64_t n_total, void* stream);
PBL_API int pbl_ic_stage_transform(pbl_ic_plan* plan, void* stream);
PBL_API int pbl_ic_stage_rank_gather(pbl_ic_plan* plan, double* Y_dev, int64_t row_stride,
                             int64_t col_stride, int32_t col0, int32_t ncols, void* stream);
PBL_API int pbl_ic_stage_status(pbl_ic_plan* plan, void* stream);

/* Row-chunk hook for a multi-GPU driver: while set (fn != NULL), the scatter by row that ends
 * rank_scores / rank_gather is enqueued chunk by chunk -- chunk g = output rows [g*chunk_rows,
 * (g+1)*chunk_rows), in the order first_chunk, first_chunk+1, ... wrapping -- and fn(column, g, user) is
 * called on the calling thread right after chunk g has been enqueued on the stream, so the driver can
 * send that row range to its owner while the rest is still being delivered. */
typedef void (*pbl_chunk_fn)(int32_t column, int32_t chunk, void* user);
PBL_API int pbl_ic_plan_set_chunk_hook(pbl_ic_plan* plan, int64_t chunk_rows, int32_t first_chunk,
                                       pbl_chunk_fn fn, void* user);

/* Device pointers to the plan's intermediates (column-major [k][n] unless noted), for parity
 * tests and for collectives: what = 0 scores / correlated scores, 1 sortedX, 2 gram [k][k],
 * 3 colsum [k], 4 T [k][k] row-major, 5 work (R then Q) [k][k]. */
PBL_API int pbl_ic_plan_buffer(pbl_ic_plan* plan, int32_t what, void** ptr_dev, uint64_t* bytes);

/* ---- unit-cube generators: the `quantiles = ...` draw of Node.sample, src/probabilit/modeling.py:479-489.
 * out_dev is (n, d) fp64 addressed with element strides (column-major: row_stride 1, col_stride n).
 * Every point depends on its global row index only: a row shard passes its first row as
 * row0 / skip / start_index and needs no communication. ---- */

/* method=None: random_state.random((n, d)), modeling.py:485-486.  Philox4x32-10 counter stream
 * (statistical parity with NumPy's generators, not bit parity); row0 must be even. */
PBL_API int pbl_uniform_f64(uint64_t seed, uint64_t row0, int64_t n, int32_t d, double* out_dev,
                            int64_t row_stride, int64_t col_stride, void* stream);

/* method="sobol": scipy.stats.qmc.Sobol(d, rng).random(n), modeling.py:482,488-489.
 *   direction numbers: Joe-Kuo tables (poly[d], vinit[d][vinit_cols], int64) -> sv[d][bits]
 *   scramble: LMS + digital shift from the host generator's random bits (ltm_bits[d][bits][bits],
 *             shift_bits[d][bits], one byte per bit, drawn exactly like scipy draws them)
 *   points skip .. skip+n-1 of the sequence; bit-exact with scipy for the same sv / shift. */
PBL_API int pbl_sobol_direction_numbers(const int64_t* poly_dev, const int64_t* vinit_dev, int32_t vinit_cols,
                                        int32_t d, int32_t bits, uint64_t* sv_dev, void* stream);
PBL_API int pbl_sobol_scramble(const uint8_t* ltm_bits_dev, const uint8_t* shift_bits_dev, int32_t d,
                               int32_t bits, uint64_t* sv_dev, uint64_t* shift_dev, void* stream);
PBL_API int pbl_sobol_f64(const uint64_t* sv_dev, const uint64_t* shift_dev, int32_t d, int32_t bits,
                          uint64_t skip, int64_t n, double* out_dev, int64_t row_stride,
                          int64_t col_stride, void* stream);

/* method="halton": scipy.stats.qmc.Halton(d, rng).random(n), modeling.py:481.  bases[d] = first d
 * primes; perms (or NULL when unscrambled): per dimension perm_count[c] x bases[c] digit
 * permutations starting at perms[perm_off[c]].  Bit-exact with scipy for the same permutations. */
PBL_API int pbl_halton_f64(const int32_t* bases_dev, const int64_t* perms_dev, const int64_t* perm_off_dev,
                           const int32_t* perm_count_dev, int32_t d, uint64_t start_index, int64_t n,
                           double* out_dev, int64_t row_stride, int64_t col_stride, void* stream);

/* method="lhs": scipy.stats.qmc.LatinHypercube(d, rng).random(n), modeling.py:480 / README.md:113.
 * (perm + 1 - U) / n with a counter-based per-column permutation (statistical parity). */
PBL_API int pbl_lhs_f64(uint64_t seed, int64_t n, int32_t d, int32_t scramble, double* out_dev,
                        int64_t row_stride, int64_t col_stride, void* stream);

/* ---- fused modeling-graph evaluation: the per-node loop of Node.sample_from_quantiles,
 * src/probabilit/modeling.py:586-612, with Distribution._sample (:795-812, scipy.stats ppf),
 * Constant._sample (:760-763) and Transform._sample (:954-956, :1007-1009, :1071-1072) fused into
 * ONE pass per sample: every node value lives in an on-chip slot, only retained nodes are written.
 *
 * A program is a list of pbl_graph_instr executed per sample (row).  Operands src[i] >= 0 name a
 * slot, src[i] < 0 means "use imm[i]" (a scalar parameter / folded Constant).  Values are fp64;
 * booleans are 0.0 / 1.0 (the host mirror keeps NumPy's result dtype and converts on download).
 * An int64 value computed by a PBL_OP_I_* instruction occupies the same 8-byte slot, accumulator and output
 * column as its int64 BIT PATTERN (__double_as_longlong / __longlong_as_double), and so does an immediate
 * operand of an integer instruction in imm[i] (like the Philox seed of PBL_OP_UNIFORM).  Integer values that
 * a table lookup produces (DiscreteDistribution values, EmpiricalDistribution data) stay exact doubles;
 * PBL_OP_F2I / PBL_OP_I2F convert between the two forms.
 *   PBL_OP_LOAD   dst <- inputs[src[0]][row]      (a quantile column, or a correlated sample column)
 *   PBL_OP_STORE  outputs[src[1]][row] <- slot src[0]                      (node.samples_ retained)
 *   PBL_OP_CHECK  if slot src[0] is not finite: report node tag src[1]      (modeling.py:600-606)
 *   PBL_OP_UNIFORM dst <- Philox uniform of (seed = imm[0] bits, global row = row0 + row, column src[0])
 *                 -- the same stream as pbl_uniform_f64, generated in-kernel (no quantile read)
 *   PBL_OP_SPILL  spill slot src[1] <- slot src[0]
 *   PBL_OP_FILL   dst <- spill slot src[0]
 *                 -- a program that needs more than PBL_GRAPH_MAX_SLOTS live values keeps the rest in spill
 *                 slots: per-row scratch in global memory (L2 resident) that the library owns, neither an input
 *                 nor an output.  Values move as 8-byte patterns (int64 bits survive).  Spill indices are below
 *                 PBL_GRAPH_MAX_SPILLS; neither instruction takes a PBL_GRAPH_* flag.
 *   PBL_PPF_*     dst <- scipy.stats.<distr>(shape..., loc, scale).ppf(q) with q = operand 0;
 *                 operands: NORM(q, loc, scale) UNIFORM_(q, loc, scale) EXPON(q, loc, scale)
 *                 TRIANG(q, c, loc, scale) GAMMA(q, a, loc, scale) LOGNORM(q, s, loc, scale)
 *                 POISSON(q, mu, loc) BINOM(q, n, p, loc) BERNOULLI(q, p, loc)
 *                 including SciPy's wrapper semantics (invalid parameters -> nan, q == 0 / 1 ->
 *                 support bounds; scipy/stats/_distn_infrastructure.py:2305-2348, :3745-3792)
 *   arithmetic    the NumPy ufunc behind each Transform class (modeling.py:962-1169). */
typedef enum pbl_graph_op {
  PBL_OP_NOP = 0, PBL_OP_LOAD = 1, PBL_OP_STORE = 2, PBL_OP_CHECK = 3, PBL_OP_MOV = 4, PBL_OP_UNIFORM = 5,
  PBL_OP_SPILL = 6, PBL_OP_FILL = 7,
  /* ppf */
  PBL_PPF_NORM = 16, PBL_PPF_UNIFORM = 17, PBL_PPF_EXPON = 18, PBL_PPF_TRIANG = 19, PBL_PPF_GAMMA = 20,
  PBL_PPF_LOGNORM = 21, PBL_PPF_POISSON = 22, PBL_PPF_BINOM = 23, PBL_PPF_BERNOULLI = 24,
  /* table-lookup distributions (modeling.py:825-927): operand 0 = q, src[1] = INDEX INTO inputs[] of a
   * device table (not a slot), imm[1] = table length m, imm[2] = method
   *   TABLE_INTERP   np.interp(q, xp, fp), table = xp[m] then fp[m]         (CumulativeDistribution)
   *   TABLE_SEARCH   np.searchsorted(cum, q, side="right") as a double       (DiscreteDistribution)
   *   TABLE_QUANTILE np.quantile(sorted data, q, method), table = data[m]    (EmpiricalDistribution)
   *                  method 0 linear 1 lower 2 higher 3 nearest 4 midpoint 5 closest_observation */
  PBL_PPF_TABLE_INTERP = 25, PBL_PPF_TABLE_SEARCH = 26, PBL_PPF_TABLE_QUANTILE = 27,
  /* four-parameter distributions: operands (q, a, b, scale), result for loc = 0 -- the caller adds loc
   * with a separate PBL_OP_ADD (scipy's `_ppf * scale + loc` is two roundings anyway)
   *   BETA      scipy.stats.beta(a, b)       (PERT, reference src/probabilit/distributions.py:79-94)
   *   TRUNCNORM scipy.stats.truncnorm(a, b)  (TruncatedNormal, distributions.py:17-29) */
  PBL_PPF_BETA = 28, PBL_PPF_TRUNCNORM = 29,
  /* binary (dst <- op(a, b)) */
  PBL_OP_ADD = 32, PBL_OP_MUL = 33, PBL_OP_SUB = 34, PBL_OP_DIV = 35, PBL_OP_POW = 36, PBL_OP_FLOORDIV = 37,
  PBL_OP_MOD = 38, PBL_OP_MAX = 39, PBL_OP_MIN = 40, PBL_OP_ATAN2 = 41, PBL_OP_LT = 42, PBL_OP_LE = 43,
  PBL_OP_GT = 44, PBL_OP_GE = 45, PBL_OP_EQ = 46, PBL_OP_NE = 47, PBL_OP_AND = 48, PBL_OP_OR = 49,
  PBL_OP_ISCLOSE = 50,
  /* int64 binary, NumPy's int64 ufuncs: + - * ** wrap modulo 2^64; FLOORDIV / MOD by 0 give 0,
   * INT64_MIN // -1 = INT64_MIN, MOD takes the sign of the divisor; POW of a negative exponent gives 1 and
   * fails the instruction's domain (see PBL_GRAPH_CHECK); comparisons give booleans (GT / GE: swap operands) */
  PBL_OP_I_ADD = 51, PBL_OP_I_SUB = 52, PBL_OP_I_MUL = 53, PBL_OP_I_FLOORDIV = 54, PBL_OP_I_MOD = 55,
  PBL_OP_I_POW = 56, PBL_OP_I_MAX = 57, PBL_OP_I_MIN = 58, PBL_OP_I_LT = 59, PBL_OP_I_LE = 60, PBL_OP_I_EQ = 61,
  PBL_OP_I_NE = 62,
  /* unary (dst <- op(a)) */
  PBL_OP_NEG = 64, PBL_OP_ABS = 65, PBL_OP_LOG = 66, PBL_OP_EXP = 67, PBL_OP_FLOOR = 68, PBL_OP_CEIL = 69,
  PBL_OP_SIGN = 70, PBL_OP_SQRT = 71, PBL_OP_SQUARE = 72, PBL_OP_LOG10 = 73, PBL_OP_SIN = 74, PBL_OP_COS = 75,
  PBL_OP_TAN = 76, PBL_OP_ASIN = 77, PBL_OP_ACOS = 78, PBL_OP_ATAN = 79, PBL_OP_SINH = 80, PBL_OP_COSH = 81,
  PBL_OP_TANH = 82, PBL_OP_ASINH = 83, PBL_OP_ACOSH = 84, PBL_OP_ATANH = 85, PBL_OP_NOT = 86,
  /* dst <- table[(int) a]; src[1] = index into inputs[] of the table, imm[1] = its length
   * (`self.values[idx]` of DiscreteDistribution, modeling.py:913); out of range -> nan */
  PBL_OP_LOOKUP = 87,
  /* int64 unary (NEG / ABS / SQUARE wrap: abs(INT64_MIN) = INT64_MIN), and the two conversions:
   *   I2F  int64 -> double rounded to nearest (NumPy's int64 -> float64 cast before a mixed operation)
   *   F2I  an integral double (a boolean's 0.0 / 1.0, a table value) -> int64 */
  PBL_OP_I_NEG = 88, PBL_OP_I_ABS = 89, PBL_OP_I_SIGN = 90, PBL_OP_I_SQUARE = 91, PBL_OP_I2F = 92, PBL_OP_F2I = 93
} pbl_graph_op;

/* Flags or-ed into pbl_graph_instr.op of a computing instruction (ppf / arithmetic / MOV) so that the
 * common load -> ppf -> check -> store chain of one node is ONE interpreted instruction:
 *   Q_INPUT    (ppf only) operand 0 is inputs[src[0]][row] instead of a slot
 *   Q_UNIFORM  (ppf only) operand 0 is the Philox uniform of column src[0], seed bits in imm[0]
 *   CHECK      after computing: if the result is not finite report node tag (dst >> 8) & 0xFFF.  Integers are
 *              always finite: on PBL_OP_I_POW (the only integer instruction that takes it) the flag reports
 *              the tag when the exponent of an active row is negative (NumPy raises ValueError there)
 *   STORE      after computing: outputs[dst >> 20][row] <- result
 * dst & 0xFF is the destination slot. */
#define PBL_GRAPH_Q_INPUT 0x100
#define PBL_GRAPH_Q_UNIFORM 0x200
#define PBL_GRAPH_CHECK 0x400
#define PBL_GRAPH_STORE 0x800

typedef struct pbl_graph_instr {
  int32_t op;     /* pbl_graph_op | PBL_GRAPH_* flags */
  int32_t dst;    /* destination slot | check tag << 8 | output index << 20 */
  int32_t src[4]; /* slot index, or < 0: imm[i] */
  double imm[4];
} pbl_graph_instr;

#define PBL_GRAPH_MAX_SLOTS 96
#define PBL_GRAPH_MAX_INSTR 4096
/* A program with spills runs on exactly the resident grid (one 128-thread block per SM at 96 slots), so its
 * scratch is n_spills x R x grid x 128 x 8 bytes whatever n is: 303 KB per spill slot at R = 2 on 148 SMs, and
 * 1024 spill slots are at most ~310 MB at that occupancy.  A model that needs more splits into several launches
 * (the host mirror does). */
#define PBL_GRAPH_MAX_SPILLS 1024

/* Evaluate `program` for rows 0..n-1.  inputs_dev / outputs_dev are HOST arrays of device column
 * pointers (contiguous fp64 columns of n rows).  *first_nonfinite receives the smallest node tag
 * whose CHECK failed, or -1.  row0 = global index of row 0 (for PBL_OP_UNIFORM on a row shard).
 * Synchronous (returns after the stream has drained).  One call holds at most PBL_GRAPH_MAX_INSTR instructions,
 * PBL_GRAPH_MAX_SLOTS slots and PBL_GRAPH_MAX_SPILLS spill slots; a larger model is several calls that pass values
 * on through n-row columns (an output of one call, an input of the next). */
PBL_API int pbl_graph_eval_f64(const pbl_graph_instr* program, int32_t n_instr, int32_t n_slots, int64_t n,
                               uint64_t row0, const double* const* inputs_dev, int32_t n_inputs,
                               double* const* outputs_dev, int32_t n_outputs, int32_t* first_nonfinite,
                               void* stream);
/* The same special functions one element at a time, for the parity tests:
 * what = a PBL_PPF_* code; p0..p2 = the distribution's operands after q (see above). */
PBL_API int pbl_ppf_f64(int32_t what, const double* q_dev, int64_t n, double p0, double p1, double p2,
                        double* out_dev, void* stream);

/* ---- statistics of sampled columns, bit-identical to NumPy on the host copy (node.samples_) ----
 * cols_dev[c] is a device column of n 8-byte values (n >= 1; every column of a call has the same n) holding
 *   PBL_STATS_F64          doubles                                   (NumPy float64)
 *   PBL_STATS_I64_BITS     int64 bit patterns                        (int64: the result of an integer instruction)
 *   PBL_STATS_I64_AS_F64   doubles holding int64 values exactly      (int64: table values)
 *   PBL_STATS_BOOL_AS_F64  0.0 / 1.0                                 (bool)
 * kinds[] and q[] are host arrays; `out` is host or device memory (ncols results, or ncols x nq row-major).  Both
 * calls are synchronous. */
typedef enum pbl_stats_kind {
  PBL_STATS_F64 = 0, PBL_STATS_I64_BITS = 1, PBL_STATS_I64_AS_F64 = 2, PBL_STATS_BOOL_AS_F64 = 3
} pbl_stats_kind;
typedef enum pbl_stats_moment { PBL_STATS_MEAN = 0, PBL_STATS_VAR = 1, PBL_STATS_STD = 2 } pbl_stats_moment;

/* np.mean / np.var(ddof) / np.std(ddof) per column: float64 pairwise summation in NumPy's tree order; an int64 or
 * bool column's mean sums chunks of `chunk` elements (np.getbufsize(): the ufunc buffer of the cast to float64) and
 * adds the chunk sums in order.  var / std divide the sum of squares by `divisor` = max(n - ddof, 0). */
PBL_API int pbl_stats_moments(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                              int64_t chunk, int32_t what, double divisor, double* out, void* stream);
/* np.quantile(column, q, method) for nq values q in [0, 1], method as for PBL_PPF_TABLE_QUANTILE (0 linear 1 lower
 * 2 higher 3 nearest 4 midpoint 5 closest_observation).  out[c * nq + i] is a double, except for an integer or bool
 * column with a method that does not interpolate: then it holds the int64 value (bool: 0 / 1).  A float column that
 * holds a NaN gives NaN for every q.  Scratch on the device: O(ncols x nq), whatever n is. */
PBL_API int pbl_stats_quantiles(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                                const double* q, int32_t nq, int32_t method, void* out, void* stream);

/* np.min and np.max per column in one read: out[2c] = min, out[2c + 1] = max, a double for PBL_STATS_F64 and the
 * int64 value for the other kinds.  A float column that holds a NaN gives the bits of its first NaN for both. */
PBL_API int pbl_stats_minmax(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n, void* out,
                             void* stream);

/* The values np.histogram keeps, `(a >= lo) & (a <= hi)`.  NumPy evaluates the two comparisons separately, each in
 * the result type of the data and that edge, so each edge has its own type: PBL_HIST_CMP_F64 compares float64(a) with
 * lo_f (hi_f), PBL_HIST_CMP_I64 compares the integer value with lo_i (hi_i); integer kinds only. */
typedef enum pbl_hist_cmp { PBL_HIST_CMP_F64 = 0, PBL_HIST_CMP_I64 = 1 } pbl_hist_cmp;
typedef struct pbl_stats_range {
  int32_t lo_cmp, hi_cmp;
  double lo_f, hi_f;
  int64_t lo_i, hi_i;
} pbl_stats_range;

/* np.histogram's counts of one column (numpy/lib/_histograms_impl.py, NumPy 2.3):
 *   PBL_HIST_UNIFORM  the equal-bin path: keep `range`, x = float64(a), i = int64(((x - first) / denom) * nbins),
 *                     i == nbins -> nbins - 1, x < table[i] -> i - 1, x >= table[i + 1] and i != nbins - 1 -> i + 1;
 *                     table = the nbins + 1 float64 edges.  nbins counts.
 *   PBL_HIST_EDGES    the edge-array path, as counts of cells: table = m distinct edge values in ascending order
 *                     (double, or int64 for PBL_HIST_CMP_I64), cell 2k + 1 counts the values equal to table[k],
 *                     cell 2k the values between table[k - 1] and table[k], cell 2m the values above table[m - 1],
 *                     cell 2m + 1 the NaNs; the caller forms searchsorted's cumulative counts from them.  nbins = m,
 *                     2m + 2 counts. */
typedef enum pbl_hist_mode { PBL_HIST_UNIFORM = 0, PBL_HIST_EDGES = 1 } pbl_hist_mode;
typedef struct pbl_stats_hist_spec {
  int32_t mode;
  int32_t cmp;           /* PBL_HIST_EDGES only: the comparison type of the table (np.result_type(data, edges)) */
  pbl_stats_range keep;  /* PBL_HIST_UNIFORM only */
  double first, denom;   /* PBL_HIST_UNIFORM only: float64(first edge), float64(_unsigned_subtract(last, first)) */
  int64_t nbins;
  const void* table;     /* host */
  int64_t offset;        /* index of the column's first count in `counts` */
} pbl_stats_hist_spec;

/* Counts of every column into counts[] (host, `total` uint64).  PBL_OUT_OF_TABLE: for every column, bad_row[c]
 * (host) is the first row whose bin index left the table, or -1; the counts are then not meaningful. */
PBL_API int pbl_stats_histogram(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                                const pbl_stats_hist_spec* specs, uint64_t* counts, int64_t total, int64_t* bad_row,
                                void* stream);

/* a[keep] of every column, in order, into out_dev[c] (kept[c] 8-byte values, the column's kind); kept[c] (host)
 * receives the number of values written.  With out_dev NULL the call only counts (one read), so that the caller can
 * size the outputs; the call that writes reads every column twice. */
PBL_API int pbl_stats_compact(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                              const pbl_stats_range* keep, void* const* out_dev, int64_t* kept, void* stream);

/* The distinct values of one column (numpy/lib/_arraysetops_impl.py:_unique1d), for np.unique / np.bincount.  The
 * host arrays have room for n entries each; the call fills the first nunique (nnan) of them:
 *   values    the double bits of each distinct non-NaN value, ascending; -0.0 and +0.0 are one value, reported with
 *             the sign of its first row.  Integer and bool kinds come back as exact doubles.
 *   first     (or NULL) the first row holding each value
 *   counts    (or NULL) the rows holding each value
 *   nan_rows  the rows holding a NaN, ascending (PBL_STATS_F64 only; NumPy sorts every NaN last)
 *   nan_bits  their bits
 *   inverse   (device, n int64, or NULL) the index of each row's value in `values`; a NaN row gets nunique with
 *             equal_nan, nunique + its index in nan_rows without.
 * PBL_STATS_I64_BITS columns must hold values within +-2^53 (else PBL_BAD_SHAPE).  n <= 2^31 - 1.  Each column is
 * sorted once (the 8-pass exact sort of the Iman-Conover engine, constant digits skipped); device scratch is about
 * 80 bytes per row, whatever ncols is.  Synchronous. */
typedef struct pbl_stats_unique_out {
  void* values;
  int64_t* first;
  int64_t* counts;
  int64_t* nan_rows;
  void* nan_bits;
  int64_t* inverse;
  int64_t nunique, nnan; /* out */
} pbl_stats_unique_out;
PBL_API int pbl_stats_unique(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                             int32_t equal_nan, pbl_stats_unique_out* outs, void* stream);
/* values_dev[i] = table[values_dev[i]] for n device int64 (an index outside [0, m) is left as it is); table is a
 * host array of m entries.  Maps the inverse of category indices to the merged categories.  Synchronous. */
PBL_API int pbl_stats_remap(int64_t* values_dev, int64_t n, const int64_t* table, int64_t m, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PROBABILIT_B200_H */
