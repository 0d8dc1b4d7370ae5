// Iman-Conover on the device: plan object + stage entry points (internal C++ API; the C ABI
// in capi.cu is a thin wrapper).  Reference: src/probabilit/correlation.py:368-425.
#pragma once
#include <vector>

#include "common.cuh"
#include "sort.cuh"

namespace pbl {

struct IcPlan {
  int device = 0;
  int64_t n = 0;       // rows (observations)
  int k = 0;           // columns (variables)
  int col_batch = 0;   // columns sorted per launch batch (bounds the sort workspace)
  int window_bits = 32;  // sort window (sort.cuh); switches to 64 after a kRetry status
  bool has_target = false;
  bool rows_only = false;  // no sort workspace: Gram / solve / transform stages only (multi-GPU row shard)

  SortBuffers sort;            // sized for col_batch columns
  uint32_t sort_epoch = 0;     // tag of the last launch that used the look-back words (sort.cuh)
  double* sortedX = nullptr;   // [k][n]  np.sort(X[:,c])
  double* vdw = nullptr;       // [n] ndtri((p+1)/(n+1)): scores of an untied column, sorted order
  bool vdw_ready = false;
  double* scores = nullptr;    // [k][n]  van der Waerden scores, then (in place) correlated scores
  double* gram_partials = nullptr;
  int gram_row_blocks = 0;
  int gram_tg = 0;             // thread-grid edge of the Gram kernel (4, 8 or 16)
  double* gram = nullptr;      // [k][k] sum_r s_ri s_rj
  double* colsum = nullptr;    // [k]
  double* work = nullptr;      // [k][k] scratch: R, then Q (lower Cholesky factor)
  double* T = nullptr;         // [k][k] row-major, upper triangular: correlated = scores @ T
  double* P = nullptr;         // [k][k] row-major lower Cholesky factor of the target C
  double* moments = nullptr;   // Cholesky correlator: [k] mean, [k] std, [k][256] partial sums (lazy)
  cudaStream_t copy_stream = nullptr;   // host-buffer entry point: copies overlap the sorts
  std::vector<cudaEvent_t> events;
  void* permcorr = nullptr;    // PermutationCorrelator state (permcorr.cu), lazy
  uint32_t* flags = nullptr;   // [8], see SortFlag in sort.cuh
  // row-chunk hook (multi-GPU driver): the scatter by row that ends rank_scores / rank_gather is issued
  // chunk by chunk (chunk g = output rows [g * chunk_rows, (g+1) * chunk_rows), starting with chunk_first
  // and wrapping) and chunk_fn(column, g, user) is called on the host right after chunk g is enqueued
  int64_t chunk_rows = 0;
  int chunk_first = 0;
  void (*chunk_fn)(int32_t, int32_t, void*) = nullptr;
  void* chunk_user = nullptr;
  size_t bytes = 0;            // device bytes held by the plan
};

// flags bit 0: rows-only plan (see IcPlan::rows_only)
int ic_plan_create(int64_t n, int k, int col_batch, int flags, IcPlan** out);
void ic_plan_destroy(IcPlan* plan);
int ic_plan_set_target(IcPlan* plan, const double* P_lower_host);

// Full transform on device-resident data.  X and Y are (n, k) with the given element strides
// (F-order: row_stride 1, col_stride n).  Synchronises the stream before returning (the reference
// call is synchronous and the status has to come back).
int ic_plan_run(IcPlan* plan, const double* X, int64_t x_row_stride, int64_t x_col_stride,
                double* Y, int64_t y_row_stride, int64_t y_col_stride, cudaStream_t stream);

// Same with HOST buffers (column-major or C order), copies inside and overlapped with the sorts.
int ic_plan_run_host(IcPlan* plan, const double* X_host, int64_t x_row_stride, int64_t x_col_stride,
                     double* Y_host, int64_t y_row_stride, int64_t y_col_stride, double* dX, double* dY,
                     cudaStream_t stream);

// Stage-level entry points (parity tests, and the multi-GPU host driver which interleaves
// collectives between them).  All asynchronous on `stream`.
// ranks_only: leave scipy.stats.rankdata(X[:, c]) (average ranks) in plan->scores instead of the scores
int ic_stage_rank_scores(IcPlan* plan, const double* X, int64_t row_stride, int64_t col_stride,
                         int col0, int ncols, cudaStream_t stream, bool ranks_only = false);
int ic_stage_gram(IcPlan* plan, cudaStream_t stream);
int ic_stage_solve(IcPlan* plan, int64_t n_total, cudaStream_t stream);
int ic_stage_transform(IcPlan* plan, cudaStream_t stream);
int ic_stage_rank_gather(IcPlan* plan, double* Y, int64_t row_stride, int64_t col_stride,
                         int col0, int ncols, cudaStream_t stream);
int ic_read_status(IcPlan* plan, cudaStream_t stream);

int column_moments(IcPlan* plan, const double* X, int64_t xrs, int64_t xcs, const double* mean_dev,
                   double* out_dev, int mode, cudaStream_t stream);
int centre_columns(IcPlan* plan, const double* X, int64_t xrs, int64_t xcs, const double* mean_dev, double* S,
                   cudaStream_t stream);

// PermutationCorrelator (permcorr.cu; reference correlation.py:473-703, :757-921)
void permcorr_free(void* state);
int permcorr_begin(IcPlan* plan, const double* X, int64_t xrs, int64_t xcs, double* Y, int spearman,
                   const double* target_host, const double* weights_host, cudaStream_t stream);
int permcorr_steps(IcPlan* plan, double* Y, const int32_t* step_col, const int32_t* step_off,
                   const int32_t* step_cnt, const int64_t* swaps, int64_t n_swaps_total, int64_t n_steps,
                   double tol, int64_t* steps_done, int32_t* converged, double* errors_host,
                   int64_t errors_cap, int64_t* n_errors, cudaStream_t stream);
int permcorr_read_corr(IcPlan* plan, double* corr_host);

int corrcoef_run(IcPlan* plan, const double* X, int64_t xrs, int64_t xcs, int spearman, double* out_host,
                 cudaStream_t stream);

// (n, k) fp64 matrix from one strided layout to another on the device (non-overlapping buffers)
int copy_strided(const double* src, int64_t srs, int64_t scs, double* dst, int64_t drs, int64_t dcs, int64_t n, int k,
                 cudaStream_t stream);

// Cholesky correlator (reference correlation.py:205-285); synchronous like ic_plan_run.
int cholesky_correlator_run(IcPlan* plan, const double* X, int64_t x_row_stride, int64_t x_col_stride,
                            double* Y, int64_t y_row_stride, int64_t y_col_stride, cudaStream_t stream);

}  // namespace pbl
