// np.quantile's index arithmetic (numpy/lib/_function_base_impl.py: _QuantileMethods, _get_indexes, _get_gamma,
// _lerp), split into "which two order statistics and gamma" and "combine a[lo], a[hi]".  Shared by the
// EmpiricalDistribution lookup of the graph kernel (graph.cu, TABLE_QUANTILE) and the column quantiles of stats.cu,
// so that the two cannot drift apart.  Callers compile without FMA contraction (or use the _rn intrinsics, as here).
#pragma once
#include <cuda_runtime.h>

namespace pbl {

// method codes of PBL_PPF_TABLE_QUANTILE and pbl_stats_quantiles
enum QuantileMethod { kQLinear = 0, kQLower = 1, kQHigher = 2, kQNearest = 3, kQMidpoint = 4, kQClosest = 5 };

__host__ __device__ __forceinline__ bool quantile_interpolates(int method) {
  return method == kQLinear || method == kQMidpoint;
}

// The ranks (integral doubles in [0, m - 1]) of the order statistics that quantile q of m sorted values reads, and
// the interpolation weight.  Methods that do not interpolate give lo == hi.  q is not NaN.
struct QuantilePick {
  double lo, hi, gamma;
};
__device__ __forceinline__ QuantilePick quantile_pick(double q, double m, int method) {
  const double n1 = m - 1.0;
  const double vi = __dmul_rn(n1, q);  // (n - 1) * quantiles
  if (method == kQLower || method == kQHigher || method == kQNearest) {
    double idx = method == kQLower ? floor(vi) : (method == kQHigher ? ceil(vi) : rint(vi));
    if (idx < 0.0) idx = 0.0;
    if (idx > n1) idx = n1;
    return {idx, idx, 0.0};
  }
  if (method == kQClosest) {  // discontinuous, index from n*q - 1.5, ties to odd
    const double index = __dadd_rn(__dadd_rn(__dmul_rn(m, q), -1.0), -0.5);
    const double prev = floor(index);
    const double gamma = index - prev;
    double res = (gamma == 0.0 && fmod(prev, 2.0) == 1.0) ? prev : prev + 1.0;
    if (res < 0.0) res = 0.0;
    if (res > n1) res = n1;
    return {res, res, 0.0};
  }
  double index = vi;
  if (method == kQMidpoint) index = __dmul_rn(0.5, __dadd_rn(floor(vi), ceil(vi)));
  double prev = floor(index), next = prev + 1.0;
  if (index >= n1) prev = next = n1;  // _get_indexes: at / above the last element both are the last
  if (index < 0.0) prev = next = 0.0;
  double gamma = __dsub_rn(index, prev);
  if (method == kQMidpoint) gamma = (fmod(index, 1.0) == 0.0) ? 0.0 : 0.5;
  return {prev, next, gamma};
}

// _lerp(a, b, t): a + (b - a) * t, or b - (b - a) * (1 - t) where t >= 0.5.  `diff` is b - a in the data's own
// arithmetic (int64 data subtract in int64, wrapping, before the cast), lo / hi are a and b as doubles.
__device__ __forceinline__ double quantile_lerp(double lo, double hi, double diff, double gamma) {
  double r = __dadd_rn(lo, __dmul_rn(diff, gamma));
  if (gamma >= 0.5) r = __dsub_rn(hi, __dmul_rn(diff, __dsub_rn(1.0, gamma)));
  return r;
}

}  // namespace pbl
