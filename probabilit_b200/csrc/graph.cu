// Fused evaluation of a probabilit modeling graph: ONE kernel evaluates every node of the graph
// for each sample instead of one NumPy temporary (n doubles through DRAM) per node.
//
// Replaces the per-node loop of Node.sample_from_quantiles (reference
// src/probabilit/modeling.py:586-612): Distribution._sample = scipy.stats ppf (:795-812),
// Constant._sample (:760-763), Transform._sample (:954-956, :986-990, :1007-1009, :1071-1072) and
// the per-node finite check (:600-606).  The host mirror (probabilit_b200/modeling.py) compiles
// the graph, in the reference's evaluation order, into the bytecode of include/probabilit_b200.h.
//
// Execution model: one thread per sample; node values live in shared-memory "slots"
// ([slot][thread], conflict-free), the program is staged in shared memory and decoded uniformly
// by the whole block (no divergence except inside the iterative inverse CDFs).  HBM traffic is
// 8 B per quantile column read + 8 B per retained node written; with PBL_OP_UNIFORM the quantiles
// are generated in-kernel and only retained nodes touch HBM.  A program with more live values than slots keeps the
// rest in spill slots (PBL_OP_SPILL / PBL_OP_FILL): per-thread scratch in global memory that stays in L2, because
// such a program runs on the resident grid only.
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/probabilit_b200.h"
#include "common.cuh"
#include "philox.cuh"
#include "quantile.cuh"
#include "special.cuh"

namespace pbl {
namespace {


__device__ __forceinline__ double rn_scale_loc(double v, double scale, double loc) {
  return __dadd_rn(__dmul_rn(v, scale), loc);  // `_ppf(q) * scale + loc` as two NumPy ufuncs (no FMA)
}

// scipy rv_continuous.ppf wrapper (scipy/stats/_distn_infrastructure.py:2305-2348); `core` is
// only evaluated for valid parameters and 0 < q < 1
template <typename F>
__device__ __forceinline__ double ppf_continuous(double q, bool args_ok, double a, double b, double loc,
                                                 double scale, F core) {
  const bool cond0 = args_ok && (scale > 0.0) && (loc == loc);
  if (!cond0) return PBL_NAN;
  if (q == 0.0) return rn_scale_loc(a, scale, loc);
  if (q == 1.0) return rn_scale_loc(b, scale, loc);
  if (q > 0.0 && q < 1.0) return rn_scale_loc(core(), scale, loc);
  return PBL_NAN;
}

// scipy rv_discrete.ppf wrapper (:3745-3792): q == 0 -> a - 1 + loc even for invalid parameters
template <typename F>
__device__ __forceinline__ double ppf_discrete(double q, bool args_ok, double a, double b, double loc, F core) {
  const bool cond0 = args_ok && (loc == loc);
  if (q == 0.0) return __dadd_rn(a - 1.0, loc);
  if (!cond0) return PBL_NAN;
  if (q == 1.0) return __dadd_rn(b, loc);
  if (q > 0.0 && q < 1.0) return __dadd_rn(core(), loc);
  return PBL_NAN;
}

__device__ __forceinline__ double triang_core(double q, double c) {
  // scipy/stats/_continuous_distns.py:10126  where(q < c, sqrt(c*q), 1 - sqrt((1-c)*(1-q)))
  if (q < c) return __dsqrt_rn(__dmul_rn(c, q));
  return __dadd_rn(1.0, -__dsqrt_rn(__dmul_rn(__dadd_rn(1.0, -c), __dadd_rn(1.0, -q))));
}

__device__ __noinline__ double eval_ppf(int op, double q, double p0, double p1, double p2) {
  switch (op) {
    case PBL_PPF_NORM:
      return ppf_continuous(q, true, -kInf, kInf, p0, p1, [&] { return ndtri(q); });
    case PBL_PPF_UNIFORM:
      return ppf_continuous(q, true, 0.0, 1.0, p0, p1, [&] { return q; });
    case PBL_PPF_EXPON:
      return ppf_continuous(q, true, 0.0, kInf, p0, p1, [&] { return -log1p(-q); });
    case PBL_PPF_TRIANG:
      return ppf_continuous(q, p0 >= 0.0 && p0 <= 1.0, 0.0, 1.0, p1, p2, [&] { return triang_core(q, p0); });
    case PBL_PPF_GAMMA:
      return ppf_continuous(q, p0 > 0.0, 0.0, kInf, p1, p2, [&] { return igami(p0, q); });
    case PBL_PPF_LOGNORM:
      return ppf_continuous(q, p0 > 0.0, 0.0, kInf, p1, p2, [&] { return exp(__dmul_rn(p0, ndtri(q))); });
    case PBL_PPF_POISSON:
      return ppf_discrete(q, p0 >= 0.0, 0.0, kInf, p1, [&] { return poisson_ppf_core(q, p0); });
    case PBL_PPF_BINOM:
      return ppf_discrete(q, p0 >= 0.0 && p1 >= 0.0 && p1 <= 1.0 && p0 == rint(p0), 0.0, p0, p2,
                          [&] { return binom_ppf_core(q, p0, p1); });
    case PBL_PPF_BERNOULLI:
      return ppf_discrete(q, p0 >= 0.0 && p0 <= 1.0, 0.0, 1.0, p1, [&] { return binom_ppf_core(q, 1.0, p0); });
  }
  return PBL_NAN;
}

// four-parameter distributions: (a, b, loc, scale)
__device__ __noinline__ double eval_ppf4(int op, double q, double a, double b, double loc, double scale) {
  if (op == PBL_PPF_BETA)
    return ppf_continuous(q, a > 0.0 && b > 0.0, 0.0, 1.0, loc, scale, [&] { return ibeta_inv(a, b, q); });
  // truncnorm: support [a, b] in standard units, scipy argcheck a < b
  return ppf_continuous(q, a < b, a, b, loc, scale, [&] { return truncnorm_ppf_core(q, a, b); });
}

// ---- table-lookup distributions (reference modeling.py:825-927) ----
// np.interp(x, xp, fp) (numpy compiled_base.c arr_interp): clamp outside, exact knots return fp[j]
__device__ __noinline__ double table_interp(double x, const double* __restrict__ t, int m) {
  const double* xp = t;
  const double* fp = t + m;
  if (x != x) return x;
  if (x >= xp[m - 1]) return fp[m - 1];
  if (x < xp[0]) return fp[0];
  int lo = 0, hi = m - 1;  // xp[lo] <= x < xp[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (x >= xp[mid]) lo = mid; else hi = mid;
  }
  if (xp[lo] == x) return fp[lo];
  const double slope = __ddiv_rn(__dsub_rn(fp[lo + 1], fp[lo]), __dsub_rn(xp[lo + 1], xp[lo]));
  double r = __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xp[lo])), fp[lo]);
  if (r != r) {
    r = __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xp[lo + 1])), fp[lo + 1]);
    if (r != r && fp[lo] == fp[lo + 1]) r = fp[lo];
  }
  return r;
}
// np.searchsorted(cum, q, side="right"): the first index with cum[idx] > q
__device__ __noinline__ double table_search_right(double q, const double* __restrict__ cum, int m) {
  int lo = 0, hi = m;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (cum[mid] <= q) lo = mid + 1; else hi = mid;
  }
  return (double)lo;
}
// np.quantile(data, q, method=...) on sorted data (numpy/lib/_function_base_impl.py _quantile, _lerp)
__device__ __noinline__ double table_quantile(double q, const double* __restrict__ a, int m, int method) {
  if (q != q) return q;
  const QuantilePick p = quantile_pick(q, (double)m, method);
  if (!quantile_interpolates(method)) return a[(int)p.lo];
  const double lo = a[(int)p.lo], hi = a[(int)p.hi];
  return quantile_lerp(lo, hi, __dsub_rn(hi, lo), p.gamma);
}

// numpy npy_divmod for doubles (numpy/_core/src/npymath/npy_math_internal.h.src)
__device__ __forceinline__ double np_divmod(double a, double b, double* modulus) {
  double mod = fmod(a, b);
  if (b == 0.0) {
    *modulus = mod;
    return a / b;
  }
  double div = (a - mod) / b;
  if (mod != 0.0) {
    if ((b < 0.0) != (mod < 0.0)) {
      mod += b;
      div -= 1.0;
    }
  } else {
    mod = copysign(0.0, b);
  }
  double floordiv;
  if (div != 0.0) {
    floordiv = floor(div);
    if (div - floordiv > 0.5) floordiv += 1.0;
  } else {
    floordiv = copysign(0.0, a / b);
  }
  *modulus = mod;
  return floordiv;
}

__device__ __forceinline__ double b2d(bool b) { return b ? 1.0 : 0.0; }

// ---- int64 values (NumPy's int64 ufuncs, numpy/_core/src/umath/loops_arithmetic.dispatch.c.src): the slot holds
// the bit pattern.  Wrapping arithmetic goes through uint64, where overflow is defined.
__device__ __forceinline__ int64_t d2i(double v) { return __double_as_longlong(v); }
__device__ __forceinline__ double i2d(int64_t v) { return __longlong_as_double(v); }
__device__ __forceinline__ int64_t wrap_mul(int64_t a, int64_t b) { return (int64_t)((uint64_t)a * (uint64_t)b); }
__device__ __forceinline__ int64_t int_floordiv(int64_t a, int64_t b) {
  if (b == 0) return 0;     // NumPy: 0 (with a divide-by-zero warning)
  if (b == -1) return (int64_t)(0 - (uint64_t)a);  // INT64_MIN // -1 wraps to INT64_MIN
  const int64_t q = a / b;
  return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q;
}
__device__ __forceinline__ int64_t int_mod(int64_t a, int64_t b) {
  if (b == 0 || b == -1) return 0;  // (INT64_MIN % -1 is undefined in C)
  const int64_t m = a % b;
  return (m != 0 && ((m < 0) != (b < 0))) ? m + b : m;  // the sign of the divisor
}
__device__ __forceinline__ int64_t int_pow(int64_t a, int64_t e) {  // e < 0: 1 (the caller reports the domain)
  int64_t r = 1;
  for (; e > 0; e >>= 1) {
    if (e & 1) r = wrap_mul(r, a);
    a = wrap_mul(a, a);
  }
  return r;
}

__device__ __noinline__ double eval_binary(int op, double a, double b) {
  switch (op) {
    case PBL_OP_I_ADD: return i2d((int64_t)((uint64_t)d2i(a) + (uint64_t)d2i(b)));
    case PBL_OP_I_SUB: return i2d((int64_t)((uint64_t)d2i(a) - (uint64_t)d2i(b)));
    case PBL_OP_I_MUL: return i2d(wrap_mul(d2i(a), d2i(b)));
    case PBL_OP_I_FLOORDIV: return i2d(int_floordiv(d2i(a), d2i(b)));
    case PBL_OP_I_MOD: return i2d(int_mod(d2i(a), d2i(b)));
    case PBL_OP_I_POW: return i2d(int_pow(d2i(a), d2i(b)));
    case PBL_OP_I_MAX: return i2d(max(d2i(a), d2i(b)));
    case PBL_OP_I_MIN: return i2d(min(d2i(a), d2i(b)));
    case PBL_OP_I_LT: return b2d(d2i(a) < d2i(b));
    case PBL_OP_I_LE: return b2d(d2i(a) <= d2i(b));
    case PBL_OP_I_EQ: return b2d(d2i(a) == d2i(b));
    case PBL_OP_I_NE: return b2d(d2i(a) != d2i(b));
    case PBL_OP_POW: return pow(a, b);
    case PBL_OP_FLOORDIV: {
      double m;
      return np_divmod(a, b, &m);
    }
    case PBL_OP_MOD: {
      double m;
      np_divmod(a, b, &m);
      return m;
    }
    case PBL_OP_MAX: return (a >= b || a != a) ? a : b;   // np.maximum propagates NaN
    case PBL_OP_MIN: return (a <= b || a != a) ? a : b;
    case PBL_OP_ATAN2: return atan2(a, b);
    case PBL_OP_LT: return b2d(a < b);
    case PBL_OP_LE: return b2d(a <= b);
    case PBL_OP_GT: return b2d(a > b);
    case PBL_OP_GE: return b2d(a >= b);
    case PBL_OP_EQ: return b2d(a == b);
    case PBL_OP_NE: return b2d(a != b);
    case PBL_OP_AND: return b2d(a != 0.0 && b != 0.0);
    case PBL_OP_OR: return b2d(a != 0.0 || b != 0.0);
    case PBL_OP_ISCLOSE: {  // np.isclose(a, b): rtol 1e-5, atol 1e-8, equal_nan False
      if (isfinite(a) && isfinite(b)) return b2d(fabs(a - b) <= __dadd_rn(1e-8, __dmul_rn(1e-5, fabs(b))));
      return b2d(a == b);
    }
  }
  return PBL_NAN;
}

__device__ __noinline__ double eval_unary(int op, double a) {
  switch (op) {
    case PBL_OP_LOG: return log(a);
    case PBL_OP_EXP: return exp(a);
    case PBL_OP_SIGN: return a > 0.0 ? 1.0 : (a < 0.0 ? -1.0 : (a == 0.0 ? 0.0 : a));
    case PBL_OP_LOG10: return log10(a);
    case PBL_OP_SIN: return sin(a);
    case PBL_OP_COS: return cos(a);
    case PBL_OP_TAN: return tan(a);
    case PBL_OP_ASIN: return asin(a);
    case PBL_OP_ACOS: return acos(a);
    case PBL_OP_ATAN: return atan(a);
    case PBL_OP_SINH: return sinh(a);
    case PBL_OP_COSH: return cosh(a);
    case PBL_OP_TANH: return tanh(a);
    case PBL_OP_ASINH: return asinh(a);
    case PBL_OP_ACOSH: return acosh(a);
    case PBL_OP_ATANH: return atanh(a);
    case PBL_OP_I_NEG: return i2d((int64_t)(0 - (uint64_t)d2i(a)));
    case PBL_OP_I_ABS: return i2d(d2i(a) < 0 ? (int64_t)(0 - (uint64_t)d2i(a)) : d2i(a));
    case PBL_OP_I_SIGN: return i2d((int64_t)(d2i(a) > 0) - (int64_t)(d2i(a) < 0));
    case PBL_OP_I_SQUARE: return i2d(wrap_mul(d2i(a), d2i(a)));
    case PBL_OP_I2F: return __ll2double_rn(d2i(a));
    case PBL_OP_F2I: return i2d(__double2ll_rz(a));
  }
  return PBL_NAN;
}

// ---- device form of a program -------------------------------------------------------------------------
// pbl_graph_eval_f64 translates the caller's pbl_graph_instr list (the ABI) into this 64-byte form (four
// 128-bit shared-memory loads per decoded instruction) and runs a liveness pass over it:
//   kAcc0 / kAcc1   operand 0 / 1 is the value the PREVIOUS instruction produced: it is taken from the
//                   accumulator registers instead of a shared-memory slot
//   kNoWrite        nothing reads the destination slot before it is overwritten (every consumer takes the
//                   value from the accumulator, or the node is only stored): the slot store is skipped
// so that chains like  ppf -> MUL -> ADD  (README "mutual fund": 20 of them) keep their values in registers.
constexpr int kAcc0 = 0x1000, kAcc1 = 0x2000, kNoWrite = 0x4000;
struct __align__(16) DevInstr {
  int32_t op;   // pbl_graph_op | PBL_GRAPH_* flags | kAcc0 | kAcc1 | kNoWrite
  int32_t dst;  // destination slot
  int32_t tag;  // node tag reported by CHECK
  int32_t out;  // output column written by STORE
  int32_t src[4];
  double imm[4];
};
static_assert(sizeof(DevInstr) == 64, "DevInstr is four 16-byte words");

struct GraphArgs {
  const DevInstr* program;
  int n_instr, n_slots;
  int program_in_smem;
  int64_t n;
  uint64_t row0;
  const double* const* inputs;
  double* const* outputs;
  int* first_nonfinite;
  const int32_t* row_inputs;  // indices into inputs[] of the columns that are read row by row (not tables)
  int n_row_inputs;
  double* spill;  // spill scratch (programs with PBL_OP_SPILL, launched on the resident grid), see spill_index
};

__device__ __forceinline__ double2 ld_stream_f64x2(const double* p) {
  double2 v;
  asm volatile("ld.global.cs.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
}

// Rows of a thread: R / 2 PAIRS of adjacent rows (2t, 2t + 1), the pairs 2 * kGraphBlock rows apart.  A pair
// shares one Philox block (philox.cuh: one block serves the row pair (g & ~1, g | 1)) and one 128-bit load /
// store per column when the column is 16-byte aligned there.
template <int R>
struct Rows {
  int64_t first[R / 2];  // row of the pair's first member (may be -1: the pair is aligned to the GLOBAL row parity)
  bool active[R];
};

template <int R>
__device__ __forceinline__ void load_rows(const double* __restrict__ col, const Rows<R>& rw, double (&v)[R], double dflt) {
#pragma unroll
  for (int p = 0; p < R / 2; ++p) {
    const double* a = col + rw.first[p];
    if (rw.active[2 * p] && rw.active[2 * p + 1] && (reinterpret_cast<uintptr_t>(a) & 15u) == 0) {
      const double2 t = ld_stream_f64x2(a);
      v[2 * p] = t.x;
      v[2 * p + 1] = t.y;
    } else {
      v[2 * p] = rw.active[2 * p] ? ld_stream_f64(a) : dflt;
      v[2 * p + 1] = rw.active[2 * p + 1] ? ld_stream_f64(a + 1) : dflt;
    }
  }
}
template <int R>
__device__ __forceinline__ void store_rows(double* __restrict__ col, const Rows<R>& rw, const double (&v)[R]) {
#pragma unroll
  for (int p = 0; p < R / 2; ++p) {
    double* a = col + rw.first[p];
    if (rw.active[2 * p] && rw.active[2 * p + 1] && (reinterpret_cast<uintptr_t>(a) & 15u) == 0) {
      __stcs(reinterpret_cast<double2*>(a), make_double2(v[2 * p], v[2 * p + 1]));
    } else {
      if (rw.active[2 * p]) __stcs(a, v[2 * p]);
      if (rw.active[2 * p + 1]) __stcs(a + 1, v[2 * p + 1]);
    }
  }
}
// the Philox uniforms of column c for the thread's rows: one block per pair (same values as philox_uniform_at)
template <int R>
__device__ __forceinline__ void uniform_rows(uint64_t seed, const uint64_t (&gpair)[R / 2], uint32_t c, double (&v)[R]) {
#pragma unroll
  for (int p = 0; p < R / 2; ++p) {
    const U4 ctr = {(uint32_t)gpair[p], (uint32_t)(gpair[p] >> 32), c, 0x50424C31u};
    const U4 o = philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
    v[2 * p] = u01_53(o.x, o.y);
    v[2 * p + 1] = u01_53(o.z, o.w);
  }
}

// ndtri for the R values of every lane of a warp.  Cephes ndtri has a cheap central branch (exp(-2) < q <
// 1 - exp(-2): 73 % of uniform quantiles; one rational function) and an expensive tail branch (two logs, a
// square root, three divisions, two polynomials: ~3x the fp64 work).  Evaluated per lane, every warp runs
// BOTH for each of its values (some lane always sits in the tail).  Here the central branch runs in place,
// and the tail arguments of the warp's 32 R values are COMPACTED through a shared-memory queue so that the
// tail code runs ceil(#tails / 32) times instead of R times (R = 4: 35 tails on average -> 1-2 rounds instead
// of 4).  Values are bit-identical to ndtri() (ndtri.cuh): same operations on the same operands.
// All 32 lanes must call it together; `queue` holds 32 * R doubles private to the warp.
// The Cephes coefficient tables live in CONSTANT memory here: fp64 instructions take a constant-bank operand
// directly, whereas a literal costs two UMOVs (a 64-bit immediate does not fit the instruction) -- in the ncu
// capture of the first version of this kernel 16 % of all executed instructions were UMOVs.
__constant__ double kNdP0[5] = {-5.99633501014107895267E1, 9.80010754185999661536E1, -5.66762857469070293439E1,
                                1.39312609387279679503E1, -1.23916583867381258016E0};
__constant__ double kNdQ0[8] = {1.95448858338141759834E0, 4.67627912898881538453E0,  8.63602421390890590575E1,
                                -2.25462687854119370527E2, 2.00260212380060660359E2, -8.20372256168333339912E1,
                                1.59056225126211695515E1, -1.18331621121330003142E0};
__constant__ double kNdP1[9] = {4.05544892305962419923E0,  3.15251094599893866154E1,  5.71628192246421288162E1,
                                4.40805073893200834700E1,  1.46849561928858024014E1,  2.18663306850790267539E0,
                                -1.40256079171354495875E-1, -3.50424626827848203418E-2, -8.57456785154685413611E-4};
__constant__ double kNdQ1[8] = {1.57799883256466749731E1,  4.53907635128879210584E1,  4.13172038254672030440E1,
                                1.50425385692907503408E1,  2.50464946208309415979E0,  -1.42182922854787788574E-1,
                                -3.80806407691578277194E-2, -9.33259480895457427372E-4};
__constant__ double kNdP2[9] = {3.23774891776946035970E0,  6.91522889068984211695E0,  3.93881025292474443415E0,
                                1.33303460815807542389E0,  2.01485389549179081538E-1, 1.23716634817820021358E-2,
                                3.01581553508235416007E-4, 2.65806974686737550832E-6, 6.23974539184983293730E-9};
__constant__ double kNdQ2[8] = {6.02427039364742014255E0,  3.67983563856160859403E0,  1.37702099489081330271E0,
                                2.16236993594496635890E-1, 1.34204006088543189037E-2, 3.28014464682127739104E-4,
                                2.89247864745380683936E-6, 6.79019408009981274425E-9};
template <int N>
__device__ __forceinline__ double ndc_polevl(double x, const double* c) {  // c: a __constant__ table
  double r = c[0];
#pragma unroll
  for (int i = 1; i < N; ++i) r = nd_add(nd_mul(r, x), c[i]);
  return r;
}
template <int N>
__device__ __forceinline__ double ndc_p1evl(double x, const double* c) {
  double r = nd_add(x, c[0]);
#pragma unroll
  for (int i = 1; i < N; ++i) r = nd_add(nd_mul(r, x), c[i]);
  return r;
}
__device__ __forceinline__ double ndtri_central(double y) {  // y = q - 0.5
  const double s2pi = 2.50662827463100050242E0;
  const double y2 = nd_mul(y, y);
  const double x = nd_add(y, nd_mul(y, __ddiv_rn(nd_mul(y2, ndc_polevl<5>(y2, kNdP0)), ndc_p1evl<8>(y2, kNdQ0))));
  return nd_mul(x, s2pi);
}
__device__ __noinline__ double ndtri_tail(double y) {  // 0 < y <= exp(-2); returns |ndtri|
  const double x = __dsqrt_rn(nd_mul(-2.0, log(y)));
  const double x0 = nd_add(x, -__ddiv_rn(log(x), x));
  const double z = __ddiv_rn(1.0, x);
  double x1;
  if (x < 8.0)
    x1 = __ddiv_rn(nd_mul(z, ndc_polevl<9>(z, kNdP1)), ndc_p1evl<8>(z, kNdQ1));
  else
    x1 = __ddiv_rn(nd_mul(z, ndc_polevl<9>(z, kNdP2)), ndc_p1evl<8>(z, kNdQ2));
  return nd_add(x0, -x1);
}
template <int R>
__device__ __forceinline__ void ndtri_rows(const double (&q)[R], double (&x)[R], double* __restrict__ queue,
                                           const uint32_t lane) {
  const double expm2 = 0.13533528323661269189;
  const uint32_t lt = lanemask_lt();
  uint32_t tails = 0, negate = 0, total = 0;
  uint32_t idx[R];
#pragma unroll
  for (int j = 0; j < R; ++j) {
    const double y0 = q[j];
    bool tail = false;
    if (y0 == 0.0) {
      x[j] = -kInf;
    } else if (y0 == 1.0) {
      x[j] = kInf;
    } else if (!(y0 > 0.0 && y0 < 1.0)) {
      x[j] = PBL_NAN;
    } else {
      double y = y0;
      bool neg = true;
      if (y > nd_add(1.0, -expm2)) {
        y = nd_add(1.0, -y);
        neg = false;
      }
      if (y > expm2) {
        x[j] = ndtri_central(nd_add(y, -0.5));
      } else {
        tail = true;
        x[j] = y;
        negate |= (neg ? 1u : 0u) << j;
      }
    }
    const uint32_t bal = __ballot_sync(0xFFFFFFFFu, tail);
    idx[j] = total + __popc(bal & lt);
    total += __popc(bal);
    tails |= (tail ? 1u : 0u) << j;
  }
  if (total == 0) return;  // (warp-uniform)
#pragma unroll
  for (int j = 0; j < R; ++j)
    if ((tails >> j) & 1u) queue[idx[j]] = x[j];
  __syncwarp();
  for (uint32_t k = lane; k < total; k += 32) queue[k] = ndtri_tail(queue[k]);
  __syncwarp();
#pragma unroll
  for (int j = 0; j < R; ++j)
    if ((tails >> j) & 1u) {
      const double v = queue[idx[j]];
      x[j] = ((negate >> j) & 1u) ? -v : v;
    }
  __syncwarp();  // the queue is free for the next call
}

constexpr int kGraphBlockR = 128;  // threads per block of graph_eval_kernel (R rows each)

// Spill slots (PBL_OP_SPILL / PBL_OP_FILL): scratch [spill][R][gridDim.x * 128], row j of thread tid of block b at
// ((spill * R + j) * gridDim.x + b) * 128 + tid -- coalesced per warp, and every chunk of the grid-stride loop
// reuses the same positions (a thread finishes a chunk's program before it starts the next).  A thread reads back
// what it wrote in the same kernel, so neither the non-coherent path nor evict-first: .cg keeps the values in L2,
// and program order of the same thread needs no fence.  Out of line, so that the interpreter loop keeps its
// registers.
__device__ __forceinline__ size_t spill_index(int spill, int j, int R) {
  return (((size_t)spill * R + j) * gridDim.x + blockIdx.x) * kGraphBlockR + threadIdx.x;
}
__device__ __noinline__ double fill_value(const double* scratch, int spill, int j, int R) {
  double v;
  asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(scratch + spill_index(spill, j, R)) : "memory");
  return v;
}
__device__ __noinline__ void spill_value(double* scratch, int spill, int j, int R, double v) {
  asm volatile("st.global.cg.f64 [%0], %1;" ::"l"(scratch + spill_index(spill, j, R)), "d"(v) : "memory");
}

template <int R>
__global__ void __launch_bounds__(kGraphBlockR, 4) graph_eval_kernel(const GraphArgs g) {
  constexpr int TB = kGraphBlockR;
  extern __shared__ __align__(16) unsigned char gsm_raw[];
  double* slots = reinterpret_cast<double*>(gsm_raw);  // [n_slots + 1][R][TB]; the last "slot" is the tail queue
  const DevInstr* prog = g.program;
  if (g.program_in_smem) {
    DevInstr* sp = reinterpret_cast<DevInstr*>(slots + (size_t)(g.n_slots + 1) * R * TB);
    const int words = g.n_instr * (int)(sizeof(DevInstr) / 16);
    const uint4* src = reinterpret_cast<const uint4*>(g.program);
    uint4* dst = reinterpret_cast<uint4*>(sp);
    for (int i = threadIdx.x; i < words; i += TB) dst[i] = src[i];
    prog = sp;
    __syncthreads();
  }
  const int tid = threadIdx.x;
  const uint32_t lane = tid & 31u, warp = tid >> 5;
  double* S = slots + tid;
  double* queue = slots + (size_t)g.n_slots * R * TB + warp * (32 * R);
#define SLOT(i, j) S[((size_t)(i) * R + (j)) * TB]
  // rows are walked in r' = row + (row0 & 1), so that a thread's pairs are the generator's pairs
  const int par = (int)(g.row0 & 1u);
  const int64_t n_shift = g.n + par;
  const uint64_t g_even = g.row0 - (uint64_t)par;
  for (int64_t base = (int64_t)blockIdx.x * (TB * R); base < n_shift; base += (int64_t)gridDim.x * (TB * R)) {
    Rows<R> rw;
    uint64_t gpair[R / 2];
#pragma unroll
    for (int p = 0; p < R / 2; ++p) {
      const int64_t rp = base + (int64_t)p * (2 * TB) + 2 * tid;
      rw.first[p] = rp - par;
      rw.active[2 * p] = rw.first[p] >= 0 && rw.first[p] < g.n;
      rw.active[2 * p + 1] = rw.first[p] + 1 < g.n;
      gpair[p] = (g_even + (uint64_t)rp) >> 1;
    }
    // the quantile / sample columns of this chunk are asked for now (HBM -> L2): the loads are fused into the
    // instructions that consume them, one column at a time, and would each expose a full HBM round trip
    for (int i = 0; i < g.n_row_inputs; ++i) {
      const double* col = g.inputs[g.row_inputs[i]];
#pragma unroll
      for (int p = 0; p < R / 2; ++p)
        if (rw.active[2 * p + 1]) asm volatile("prefetch.global.L2 [%0];" ::"l"(col + rw.first[p] + 1));
    }
    double acc[R];
#pragma unroll
    for (int j = 0; j < R; ++j) acc[j] = 0.0;
    for (int pc = 0; pc < g.n_instr; ++pc) {
      const int4 head = *reinterpret_cast<const int4*>(&prog[pc]);
      const int4 srcs = *reinterpret_cast<const int4*>(&prog[pc].src[0]);
      int flags = head.x;
      const int op = head.x & 0xFF, dst = head.y;
      const int s0 = srcs.x, s1 = srcs.y;
      double r[R];
      if (op < 16) {
        if (op == PBL_OP_LOAD) {
          load_rows<R>(g.inputs[s0], rw, r, 0.5);
        } else if (op == PBL_OP_STORE) {
#pragma unroll
          for (int j = 0; j < R; ++j) r[j] = SLOT(s0, j);
          store_rows<R>(g.outputs[s1], rw, r);
          continue;
        } else if (op == PBL_OP_CHECK) {
#pragma unroll
          for (int j = 0; j < R; ++j)
            if (rw.active[j] && !isfinite(SLOT(s0, j))) atomicMin(g.first_nonfinite, s1);
          continue;
        } else if (op == PBL_OP_MOV) {
          const double imm0 = prog[pc].imm[0];
#pragma unroll
          for (int j = 0; j < R; ++j) r[j] = (flags & kAcc0) ? acc[j] : (s0 >= 0 ? SLOT(s0, j) : imm0);
        } else if (op == PBL_OP_UNIFORM) {
          uniform_rows<R>((uint64_t)__double_as_longlong(prog[pc].imm[0]), gpair, (uint32_t)s0, r);
        } else if (op == PBL_OP_FILL) {
#pragma unroll
          for (int j = 0; j < R; ++j) r[j] = fill_value(g.spill, s0, j, R);
        } else if (op == PBL_OP_SPILL) {
#pragma unroll
          for (int j = 0; j < R; ++j) spill_value(g.spill, s1, j, R, SLOT(s0, j));
          continue;
        } else {
          continue;
        }
      } else {
        double a[R];
        if (flags & kAcc0) {
#pragma unroll
          for (int j = 0; j < R; ++j) a[j] = acc[j];
        } else if (flags & PBL_GRAPH_Q_INPUT) {  // fused LOAD: the quantile comes straight from its column
          load_rows<R>(g.inputs[s0], rw, a, 0.5);
        } else if (flags & PBL_GRAPH_Q_UNIFORM) {  // fused UNIFORM: generated in-kernel
          uniform_rows<R>((uint64_t)__double_as_longlong(prog[pc].imm[0]), gpair, (uint32_t)s0, a);
        } else if (s0 >= 0) {
#pragma unroll
          for (int j = 0; j < R; ++j) a[j] = SLOT(s0, j);
        } else {
          const double imm0 = prog[pc].imm[0];
#pragma unroll
          for (int j = 0; j < R; ++j) a[j] = imm0;
        }
        if (op >= 64) {  // unary
          switch (op) {
#define PBL_UNARY(CASE, EXPR) \
  case CASE:                  \
    _Pragma("unroll") for (int j = 0; j < R; ++j) r[j] = (EXPR); \
    break;
            PBL_UNARY(PBL_OP_NEG, -a[j])
            PBL_UNARY(PBL_OP_ABS, fabs(a[j]))
            PBL_UNARY(PBL_OP_FLOOR, floor(a[j]))
            PBL_UNARY(PBL_OP_CEIL, ceil(a[j]))
            PBL_UNARY(PBL_OP_SQRT, __dsqrt_rn(a[j]))
            PBL_UNARY(PBL_OP_SQUARE, __dmul_rn(a[j], a[j]))
            PBL_UNARY(PBL_OP_NOT, b2d(a[j] == 0.0))
#undef PBL_UNARY
            case PBL_OP_LOOKUP: {
              const int m = (int)prog[pc].imm[1];
              const double* tab = g.inputs[s1];
#pragma unroll
              for (int j = 0; j < R; ++j) r[j] = (a[j] >= 0.0 && a[j] < (double)m) ? tab[(int)a[j]] : PBL_NAN;
              break;
            }
            default:
#pragma unroll
              for (int j = 0; j < R; ++j) r[j] = eval_unary(op, a[j]);
              break;
          }
        } else if (op >= 32) {  // binary
          double b[R];
          if (flags & kAcc1) {
#pragma unroll
            for (int j = 0; j < R; ++j) b[j] = acc[j];
          } else if (s1 >= 0) {
#pragma unroll
            for (int j = 0; j < R; ++j) b[j] = SLOT(s1, j);
          } else {
            const double imm1 = prog[pc].imm[1];
#pragma unroll
            for (int j = 0; j < R; ++j) b[j] = imm1;
          }
          switch (op) {
#define PBL_BINARY(CASE, EXPR) \
  case CASE:                   \
    _Pragma("unroll") for (int j = 0; j < R; ++j) r[j] = (EXPR); \
    break;
            PBL_BINARY(PBL_OP_ADD, __dadd_rn(a[j], b[j]))
            PBL_BINARY(PBL_OP_MUL, __dmul_rn(a[j], b[j]))
            PBL_BINARY(PBL_OP_SUB, __dsub_rn(a[j], b[j]))
            PBL_BINARY(PBL_OP_DIV, __ddiv_rn(a[j], b[j]))
            PBL_BINARY(PBL_OP_LT, b2d(a[j] < b[j]))
            PBL_BINARY(PBL_OP_GT, b2d(a[j] > b[j]))
#undef PBL_BINARY
            default:
              if (op == PBL_OP_I_POW && (flags & PBL_GRAPH_CHECK)) {  // an integer is finite: check the domain
#pragma unroll
                for (int j = 0; j < R; ++j)
                  if (rw.active[j] && d2i(b[j]) < 0) atomicMin(g.first_nonfinite, head.z);
                flags &= ~PBL_GRAPH_CHECK;
              }
#pragma unroll
              for (int j = 0; j < R; ++j) r[j] = eval_binary(op, a[j], b[j]);
              break;
          }
        } else if (op >= PBL_PPF_TABLE_INTERP && op <= PBL_PPF_TABLE_QUANTILE) {
          // table lookups: src[1] names a device table
          const double* tab = g.inputs[s1];
          const int m = (int)prog[pc].imm[1];
          const int method = (int)prog[pc].imm[2];
#pragma unroll
          for (int j = 0; j < R; ++j)
            r[j] = op == PBL_PPF_TABLE_INTERP ? table_interp(a[j], tab, m)
                   : (op == PBL_PPF_TABLE_SEARCH ? table_search_right(a[j], tab, m) : table_quantile(a[j], tab, m, method));
        } else {  // ppf: operand 0 = q, then up to three parameters (slots: one value per row)
          const int s2 = srcs.z, s3 = srcs.w;
          double p0[R], p1[R], p2[R];
          {
            const double i1 = prog[pc].imm[1], i2 = prog[pc].imm[2], i3 = prog[pc].imm[3];
#pragma unroll
            for (int j = 0; j < R; ++j) {
              p0[j] = (flags & kAcc1) ? acc[j] : (s1 >= 0 ? SLOT(s1, j) : i1);
              p1[j] = s2 >= 0 ? SLOT(s2, j) : i2;
              p2[j] = s3 >= 0 ? SLOT(s3, j) : i3;
            }
          }
          if (op == PBL_PPF_NORM) {  // the common case: inline, tails compacted across the warp
            double x[R];
            ndtri_rows<R>(a, x, queue, lane);
#pragma unroll
            for (int j = 0; j < R; ++j) {
              // scipy's wrapper: nan unless scale > 0 and loc is a number; q = 0 / 1 / outside [0, 1] give
              // -inf / inf / nan through ndtri itself, scaled like any other value
              const bool cond0 = (p1[j] > 0.0) && (p0[j] == p0[j]);
              r[j] = cond0 ? rn_scale_loc(x[j], p1[j], p0[j]) : PBL_NAN;
            }
          } else if (op >= PBL_PPF_BETA) {  // (q, a, b, scale); the host adds loc with a separate ADD
#pragma unroll
            for (int j = 0; j < R; ++j) r[j] = eval_ppf4(op, a[j], p0[j], p1[j], 0.0, p2[j]);
          } else {
#pragma unroll
            for (int j = 0; j < R; ++j) r[j] = eval_ppf(op, a[j], p0[j], p1[j], p2[j]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < R; ++j) acc[j] = r[j];
      if (!(flags & kNoWrite)) {
#pragma unroll
        for (int j = 0; j < R; ++j) SLOT(dst, j) = r[j];
      }
      if (flags & PBL_GRAPH_CHECK) {
#pragma unroll
        for (int j = 0; j < R; ++j)
          if (rw.active[j] && !isfinite(r[j])) atomicMin(g.first_nonfinite, head.z);
      }
      if (flags & PBL_GRAPH_STORE) store_rows<R>(g.outputs[head.w], rw, r);
    }
  }
#undef SLOT
}

__global__ void __launch_bounds__(256) ppf_kernel(int what, const double* __restrict__ q, int64_t n, double p0,
                                                  double p1, double p2, double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256)
    out[i] = what >= PBL_PPF_BETA ? eval_ppf4(what, q[i], p0, p1, 0.0, p2) : eval_ppf(what, q[i], p0, p1, p2);
}

}  // namespace
}  // namespace pbl

namespace pbl {
// Caller's program -> device form.  Operands are assumed validated.  Three host passes:
//  (1) SINK the quantile-fed inverse CDFs (fused LOAD / UNIFORM, immediate parameters) down to just before
//      their first consumer.  The host mirror emits nodes in the reference's topological order, which puts
//      every distribution first (20 live values for the README mutual-fund graph); a value that is produced
//      right before it is consumed travels in the accumulator and needs no slot.  Legal: such an instruction
//      reads no slot, its destination slot is reserved for it from its original position to its last reader,
//      and CHECK / STORE are order-independent (smallest failing tag; one column per node).
//      SPILL / FILL stay in place: they read / write their slot like any other instruction.
//  (2) accumulator chaining + dead slot stores (kAcc0 / kAcc1 / kNoWrite).
//  (3) slots that are never materialised any more are dropped and the rest renumbered: fewer live values
//      per sample = less shared memory per block = more rows per thread / more resident warps.
// Returns the number of slots the device form needs.
static int translate_program(const pbl_graph_instr* program, int n_instr, std::vector<DevInstr>& out) {
  // slots an instruction READS, by operand position (-1: not a slot)
  auto slot_reads = [](const DevInstr& in, int (&r)[4]) {
    r[0] = r[1] = r[2] = r[3] = -1;
    const int op = in.op & 0xFF;
    const bool fused_q = (in.op & (PBL_GRAPH_Q_INPUT | PBL_GRAPH_Q_UNIFORM)) != 0;
    if (op == PBL_OP_STORE || op == PBL_OP_CHECK || op == PBL_OP_MOV || op == PBL_OP_SPILL) {
      r[0] = in.src[0];
    } else if (op >= 64) {
      r[0] = in.src[0];
    } else if (op >= 32) {
      r[0] = in.src[0];
      r[1] = in.src[1];
    } else if (op >= 16) {
      if (!fused_q) r[0] = in.src[0];
      if (!(op >= PBL_PPF_TABLE_INTERP && op <= PBL_PPF_TABLE_QUANTILE)) {
        r[1] = in.src[1];
        r[2] = in.src[2];
        r[3] = in.src[3];
      }
    }
    for (int i = 0; i < 4; ++i)
      if (r[i] < 0) r[i] = -1;
  };
  auto slot_written = [](const DevInstr& in) {
    const int op = in.op & 0xFF;
    return (op >= 16 || op == PBL_OP_MOV || op == PBL_OP_LOAD || op == PBL_OP_UNIFORM || op == PBL_OP_FILL) ? in.dst
                                                                                                          : -1;
  };
  std::vector<DevInstr> prog((size_t)n_instr);
  for (int i = 0; i < n_instr; ++i) {
    const pbl_graph_instr& in = program[i];
    DevInstr& d = prog[(size_t)i];
    d.op = in.op & 0xFFF;
    d.dst = in.dst & 0xFF;
    d.tag = (in.dst >> 8) & 0xFFF;
    d.out = (int32_t)((uint32_t)in.dst >> 20);
    for (int j = 0; j < 4; ++j) {
      d.src[j] = in.src[j];
      d.imm[j] = in.imm[j];
    }
  }
  // (1)
  out.clear();
  out.reserve((size_t)n_instr);
  {
    std::map<int, DevInstr> pending;  // destination slot -> held-back producer
    auto flush = [&](int slot) {
      auto it = pending.find(slot);
      if (it != pending.end()) {
        out.push_back(it->second);
        pending.erase(it);
      }
    };
    for (const DevInstr& in : prog) {
      int r[4];
      slot_reads(in, r);
      for (int j = 0; j < 4; ++j)
        if (r[j] >= 0) flush(r[j]);
      const int w = slot_written(in);
      if (w >= 0) flush(w);  // (a held-back value nobody read: keep the original write order on the slot)
      const int op = in.op & 0xFF;
      const bool sinkable = op >= 16 && op < 32 && (in.op & (PBL_GRAPH_Q_INPUT | PBL_GRAPH_Q_UNIFORM)) &&
                            r[1] < 0 && r[2] < 0 && r[3] < 0 &&
                            !(op >= PBL_PPF_TABLE_INTERP && op <= PBL_PPF_TABLE_QUANTILE);
      if (sinkable)
        pending[w] = in;
      else
        out.push_back(in);
    }
    while (!pending.empty()) flush(pending.begin()->first);
  }
  // (2)
  for (int i = 0; i < n_instr; ++i) {
    const int w = slot_written(out[(size_t)i]);
    if (w < 0) continue;
    if (i + 1 < n_instr) {  // the next instruction takes the value from the accumulator
      DevInstr& nx = out[(size_t)i + 1];
      const int nop = nx.op & 0xFF;
      int r[4];
      slot_reads(nx, r);
      if (nop >= 16 || nop == PBL_OP_MOV) {
        if (r[0] == w) nx.op |= kAcc0;
        if (r[1] == w && nop < 64) nx.op |= kAcc1;
      }
    }
    bool needed = false;  // does anything read the SLOT before it is overwritten?
    for (int k = i + 1; k < n_instr && !needed; ++k) {
      int r[4];
      slot_reads(out[(size_t)k], r);
      for (int j = 0; j < 4; ++j) {
        const bool via_acc =
            k == i + 1 && ((j == 0 && (out[(size_t)k].op & kAcc0)) || (j == 1 && (out[(size_t)k].op & kAcc1)));
        if (r[j] == w && !via_acc) needed = true;
      }
      if (slot_written(out[(size_t)k]) == w) break;
    }
    if (!needed) out[(size_t)i].op |= kNoWrite;
  }
  // (3) linear-scan reallocation of the values that still live in a slot
  std::vector<int> last_use((size_t)n_instr, -1);  // per defining instruction: its last slot reader
  {
    int def_of[256];
    for (int& x : def_of) x = -1;
    for (int k = 0; k < n_instr; ++k) {
      const DevInstr& in = out[(size_t)k];
      int r[4];
      slot_reads(in, r);
      for (int j = 0; j < 4; ++j) {
        const bool via_acc = (j == 0 && (in.op & kAcc0)) || (j == 1 && (in.op & kAcc1));
        if (r[j] >= 0 && !via_acc && def_of[r[j]] >= 0) last_use[(size_t)def_of[r[j]]] = k;
      }
      const int w = slot_written(in);
      if (w >= 0) def_of[w] = (in.op & kNoWrite) ? -1 : k;
    }
  }
  int n_used = 0;
  {
    int cur[256], def_of[256];  // original slot -> physical slot / defining instruction of its live value
    for (int i = 0; i < 256; ++i) cur[i] = def_of[i] = -1;
    std::vector<int> free_list;
    for (int k = 0; k < n_instr; ++k) {
      DevInstr& in = out[(size_t)k];
      int r[4];
      slot_reads(in, r);
      int released[4], n_released = 0;
      for (int j = 0; j < 4; ++j) {
        if (r[j] < 0) continue;
        const bool via_acc = (j == 0 && (in.op & kAcc0)) || (j == 1 && (in.op & kAcc1));
        if (via_acc || cur[r[j]] < 0) {  // (an accumulator operand names no slot any more)
          in.src[j] = 0;
          continue;
        }
        in.src[j] = cur[r[j]];
        if (def_of[r[j]] >= 0 && last_use[(size_t)def_of[r[j]]] == k) {
          bool seen = false;
          for (int q = 0; q < n_released; ++q) seen = seen || released[q] == r[j];
          if (!seen) released[n_released++] = r[j];
        }
      }
      for (int q = 0; q < n_released; ++q) {  // operands are read before the result is written: reusable now
        free_list.push_back(cur[released[q]]);
        cur[released[q]] = def_of[released[q]] = -1;
      }
      const int w = slot_written(in);
      if (w >= 0) {
        if (in.op & kNoWrite) {
          in.dst = 0;
          if (cur[w] >= 0) {  // nothing reads the old value of this slot any more either
            free_list.push_back(cur[w]);
            cur[w] = def_of[w] = -1;
          }
        } else {
          int phys;
          if (!free_list.empty()) {
            phys = free_list.back();
            free_list.pop_back();
          } else {
            phys = n_used++;
          }
          // (a live value of the same original slot that is overwritten without having been read again)
          if (cur[w] >= 0) free_list.push_back(cur[w]);
          cur[w] = phys;
          def_of[w] = k;
          in.dst = phys;
        }
      }
    }
  }
  return std::max(n_used, 1);
}
}  // namespace pbl

using pbl::kBadShape;
using pbl::kOk;

extern "C" {

int pbl_graph_eval_f64(const pbl_graph_instr* program, int32_t n_instr, int32_t n_slots, int64_t n, uint64_t row0,
                       const double* const* inputs_dev, int32_t n_inputs, double* const* outputs_dev,
                       int32_t n_outputs, int32_t* first_nonfinite, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (first_nonfinite) *first_nonfinite = -1;
  if (!program || n_instr < 0 || n_instr > PBL_GRAPH_MAX_INSTR || n_slots < 0 || n_slots > PBL_GRAPH_MAX_SLOTS ||
      n < 0 || n_inputs < 0 || n_outputs < 0) {
    pbl::set_last_error("pbl_graph_eval_f64: bad arguments (program size / slot count out of range)");
    return kBadShape;
  }
  int n_spills = 0;
  for (int i = 0; i < n_instr; ++i) {  // validate every operand before it reaches the device
    const pbl_graph_instr& in = program[i];
    const int op = in.op & 0xFF;
    bool ok = (in.dst & 0xFF) < std::max(n_slots, 1) && in.dst >= 0;
    const bool fused_q = (in.op & (PBL_GRAPH_Q_INPUT | PBL_GRAPH_Q_UNIFORM)) != 0;
    const int nsrc = op == PBL_OP_STORE || op == PBL_OP_CHECK || op == PBL_OP_LOAD || op == PBL_OP_UNIFORM ||
                     op == PBL_OP_SPILL || op == PBL_OP_FILL ? 0 : 4;
    const bool table_op = (op >= PBL_PPF_TABLE_INTERP && op <= PBL_PPF_TABLE_QUANTILE) || op == PBL_OP_LOOKUP;
    for (int s = fused_q ? 1 : 0; s < nsrc; ++s) ok = ok && (in.src[s] < n_slots || (table_op && s == 1));
    if (table_op) ok = ok && in.src[1] >= 0 && in.src[1] < n_inputs && in.imm[1] >= 1.0 && in.imm[1] < 2147483647.0;
    if (op == PBL_OP_LOAD || (in.op & PBL_GRAPH_Q_INPUT)) ok = ok && in.src[0] >= 0 && in.src[0] < n_inputs;
    if (fused_q) ok = ok && op >= PBL_PPF_NORM && op <= PBL_PPF_TRUNCNORM && in.src[0] >= 0;
    if (in.op & PBL_GRAPH_STORE) ok = ok && (int)((uint32_t)in.dst >> 20) < n_outputs && (op >= 16 || op == PBL_OP_MOV);
    const bool int_result = (op >= PBL_OP_I_ADD && op <= PBL_OP_I_MIN) || (op >= PBL_OP_I_NEG && op <= PBL_OP_I_SQUARE) ||
                            op == PBL_OP_F2I;
    if (in.op & PBL_GRAPH_CHECK) ok = ok && op >= 16 && (!int_result || op == PBL_OP_I_POW);
    if (op == PBL_OP_STORE) ok = ok && in.src[0] >= 0 && in.src[0] < n_slots && in.src[1] >= 0 && in.src[1] < n_outputs;
    if (op == PBL_OP_CHECK) ok = ok && in.src[0] >= 0 && in.src[0] < n_slots && in.src[1] >= 0;
    if (op == PBL_OP_SPILL || op == PBL_OP_FILL) {
      const int spill_idx = op == PBL_OP_SPILL ? in.src[1] : in.src[0];
      ok = ok && (in.op & ~0xFF) == 0 && spill_idx >= 0 && spill_idx < PBL_GRAPH_MAX_SPILLS;
      if (op == PBL_OP_SPILL) ok = ok && in.src[0] >= 0 && in.src[0] < n_slots;
      n_spills = std::max(n_spills, spill_idx + 1);
    }
    if (!ok) {
      pbl::set_last_error("pbl_graph_eval_f64: instruction " + std::to_string(i) + " has an operand out of range");
      return kBadShape;
    }
  }
  if (n == 0 || n_instr == 0) return kOk;

  std::vector<pbl::DevInstr> dev_prog;
  n_slots = pbl::translate_program(program, n_instr, dev_prog);  // (the device form may need fewer)

  // rows per thread and shared memory: (n_slots + 1 queue) x R x 128 doubles + the program.  R = 4 while a
  // block stays below 64 KB (>= 3 blocks / 12 warps per SM), else R = 2; a program that does not fit beside
  // the slots is decoded from global memory (uniform loads, L1-resident).
  const size_t prog_bytes = (size_t)n_instr * sizeof(pbl::DevInstr);
  const size_t slot_bytes2 = (size_t)(n_slots + 1) * 2 * pbl::kGraphBlockR * 8;
  int R = (2 * slot_bytes2 + prog_bytes <= 64 * 1024) ? 4 : 2;
  if (const char* e = getenv("PBL_GRAPH_ROWS")) R = atoi(e) == 2 ? 2 : (atoi(e) == 4 && 2 * slot_bytes2 <= 200 * 1024 ? 4 : R);
  const size_t slot_bytes = slot_bytes2 * (size_t)(R / 2);
  const size_t kSmemCap = 227 * 1024;
  // (PBL_GRAPH_PROGRAM=global forces the decode-from-global path, for the parity tests)
  const char* prog_env = getenv("PBL_GRAPH_PROGRAM");
  const int prog_in_smem = (slot_bytes + prog_bytes <= kSmemCap && !(prog_env && prog_env[0] == 'g')) ? 1 : 0;
  const size_t smem = slot_bytes + (prog_in_smem ? prog_bytes : 0);
  if (smem > kSmemCap) {
    pbl::set_last_error("pbl_graph_eval_f64: " + std::to_string(n_slots) + " live values per sample do not fit the kernel's shared memory");
    return kBadShape;
  }

  // input columns that are read row by row (LOAD / fused quantile loads), for the kernel's L2 prefetch
  std::vector<int32_t> row_inputs;
  {
    std::vector<char> seen((size_t)std::max(n_inputs, 1), 0);
    for (const pbl::DevInstr& d : dev_prog)
      if ((d.op & 0xFF) == PBL_OP_LOAD || (d.op & PBL_GRAPH_Q_INPUT))
        if (!seen[(size_t)d.src[0]]) {
          seen[(size_t)d.src[0]] = 1;
          row_inputs.push_back(d.src[0]);
        }
  }
  // one staging buffer (cached, grown on demand): [flag | program | input pointers | output pointers | row inputs]
  const size_t off_prog = 64, off_in = off_prog + prog_bytes, off_out = off_in + (size_t)n_inputs * 8;
  const size_t off_rows = off_out + (size_t)n_outputs * 8;
  const size_t total = off_rows + row_inputs.size() * 4 + 16;
  std::vector<unsigned char> host(total, 0);
  *reinterpret_cast<int*>(host.data()) = 0x7FFFFFFF;
  memcpy(host.data() + off_prog, dev_prog.data(), prog_bytes);
  if (n_inputs) memcpy(host.data() + off_in, inputs_dev, (size_t)n_inputs * 8);
  if (n_outputs) memcpy(host.data() + off_out, outputs_dev, (size_t)n_outputs * 8);
  if (!row_inputs.empty()) memcpy(host.data() + off_rows, row_inputs.data(), row_inputs.size() * 4);
  static std::mutex mu;
  static std::map<int, std::pair<unsigned char*, size_t>> staging;  // per device
  static std::map<int, int> attr_set;  // per device: bit 0 = R 2, bit 1 = R 4 (the attribute is per context)
  static std::map<int, std::pair<double*, size_t>> spill_scratch;  // per device, cached like the staging buffer
  std::lock_guard<std::mutex> lock(mu);
  int device = 0;
  PBL_CUDA_CHECK(cudaGetDevice(&device));
  auto& slot = staging[device];
  if (slot.second < total) {
    if (slot.first) cudaFree(slot.first);
    slot = {nullptr, 0};
    const size_t cap = std::max<size_t>(total * 2, 64 * 1024);
    PBL_CUDA_CHECK(cudaMalloc((void**)&slot.first, cap));
    slot.second = cap;
  }
  unsigned char* dev = slot.first;
  PBL_CUDA_CHECK(cudaMemcpyAsync(dev, host.data(), total, cudaMemcpyHostToDevice, stream));
  pbl::GraphArgs a;
  a.program = reinterpret_cast<const pbl::DevInstr*>(dev + off_prog);
  a.n_instr = n_instr;
  a.n_slots = n_slots;
  a.program_in_smem = prog_in_smem;
  a.n = n;
  a.row0 = row0;
  a.inputs = reinterpret_cast<const double* const*>(dev + off_in);
  a.outputs = reinterpret_cast<double* const*>(dev + off_out);
  a.first_nonfinite = reinterpret_cast<int*>(dev);
  a.row_inputs = reinterpret_cast<const int32_t*>(dev + off_rows);
  a.n_row_inputs = (int)row_inputs.size();
  const int attr_bit = R == 4 ? 2 : 1;
  if (!(attr_set[device] & attr_bit)) {
    if (R == 4)
      PBL_CUDA_CHECK(cudaFuncSetAttribute(pbl::graph_eval_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap));
    else
      PBL_CUDA_CHECK(cudaFuncSetAttribute(pbl::graph_eval_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap));
    attr_set[device] |= attr_bit;
  }
  const int64_t per_block = (int64_t)pbl::kGraphBlockR * R;
  const int64_t blocks_needed = (n + 1 + per_block - 1) / per_block;
  int64_t cap_blocks = (int64_t)pbl::num_sms() * 32;
  a.spill = nullptr;
  if (n_spills > 0) {
    // exactly the resident grid: the scratch ([spill][R][grid x 128] doubles) then does not grow with n, and the
    // grid-stride loop reuses it chunk after chunk
    int per_sm = 0;
    if (R == 4)
      PBL_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pbl::graph_eval_kernel<4>, pbl::kGraphBlockR, smem));
    else
      PBL_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pbl::graph_eval_kernel<2>, pbl::kGraphBlockR, smem));
    cap_blocks = (int64_t)pbl::num_sms() * std::max(per_sm, 1);
    const size_t bytes = (size_t)n_spills * R * (size_t)std::min(blocks_needed, cap_blocks) * pbl::kGraphBlockR * 8;
    auto& sc = spill_scratch[device];
    if (sc.second < bytes) {
      if (sc.first) cudaFree(sc.first);
      sc = {nullptr, 0};
      PBL_CUDA_CHECK(cudaMalloc((void**)&sc.first, bytes));
      sc.second = bytes;
    }
    a.spill = sc.first;
  }
  const unsigned grid = (unsigned)std::min(blocks_needed, cap_blocks);
  if (R == 4)
    pbl::graph_eval_kernel<4><<<grid, pbl::kGraphBlockR, smem, stream>>>(a);
  else
    pbl::graph_eval_kernel<2><<<grid, pbl::kGraphBlockR, smem, stream>>>(a);
  pbl::g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
  PBL_CUDA_CHECK(cudaGetLastError());
  int flag = 0x7FFFFFFF;
  PBL_CUDA_CHECK(cudaMemcpyAsync(&flag, dev, sizeof(int), cudaMemcpyDeviceToHost, stream));
  // synchronous by contract; the staging buffer may be reused by the next call once the stream has drained
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  if (first_nonfinite) *first_nonfinite = (flag == 0x7FFFFFFF) ? -1 : flag;
  return kOk;
}

// developer / test aid (host only, no GPU needed): the device form of a program as pbl_graph_instr records
// (reordered, slots renumbered; dst carries slot | tag << 8 | output << 20 like the ABI form) + its op words
// with the internal flags 0x1000 (operand 0 from the accumulator), 0x2000 (operand 1), 0x4000 (slot store
// skipped), + the slot count it needs.
__attribute__((visibility("default"))) int pbl_graph_debug_translate(const pbl_graph_instr* program, int32_t n_instr,
                                                                     pbl_graph_instr* prog_out, int32_t* op_out,
                                                                     int32_t* n_slots_out) {
  if (!program || !op_out || !prog_out || n_instr < 0) return kBadShape;
  std::vector<pbl::DevInstr> dev_prog;
  const int ns = pbl::translate_program(program, n_instr, dev_prog);
  for (int i = 0; i < n_instr; ++i) {
    const pbl::DevInstr& d = dev_prog[(size_t)i];
    op_out[i] = d.op;
    prog_out[i].op = d.op & 0xFFF;
    prog_out[i].dst = d.dst | (d.tag << 8) | (int32_t)((uint32_t)d.out << 20);
    for (int j = 0; j < 4; ++j) {
      prog_out[i].src[j] = d.src[j];
      prog_out[i].imm[j] = d.imm[j];
    }
  }
  if (n_slots_out) *n_slots_out = ns;
  return kOk;
}

int pbl_ppf_f64(int32_t what, const double* q_dev, int64_t n, double p0, double p1, double p2, double* out_dev,
                void* stream) {
  if (n < 0 || (n > 0 && (!q_dev || !out_dev)) || what < PBL_PPF_NORM || what > PBL_PPF_TRUNCNORM ||
      (what >= PBL_PPF_TABLE_INTERP && what <= PBL_PPF_TABLE_QUANTILE)) {
    pbl::set_last_error("pbl_ppf_f64: bad arguments");
    return kBadShape;
  }
  if (n == 0) return kOk;
  const int64_t blocks = std::min<int64_t>((n + 255) / 256, (int64_t)pbl::num_sms() * 32);
  pbl::ppf_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(what, q_dev, n, p0, p1, p2, out_dev);
  PBL_LAUNCH_CHECK();
  return kOk;
}

}  // extern "C"
