// Column statistics of sampled nodes with NumPy's bits: np.mean / np.var / np.std and np.quantile / np.percentile
// of the columns a graph run leaves in HBM, without copying them to the host.
//
// Moments.  NumPy sums float64 with one pairwise tree (numpy/_core/src/umath/loops_utils.h.src, pairwise_sum): a
// node of m > 128 elements is pw(first n2) + pw(rest) with n2 = m/2 - (m/2) % 8, a leaf of 8..128 elements runs
// eight accumulators, fewer than 8 elements are added in order; the reduction adds that to its initial 0.0.  int64
// and bool means cast through the ufunc buffer: one such tree per chunk of `chunk` elements (np.getbufsize()), the
// chunk sums added in order.  The tree depends on n alone, so it is cut at the depth where every subtree fits one
// block's shared memory: a block stages its subtree (coalesced), sums the leaves in parallel and walks the subtree in
// NumPy's order; one block per column then adds the subtrees level by level (the top of the tree is perfect) and the
// chunks in order.  No floating-point atomics: the result does not depend on the grid.  var / std is a second pass
// over (x - mean)^2, the mean read from device memory.
//
// Quantiles.  MSD radix select of the order statistics that (n, q, method) needs, 8 bits per pass, at most 8
// passes, every pass one read of the column.  Values map to order-preserving u64 keys.  Targets that share a key
// prefix share one histogram (a "group"); a pass histograms the next digit of the keys of every group and keeps
// their min / max, so a target whose group holds a single distinct key ends there.  Prefix, remaining rank and
// groups advance on the device (no host round trip).  Scratch is O(columns x targets).
//
// Min / max and histograms (numpy/lib/_histograms_impl.py).  Min / max: one read of every column into
// order-preserving keys, NaNs set aside (the first NaN's row is kept: NumPy propagates it).  Histograms: one read of
// every column with its own edges and bin count.  The equal-bin path repeats NumPy's float64 index arithmetic
// (x - first) / denom * nbins and its two fix-ups against the edge table, so a value lands where NumPy puts it, not in
// "the mathematically right bin"; an index that leaves the table is reported with its row (NumPy raises there).  An
// edge array counts cells around its distinct values (below / equal to each, NaN apart), from which the host forms
// searchsorted's counts.  Counts are u32 in shared memory with warp-aggregated adds, flushed to u64 with integer
// atomics (the result does not depend on the grid); past kHistSmemCounts bins every add is a u64 global atomic.
// Compaction writes a[keep] in order (tile counts, a scan, an ordered scatter) for the estimators under a range.
#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/probabilit_b200.h"
#include "common.cuh"
#include "quantile.cuh"

namespace pbl {
namespace {

// ---------------------------------------------------------------------------------------------------------------
// moments
constexpr int kSumThreads = 256;
constexpr int kLeaf = 128;                 // numpy's PW_BLOCKSIZE
constexpr int64_t kSubtreeCap = 8192 + 32;  // doubles of one block's subtree (a whole 8192-element chunk fits)
constexpr int kMaxLeaves = 160;             // leaves of a subtree: each has >= 56 elements once the subtree has > 128
constexpr int kMaxDepth = 24;               // frames of a subtree walk (log2(kSubtreeCap / 56) + 1 would do)

struct SumArgs {
  const uint64_t* const* cols;
  const int32_t* kinds;
  int64_t n, chunk;
  const double* means;  // squares pass: the column means
  double* partials;     // [col][stride] subtree sums
  double* pingpong;     // [col][stride] scratch of the top levels
  int64_t stride;       // blocks per column (gridDim.x)
};

// The subtrees of an L-element tree cut at depth d differ from L / 2^d by at most 17 elements (a split moves at
// most 8.5 from the half), so this depth fits them in a block, and every node above it has > 128 elements.
__host__ __device__ __forceinline__ int cut_depth(int64_t L) {
  int d = 0;
  while ((L >> d) + 24 > kSubtreeCap) ++d;
  return d;
}
__host__ __device__ __forceinline__ int64_t seg_len(int kind, bool squares, int64_t n, int64_t chunk) {
  return (kind == PBL_STATS_F64 || squares) ? n : chunk;  // (the squares are float64 already: no cast, no chunks)
}
__host__ __device__ __forceinline__ int64_t min64(int64_t x, int64_t y) { return x < y ? x : y; }
__host__ __device__ __forceinline__ int64_t pw_split(int64_t m) {
  const int64_t h = m / 2;
  return h - h % 8;
}

__device__ __forceinline__ double value_f64(uint64_t bits, int kind) {
  if (kind == PBL_STATS_I64_BITS) return __ll2double_rn((long long)bits);
  return __longlong_as_double((long long)bits);  // doubles, and int64 / bool values held as exact doubles
}
__device__ __forceinline__ double load_value(const uint64_t* col, int kind, int64_t i) {
  return value_f64(ld_stream_u64(col + i), kind);
}

__device__ double leaf_sum(const double* a, int m) {
  if (m < 8) {
    double r = -0.0;
    for (int i = 0; i < m; ++i) r = __dadd_rn(r, a[i]);
    return r;
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i = 8;
  for (; i < m - m % 8; i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], a[i + j]);
  }
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < m; ++i) res = __dadd_rn(res, a[i]);
  return res;
}

// leaves (offset, length) of the pairwise tree of m elements, in order
__device__ int tree_leaves(int64_t m, int* off, int* len) {
  int64_t stack[kMaxDepth];
  int sp = 0, nl = 0;
  int64_t cur = m, at = 0;
  while (true) {
    while (cur > kLeaf) {
      const int64_t n2 = pw_split(cur);
      stack[sp++] = cur - n2;
      cur = n2;
    }
    off[nl] = (int)at;
    len[nl] = (int)cur;
    ++nl;
    at += cur;
    if (sp == 0) return nl;
    cur = stack[--sp];
  }
}

// the pairwise tree of m elements whose leaf sums are leafv[0..], added in NumPy's order
__device__ double tree_combine(int64_t m, const double* leafv) {
  int64_t right[kMaxDepth];
  double left[kMaxDepth];
  bool has_left[kMaxDepth];
  int sp = 0, li = 0;
  int64_t cur = m;
  while (true) {
    while (cur > kLeaf) {
      const int64_t n2 = pw_split(cur);
      right[sp] = cur - n2;
      has_left[sp] = false;
      ++sp;
      cur = n2;
    }
    double v = leafv[li++];
    while (sp > 0 && has_left[sp - 1]) {
      v = __dadd_rn(left[sp - 1], v);
      --sp;
    }
    if (sp == 0) return v;
    left[sp - 1] = v;
    has_left[sp - 1] = true;
    cur = right[sp - 1];
  }
}

// one block per subtree: blockIdx.x = segment << dmax | subtree, blockIdx.y = column
template <bool kSquares>
__global__ void __launch_bounds__(kSumThreads) pairwise_subtree_kernel(SumArgs a) {
  extern __shared__ double s_val[];
  __shared__ int s_off[kMaxLeaves], s_len[kMaxLeaves], s_nl;
  __shared__ double s_leaf[kMaxLeaves];
  const int col = blockIdx.y;
  const int kind = a.kinds[col];
  const int64_t L0 = seg_len(kind, kSquares, a.n, a.chunk);
  const int dmax = cut_depth(min64(L0, a.n));
  const int64_t seg = (int64_t)blockIdx.x >> dmax, local = (int64_t)blockIdx.x & ((1ll << dmax) - 1);
  const int64_t seg0 = seg * L0;
  if (seg0 >= a.n) return;
  const int64_t L = min64(L0, a.n - seg0);
  const int d = cut_depth(L);
  if (local >= (1ll << d)) return;
  int64_t off = 0, m = L;
  for (int k = d - 1; k >= 0; --k) {
    const int64_t n2 = pw_split(m);
    if ((local >> k) & 1) {
      off += n2;
      m -= n2;
    } else {
      m = n2;
    }
  }
  const uint64_t* col_ptr = a.cols[col];
  const double mean = kSquares ? a.means[col] : 0.0;
  for (int64_t i = threadIdx.x; i < m; i += kSumThreads) {
    double v = load_value(col_ptr, kind, seg0 + off + i);
    if (kSquares) {
      v = __dsub_rn(v, mean);  // x = float64(a) - mean, then x * x
      v = __dmul_rn(v, v);
    }
    s_val[i] = v;
  }
  if (threadIdx.x == 0) s_nl = tree_leaves(m, s_off, s_len);
  __syncthreads();
  for (int t = threadIdx.x; t < s_nl; t += kSumThreads) s_leaf[t] = leaf_sum(s_val + s_off[t], s_len[t]);
  __syncthreads();
  if (threadIdx.x == 0) a.partials[col * a.stride + blockIdx.x] = tree_combine(m, s_leaf);
}

// one block per column: the top levels of every segment's tree, the segments in order, then the statistic
__global__ void __launch_bounds__(1024) pairwise_finish_kernel(SumArgs a, bool squares, int what, double divisor,
                                                               double* means_out, double* out) {
  const int col = blockIdx.x;
  const int kind = a.kinds[col];
  const int64_t L0 = seg_len(kind, squares, a.n, a.chunk);
  const int dmax = cut_depth(min64(L0, a.n));
  const int64_t nseg = (a.n + L0 - 1) / L0;
  double* base = a.partials + col * a.stride;
  double* pp = a.pingpong + col * a.stride;
  double total = 0.0;  // the reduction's initial value
  for (int64_t seg = 0; seg < nseg; ++seg) {
    const int64_t L = min64(L0, a.n - seg * L0);
    const int d = cut_depth(L);
    double* src = base + (seg << dmax);
    if (d > 0) {  // perfect binary tree of 2^d subtree sums: level by level, left + right
      double* dst = pp + (seg << dmax);
      for (int64_t cnt = 1ll << (d - 1); cnt >= 1; cnt >>= 1) {
        for (int64_t i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = __dadd_rn(src[2 * i], src[2 * i + 1]);
        __syncthreads();
        double* t = src;
        src = dst;
        dst = t;
      }
    }
    if (threadIdx.x == 0) total = __dadd_rn(total, src[0]);
    if (d > 0) __syncthreads();  // (the next segment overwrites the ping-pong area)
  }
  if (threadIdx.x != 0) return;
  double r;
  if (!squares) {
    r = __ddiv_rn(total, (double)a.n);
    if (means_out) means_out[col] = r;
  } else {
    r = __ddiv_rn(total, divisor);
    if (what == PBL_STATS_STD) r = __dsqrt_rn(r);
  }
  if (what == PBL_STATS_MEAN || squares) out[col] = r;
}

// ---------------------------------------------------------------------------------------------------------------
// quantiles
constexpr int kSelThreads = 256;
constexpr int kDigitBits = 8, kBins = 1 << kDigitBits, kPasses = 64 / kDigitBits;
constexpr int kGroupsPerBlock = 32;  // histograms one pass block keeps in shared memory (32 KB)
constexpr uint64_t kSign = 0x8000000000000000ull;

struct Target {
  uint64_t prefix;  // key bits decided so far (8 per pass)
  uint64_t rank;    // rank among the keys that share the prefix
  uint64_t key;     // done: the key of the order statistic
  int32_t group, done;
};

struct SelArgs {
  const uint64_t* const* cols;
  const int32_t* kinds;
  int64_t n;
  int32_t ntargets;    // per column: 2 per q (lo, hi)
  const double* q;     // [nq]
  int32_t nq, method;
  Target* targets;     // [col][ntargets]
  uint64_t* gprefix;   // [col][ntargets] sorted distinct prefixes of the unresolved targets
  int32_t* first;      // [col][ntargets] scratch of the regrouping
  int32_t* ngroups;    // [col]
  int32_t* has_nan;    // [col]
  unsigned long long* hist;  // [col][ntargets][kBins]
  unsigned long long* gmin;  // [col][ntargets]
  unsigned long long* gmax;  // [col][ntargets]
};

// order-preserving keys: doubles flip the sign bit (positive) or all bits (negative); integers flip the sign bit
__device__ __forceinline__ uint64_t value_key(uint64_t bits, int kind) {
  if (kind == PBL_STATS_F64) return flip_f64(bits);
  if (kind == PBL_STATS_I64_BITS) return bits ^ kSign;
  return (uint64_t)(int64_t)__longlong_as_double((long long)bits) ^ kSign;  // an exact double of an integer
}

__global__ void select_init_kernel(SelArgs a) {
  const int col = blockIdx.x;
  Target* tg = a.targets + (int64_t)col * a.ntargets;
  for (int t = threadIdx.x; t < a.ntargets; t += blockDim.x) {
    const QuantilePick p = quantile_pick(a.q[t >> 1], (double)a.n, a.method);
    tg[t] = Target{0, (uint64_t)((t & 1) ? p.hi : p.lo), 0, 0, 0};
  }
  unsigned long long* h = a.hist + (int64_t)col * a.ntargets * kBins;
  for (int b = threadIdx.x; b < kBins; b += blockDim.x) h[b] = 0;
  if (threadIdx.x == 0) {
    a.gprefix[(int64_t)col * a.ntargets] = 0;
    a.ngroups[col] = 1;
    a.has_nan[col] = 0;
    a.gmin[(int64_t)col * a.ntargets] = ~0ull;
    a.gmax[(int64_t)col * a.ntargets] = 0;
  }
}

// one read of the column: blockIdx.y = column, blockIdx.z = a range of kGroupsPerBlock groups
__global__ void __launch_bounds__(kSelThreads) select_pass_kernel(SelArgs a, int pass) {
  __shared__ unsigned s_hist[kGroupsPerBlock * kBins];
  __shared__ unsigned long long s_min[kGroupsPerBlock], s_max[kGroupsPerBlock];
  const int col = blockIdx.y;
  const int ng = a.ngroups[col];
  const int g0 = blockIdx.z * kGroupsPerBlock;
  if (g0 >= ng) return;
  const int g1 = min(ng, g0 + kGroupsPerBlock);
  const int64_t cbase = (int64_t)col * a.ntargets;
  const uint64_t* gp = a.gprefix + cbase;
  for (int i = threadIdx.x; i < (g1 - g0) * kBins; i += kSelThreads) s_hist[i] = 0;
  for (int i = threadIdx.x; i < g1 - g0; i += kSelThreads) {
    s_min[i] = ~0ull;
    s_max[i] = 0;
  }
  __syncthreads();
  const int kind = a.kinds[col];
  const uint64_t* x = a.cols[col];
  const int pshift = 64 - kDigitBits * pass;  // prefix = key >> pshift (pass 0: every key, group 0)
  const int dshift = 64 - kDigitBits * (pass + 1);
  const uint64_t plo = gp[g0], phi = gp[g1 - 1];
  const int lane = threadIdx.x & 31;
  int cur = -1;
  unsigned long long tmin = 0, tmax = 0;
  bool nan = false;
  const int64_t stride = (int64_t)gridDim.x * kSelThreads;
  // warp-uniform trip count (the histogram adds are aggregated across the warp)
  for (int64_t base = (int64_t)blockIdx.x * kSelThreads + (threadIdx.x & ~31); base < a.n; base += stride) {
    const int64_t i = base + lane;
    int g = -1;
    uint64_t key = 0;
    if (i < a.n) {
      const uint64_t bits = ld_stream_u64(x + i);
      if (kind == PBL_STATS_F64) nan |= ((bits & ~kSign) > 0x7FF0000000000000ull);
      key = value_key(bits, kind);
      if (pass == 0) {
        g = 0;
      } else {
        const uint64_t p = key >> pshift;
        if (p >= plo && p <= phi) {
          int lo = g0, hi = g1 - 1;
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (gp[mid] < p) lo = mid + 1; else hi = mid;
          }
          if (gp[lo] == p) g = lo;
        }
      }
    }
    unsigned bin = 0xFFFFFFFFu;
    if (g >= 0) {
      bin = (unsigned)((g - g0) * kBins) + (unsigned)((key >> dshift) & (kBins - 1));
      if (g != cur) {
        if (cur >= 0) {
          atomicMin(&s_min[cur - g0], tmin);
          atomicMax(&s_max[cur - g0], tmax);
        }
        cur = g;
        tmin = tmax = key;
      } else {
        tmin = min(tmin, (unsigned long long)key);
        tmax = max(tmax, (unsigned long long)key);
      }
    }
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, bin);
    if (bin != 0xFFFFFFFFu && lane == __ffs(peers) - 1) atomicAdd(&s_hist[bin], (unsigned)__popc(peers));
  }
  if (cur >= 0) {
    atomicMin(&s_min[cur - g0], tmin);
    atomicMax(&s_max[cur - g0], tmax);
  }
  if (nan) a.has_nan[col] = 1;
  __syncthreads();
  unsigned long long* h = a.hist + (cbase + g0) * kBins;
  for (int i = threadIdx.x; i < (g1 - g0) * kBins; i += kSelThreads)
    if (s_hist[i]) atomicAdd(&h[i], (unsigned long long)s_hist[i]);
  for (int i = threadIdx.x; i < g1 - g0; i += kSelThreads) {
    if (s_max[i] >= s_min[i]) {
      atomicMin(&a.gmin[cbase + g0 + i], s_min[i]);
      atomicMax(&a.gmax[cbase + g0 + i], s_max[i]);
    }
  }
}

// one block per column: advance every unresolved target by the pass's histogram, then regroup
__global__ void __launch_bounds__(kSelThreads) select_update_kernel(SelArgs a, int pass) {
  __shared__ int s_count;
  const int col = blockIdx.x;
  if (a.ngroups[col] == 0) return;
  const int64_t cbase = (int64_t)col * a.ntargets;
  Target* tg = a.targets + cbase;
  const bool nan = a.has_nan[col] != 0;  // every quantile is NaN: nothing to select
  for (int t = threadIdx.x; t < a.ntargets; t += kSelThreads) {
    Target v = tg[t];
    if (v.done) continue;
    const int64_t g = cbase + v.group;
    if (nan) {
      v.done = 1;
    } else if (a.gmin[g] == a.gmax[g]) {  // one distinct key left
      v.done = 1;
      v.key = a.gmin[g];
    } else {
      const unsigned long long* h = a.hist + g * kBins;
      uint64_t cum = 0;
      int b = 0;
      for (; b < kBins - 1; ++b) {
        if (v.rank < cum + h[b]) break;
        cum += h[b];
      }
      v.rank -= cum;
      v.prefix = (v.prefix << kDigitBits) | (uint64_t)b;
      if (pass == kPasses - 1) {
        v.done = 1;
        v.key = v.prefix;
      }
    }
    tg[t] = v;
  }
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  // groups of the next pass: the distinct prefixes of the unresolved targets, ascending
  for (int t = threadIdx.x; t < a.ntargets; t += kSelThreads) {
    int f = 0;
    if (!tg[t].done) {
      f = 1;
      for (int u = 0; u < t && f; ++u)
        if (!tg[u].done && tg[u].prefix == tg[t].prefix) f = 0;
    }
    a.first[cbase + t] = f;
    if (f) atomicAdd(&s_count, 1);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < a.ntargets; t += kSelThreads) {
    if (tg[t].done) continue;
    int g = 0;
    for (int u = 0; u < a.ntargets; ++u)
      if (a.first[cbase + u] && tg[u].prefix < tg[t].prefix) ++g;
    tg[t].group = g;
    if (a.first[cbase + t]) a.gprefix[cbase + g] = tg[t].prefix;
  }
  const int ng = s_count;
  for (int64_t i = threadIdx.x; i < (int64_t)ng * kBins; i += kSelThreads) a.hist[cbase * kBins + i] = 0;
  for (int i = threadIdx.x; i < ng; i += kSelThreads) {
    a.gmin[cbase + i] = ~0ull;
    a.gmax[cbase + i] = 0;
  }
  if (threadIdx.x == 0) a.ngroups[col] = ng;
}

// the quantiles from the selected order statistics: out[col][q] holds a double, or int64 bits for a method that
// does not interpolate on an integer column
__global__ void select_finish_kernel(SelArgs a, uint64_t* out) {
  const int col = blockIdx.x;
  const int kind = a.kinds[col];
  const Target* tg = a.targets + (int64_t)col * a.ntargets;
  const bool interp = quantile_interpolates(a.method);
  for (int i = threadIdx.x; i < a.nq; i += blockDim.x) {
    const uint64_t klo = tg[2 * i].key, khi = tg[2 * i + 1].key;
    uint64_t r;
    if (kind == PBL_STATS_F64) {
      double v;
      if (a.has_nan[col]) {
        v = __longlong_as_double(0x7FF8000000000000ll);
      } else {
        const double lo = key_to_double(klo), hi = key_to_double(khi);
        v = lo;
        if (interp) v = quantile_lerp(lo, hi, __dsub_rn(hi, lo), quantile_pick(a.q[i], (double)a.n, a.method).gamma);
      }
      r = (uint64_t)__double_as_longlong(v);
    } else {
      const int64_t lo = (int64_t)(klo ^ kSign), hi = (int64_t)(khi ^ kSign);
      if (interp) {  // b - a in int64 (wrapping), then float64
        const double diff = __ll2double_rn((long long)((uint64_t)hi - (uint64_t)lo));
        const double v = quantile_lerp(__ll2double_rn(lo), __ll2double_rn(hi), diff,
                                       quantile_pick(a.q[i], (double)a.n, a.method).gamma);
        r = (uint64_t)__double_as_longlong(v);
      } else {
        r = (uint64_t)lo;
      }
    }
    out[(int64_t)col * a.nq + i] = r;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// min / max, histograms and the ordered compaction of a range
constexpr int kScanThreads = 256;
constexpr int kHistThreads = 512;
// Counts of one histogram column live in a block's shared memory (u32, flushed to u64 global counts with integer
// atomics) up to kHistSmemCounts; above, every value is a warp-aggregated u64 atomic in global memory.  The edge
// table joins the counts in shared memory when both fit kHistSmemBytes, else it is read through the read-only path.
constexpr int64_t kHistSmemCounts = 16384;
constexpr int kHistSmemBytes = 96 * 1024;
constexpr int kTile = 8192;  // values of one compaction block: its keep count, scanned, orders the scatter
constexpr unsigned long long kNone = ~0ull;

__device__ __forceinline__ int64_t value_i64(uint64_t bits, int kind) {  // integer kinds only
  if (kind == PBL_STATS_I64_BITS) return (int64_t)bits;
  return (int64_t)__longlong_as_double((long long)bits);  // an exact double of an integer
}
__device__ __forceinline__ bool is_nan_bits(uint64_t bits, int kind) {
  return kind == PBL_STATS_F64 && (bits & ~kSign) > 0x7FF0000000000000ull;
}
// (a >= lo) & (a <= hi), each comparison in its own type, as NumPy evaluates them
__device__ __forceinline__ bool keep_value(uint64_t bits, int kind, const pbl_stats_range& r) {
  const bool lo = r.lo_cmp == PBL_HIST_CMP_I64 ? value_i64(bits, kind) >= r.lo_i : value_f64(bits, kind) >= r.lo_f;
  const bool hi = r.hi_cmp == PBL_HIST_CMP_I64 ? value_i64(bits, kind) <= r.hi_i : value_f64(bits, kind) <= r.hi_f;
  return lo && hi;
}

struct ColArgs {
  const uint64_t* const* cols;
  const int32_t* kinds;
  int64_t n;
};

// grid (blocks, columns): NaNs are left out of the keys and their first row is kept instead
__global__ void __launch_bounds__(kScanThreads) minmax_kernel(ColArgs a, unsigned long long* kmin,
                                                              unsigned long long* kmax, unsigned long long* nan_row) {
  const int col = blockIdx.y;
  const int kind = a.kinds[col];
  const uint64_t* x = a.cols[col];
  unsigned long long lo = kNone, hi = 0, nan = kNone;
  for (int64_t i = (int64_t)blockIdx.x * kScanThreads + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * kScanThreads) {
    const uint64_t bits = ld_stream_u64(x + i);
    if (is_nan_bits(bits, kind)) {
      nan = min(nan, (unsigned long long)i);
      continue;
    }
    const unsigned long long key = value_key(bits, kind);
    lo = min(lo, key);
    hi = max(hi, key);
  }
  for (int o = 16; o; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
    nan = min(nan, __shfl_xor_sync(0xFFFFFFFFu, nan, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (lo != kNone) atomicMin(&kmin[col], lo);
    if (hi != 0) atomicMax(&kmax[col], hi);
    if (nan != kNone) atomicMin(&nan_row[col], nan);
  }
}

__global__ void minmax_finish_kernel(ColArgs a, int ncols, const unsigned long long* kmin,
                                     const unsigned long long* kmax, const unsigned long long* nan_row, uint64_t* out) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncols) return;
  const int kind = a.kinds[col];
  if (kind == PBL_STATS_F64) {
    if (nan_row[col] != kNone) {
      out[2 * col] = out[2 * col + 1] = a.cols[col][nan_row[col]];
    } else {
      out[2 * col] = unflip_f64(kmin[col]);
      out[2 * col + 1] = unflip_f64(kmax[col]);
    }
  } else {
    out[2 * col] = kmin[col] ^ kSign;
    out[2 * col + 1] = kmax[col] ^ kSign;
  }
}

// grid (blocks, columns); one read of every column, counts per spec
__global__ void __launch_bounds__(kHistThreads) histogram_kernel(ColArgs a, const pbl_stats_hist_spec* specs,
                                                                 int smem_bytes, unsigned long long* counts,
                                                                 unsigned long long* bad_row) {
  extern __shared__ double s_hist_raw[];
  const int col = blockIdx.y;
  const pbl_stats_hist_spec sp = specs[col];
  const int kind = a.kinds[col];
  const bool uniform = sp.mode == PBL_HIST_UNIFORM;
  const int64_t m = sp.nbins;
  const int64_t ncount = uniform ? m : 2 * m + 2, ntable = uniform ? m + 1 : m;
  const bool smem_counts = ncount <= kHistSmemCounts;
  const bool smem_table = ntable * 8 + (smem_counts ? ncount * 4 : 0) <= smem_bytes;
  uint64_t* s_tab = reinterpret_cast<uint64_t*>(s_hist_raw);
  unsigned* s_cnt = reinterpret_cast<unsigned*>(s_hist_raw + (smem_table ? ntable : 0));
  const uint64_t* g_tab = static_cast<const uint64_t*>(sp.table);
  if (smem_table)
    for (int64_t k = threadIdx.x; k < ntable; k += kHistThreads) s_tab[k] = __ldg(g_tab + k);
  if (smem_counts)
    for (int64_t k = threadIdx.x; k < ncount; k += kHistThreads) s_cnt[k] = 0;
  __syncthreads();
  auto tab = [&](int64_t k) -> uint64_t { return smem_table ? s_tab[k] : __ldg(g_tab + k); };
  unsigned long long* g_cnt = counts + sp.offset;
  const uint64_t* x = a.cols[col];
  const int lane = threadIdx.x & 31;
  const double nb = (double)m;
  unsigned long long bad = kNone;
  const int64_t stride = (int64_t)gridDim.x * kHistThreads;
  // warp-uniform trip count (the count adds are aggregated across the warp)
  for (int64_t base = (int64_t)blockIdx.x * kHistThreads + (threadIdx.x & ~31); base < a.n; base += stride) {
    const int64_t i = base + lane;
    unsigned long long bin = kNone;
    if (i < a.n) {
      const uint64_t bits = ld_stream_u64(x + i);
      if (uniform) {
        if (keep_value(bits, kind, sp.keep)) {
          const double v = value_f64(bits, kind);
          const double f = __dmul_rn(__ddiv_rn(__dsub_rn(v, sp.first), sp.denom), nb);
          long long b = -1;
          if (f >= 0.0 && f < 9.0e18) {  // intp(f); NumPy's cast of anything else indexes outside the table
            b = (long long)f;
            if (b == m) b = m - 1;
            if (b < m) {
              if (v < __longlong_as_double((long long)tab(b))) --b;
              if (v >= __longlong_as_double((long long)tab(b + 1)) && b != m - 1) ++b;
            } else {
              b = -1;
            }
          }
          if (b >= 0) bin = (unsigned long long)b; else bad = min(bad, (unsigned long long)i);
        }
      } else {
        int64_t lo = 0, hi = m;
        bool eq;
        if (sp.cmp == PBL_HIST_CMP_I64) {
          const int64_t v = value_i64(bits, kind);
          while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if ((int64_t)tab(mid) < v) lo = mid + 1; else hi = mid;
          }
          eq = lo < m && (int64_t)tab(lo) == v;
          bin = 2 * lo + eq;
        } else if (is_nan_bits(bits, kind)) {
          bin = 2 * m + 1;
        } else {
          const double v = value_f64(bits, kind);
          while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (__longlong_as_double((long long)tab(mid)) < v) lo = mid + 1; else hi = mid;
          }
          eq = lo < m && __longlong_as_double((long long)tab(lo)) == v;
          bin = 2 * lo + eq;
        }
      }
    }
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, bin);
    if (bin != kNone && lane == __ffs(peers) - 1) {
      if (smem_counts) atomicAdd(&s_cnt[bin], (unsigned)__popc(peers));
      else atomicAdd(&g_cnt[bin], (unsigned long long)__popc(peers));
    }
  }
  if (bad != kNone) atomicMin(&bad_row[col], bad);
  if (!smem_counts) return;
  __syncthreads();
  for (int64_t k = threadIdx.x; k < ncount; k += kHistThreads)
    if (s_cnt[k]) atomicAdd(&g_cnt[k], (unsigned long long)s_cnt[k]);
}

// grid (tiles, columns): the number of kept values of every tile
__global__ void __launch_bounds__(kScanThreads) compact_count_kernel(ColArgs a, const pbl_stats_range* keep,
                                                                     int64_t* tile_count) {
  const int col = blockIdx.y;
  const int kind = a.kinds[col];
  const pbl_stats_range r = keep[col];
  const int64_t t0 = (int64_t)blockIdx.x * kTile, t1 = min64(t0 + kTile, a.n);
  int c = 0;
  for (int64_t i = t0 + threadIdx.x; i - threadIdx.x < t1; i += kScanThreads)
    c += __syncthreads_count(i < t1 && keep_value(ld_stream_u64(a.cols[col] + i), kind, r));
  if (threadIdx.x == 0) tile_count[(int64_t)col * gridDim.x + blockIdx.x] = c;
}

// one block per column: exclusive scan of the tile counts in place, the total into kept[col]
__global__ void __launch_bounds__(1024) compact_scan_kernel(int64_t tiles, int64_t* tile_count, int64_t* kept) {
  __shared__ int64_t s_warp[32];
  int64_t* t = tile_count + (int64_t)blockIdx.x * tiles;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int64_t carry = 0;
  for (int64_t c0 = 0; c0 < tiles; c0 += 1024) {
    const int64_t i = c0 + threadIdx.x;
    const int64_t v = i < tiles ? t[i] : 0;
    int64_t s = v;  // inclusive scan within the warp
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t u = __shfl_up_sync(0xFFFFFFFFu, s, o);
      if (lane >= o) s += u;
    }
    if (lane == 31) s_warp[warp] = s;
    __syncthreads();
    int64_t before = carry;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    int64_t chunk = 0;
    for (int w = 0; w < 32; ++w) chunk += s_warp[w];
    if (i < tiles) t[i] = before + s - v;
    carry += chunk;
    __syncthreads();
  }
  if (threadIdx.x == 0) kept[blockIdx.x] = carry;
}

// grid (tiles, columns): the kept values of a tile in order, from the tile's scanned offset
__global__ void __launch_bounds__(kScanThreads) compact_scatter_kernel(ColArgs a, const pbl_stats_range* keep,
                                                                       const int64_t* tile_offset,
                                                                       uint64_t* const* out) {
  __shared__ int s_warp[kScanThreads / 32];
  const int col = blockIdx.y;
  const int kind = a.kinds[col];
  const pbl_stats_range r = keep[col];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t t0 = (int64_t)blockIdx.x * kTile, t1 = min64(t0 + kTile, a.n);
  int64_t at = tile_offset[(int64_t)col * gridDim.x + blockIdx.x];
  uint64_t* dst = out[col];
  for (int64_t c0 = t0; c0 < t1; c0 += kScanThreads) {
    const int64_t i = c0 + threadIdx.x;
    uint64_t bits = 0;
    bool k = false;
    if (i < t1) {
      bits = ld_stream_u64(a.cols[col] + i);
      k = keep_value(bits, kind, r);
    }
    const unsigned ballot = __ballot_sync(0xFFFFFFFFu, k);
    if (lane == 0) s_warp[warp] = __popc(ballot);
    __syncthreads();
    int64_t pos = at;
    int total = 0;
    for (int w = 0; w < kScanThreads / 32; ++w) {
      if (w < warp) pos += s_warp[w];
      total += s_warp[w];
    }
    if (k) dst[pos + __popc(ballot & lanemask_lt())] = bits;
    at += total;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------------------------
// one scratch buffer per device, grown on demand; the calls are synchronous, so it is free again when they return
std::mutex g_mu;
std::map<int, std::pair<unsigned char*, size_t>> g_scratch;

int scratch(size_t bytes, unsigned char** p) {
  int device = 0;
  PBL_CUDA_CHECK(cudaGetDevice(&device));
  auto& s = g_scratch[device];
  if (s.second < bytes) {
    if (s.first) cudaFree(s.first);
    s = {nullptr, 0};
    const size_t cap = std::max<size_t>(bytes + bytes / 4, 1 << 20);
    PBL_CUDA_CHECK(cudaMalloc((void**)&s.first, cap));
    s.second = cap;
  }
  *p = s.first;
  return kOk;
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

bool columns_ok(const void* const* cols, const int32_t* kinds, int32_t ncols, int64_t n, const char* what) {
  if (ncols < 1 || ncols > 65535 || n < 1 || !cols || !kinds) {
    set_last_error(std::string(what) + ": bad arguments");
    return false;
  }
  for (int c = 0; c < ncols; ++c) {
    if (!cols[c] || kinds[c] < PBL_STATS_F64 || kinds[c] > PBL_STATS_BOOL_AS_F64) {
      set_last_error(std::string(what) + ": column " + std::to_string(c) + " has no pointer or an unknown kind");
      return false;
    }
  }
  return true;
}

}  // namespace
}  // namespace pbl

using namespace pbl;

extern "C" {

int pbl_stats_moments(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n, int64_t chunk,
                      int32_t what, double divisor, double* out, void* stream_) {
  if (!columns_ok(cols_dev, kinds, ncols, n, "pbl_stats_moments")) return kBadShape;
  if (chunk < 1 || what < PBL_STATS_MEAN || what > PBL_STATS_STD || !out) {
    set_last_error("pbl_stats_moments: bad chunk, statistic or output");
    return kBadShape;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  // grid: the most subtrees any column needs, for the mean pass and (var / std) the squares pass
  int64_t blocks[2] = {0, 0};
  for (int p = 0; p < 2; ++p)
    for (int c = 0; c < ncols; ++c) {
      const int64_t L0 = seg_len(kinds[c], p == 1, n, chunk);
      blocks[p] = std::max(blocks[p], ((n + L0 - 1) / L0) << cut_depth(std::min(L0, n)));
    }
  if (std::max(blocks[0], blocks[1]) > 0x7FFFFFFF) {
    set_last_error("pbl_stats_moments: too many chunks for one launch");
    return kBadShape;
  }
  const int64_t stride = std::max(blocks[0], blocks[1]);
  const size_t off_cols = 0, off_kinds = align256((size_t)ncols * 8), off_means = off_kinds + align256((size_t)ncols * 4);
  const size_t off_out = off_means + align256((size_t)ncols * 8), off_part = off_out + align256((size_t)ncols * 8);
  const size_t total = off_part + 2 * (size_t)ncols * (size_t)stride * 8;
  std::vector<unsigned char> host(off_means, 0);
  memcpy(host.data() + off_cols, cols_dev, (size_t)ncols * 8);
  memcpy(host.data() + off_kinds, kinds, (size_t)ncols * 4);
  std::lock_guard<std::mutex> lock(g_mu);
  unsigned char* dev = nullptr;
  PBL_RETURN_IF(scratch(total, &dev));
  PBL_CUDA_CHECK(cudaMemcpyAsync(dev, host.data(), host.size(), cudaMemcpyHostToDevice, stream));
  SumArgs a;
  a.cols = reinterpret_cast<const uint64_t* const*>(dev + off_cols);
  a.kinds = reinterpret_cast<const int32_t*>(dev + off_kinds);
  a.n = n;
  a.chunk = chunk;
  a.means = reinterpret_cast<const double*>(dev + off_means);
  a.partials = reinterpret_cast<double*>(dev + off_part);
  a.pingpong = a.partials + (size_t)ncols * stride;
  a.stride = stride;
  double* means = reinterpret_cast<double*>(dev + off_means);
  double* res = reinterpret_cast<double*>(dev + off_out);
  const size_t smem = (size_t)kSubtreeCap * 8;
  static bool attr = false;  // (per process: the attribute only raises a limit)
  if (!attr) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(pairwise_subtree_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    PBL_CUDA_CHECK(cudaFuncSetAttribute(pairwise_subtree_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  pairwise_subtree_kernel<false><<<dim3((unsigned)blocks[0], (unsigned)ncols), kSumThreads, smem, stream>>>(a);
  PBL_LAUNCH_CHECK();
  pairwise_finish_kernel<<<ncols, 1024, 0, stream>>>(a, false, what, divisor, means, res);
  PBL_LAUNCH_CHECK();
  if (what != PBL_STATS_MEAN) {
    pairwise_subtree_kernel<true><<<dim3((unsigned)blocks[1], (unsigned)ncols), kSumThreads, smem, stream>>>(a);
    PBL_LAUNCH_CHECK();
    pairwise_finish_kernel<<<ncols, 1024, 0, stream>>>(a, true, what, divisor, nullptr, res);
    PBL_LAUNCH_CHECK();
  }
  PBL_CUDA_CHECK(cudaMemcpyAsync(out, res, (size_t)ncols * 8, cudaMemcpyDefault, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  return kOk;
}

int pbl_stats_quantiles(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n, const double* q,
                        int32_t nq, int32_t method, void* out, void* stream_) {
  if (!columns_ok(cols_dev, kinds, ncols, n, "pbl_stats_quantiles")) return kBadShape;
  if (nq < 1 || nq > (1 << 24) || !q || !out || method < kQLinear || method > kQClosest) {
    set_last_error("pbl_stats_quantiles: bad q, method or output");
    return kBadShape;
  }
  for (int i = 0; i < nq; ++i)
    if (!(q[i] >= 0.0 && q[i] <= 1.0)) {
      set_last_error("pbl_stats_quantiles: q outside [0, 1]");
      return kBadShape;
    }
  cudaStream_t stream = (cudaStream_t)stream_;
  const int64_t T = 2 * (int64_t)nq, CT = (int64_t)ncols * T;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align256(bytes);
    return o;
  };
  const size_t o_cols = take((size_t)ncols * 8), o_kinds = take((size_t)ncols * 4), o_q = take((size_t)nq * 8);
  const size_t host_bytes = off;
  const size_t o_tg = take((size_t)CT * sizeof(Target)), o_gp = take((size_t)CT * 8), o_first = take((size_t)CT * 4);
  const size_t o_ng = take((size_t)ncols * 4), o_nan = take((size_t)ncols * 4), o_hist = take((size_t)CT * kBins * 8);
  const size_t o_min = take((size_t)CT * 8), o_max = take((size_t)CT * 8), o_out = take((size_t)ncols * nq * 8);
  std::vector<unsigned char> host(host_bytes, 0);
  memcpy(host.data() + o_cols, cols_dev, (size_t)ncols * 8);
  memcpy(host.data() + o_kinds, kinds, (size_t)ncols * 4);
  memcpy(host.data() + o_q, q, (size_t)nq * 8);
  std::lock_guard<std::mutex> lock(g_mu);
  unsigned char* dev = nullptr;
  PBL_RETURN_IF(scratch(off, &dev));
  PBL_CUDA_CHECK(cudaMemcpyAsync(dev, host.data(), host_bytes, cudaMemcpyHostToDevice, stream));
  SelArgs a;
  a.cols = reinterpret_cast<const uint64_t* const*>(dev + o_cols);
  a.kinds = reinterpret_cast<const int32_t*>(dev + o_kinds);
  a.n = n;
  a.ntargets = (int32_t)T;
  a.q = reinterpret_cast<const double*>(dev + o_q);
  a.nq = nq;
  a.method = method;
  a.targets = reinterpret_cast<Target*>(dev + o_tg);
  a.gprefix = reinterpret_cast<uint64_t*>(dev + o_gp);
  a.first = reinterpret_cast<int32_t*>(dev + o_first);
  a.ngroups = reinterpret_cast<int32_t*>(dev + o_ng);
  a.has_nan = reinterpret_cast<int32_t*>(dev + o_nan);
  a.hist = reinterpret_cast<unsigned long long*>(dev + o_hist);
  a.gmin = reinterpret_cast<unsigned long long*>(dev + o_min);
  a.gmax = reinterpret_cast<unsigned long long*>(dev + o_max);
  uint64_t* res = reinterpret_cast<uint64_t*>(dev + o_out);
  select_init_kernel<<<ncols, kSelThreads, 0, stream>>>(a);
  PBL_LAUNCH_CHECK();
  // a pass block counts at most 2^32 - 1 keys per bin in shared memory
  int64_t gx = std::max<int64_t>(1, std::min<int64_t>((n + 4095) / 4096, ((int64_t)num_sms() * 8 + ncols - 1) / ncols));
  gx = std::max<int64_t>(gx, (n >> 31) + 1);
  const unsigned gz = (unsigned)((T + kGroupsPerBlock - 1) / kGroupsPerBlock);
  for (int pass = 0; pass < kPasses; ++pass) {
    select_pass_kernel<<<dim3((unsigned)gx, (unsigned)ncols, pass == 0 ? 1u : gz), kSelThreads, 0, stream>>>(a, pass);
    PBL_LAUNCH_CHECK();
    select_update_kernel<<<ncols, kSelThreads, 0, stream>>>(a, pass);
    PBL_LAUNCH_CHECK();
  }
  select_finish_kernel<<<ncols, kSelThreads, 0, stream>>>(a, res);
  PBL_LAUNCH_CHECK();
  PBL_CUDA_CHECK(cudaMemcpyAsync(out, res, (size_t)ncols * nq * 8, cudaMemcpyDefault, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  return kOk;
}

int pbl_stats_minmax(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n, void* out,
                     void* stream_) {
  if (!columns_ok(cols_dev, kinds, ncols, n, "pbl_stats_minmax")) return kBadShape;
  if (!out) {
    set_last_error("pbl_stats_minmax: no output");
    return kBadShape;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  const size_t o_cols = 0, o_kinds = align256((size_t)ncols * 8), o_min = o_kinds + align256((size_t)ncols * 4);
  const size_t o_max = o_min + align256((size_t)ncols * 8), o_nan = o_max + align256((size_t)ncols * 8);
  const size_t o_out = o_nan + align256((size_t)ncols * 8), total = o_out + (size_t)ncols * 16;
  std::vector<unsigned char> host(o_min, 0);
  memcpy(host.data() + o_cols, cols_dev, (size_t)ncols * 8);
  memcpy(host.data() + o_kinds, kinds, (size_t)ncols * 4);
  std::lock_guard<std::mutex> lock(g_mu);
  unsigned char* dev = nullptr;
  PBL_RETURN_IF(scratch(total, &dev));
  PBL_CUDA_CHECK(cudaMemcpyAsync(dev, host.data(), host.size(), cudaMemcpyHostToDevice, stream));
  PBL_CUDA_CHECK(cudaMemsetAsync(dev + o_min, 0xFF, (size_t)ncols * 8, stream));
  PBL_CUDA_CHECK(cudaMemsetAsync(dev + o_max, 0, (size_t)ncols * 8, stream));
  PBL_CUDA_CHECK(cudaMemsetAsync(dev + o_nan, 0xFF, (size_t)ncols * 8, stream));
  ColArgs a{reinterpret_cast<const uint64_t* const*>(dev + o_cols), reinterpret_cast<const int32_t*>(dev + o_kinds), n};
  auto* kmin = reinterpret_cast<unsigned long long*>(dev + o_min);
  auto* kmax = reinterpret_cast<unsigned long long*>(dev + o_max);
  auto* nan = reinterpret_cast<unsigned long long*>(dev + o_nan);
  auto* res = reinterpret_cast<uint64_t*>(dev + o_out);
  const int64_t gx = std::max<int64_t>(1, std::min<int64_t>((n + 4095) / 4096, ((int64_t)num_sms() * 8 + ncols - 1) / ncols));
  minmax_kernel<<<dim3((unsigned)gx, (unsigned)ncols), kScanThreads, 0, stream>>>(a, kmin, kmax, nan);
  PBL_LAUNCH_CHECK();
  minmax_finish_kernel<<<(ncols + 255) / 256, 256, 0, stream>>>(a, ncols, kmin, kmax, nan, res);
  PBL_LAUNCH_CHECK();
  PBL_CUDA_CHECK(cudaMemcpyAsync(out, res, (size_t)ncols * 16, cudaMemcpyDefault, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  return kOk;
}

// a comparison type is F64 or I64, and I64 only for a column of integers
static bool cmp_ok(int32_t cmp, int32_t kind) {
  return cmp == PBL_HIST_CMP_F64 || (cmp == PBL_HIST_CMP_I64 && kind != PBL_STATS_F64);
}
static bool range_ok(const pbl_stats_range& r, int32_t kind) { return cmp_ok(r.lo_cmp, kind) && cmp_ok(r.hi_cmp, kind); }

int pbl_stats_histogram(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                        const pbl_stats_hist_spec* specs, uint64_t* counts, int64_t total, int64_t* bad_row,
                        void* stream_) {
  if (!columns_ok(cols_dev, kinds, ncols, n, "pbl_stats_histogram")) return kBadShape;
  if (!specs || !counts || !bad_row || total < 1) {
    set_last_error("pbl_stats_histogram: bad specs or outputs");
    return kBadShape;
  }
  int64_t table_bytes = 0;
  int smem = 0;
  for (int c = 0; c < ncols; ++c) {
    const pbl_stats_hist_spec& s = specs[c];
    const bool uniform = s.mode == PBL_HIST_UNIFORM;
    const int64_t ncount = uniform ? s.nbins : 2 * s.nbins + 2, ntable = uniform ? s.nbins + 1 : s.nbins;
    const bool cmps = uniform ? range_ok(s.keep, kinds[c]) : (s.mode == PBL_HIST_EDGES && cmp_ok(s.cmp, kinds[c]));
    if (!cmps || s.nbins < 1 || s.nbins > (1ll << 40) ||
        !s.table || s.offset < 0 || s.offset > total - ncount) {
      set_last_error("pbl_stats_histogram: column " + std::to_string(c) + " has a bad spec");
      return kBadShape;
    }
    table_bytes += (int64_t)align256((size_t)ntable * 8);
    const int64_t cnt = ncount <= kHistSmemCounts ? ncount * 4 : 0;
    const int64_t need = cnt + ntable * 8 <= kHistSmemBytes ? cnt + ntable * 8 : cnt;
    smem = std::max(smem, (int)need);
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align256(bytes);
    return o;
  };
  const size_t o_cols = take((size_t)ncols * 8), o_kinds = take((size_t)ncols * 4);
  const size_t o_specs = take((size_t)ncols * sizeof(pbl_stats_hist_spec)), o_tab = take((size_t)table_bytes);
  const size_t host_bytes = off;
  const size_t o_cnt = take((size_t)total * 8), o_bad = take((size_t)ncols * 8);
  std::vector<unsigned char> host(host_bytes, 0);
  memcpy(host.data() + o_cols, cols_dev, (size_t)ncols * 8);
  memcpy(host.data() + o_kinds, kinds, (size_t)ncols * 4);
  std::lock_guard<std::mutex> lock(g_mu);
  unsigned char* dev = nullptr;
  PBL_RETURN_IF(scratch(off, &dev));
  auto* dspecs = reinterpret_cast<pbl_stats_hist_spec*>(host.data() + o_specs);
  size_t at = o_tab;
  for (int c = 0; c < ncols; ++c) {  // the tables follow the specs, which point at their device copies
    const int64_t ntable = specs[c].mode == PBL_HIST_UNIFORM ? specs[c].nbins + 1 : specs[c].nbins;
    dspecs[c] = specs[c];
    dspecs[c].table = dev + at;
    memcpy(host.data() + at, specs[c].table, (size_t)ntable * 8);
    at += align256((size_t)ntable * 8);
  }
  PBL_CUDA_CHECK(cudaMemcpyAsync(dev, host.data(), host_bytes, cudaMemcpyHostToDevice, stream));
  PBL_CUDA_CHECK(cudaMemsetAsync(dev + o_cnt, 0, (size_t)total * 8, stream));
  PBL_CUDA_CHECK(cudaMemsetAsync(dev + o_bad, 0xFF, (size_t)ncols * 8, stream));
  static std::map<int, bool> attr;  // per device: the attribute belongs to the device's context
  int device = 0;
  PBL_CUDA_CHECK(cudaGetDevice(&device));
  if (!attr[device]) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(histogram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHistSmemBytes));
    attr[device] = true;
  }
  ColArgs a{reinterpret_cast<const uint64_t* const*>(dev + o_cols), reinterpret_cast<const int32_t*>(dev + o_kinds), n};
  auto* cnt = reinterpret_cast<unsigned long long*>(dev + o_cnt);
  auto* bad = reinterpret_cast<unsigned long long*>(dev + o_bad);
  // a block counts at most 2^32 - 1 values per bin in shared memory
  int64_t gx = std::max<int64_t>(1, std::min<int64_t>((n + 8191) / 8192, ((int64_t)num_sms() * 8 + ncols - 1) / ncols));
  gx = std::max<int64_t>(gx, (n >> 31) + 1);
  histogram_kernel<<<dim3((unsigned)gx, (unsigned)ncols), kHistThreads, (size_t)smem, stream>>>(
      a, reinterpret_cast<const pbl_stats_hist_spec*>(dev + o_specs), smem, cnt, bad);
  PBL_LAUNCH_CHECK();
  PBL_CUDA_CHECK(cudaMemcpyAsync(counts, cnt, (size_t)total * 8, cudaMemcpyDeviceToHost, stream));
  PBL_CUDA_CHECK(cudaMemcpyAsync(bad_row, bad, (size_t)ncols * 8, cudaMemcpyDeviceToHost, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  bool out_of_table = false;
  for (int c = 0; c < ncols; ++c) out_of_table |= bad_row[c] >= 0;  // (kNone reads as -1)
  return out_of_table ? (int)PBL_OUT_OF_TABLE : (int)kOk;
}

int pbl_stats_compact(const void* const* cols_dev, const int32_t* kinds, int32_t ncols, int64_t n,
                      const pbl_stats_range* keep, void* const* out_dev, int64_t* kept, void* stream_) {
  if (!columns_ok(cols_dev, kinds, ncols, n, "pbl_stats_compact")) return kBadShape;
  if (!keep || !kept) {
    set_last_error("pbl_stats_compact: bad ranges or outputs");
    return kBadShape;
  }
  for (int c = 0; c < ncols; ++c)
    if (!range_ok(keep[c], kinds[c]) || (out_dev && !out_dev[c])) {
      set_last_error("pbl_stats_compact: column " + std::to_string(c) + " has a bad range or no output");
      return kBadShape;
    }
  cudaStream_t stream = (cudaStream_t)stream_;
  const int64_t tiles = (n + kTile - 1) / kTile;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += align256(bytes);
    return o;
  };
  const size_t o_cols = take((size_t)ncols * 8), o_kinds = take((size_t)ncols * 4);
  const size_t o_keep = take((size_t)ncols * sizeof(pbl_stats_range)), o_out = take((size_t)ncols * 8);
  const size_t host_bytes = off;
  const size_t o_tiles = take((size_t)ncols * tiles * 8), o_kept = take((size_t)ncols * 8);
  std::vector<unsigned char> host(host_bytes, 0);
  memcpy(host.data() + o_cols, cols_dev, (size_t)ncols * 8);
  memcpy(host.data() + o_kinds, kinds, (size_t)ncols * 4);
  memcpy(host.data() + o_keep, keep, (size_t)ncols * sizeof(pbl_stats_range));
  if (out_dev) memcpy(host.data() + o_out, out_dev, (size_t)ncols * 8);
  std::lock_guard<std::mutex> lock(g_mu);
  unsigned char* dev = nullptr;
  PBL_RETURN_IF(scratch(off, &dev));
  PBL_CUDA_CHECK(cudaMemcpyAsync(dev, host.data(), host_bytes, cudaMemcpyHostToDevice, stream));
  ColArgs a{reinterpret_cast<const uint64_t* const*>(dev + o_cols), reinterpret_cast<const int32_t*>(dev + o_kinds), n};
  auto* dkeep = reinterpret_cast<const pbl_stats_range*>(dev + o_keep);
  auto* tc = reinterpret_cast<int64_t*>(dev + o_tiles);
  auto* dkept = reinterpret_cast<int64_t*>(dev + o_kept);
  compact_count_kernel<<<dim3((unsigned)tiles, (unsigned)ncols), kScanThreads, 0, stream>>>(a, dkeep, tc);
  PBL_LAUNCH_CHECK();
  compact_scan_kernel<<<ncols, 1024, 0, stream>>>(tiles, tc, dkept);
  PBL_LAUNCH_CHECK();
  if (out_dev) {
    compact_scatter_kernel<<<dim3((unsigned)tiles, (unsigned)ncols), kScanThreads, 0, stream>>>(
        a, dkeep, tc, reinterpret_cast<uint64_t* const*>(dev + o_out));
    PBL_LAUNCH_CHECK();
  }
  PBL_CUDA_CHECK(cudaMemcpyAsync(kept, dkept, (size_t)ncols * 8, cudaMemcpyDeviceToHost, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  return kOk;
}

}  // extern "C"
