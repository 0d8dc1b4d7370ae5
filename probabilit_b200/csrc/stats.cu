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

__device__ __forceinline__ double load_value(const uint64_t* col, int kind, int64_t i) {
  const uint64_t bits = ld_stream_u64(col + i);
  if (kind == PBL_STATS_I64_BITS) return __ll2double_rn((long long)bits);
  return __longlong_as_double((long long)bits);  // doubles, and int64 / bool values held as exact doubles
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

}  // extern "C"
