// Batched per-column LSD radix sort ("onesweep": one read + one write of every key per digit
// pass, chained-scan decoupled look-back between tiles) of 64-bit keys with 32-bit row-index
// payloads.  This is the engine under both ranking steps of Iman-Conover; it replaces NumPy's
// stable argsort inside scipy.stats.rankdata (reference call sites
// src/probabilit/correlation.py:394 and :422) and np.sort (:423).
//
// Layout in HBM (all SoA, one contiguous run per column):
//   keys  [ncols][n]  u64   COMPACT order-preserving image of the fp64 values (common.cuh::flip_f64
//                           followed by KeyMap's gap removal), -0.0 stored as +0.0 (they tie in
//                           the reference; the sign travels in bit 31 of the payload and is
//                           restored when the sorted column is read)
//   vals  [ncols][n]  u32   source row of each key (bits 0..30), bit 31 = "was -0.0"
//   hist  [ncols][8][256] u32   digit histograms -> exclusive bin bases
//   status[ncols][ntiles][256]   look-back words of the chained scans between tiles: u64 epoch-tagged words
//                           (below) for the bulk-async kernels and the row-window partition; u32 words (bit31
//                           inclusive, bit30 partial, 30-bit count), cleared before every pass, for the
//                           one-tile-per-block digit pass
//   kminmax[ncols][4] u64   smallest / largest key of the column, largest negative / smallest positive key
// Columns are independent: blockIdx.y is the column, so one launch per digit pass covers the
// whole batch.  The first pass reads the caller's doubles in place (any row stride) and
// synthesises the payload (row index), so X is never copied or converted up front.
//
// WINDOWED SORT.  The passes do not sort on all 64 key bits: they sort on a 32-bit monotone image
// of the key (populated exponent range + top mantissa bits, see KeyMap) -> 4 digit passes instead
// of 8.  Keys that collide in the window end up adjacent but possibly out of order; the consumer
// (post_sort_kernel in ic.cu) completes the order inside each run of equal window values, which
// are short unless the distinct values are packed more densely than 2^-32 of the column's range.
// If a run of distinct keys is too long to complete there, a flag is raised and the caller
// repeats the sort with window_bits = 64 (plain, exact 8-pass LSD sort).  Results are identical
// either way.
//
// Digit passes in which every key of a column has the same digit are skipped on the device
// (no host round trip): the scan kernel records, per column and pass, which ping-pong buffer
// is the source, and whether the pass runs at all.
#pragma once
#include "common.cuh"

namespace pbl {

constexpr int kRadixBits = 8;
constexpr int kRadix = 1 << kRadixBits;
constexpr int kMaxPasses = 64 / kRadixBits;

constexpr uint32_t kFlagInclusive = 0x80000000u;
constexpr uint32_t kFlagPartial = 0x40000000u;
constexpr uint32_t kValueMask = 0x3FFFFFFFu;
constexpr uint32_t kMaxSortN = 0x7FFFFFFFu;  // rows per column: the payload keeps 31 bits for the row
constexpr uint32_t kMaxSortNClassic = 0x3FFFFFFFu;  // one-tile-per-block kernels: 30-bit counts in 32-bit look-back words
constexpr uint32_t kRowMask = 0x7FFFFFFFu;   // payload bits that hold the row
constexpr uint32_t kNegZeroFlag = 0x80000000u;

// Look-back words of the chained scans (digit pass, fused row-window partition) are 64-bit and tagged
// with the EPOCH of the launch that wrote them: [epoch:30 | flag:2 | count:32].  A word from an earlier
// launch reads as "not published", so the array is never cleared between launches (it used to be a
// 0.4-0.8 GB memset before each of the 10 launches of a call) and counts are full 32-bit.
constexpr uint64_t kStatusInclusive = 2ull << 32;
constexpr uint64_t kStatusPartial = 1ull << 32;
__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// error_flag[] slots shared by the sort and its consumers
enum SortFlag : int {
  kFlagWatchdog = 0,    // look-back spin limit hit
  kFlagNaN = 1,         // NaN in the input column
  kFlagNotPD = 2,       // (Iman-Conover) rank correlation not positive definite
  kFlagReserved = 3,
  kFlagWindowRetry = 4, // a run of distinct keys inside one window value was too long
  kFlagNegZeroCol0 = 5  // column 0 of X holds a -0.0 (its tie-runs then mix the two zeros)
};

// Per (column, pass) routing decided on the device by sort_scan_kernel.
struct PassPlan {
  uint8_t run[kMaxPasses];  // 1: the pass moves data, 0: skipped (constant digit)
  uint8_t src[kMaxPasses];  // 0: raw input column, 1: buffer A, 2: buffer B
  uint8_t final_buf;        // buffer holding the sorted column after the last pass (1/2)
  uint8_t pad[7];
};

// Monotone map key -> window value.
//   window_bits == 32 (default): SEGMENTED window.  In key space an fp64 column that straddles zero
//   (or contains zeros) is mostly empty: all the binades between the smallest |x| present and the
//   denormals lie between its negative and positive keys.  The map removes those gaps,
//       a(key) = key - kmin                          key <  Z   (negative values)
//                neg_al                              key == Z   (+-0.0, Z = key of +0.0)
//                neg_al + 2^sh + (key - kpos_min)    key >  Z   (positive values)
//   with kpos_min the smallest key > Z and neg_al = kneg_max - kmin + 1 rounded up to 2^sh, and
//   keeps the 32 most significant bits of a's range:  w = a >> sh.  a is strictly increasing in the
//   key, so w is a monotone image; what remains are (populated exponent range, top mantissa bits):
//   a column spanning 2^e binades keeps 32 - e mantissa bits, e.g. 26 bits (6.7e7 window values per
//   binade) for 1e8 normal samples -> 4 digit passes instead of 8, robust to heavy tails.
//   window_bits == 64: the key itself (exact 8-pass LSD sort, the fall-back).
// kminmax holds 4 words per column: kmin, kmax, kneg_max (largest key < Z, 0 if none),
// kpos_min (smallest key > Z, ~0 if none).
constexpr uint64_t kZeroKey = 0x8000000000000000ull;
constexpr int kMinMaxWords = 4;
struct KeyMap {
  uint64_t kmin;    // subtracted from negative keys
  uint64_t g0;      // subtracted from the zero key
  uint64_t g;       // subtracted from positive keys
  uint64_t neg_al;  // a(zero key); negatives are below it, positives at or above neg_al + 2^sh
  uint32_t sh;
  bool exact;
};
__device__ __forceinline__ KeyMap load_key_map(const uint64_t* __restrict__ kminmax, int col,
                                               int window_bits) {
  KeyMap m;
  m.kmin = 0;
  m.g0 = 0;
  m.g = 0;
  m.neg_al = 0;
  m.sh = 0;
  m.exact = window_bits >= 64;
  if (!m.exact) {
    const uint64_t* q = kminmax + (size_t)kMinMaxWords * col;
    const uint64_t kmin = q[0], kmax = q[1], kneg_max = q[2], kpos_min = q[3];
    const uint64_t span_neg = kmin < kZeroKey ? kneg_max - kmin + 1 : 0;
    const uint64_t span_pos = kmax > kZeroKey ? kmax - kpos_min + 1 : 0;
    // zero gets a window value of its own and the positives start on a fresh one (the segments are
    // aligned to 2^sh), so that heavily tied neighbours of zero (0 / 1 counts) never share a window
    const uint64_t rough = span_neg + 1 + span_pos;  // < 2^64: both spans are < 2^63
    const int bits = 64 - __clzll((long long)rough);
    uint32_t sh = bits > 32 ? (uint32_t)(bits - 32) : 0u;
    uint64_t neg_al = 0, unit = 1;
    for (int it = 0; it < 3; ++it) {
      unit = 1ull << sh;
      neg_al = (span_neg + unit - 1) & ~(unit - 1);
      const uint64_t last = neg_al + unit + span_pos - (span_pos ? 1 : 0);  // largest a
      if ((last >> sh) >> 32) ++sh; else break;
    }
    m.kmin = kmin;
    m.g0 = kZeroKey - neg_al;
    m.g = kpos_min - (neg_al + unit);
    m.neg_al = neg_al;
    m.sh = sh;
  }
  return m;
}
// The sort buffers hold COMPACT keys a(key): the order is the key order, the digit of pass p is
// (a >> (sh + 8 p)) & 255 -- one shift and a mask -- and a is inverted when the sorted column is read.
__device__ __forceinline__ uint64_t compact_key(uint64_t key, const KeyMap& m) {
  if (m.exact) return key;
  const uint64_t base = key > kZeroKey ? m.g : (key == kZeroKey ? m.g0 : m.kmin);
  return key - base;
}
// compact_key(key_of_double(d)) in one go, on the two 32-bit halves of the double (the digit pass that reads
// the caller's doubles spent a quarter of its instructions on 64-bit compares and selects here):
//   negative:  key = ~bits,              a = key - kmin
//   +-0.0:     key = kZeroKey,           a = neg_al            (*neg_zero: it was -0.0)
//   positive:  key = bits ^ 2^63,        a = key - g
// A FusedKeyMap holds the three constants for either window (exact: a = key).
struct FusedKeyMap {
  uint64_t base_neg, base_pos, zero_val;
};
__device__ __forceinline__ FusedKeyMap fused_key_map(const KeyMap& m) {
  FusedKeyMap f;
  f.base_neg = m.exact ? 0ull : m.kmin;
  f.base_pos = m.exact ? 0ull : m.g;
  f.zero_val = m.exact ? kZeroKey : m.neg_al;
  return f;
}
__device__ __forceinline__ uint64_t compact_key_of_double(double d, const FusedKeyMap& f, bool* neg_zero) {
  const uint32_t hi = (uint32_t)__double2hiint(d), lo = (uint32_t)__double2loint(d);
  const uint32_t m = (uint32_t)((int32_t)hi >> 31);  // all ones for a set sign bit
  const bool neg = (int32_t)hi < 0;
  const bool zero = ((hi & 0x7FFFFFFFu) | lo) == 0u;
  const uint32_t kh = hi ^ (m | 0x80000000u), kl = lo ^ m;
  const uint64_t key = ((uint64_t)kh << 32) | kl;
  const uint64_t a = key - (neg ? f.base_neg : f.base_pos);
  *neg_zero = neg && zero;
  return zero ? f.zero_val : a;
}
__device__ __forceinline__ uint64_t expand_key(uint64_t a, const KeyMap& m) {
  if (m.exact) return a;
  return a > m.neg_al ? a + m.g : (a == m.neg_al ? kZeroKey : a + m.kmin);
}
// window value / window equality of COMPACT keys
__device__ __forceinline__ uint64_t window_value(uint64_t a, const KeyMap& m) { return a >> m.sh; }
__device__ __forceinline__ bool same_window(uint64_t a, uint64_t b, const KeyMap& m) {
  return ((a ^ b) >> m.sh) == 0;
}

struct SortBuffers {
  uint64_t* keysA = nullptr;
  uint64_t* keysB = nullptr;
  uint32_t* valsA = nullptr;
  uint32_t* valsB = nullptr;
  uint32_t* hist = nullptr;          // [ncols][8][256]
  uint32_t* status = nullptr;        // [ncols][ntiles][256] look-back words, sort_status_bytes() of them
  uint32_t* tile_counter = nullptr;  // [8 passes + 1 scatter pass][ncols]
  PassPlan* plan = nullptr;          // [ncols]
  uint64_t* kminmax = nullptr;       // [ncols][4], see KeyMap
  KeyMap* maps = nullptr;            // [ncols] the window map of every column (written by sort_scan_kernel)
  uint32_t* error_flag = nullptr;    // [8], see SortFlag
  uint32_t* epoch = nullptr;         // host counter: launches that have used `status` with epoch-tagged words
};

size_t sort_status_bytes(int ncols, uint32_t n);

// The long-column rule (sort.cu): columns of n rows, n > 3e8 (PBL_CLASSIC_ABOVE=<rows> moves the threshold) and
// n <= kMaxSortNClassic, are finished by the one-tile-per-block consumer (post_sort_kernel in ic.cu) instead of
// post_tma_kernel, and sorted by the one-tile-per-block digit pass (partition_pass_kernel) instead of
// pass_tma_kernel when the launch holds one or two such columns.
bool sort_classic_consumer(uint32_t n);
bool sort_classic_pass(uint32_t n, int ncols);

// Optional CUDA-event timing of every digit-pass launch (bench.py's roofline leg): when enabled,
// sort_columns_f64 brackets each partition_pass_kernel launch with events on the launching stream.
void sort_profile_enable(bool on);
// Drains the recorded events (synchronises them): number of pass launches, their total
// duration in ms and the number of keys they moved.
void sort_profile_read(int64_t* launches, double* total_ms, int64_t* keys);

// Sort `ncols` columns of n <= kMaxSortN doubles each on their `window_bits`-bit window (see above);
// column c starts at in + c*col_stride and its rows are row_stride elements apart.  On return (stream
// order) column c's keys/rows, ordered by window value, are in buffer plan[c].final_buf
// (1 = A, 2 = B).  error_flag[kFlagNaN] is set if any input is NaN.
int sort_columns_f64(const double* in, int64_t row_stride, int64_t col_stride, uint32_t n,
                     int ncols, int window_bits, const SortBuffers& buf, cudaStream_t stream);

// "Scatter by row" that follows each sort: out[col][row * row_stride] = value for the (row, value)
// pairs the sort's consumer staged in the "other" ping-pong buffer (vals[other] / keys[other]).
// For columns of 2^19 rows and more written with row_stride 1, the consumer first groups the pairs into
// <= 256 L2-sized row windows (a fused partition step, chained scan between its tiles of `consumer_tile`
// elements): scatter_prepare returns the window shift (32 = no grouping), the tile count, the ticket counter
// and the epoch tag of the launch's look-back words.  scatter_rows then writes every 128 B line of the output
// once, from L2.
int scatter_prepare(uint32_t n, int ncols, const SortBuffers& buf, int64_t row_stride, int consumer_tile,
                    int* shift_out, int* ntiles_out, uint32_t** tile_counter_out, uint32_t* epoch_out,
                    cudaStream_t stream);
// [pos_begin, pos_end): the staged positions to deliver.  With grouped pairs (shift < 32) the pairs of
// rows [a << shift, b << shift) are exactly the positions [a << shift, b << shift), so a caller can
// deliver the output row range by row range (the multi-GPU driver sends each range off as it completes).
int scatter_rows(uint32_t n, int ncols, const SortBuffers& buf, double* out, int64_t row_stride,
                 int64_t col_stride, cudaStream_t stream, uint32_t pos_begin = 0, uint32_t pos_end = 0xFFFFFFFFu);

}  // namespace pbl
