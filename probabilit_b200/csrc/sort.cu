// Batched per-column windowed onesweep LSD radix sort + scatter-by-row (see sort.cuh).
#include "sort.cuh"

#include "tile_pipeline.cuh"

#include <algorithm>
#include <cstdlib>
#include <vector>

namespace pbl {

namespace {

constexpr uint32_t kSpinLimit = 1u << 24;  // look-back watchdog: fail loudly instead of hanging

// fp64 -> sort key (order-preserving, -0.0 folded onto +0.0); *neg_zero tells the caller
__device__ __forceinline__ uint64_t key_of_double(double d, bool* neg_zero) {
  uint64_t bits = (uint64_t)__double_as_longlong(d);
  const bool nz = bits == 0x8000000000000000ull;
  if (nz) bits = 0;
  *neg_zero = nz;
  return flip_f64(bits);
}

// --------------------------------------------------------------------------------------
// Kernel 0: per-column min / max key (for the window map) and the NaN check the reference
// gets from scipy's check_finite (correlation.py:409).  8 B / key, pure streaming.
// --------------------------------------------------------------------------------------
__global__ void minmax_init_kernel(uint64_t* __restrict__ kminmax, int ncols) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < ncols) {
    kminmax[kMinMaxWords * c] = ~0ull;
    kminmax[kMinMaxWords * c + 1] = 0ull;
    kminmax[kMinMaxWords * c + 2] = 0ull;   // largest key below the zero key
    kminmax[kMinMaxWords * c + 3] = ~0ull;  // smallest key above the zero key
  }
}

// Order-preserving 32-bit image of the HIGH word of an fp64 (sign, exponent, top 20 mantissa bits):
// monotone (not strictly) in the value, NaNs land beyond the infinities on either side.
__device__ __forceinline__ uint32_t hi_image(uint32_t hi32) {
  return hi32 ^ ((uint32_t)((int32_t)hi32 >> 31) | 0x80000000u);
}
__device__ __forceinline__ uint32_t hi_image_of(double d) { return hi_image((uint32_t)__double2hiint(d)); }

template <int BLOCK, int UNROLL>
__global__ void __launch_bounds__(BLOCK)
col_minmax_kernel(const double* __restrict__ raw, int64_t row_stride, int64_t col_stride, uint32_t n,
                  uint64_t* __restrict__ kminmax, uint32_t* __restrict__ error_flag) {
  // The four extremes are tracked exactly as doubles per thread, but an element only reaches that
  // code (several emulated fp64 min/max, ~45 instructions) when a 32-bit FILTER on the image of its
  // high word says it could move one of them: outside [f_min, f_max] of what the warp has seen, or
  // inside the gap [f_neg, f_pos] between the warp's largest negative and smallest positive value.
  // The filters are shared by the warp and refreshed after every exact update, so after the first
  // few batches an element costs 2 + 4 integer instructions (records are O(log n) per warp).
  // Zeros, infinities and NaNs always pass the filter.
  __shared__ double s_lo[BLOCK / 32], s_hi[BLOCK / 32], s_nm[BLOCK / 32], s_pm[BLOCK / 32];
  const double inf = __longlong_as_double(0x7FF0000000000000LL);
  const int col = blockIdx.y;
  const double* colp = raw + (int64_t)col * col_stride;
  double lo = inf, hi = -inf, negmax = -inf, posmin = inf;  // fmin / fmax drop NaNs
  bool saw_nan = false;
  uint32_t f_min = 0xFFFFFFFFu, f_max = 0u, f_neg = 0u, f_pos = 0xFFFFFFFFu;  // everything passes
  const uint64_t step = (uint64_t)gridDim.x * BLOCK * UNROLL;
  for (uint64_t base = (uint64_t)blockIdx.x * BLOCK * UNROLL; base < n; base += step) {
    double d[UNROLL];
    if (base + (uint64_t)BLOCK * UNROLL <= n) {  // interior batch: no bounds tests
      const double* p0 = colp + (int64_t)(base + threadIdx.x) * row_stride;
      const int64_t du = (int64_t)BLOCK * row_stride;
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) d[u] = ld_stream_f64(p0 + u * du);
    } else {
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        uint64_t i = base + (uint64_t)u * BLOCK + threadIdx.x;
        d[u] = (i < n) ? ld_stream_f64(colp + (int64_t)i * row_stride) : colp[0];
      }
    }
    bool pass = false;
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const uint32_t h = hi_image_of(d[u]);
      pass |= (h <= f_min) | (h >= f_max) | ((h >= f_neg) & (h <= f_pos));
    }
    if (__any_sync(0xFFFFFFFFu, pass)) {
      if (pass) {
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          saw_nan |= (d[u] != d[u]);
          lo = fmin(lo, d[u]);
          hi = fmax(hi, d[u]);
          negmax = fmax(negmax, d[u] < 0.0 ? d[u] : -inf);
          posmin = fmin(posmin, d[u] > 0.0 ? d[u] : inf);
        }
      }
      // (a lane without candidates contributes its neutral starting values)
      f_min = __reduce_min_sync(0xFFFFFFFFu, hi_image_of(lo));
      f_max = __reduce_max_sync(0xFFFFFFFFu, hi_image_of(hi));
      f_neg = __reduce_max_sync(0xFFFFFFFFu, hi_image_of(negmax));
      f_pos = __reduce_min_sync(0xFFFFFFFFu, hi_image_of(posmin));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
    hi = fmax(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
    negmax = fmax(negmax, __shfl_xor_sync(0xFFFFFFFFu, negmax, o));
    posmin = fmin(posmin, __shfl_xor_sync(0xFFFFFFFFu, posmin, o));
  }
  if ((threadIdx.x & 31) == 0) {
    s_lo[threadIdx.x >> 5] = lo;
    s_hi[threadIdx.x >> 5] = hi;
    s_nm[threadIdx.x >> 5] = negmax;
    s_pm[threadIdx.x >> 5] = posmin;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < BLOCK / 32; ++w) {
      lo = fmin(lo, s_lo[w]);
      hi = fmax(hi, s_hi[w]);
      negmax = fmax(negmax, s_nm[w]);
      posmin = fmin(posmin, s_pm[w]);
    }
    if (lo <= hi) {  // at least one non-NaN value seen
      bool nz;
      unsigned long long* q = (unsigned long long*)&kminmax[kMinMaxWords * col];
      atomicMin(q, (unsigned long long)key_of_double(lo, &nz));
      atomicMax(q + 1, (unsigned long long)key_of_double(hi, &nz));
      if (lo < 0.0) atomicMax(q + 2, (unsigned long long)key_of_double(negmax, &nz));
      if (hi > 0.0) atomicMin(q + 3, (unsigned long long)key_of_double(posmin, &nz));
    }
  }
  if (saw_nan) error_flag[kFlagNaN] = 1u;
}

// --------------------------------------------------------------------------------------
// Kernel 1: the digit histograms of every column's window values in one read of the input
// (8 B / key).  Plain shared-memory reductions: with the compact window every digit, including
// the most significant one, is spread over many values, so same-address conflicts are rare and
// warp aggregation (MATCH.ANY, ~2 cycles per distinct value per SM) would cost more than it saves.
// --------------------------------------------------------------------------------------
template <int BLOCK, int UNROLL, int NP>
__global__ void __launch_bounds__(BLOCK)
sort_hist_kernel(const double* __restrict__ raw, int64_t row_stride, int64_t col_stride, uint32_t n,
                 uint32_t* __restrict__ hist, const uint64_t* __restrict__ kminmax, int window_bits) {
  __shared__ uint32_t sh[NP][kRadix];
  for (int i = threadIdx.x; i < NP * kRadix; i += BLOCK) (&sh[0][0])[i] = 0;
  __syncthreads();
  const int col = blockIdx.y;
  const KeyMap map = load_key_map(kminmax, col, window_bits);
  const double* colp = raw + (int64_t)col * col_stride;
  const uint32_t sh_addr = (uint32_t)__cvta_generic_to_shared(&sh[0][0]);
  const uint64_t step = (uint64_t)gridDim.x * BLOCK * UNROLL;
  for (uint64_t base = (uint64_t)blockIdx.x * BLOCK * UNROLL; base < n; base += step) {
    double d[UNROLL];
    bool valid[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      uint64_t i = base + (uint64_t)u * BLOCK + threadIdx.x;
      valid[u] = i < n;
      d[u] = valid[u] ? ld_stream_f64(colp + (int64_t)i * row_stride) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      bool nz;
      const uint64_t w = window_value(compact_key(key_of_double(d[u], &nz), map), map);
      if (valid[u]) {
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          const uint32_t dg = (uint32_t)(w >> (8 * p)) & 255u;
          asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(sh_addr + (uint32_t)(p * kRadix + dg) * 4u), "r"(1u)
                       : "memory");
        }
      }
    }
  }
  __syncthreads();
  uint32_t* h = hist + (size_t)col * kMaxPasses * kRadix;
  for (int i = threadIdx.x; i < NP * kRadix; i += BLOCK) {
    uint32_t v = (&sh[0][0])[i];
    if (v) atomicAdd(&h[i], v);
  }
}

// block-wide exclusive scan over kRadix values held one per thread (blockDim.x == kRadix)
__device__ __forceinline__ uint32_t block_excl_scan_256(uint32_t v, uint32_t* s_wsum) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
    if (lane >= (uint32_t)d) incl += t;
  }
  if (lane == 31) s_wsum[warp] = incl;
  __syncthreads();
  uint32_t prefix = 0;
#pragma unroll
  for (int w = 0; w < kRadix / 32; ++w)
    if ((uint32_t)w < warp) prefix += s_wsum[w];
  __syncthreads();
  return prefix + incl - v;
}

// --------------------------------------------------------------------------------------
// Kernel 2: histograms -> exclusive bin bases, and the per-column pass plan (which digit
// passes are no-ops, which buffer each pass reads).  One block of 256 threads per column.
// --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kRadix)
sort_scan_kernel(uint32_t* __restrict__ hist, PassPlan* __restrict__ plan, uint32_t n, int npasses,
                 const uint64_t* __restrict__ kminmax, int window_bits, KeyMap* __restrict__ maps) {
  __shared__ uint32_t s_wsum[kRadix / 32];
  __shared__ int s_const[kMaxPasses];
  const int col = blockIdx.x;
  if (threadIdx.x == 32) maps[col] = load_key_map(kminmax, col, window_bits);  // once per column, not per tile
  if (threadIdx.x < kMaxPasses) s_const[threadIdx.x] = 0;
  __syncthreads();
  for (int p = 0; p < npasses; ++p) {
    uint32_t* h = hist + ((size_t)col * kMaxPasses + p) * kRadix;
    uint32_t c = h[threadIdx.x];
    if (c == n) s_const[p] = 1;
    uint32_t e = block_excl_scan_256(c, s_wsum);
    h[threadIdx.x] = e;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    PassPlan pp;
    int cur = 0;
    for (int p = 0; p < kMaxPasses; ++p) {
      bool run = p < npasses && !s_const[p];
      // the data must leave the caller's array at least once: force the last pass if needed
      if (p == npasses - 1 && cur == 0) run = true;
      pp.run[p] = run ? 1 : 0;
      pp.src[p] = (uint8_t)cur;
      if (run) cur = (cur == 1) ? 2 : 1;
    }
    pp.final_buf = (uint8_t)cur;
    for (int i = 0; i < 7; ++i) pp.pad[i] = 0;
    plan[col] = pp;
  }
}

// --------------------------------------------------------------------------------------
// Kernel 3: one radix digit pass (the onesweep step) of compact u64 keys with u32 row payloads.
// Tile = BLOCK*ITEMS elements, warp-striped so that (warp, item, lane) order == position order
// (every LSD pass must be stable).
//   load -> early per-warp digit counts -> tile counts published for the tiles behind us
//   -> ballot-based ranking, one shared-memory atomic per distinct digit and warp
//   -> scatter key + payload into shared memory in digit order -> look back for the
//   exclusive tile prefix per bin -> coalesced runs out to HBM.
//
// The kernel is bound by the integer ALU pipe on B200 (ncu: issue ~50 %, alu pipe saturated; a
// B200 has about half the integer issue rate per byte of HBM bandwidth of an H100), so the code
// is organised to minimise ALU instructions per key:
//   * keys are stored COMPACT (sort.cuh): the digit is one 64-bit shift + mask;
//   * full tiles (all but the last tile of a column) run a path without any bounds predicate;
//   * global addresses are formed with mad.wide (fma pipe) instead of shift/add pairs.
// --------------------------------------------------------------------------------------
struct PassArgs {
  const double* raw;        // caller's column-major-or-strided doubles (src == 0)
  int64_t row_stride, col_stride;
  uint64_t* keysA;
  uint64_t* keysB;
  uint32_t* valsA;
  uint32_t* valsB;
  const uint32_t* bin_base_all;  // [ncols][8][256] exclusive digit histograms
  uint32_t* status;              // [ncols][ntiles][256] 32-bit look-back words (cleared before each pass)
  uint32_t* tile_counter;        // [ncols]
  const PassPlan* plan;
  const uint64_t* kminmax;       // [ncols][4]
  uint32_t* error_flag;
  uint32_t n;
  int pass;                      // digit index
  int window_bits;
  int ntiles;
};

#include "pass_tma.cuh"

#ifdef PBL_PASS_PROFILE
// developer instrumentation (tools/pass_phases.py): cycle stamps of every 64th tile at the phase boundaries
__device__ long long g_pass_stamps[8][8192];
__device__ unsigned int g_pass_stamp_count;
#define PBL_STAMP(i)                                                                                  \
  do {                                                                                                \
    if (threadIdx.x == 0 && stamp_slot >= 0) g_pass_stamps[i][stamp_slot] = clock64();                \
  } while (0)
#else
#define PBL_STAMP(i)
#endif

struct PassSmem {
  uint64_t* big;      // [TILE] 8-byte member
  uint32_t* small_;   // [TILE] 4-byte member
  uint32_t* hist;     // [NWARPS][kRadix]
  uint32_t* goff;     // [kRadix] global slot - tile position
  uint32_t* bstart;   // [kRadix] tile-local bin start
  uint32_t* wsum;     // [8]
};

template <int BLOCK, int ITEMS, bool FULL>
__device__ __forceinline__ void pass_body(const PassArgs& a, const PassSmem& sm, const int col,
                                          const uint32_t tile, const uint32_t nvalid, const int src,
                                          const int dst, const uint32_t dshift, const KeyMap& map, const int stamp_slot) {
  constexpr int TILE = BLOCK * ITEMS;
  constexpr int NWARPS = BLOCK / 32;
  uint64_t* s_keys = sm.big;
  uint32_t* s_vals = sm.small_;
  const int tid = threadIdx.x;
  const uint32_t n = a.n;
  const uint32_t tile_start = tile * (uint32_t)TILE;
  const uint32_t warp = tid >> 5, lane = tid & 31;
  const uint32_t pos0 = warp * (ITEMS * 32) + lane;

  // ---- load keys and take their digits; padding (positions >= nvalid, partial tiles only) is
  //      forced into the last bin, where it sorts after every real key of the tile because it
  //      also has the highest positions ----
  uint64_t key[ITEMS];
  uint32_t dig[ITEMS];
  uint32_t negzero = 0;  // first pass (raw input): bit u set if item u was -0.0
  if (src == 0) {
    const double* colp = a.raw + (int64_t)col * a.col_stride + (int64_t)(tile_start + pos0) * a.row_stride;
    const int64_t step = 32 * a.row_stride;
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) {
      key[u] = 0ull;
      if (FULL || pos0 + u * 32 < nvalid) {
        bool nz;
        const uint64_t k = key_of_double(ld_stream_f64(colp + u * step), &nz);
        key[u] = compact_key(k, map);
        negzero |= (nz ? 1u : 0u) << u;
      }
    }
  } else {
    const uint64_t* kin = (src == 1 ? a.keysA : a.keysB) + (size_t)col * n + tile_start + pos0;
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) key[u] = (FULL || pos0 + u * 32 < nvalid) ? ld_stream_u64(kin + u * 32) : 0ull;
  }
#pragma unroll
  for (int u = 0; u < ITEMS; ++u) dig[u] = (uint32_t)(key[u] >> dshift) & (uint32_t)(kRadix - 1);
  if (!FULL) {
#pragma unroll
    for (int u = 0; u < ITEMS; ++u)
      if (pos0 + u * 32 >= nvalid) dig[u] = (uint32_t)(kRadix - 1);
  }

  // ---- rank inside the warp FIRST, against warp-private counters that start at zero: what the
  //      counters hold afterwards are the warp's digit counts, so no separate counting phase (one
  //      shared-memory reduction per key and a block barrier) is needed.
  //      (1) the mask of lanes holding the same digit, built from 8 ballots (one per digit bit;
  //      MATCH.ANY is avoided on purpose: its cost grows with the number of distinct digits in the
  //      warp and saturates the ADU pipe), (2) the highest lane of every digit group reads and bumps
  //      the group's counter -- plain load / store, the counters are private to the warp and a warp
  //      barrier orders item u's stores before item u+1's loads (a returning shared atomic costs ~2
  //      cycles per active lane here), (3) broadcast + lane offset. ----
  uint32_t* wh = sm.hist + warp * kRadix;
  uint32_t rank[ITEMS];
  {
    const uint32_t lt = lanemask_lt();
    uint32_t m[ITEMS];
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) {
      const uint32_t d = dig[u];
      uint32_t mm = 0xFFFFFFFFu;
#pragma unroll
      for (int b = 0; b < kRadixBits; ++b) {
        const bool bit = (d >> b) & 1u;
        const uint32_t bal = __ballot_sync(0xFFFFFFFFu, bit);
        mm &= bit ? bal : ~bal;
      }
      m[u] = mm;
    }
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) {
      uint32_t base = 0;
      if ((m[u] >> lane) == 1u) {  // highest lane of its group
        uint32_t* ctr = wh + dig[u];
        base = *ctr;
        *ctr = base + __popc(m[u]);
      }
      __syncwarp();
      rank[u] = base;
    }
#pragma unroll
    for (int u = 0; u < ITEMS; ++u)
      rank[u] = __shfl_sync(0xFFFFFFFFu, rank[u], 31 - __clz(m[u])) + __popc(m[u] & lt);
  }
  __syncthreads();
  PBL_STAMP(2);

  // ---- per bin: the warps' counts -> tile total, published for the tiles behind us; exclusive scan
  //      over warps and over bins; the counters are overwritten with (bin start in the tile + the
  //      keys of earlier warps in that bin), which is what a key adds to its in-warp rank ----
  uint32_t cnt = 0, bin_start = 0;
  uint32_t* st = a.status + (size_t)col * a.ntiles * kRadix;
  if (tid < kRadix) {
#pragma unroll
    for (int w = 0; w < NWARPS; ++w) cnt += sm.hist[w * kRadix + tid];
    if (!FULL && tid == kRadix - 1) cnt -= (uint32_t)TILE - nvalid;  // drop the padding keys (last in the last bin)
    st_relaxed_u32(&st[(size_t)tile * kRadix + tid], cnt | (tile == 0 ? kFlagInclusive : kFlagPartial));
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if (lane >= (uint32_t)d) incl += t;
    }
    if (lane == 31) sm.wsum[warp] = incl;
    bin_start = incl - cnt;
  }
  __syncthreads();
  if (tid < kRadix) {
#pragma unroll
    for (int w = 0; w < kRadix / 32; ++w)
      if ((uint32_t)w < warp) bin_start += sm.wsum[w];
    uint32_t run = bin_start;
#pragma unroll
    for (int w = 0; w < NWARPS; ++w) {
      const uint32_t c = sm.hist[w * kRadix + tid];
      sm.hist[w * kRadix + tid] = run;
      run += c;
    }
  }
  PBL_STAMP(3);
  __syncthreads();  // offsets visible to everyone
  PBL_STAMP(4);

  // ---- scatter to shared memory in digit order ----
#pragma unroll
  for (int u = 0; u < ITEMS; ++u) {
    rank[u] += wh[dig[u]];
    s_keys[rank[u]] = key[u];
  }
  if (src == 0) {
#pragma unroll
    for (int u = 0; u < ITEMS; ++u)
      s_vals[rank[u]] = (tile_start + pos0 + u * 32) | (((negzero >> u) & 1u) ? kNegZeroFlag : 0u);
  } else {
    uint32_t v[ITEMS];
    const uint32_t* vin = (src == 1 ? a.valsA : a.valsB) + (size_t)col * n + tile_start + pos0;
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) v[u] = (FULL || pos0 + u * 32 < nvalid) ? ld_stream_u32(vin + u * 32) : 0u;
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) s_vals[rank[u]] = v[u];
  }

  PBL_STAMP(5);
  // ---- exclusive prefix of this bin over all earlier tiles (they published long ago) ----
  if (tid < kRadix) {
    uint32_t excl = 0;
    if (tile != 0) {
      // walk back over the predecessors LB at a time: the LB status words are fetched together
      // (one L2 round trip per batch instead of one per predecessor), consumed in order, and the
      // walk stops at the first inclusive word; an unpublished word restarts the batch there
      constexpr int LB = 8;
      int64_t t = (int64_t)tile - 1;
      bool done = false;
      uint32_t spins = 0;
      while (!done) {
        uint32_t pre[LB];
#pragma unroll
        for (int i = 0; i < LB; ++i)
          pre[i] = (t - i >= 0) ? ld_relaxed_u32(&st[(size_t)(t - i) * kRadix + tid]) : kFlagInclusive;
#pragma unroll
        for (int i = 0; i < LB; ++i) {
          if (!done) {
            const uint32_t w = pre[i];
            if ((w & (kFlagInclusive | kFlagPartial)) == 0) {  // not published yet: poll again from here
              if (++spins > kSpinLimit) {
                atomicExch(&a.error_flag[kFlagWatchdog], 1u);
                done = true;
              }
              break;
            }
            excl += w & kValueMask;
            --t;
            if (w & kFlagInclusive) done = true;
          }
        }
      }
      st_relaxed_u32(&st[(size_t)tile * kRadix + tid], ((excl + cnt) & kValueMask) | kFlagInclusive);
    }
    const uint32_t base = a.bin_base_all[((size_t)col * kMaxPasses + a.pass) * kRadix + tid];
    sm.goff[tid] = base + excl - bin_start;  // + position in tile order = global slot
  }
  __syncthreads();
  PBL_STAMP(6);

  // ---- coalesced runs out to HBM ----
  uint64_t* out_big = (dst == 1 ? a.keysA : a.keysB) + (size_t)col * n;
  uint32_t* out_small = (dst == 1 ? a.valsA : a.valsB) + (size_t)col * n;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const uint32_t pos = j * BLOCK + tid;
    if (FULL || pos < nvalid) {
      const uint64_t k = s_keys[pos];
      const uint32_t g = sm.goff[(uint32_t)(k >> dshift) & (uint32_t)(kRadix - 1)] + pos;
      st_u64_at(out_big, g, k);
      st_u32_at(out_small, g, s_vals[pos]);
    }
  }
  PBL_STAMP(7);
}

template <int BLOCK, int ITEMS, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB)
partition_pass_kernel(const PassArgs a) {
  constexpr int TILE = BLOCK * ITEMS;
  constexpr int NWARPS = BLOCK / 32;
  static_assert(BLOCK >= kRadix && BLOCK % 32 == 0, "one thread per bin is assumed");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  PassSmem sm;
  sm.big = reinterpret_cast<uint64_t*>(smem_raw);
  sm.small_ = reinterpret_cast<uint32_t*>(sm.big + TILE);
  sm.hist = sm.small_ + TILE;
  sm.goff = sm.hist + NWARPS * kRadix;
  sm.bstart = sm.goff + kRadix;
  sm.wsum = sm.bstart + kRadix;
  uint32_t* s_tile = sm.wsum + 8;

  const int col = blockIdx.y;
  const int tid = threadIdx.x;
  // reads (keys, rows)[src] (or the raw column), writes (keys, rows)[dst]
  if (!a.plan[col].run[a.pass]) return;
  const int src = a.plan[col].src[a.pass];
  const int dst = (src == 1) ? 2 : 1;
  const KeyMap map = load_key_map(a.kminmax, col, a.window_bits);
  const uint32_t dshift = map.sh + (uint32_t)a.pass * kRadixBits;
  int stamp_slot = -1;
#ifdef PBL_PASS_PROFILE
  const long long t_entry = clock64();
#endif
  if (tid == 0) *s_tile = atomicAdd(&a.tile_counter[col], 1u);
  for (int i = tid; i < NWARPS * kRadix; i += BLOCK) sm.hist[i] = 0;
  __syncthreads();
  const uint32_t tile = *s_tile;
#ifdef PBL_PASS_PROFILE
  if (tid == 0) {
    if ((tile & 63u) == 17u && a.pass == 1) {
      stamp_slot = (int)atomicAdd(&g_pass_stamp_count, 1u);
      if (stamp_slot >= 8192) stamp_slot = -1;
    }
    if (stamp_slot >= 0) {
      g_pass_stamps[0][stamp_slot] = t_entry;
      g_pass_stamps[1][stamp_slot] = clock64();
    }
  }
#endif
  const uint32_t nvalid = min((uint32_t)TILE, a.n - tile * (uint32_t)TILE);
  if (nvalid == (uint32_t)TILE)
    pass_body<BLOCK, ITEMS, true>(a, sm, col, tile, nvalid, src, dst, dshift, map, stamp_slot);
  else
    pass_body<BLOCK, ITEMS, false>(a, sm, col, tile, nvalid, src, dst, dshift, map, stamp_slot);
}

// Second half of the scatter by row: out[row] = value for the (row, value) pairs the sort's consumer staged in
// the "other" ping-pong buffer, grouped by destination row window for long columns (scatter_prepare).  Blocks
// walk the column in order, so the windows being written at any moment total a few MB and stay in L2 until
// every line is complete.
__global__ void __launch_bounds__(256)
scatter_rows_kernel(const uint64_t* __restrict__ keysA, const uint64_t* __restrict__ keysB,
                    const uint32_t* __restrict__ valsA, const uint32_t* __restrict__ valsB,
                    const PassPlan* __restrict__ plan, uint32_t n,
                    double* __restrict__ out, int64_t out_row_stride, int64_t out_col_stride,
                    uint32_t pos_begin, uint32_t pos_end) {
  const int col = blockIdx.y;
  const int b = (plan[col].final_buf == 1) ? 2 : 1;
  const uint32_t* rows = (b == 1 ? valsA : valsB) + (size_t)col * n;
  const uint64_t* vals = (b == 1 ? keysA : keysB) + (size_t)col * n;
  double* outc = out + (int64_t)col * out_col_stride;
  constexpr int U = 8;
  const uint32_t base = pos_begin + blockIdx.x * (256u * U) + threadIdx.x;  // pos_end <= n < 2^31: no overflow
  uint32_t r[U];
  uint64_t v[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    uint32_t i = base + u * 256u;
    if (i < pos_end) {  // evict-first: the pairs stream through L2 once, the output lines must stay
      r[u] = __ldcs(rows + i);
      v[u] = __ldcs((const unsigned long long*)vals + i);
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    uint32_t i = base + u * 256u;
    if (i < pos_end) outc[(int64_t)r[u] * out_row_stride] = __longlong_as_double((long long)v[u]);
  }
}

// The one-tile-per-block digit pass: 256 threads x 16 keys, 3 blocks per SM.
constexpr int kPassBlock = 256;
constexpr int kPassItems = 16;
constexpr int kPassTile = kPassBlock * kPassItems;

int launch_pass(const PassArgs& a, int ncols, cudaStream_t stream) {
  auto kern = partition_pass_kernel<kPassBlock, kPassItems, 3>;
  constexpr size_t smem = (size_t)kPassTile * 12 + (size_t)(kPassBlock / 32) * kRadix * 4 + 2 * kRadix * 4 + 8 * 4 + 16;
  static bool attr_set = false;
  if (!attr_set) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  kern<<<dim3(a.ntiles, ncols), kPassBlock, smem, stream>>>(a);
  return kOk;
}

int next_epoch(const SortBuffers& buf, size_t status_bytes, cudaStream_t stream, uint32_t* out) {
  // a fresh tag for every launch; the array is cleared once per 2^28 launches (and at allocation)
  if (*buf.epoch >= (1u << 28)) {
    PBL_CUDA_CHECK(cudaMemsetAsync(buf.status, 0, status_bytes, stream));
    *buf.epoch = 0;
  }
  *out = ++*buf.epoch;
  return kOk;
}

int launch_pass_tma(const PassArgs& a, int ncols, const SortBuffers& buf, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(pass_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTmaSmemBytes));
    attr_set = true;
  }
  TmaArgs t;
  t.p = a;
  t.maps = buf.maps;
  t.status64 = reinterpret_cast<uint64_t*>(buf.status);
  t.ticket = a.tile_counter;
  t.total_tiles = (uint32_t)ncols * (uint32_t)a.ntiles;
  t.ncols = (uint32_t)ncols;
  t.ncols_interleave = std::min<uint32_t>((uint32_t)ncols, kInterleaveWidth);
  PBL_RETURN_IF(next_epoch(buf, sort_status_bytes(ncols, a.n), stream, &t.epoch));
  const unsigned grid = (unsigned)std::min<size_t>((size_t)2 * num_sms(), (size_t)t.total_tiles);
  pass_tma_kernel<<<grid, kTileThreads, kTmaSmemBytes, stream>>>(t);
  return kOk;
}

struct PassEvent {
  cudaEvent_t start, stop;
  int64_t keys;
};
bool g_profile = false;
std::vector<PassEvent> g_events;

}  // namespace

#ifdef PBL_PASS_PROFILE
}  // namespace pbl
extern "C" __attribute__((visibility("default"))) int pbl_debug_pass_stamps(long long* out, int cap) {
  unsigned int cnt = 0;
  cudaMemcpyFromSymbol(&cnt, pbl::g_pass_stamp_count, sizeof(cnt));
  int take = (int)std::min<unsigned int>(cnt, (unsigned int)std::min(cap, 8192));
  for (int i = 0; i < 8; ++i)
    cudaMemcpyFromSymbol(out + (size_t)i * cap, pbl::g_pass_stamps, (size_t)take * 8, (size_t)i * 8192 * 8);
  unsigned int zero = 0;
  cudaMemcpyToSymbol(pbl::g_pass_stamp_count, &zero, sizeof(zero));
  return take;
}
namespace pbl {
#endif

#ifdef PBL_TILE_STATS
}  // namespace pbl
// developer instrumentation: read and clear the tile statistics (tile_pipeline.cuh)
extern "C" __attribute__((visibility("default"))) int pbl_debug_tile_stats(unsigned long long* out) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, pbl::g_tile_stats, 8 * sizeof(unsigned long long));
  unsigned long long zero[8] = {0};
  cudaMemcpyToSymbol(pbl::g_tile_stats, zero, sizeof(zero));
  return 0;
}
namespace pbl {
#endif

void sort_profile_enable(bool on) { g_profile = on; }

void sort_profile_read(int64_t* launches, double* total_ms, int64_t* keys) {
  int64_t nl = 0, nk = 0;
  double ms = 0.0;
  for (auto& e : g_events) {
    float t = 0.f;
    if (cudaEventSynchronize(e.stop) == cudaSuccess &&
        cudaEventElapsedTime(&t, e.start, e.stop) == cudaSuccess) {
      ++nl;
      ms += t;
      nk += e.keys;
    }
    cudaEventDestroy(e.start);
    cudaEventDestroy(e.stop);
  }
  g_events.clear();
  if (launches) *launches = nl;
  if (total_ms) *total_ms = ms;
  if (keys) *keys = nk;
}

// The long-column rule.  The persistent bulk-async kernels (pass_tma.cuh, post_tma.cuh) everywhere, except
// on columns longer than 3e8 rows (the multi-GPU driver's shapes), where the one-tile-per-block kernels are the
// faster ones:
//   consumer: the 32-bit windows of such columns are dense (1.5 keys per window value at n = 8e8) and
//     post_sort_kernel (ic.cu: 2048-key tiles, run extents from ballot masks) wins: 108 vs 127 ms per
//     rank_scores of 2 x 8e8 keys (profiles/r2_narrow_launch_experiments.txt);
//   digit pass, on launches of one or two such columns: all tiles in flight share one look-back chain, the
//     ticket taken a tile ahead buys nothing, and partition_pass_kernel wins (8 GPUs, 8e8-row columns: 5.97
//     vs 6.35 ms per pass, profiles/r1_bench_n8.json vs r2_bench_n8_weak.json; one GPU, same shape: 125.5 vs
//     127.4 ms per rank_scores).
// The one-tile-per-block kernels keep 30-bit counts in their look-back words: at most kMaxSortNClassic rows.
// PBL_CLASSIC_ABOVE=<rows> moves the 3e8 threshold (read per call: the tests run the classic kernels on small
// columns with it).
static uint64_t classic_above() {
  const char* e = getenv("PBL_CLASSIC_ABOVE");
  return (e && e[0]) ? strtoull(e, nullptr, 10) : 300000000ull;
}
bool sort_classic_consumer(uint32_t n) { return n > classic_above() && n <= kMaxSortNClassic; }
bool sort_classic_pass(uint32_t n, int ncols) { return ncols <= 2 && sort_classic_consumer(n); }

size_t sort_status_bytes(int ncols, uint32_t n) {
  // sized for the smallest tile that uses the words: the 2048 keys of post_sort_kernel (ic.cu)
  constexpr size_t tile = 2048;
  size_t ntiles = ((size_t)n + tile - 1) / tile;
  return (size_t)ncols * ntiles * kRadix * sizeof(uint64_t);  // 64-bit epoch-tagged words (pass_tma.cuh)
}

int sort_columns_f64(const double* in, int64_t row_stride, int64_t col_stride, uint32_t n,
                     int ncols, int window_bits, const SortBuffers& buf, cudaStream_t stream) {
  if (n == 0 || ncols <= 0) return kOk;
  if (n > kMaxSortN) {
    set_last_error("sort_columns_f64: n exceeds 2^31-1 rows per column");
    return kBadShape;
  }
  if (window_bits != 32 && window_bits != 64) {
    set_last_error("sort_columns_f64: window_bits must be 32 or 64");
    return kBadShape;
  }
  const int npasses = window_bits / kRadixBits;
  PBL_CUDA_CHECK(cudaMemsetAsync(buf.hist, 0, (size_t)ncols * kMaxPasses * kRadix * 4, stream));
  PBL_CUDA_CHECK(cudaMemsetAsync(buf.tile_counter, 0, (size_t)ncols * (kMaxPasses + 1) * 4, stream));

  const int sms = num_sms();
  {
    constexpr int MB = 512, MU = 8;
    int per_col = (int)(((size_t)n + MB * MU - 1) / (MB * MU));
    int want = (sms * 4 + ncols - 1) / ncols;
    dim3 grid((unsigned)std::max(1, std::min(per_col, want)), (unsigned)ncols);
    minmax_init_kernel<<<(ncols + 255) / 256, 256, 0, stream>>>(buf.kminmax, ncols);
    PBL_LAUNCH_CHECK();
    col_minmax_kernel<MB, MU><<<grid, MB, 0, stream>>>(in, row_stride, col_stride, n, buf.kminmax,
                                                      buf.error_flag);
    PBL_LAUNCH_CHECK();
  }
  {
    constexpr int HB = 512, HU = 4;
    int per_col = (int)(((size_t)n + HB * HU - 1) / (HB * HU));
    int want = (sms * 4 + ncols - 1) / ncols;  // ~4 resident blocks per SM over the batch
    dim3 grid((unsigned)std::max(1, std::min(per_col, want)), (unsigned)ncols);
    if (npasses == 4)
      sort_hist_kernel<HB, HU, 4><<<grid, HB, 0, stream>>>(in, row_stride, col_stride, n, buf.hist,
                                                          buf.kminmax, window_bits);
    else
      sort_hist_kernel<HB, HU, 8><<<grid, HB, 0, stream>>>(in, row_stride, col_stride, n, buf.hist,
                                                          buf.kminmax, window_bits);
    PBL_LAUNCH_CHECK();
  }
  sort_scan_kernel<<<ncols, kRadix, 0, stream>>>(buf.hist, buf.plan, n, npasses, buf.kminmax, window_bits, buf.maps);
  PBL_LAUNCH_CHECK();

  const bool classic = sort_classic_pass(n, ncols);
  const int tile = classic ? kPassTile : kTmaTile;
  PassArgs a{};
  a.raw = in;
  a.row_stride = row_stride;
  a.col_stride = col_stride;
  a.keysA = buf.keysA;
  a.keysB = buf.keysB;
  a.valsA = buf.valsA;
  a.valsB = buf.valsB;
  a.bin_base_all = buf.hist;
  a.status = buf.status;
  a.plan = buf.plan;
  a.kminmax = buf.kminmax;
  a.error_flag = buf.error_flag;
  a.n = n;
  a.window_bits = window_bits;
  a.ntiles = (int)(((size_t)n + tile - 1) / tile);
  for (int pass = 0; pass < npasses; ++pass) {
    // the one-tile-per-block pass keeps 32-bit words [ncols][ntiles][256]: clear those, not the whole allocation
    // (the bulk-async pass uses epoch-tagged words: nothing to clear)
    if (classic) PBL_CUDA_CHECK(cudaMemsetAsync(buf.status, 0, (size_t)ncols * a.ntiles * kRadix * 4, stream));
    a.pass = pass;
    a.tile_counter = buf.tile_counter + (size_t)pass * ncols;
    PassEvent ev{};
    if (g_profile) {
      cudaEventCreate(&ev.start);
      cudaEventCreate(&ev.stop);
      ev.keys = (int64_t)n * ncols;
      cudaEventRecord(ev.start, stream);
    }
    if (classic)
      PBL_RETURN_IF(launch_pass(a, ncols, stream));
    else
      PBL_RETURN_IF(launch_pass_tma(a, ncols, buf, stream));
    if (g_profile) {
      cudaEventRecord(ev.stop, stream);
      g_events.push_back(ev);
    }
    PBL_LAUNCH_CHECK();
  }
  return kOk;
}

static int scatter_shift_for(uint32_t n) {
  // <= 256 destination windows; a single window (no partition pass) below 2^19 rows
  int bits = 0;
  while (bits < 32 && (1ull << bits) < (uint64_t)n) ++bits;
  return bits > 19 ? std::max(19, bits - 8) : 32;
}

// Scatter by row, second half.  The consumer of the sort (post_sort_kernel / post_tma_kernel in ic.cu) leaves
// (row, value) pairs in the "other" ping-pong buffer, already grouped by destination window when
// scatter_prepare() returned a shift < 32; this kernel delivers value -> out[row].
int scatter_prepare(uint32_t n, int ncols, const SortBuffers& buf, int64_t row_stride, int consumer_tile,
                    int* shift_out, int* ntiles_out, uint32_t** tile_counter_out, uint32_t* epoch_out,
                    cudaStream_t stream) {
  const int shift = row_stride == 1 ? scatter_shift_for(n) : 32;
  const int ntiles = (int)(((size_t)n + consumer_tile - 1) / consumer_tile);
  *shift_out = shift;
  *ntiles_out = ntiles;
  *tile_counter_out = buf.tile_counter + (size_t)kMaxPasses * ncols;
  *epoch_out = 0;
  if (shift < 32) {
    PBL_RETURN_IF(next_epoch(buf, sort_status_bytes(ncols, n), stream, epoch_out));
    PBL_CUDA_CHECK(cudaMemsetAsync(*tile_counter_out, 0, (size_t)ncols * 4, stream));
  }
  return kOk;
}

int scatter_rows(uint32_t n, int ncols, const SortBuffers& buf, double* out, int64_t row_stride,
                 int64_t col_stride, cudaStream_t stream, uint32_t pos_begin, uint32_t pos_end) {
  pos_end = std::min(pos_end, n);
  if (n == 0 || ncols <= 0 || pos_begin >= pos_end) return kOk;
  dim3 grid((unsigned)(((size_t)(pos_end - pos_begin) + 2047) / 2048), (unsigned)ncols);
  scatter_rows_kernel<<<grid, 256, 0, stream>>>(buf.keysA, buf.keysB, buf.valsA, buf.valsB, buf.plan,
                                               n, out, row_stride, col_stride, pos_begin, pos_end);
  PBL_LAUNCH_CHECK();
  return kOk;
}

}  // namespace pbl
