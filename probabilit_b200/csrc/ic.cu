// Iman-Conover correlator on one B200 (reference: src/probabilit/correlation.py:368-425).
//
//   stage rank_scores  : per-column sort of X  -> tie-run average ranks -> van der Waerden scores
//                        scattered back to row order, plus np.sort(X[:,c])      (:394-395, :423)
//   stage gram         : fp64 Gram  S^T S  and column sums of the scores        (:398 np.corrcoef)
//   stage solve        : corrcoef normalisation + clip, single-block Cholesky Q, T = Q^-T P^T
//                                                                               (:398-414)
//   stage transform    : correlated = scores @ T  (T upper triangular), in place (:409-414)
//   stage rank_gather  : per-column sort of the correlated scores -> tie-run midpoint index
//                        -> Y[row, c] = sortedX[c][index]                       (:419-423)
//
// Everything is column-major on the device ([k][n], one contiguous run per variable), which is
// what the graph path hands over (np.vstack(...).T, reference src/probabilit/modeling.py:580).
#include "ic.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cooperative_groups.h>

#include "ndtri.cuh"
#include "tile_pipeline.cuh"

namespace cg = cooperative_groups;

namespace pbl {

namespace {

// ======================================================================================
// post-sort kernel: tie runs on the sorted column, then either scores (MODE 0) or the gather
// of the sorted marginal (MODE 1)
// ======================================================================================
constexpr int kPostBlock = 512;
constexpr int kPostItems = 4;
constexpr int kPostTile = kPostBlock * kPostItems;
constexpr int kHalo = 64;                      // window values may repeat in runs of < kHalo keys
constexpr int kWin = kPostTile + 2 * kHalo;
constexpr int kMaxRun = 32;                    // ... and are re-ordered here when shorter than this
constexpr size_t kPostSmem = (size_t)kWin * 8 * 2 + (size_t)kWin * 4 * 2 + (size_t)kPostTile * 4 * 2 + 128 +
                             2 * kRadix * 4 + 16 + (kWin / 32) * 4 + sizeof(KeyMap);
static_assert(kWin % 32 == 0 && kHalo >= 2 * kMaxRun - 1, "run masks are per 32 slots; halo covers two runs");

__device__ __forceinline__ uint32_t block_excl_prefix_max(uint32_t v, uint32_t* s_w) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
    if (lane >= (uint32_t)d) incl = max(incl, t);
  }
  if (lane == 31) s_w[warp] = incl;
  uint32_t excl = __shfl_up_sync(0xFFFFFFFFu, incl, 1);
  if (lane == 0) excl = 0;
  __syncthreads();
  for (uint32_t w = 0; w < warp; ++w) excl = max(excl, s_w[w]);
  __syncthreads();
  return excl;
}

__device__ __forceinline__ uint32_t block_excl_suffix_min(uint32_t v, uint32_t* s_w) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_down_sync(0xFFFFFFFFu, incl, d);
    if (lane + d < 32) incl = min(incl, t);
  }
  if (lane == 0) s_w[warp] = incl;
  uint32_t excl = __shfl_down_sync(0xFFFFFFFFu, incl, 1);
  if (lane == 31) excl = 0xFFFFFFFFu;
  __syncthreads();
  for (uint32_t w = warp + 1; w < kPostBlock / 32; ++w) excl = min(excl, s_w[w]);
  __syncthreads();
  return excl;
}

// Consumes one column that the windowed sort left ordered by window value (sort.cuh):
//  (1) completes the order inside every run of equal window values (runs of < kHalo keys are
//      re-ordered by their full 64-bit keys in shared memory; a longer run of *distinct* keys
//      raises kFlagWindowRetry and the caller repeats the sort on all 64 bits);
//  (2) finds the tie runs (equal values) and, for every sorted position p, the value its source
//      row must receive:
//      MODE 0: ndtri(average_rank / (n+1)), and sortedX[col][p] = the p-th smallest input
//              (scipy.stats.rankdata 'average' + norm.ppf, correlation.py:394-395; np.sort, :423)
//      MODE 1: sortedX[col][run_start + (run_len-1)/2]
//              (rankdata(...).astype(int) - 1 then the gather, correlation.py:422-423)
//  (3) stages value and row, in sorted order, in the "other" ping-pong buffer (the one that does
//      not hold the sorted keys); scatter_by_row (sort.cu) then delivers value -> row.
// van der Waerden scores of an untied column in sorted order: vdw[p] = ndtri((p+1)/(n+1)).
// They depend on n only, so the table is built once per plan and shared by all columns
// (the per-element ndtri -- several fp64 divisions, log, sqrt -- is then paid for ties only).
__global__ void __launch_bounds__(256) vdw_table_kernel(uint32_t n, double* __restrict__ vdw) {
  for (uint64_t p = (uint64_t)blockIdx.x * 256 + threadIdx.x; p < n; p += (uint64_t)gridDim.x * 256)
    vdw[p] = ndtri(__ddiv_rn((double)(p + 1), (double)((uint64_t)n + 1ull)));
}

template <int MODE>
__global__ void __launch_bounds__(kPostBlock, 3)
post_sort_kernel(uint64_t* keysA, uint64_t* keysB, uint32_t* valsA, uint32_t* valsB,
                 const PassPlan* __restrict__ plan, const uint64_t* __restrict__ kminmax,
                 int window_bits, uint32_t n, double* __restrict__ sortedX,
                 const double* __restrict__ vdw, uint32_t* __restrict__ flags, int col_base,
                 int part_shift, uint64_t* __restrict__ status, uint32_t* __restrict__ tile_counter,
                 int ntiles, uint32_t epoch) {
  extern __shared__ __align__(16) unsigned char psm[];
  uint64_t* s_raw = reinterpret_cast<uint64_t*>(psm);        // [kWin] keys as the sort left them
  uint64_t* s_key = s_raw + kWin;                            // [kWin] completed order
  uint32_t* s_rawv = reinterpret_cast<uint32_t*>(s_key + kWin);  // [kWin] rows as sorted
  uint32_t* s_row = s_rawv + kWin;                           // [kWin] rows, completed order
  uint32_t* s_start = s_row + kWin;                          // [kPostTile]
  uint32_t* s_end = s_start + kPostTile;                     // [kPostTile]
  uint32_t* s_w = s_end + kPostTile;                         // [kPostBlock / 32]
  uint32_t* s_lohi = s_w + kPostBlock / 32;                  // [2]
  uint32_t* s_bstart = s_lohi + 4;                           // [kRadix]
  uint32_t* s_goff = s_bstart + kRadix;                      // [kRadix]
  // warp-private window counters of the fused partition: [16 warps][kRadix], on top of s_start / s_end
  // (dead once step (3) has read them)
  uint32_t* s_hist = s_start;
  static_assert(2 * kPostTile == (kPostBlock / 32) * kRadix, "the counters alias s_start + s_end exactly");
  uint32_t* s_ticket = s_goff + kRadix;                      // [1] (+3 pad)
  uint32_t* s_mask = s_ticket + 4;                           // [kWin / 32] "same window as the slot to the left"
  KeyMap* s_map = reinterpret_cast<KeyMap*>(s_mask + kWin / 32);  // 8-byte aligned: all sizes above are
  // staging of the partitioned (value, row) pairs: the raw window copies are dead by then
  double* s_pval = reinterpret_cast<double*>(s_raw);         // [kPostTile]
  uint32_t* s_prow = s_rawv;                                 // [kPostTile]

  const int col = blockIdx.y;
  const int tid = threadIdx.x;
  const bool partition = part_shift < 32;
  // tiles take tickets so that the look-back between tiles can never wait on a tile that has not
  // started (blockIdx order is not a scheduling guarantee)
  uint32_t tile = blockIdx.x;
  if (partition && tid == 0) *s_ticket = atomicAdd(&tile_counter[col], 1u);
  if (tid == 32) *s_map = load_key_map(kminmax, col, window_bits);  // once per block, not per thread
  __syncthreads();
  if (partition) tile = *s_ticket;
  const KeyMap map = *s_map;
  const int fb = plan[col].final_buf;
  const uint64_t* keys = (fb == 1 ? keysA : keysB) + (size_t)col * n;
  const uint32_t* rows_in = (fb == 1 ? valsA : valsB) + (size_t)col * n;
  double* stage = reinterpret_cast<double*>((fb == 1 ? keysB : keysA) + (size_t)col * n);
  uint32_t* rows_out = (fb == 1 ? valsB : valsA) + (size_t)col * n;
  double* sx = sortedX + (size_t)col * n;
  const uint32_t tile_start = tile * (uint32_t)kPostTile;
  const uint32_t nvalid = min((uint32_t)kPostTile, n - tile_start);
  const int64_t wbase = (int64_t)tile_start - kHalo;  // global index of window slot 0

  // the position-indexed operand of step (3) is fetched now, together with the window, so that its
  // HBM latency is not a separate link of the tile's dependency chain: the van der Waerden score of
  // the position (MODE 0) / the sorted marginal at the position (MODE 1; used unless the position
  // sits in a tie-run, whose midpoint is then fetched instead)
  double pre_val[kPostItems];
#pragma unroll
  for (int j = 0; j < kPostItems; ++j) {
    const uint32_t p = j * kPostBlock + tid;
    pre_val[j] = 0.0;
    if (MODE != 2 && p < nvalid) pre_val[j] = ld_stream_f64((MODE == 0 ? vdw : sx) + tile_start + p);
  }
  for (int i = tid; i < kWin; i += kPostBlock) {
    int64_t g = wbase + i;
    uint64_t k = 0;
    uint32_t r = 0;
    if (g >= 0 && g < (int64_t)n) {
      k = ld_stream_u64(keys + g);
      r = ld_stream_u32(rows_in + g);
    }
    s_raw[i] = k;
    s_rawv[i] = r;
  }
  __syncthreads();

  // ---- (1) complete the order inside runs of equal window values ----
  // (1a) one bit per slot: "same window value as the slot to its left" (ballot words in shared memory)
  const int lo_i = (int)max((int64_t)0, -wbase);                  // first slot inside the column
  const int hi_i = (int)min((int64_t)kWin, (int64_t)n - wbase);   // one past the last such slot
  for (int i = tid; i < kWin; i += kPostBlock) {  // kWin and the tail of the loop are whole warps
    const bool sl = i > lo_i && i < hi_i && same_window(s_raw[i], s_raw[i - 1], map);
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, sl);
    if ((tid & 31) == 0) s_mask[i >> 5] = m;
  }
  __syncthreads();
  // (1b) a slot's run is the stretch of set bits around it: its extent comes from bit scans, and only
  //      members of a run (a fifth of the keys at 0.2 keys per window value) walk it.  Runs of up to
  //      kMaxRun keys are re-ordered by their full keys (equal keys keep their order); every member sees
  //      the whole run (kHalo >= 2 kMaxRun - 1 slots on either side of the tile), so all reach the same
  //      verdict.  A longer run is left as it is -- fine if it is pure (a tie run) -- and any adjacent
  //      pair of DIFFERENT keys inside it raises kFlagWindowRetry in the tile that owns either key.
  int retry = 0, tie = 0;
  for (int i = tid; i < kWin; i += kPostBlock) {
    if (i < lo_i || i >= hi_i) continue;
    const uint64_t my = s_raw[i];
    int dst = i;
    const int c = i >> 5, l = i & 31;
    const uint32_t cur = s_mask[c];
    const uint32_t prev = c > 0 ? s_mask[c - 1] : 0u;
    const uint32_t next = c + 1 < kWin / 32 ? s_mask[c + 1] : 0u;
    const uint64_t left = (((uint64_t)cur << 32) | prev) << (31 - l);      // bit 63 = this slot's flag
    const uint64_t right = (((uint64_t)next << 32) | cur) >> (l + 1);      // bit 0 = flag of slot i + 1
    if ((left >> 63) | (right & 1ull)) {
      const int L = __clzll((long long)~left);                            // set flags at i, i-1, ...
      const int R = (~right) ? __ffsll((long long)~right) - 1 : 64;        // set flags at i+1, i+2, ...
      if (L + R + 1 <= kMaxRun) {
        uint32_t cnt = 0;
        for (int j = i - L; j <= i + R; ++j) {
          const uint64_t kj = s_raw[j];
          cnt += (kj < my || (kj == my && j < i)) ? 1u : 0u;
          tie |= (kj == my && j != i) ? 1 : 0;
        }
        dst = i - L + (int)cnt;
      } else if (L > 0) {
        const bool differs = s_raw[i - 1] != my;
        tie |= differs ? 0 : 1;
        if (differs && i >= kHalo && i - 1 < kHalo + (int)nvalid) retry = 1;
      }
    }
    s_key[dst] = my;
    s_row[dst] = s_rawv[i];
  }
  if (retry) flags[kFlagWindowRetry] = 1u;

  // ---- (2) tie runs.  teq(q): tile position q holds the same value as position q-1
  //      (q = 0 .. nvalid; positions outside the column never tie).  Keys are canonical
  //      (-0.0 folded onto +0.0), so key equality is value equality.  Equal keys share a window value,
  //      so step (1) has seen every tie (possibly one that lies in the halo only: harmless). ----
  auto teq = [&](uint32_t q) -> bool {
    const int64_t g = (int64_t)tile_start + q;  // global index of position q
    if (g <= 0 || g >= (int64_t)n) return false;
    return s_key[kHalo + q] == s_key[kHalo + q - 1];
  };
  tie = __syncthreads_or(tie);

  if (tie) {
    // blocked arrangement: thread t owns positions t*ITEMS .. t*ITEMS+ITEMS-1
    uint32_t st[kPostItems], en[kPostItems];
    uint32_t run = 0;
#pragma unroll
    for (int i = 0; i < kPostItems; ++i) {
      uint32_t p = tid * kPostItems + i;
      uint32_t v = 0;
      if (p < nvalid && !teq(p)) v = tile_start + p + 1;  // head: pos+1
      run = max(run, v);
      st[i] = run;
    }
    uint32_t pre = block_excl_prefix_max(run, s_w);
    run = 0xFFFFFFFFu;
#pragma unroll
    for (int i = kPostItems - 1; i >= 0; --i) {
      uint32_t p = tid * kPostItems + i;
      uint32_t v = 0xFFFFFFFFu;
      if (p < nvalid && !teq(p + 1)) v = tile_start + p;  // tail: pos
      run = min(run, v);
      en[i] = run;
    }
    uint32_t suf = block_excl_suffix_min(run, s_w);
    // tie runs that cross the tile boundary: binary search on the window value in the column
    // (valid because such a run is pure: any impure long run has raised kFlagWindowRetry)
    if (tid == 0) {
      uint32_t lo = tile_start, hi = tile_start + nvalid - 1;
      if (teq(0)) {
        const uint64_t w = window_value(s_key[kHalo], map);
        uint32_t a = 0, b = tile_start;  // first q in [0, tile_start) with window(q) >= w
        while (a < b) {
          uint32_t mid = a + (b - a) / 2;
          if (window_value(keys[mid], map) < w) a = mid + 1; else b = mid;
        }
        lo = a;
      }
      if (teq(nvalid)) {
        const uint64_t w = window_value(s_key[kHalo + nvalid - 1], map);
        uint32_t a = tile_start + nvalid, b = n;  // first q with window(q) > w
        while (a < b) {
          uint32_t mid = a + (b - a) / 2;
          if (window_value(keys[mid], map) > w) b = mid; else a = mid + 1;
        }
        hi = a - 1;
      }
      s_lohi[0] = lo;
      s_lohi[1] = hi;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kPostItems; ++i) {
      uint32_t p = tid * kPostItems + i;
      if (p < nvalid) {
        uint32_t s = max(st[i], pre);
        uint32_t e = min(en[i], suf);
        s_start[p] = (s == 0) ? s_lohi[0] : s - 1;
        s_end[p] = (e == 0xFFFFFFFFu) ? s_lohi[1] : e;
      }
    }
    __syncthreads();
  }

  // ---- (3) the value every source row must receive ----
  double out_val[kPostItems];
  uint32_t out_row[kPostItems];
#pragma unroll
  for (int j = 0; j < kPostItems; ++j) {
    uint32_t p = j * kPostBlock + tid;
    out_val[j] = 0.0;
    out_row[j] = 0;
    if (p < nvalid) {
      uint32_t g = tile_start + p;
      uint32_t s = g, e = g;
      if (tie) {
        s = s_start[p];
        e = s_end[p];
      }
      const uint32_t row = s_row[kHalo + p];
      out_row[j] = row & kRowMask;
      if (MODE == 2) {
        // scipy.stats.rankdata(x) itself (average ranks as doubles): the Spearman mode of
        // CorrelationMatrix, correlation.py:835-837
        out_val[j] = (double)((uint64_t)s + (uint64_t)e + 2ull) * 0.5;
      } else if (MODE == 0) {
        double sc;
        if (s == e) {
          sc = pre_val[j];  // untied: the score depends on the position only
        } else {
          double avg = (double)((uint64_t)s + (uint64_t)e + 2ull) * 0.5;
          sc = ndtri(__ddiv_rn(avg, (double)((uint64_t)n + 1ull)));
        }
        out_val[j] = sc;
        sx[g] = (row & kNegZeroFlag) ? -0.0 : key_to_double(expand_key(s_key[kHalo + p], map));
        if ((row & kNegZeroFlag) && col + col_base == 0) flags[kFlagNegZeroCol0] = 1u;
      } else {
        uint32_t m = s + (e - s) / 2;
        out_val[j] = (m == g) ? pre_val[j] : sx[m];
      }
    }
  }
  if (!partition) {  // short columns: scatter_rows_kernel delivers straight from sorted order
#pragma unroll
    for (int j = 0; j < kPostItems; ++j) {
      uint32_t p = j * kPostBlock + tid;
      if (p < nvalid) {
        rows_out[tile_start + p] = out_row[j];
        stage[tile_start + p] = out_val[j];
      }
    }
    return;
  }

  // ---- (4) first half of the scatter by row, fused: group the tile's (row, value) pairs by
  //      destination window (row >> part_shift, <= 256 windows of L2 size) with a chained scan
  //      between tiles, like the digit pass but without an extra round trip of the pairs through
  //      HBM.  In-warp ranking by ballots against warp-private counters (rank.cuh) instead of returning
  //      shared atomics on block-wide counters (~2 cycles per lane on B200: 43 % of this kernel). ----
  if (tie) __syncthreads();  // step (3) has read s_start / s_end, which the counters overwrite
  const uint32_t lane = tid & 31, warp = tid >> 5;
  uint32_t* wh = s_hist + warp * kRadix;
  {
    const uint4 z = make_uint4(0, 0, 0, 0);
    reinterpret_cast<uint4*>(wh)[lane] = z;
    reinterpret_cast<uint4*>(wh)[lane + 32] = z;
  }
  __syncwarp();
  uint32_t dig[kPostItems], slot[kPostItems];
#pragma unroll
  for (int j = 0; j < kPostItems; ++j) dig[j] = out_row[j] >> part_shift;
  if (nvalid == (uint32_t)kPostTile) {
    warp_rank_digits<kPostItems>(dig, wh, slot, lane);
  } else {
    bool valid[kPostItems];
#pragma unroll
    for (int j = 0; j < kPostItems; ++j) valid[j] = j * kPostBlock + tid < nvalid;
    warp_rank_digits_masked<kPostItems>(dig, valid, wh, slot, lane);
  }
  __syncthreads();
  uint32_t cnt = 0, bin_start = 0;
  uint64_t* st = status + (size_t)col * ntiles * kRadix;
  const uint64_t tag = (uint64_t)epoch << 34;
  if (tid < kRadix) {
#pragma unroll
    for (int w = 0; w < kPostBlock / 32; ++w) cnt += s_hist[w * kRadix + tid];
    st_relaxed_u64(&st[(size_t)tile * kRadix + tid], tag | (tile == 0 ? kStatusInclusive : kStatusPartial) | cnt);
  }
  {
    // exclusive scan of the 256 counts (threads >= 256 carry zeros)
    uint32_t incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
      if (lane >= (uint32_t)d) incl += t;
    }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    bin_start = incl - cnt;
    for (uint32_t w = 0; w < warp; ++w) bin_start += s_w[w];
  }
  if (tid < kRadix) {  // the counters become (window start in the tile + pairs of earlier warps in the window)
    uint32_t run = bin_start;
#pragma unroll
    for (int w = 0; w < kPostBlock / 32; ++w) {
      const uint32_t c = s_hist[w * kRadix + tid];
      s_hist[w * kRadix + tid] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kPostItems; ++j) {
    uint32_t p = j * kPostBlock + tid;
    if (p < nvalid) {
      const uint32_t q = wh[dig[j]] + slot[j];
      s_pval[q] = out_val[j];
      s_prow[q] = out_row[j];
    }
  }
  if (tid < kRadix) {
    const uint32_t excl = lookback_u64(st, tile, epoch, cnt, flags);
    const uint64_t b = (uint64_t)tid << part_shift;  // rows are a permutation of 0..n-1
    const uint32_t base = (uint32_t)(b < n ? b : n);
    s_goff[tid] = base + excl - bin_start;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kPostItems; ++j) {
    uint32_t p = j * kPostBlock + tid;
    if (p < nvalid) {
      const uint32_t r = s_prow[p];
      const uint32_t g = s_goff[r >> part_shift] + p;
      rows_out[g] = r;
      stage[g] = s_pval[p];
    }
  }
}

#include "post_tma.cuh"

// ======================================================================================
// Gram: per (row block, column-tile pair) partial sums of s_i s_j and of s_i, then a fixed-order
// reduction over row blocks (deterministic: no floating-point atomics).
// Thread grid TG x TG, 4x4 outputs per thread, 256/TG^2 row groups per block.
// ======================================================================================
constexpr int kGramRows = 64;  // rows staged per step

template <int TG>
__global__ void __launch_bounds__(256)
gram_kernel(const double* __restrict__ S, int64_t n, int k, double* __restrict__ partials,
            int nrb, int64_t rows_per_block) {
  constexpr int CT = 4 * TG;
  constexpr int RG = 256 / (TG * TG);
  constexpr int R = kGramRows;
  constexpr int LD = R + 1;
  extern __shared__ double gsm[];
  double* sI = gsm;
  double* sJ = gsm + CT * LD;

  const int nt = (k + CT - 1) / CT;
  int I = 0, J = 0;
  {
    int p = blockIdx.y;
    for (I = 0; I < nt; ++I) {
      int cnt = nt - I;
      if (p < cnt) { J = I + p; break; }
      p -= cnt;
    }
  }
  const bool diag = (I == J);
  if (diag) sJ = sI;
  const int tid = threadIdx.x;
  const int rg = tid / (TG * TG);
  const int tt = tid % (TG * TG);
  const int ti = tt / TG, tj = tt % TG;
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r_end = min(n, r_begin + rows_per_block);

  double acc[4][4];
  double sum[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    sum[i] = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  }

  for (int64_t r0 = r_begin; r0 < r_end; r0 += R) {
    for (int idx = tid; idx < CT * R; idx += 256) {
      int c = idx / R, r = idx % R;
      int64_t row = r0 + r;
      int colI = I * CT + c;
      sI[c * LD + r] = (colI < k && row < r_end) ? ld_stream_f64(S + (int64_t)colI * n + row) : 0.0;
      if (!diag) {
        int colJ = J * CT + c;
        sJ[c * LD + r] = (colJ < k && row < r_end) ? ld_stream_f64(S + (int64_t)colJ * n + row) : 0.0;
      }
    }
    __syncthreads();
#pragma unroll 4
    for (int r = rg; r < R; r += RG) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sI[(ti + TG * i) * LD + r];  // columns interleaved by TG: the TG
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = sJ[(tj + TG * j) * LD + r];  // threads of a row hit distinct banks
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
      if (diag && tj == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) sum[i] += a[i];
      }
    }
    __syncthreads();
  }

  // fold the row groups in a fixed order
  if (RG > 1) {
    double* red = gsm;  // [TG*TG][20]
    for (int g = 1; g < RG; ++g) {
      if (rg == g) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int j = 0; j < 4; ++j) red[tt * 20 + i * 4 + j] = acc[i][j];
          red[tt * 20 + 16 + i] = sum[i];
        }
      }
      __syncthreads();
      if (rg == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] += red[tt * 20 + i * 4 + j];
          sum[i] += red[tt * 20 + 16 + i];
        }
      }
      __syncthreads();
    }
  }
  if (rg == 0) {
    double* out = partials + ((size_t)blockIdx.y * nrb + blockIdx.x) * (CT * CT + CT);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) out[(ti + TG * i) * CT + tj + TG * j] = acc[i][j];
      if (tj == 0) out[CT * CT + ti + TG * i] = sum[i];
    }
  }
}

// k <= 16 (one 16 x 16 tile, HBM-bound): same thread grid and partial layout as gram_kernel<4>, but
// (a) the rows of the next step travel HBM -> shared memory with cp.async while the current step is
// multiplied (double buffer, no registers held by loads in flight), and (b) every shared-memory
// read fetches two adjacent rows of a column (LDS.128): 8 loads per 32 FMAs.  The two row groups of
// a warp sit 8 rows apart (16 banks), which keeps the 8 distinct 16-byte reads of a warp on
// distinct banks.
constexpr int kGramSmallRows = 128;
__global__ void __launch_bounds__(256, 3)
gram_small_kernel(const double* __restrict__ S, int64_t n, int k, double* __restrict__ partials,
                  int nrb, int64_t rows_per_block) {
  constexpr int TG = 4, CT = 16, R = kGramSmallRows, LD = R + 2, PER = CT * R / 256;  // 8 elements per thread and step
  __shared__ __align__(16) double sbuf[2][CT * LD];
  const int tid = threadIdx.x;
  const int rg = tid / (TG * TG);
  const int tt = tid % (TG * TG);
  const int ti = tt / TG, tj = tt % TG;
  const int rbase = (rg & 1) * 8 + (rg >> 1) * 16;
  const int64_t r_begin = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r_end = min(n, r_begin + rows_per_block);
  const int lr = tid % R, lc = tid / R;  // element e of a step: column 2 e + lc, row lr

  double acc[4][4];
  double sum[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    sum[i] = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
  }
  const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(&sbuf[0][0]) + (uint32_t)(lc * LD + lr) * 8u;
  auto issue = [&](int buf, int64_t r0) {  // rows past the end are zero-filled (src-size 0)
    const int64_t row = r0 + lr;
    const bool row_ok = row < r_end;
#pragma unroll
    for (int e = 0; e < PER; ++e) {
      const int c = 2 * e + lc;
      const bool ok = row_ok && c < k;
      const double* src = ok ? S + (int64_t)c * n + row : S;
      const uint32_t dst = s_base + (uint32_t)(buf * CT * LD + 2 * e * LD) * 8u;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(ok ? 8 : 0) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  issue(0, r_begin);
  int buf = 0;
  for (int64_t r0 = r_begin; r0 < r_end; r0 += R, buf ^= 1) {
    issue(buf ^ 1, r0 + R);  // that buffer was released by the barrier that ended the previous step
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncthreads();
    const double* sI = sbuf[buf];
#pragma unroll
    for (int pq = 0; pq < 4; ++pq) {
      const int r = rbase + 2 * pq;
      double2 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const double2*>(&sI[(ti + TG * i) * LD + r]);
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const double2*>(&sI[(tj + TG * j) * LD + r]);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc[i][j] = fma(a[i].x, b[j].x, acc[i][j]);
          acc[i][j] = fma(a[i].y, b[j].y, acc[i][j]);
        }
      if (tj == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          sum[i] += a[i].x;
          sum[i] += a[i].y;
        }
      }
    }
    __syncthreads();
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  // fold the 16 row groups in a fixed order
  double* red = sbuf[0];  // [TG*TG][20]
  for (int g = 1; g < 256 / (TG * TG); ++g) {
    if (rg == g) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) red[tt * 20 + i * 4 + j] = acc[i][j];
        red[tt * 20 + 16 + i] = sum[i];
      }
    }
    __syncthreads();
    if (rg == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] += red[tt * 20 + i * 4 + j];
        sum[i] += red[tt * 20 + 16 + i];
      }
    }
    __syncthreads();
  }
  if (rg == 0) {
    double* out = partials + (size_t)blockIdx.x * (CT * CT + CT);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = 0; j < 4; ++j) out[(ti + TG * i) * CT + tj + TG * j] = acc[i][j];
      if (tj == 0) out[CT * CT + ti + TG * i] = sum[i];
    }
  }
}

__global__ void gram_reduce_kernel(const double* __restrict__ partials, int nrb, int k, int CT,
                                   double* __restrict__ gram, double* __restrict__ colsum) {
  const int nt = (k + CT - 1) / CT;
  const int per = CT * CT + CT;
  const int pair = blockIdx.y;
  int I = 0, J = 0;
  {
    int p = pair;
    for (I = 0; I < nt; ++I) {
      int cnt = nt - I;
      if (p < cnt) { J = I + p; break; }
      p -= cnt;
    }
  }
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= per) return;
  double s = 0.0;
  const double* src = partials + (size_t)pair * nrb * per + e;
  for (int rb = 0; rb < nrb; ++rb) s += src[(size_t)rb * per];
  if (e < CT * CT) {
    int ci = I * CT + e / CT, cj = J * CT + e % CT;
    if (ci < k && cj < k) {
      gram[(size_t)ci * k + cj] = s;
      if (I != J) gram[(size_t)cj * k + ci] = s;
    }
  } else if (I == J) {
    int ci = I * CT + (e - CT * CT);
    if (ci < k) colsum[ci] = s;
  }
}

// ======================================================================================
// single-block: np.corrcoef normalisation + clip, Cholesky (lower, in place in W),
// T = Q^-T P^T (upper triangular).  numpy cov/corrcoef + np.linalg.cholesky +
// solve_triangular(...) @ P.T of correlation.py:398-414, for the k x k part.
// ======================================================================================
// MODE 0 (Iman-Conover): W = corrcoef.   MODE 1 (Cholesky correlator, correlation.py:263-285):
// W = np.cov(X_n, ddof=0) of the standardised data, and the finished T is scaled by the column
// standard deviations (`transform * std`, :285).
template <int MODE>
__global__ void __launch_bounds__(256)
chol_solve_kernel(const double* __restrict__ G, const double* __restrict__ colsum,
                  const double* __restrict__ P, double* __restrict__ W, double* __restrict__ T,
                  int k, double n_total, uint32_t* __restrict__ flags, const double* __restrict__ colstd) {
  const int tid = threadIdx.x, nth = blockDim.x;
  const double inv = 1.0 / (MODE == 0 ? n_total - 1.0 : n_total);
  for (int e = tid; e < k * k; e += nth) {
    int i = e / k, j = e % k;
    W[e] = (G[e] - colsum[i] * colsum[j] / n_total) * inv;
  }
  __syncthreads();
  if (MODE == 0) {
    for (int i = tid; i < k; i += nth) T[i] = sqrt(W[(size_t)i * k + i]);
    __syncthreads();
    for (int e = tid; e < k * k; e += nth) {
      int i = e / k, j = e % k;
      double c = W[e] / T[i];
      c = c / T[j];
      W[e] = fmin(fmax(c, -1.0), 1.0);  // NaN stays NaN only if both are NaN: checked below
      if (c != c) W[e] = c;
    }
    __syncthreads();
  }
  // right-looking Cholesky, lower triangle
  for (int j = 0; j < k; ++j) {
    double d = W[(size_t)j * k + j];
    if (!(d > 0.0)) {  // same acceptance as LAPACK dpotrf: pivot must be > 0 and not NaN
      if (tid == 0) flags[kFlagNotPD] = 1u;
      // keep the rest of the pipeline well defined (its output is discarded by the caller)
      for (int e = tid; e < k * k; e += nth) T[e] = 0.0;
      return;
    }
    double q = sqrt(d);
    __syncthreads();
    for (int i = j + 1 + tid; i < k; i += nth) W[(size_t)i * k + j] /= q;
    if (tid == 0) W[(size_t)j * k + j] = q;
    __syncthreads();
    // trailing update of the lower triangle: one warp per row i, lanes along m (coalesced, no div/mod)
    {
      const int lane = tid & 31, warp = tid >> 5, nwarps = nth >> 5;
      for (int i = j + 1 + warp; i < k; i += nwarps) {
        const double wij = W[(size_t)i * k + j];
        for (int m = j + 1 + lane; m <= i; m += 32) W[(size_t)i * k + m] -= wij * W[(size_t)m * k + j];
      }
    }
    __syncthreads();
  }
  // back substitution, one thread per column of T
  for (int c = tid; c < k; c += nth) {
    for (int i = k - 1; i >= 0; --i) {
      if (i > c) {
        T[(size_t)i * k + c] = 0.0;
        continue;
      }
      double s = P[(size_t)c * k + i];
      for (int m = i + 1; m <= c; ++m) s -= W[(size_t)m * k + i] * T[(size_t)m * k + c];
      T[(size_t)i * k + c] = s / W[(size_t)i * k + i];
    }
    if (MODE == 1) {
      const double sd = colstd[c];
      for (int i = 0; i <= c; ++i) T[(size_t)i * k + c] *= sd;
    }
  }
}

// The same computation for wide problems (k > 64), spread over the whole GPU with grid-wide barriers
// (cooperative launch): the single-block version is bound by one SM's L2 bandwidth (k^3/3 updates
// of an 8 MB matrix), this one by 3 grid barriers per column.
constexpr int kCholPanel = 32;
template <int MODE>
__global__ void __launch_bounds__(256)
chol_solve_grid_kernel(const double* __restrict__ G, const double* __restrict__ colsum,
                       const double* __restrict__ P, double* __restrict__ W, double* __restrict__ T,
                       int k, double n_total, uint32_t* __restrict__ flags, const double* __restrict__ colstd,
                       int rhs_warps) {
  cg::grid_group grid = cg::this_grid();
  const int nth = gridDim.x * blockDim.x, gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31, gwarp = gt >> 5, nwarps = nth >> 5;
  const double inv = 1.0 / (MODE == 0 ? n_total - 1.0 : n_total);
  for (int e = gt; e < k * k; e += nth) {
    int i = e / k, j = e % k;
    W[e] = (G[e] - colsum[i] * colsum[j] / n_total) * inv;
  }
  grid.sync();
  if (MODE == 0) {
    for (int i = gt; i < k; i += nth) T[i] = sqrt(W[(size_t)i * k + i]);
    grid.sync();
    for (int e = gt; e < k * k; e += nth) {
      int i = e / k, j = e % k;
      double c = W[e] / T[i];
      c = c / T[j];
      W[e] = (c != c) ? c : fmin(fmax(c, -1.0), 1.0);
    }
    grid.sync();
  }
  // Blocked right-looking Cholesky (lower triangle, in place), panels of kCholPanel columns: 3 grid barriers
  // per PANEL instead of per column (the column-by-column form spent 3 k barriers of ~15 us: 58 ms at
  // k = 1024).  (1) block 0 factors the diagonal block in shared memory, (2) every row below solves its
  // slice of the panel against it, (3) the trailing lower triangle takes the rank-kCholPanel update.
  constexpr int NB = kCholPanel;
  __shared__ double sL[NB][NB + 1];
  __shared__ int s_bad;
  for (int j0 = 0; j0 < k; j0 += NB) {
    const int nb = min(NB, k - j0);
    if (blockIdx.x == 0) {
      if (threadIdx.x == 0) s_bad = 0;
      for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) sL[e / nb][e % nb] = W[(size_t)(j0 + e / nb) * k + j0 + e % nb];
      __syncthreads();
      for (int j = 0; j < nb; ++j) {
        const double d = sL[j][j];
        if (!(d > 0.0)) {  // same acceptance as LAPACK dpotrf: the pivot must be > 0 and not NaN
          if (threadIdx.x == 0) s_bad = 1;
          break;           // (d is the same in every thread of the block)
        }
        const double q = sqrt(d);
        __syncthreads();
        for (int i = j + 1 + (int)threadIdx.x; i < nb; i += blockDim.x) sL[i][j] /= q;
        if (threadIdx.x == 0) sL[j][j] = q;
        __syncthreads();
        for (int e = threadIdx.x; e < (nb - j - 1) * (nb - j - 1); e += blockDim.x) {
          const int i = j + 1 + e / (nb - j - 1), m = j + 1 + e % (nb - j - 1);
          if (m <= i) sL[i][m] -= sL[i][j] * sL[m][j];
        }
        __syncthreads();
      }
      __syncthreads();
      for (int e = threadIdx.x; e < nb * nb; e += blockDim.x)
        if (e % nb <= e / nb) W[(size_t)(j0 + e / nb) * k + j0 + e % nb] = sL[e / nb][e % nb];
      if (threadIdx.x == 0 && s_bad) flags[kFlagNotPD] = 1u;
      __threadfence();
    }
    grid.sync();
    if (*reinterpret_cast<volatile uint32_t*>(&flags[kFlagNotPD])) {  // the same verdict in every block
      for (int e = gt; e < k * k; e += nth) T[e] = 0.0;
      return;
    }
    // (2) rows below the panel: W[i, j0 : j0+nb] <- W[i, j0 : j0+nb] L11^-T   (one thread per row)
    for (int i = j0 + nb + gt; i < k; i += nth) {
      double* wi = W + (size_t)i * k + j0;
      for (int c = 0; c < nb; ++c) {
        const double* lc = W + (size_t)(j0 + c) * k + j0;
        double v = wi[c];
        for (int m = 0; m < c; ++m) v -= wi[m] * lc[m];
        wi[c] = v / lc[c];
      }
    }
    grid.sync();
    // (3) trailing update of the lower triangle: one warp per row i, lanes along m
    for (int i = j0 + nb + gwarp; i < k; i += nwarps) {
      const double* wi = W + (size_t)i * k + j0;
      for (int m = j0 + nb + lane; m <= i; m += 32) {
        const double* wm = W + (size_t)m * k + j0;
        double acc = 0.0;
        for (int c = 0; c < nb; ++c) acc += wi[c] * wm[c];
        W[(size_t)i * k + m] -= acc;
      }
    }
    grid.sync();
  }
  // T = Q^-T P^T: column c of T solves Q^T t = P[c, :]^T (back substitution).  One WARP per column, in the
  // column-oriented (axpy) form: once t_m is final, s_i -= Q[m][i] t_m for all i < m -- a coalesced read
  // of row m of Q -- with the right-hand side in a shared-memory scratch of the warp.
  extern __shared__ double s_rhs[];  // [warps_per_block_active][k]
  const int warp_in_block = threadIdx.x >> 5;
  if (warp_in_block < rhs_warps) {
    double* sr = s_rhs + (size_t)warp_in_block * k;
    const int active_warps = gridDim.x * rhs_warps;
    for (int c = blockIdx.x * rhs_warps + warp_in_block; c < k; c += active_warps) {
      for (int i = lane; i <= c; i += 32) sr[i] = P[(size_t)c * k + i];
      for (int i = c + 1 + lane; i < k; i += 32) T[(size_t)i * k + c] = 0.0;
      __syncwarp();
      const double sd = MODE == 1 ? colstd[c] : 1.0;
      for (int m = c; m >= 0; --m) {
        const double* qm = W + (size_t)m * k;
        const double t = sr[m] / qm[m];
        for (int i = lane; i < m; i += 32) sr[i] -= qm[i] * t;
        if (lane == 0) T[(size_t)m * k + c] = MODE == 1 ? t * sd : t;
        __syncwarp();
      }
    }
  }
}

template <int MODE>
int launch_chol_solve(IcPlan* p, double n_total, const double* colstd, cudaStream_t stream) {
  if (p->k <= 64) {
    chol_solve_kernel<MODE><<<1, 256, 0, stream>>>(p->gram, p->colsum, p->P, p->work, p->T, p->k, n_total,
                                                   p->flags, colstd);
    PBL_LAUNCH_CHECK();
    return kOk;
  }
  int k = p->k;
  const double* G = p->gram;
  const double* cs = p->colsum;
  const double* P = p->P;
  double* W = p->work;
  double* T = p->T;
  uint32_t* fl = p->flags;
  // shared-memory scratch of the back substitution: one right-hand side (k doubles) per active warp
  int rhs_warps = (int)std::max<size_t>(1, std::min<size_t>(8, (size_t)(96 * 1024) / ((size_t)k * 8)));
  const size_t smem = (size_t)rhs_warps * k * 8;
  static bool attr = false;
  if (!attr) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(chol_solve_grid_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        96 * 1024));
    attr = true;
  }
  void* args[] = {&G, &cs, &P, &W, &T, &k, &n_total, &fl, &colstd, &rhs_warps};
  int per_sm = 0;
  PBL_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, chol_solve_grid_kernel<MODE>, 256, smem));
  const int blocks = std::max(1, std::min(per_sm, 2) * num_sms());
  PBL_CUDA_CHECK(cudaLaunchCooperativeKernel((void*)chol_solve_grid_kernel<MODE>, dim3(blocks), dim3(256), args, smem,
                                             stream));
  PBL_LAUNCH_CHECK();
  return kOk;
}

// ======================================================================================
// Cholesky correlator helpers (reference correlation.py:205-285): column mean / standard
// deviation (two passes, fixed-order reductions), standardisation, and the final `mean + ...`.
// ======================================================================================
constexpr int kMomBlocks = 256;  // partial sums per column

// MODE 0: sum x      MODE 1: sum (x - mean)^2
template <int MODE>
__global__ void __launch_bounds__(256)
col_moment_kernel(const double* __restrict__ X, int64_t row_stride, int64_t col_stride, int64_t n,
                  const double* __restrict__ mean, double* __restrict__ partials) {
  __shared__ double red[256];
  const int col = blockIdx.y;
  const double* xc = X + (int64_t)col * col_stride;
  const double m = MODE == 1 ? mean[col] : 0.0;
  const int64_t per = (n + gridDim.x - 1) / gridDim.x;
  const int64_t lo = (int64_t)blockIdx.x * per, hi = min(n, lo + per);
  double acc = 0.0;
  for (int64_t r = lo + threadIdx.x; r < hi; r += 256) {
    const double v = ld_stream_f64(xc + r * row_stride);
    acc += MODE == 1 ? (v - m) * (v - m) : v;
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) partials[(size_t)col * gridDim.x + blockIdx.x] = red[0];
}

template <int MODE>
__global__ void col_moment_finish_kernel(const double* __restrict__ partials, int nb, int k, double n,
                                         double* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= k) return;
  double s = 0.0;
  for (int b = 0; b < nb; ++b) s += partials[(size_t)c * nb + b];
  out[c] = MODE == 1 ? sqrt(s / n) : s / n;
}

__global__ void __launch_bounds__(256)
standardise_kernel(const double* __restrict__ X, int64_t row_stride, int64_t col_stride, int64_t n,
                   const double* __restrict__ mean, const double* __restrict__ sd, double* __restrict__ S) {
  const int col = blockIdx.y;
  const double m = mean[col], d = sd[col];
  for (int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x; r < n; r += (int64_t)gridDim.x * 256)
    S[(int64_t)col * n + r] = (ld_stream_f64(X + (int64_t)col * col_stride + r * row_stride) - m) / d;
}

__global__ void __launch_bounds__(256)
add_mean_kernel(const double* __restrict__ S, int64_t n, const double* __restrict__ mean,
                double* __restrict__ Y, int64_t row_stride, int64_t col_stride) {
  const int col = blockIdx.y;
  const double m = mean[col];
  for (int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x; r < n; r += (int64_t)gridDim.x * 256)
    Y[(int64_t)col * col_stride + r * row_stride] = m + ld_stream_f64(S + (int64_t)col * n + r);
}

// ======================================================================================
// transform: S <- S @ T in place, T upper triangular.
// small k: one thread per row, the row lives in registers, T broadcast from shared memory.
// ======================================================================================
template <int KMAX>
__global__ void __launch_bounds__(256, 2)
transform_small_kernel(double* __restrict__ S, int64_t n, int k, const double* __restrict__ T) {
  __shared__ __align__(16) double sT[KMAX * KMAX];
  for (int e = threadIdx.x; e < KMAX * KMAX; e += 256) {
    int i = e / KMAX, j = e % KMAX;
    sT[e] = (i < k && j < k) ? T[i * k + j] : 0.0;
  }
  __syncthreads();
  // one row per thread (no row loop: keeps the T loads from being hoisted into registers)
  const int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (r >= n) return;
  // acc[c] = sum_{j<=c} s_j T[j][c], accumulated in increasing j; column j is final (and can
  // overwrite its own input) as soon as row j of T has been applied.
  double acc[KMAX];
#pragma unroll
  for (int c = 0; c < KMAX; ++c) acc[c] = 0.0;
  if (KMAX <= 16) {
    // the whole row is fetched before the first store: the in-place stores may alias later loads
    // as far as the compiler can tell, so interleaving them would serialise KMAX HBM round trips
    double s[KMAX];
#pragma unroll
    for (int j = 0; j < KMAX; ++j) s[j] = (j < k) ? __ldcs(S + (int64_t)j * n + r) : 0.0;
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
#pragma unroll
      for (int c = j; c < KMAX; ++c) acc[c] = fma(s[j], sT[j * KMAX + c], acc[c]);
      if (j < k) S[(int64_t)j * n + r] = acc[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < KMAX; ++j) {
      if (j < k) {
        const double sj = S[(int64_t)j * n + r];
#pragma unroll
        for (int c = j; c < KMAX; ++c) acc[c] = fma(sj, sT[j * KMAX + c], acc[c]);
        S[(int64_t)j * n + r] = acc[j];
      }
    }
  }
}

// large k: 64-row x 64-column output tiles, 4x4 per thread, column tiles in descending order so
// that the in-place update never overwrites an input it still needs.
__global__ void __launch_bounds__(256)
transform_tiled_kernel(double* __restrict__ S, int64_t n, int k, const double* __restrict__ T) {
  constexpr int TS = 64;  // output tile edge
  constexpr int JD = 32;  // depth staged per step
  __shared__ __align__(16) double sS[JD * TS];  // [j][r]
  __shared__ __align__(16) double sT[JD * TS];  // [j][c]
  const int tid = threadIdx.x;
  const int tr = tid % 16, tc = tid / 16;
  const int64_t r0 = (int64_t)blockIdx.x * TS;
  const int nt = (k + TS - 1) / TS;
  for (int kt = nt - 1; kt >= 0; --kt) {
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    const int jmax = min(k, (kt + 1) * TS);  // T[j][c] = 0 for j > c
    for (int j0 = 0; j0 < jmax; j0 += JD) {
      for (int idx = tid; idx < JD * TS; idx += 256) {
        int j = idx / TS, x = idx % TS;
        int gj = j0 + j;
        int64_t row = r0 + x;
        sS[idx] = (gj < k && row < n) ? S[(int64_t)gj * n + row] : 0.0;
        int gc = kt * TS + x;
        sT[idx] = (gj < k && gc < k) ? T[(size_t)gj * k + gc] : 0.0;
      }
      __syncthreads();
#pragma unroll 8
      for (int j = 0; j < JD; ++j) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = sS[j * TS + 4 * tr + i];
#pragma unroll
        for (int c = 0; c < 4; ++c) b[c] = sT[j * TS + 4 * tc + c];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[i][c] = fma(a[i], b[c], acc[i][c]);
      }
      __syncthreads();
    }
    // all reads of this block's rows of column tile kt are complete (barrier above); lower
    // column tiles never read tile kt again, so it can be overwritten now
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      int gc = kt * TS + 4 * tc + c;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int64_t row = r0 + 4 * tr + i;
        if (gc < k && row < n) S[(int64_t)gc * n + row] = acc[i][c];
      }
    }
  }
}

#include "fp64_tiles.cuh"

template <typename T_>
int dev_alloc(T_** p, size_t count, IcPlan* plan) {
  size_t bytes = std::max<size_t>(count * sizeof(T_), 16);
  PBL_CUDA_CHECK(cudaMalloc((void**)p, bytes));
  plan->bytes += bytes;
  return kOk;
}

// thread-grid edge of the Gram kernel: 4 / 8 / 16 (4 x 4 outputs per thread); 32 = the 128 x 128 tiles of
// gram_big_kernel for wide problems (fp64_tiles.cuh)
int gram_tg_for(int k) { return k <= 16 ? 4 : (k <= 32 ? 8 : (k <= 64 ? 16 : 32)); }

}  // namespace

// ======================================================================================
// plan
// ======================================================================================
int ic_plan_create(int64_t n, int k, int col_batch, int flags, IcPlan** out) {
  *out = nullptr;
  if (n < 1 || k < 1 || n > (int64_t)kMaxSortN || k > 8192) {
    set_last_error("ic_plan_create: need 1 <= n < 2^31 and 1 <= k <= 8192");
    return kBadShape;
  }
  int device = 0;
  size_t free_b = 0, total_b = 0;
  PBL_CUDA_CHECK(cudaGetDevice(&device));  // (before the plan exists: an early CUDA failure leaks nothing)
  PBL_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  IcPlan* p = new IcPlan();
  p->n = n;
  p->k = k;
  p->rows_only = (flags & 1) != 0;
  p->device = device;

  // column batch: as many columns per launch as fit in ~45% of free memory
  const size_t fixed = (size_t)2 * k * n * 8;  // sortedX + scores
  const size_t per_col = (size_t)n * 24 + sort_status_bytes(1, (uint32_t)n) + 16384;
  if (col_batch <= 0) {
    size_t budget = free_b > fixed ? (size_t)((free_b - fixed) * 0.6) : 0;
    col_batch = (int)std::min<size_t>((size_t)k, std::max<size_t>(1, budget / per_col));
  }
  col_batch = std::max(1, std::min(col_batch, k));
  p->col_batch = col_batch;
  const int cb = col_batch;

  int rc = kOk;
  auto A = [&](auto** ptr, size_t count) {
    if (rc == kOk) rc = dev_alloc(ptr, count, p);
  };
  if (!p->rows_only) {
    // + 16 B: the bulk copies of the digit pass read whole 16 B units around a tile (pass_tma.cuh)
    A(&p->sort.keysA, (size_t)cb * n + 2);
    A(&p->sort.keysB, (size_t)cb * n + 2);
    A(&p->sort.valsA, (size_t)cb * n + 4);
    A(&p->sort.valsB, (size_t)cb * n + 4);
    A(&p->sort.hist, (size_t)cb * kMaxPasses * kRadix);
    A((unsigned char**)&p->sort.status, sort_status_bytes(cb, (uint32_t)n));
    if (rc == kOk && cudaMemset(p->sort.status, 0, sort_status_bytes(cb, (uint32_t)n)) != cudaSuccess) rc = kCudaError;
    A(&p->sort.maps, (size_t)cb);
    p->sort.epoch = &p->sort_epoch;
    A(&p->sort.tile_counter, (size_t)cb * (kMaxPasses + 1));
    A(&p->sort.kminmax, (size_t)cb * kMinMaxWords);
    A(&p->sort.plan, (size_t)cb);
    A(&p->sortedX, (size_t)k * n);
    A(&p->vdw, (size_t)n);
  }
  A(&p->flags, 8);
  p->sort.error_flag = p->flags;
  A(&p->scores, (size_t)k * n);
  A(&p->gram, (size_t)k * k);
  A(&p->colsum, (size_t)k);
  A(&p->work, (size_t)k * k);
  A(&p->T, (size_t)k * k);
  A(&p->P, (size_t)k * k);

  p->gram_tg = gram_tg_for(k);
  const int CT = 4 * p->gram_tg;
  const int nt = (k + CT - 1) / CT;
  const int npairs = nt * (nt + 1) / 2;
  int64_t max_rb = (n + kGramSmallRows - 1) / kGramSmallRows;
  // whole waves: gram_small_kernel runs 3 blocks per SM, gram_kernel 4
  int want = std::max(1, ((p->gram_tg == 4 ? 3 : (p->gram_tg == 32 ? 1 : 4)) * num_sms() + npairs - 1) / npairs);
  if (p->gram_tg == 32) {
    // one 254-register block per SM: pick the row-block count whose grid fills whole waves best (36 tile
    // pairs at k = 1024: 4 row blocks = 144 of 148 SMs in one wave, where 5 would run 1.2 waves)
    double best_eff = 0.0;
    for (int nrb = 1; nrb <= 16; ++nrb) {
      const int blocks = npairs * nrb, waves = (blocks + num_sms() - 1) / num_sms();
      const double eff = (double)blocks / ((double)waves * num_sms());
      if (eff > best_eff + 1e-9) {
        best_eff = eff;
        want = nrb;
      }
    }
  }
  p->gram_row_blocks = (int)std::max<int64_t>(1, std::min<int64_t>(max_rb, want));
  A(&p->gram_partials, (size_t)npairs * p->gram_row_blocks * (CT * CT + CT));
  if (rc != kOk) {
    ic_plan_destroy(p);
    return rc;
  }
  *out = p;
  return kOk;
}

void ic_plan_destroy(IcPlan* p) {
  if (!p) return;
  cudaFree(p->sort.keysA);
  cudaFree(p->sort.keysB);
  cudaFree(p->sort.valsA);
  cudaFree(p->sort.valsB);
  cudaFree(p->sort.hist);
  cudaFree(p->sort.status);
  cudaFree(p->sort.tile_counter);
  cudaFree(p->sort.plan);
  cudaFree(p->sort.kminmax);
  cudaFree(p->sort.maps);
  cudaFree(p->flags);
  cudaFree(p->sortedX);
  cudaFree(p->vdw);
  cudaFree(p->scores);
  cudaFree(p->gram);
  cudaFree(p->colsum);
  cudaFree(p->work);
  cudaFree(p->T);
  cudaFree(p->P);
  cudaFree(p->gram_partials);
  cudaFree(p->moments);
  permcorr_free(p->permcorr);
  for (cudaEvent_t e : p->events) cudaEventDestroy(e);
  if (p->copy_stream) cudaStreamDestroy(p->copy_stream);
  delete p;
}

int ic_plan_set_target(IcPlan* p, const double* P_lower_host) {
  PBL_CUDA_CHECK(cudaMemcpy(p->P, P_lower_host, (size_t)p->k * p->k * 8, cudaMemcpyHostToDevice));
  p->has_target = true;
  return kOk;
}

// ======================================================================================
// stages
// ======================================================================================
static SortBuffers sort_view(const IcPlan* p) { return p->sort; }

template <int MODE>
// c: global index of the batch's first column; the launch covers the batch-local columns [j0, j0 + nb)
static int launch_post_tma(IcPlan* p, int c, int nb, int shift, uint32_t epoch, uint32_t* counter,
                           cudaStream_t stream, int j0 = 0) {
  static bool attr_set = false;
  if (!attr_set) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(post_tma_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kPostTmaSmemBytes));
    attr_set = true;
  }
  PostArgs a;
  const size_t off = (size_t)j0 * p->n;
  a.keysA = p->sort.keysA + off;
  a.keysB = p->sort.keysB + off;
  a.valsA = p->sort.valsA + off;
  a.valsB = p->sort.valsB + off;
  a.plan = p->sort.plan + j0;
  a.maps = p->sort.maps + j0;
  a.sortedX = p->sortedX + (size_t)(c + j0) * p->n;
  a.vdw = p->vdw;
  a.flags = p->flags;
  a.ticket = counter;
  a.n = (uint32_t)p->n;
  a.ntiles = (uint32_t)((p->n + kTile - 1) / kTile);
  a.status64 = reinterpret_cast<uint64_t*>(p->sort.status) + (size_t)j0 * a.ntiles * kRadix;
  a.total_tiles = a.ntiles * (uint32_t)nb;
  a.epoch = epoch;
  a.col_base = c + j0;
  a.part_shift = shift;
  a.ncols = (uint32_t)nb;
  a.ncols_interleave = std::min<uint32_t>((uint32_t)nb, kInterleaveWidth);
  PBL_CUDA_CHECK(cudaMemsetAsync(counter, 0, sizeof(uint32_t), stream));
  const unsigned grid = (unsigned)std::min<size_t>((size_t)2 * num_sms(), (size_t)a.total_tiles);
  post_tma_kernel<MODE><<<grid, kTileThreads, kPostTmaSmemBytes, stream>>>(a);
  PBL_LAUNCH_CHECK();
  return kOk;
}

static int post_sort_attr() {
  static bool done = false;
  if (!done) {
    PBL_CUDA_CHECK(cudaFuncSetAttribute(post_sort_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPostSmem));
    PBL_CUDA_CHECK(cudaFuncSetAttribute(post_sort_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPostSmem));
    PBL_CUDA_CHECK(cudaFuncSetAttribute(post_sort_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPostSmem));
    done = true;
  }
  return kOk;
}

// The scatter by row, in one launch or (row-chunk hook set) chunk by chunk with the hook called after each.
static int scatter_rows_hooked(IcPlan* p, int c, int nb, int shift, double* out, int64_t row_stride,
                               int64_t col_stride, cudaStream_t stream) {
  const uint32_t n = (uint32_t)p->n;
  if (!p->chunk_fn || p->chunk_rows <= 0) return scatter_rows(n, nb, sort_view(p), out, row_stride, col_stride, stream);
  const int nchunks = (int)((p->n + p->chunk_rows - 1) / p->chunk_rows);
  if (shift >= 32) {  // short columns: the pairs are not grouped by row window
    PBL_RETURN_IF(scatter_rows(n, nb, sort_view(p), out, row_stride, col_stride, stream));
    for (int i = 0; i < nchunks; ++i)
      for (int j = 0; j < nb; ++j) p->chunk_fn(c + j, (p->chunk_first + i) % nchunks, p->chunk_user);
    return kOk;
  }
  const uint64_t w = 1ull << shift;
  for (int i = 0; i < nchunks; ++i) {
    const int g = (p->chunk_first + i) % nchunks;
    // whole windows covering the chunk's rows (a window shared with the neighbouring chunk is delivered
    // twice, with identical values)
    const uint64_t lo = (uint64_t)g * p->chunk_rows / w * w;
    const uint64_t hi = std::min<uint64_t>(n, (std::min<uint64_t>(n, (uint64_t)(g + 1) * p->chunk_rows) + w - 1) / w * w);
    PBL_RETURN_IF(scatter_rows(n, nb, sort_view(p), out, row_stride, col_stride, stream, (uint32_t)lo, (uint32_t)hi));
    for (int j = 0; j < nb; ++j) p->chunk_fn(c + j, g, p->chunk_user);
  }
  return kOk;
}

int ic_stage_rank_scores(IcPlan* p, const double* X, int64_t row_stride, int64_t col_stride,
                         int col0, int ncols, cudaStream_t stream, bool ranks_only) {
  if (p->rows_only) {
    set_last_error("this plan was created without a sort workspace (rows-only)");
    return kBadShape;
  }
  const uint32_t n = (uint32_t)p->n;
  if (!p->vdw_ready) {
    vdw_table_kernel<<<(unsigned)std::min<int64_t>((p->n + 255) / 256, (int64_t)num_sms() * 16), 256, 0, stream>>>(n, p->vdw);
    PBL_LAUNCH_CHECK();
    p->vdw_ready = true;
  }
  for (int c = col0; c < col0 + ncols; c += p->col_batch) {
    int nb = std::min(p->col_batch, col0 + ncols - c);
    PBL_RETURN_IF(sort_columns_f64(X + (int64_t)c * col_stride, row_stride, col_stride, n, nb,
                                   p->window_bits, sort_view(p), stream));
    dim3 grid((unsigned)((n + kPostTile - 1) / kPostTile), (unsigned)nb);
    PBL_RETURN_IF(post_sort_attr());
    int shift = 32, ntiles = 0;
    uint32_t* counter = nullptr;
    uint32_t epoch = 0;
    PBL_RETURN_IF(scatter_prepare(n, nb, sort_view(p), 1, kPostTile, &shift, &ntiles, &counter, &epoch, stream));
    if (!sort_classic_consumer(n)) {
      if (ranks_only)
        PBL_RETURN_IF(launch_post_tma<2>(p, c, nb, shift, epoch, counter, stream));
      else
        PBL_RETURN_IF(launch_post_tma<0>(p, c, nb, shift, epoch, counter, stream));
    } else {
      uint64_t* st64 = reinterpret_cast<uint64_t*>(p->sort.status);
      if (ranks_only)
        post_sort_kernel<2><<<grid, kPostBlock, kPostSmem, stream>>>(
            p->sort.keysA, p->sort.keysB, p->sort.valsA, p->sort.valsB, p->sort.plan, p->sort.kminmax,
            p->window_bits, n, p->sortedX + (size_t)c * n, p->vdw, p->flags, c, shift, st64, counter, ntiles, epoch);
      else
        post_sort_kernel<0><<<grid, kPostBlock, kPostSmem, stream>>>(
            p->sort.keysA, p->sort.keysB, p->sort.valsA, p->sort.valsB, p->sort.plan, p->sort.kminmax,
            p->window_bits, n, p->sortedX + (size_t)c * n, p->vdw, p->flags, c, shift, st64, counter, ntiles, epoch);
      PBL_LAUNCH_CHECK();
    }
    PBL_RETURN_IF(scatter_rows_hooked(p, c, nb, shift, p->scores + (size_t)c * n, 1, (int64_t)n, stream));
  }
  return kOk;
}

int ic_stage_gram(IcPlan* p, cudaStream_t stream) {
  const int TG = p->gram_tg, CT = 4 * TG;
  const int nt = (p->k + CT - 1) / CT;
  const int npairs = nt * (nt + 1) / 2;
  const int nrb = p->gram_row_blocks;
  int64_t rows_per = (p->n + nrb - 1) / nrb;
  const int step_rows = TG == 4 ? kGramSmallRows : (TG == 32 ? kBD : kGramRows);
  rows_per = (rows_per + step_rows - 1) / step_rows * step_rows;
  dim3 grid((unsigned)nrb, (unsigned)npairs);
  size_t smem = (size_t)2 * CT * (kGramRows + 1) * 8;
  smem = std::max(smem, (size_t)TG * TG * 20 * 8);
  if (TG == 32) {  // wide: FP64-bound 128 x 128 tiles
    static bool attr = false;
    if (!attr) {
      PBL_CUDA_CHECK(cudaFuncSetAttribute(gram_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGramBigSmem));
      attr = true;
    }
    gram_big_kernel<<<grid, 256, kGramBigSmem, stream>>>(p->scores, p->n, p->k, p->gram_partials, nrb, rows_per);
  } else if (TG == 4)  // k <= 16: one tile pair
    gram_small_kernel<<<(unsigned)nrb, 256, 0, stream>>>(p->scores, p->n, p->k, p->gram_partials, nrb, rows_per);
  else if (TG == 8)
    gram_kernel<8><<<grid, 256, smem, stream>>>(p->scores, p->n, p->k, p->gram_partials, nrb, rows_per);
  else {
    static bool attr = false;
    if (!attr) {
      PBL_CUDA_CHECK(cudaFuncSetAttribute(gram_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      attr = true;
    }
    gram_kernel<16><<<grid, 256, smem, stream>>>(p->scores, p->n, p->k, p->gram_partials, nrb, rows_per);
  }
  PBL_LAUNCH_CHECK();
  const int per = CT * CT + CT;
  gram_reduce_kernel<<<dim3((per + 255) / 256, npairs), 256, 0, stream>>>(
      p->gram_partials, nrb, p->k, CT, p->gram, p->colsum);
  PBL_LAUNCH_CHECK();
  return kOk;
}

int ic_stage_solve(IcPlan* p, int64_t n_total, cudaStream_t stream) {
  if (!p->has_target) {
    set_last_error("ic: set_target has not been called");
    return kBadShape;
  }
  PBL_RETURN_IF(launch_chol_solve<0>(p, (double)n_total, nullptr, stream));
  return kOk;
}

int ic_stage_transform(IcPlan* p, cudaStream_t stream) {
  const int k = p->k;
  const int64_t n = p->n;
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (k <= 8)
    transform_small_kernel<8><<<blocks, 256, 0, stream>>>(p->scores, n, k, p->T);
  else if (k <= 16)
    transform_small_kernel<16><<<blocks, 256, 0, stream>>>(p->scores, n, k, p->T);
  else if (k <= 32)
    transform_small_kernel<32><<<blocks, 256, 0, stream>>>(p->scores, n, k, p->T);
  else if (k <= 64)
    transform_tiled_kernel<<<(unsigned)((n + 63) / 64), 256, 0, stream>>>(p->scores, n, k, p->T);
  else {
    static bool attr = false;
    if (!attr) {
      PBL_CUDA_CHECK(cudaFuncSetAttribute(transform_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)kTransformBigSmem));
      attr = true;
    }
    transform_big_kernel<<<(unsigned)((n + kBT - 1) / kBT), 256, kTransformBigSmem, stream>>>(p->scores, n, k, p->T);
  }
  PBL_LAUNCH_CHECK();
  return kOk;
}

int ic_stage_rank_gather(IcPlan* p, double* Y, int64_t row_stride, int64_t col_stride, int col0,
                         int ncols, cudaStream_t stream) {
  if (p->rows_only) {
    set_last_error("this plan was created without a sort workspace (rows-only)");
    return kBadShape;
  }
  const uint32_t n = (uint32_t)p->n;
  for (int c = col0; c < col0 + ncols; c += p->col_batch) {
    int nb = std::min(p->col_batch, col0 + ncols - c);
    PBL_RETURN_IF(sort_columns_f64(p->scores + (size_t)c * n, 1, (int64_t)n, n, nb, p->window_bits,
                                   sort_view(p), stream));
    dim3 grid((unsigned)((n + kPostTile - 1) / kPostTile), (unsigned)nb);
    PBL_RETURN_IF(post_sort_attr());
    int shift = 32, ntiles = 0;
    uint32_t* counter = nullptr;
    uint32_t epoch = 0;
    PBL_RETURN_IF(scatter_prepare(n, nb, sort_view(p), row_stride, kPostTile, &shift, &ntiles, &counter, &epoch,
                                  stream));
    if (!sort_classic_consumer(n)) {
      // Batches of 2 .. 7 columns go column by column: with so few columns interleaved the gather-mode consumer,
      // whose tiles are short, spends most of its time polling look-back words (ncu, 1e8 x 2: 2.1x the
      // instructions and 5.4 ms in one launch against 1.0 + 1.4 ms in two; 3 / 4 columns: +0.8 / +0.6 ms per
      // column); from ~8 columns on the interleave wins (15 columns: 1.2 ms per column).
      if (nb > 1 && nb < 8) {
        for (int j = 0; j < nb; ++j) PBL_RETURN_IF(launch_post_tma<1>(p, c, 1, shift, epoch, counter, stream, j));
      } else {
        PBL_RETURN_IF(launch_post_tma<1>(p, c, nb, shift, epoch, counter, stream));
      }
    } else {
      post_sort_kernel<1><<<grid, kPostBlock, kPostSmem, stream>>>(
          p->sort.keysA, p->sort.keysB, p->sort.valsA, p->sort.valsB, p->sort.plan, p->sort.kminmax,
          p->window_bits, n, p->sortedX + (size_t)c * n, p->vdw, p->flags, c, shift,
          reinterpret_cast<uint64_t*>(p->sort.status), counter, ntiles, epoch);
      PBL_LAUNCH_CHECK();
    }
    PBL_RETURN_IF(scatter_rows_hooked(p, c, nb, shift, Y + (int64_t)c * col_stride, row_stride, col_stride,
                                      stream));
  }
  return kOk;
}

// Cholesky().set_target(C)(X) (reference correlation.py:248-285) on device-resident data:
//   mean / std (ddof 0) per column, X_n = (X - mean) / std, cov = np.cov(X_n, ddof=0),
//   T = chol(cov)^-T P^T scaled by std per column, Y = mean + X_n @ T.
// Works on any plan (rows-only is enough: no sorts).
int cholesky_correlator_run(IcPlan* p, const double* X, int64_t xrs, int64_t xcs, double* Y, int64_t yrs,
                            int64_t ycs, cudaStream_t stream) {
  if (!p->has_target) {
    set_last_error("User must call `set_target` first.");
    return kBadShape;
  }
  const int k = p->k;
  const int64_t n = p->n;
  if (!p->moments) {
    PBL_CUDA_CHECK(cudaMalloc((void**)&p->moments, ((size_t)2 * k + (size_t)k * kMomBlocks) * 8));
    p->bytes += ((size_t)2 * k + (size_t)k * kMomBlocks) * 8;
  }
  double* mean = p->moments;
  double* sd = p->moments + k;
  double* partials = p->moments + 2 * k;
  PBL_CUDA_CHECK(cudaMemsetAsync(p->flags, 0, 8 * sizeof(uint32_t), stream));
  const dim3 mg(kMomBlocks, k);
  col_moment_kernel<0><<<mg, 256, 0, stream>>>(X, xrs, xcs, n, nullptr, partials);
  PBL_LAUNCH_CHECK();
  col_moment_finish_kernel<0><<<(k + 127) / 128, 128, 0, stream>>>(partials, kMomBlocks, k, (double)n, mean);
  PBL_LAUNCH_CHECK();
  col_moment_kernel<1><<<mg, 256, 0, stream>>>(X, xrs, xcs, n, mean, partials);
  PBL_LAUNCH_CHECK();
  col_moment_finish_kernel<1><<<(k + 127) / 128, 128, 0, stream>>>(partials, kMomBlocks, k, (double)n, sd);
  PBL_LAUNCH_CHECK();
  const unsigned rb = (unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)num_sms() * 8);
  standardise_kernel<<<dim3(rb, k), 256, 0, stream>>>(X, xrs, xcs, n, mean, sd, p->scores);
  PBL_LAUNCH_CHECK();
  PBL_RETURN_IF(ic_stage_gram(p, stream));
  PBL_RETURN_IF(launch_chol_solve<1>(p, (double)n, sd, stream));
  PBL_RETURN_IF(ic_stage_transform(p, stream));
  add_mean_kernel<<<dim3(rb, k), 256, 0, stream>>>(p->scores, n, mean, Y, yrs, ycs);
  PBL_LAUNCH_CHECK();
  uint32_t h[8];
  PBL_CUDA_CHECK(cudaMemcpyAsync(h, p->flags, sizeof(h), cudaMemcpyDeviceToHost, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  if (h[kFlagNotPD]) {
    set_last_error("Matrix is not positive definite");
    return kNotPositiveDefinite;
  }
  return kOk;
}

__global__ void __launch_bounds__(256)
copy_column_kernel(const double* __restrict__ X, int64_t xrs, double* __restrict__ Y, int64_t yrs, int64_t n) {
  for (int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x; r < n; r += (int64_t)gridDim.x * 256)
    Y[r * yrs] = ld_stream_f64(X + r * xrs);
}

// Column 0 needs no second sort when T[0][0] == 1 exactly: its correlated score is then the van der
// Waerden score itself (T is upper triangular), whose order and tie-runs are those of X[:, 0], so
// the reference's gather returns X[:, 0] unchanged (every member of a tie-run receives the run's
// common value).  Only a column holding both zeros is excluded (its tie-run mixes -0.0 and +0.0).
// Returns the first column that still has to be ranked (0 or 1); Y[:, 0] <- X[:, 0] when skipped.
static int first_column_to_rank(IcPlan* p, const double* X, int64_t xrs, double* Y, int64_t yrs,
                                cudaStream_t stream) {
  double t00 = 0.0;
  uint32_t h[8];
  if (cudaMemcpyAsync(&t00, p->T, sizeof(double), cudaMemcpyDeviceToHost, stream) != cudaSuccess) return 0;
  if (cudaMemcpyAsync(h, p->flags, sizeof(h), cudaMemcpyDeviceToHost, stream) != cudaSuccess) return 0;
  if (cudaStreamSynchronize(stream) != cudaSuccess) return 0;
  if (t00 != 1.0 || h[kFlagNegZeroCol0] || h[kFlagNotPD] || h[kFlagNaN] || h[kFlagWindowRetry]) return 0;
  const unsigned rb = (unsigned)std::min<int64_t>((p->n + 255) / 256, (int64_t)num_sms() * 16);
  copy_column_kernel<<<rb, 256, 0, stream>>>(X, xrs, Y, yrs, p->n);
  g_kernel_launches.fetch_add(1, std::memory_order_relaxed);
  return 1;
}

// ImanConover.__call__ with HOST buffers, pipelined: the host->device copy of column batch b+1
// overlaps the rank_scores sorts of batch b, and the device->host copy of batch b overlaps the
// rank_gather sorts of batch b+1 (columns are independent in both sort stages; only the Gram /
// solve / transform in the middle need every column).  dX / dY: device staging of n*k doubles each.
int ic_plan_run_host(IcPlan* p, const double* Xh, int64_t xrs, int64_t xcs, double* Yh, int64_t yrs,
                     int64_t ycs, double* dX, double* dY, cudaStream_t stream) {
  const int64_t n = p->n;
  const int k = p->k;
  const size_t bytes = (size_t)n * k * 8;
  const bool colmajor = (xrs == 1 && xcs == n && yrs == 1 && ycs == n) || k == 1;
  if (!colmajor) {  // C order: one block each way, no overlap
    PBL_CUDA_CHECK(cudaMemcpyAsync(dX, Xh, bytes, cudaMemcpyHostToDevice, stream));
    int st = ic_plan_run(p, dX, xrs, xcs, dY, yrs, ycs, stream);
    if (st != kOk) return st;
    PBL_CUDA_CHECK(cudaMemcpyAsync(Yh, dY, bytes, cudaMemcpyDeviceToHost, stream));
    PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
    return kOk;
  }
  if (!p->copy_stream) {
    PBL_CUDA_CHECK(cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
  }
  const int bc = std::max(1, std::min(p->col_batch, k >= 8 ? 2 : 1));  // columns per pipeline stage
  const int nb = (k + bc - 1) / bc;
  while ((int)p->events.size() < 2 * nb) {
    cudaEvent_t e;
    PBL_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    p->events.push_back(e);
  }
  // every exit -- including the early error returns below -- first drains the copy stream: its copies target
  // the caller's host buffers and dX / dY, which the caller may reuse or free as soon as this returns
  struct DrainCopies {
    cudaStream_t s;
    ~DrainCopies() { cudaStreamSynchronize(s); }
  } drain{p->copy_stream};
  while ((int)p->events.size() < 2 * nb + 1) {
    cudaEvent_t e;
    PBL_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    p->events.push_back(e);
  }
  for (int attempt = 0; attempt < 2; ++attempt) {
    PBL_CUDA_CHECK(cudaMemsetAsync(p->flags, 0, 8 * sizeof(uint32_t), stream));
    // the copy stream must not run ahead of work queued earlier on `stream` (e.g. the caller's last use of
    // dX / dY, or the first attempt's sorts that still read dX)
    PBL_CUDA_CHECK(cudaEventRecord(p->events[2 * nb], stream));
    PBL_CUDA_CHECK(cudaStreamWaitEvent(p->copy_stream, p->events[2 * nb], 0));
    for (int b = 0; b < nb; ++b) {
      const int c0 = b * bc, nc = std::min(bc, k - c0);
      PBL_CUDA_CHECK(cudaMemcpyAsync(dX + (size_t)c0 * n, Xh + (size_t)c0 * n, (size_t)nc * n * 8,
                                     cudaMemcpyHostToDevice, p->copy_stream));
      PBL_CUDA_CHECK(cudaEventRecord(p->events[b], p->copy_stream));
      PBL_CUDA_CHECK(cudaStreamWaitEvent(stream, p->events[b], 0));
      PBL_RETURN_IF(ic_stage_rank_scores(p, dX, 1, n, c0, nc, stream));
    }
    PBL_RETURN_IF(ic_stage_gram(p, stream));
    PBL_RETURN_IF(ic_stage_solve(p, p->n, stream));
    PBL_RETURN_IF(ic_stage_transform(p, stream));
    const int skip0 = first_column_to_rank(p, dX, 1, dY, 1, stream);
    for (int b = 0; b < nb; ++b) {
      const int c0 = b * bc, nc = std::min(bc, k - c0);
      const int r0 = std::max(c0, skip0);
      if (r0 < c0 + nc) PBL_RETURN_IF(ic_stage_rank_gather(p, dY, 1, n, r0, c0 + nc - r0, stream));
      PBL_CUDA_CHECK(cudaEventRecord(p->events[nb + b], stream));
      PBL_CUDA_CHECK(cudaStreamWaitEvent(p->copy_stream, p->events[nb + b], 0));
      PBL_CUDA_CHECK(cudaMemcpyAsync(Yh + (size_t)c0 * n, dY + (size_t)c0 * n, (size_t)nc * n * 8,
                                     cudaMemcpyDeviceToHost, p->copy_stream));
    }
    int st = ic_read_status(p, stream);
    PBL_CUDA_CHECK(cudaStreamSynchronize(p->copy_stream));
    if (st != kRetry) return st;
  }
  set_last_error("windowed sort retry did not converge (internal error)");
  return kInternal;
}

// Column means (MODE 0) or population standard deviations about `mean` (MODE 1) of an (n, k) matrix,
// fixed-order reductions (used by the Cholesky and permutation correlators).
int column_moments(IcPlan* p, const double* X, int64_t xrs, int64_t xcs, const double* mean_dev, double* out_dev,
                   int mode, cudaStream_t stream) {
  const int k = p->k;
  const int64_t n = p->n;
  if (!p->moments) {
    PBL_CUDA_CHECK(cudaMalloc((void**)&p->moments, ((size_t)2 * k + (size_t)k * kMomBlocks) * 8));
    p->bytes += ((size_t)2 * k + (size_t)k * kMomBlocks) * 8;
  }
  double* partials = p->moments + 2 * k;
  const dim3 mg(kMomBlocks, k);
  if (mode == 0) {
    col_moment_kernel<0><<<mg, 256, 0, stream>>>(X, xrs, xcs, n, nullptr, partials);
    PBL_LAUNCH_CHECK();
    col_moment_finish_kernel<0><<<(k + 127) / 128, 128, 0, stream>>>(partials, kMomBlocks, k, (double)n, out_dev);
  } else {
    col_moment_kernel<1><<<mg, 256, 0, stream>>>(X, xrs, xcs, n, mean_dev, partials);
    PBL_LAUNCH_CHECK();
    col_moment_finish_kernel<1><<<(k + 127) / 128, 128, 0, stream>>>(partials, kMomBlocks, k, (double)n, out_dev);
  }
  PBL_LAUNCH_CHECK();
  return kOk;
}

__global__ void __launch_bounds__(256)
centre_kernel(const double* __restrict__ X, int64_t row_stride, int64_t col_stride, int64_t n,
              const double* __restrict__ mean, double* __restrict__ S) {
  const int col = blockIdx.y;
  const double m = mean[col];
  for (int64_t r = (int64_t)blockIdx.x * 256 + threadIdx.x; r < n; r += (int64_t)gridDim.x * 256)
    S[(int64_t)col * n + r] = ld_stream_f64(X + (int64_t)col * col_stride + r * row_stride) - m;
}

// S[c][r] = X[r, c] - mean[c]  (column-major destination)
int centre_columns(IcPlan* p, const double* X, int64_t xrs, int64_t xcs, const double* mean_dev, double* S,
                   cudaStream_t stream) {
  const unsigned rb = (unsigned)std::min<int64_t>((p->n + 255) / 256, (int64_t)num_sms() * 8);
  centre_kernel<<<dim3(rb, p->k), 256, 0, stream>>>(X, xrs, xcs, p->n, mean_dev, S);
  PBL_LAUNCH_CHECK();
  return kOk;
}

__global__ void corr_from_gram_kernel(const double* __restrict__ G, int k, double* __restrict__ R) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < k * k; e += gridDim.x * blockDim.x) {
    const int i = e / k, j = e % k;
    double c = G[e] / sqrt(G[(size_t)i * k + i]);
    c = c / sqrt(G[(size_t)j * k + j]);
    R[e] = (c != c) ? c : fmin(fmax(c, -1.0), 1.0);
  }
}

// np.corrcoef(X, rowvar=False) (spearman == 0) or the Spearman rank correlation matrix
// (scipy.stats.spearmanr: Pearson correlation of the average ranks) of device-resident X, written to
// host memory.  Verification helper: lets the acceptance checks of the correlators run on the device
// at sizes the host cannot hold.  Uses plan->scores (and the sort workspace for Spearman).
int corrcoef_run(IcPlan* p, const double* X, int64_t xrs, int64_t xcs, int spearman, double* out_host,
                 cudaStream_t stream) {
  const int k = p->k;
  const int64_t n = p->n;
  if (!p->moments) {
    PBL_CUDA_CHECK(cudaMalloc((void**)&p->moments, ((size_t)2 * k + (size_t)k * kMomBlocks) * 8));
    p->bytes += ((size_t)2 * k + (size_t)k * kMomBlocks) * 8;
  }
  double* mean = p->moments;
  PBL_CUDA_CHECK(cudaMemsetAsync(p->flags, 0, 8 * sizeof(uint32_t), stream));
  const double* basis = X;
  int64_t brs = xrs, bcs = xcs;
  if (spearman) {
    if (p->rows_only) {
      set_last_error("corrcoef: the Spearman mode needs a plan with a sort workspace");
      return kBadShape;
    }
    PBL_RETURN_IF(ic_stage_rank_scores(p, X, xrs, xcs, 0, k, stream, /*ranks_only=*/true));
    basis = p->scores;
    brs = 1;
    bcs = n;
  }
  PBL_RETURN_IF(column_moments(p, basis, brs, bcs, nullptr, mean, 0, stream));
  PBL_RETURN_IF(centre_columns(p, basis, brs, bcs, mean, p->scores, stream));
  PBL_RETURN_IF(ic_stage_gram(p, stream));
  corr_from_gram_kernel<<<std::min(64, (k * k + 255) / 256), 256, 0, stream>>>(p->gram, k, p->work);
  PBL_LAUNCH_CHECK();
  PBL_CUDA_CHECK(cudaMemcpyAsync(out_host, p->work, (size_t)k * k * 8, cudaMemcpyDeviceToHost, stream));
  int st = ic_read_status(p, stream);
  return st == kRetry ? corrcoef_run(p, X, xrs, xcs, spearman, out_host, stream) : st;
}

int ic_read_status(IcPlan* p, cudaStream_t stream) {
  uint32_t h[8];
  PBL_CUDA_CHECK(cudaMemcpyAsync(h, p->flags, sizeof(h), cudaMemcpyDeviceToHost, stream));
  PBL_CUDA_CHECK(cudaStreamSynchronize(stream));
  if (h[kFlagWatchdog]) {
    set_last_error("radix sort look-back watchdog fired (internal error)");
    return kInternal;
  }
  if (h[kFlagNaN]) {
    set_last_error("array must not contain infs or NaNs");
    return kNonFinite;
  }
  if (h[kFlagWindowRetry] && p->window_bits < 64) {
    // the data are too dense for the 32-bit window: from now on this plan sorts on all 64 bits
    p->window_bits = 64;
    set_last_error("windowed sort could not be completed; repeat the call (full 64-bit sort)");
    return kRetry;
  }
  if (h[kFlagNotPD]) {
    set_last_error("Rank data correlation not positive definite.");
    return kNotPositiveDefinite;
  }
  return kOk;
}

int ic_plan_run(IcPlan* p, const double* X, int64_t xrs, int64_t xcs, double* Y, int64_t yrs,
                int64_t ycs, cudaStream_t stream) {
  for (int attempt = 0; attempt < 2; ++attempt) {
    PBL_CUDA_CHECK(cudaMemsetAsync(p->flags, 0, 8 * sizeof(uint32_t), stream));
    PBL_RETURN_IF(ic_stage_rank_scores(p, X, xrs, xcs, 0, p->k, stream));
    PBL_RETURN_IF(ic_stage_gram(p, stream));
    PBL_RETURN_IF(ic_stage_solve(p, p->n, stream));
    PBL_RETURN_IF(ic_stage_transform(p, stream));
    const int c0 = first_column_to_rank(p, X, xrs, Y, yrs, stream);
    if (c0 < p->k) PBL_RETURN_IF(ic_stage_rank_gather(p, Y, yrs, ycs, c0, p->k - c0, stream));
    int st = ic_read_status(p, stream);
    if (st != kRetry) return st;
  }
  set_last_error("windowed sort retry did not converge (internal error)");
  return kInternal;
}

}  // namespace pbl
