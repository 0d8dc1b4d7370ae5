// Building blocks shared by the two persistent, bulk-async (TMA) tile kernels of the sort:
//   pass_tma_kernel (sort.cu)  -- one onesweep digit pass
//   post_tma_kernel (ic.cu)    -- order completion + tie runs + scores / gather + row-window partition
// Both walk a column in tiles of 4096 elements (8 B "big" member + 4 B "small" member), pull a tile into
// a shared-memory stage with cp.async.bulk + mbarrier (SASS: UBLKCP / SYNCS), and finish with the
// same multi-split: rank the elements by an 8-bit digit, chain the per-bin counts to the previous
// tiles by decoupled look-back, stage the tile in digit order in place, write coalesced runs.
#pragma once
#include "rank.cuh"
#include "sort.cuh"

namespace pbl {

constexpr int kTileThreads = 256;
constexpr int kTileItems = 16;
constexpr int kTile = kTileThreads * kTileItems;  // 4096
constexpr int kTileWarps = kTileThreads / 32;
constexpr uint32_t kTileSpinLimit = 1u << 24;     // look-back watchdog: fail loudly instead of hanging

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait suspends the thread in hardware until the phase completes or a time limit passes; the loop
// around it is bounded so that a lost transaction traps (CUDA error on the host) instead of hanging
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t* error_flag) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 22)) {
      atomicExch(&error_flag[kFlagWatchdog], 1u);
      __trap();
    }
  }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// generic-proxy accesses to shared memory (this thread's, and by cumulativity those ordered before it by
// a barrier) -> visible to / ordered before subsequent async-proxy (bulk copy) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void st_u64_at(uint64_t* base, uint32_t idx, uint64_t v) {
  uint64_t addr;
  asm("mad.wide.u32 %0, %1, 8, %2;" : "=l"(addr) : "r"(idx), "l"(base));
  *reinterpret_cast<uint64_t*>(addr) = v;
}
__device__ __forceinline__ void st_u32_at(uint32_t* base, uint32_t idx, uint32_t v) {
  uint64_t addr;
  asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(addr) : "r"(idx), "l"(base));
  *reinterpret_cast<uint32_t*>(addr) = v;
}

#ifdef PBL_TILE_STATS
// developer instrumentation (tools/tile_stats.py; build with PBL_EXTRA_NVCC_FLAGS=-DPBL_TILE_STATS):
// per-launch totals taken by thread 0 -- [0] tiles of the digit pass, [1] look-back words consumed,
// [2] polls that found an unpublished word, [3] cycles in the look-back, [4] cycles from "tile data landed"
// to the end of the tile, [5] cycles waiting for the data, [6] tiles that walked
__device__ unsigned long long g_tile_stats[8];
#endif

// Decoupled look-back over 64-bit epoch-tagged words (sort.cuh) for bin threadIdx.x: walks back over the
// predecessors of `tile` in `st` ([ntiles][kRadix] of this column; the caller has published `cnt` for `tile`)
// until an inclusive word, stores this tile's inclusive word and returns the exclusive prefix.  The walk
// fetches 4 words per round trip; an unpublished word (not this epoch yet) restarts the batch there, and
// kTileSpinLimit polls raise error_flag[kFlagWatchdog] instead of hanging.  Shared by split_tile below and
// post_sort_kernel (ic.cu).
__device__ __forceinline__ uint32_t lookback_u64(uint64_t* __restrict__ st, const uint32_t tile, const uint32_t epoch,
                                                 const uint32_t cnt, uint32_t* __restrict__ error_flag) {
  const uint32_t bin = threadIdx.x;
  uint32_t excl = 0;
  if (tile == 0) return excl;
#ifdef PBL_TILE_STATS
  const long long lb_t0 = clock64();
  unsigned long long lb_steps = 0;
#endif
  const uint64_t tag = (uint64_t)epoch << 34;
  constexpr int LB = 4;
  int64_t t = (int64_t)tile - 1;
  bool done = false;
  uint32_t spins = 0;
  while (!done) {
    uint64_t pre[LB];
#pragma unroll
    for (int i = 0; i < LB; ++i)
      pre[i] = (t - i >= 0) ? ld_relaxed_u64(&st[(size_t)(t - i) * kRadix + bin]) : (tag | kStatusInclusive);
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      if (!done) {
        const uint64_t w = pre[i];
        if ((w >> 34) != (uint64_t)epoch || (w & (kStatusInclusive | kStatusPartial)) == 0) {  // not published yet
          if (++spins > kTileSpinLimit) {
            atomicExch(&error_flag[kFlagWatchdog], 1u);
            done = true;
          }
          break;
        }
        excl += (uint32_t)w;
        --t;
#ifdef PBL_TILE_STATS
        ++lb_steps;
#endif
        if (w & kStatusInclusive) done = true;
      }
    }
  }
  st_relaxed_u64(&st[(size_t)tile * kRadix + bin], tag | kStatusInclusive | (uint32_t)(excl + cnt));
#ifdef PBL_TILE_STATS
  if (bin == 0) {
    atomicAdd(&g_tile_stats[6], 1ull);
    atomicAdd(&g_tile_stats[1], lb_steps);
    atomicAdd(&g_tile_stats[2], (unsigned long long)spins);
    atomicAdd(&g_tile_stats[3], (unsigned long long)(clock64() - lb_t0));
  }
#endif
  return excl;
}

// Ticket -> (column, tile).  Tickets are handed out in GROUPS of `width` columns (the last group may be
// narrower): inside a group ticket r works on column r % w, tile r / w, so that the tiles in flight at any
// moment (2 per SM) are spread over the group's columns and a tile's look-back finds an inclusive
// predecessor a few tiles back instead of a few hundred (the chained scan is per column).  The width is
// capped (kInterleaveWidth): every column in flight keeps 256 partly written 128 B lines per output array in
// L2, and with 1024 columns interleaved (d = 1024: 67 MB of write frontier) they were evicted half
// written -- the passes ran at half speed.  width = min(ncols, kInterleaveWidth) >= 1.
constexpr uint32_t kInterleaveWidth = 32;
__device__ __forceinline__ void ticket_to_tile(uint32_t g, uint32_t ncols, uint32_t ntiles, uint32_t width,
                                               uint32_t* col, uint32_t* tile) {
  const uint32_t per_group = width * ntiles;
  const uint32_t group = g / per_group, r = g - group * per_group;
  const uint32_t c0 = group * width;
  const uint32_t w = min(width, ncols - c0);  // the last group holds what is left
  // (tickets of a narrower last group: r runs over w * ntiles values only, because the launch's ticket
  //  space is ncols * ntiles and earlier groups are full)
  *tile = r / w;
  *col = c0 + (r - *tile * w);
}

// Shared-memory scratch of the multi-split.
struct SplitSmem {
  uint32_t* hist;  // [kTileWarps][kRadix] warp-private digit counters
  uint32_t* goff;  // [kRadix]
  uint32_t* wsum;  // [kTileWarps]
};
constexpr size_t kSplitSmemBytes = (size_t)kTileWarps * kRadix * 4 + kRadix * 4 + 64;

// The multi-split of one tile.  On entry every thread holds its kTileItems elements' digits and 8 B
// members in registers (warp-striped: item u of lane l of warp w is tile position w*512 + u*32 + l) and
// NOTHING else of the tile is needed from the stage any more once `load_small` has run, because the
// stage is reused, in place, as the digit-ordered staging area.
//   dig          digits; positions >= nvalid of a partial tile must carry kRadix-1 (they sort last)
//   load_small   callable(uint32_t (&small)[ITEMS]): produces the 4 B members; called after the 8 B
//                members have been staged (keeps them out of the registers during the ranking)
//   digit_at     callable(pos) -> digit of the staged element at tile position pos
//   after_first_barrier  callable(): runs once, right after the first block barrier (at that point every
//                warp has finished the PREVIOUS tile: the other stage may be refilled)
//   st           look-back words of this column: [ntiles][kRadix]
//   bin_base     (thread tid owns bin tid) global slot of the bin's first element
template <bool FULL, class LoadSmall, class DigitAt, class AfterFirstBarrier>
__device__ __forceinline__ void split_tile(const uint32_t (&dig)[kTileItems], const uint64_t (&big)[kTileItems],
                                           LoadSmall load_small, DigitAt digit_at,
                                           AfterFirstBarrier after_first_barrier, const SplitSmem& sm,
                                           uint64_t* s_big, uint32_t* s_small, uint64_t* __restrict__ st,
                                           const uint32_t tile, const uint32_t nvalid, const uint32_t epoch,
                                           const uint32_t bin_base, uint64_t* __restrict__ out_big,
                                           uint32_t* __restrict__ out_small, uint32_t* __restrict__ error_flag) {
  constexpr int ITEMS = kTileItems;
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  // the warp's private digit counters start at zero
  uint32_t* wh = sm.hist + warp * kRadix;
  {
    const uint4 z = make_uint4(0, 0, 0, 0);
    reinterpret_cast<uint4*>(wh)[lane] = z;
    reinterpret_cast<uint4*>(wh)[lane + 32] = z;
  }
  __syncwarp();
  uint32_t rank[ITEMS];
  warp_rank_digits<ITEMS>(dig, wh, rank, lane);
  __syncthreads();  // every element of the stage is in registers; all warps' counts are final
  after_first_barrier();

  // ---- per bin: the warps' counts -> tile total, published for the tiles behind us; exclusive scan over
  //      warps and bins; the counters become (bin start in the tile + elements of earlier warps in the bin) ----
  const uint64_t tag = (uint64_t)epoch << 34;
  uint32_t cnt = 0;
#pragma unroll
  for (int w = 0; w < kTileWarps; ++w) cnt += sm.hist[w * kRadix + tid];
  if (!FULL && tid == kRadix - 1) cnt -= (uint32_t)kTile - nvalid;  // the padding
  st_relaxed_u64(&st[(size_t)tile * kRadix + tid], tag | (tile == 0 ? kStatusInclusive : kStatusPartial) | cnt);
  uint32_t incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
    if (lane >= (uint32_t)d) incl += t;
  }
  if (lane == 31) sm.wsum[warp] = incl;
  uint32_t bin_start = incl - cnt;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < kTileWarps; ++w)
    if ((uint32_t)w < warp) bin_start += sm.wsum[w];
  {
    uint32_t run = bin_start;
#pragma unroll
    for (int w = 0; w < kTileWarps; ++w) {
      const uint32_t c = sm.hist[w * kRadix + tid];
      sm.hist[w * kRadix + tid] = run;
      run += c;
    }
  }
  __syncthreads();  // offsets visible to everyone

  // ---- into digit order, in place: the 8 B members now, the 4 B members after one more barrier ----
  uint32_t small[ITEMS];
  load_small(small);
#pragma unroll
  for (int u = 0; u < ITEMS; ++u) {
    rank[u] += wh[dig[u]];
    s_big[rank[u]] = big[u];
  }

  // ---- exclusive prefix of this bin over all earlier tiles of the column (decoupled look-back) ----
  sm.goff[tid] = bin_base + lookback_u64(st, tile, epoch, cnt, error_flag) - bin_start;  // + position in tile order = global slot
  __syncthreads();  // every 4 B member has been fetched
#pragma unroll
  for (int u = 0; u < ITEMS; ++u) s_small[rank[u]] = small[u];
  __syncthreads();

  // ---- coalesced runs out to HBM ----
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const uint32_t pos = j * kTileThreads + tid;
    if (FULL || pos < nvalid) {
      const uint32_t g = sm.goff[digit_at(pos)] + pos;
      st_u64_at(out_big, g, s_big[pos]);
      st_u32_at(out_small, g, s_small[pos]);
    }
  }
  // this thread's accesses to the stage (generic proxy) are ordered before the bulk copy (async proxy) that
  // refills it after the next block barrier
  fence_proxy_async();
}

}  // namespace pbl
