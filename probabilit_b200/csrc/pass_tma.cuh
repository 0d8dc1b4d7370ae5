// The onesweep digit pass as a PERSISTENT kernel with double-buffered bulk-async (TMA) tile loads.
// Included by sort.cu (inside namespace pbl, after PassArgs).
//
// A CTA of 8 warps loops over tiles of 4096 keys.  Each tile lives in one of two 48 KB shared-memory
// stages: thread 0 takes the ticket (col, tile) of the NEXT tile while the current one is being ranked,
// arms that stage's mbarrier with the byte count and issues cp.async.bulk.shared.global for the tile's
// keys (8 B each, or the caller's raw doubles in the first pass) and rows (4 B each) -- SASS: UBLKCP +
// SYNCS -- as soon as the first block barrier of the current tile has shown that the stage's previous
// occupant has been written out.  The warps wait on the mbarrier, pull their 16 keys + rows out of
// the stage into registers (conflict-free LDS), rank them (rank.cuh), and then REUSE the stage as the
// digit-ordered staging area from which coalesced runs go out to HBM.  Two CTAs per SM: while a tile
// is ranked and written out, the next one is already landing, and its ticket was taken a tile
// earlier, so that neither the global-load latency nor the ticket's L2 round trip is on the critical path.
//
// Look-back words: 64-bit, epoch-tagged (sort.cuh) -- the array is never cleared between passes.
//
// Global addresses of a tile are only 8 B (keys) / 4 B (rows) aligned when the column length is odd;
// a bulk copy needs 16 B: the copy covers the enclosing aligned range and the ticket carries the
// offset of the first element (the buffers have 16 B of slack at the end, see ic_plan_create).
#pragma once

constexpr int kTmaTile = kTile;
constexpr uint32_t kTmaKeyBytes = (kTile + 2) * 8;  // + one 16 B unit of alignment slack
constexpr uint32_t kTmaValBytes = (kTile + 4) * 4;
constexpr uint32_t kTmaStageBytes = kTmaKeyBytes + kTmaValBytes;
constexpr size_t kTmaSmemBytes = 2 * (size_t)kTmaStageBytes + kSplitSmemBytes + 2 * 32 + 2 * 8;

enum TmaMode : uint32_t { kModeBuffers = 0, kModeRawBulk = 1, kModeRawDirect = 2, kModeEnd = 3 };
struct __align__(16) TmaTicket {
  uint32_t col, tile, nvalid;
  uint32_t mode_off;  // mode | key offset << 8 | row offset << 16   (offsets in elements inside the stage)
  uint32_t dshift;    // digit = (compact key >> dshift) & 255
  uint32_t dst;       // ping-pong buffer the pass writes (1 = A, 2 = B)
  uint32_t pad[2];
};

struct TmaArgs {
  PassArgs p;
  const KeyMap* maps;       // [ncols], written by sort_scan_kernel
  uint64_t* status64;       // [ncols][ntiles][256]
  uint32_t* ticket;         // one counter for the launch
  uint32_t total_tiles;     // ncols * ntiles
  uint32_t epoch;           // 1 .. 2^28, different for every launch that uses status64
  uint32_t ncols;
  // Ticket order (ticket_to_tile): width of the column groups whose tiles are interleaved.
  uint32_t ncols_interleave;
};


// Thread 0 only: decode ticket g (columns that skip this pass are stepped over with further tickets),
// publish it in s_tk and start the bulk copies of its tile into `stage` (completion on `full`).
__device__ __forceinline__ void tma_issue(const TmaArgs& a, uint32_t g, TmaTicket* s_tk, uint32_t stage, uint32_t full) {
  const int pass = a.p.pass;
  const uint32_t ntiles = (uint32_t)a.p.ntiles;
  TmaTicket tk;
  int src = 0;
  for (;;) {
    if (g >= a.total_tiles) {
      tk.col = tk.tile = tk.nvalid = tk.dshift = tk.dst = tk.pad[0] = tk.pad[1] = 0;
      tk.mode_off = kModeEnd;
      *s_tk = tk;
      mbar_arrive(full);
      return;
    }
    ticket_to_tile(g, a.ncols, ntiles, a.ncols_interleave, &tk.col, &tk.tile);
    if (a.p.plan[tk.col].run[pass]) break;
    g = atomicAdd(a.ticket, 1u);  // constant digit: the column sits this pass out
  }
  src = a.p.plan[tk.col].src[pass];
  tk.dst = (src == 1) ? 2u : 1u;
  tk.dshift = a.maps[tk.col].sh + (uint32_t)pass * kRadixBits;
  tk.pad[0] = tk.pad[1] = 0;
  tk.nvalid = min((uint32_t)kTmaTile, a.p.n - tk.tile * (uint32_t)kTmaTile);
  const size_t first = (size_t)tk.col * a.p.n + (size_t)tk.tile * kTmaTile;
  // the stage was last touched through the generic proxy (the previous occupant's staging); the barrier
  // that let this thread get here ordered those accesses, the fence hands the stage to the async proxy
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (src == 0) {
    const double* gp = a.p.raw + (int64_t)tk.col * a.p.col_stride + (int64_t)tk.tile * kTmaTile * a.p.row_stride;
    const bool bulk = a.p.row_stride == 1 && ((uintptr_t)gp & 15u) == 0 && (tk.nvalid & 1u) == 0;
    tk.mode_off = bulk ? kModeRawBulk : kModeRawDirect;
    *s_tk = tk;
    if (bulk) {
      mbar_arrive_expect_tx(full, tk.nvalid * 8u);
      bulk_g2s(stage, gp, tk.nvalid * 8u, full);
    } else {
      mbar_arrive(full);
    }
  } else {
    const uint64_t* gk = (src == 1 ? a.p.keysA : a.p.keysB) + first;
    const uint32_t* gv = (src == 1 ? a.p.valsA : a.p.valsB) + first;
    const uint32_t mk = (uint32_t)((uintptr_t)gk & 15u), mv = (uint32_t)((uintptr_t)gv & 15u);
    const uint32_t kb = (mk + tk.nvalid * 8u + 15u) & ~15u, vb = (mv + tk.nvalid * 4u + 15u) & ~15u;
    tk.mode_off = kModeBuffers | ((mk >> 3) << 8) | ((mv >> 2) << 16);
    *s_tk = tk;
    mbar_arrive_expect_tx(full, kb + vb);
    bulk_g2s(stage, reinterpret_cast<const unsigned char*>(gk) - mk, kb, full);
    bulk_g2s(stage + kTmaKeyBytes, reinterpret_cast<const unsigned char*>(gv) - mv, vb, full);
  }
}

struct TmaSmem {
  unsigned char* stage0;  // two stages, kTmaStageBytes apart
  SplitSmem split;
  TmaTicket* tk;    // [2]
  uint32_t full0;   // shared-space address of the two mbarriers (8 B apart)
  __device__ __forceinline__ unsigned char* stage(uint32_t s) const { return stage0 + s * kTmaStageBytes; }
  __device__ __forceinline__ uint32_t full(uint32_t s) const { return full0 + 8u * s; }
};

template <bool FULL>
__device__ __forceinline__ void tma_tile(const TmaArgs& a, const TmaSmem& sm, const uint32_t s, const TmaTicket tk) {
  constexpr int ITEMS = kTileItems;
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t n = a.p.n;
  const uint32_t col = tk.col, tile = tk.tile, nvalid = tk.nvalid, dshift = tk.dshift, dst = tk.dst;
  // global slot of this thread's bin: asked for now, needed after the look-back
  const uint32_t bin_base = a.p.bin_base_all[((size_t)col * kMaxPasses + a.p.pass) * kRadix + tid];
  const uint32_t mode = tk.mode_off & 255u, koff = (tk.mode_off >> 8) & 255u, voff = (tk.mode_off >> 16) & 255u;
  const uint32_t tile_start = tile * (uint32_t)kTile;
  const uint32_t pos0 = warp * (ITEMS * 32) + lane;
  uint64_t* s_keys = reinterpret_cast<uint64_t*>(sm.stage(s));
  uint32_t* s_vals = reinterpret_cast<uint32_t*>(sm.stage(s) + kTmaKeyBytes);

  // the ticket of the tile after this one: asked for now, needed after the first barrier
  uint32_t next_ticket = 0;
  if (tid == 0) next_ticket = atomicAdd(a.ticket, 1u);

  // ---- keys: stage -> registers ----
  uint64_t key[ITEMS];
  uint32_t negzero = 0;  // raw input: bit u set if item u was -0.0
  if (mode == kModeBuffers) {
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) key[u] = (FULL || pos0 + u * 32 < nvalid) ? s_keys[koff + pos0 + u * 32] : 0ull;
  } else {
    // first pass of a column: the caller's doubles (a bulk copy landed them in the key area, or -- strided /
    // misaligned input -- straight from global memory); the payload is the row index + the -0.0 flag
    const double* colp = a.p.raw + (int64_t)col * a.p.col_stride + (int64_t)(tile_start + pos0) * a.p.row_stride;
    const int64_t step = 32 * a.p.row_stride;
    const double* s_raw = reinterpret_cast<const double*>(sm.stage(s));
    const KeyMap map = a.maps[col];
    double d[ITEMS];
    if (mode == kModeRawBulk) {
#pragma unroll
      for (int u = 0; u < ITEMS; ++u) d[u] = (FULL || pos0 + u * 32 < nvalid) ? s_raw[pos0 + u * 32] : 0.0;
    } else {
#pragma unroll
      for (int u = 0; u < ITEMS; ++u) d[u] = (FULL || pos0 + u * 32 < nvalid) ? ld_stream_f64(colp + u * step) : 0.0;
    }
    const FusedKeyMap fmap = fused_key_map(map);
#pragma unroll
    for (int u = 0; u < ITEMS; ++u) {
      bool nz;
      key[u] = compact_key_of_double(d[u], fmap, &nz);
      negzero |= (nz ? 1u : 0u) << u;
    }
  }
  uint32_t dig[ITEMS];
#pragma unroll
  for (int u = 0; u < ITEMS; ++u) {
    dig[u] = (uint32_t)(key[u] >> dshift) & (uint32_t)(kRadix - 1);
    // padding of a partial tile goes to the last bin, behind every real key of the tile
    if (!FULL && pos0 + u * 32 >= nvalid) dig[u] = (uint32_t)(kRadix - 1);
  }

  // the rows are only fetched once the keys have been staged (keeps them out of the registers while the
  // keys are ranked); the first pass synthesises them
  auto load_rows = [&](uint32_t (&val)[ITEMS]) {
    if (mode == kModeBuffers) {
#pragma unroll
      for (int u = 0; u < ITEMS; ++u) val[u] = (FULL || pos0 + u * 32 < nvalid) ? s_vals[voff + pos0 + u * 32] : 0u;
    } else {
#pragma unroll
      for (int u = 0; u < ITEMS; ++u)
        val[u] = (tile_start + pos0 + u * 32) | (((negzero >> u) & 1u) ? kNegZeroFlag : 0u);
    }
  };
  auto digit_at = [&](uint32_t pos) { return (uint32_t)(s_keys[pos] >> dshift) & (uint32_t)(kRadix - 1); };
  // after the first barrier every warp has finished writing out the PREVIOUS tile: its stage takes the next one
  auto prefetch = [&]() {
    if (tid == 0) tma_issue(a, next_ticket, &sm.tk[s ^ 1u], smem_u32(sm.stage(s ^ 1u)), sm.full(s ^ 1u));
  };
  split_tile<FULL>(dig, key, load_rows, digit_at, prefetch, sm.split, s_keys, s_vals,
                   a.status64 + ((size_t)col * a.p.ntiles) * kRadix, tile, nvalid, a.epoch, bin_base,
                   (dst == 1 ? a.p.keysA : a.p.keysB) + (size_t)col * n,
                   (dst == 1 ? a.p.valsA : a.p.valsB) + (size_t)col * n, a.p.error_flag);
}

__global__ void __launch_bounds__(kTileThreads, 2) pass_tma_kernel(const TmaArgs a) {
  extern __shared__ __align__(128) unsigned char tsm[];
  TmaSmem sm;
  sm.stage0 = tsm;
  sm.split.hist = reinterpret_cast<uint32_t*>(tsm + 2 * kTmaStageBytes);
  sm.split.goff = sm.split.hist + kTileWarps * kRadix;
  sm.split.wsum = sm.split.goff + kRadix;                   // [8] (+8 pad)
  sm.tk = reinterpret_cast<TmaTicket*>(sm.split.wsum + 16);  // [2]
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(sm.tk + 2);  // full[2]
  sm.full0 = smem_u32(s_bar);
  const uint32_t tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(sm.full(0), 1);
    mbar_init(sm.full(1), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tma_issue(a, atomicAdd(a.ticket, 1u), &sm.tk[0], smem_u32(sm.stage(0)), sm.full(0));
  }
  __syncthreads();
  for (uint32_t it = 0;; ++it) {
    const uint32_t s = it & 1u;
#ifdef PBL_TILE_STATS
    const long long w0 = clock64();
#endif
    mbar_wait(sm.full(s), (it >> 1) & 1u, a.p.error_flag);
#ifdef PBL_TILE_STATS
    const long long w1 = clock64();
#endif
    const TmaTicket tk = sm.tk[s];
    if ((tk.mode_off & 255u) == kModeEnd) break;
    if (tk.nvalid == (uint32_t)kTmaTile)
      tma_tile<true>(a, sm, s, tk);
    else
      tma_tile<false>(a, sm, s, tk);
#ifdef PBL_TILE_STATS
    if (tid == 0) {
      atomicAdd(&g_tile_stats[0], 1ull);
      atomicAdd(&g_tile_stats[4], (unsigned long long)(clock64() - w1));
      atomicAdd(&g_tile_stats[5], (unsigned long long)(w1 - w0));
    }
#endif
  }
}
