// k_tile_tma.cuh -- second kernel of the fused path, warp-specialised: a producer warp feeds the
// tiles' records through a ring of shared-memory stages with TMA bulk copies behind mbarriers,
// four consumer warps turn them into depth.
//
// A tile's +1 / +1 go to packed start|end counters in shared memory, the ends of near reads that
// started before the tile are found by walking back in the sorted order (their number IS the depth
// entering the tile, see k_fused.cuh), far ends come from the buckets, block scan, 128-bit streaming
// stores.  How the work is split:
//   * everything that is latency and bookkeeping -- drawing tickets, resolving them to tiles,
//     loading tile_first, staging records -- is done by ONE thread of a separate warp, several
//     tiles ahead of the consumers, instead of by every thread of the CTA in front of every tile
//     (done that way, ~70 % of the tile kernel's 54 M warp instructions lay outside the scan);
//   * records arrive by cp.async.bulk (one copy per tile: walk-back candidates and own records are
//     contiguous in the sorted order), consumers read them from shared memory;
//   * two barriers per tile (a thread clears exactly the counter vectors it has just read), over
//     the four consumer warps only;
//   * tiles touched by >= 32 768 reads take two 32-bit passes (starts, then ends) over the same
//     8 KB of counters instead of a second counter array, so a CTA needs 8 KB + the ring.
// Tile order: tickets, heavy tiles (listed by k_far_scatter) first, then all tiles in position order.
// The depth does not depend on the order: every tile is self-contained.  A pass may be restricted to
// the tile range [tile_lo, tile_hi) (streaming: successive batches of a sorted file).
#pragma once
#include "k_fused.cuh"
#include "k_stats.cuh"

namespace mcov {

#ifndef MCOV_TT_STAGES
#define MCOV_TT_STAGES 3
#endif
#ifndef MCOV_TT_STAGE_RECS
#define MCOV_TT_STAGE_RECS 1536
#endif
#ifndef MCOV_TT_CTAS
#define MCOV_TT_CTAS 8
#endif
#ifndef MCOV_TT_BATCH
#define MCOV_TT_BATCH 4               // records a thread of a dense tile fetches from global memory before it scatters them
#endif
constexpr int kTtStages = MCOV_TT_STAGES;
constexpr int kTtStageRecs = MCOV_TT_STAGE_RECS;             // records staged per tile (walk-back candidates + own)
constexpr int kTtThreads = kFusedThreads + 32;               // 4 consumer warps + the producer warp
static_assert(kTtStageRecs % 4 == 0, "stage = whole 16-byte vectors");

struct TtMeta {
  int64_t tile;           // < 0: no more tiles
  uint32_t r0, r1, jmin;  // own records [r0, r1); walk-back candidates [jmin, r0)
  uint32_t jb, nst;       // records [jb, jb + nst) are in the stage
  uint32_t touching;      // own records + walk-back candidates + far ends: every +1 the tile can receive
  int32_t carry;          // far reads open at the tile border
  int32_t n_vec;          // 16-byte vectors of the tile inside the depth array (only the last tile is short)
  int32_t pad;
};

// inclusive warp scan step: x += (value of lane - o), lanes below o unchanged -- the shuffle's own predicate guards the
// add (two instructions per step; the C++ form `if (lane >= o) x += y` compiles to SHFL + SEL + IADD)
__device__ __forceinline__ int scan_step_up(int x, int o) {
  int r;
  asm volatile("{ .reg .s32 t; .reg .pred p; shfl.sync.up.b32 t|p, %1, %2, 0, 0xffffffff; @p add.s32 t, t, %1; mov.s32 %0, t; }"
               : "=r"(r) : "r"(x), "r"(o));
  return r;
}
__device__ __forceinline__ int warp_scan_incl(int x) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) x = scan_step_up(x, o);
  return x;
}

// ALL_STAGED: every record the tile looks at is in the stage (the normal case, decided once per tile)
template <bool ALL_STAGED>
__device__ __forceinline__ uint32_t tt_rec(const FusedArgs& f, const TtMeta& m, const uint32_t* s_rec, uint32_t j) {
  const uint32_t k = j - m.jb;
  if (ALL_STAGED) return s_rec[k];
  return k < m.nst ? s_rec[k] : __ldg(f.rec + j);               // dense tiles: what does not fit the stage, from global
}

// scatter of one tile's records into the counters.  WHAT: 0 = packed starts|ends, 1 = starts only, 2 = ends only
template <int WHAT, bool ALL_STAGED>
__device__ __forceinline__ int tt_scatter(const FusedArgs& f, const TtMeta& m, const uint32_t* s_rec, int* s_cnt, uint32_t reach,
                                          bool has_far) {
  const int t = threadIdx.x;
  if (WHAT == 0 && ALL_STAGED) {
    // the common case, branch-free: both atomics of every record are issued; an end beyond the tile goes to the spare
    // counter behind the tile, a record that does not count here (code 0: filtered, or far) to the lane's own spare
    // counter (spares are never read and never cleared)
    const uint32_t spare = (uint32_t)kTile + 1u + (threadIdx.x & 31u);
    const uint32_t* p = s_rec + (m.r0 - m.jb) + t;
    const uint32_t* const pe = s_rec + (m.r1 - m.jb);
#pragma unroll 2
    for (; p < pe; p += kFusedThreads) {
      const uint32_t r = *p;
      const uint32_t code = r >> kTileShift, local = r & (kTile - 1);
      const bool counts = code != 0;
      const uint32_t a = counts ? local : spare;
      const uint32_t e = counts ? min(local + code, (uint32_t)kTile) : spare;
      atomicAdd(&s_cnt[a], 1);
      atomicAdd(&s_cnt[e], 0x10000);
    }
  } else {
    // dense tiles (more records than a stage holds) read theirs from global memory: eight independent loads per thread
    // in flight, THEN the atomics -- one load per iteration behind its atomics is a DRAM round trip per record (a
    // 38 000-read tile of config C3 took 400 us that way and the whole pass waited for it)
    constexpr int kBatch = MCOV_TT_BATCH;
    for (uint32_t j0 = m.r0 + t; j0 < m.r1; j0 += kBatch * kFusedThreads) {
      uint32_t r[kBatch];
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const uint32_t j = j0 + (uint32_t)u * kFusedThreads;
        r[u] = j < m.r1 ? tt_rec<ALL_STAGED>(f, m, s_rec, j) : 0u;           // (code 0: does not count)
      }
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const uint32_t code = r[u] >> kTileShift;
        if (code) {
          const uint32_t local = r[u] & (kTile - 1);
          if (WHAT != 2) atomicAdd(&s_cnt[local], 1);
          const uint32_t el = local + code;
          if (WHAT != 1 && el < (uint32_t)kTile) atomicAdd(&s_cnt[el], WHAT == 0 ? 0x10000 : 1);
        }
      }
    }
  }
  // near reads that started before the tile and end inside it (see k_fused.cuh): walk back while the
  // start is within `reach` slots of the tile; every hit covers the last slot before the tile
  int open = 0;
  if (WHAT != 1) {
    for (uint32_t k = (uint32_t)t; k < m.r0 - m.jmin; k += kFusedThreads) {       // candidate m.r0 - 1 - k (sanitised ranges: jmin <= r0)
      const uint32_t r = tt_rec<ALL_STAGED>(f, m, s_rec, m.r0 - 1u - k);
      const uint32_t d = (uint32_t)kTile - (r & (kTile - 1));
      if (d > reach) break;
      const uint32_t code = r >> kTileShift;
      if (code >= d && code <= kNearSpan) { atomicAdd(&s_cnt[code - d], WHAT == 0 ? 0x10000 : 1); ++open; }
    }
    if (has_far) {
      const uint32_t k0 = m.tile > 0 ? f.tile_cnt[m.tile - 1] : 0u, k1 = f.tile_cnt[m.tile];
      for (uint32_t k = k0 + t; k < k1; k += kFusedThreads) atomicAdd(&s_cnt[f.far_sorted[k] & (kTile - 1)], WHAT == 0 ? 0x10000 : 1);
    }
  }
  return open;
}

// The depth histogram of the previous tile (f.tile_hist): one u16 per consumer thread, and its bins cleared for the
// next tile.  Called after the current tile's first barrier, which every consumer passes only when it has counted the
// previous tile; the current tile counts after its second barrier.
static_assert(kFusedThreads == kTileHistWords, "one histogram word per consumer thread");
static_assert(kHistBins - 1 - kTileHistBins < (int)kTileHistNone, "anchors stay below kTileHistNone");
__device__ __forceinline__ void tt_hist_flush(const FusedArgs& f, uint32_t* s_th, const int* s_th_tile) {
  const int tile = s_th_tile[0];
  if (tile < 0) return;
  const int t = threadIdx.x, b = (t + kTileHistWords - 1) & (kTileHistWords - 1);      // thread 0: the outside-window bin
  const uint32_t c = s_th[b];
  s_th[b] = 0u;
  const int anchor = s_th_tile[1];
  // anchor + kTileHistBins <= kHistBins - 1: the histogram holds no value of the statistics' overflow bin
  const bool ok = c == 0u && anchor + kTileHistBins <= kHistBins - 1;
  f.tile_hist[(int64_t)tile * kTileHistWords + t] = t == 0 ? (ok ? (uint16_t)anchor : kTileHistNone) : (uint16_t)c;
}

// HIST: also write the depth histogram of every tile to f.tile_hist (a pass without histograms runs code without them)
template <bool HIST>
__global__ void __launch_bounds__(kTtThreads, MCOV_TT_CTAS)
k_fused_tile_tma(const __grid_constant__ FusedArgs f) {
  __shared__ __align__(16) int s_cnt[kTile + 36];       // [kTile ..]: spare counters (tt_scatter)
  __shared__ __align__(16) uint32_t s_rec[kTtStages][kTtStageRecs];
  __shared__ __align__(8) uint64_t s_full[kTtStages], s_empty[kTtStages];
  __shared__ TtMeta s_meta[kTtStages];
  __shared__ int s_warp[kFusedThreads / 32], s_warp2[kFusedThreads / 32];
  __shared__ int s_open[2];
  // depth histogram of the tile (f.tile_hist): bins [anchor, anchor + kTileHistBins), then one bin for everything
  // outside; the tile and the anchor it was counted with, kept for tt_hist_flush
  __shared__ uint32_t s_th[kTileHistWords];
  __shared__ int s_th_tile[2];
  PassCounters* pc = f.e.pc;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  {                                                     // (before the dependency wait: touches nothing global)
    int4* z0 = reinterpret_cast<int4*>(s_cnt);
    for (int k = threadIdx.x; k < kTile / 4; k += kTtThreads) z0[k] = make_int4(0, 0, 0, 0);
    if (HIST && threadIdx.x < kTileHistWords) s_th[threadIdx.x] = 0u;
    if (HIST && threadIdx.x == 0) s_th_tile[0] = -1;
    if (threadIdx.x < 2) s_open[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
      for (int s = 0; s < kTtStages; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], kFusedThreads / 32); }
      mbar_fence_init();
    }
  }
  __syncthreads();
  pdl_wait();                                           // records, tile_first and the far tables are complete
  pdl_launch_dependents();

  if (warp == kFusedThreads / 32) {
    // ---------------- producer: one thread ----------------
    if (lane != 0) return;
    const uint32_t n_heavy = pc->n_heavy;
    const bool has_far = pc->n_far != 0;                // else the far tables are all zero and are not read
    const unsigned G = gridDim.x;
    auto resolve = [&](unsigned tk, TtMeta& m) {        // ticket -> tile + its record ranges; tile = -1: skip, -2: past the end
      m.r0 = m.r1 = m.jmin = m.jb = m.nst = 0;
      m.touching = 0; m.carry = 0; m.n_vec = 0; m.pad = 0;
      int64_t T;
      if (tk < n_heavy) T = f.tile_heavy[tk];
      else {
        T = f.tile_lo + (int64_t)(tk - n_heavy);
        if (T >= f.tile_hi) { m.tile = -2; return; }
      }
      m.r0 = f.tile_first[T]; m.r1 = f.tile_first[T + 1];
      m.jmin = T > 0 ? f.tile_first[T - 1] : 0u;
      // unsorted input (the pass is rejected by the verdict) leaves tile_first non-monotone: such a tile is treated
      // as empty, so that no copy or index is formed from an inverted range
      if (!(m.jmin <= m.r0 && m.r0 <= m.r1)) m.r0 = m.r1 = m.jmin = 0u;
      m.touching = m.r1 - m.jmin;
      m.carry = 0;
      if (has_far) {
        const uint32_t k0 = T > 0 ? f.tile_cnt[T - 1] : 0u;
        m.touching += f.tile_cnt[T] - k0;
        if (T > 0) m.carry = f.tile_agg[T - 1];
      }
      m.n_vec = (int32_t)min((int64_t)(kTile / 4), (f.n_slots - (T << kTileShift)) >> 2);
      m.tile = (tk >= n_heavy && n_heavy != 0 && m.r1 - m.r0 >= f.heavy_min) ? -1 : T;   // a heavy tile met again in position order
    };
    TtMeta m_cur, m_nxt;
    resolve(blockIdx.x, m_cur);
    unsigned tk_nxt = blockIdx.x + G;
    unsigned it = 0;
    while (true) {
      // the ticket after next (one atomic per tile) and the metadata of the next tile: in flight while this tile is published
      const unsigned tk_new = 2u * G + atomicAdd(&pc->ticket2, 1u);
      resolve(tk_nxt, m_nxt);
      if (m_cur.tile != -1) {
        const unsigned s = it % kTtStages, k = it / kTtStages;
        if (k > 0) mbar_wait_relaxed(&s_empty[s], (k - 1) & 1);
        if (m_cur.tile >= 0) {
          m_cur.jb = m_cur.jmin & ~3u;
          const uint32_t want = ((m_cur.r1 + 3u) & ~3u) - m_cur.jb;        // (the record buffer is padded past n)
          m_cur.nst = min(want, (uint32_t)kTtStageRecs);
        }
        s_meta[s] = m_cur;
        if (m_cur.tile >= 0 && m_cur.nst) {
          mbar_arrive_expect_tx(&s_full[s], 4u * m_cur.nst);
          tma_load_1d(&s_rec[s][0], f.rec + m_cur.jb, 4u * m_cur.nst, &s_full[s]);
        } else {
          mbar_arrive(&s_full[s]);
        }
        ++it;
        if (m_cur.tile < 0) break;                      // -2: the consumers have been told to stop
      }
      m_cur = m_nxt; tk_nxt = tk_new;
    }
    return;
  }

  // ---------------- consumers: 4 warps ----------------
  const uint32_t reach = pc->max_span;                  // written by the prep kernel
  const bool has_far = pc->n_far != 0;                  // else the far tables are all zero and are not read
  int mx = 0, cap = 0;
  int par = 0;
  unsigned s = 0, ph = 0;                                 // stage of this iteration and the parity of its "full" phase
#pragma unroll 1
  for (;; par ^= 1, s = (s + 1 == kTtStages) ? 0u : s + 1, ph ^= (s == 0) ? 1u : 0u) {
    mbar_wait(&s_full[s], ph);
    const TtMeta m = s_meta[s];
    if (m.tile < 0) break;
    const uint32_t* rec = s_rec[s];
    // every +1 of the tile comes from an own record, a walk-back candidate or a far end: fewer than 32 768 of
    // them keep both halves of the packed counters within a signed 16-bit value (the scan below subtracts the halves
    // with one two-way dot product per slot)
    const bool packed = m.touching < 32768u;
    // v[j] = prefix sums of (starts - ends) inside vector j; capv[j] = max over its slots of (prefix before the slot +
    // starts of the slot): cap[p] = depth[p-1] + starts[p] relative to the vector's incoming depth.
    // Vectors are warp-striped, so a warp's 128-bit depth stores are contiguous; a blocked layout (one warp scan per
    // thread instead of four) half-fills every store's sectors and measured slower (DESIGN.md 3.1).
    int4 v[kTileVec];
    int capv[kTileVec];
    if (packed) {
      int open = (m.r1 - m.jb <= m.nst) ? tt_scatter<0, true>(f, m, rec, s_cnt, reach, has_far)
                                        : tt_scatter<0, false>(f, m, rec, s_cnt, reach, has_far);
      open = __reduce_add_sync(0xffffffffu, open);
      if (lane == 0) { if (open) atomicAdd(&s_open[par], open); mbar_arrive(&s_empty[s]); }   // stage free: the records have been read
      named_bar_sync<1, kFusedThreads>();
      if (HIST) tt_hist_flush(f, s_th, s_th_tile);
      const int4* vs = reinterpret_cast<const int4*>(s_cnt);
#pragma unroll
      for (int j = 0; j < kTileVec; ++j) {
        const int idx = (warp * kTileVec + j) * 32 + lane;
        const int4 c = vs[idx];
        reinterpret_cast<int4*>(s_cnt)[idx] = make_int4(0, 0, 0, 0);      // cleared by the thread that read it
        // starts - ends of a packed counter, accumulated: ONE instruction (IDP.2A: lo * 1 + hi * -1 + acc)
        constexpr int kPlusMinus = 0x0000FF01;
        v[j].x = __dp2a_lo(c.x, kPlusMinus, 0);
        v[j].y = __dp2a_lo(c.y, kPlusMinus, v[j].x);
        v[j].z = __dp2a_lo(c.z, kPlusMinus, v[j].y);
        v[j].w = __dp2a_lo(c.w, kPlusMinus, v[j].z);
        capv[j] = max(max(c.x & 0xffff, v[j].x + (c.y & 0xffff)), max(v[j].y + (c.z & 0xffff), v[j].z + (c.w & 0xffff)));
      }
    } else {
      int4 st[kTileVec], en[kTileVec];
      // dense tile: starts and ends counted in two 32-bit passes over the same counters
      tt_scatter<1, false>(f, m, rec, s_cnt, reach, has_far);
      named_bar_sync<1, kFusedThreads>();
      if (HIST) tt_hist_flush(f, s_th, s_th_tile);
#pragma unroll
      for (int j = 0; j < kTileVec; ++j) {
        const int idx = (warp * kTileVec + j) * 32 + lane;
        st[j] = reinterpret_cast<const int4*>(s_cnt)[idx];
        reinterpret_cast<int4*>(s_cnt)[idx] = make_int4(0, 0, 0, 0);
      }
      named_bar_sync<1, kFusedThreads>();
      int open = tt_scatter<2, false>(f, m, rec, s_cnt, reach, has_far);
      open = __reduce_add_sync(0xffffffffu, open);
      if (lane == 0) { if (open) atomicAdd(&s_open[par], open); mbar_arrive(&s_empty[s]); }
      named_bar_sync<1, kFusedThreads>();
#pragma unroll
      for (int j = 0; j < kTileVec; ++j) {
        const int idx = (warp * kTileVec + j) * 32 + lane;
        en[j] = reinterpret_cast<const int4*>(s_cnt)[idx];
        reinterpret_cast<int4*>(s_cnt)[idx] = make_int4(0, 0, 0, 0);
        v[j].x = st[j].x - en[j].x;
        v[j].y = v[j].x + st[j].y - en[j].y;
        v[j].z = v[j].y + st[j].z - en[j].z;
        v[j].w = v[j].z + st[j].w - en[j].w;
        capv[j] = max(max(st[j].x, v[j].x + st[j].y), max(v[j].y + st[j].z, v[j].z + st[j].w));
      }
    }
    // block scan of (starts - ends).  cap[p] = depth[p-1] + starts[p] is folded into one value per vector, relative
    // to the vector's incoming depth.  run[j] = exclusive offset of vector j inside the warp's 512 slots.
    int run[kTileVec];
#pragma unroll
    for (int j = 0; j < kTileVec; ++j) run[j] = v[j].w;
    int acc = 0;
    if (packed) {
      // the totals of two rows share one scan: |partial sums| < 32 768 in a packed tile, so two signed 16-bit
      // halves add independently modulo a borrow that the unpacking undoes (lo = sign-extended low half,
      // hi = (x - lo) >> 16)
      const int p01 = run[1] * 65536 + run[0], p23 = run[3] * 65536 + run[2];
      const int x01 = warp_scan_incl(p01), x23 = warp_scan_incl(p23);
      const int t01 = __shfl_sync(0xffffffffu, x01, 31), t23 = __shfl_sync(0xffffffffu, x23, 31);
      const int e01 = x01 - p01, e23 = x23 - p23;                          // exclusive, still packed
      const int e0 = __dp2a_lo(e01, 0x0001, 0), e2 = __dp2a_lo(e23, 0x0001, 0);
      const int e1 = (e01 - e0) >> 16, e3 = (e23 - e2) >> 16;
      const int T0 = __dp2a_lo(t01, 0x0001, 0), T2 = __dp2a_lo(t23, 0x0001, 0);
      const int T1 = (t01 - T0) >> 16, T3 = (t23 - T2) >> 16;
      run[0] = e0; run[1] = e1 + T0; run[2] = e2 + T0 + T1; run[3] = e3 + T0 + T1 + T2;
      acc = T0 + T1 + T2 + T3;
    } else {
#pragma unroll
      for (int j = 0; j < kTileVec; ++j) {
        int x = run[j];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, x, o);
          if (lane >= o) x += y;
        }
        const int total = __shfl_sync(0xffffffffu, x, 31);
        run[j] = x - run[j] + acc;
        acc += total;
      }
    }
    if (lane == 31) s_warp[warp] = acc;
    // the other s_open buffer: last read after the previous tile's second barrier (every thread has passed this
    // tile's first barrier since), next added to after this tile's second barrier
    if (threadIdx.x == 0) s_open[par ^ 1] = 0;
    named_bar_sync<1, kFusedThreads>();
    int off = m.carry + s_open[par];                     // far reads + near reads open at the border
    // the histogram window is centred on the depth entering the tile
    const int anchor = max(0, off - kTileHistBins / 2);
    if (HIST && threadIdx.x == 0) { s_th_tile[0] = (int)m.tile; s_th_tile[1] = anchor; }
#pragma unroll
    for (int w = 0; w < kFusedThreads / 32; ++w) off += (w < warp) ? s_warp[w] : 0;
    const int64_t base = m.tile << kTileShift;
    int4* out = reinterpret_cast<int4*>(f.depth + base);
    const int n_vec = m.n_vec;
    int cap_t = 0;
#pragma unroll
    for (int j = 0; j < kTileVec; ++j) {
      const int idx = (warp * kTileVec + j) * 32 + lane;
      const int o = off + run[j];
      cap_t = max(cap_t, o + capv[j]);
      v[j].x += o; v[j].y += o; v[j].z += o; v[j].w += o;
      mx = max(mx, max(max(v[j].x, v[j].y), max(v[j].z, v[j].w)));
      if (idx < n_vec) {
        st_stream_int4(out + idx, v[j]);
        if (HIST) {
          // plain +1 updates (ATOMS.POPC.INC, see hist_vec); a value outside the window lands in the last bin
          atomicAdd(&s_th[min((unsigned)(v[j].x - anchor), (unsigned)kTileHistBins)], 1u);
          atomicAdd(&s_th[min((unsigned)(v[j].y - anchor), (unsigned)kTileHistBins)], 1u);
          atomicAdd(&s_th[min((unsigned)(v[j].z - anchor), (unsigned)kTileHistBins)], 1u);
          atomicAdd(&s_th[min((unsigned)(v[j].w - anchor), (unsigned)kTileHistBins)], 1u);
        }
      }
    }
    cap = max(cap, cap_t);
    // htslib's cap could fire somewhere in this tile (rare): remember the tile for the exact replay
    if (f.max_depth > 0 && cap_t > f.max_depth) atomicMax(f.tile_cap + m.tile, cap_t);
  }
  mx = warp_max(mx);
  cap = warp_max(cap);
  if (lane == 0) { s_warp2[warp] = cap; }
  named_bar_sync<1, kFusedThreads>();                    // (s_warp of the last tile has been read by everyone)
  if (HIST) tt_hist_flush(f, s_th, s_th_tile);
  if (lane == 0) s_warp[warp] = mx;
  named_bar_sync<1, kFusedThreads>();
  if (threadIdx.x == 0) {
    int m2 = 0, c2 = 0;
    for (int w = 0; w < kFusedThreads / 32; ++w) { m2 = max(m2, s_warp[w]); c2 = max(c2, s_warp2[w]); }
    if (m2 > 0) atomicMax(&pc->max_depth_seen, m2);
    if (c2 > 0) atomicMax(&pc->cap_metric, c2);
  }
}

}  // namespace mcov
