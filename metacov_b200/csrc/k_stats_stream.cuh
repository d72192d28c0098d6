// k_stats_stream.cuh -- region statistics as ONE balanced stream over the depth (large regions).
//
// One CTA per region (or per chunk of a region) leaves the machine badly balanced: on config C2,
// 1 000 equal CTAs on 592 resident slots = 1.69 waves, each CTA starting with a cold pipeline and
// ending with a clear / walk during which it loads nothing (DESIGN.md 3.3).  Here the
// concatenation of all large regions is cut into EQUAL slices, one per persistent CTA (2 per SM),
// whatever the region boundaries are:
//   * a producer warp streams the CTA's slice through a ring of 16 KB shared-memory stages with
//     TMA bulk copies behind mbarriers -- it runs ahead across region boundaries, so the stream
//     never stops while the consumers finish a region;
//   * 8 consumer warps feed the exact counting histogram (8192 one-value bins, ATOMS.POPC.INC)
//     from shared memory;
//   * a region that lies wholly inside a slice is walked and written by its CTA; a region cut by
//     a slice border (at most one per border) adds its touched bins to a per-split-region
//     histogram in global memory (fire-and-forget reductions, nobody waits), and the CTA whose
//     piece of it arrives last pulls the merged bin range back and walks the region.
// The walk is hist_walk (k_stats.cuh), the same as for the small regions.
//
// When the tile kernel has left a depth histogram of every tile (FusedArgs::tile_hist, k_fused.cuh) that still
// describes the depth, the tiles that lie wholly inside a piece are counted from their histograms (256 bytes each
// instead of 8 KB of depth); only the piece's ends, and the tiles whose depth left the histogram's window, are read
// from the depth.
#pragma once
#include "k_fused.cuh"
#include "k_stats.cuh"

namespace mcov {

#ifndef MCOV_SS_STAGES
#define MCOV_SS_STAGES 4
#endif
#ifndef MCOV_SS_BLK
#define MCOV_SS_BLK 4096
#endif
#ifndef MCOV_SS_CTAS
#define MCOV_SS_CTAS 2
#endif
constexpr int kSsStages = MCOV_SS_STAGES;
constexpr int kSsBlk = MCOV_SS_BLK;                  // slots per stage (16 KB)
constexpr int kSsConsumers = 256;
constexpr int kSsThreads = kSsConsumers + 32;
constexpr int kSsSmemBytes = kSsStages * kSsBlk * 4 + kHistBins * 4;

struct SsPiece {          // a region, or the part of a region inside one slice
  int64_t slot;           // first slot
  int32_t n;              // slots
  int32_t region;
  int32_t pad;            // zeros to add to bin 0 (positions beyond the contig end; first piece of the region only)
  int32_t split;          // -1: the whole region is this piece; else index of the region's global histogram
};

// cnt < 0: end of the slice.  tile < 0: the stage holds depth, valid elements [skip, skip + cnt); else the histograms
// of the cnt tiles from `tile` on
struct SsDesc { int32_t region, split, pad, skip, cnt, last, tile; };
constexpr int kSsHistTiles = kSsBlk * 4 / (kTileHistWords * 2);     // tile histograms per stage

struct SsArgs {
  const int32_t* depth;
  const SsPiece* pieces;
  const int32_t* cta_piece_start;   // [grid + 1]
  const int32_t* region_len;
  const int32_t* region_pad;
  uint32_t* split_hist;             // [n_split][kHistBins], zero between runs
  RegionScratch* split_scratch;     // [n_split] arrival counter + bin range of the merged histogram, zero between runs
  const int32_t* split_pieces;      // [n_split] pieces of the split region: the CTA that merges the last one walks the region
  const uint16_t* tile_hist;        // [n_tiles][kTileHistWords] histograms of the depth's tiles (k_fused.cuh), nullptr: none
  mcov_region_stats* out;
  int32_t breadth_n;
};

__global__ void __launch_bounds__(kSsThreads, MCOV_SS_CTAS)
k_stats_stream(const __grid_constant__ SsArgs a) {
  extern __shared__ __align__(128) char ss_smem[];
  int32_t* s_ring = reinterpret_cast<int32_t*>(ss_smem);
  uint32_t* s_hist = reinterpret_cast<uint32_t*>(ss_smem + (size_t)kSsStages * kSsBlk * 4);
  __shared__ __align__(8) uint64_t s_full[kSsStages], s_empty[kSsStages];
  __shared__ SsDesc s_desc[kSsStages];
  __shared__ unsigned long long s_u64[6 * (kSsConsumers / 32)];
  __shared__ int s_i32[4 * (kSsConsumers / 32)];
  __shared__ int s_med[2];
  __shared__ int s_last;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  {
    uint4* h4 = reinterpret_cast<uint4*>(s_hist);
    for (int k = t; k < kHistBins / 4; k += kSsThreads) h4[k] = make_uint4(0, 0, 0, 0);
    if (t == 0) {
      for (int s = 0; s < kSsStages; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], kSsConsumers / 32); }
      mbar_fence_init();
    }
  }
  __syncthreads();
  pdl_wait();                                           // the depth is complete
  pdl_launch_dependents();
  const int p0 = a.cta_piece_start[blockIdx.x], p1 = a.cta_piece_start[blockIdx.x + 1];

  if (warp == kSsConsumers / 32) {
    // ---------------- producer: one thread streams the slice ----------------
    if (lane != 0) return;
    const uint64_t pol = l2_policy_evict_first();
    unsigned it = 0;
    auto publish = [&](const SsDesc& d, const int32_t* src, uint32_t bytes) {
      const unsigned s = it % kSsStages, k = it / kSsStages;
      if (k > 0) mbar_wait_relaxed(&s_empty[s], (k - 1) & 1);
      s_desc[s] = d;
      if (bytes) {
        mbar_arrive_expect_tx(&s_full[s], bytes);
        tma_load_1d_hint(s_ring + (size_t)s * kSsBlk, src, bytes, &s_full[s], pol);
      } else {
        mbar_arrive(&s_full[s]);
      }
      ++it;
    };
    // the depth of the slots [s0, s1) of a piece; `last`: the piece ends there (a piece without slots still finishes its region)
    auto depth_stages = [&](const SsPiece& pc, int64_t s0, int64_t s1, bool last) {
      const int64_t a0 = s0 & ~(int64_t)3;
      const int64_t nblk = s1 > s0 ? (s1 - a0 + kSsBlk - 1) / kSsBlk : (last ? 1 : 0);
      for (int64_t k = 0; k < nblk; ++k) {
        const int64_t b0 = a0 + k * kSsBlk;
        const int64_t lo = max(b0, s0), hi = min(b0 + kSsBlk, s1);
        SsDesc d;
        d.region = pc.region; d.split = pc.split; d.pad = pc.pad; d.tile = -1;
        d.skip = (int32_t)(lo - b0); d.cnt = (int32_t)max((int64_t)0, hi - lo); d.last = (last && k == nblk - 1) ? 1 : 0;
        const uint32_t bytes = d.cnt > 0 ? (uint32_t)((d.skip + d.cnt + 3) & ~3) * 4u : 0u;   // whole 16-byte vectors inside the padded depth array
        publish(d, a.depth + b0, bytes);
      }
    };
    for (int p = p0; p < p1; ++p) {
      const SsPiece pc = a.pieces[p];
      const int64_t end = pc.slot + pc.n;
      // tiles [t0, t1) lie wholly inside the piece
      const int64_t t0 = a.tile_hist ? (pc.slot + kTile - 1) >> kTileShift : 0, t1 = a.tile_hist ? end >> kTileShift : 0;
      if (t1 <= t0) { depth_stages(pc, pc.slot, end, true); continue; }
      depth_stages(pc, pc.slot, t0 << kTileShift, false);
      for (int64_t t = t0; t < t1; t += kSsHistTiles) {
        SsDesc d;
        d.region = pc.region; d.split = pc.split; d.pad = pc.pad;
        d.skip = 0; d.cnt = (int32_t)min((int64_t)kSsHistTiles, t1 - t); d.last = 0; d.tile = (int32_t)t;
        publish(d, reinterpret_cast<const int32_t*>(a.tile_hist + t * kTileHistWords), (uint32_t)d.cnt * kTileHistWords * 2u);
      }
      depth_stages(pc, t1 << kTileShift, end, true);
    }
    SsDesc e; e.region = -1; e.split = -1; e.pad = 0; e.skip = 0; e.cnt = -1; e.last = 0; e.tile = -1;
    publish(e, nullptr, 0u);
    return;
  }

  // ---------------- consumers ----------------
  int lo = kHistBins, hi = -1;
#pragma unroll 1
  for (unsigned it = 0;; ++it) {
    const unsigned s = it % kSsStages, k = it / kSsStages;
    mbar_wait(&s_full[s], k & 1);
    const SsDesc d = s_desc[s];
    if (d.cnt < 0) break;
    if (d.tile >= 0) {
      // 64 threads per tile histogram, a u32 (two u16 words) each: word 2w holds bin 2w - 1, word 2w + 1 bin 2w
      const uint32_t* h = reinterpret_cast<const uint32_t*>(s_ring + (size_t)s * kSsBlk);
      constexpr int kPer = kTileHistWords / 2;
      for (int q = t; q < d.cnt * kPer; q += kSsConsumers) {
        const int r = q / kPer, w = q % kPer;
        const int anchor = (int)(h[r * kPer] & 0xffffu);
        if (anchor != kTileHistNone) {
          const uint32_t x = h[q];
          const int b = anchor + 2 * w;
          if (w > 0 && (x & 0xffffu)) { atomicAdd(&s_hist[b - 1], x & 0xffffu); lo = min(lo, b - 1); hi = max(hi, b - 1); }
          if (x >> 16) { atomicAdd(&s_hist[b], x >> 16); lo = min(lo, b); hi = max(hi, b); }
        } else {
          // no histogram: the tile's depth, read by the 64 threads of its histogram (eight loads in flight each)
          const int4* v = reinterpret_cast<const int4*>(a.depth + ((int64_t)(d.tile + r) << kTileShift)) + w;
          int4 x[kTile / 4 / kPer];
#pragma unroll
          for (int u = 0; u < kTile / 4 / kPer; ++u) x[u] = __ldcs(v + u * kPer);
#pragma unroll
          for (int u = 0; u < kTile / 4 / kPer; ++u) hist_vec(s_hist, x[u], lo, hi);
        }
      }
    } else if (d.cnt > 0) {
      const int4* v = reinterpret_cast<const int4*>(s_ring + (size_t)s * kSsBlk);
      const int stop = d.skip + d.cnt;                                  // valid elements [skip, stop)
      const int nvec = (stop + 3) >> 2;
      const int tail = stop & 3;
      const int jf0 = d.skip ? 1 : 0, jf1 = nvec - (tail ? 1 : 0);       // full vectors [jf0, jf1)
      for (int j = jf0 + t; j < jf1; j += kSsConsumers) hist_vec(s_hist, v[j], lo, hi);
      if (nvec == 1) { if (t == 0 && (d.skip || tail)) hist_partial(s_hist, v[0], d.skip, stop, lo, hi); }
      else {
        if (t == 0 && d.skip) hist_partial(s_hist, v[0], d.skip, 4, lo, hi);
        if (t == 32 && tail) hist_partial(s_hist, v[nvec - 1], 0, tail, lo, hi);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&s_empty[s]);                             // the stage may be refilled
    if (!d.last) continue;
    // ---- end of a piece: bin range over the CTA, then walk (whole region) or merge (split region) ----
    lo = warp_min(lo); hi = warp_max(hi);
    if (lane == 0) { s_i32[warp] = lo; s_i32[kSsConsumers / 32 + warp] = hi; }
    named_bar_sync<1, kSsConsumers>();                                  // also: the histogram of the piece is complete
    lo = kHistBins; hi = -1;
#pragma unroll
    for (int w = 0; w < kSsConsumers / 32; ++w) { lo = min(lo, s_i32[w]); hi = max(hi, s_i32[kSsConsumers / 32 + w]); }
    if (d.split < 0) {
      if (d.pad > 0) {                                                   // zeros beyond the contig end join the multiset
        if (t == 0) s_hist[0] += (uint32_t)d.pad;
        if (hi < 0) hi = 0;
        lo = 0;
      }
      if (hi < lo) { lo = 0; hi = 0; }
      named_bar_sync<1, kSsConsumers>();
      const long long n_region = (long long)a.region_len[d.region] + a.region_pad[d.region];
      const WalkOut w = hist_walk<kSsConsumers, true>(s_hist, n_region, a.breadth_n, lo, hi, s_u64, s_i32, s_med);
      if (t == 0) write_stats(a.out + d.region, w);
    } else {
      uint32_t* gh = a.split_hist + (int64_t)d.split * kHistBins;
      RegionScratch* rs = a.split_scratch + d.split;
      for (int b = lo + t; b <= hi; b += kSsConsumers) {
        const uint32_t c = s_hist[b];
        if (c) atomicAdd(gh + b, c);
      }
      named_bar_sync<1, kSsConsumers>();                                 // the CTA's merges are issued before its arrival
      if (t == 0) {
        if (d.pad > 0) { atomicAdd(gh, (uint32_t)d.pad); lo = 0; if (hi < 0) hi = 0; }
        if (hi >= lo) {
          atomicMax(&rs->max_bin, (uint32_t)hi);
          atomicMax(&rs->min_bin_inv, (uint32_t)(kHistBins - 1 - lo));
        }
        __threadfence();
        const unsigned prev = atomicAdd(&rs->done, 1u);
        s_last = prev == (unsigned)(a.split_pieces[d.split] - 1) ? 1 : 0;
      }
      if (hi < lo) { lo = 0; hi = -1; }
      named_bar_sync<1, kSsConsumers>();
      if (s_last) {
        // the last piece of the region has arrived here: pull the merged bin range (it contains this piece's), leave the
        // global copy zeroed for the next run, walk
        __threadfence();
        int mlo = kHistBins - 1 - (int)*((volatile uint32_t*)&rs->min_bin_inv), mhi = (int)*((volatile uint32_t*)&rs->max_bin);
        if (mhi < mlo) { mlo = 0; mhi = 0; }
        for (int b = mlo + t; b <= mhi; b += kSsConsumers) { s_hist[b] = __ldcg(gh + b); gh[b] = 0u; }
        named_bar_sync<1, kSsConsumers>();
        if (t == 0) { rs->done = 0u; rs->max_bin = 0u; rs->min_bin_inv = 0u; }
        const long long n_region = (long long)a.region_len[d.region] + a.region_pad[d.region];
        const WalkOut w = hist_walk<kSsConsumers, true>(s_hist, n_region, a.breadth_n, mlo, mhi, s_u64, s_i32, s_med);
        if (t == 0) write_stats(a.out + d.region, w);
        lo = mlo; hi = mhi;                                              // (the range to clear below)
      }
    }
    named_bar_sync<1, kSsConsumers>();                                  // walk / merge have read the bins
    for (int b = lo + t; b <= hi; b += kSsConsumers) s_hist[b] = 0u;     // only the touched range needs clearing
    lo = kHistBins; hi = -1;
    named_bar_sync<1, kSsConsumers>();
  }
}

}  // namespace mcov
