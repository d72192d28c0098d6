// k_stats_stream.cuh -- region statistics as ONE balanced stream over the depth (large regions).
//
// One CTA per region (or per chunk of a region) leaves the machine badly balanced: on config C2,
// 1 000 equal CTAs on 592 resident slots = 1.69 waves, each CTA starting with a cold pipeline and
// ending with a clear / walk during which it loads nothing (DESIGN.md 3.3).  Here the large regions
// are cut into slices of equal COST, one per persistent CTA (2 per SM); the plan (mcov_api.cu) puts a
// slice border on a region border wherever that costs less imbalance than a split region costs chain:
//   * a producer warp streams the CTA's slice through a ring of 8 KB shared-memory stages with
//     TMA bulk copies behind mbarriers -- it runs ahead across region boundaries, so the stream
//     never stops while the consumers finish a region; a tile shared by two pieces that follow
//     each other in slot order is staged once, the slots of each counted into its own piece;
//   * 8 consumer warps feed the exact counting histogram (8192 one-value bins, ATOMS.POPC.INC)
//     from shared memory; there are two, so that the consumers count piece p into one while a
//     walker warp walks piece p - 1 in the other;
//   * a region that lies wholly inside a slice is walked and written by its CTA; a region cut by
//     a slice border adds its touched bins to a per-split-region histogram in global memory
//     (fire-and-forget reductions, nobody waits), and the CTA whose piece of it arrives last pulls
//     the merged bin range back and walks the region.
// The walk is hist_walk (k_stats.cuh), the same as for the small regions; it also clears the bins it walks, so a
// whole piece ends for the consumers with one barrier and a hand-off to the walker.
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
#define MCOV_SS_STAGES 5
#endif
#ifndef MCOV_SS_BLK
#define MCOV_SS_BLK 2048
#endif
#ifndef MCOV_SS_CTAS
#define MCOV_SS_CTAS 2
#endif
constexpr int kSsStages = MCOV_SS_STAGES;
constexpr int kSsBlk = MCOV_SS_BLK;                  // slots per stage (8 KB)
constexpr int kSsConsumers = 256;
constexpr int kSsThreads = kSsConsumers + 64;        // + the producer warp + the walker warp
constexpr int kSsSmemBytes = kSsStages * kSsBlk * 4 + 2 * kHistBins * 4;   // 104 KB: 2 CTAs per SM

struct SsPiece {          // a region, or the part of a region inside one slice
  int64_t slot;           // first slot
  int32_t n;              // slots
  int32_t region;
  int32_t pad;            // zeros to add to bin 0 (positions beyond the contig end; first piece of the region only)
  int32_t split;          // -1: the whole region is this piece; else index of the region's global histogram
  int32_t n_region;       // values the region's histogram describes (slots inside the contig + pad)
  int32_t reserved;
};

// cnt < 0: end of the slice.  tile < 0: the stage holds depth, valid elements [skip, skip + cnt) of the piece, then
// (after the piece's end when `last`) [skip + cnt, skip + cnt + next) of the piece that follows it in slot order;
// else the histograms of the cnt tiles from `tile` on
struct SsDesc { int32_t region, split, pad, skip, cnt, last, tile, n_region, next; };
struct SsJob { int32_t region, n_region, lo, hi; };  // a histogram handed to the walker; region < 0: end of the slice
constexpr int kSsHistTiles = kSsBlk * 4 / (kTileHistWords * 2);     // tile histograms per stage
// Slice costs of the plan (mcov_api.cu), in staged bytes.  Measured with tools/probe_stats_chain.py on C2 (B200):
// the consumers of a CTA take about 1 us per 16 KB staged, 1.65 us to end a whole piece and walk it, and about 5 us
// more for a region split between two CTAs (two merges into global memory, arrival, pull-back, one more piece end).
constexpr int64_t kSsPieceCost = 26 << 10;
constexpr int64_t kSsSplitCost = 80 << 10;

#ifdef MCOV_SS_PROBE
// Phase timer of the consumers' serial chain (tools/probe_stats_chain.py builds a library with it; the product build
// has none of this): clock64 cycles per CTA and phase, kept in registers of consumer thread 0 and stored at the end.
enum { kPrWait, kPrAccum, kPrEndWhole, kPrEndSplit, kPrWalk, kPrTotal, kPrPieces, kPrSplits, kPrNs, kPrPhases };
constexpr int kPrMaxCtas = 4096;
__device__ unsigned long long g_ss_probe[kPrMaxCtas][kPrPhases];
struct SsProbe {
  long long t, t0, acc[kPrPhases];
  unsigned long long ns0;
  __device__ __forceinline__ void start() {
    for (int k = 0; k < kPrPhases; ++k) acc[k] = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns0));
    t = t0 = clock64();
  }
  __device__ __forceinline__ void lap(int phase) { const long long n = clock64(); acc[phase] += n - t; t = n; }
  __device__ __forceinline__ void store() {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    acc[kPrTotal] = clock64() - t0; acc[kPrNs] = (long long)(ns - ns0);
    if (threadIdx.x == 0 && blockIdx.x < kPrMaxCtas)
      for (int k = 0; k < kPrPhases; ++k) g_ss_probe[blockIdx.x][k] = (unsigned long long)acc[k];
  }
};
#define SS_PROBE(...) __VA_ARGS__
#else
#define SS_PROBE(...)
#endif

struct SsArgs {
  const int32_t* depth;
  const SsPiece* pieces;
  const int32_t* cta_piece_start;   // [grid + 1]
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
  uint32_t* s_hist2 = reinterpret_cast<uint32_t*>(ss_smem + (size_t)kSsStages * kSsBlk * 4);   // [2][kHistBins]
  __shared__ __align__(8) uint64_t s_full[kSsStages], s_empty[kSsStages];
  __shared__ __align__(8) uint64_t s_hfull[2], s_hfree[2];   // histogram b handed to the walker / walked and cleared
  __shared__ SsDesc s_desc[kSsStages];
  __shared__ SsJob s_job[2];
  __shared__ int s_rng[2][2 * (kSsConsumers / 32)];  // bin range of a piece per consumer warp, by the parity of the piece
  __shared__ int s_last;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  constexpr int kW = kSsConsumers / 32;
  {
    uint4* h4 = reinterpret_cast<uint4*>(s_hist2);
    for (int k = t; k < 2 * kHistBins / 4; k += kSsThreads) h4[k] = make_uint4(0, 0, 0, 0);
    if (t == 0) {
      for (int s = 0; s < kSsStages; ++s) { mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], kW); }
      for (int b = 0; b < 2; ++b) { mbar_init(&s_hfull[b], 1); mbar_init(&s_hfree[b], 1); }
      mbar_fence_init();
    }
  }
  __syncthreads();
  pdl_wait();                                           // the depth is complete
  pdl_launch_dependents();
  const int p0 = a.cta_piece_start[blockIdx.x], p1 = a.cta_piece_start[blockIdx.x + 1];

  if (warp == kW) {
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
    // tiles [t0, t1) lie wholly inside the piece and are staged as histograms; t1 <= t0: none
    auto hist_tiles = [&](const SsPiece& pc, int64_t& t0, int64_t& t1) {
      t0 = a.tile_hist ? (pc.slot + kTile - 1) >> kTileShift : 0;
      t1 = a.tile_hist ? (pc.slot + pc.n) >> kTileShift : 0;
    };
    // the depth of the slots [s0, s1) of a piece; `last`: the piece ends there (a piece without slots still finishes
    // its region).  The last block also takes the slots [s1, nlim) of the next piece, as far as they fit; returns
    // where that piece's staging resumes (-1 when it takes none)
    auto depth_stages = [&](const SsPiece& pc, int64_t s0, int64_t s1, bool last, int64_t nlim) {
      const int64_t a0 = s0 & ~(int64_t)3;
      const int64_t nblk = s1 > s0 ? (s1 - a0 + kSsBlk - 1) / kSsBlk : (last ? 1 : 0);
      int64_t resume = -1;
      for (int64_t k = 0; k < nblk; ++k) {
        const int64_t b0 = a0 + k * kSsBlk;
        const int64_t lo = max(b0, s0), hi = min(b0 + kSsBlk, s1);
        SsDesc d;
        d.region = pc.region; d.split = pc.split; d.pad = pc.pad; d.n_region = pc.n_region; d.tile = -1;
        d.skip = (int32_t)(lo - b0); d.cnt = (int32_t)max((int64_t)0, hi - lo); d.last = (last && k == nblk - 1) ? 1 : 0;
        d.next = d.last ? (int32_t)max((int64_t)0, min(b0 + kSsBlk, nlim) - s1) : 0;
        if (d.next) resume = s1 + d.next;
        const int32_t stop = d.skip + d.cnt + d.next;
        const uint32_t bytes = stop > d.skip ? (uint32_t)((stop + 3) & ~3) * 4u : 0u;   // whole 16-byte vectors inside the padded depth array
        publish(d, a.depth + b0, bytes);
      }
      return resume;
    };
    int64_t from = -1;                       // first slot of piece p not staged with piece p - 1 (-1: none was)
    for (int p = p0; p < p1; ++p) {
      const SsPiece pc = a.pieces[p];
      const int64_t end = pc.slot + pc.n;
      const int64_t s0 = from >= 0 ? from : pc.slot;
      // the next piece begins where this one ends: its leading depth slots (up to its first histogram tile, and short
      // of its last slot, which ends it) ride in this piece's last block
      int64_t nlim = end;
      if (p + 1 < p1) {
        const SsPiece nx = a.pieces[p + 1];
        if (nx.slot == end) {
          int64_t n0, n1;
          hist_tiles(nx, n0, n1);
          nlim = min(n1 > n0 ? n0 << kTileShift : nx.slot + nx.n, nx.slot + nx.n - 1);
        }
      }
      int64_t t0, t1;
      hist_tiles(pc, t0, t1);
      if (t1 <= t0) { from = depth_stages(pc, s0, end, true, nlim); continue; }
      depth_stages(pc, s0, t0 << kTileShift, false, 0);
      for (int64_t t = t0; t < t1; t += kSsHistTiles) {
        SsDesc d;
        d.region = pc.region; d.split = pc.split; d.pad = pc.pad; d.n_region = pc.n_region; d.next = 0;
        d.skip = 0; d.cnt = (int32_t)min((int64_t)kSsHistTiles, t1 - t); d.last = 0; d.tile = (int32_t)t;
        publish(d, reinterpret_cast<const int32_t*>(a.tile_hist + t * kTileHistWords), (uint32_t)d.cnt * kTileHistWords * 2u);
      }
      from = depth_stages(pc, t1 << kTileShift, end, true, nlim);
    }
    SsDesc e;
    e.region = -1; e.split = -1; e.pad = 0; e.skip = 0; e.cnt = -1; e.last = 0; e.tile = -1; e.n_region = 0; e.next = 0;
    publish(e, nullptr, 0u);
    return;
  }

  if (warp == kW + 1) {
    // ---------------- walker: one warp walks each finished histogram while the consumers count the next piece ----
    __shared__ unsigned long long w_u64[6];
    __shared__ int w_i32[4];
    __shared__ int w_med[2];
    for (unsigned n = 0;; ++n) {
      const unsigned b = n & 1;
      mbar_wait(&s_hfull[b], (n >> 1) & 1);
      const SsJob j = s_job[b];
      if (j.region < 0) break;
      const WalkOut w = hist_walk<32, true, true, 2>(s_hist2 + b * kHistBins, j.n_region, a.breadth_n, j.lo, j.hi, w_u64, w_i32, w_med);
      if (lane == 0) write_stats(a.out + j.region, w);
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_hfree[b]);                           // (the walk has cleared [lo, hi])
    }
    return;
  }

  // ---------------- consumers ----------------
  int lo = kHistBins, hi = -1;
  unsigned buf = 0, handoffs = 0, piece = 0;   // the histogram being counted (handoffs & 1), hand-offs, pieces ended
  uint32_t* s_hist = s_hist2;
  // elements [e0, e1) of a depth stage: whole vectors by all threads, a partial head vector by thread 0, a partial
  // tail vector by thread 32
  auto count_depth = [&](const int4* v, int e0, int e1) {
    if (e1 <= e0) return;
    const int hv = e0 >> 2, tv = e1 >> 2;
    for (int j = ((e0 + 3) >> 2) + t; j < tv; j += kSsConsumers) hist_vec(s_hist, v[j], lo, hi);
    if (t == 0 && (e0 & 3)) hist_partial(s_hist, v[hv], e0 & 3, hv == tv ? (e1 & 3) : 4, lo, hi);
    if (t == 32 && (e1 & 3) && (hv != tv || !(e0 & 3))) hist_partial(s_hist, v[tv], 0, e1 & 3, lo, hi);
  };
  SS_PROBE(SsProbe pr; pr.start();)
#pragma unroll 1
  for (unsigned it = 0;; ++it) {
    const unsigned s = it % kSsStages, k = it / kSsStages;
    mbar_wait(&s_full[s], k & 1);
    SS_PROBE(pr.lap(kPrWait);)
    const SsDesc d = s_desc[s];
    if (d.cnt < 0) {
      if (t == 0) { s_job[buf].region = -1; mbar_arrive(&s_hfull[buf]); }   // (buffer buf is free: waited for below)
      break;
    }
    const int4* v = reinterpret_cast<const int4*>(s_ring + (size_t)s * kSsBlk);
    if (d.tile >= 0) {
      // 64 threads per tile histogram, a u32 (two u16 words) each: word 2w holds bin 2w - 1, word 2w + 1 bin 2w
      const uint32_t* h = reinterpret_cast<const uint32_t*>(v);
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
          const int4* dv = reinterpret_cast<const int4*>(a.depth + ((int64_t)(d.tile + r) << kTileShift)) + w;
          int4 x[kTile / 4 / kPer];
#pragma unroll
          for (int u = 0; u < kTile / 4 / kPer; ++u) x[u] = __ldcs(dv + u * kPer);
#pragma unroll
          for (int u = 0; u < kTile / 4 / kPer; ++u) hist_vec(s_hist, x[u], lo, hi);
        }
      }
    } else {
      count_depth(v, d.skip, d.skip + d.cnt);
    }
    if (!d.next) {
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_empty[s]);                           // the stage may be refilled
    }
    SS_PROBE(pr.lap(kPrAccum);)
    if (d.last) {
      SS_PROBE(pr.acc[kPrPieces] += 1; pr.acc[kPrSplits] += d.split >= 0;)
      // ---- end of a piece: bin range over the CTA, then walk (whole region) or merge (split region) ----
      if (t == 0 && d.pad > 0) {                                         // zeros beyond the contig end join the multiset
        atomicAdd(&s_hist[0], (uint32_t)d.pad);
        lo = 0; hi = max(hi, 0);
      }
      lo = warp_min(lo); hi = warp_max(hi);
      int* rng = s_rng[piece++ & 1];                                     // (a warp may reach the next piece's end first)
      if (lane == 0) { rng[warp] = lo; rng[kW + warp] = hi; }
      named_bar_sync<1, kSsConsumers>();                                // also: the histogram of the piece is complete
      lo = kHistBins; hi = -1;
#pragma unroll
      for (int w = 0; w < kW; ++w) { lo = min(lo, rng[w]); hi = max(hi, rng[kW + w]); }
      bool walk = true;
      if (d.split >= 0) {
        uint32_t* gh = a.split_hist + (int64_t)d.split * kHistBins;
        RegionScratch* rs = a.split_scratch + d.split;
        for (int b = lo + t; b <= hi; b += kSsConsumers) {              // each thread clears the bins it merged
          const uint32_t c = s_hist[b];
          if (c) { atomicAdd(gh + b, c); s_hist[b] = 0u; }
        }
        named_bar_sync<1, kSsConsumers>();                               // the CTA's merges are issued before its arrival
        if (t == 0) {
          if (hi >= lo) {
            atomicMax(&rs->max_bin, (uint32_t)hi);
            atomicMax(&rs->min_bin_inv, (uint32_t)(kHistBins - 1 - lo));
          }
          __threadfence();
          const unsigned prev = atomicAdd(&rs->done, 1u);
          s_last = prev == (unsigned)(a.split_pieces[d.split] - 1) ? 1 : 0;
        }
        named_bar_sync<1, kSsConsumers>();
        walk = s_last != 0;
        if (walk) {
          // the last piece of the region has arrived here: pull the merged bin range (it contains this piece's), leave
          // the global copy zeroed for the next run, walk
          __threadfence();
          lo = kHistBins - 1 - (int)*((volatile uint32_t*)&rs->min_bin_inv); hi = (int)*((volatile uint32_t*)&rs->max_bin);
          if (hi < lo) { lo = 0; hi = 0; }
          for (int b = lo + t; b <= hi; b += kSsConsumers) { s_hist[b] = __ldcg(gh + b); gh[b] = 0u; }
          named_bar_sync<1, kSsConsumers>();
          if (t == 0) { rs->done = 0u; rs->max_bin = 0u; rs->min_bin_inv = 0u; }
        }
      }
      if (walk) {
        // hand the histogram to the walker (the barrier above made it complete), count on in the other one once the
        // walker has finished with it
        if (hi < lo) { lo = 0; hi = 0; }
        if (t == 0) { s_job[buf] = SsJob{d.region, d.n_region, lo, hi}; mbar_arrive(&s_hfull[buf]); }
        buf = ++handoffs & 1;
        s_hist = s_hist2 + buf * kHistBins;
        SS_PROBE(if (d.split < 0) pr.lap(kPrEndWhole); else pr.lap(kPrEndSplit);)
        const unsigned uses = handoffs >> 1;                            // earlier hand-offs of this buffer
        if (uses) mbar_wait(&s_hfree[buf], (uses - 1) & 1);
        SS_PROBE(pr.lap(kPrWalk);)
      }
      lo = kHistBins; hi = -1;
      SS_PROBE(if (d.split < 0) pr.lap(kPrEndWhole); else pr.lap(kPrEndSplit);)
    }
    if (d.next) {                                                        // the next piece's head shares this stage
      count_depth(v, d.skip + d.cnt, d.skip + d.cnt + d.next);
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_empty[s]);
      SS_PROBE(pr.lap(kPrAccum);)
    }
  }
  SS_PROBE(pr.store();)
}

}  // namespace mcov
