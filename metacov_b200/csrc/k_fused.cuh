// k_fused.cuh -- fused depth path for coordinate-sorted reads.
//
// Same result as K0 (clear) + K1 (expand, k_expand.cuh) + K2 (scan, k_scan.cuh)
// -- the per-base `column.n` of reference metacov/pileup.py:13-16 -- but the
// slot space is written exactly once and never read, no atomic ever reaches
// L2 per read, and no CTA waits on another:
//
//   k_fused_prep   one pass over the reads, 4 consecutive reads per thread with
//                  128-bit loads: filter + CIGAR reduce, emits the 4-byte record
//                  rec[i] = {offset of the start slot in its tile, clipped span}
//                  (span 0 = read contributes nothing).  Because the reads are
//                  sorted it also produces
//                    tile_first[T]  first read whose start slot >= T*kTile
//                  and, for reads whose span exceeds kNearSpan ("far" reads:
//                  long reads, spliced reads), the end slot list, per-tile
//                  far-end counts and tile_agg[T] = (#far starts - #far ends) in T.
//   k_scan_inplace one small scan over [tile_agg | far counts]: the inclusive
//                  sum of tile_agg up to T-1 is the number of FAR reads open at
//                  the start of tile T.
//   k_far_scatter  bucket the far ends by tile (counting sort); list the tiles that hold
//                  very many reads (scheduled first by the tile kernel).
//   k_fused_tile_tma (k_tile_tma.cuh)  persistent CTAs drawing tiles of kTile slots by
//                  ticket (heavy tiles first); a producer warp stages each tile's records
//                  with TMA bulk copies, and the consumer warps send +1/-1 of the tile's reads
//                  to SHARED-memory counters (starts and ends kept apart),
//                  the ends of near reads that started before the tile are
//                  found by walking back at most max_span slots in the sorted
//                  order -- and because kNearSpan = kTile every near read that
//                  is open at the tile border ends inside the tile, so THE
//                  NUMBER OF WALK-BACK HITS IS THE NEAR DEPTH ENTERING THE TILE:
//                  no look-back, no ordering between CTAs, and no per-tile
//                  aggregate for near reads at all.  Far ends come from the
//                  tile's bucket; block scan from the carry; 128-bit streaming
//                  stores.  Keeping starts and ends apart gives htslib's
//                  max_depth no-op condition exactly: cap[p] = depth[p-1] +
//                  starts[p] = depth[p] + ends[p] (SURVEY.md Appendix A-6).
//
// HBM bytes (algorithmic): prep 15R + 4*sum(n_cigar of passing reads) + 4R;
// tile 4R + 4(L+C).  The kernels of one pass are chained with programmatic
// dependent launches (pdl_wait / pdl_launch_dependents, common.cuh).
#pragma once
#include <type_traits>
#include "ctx.cuh"
#include "k_expand.cuh"
#include "k_scan.cuh"

namespace mcov {

#ifndef MCOV_TILE_SHIFT
#define MCOV_TILE_SHIFT 11
#endif
constexpr int kTileShift = MCOV_TILE_SHIFT;
constexpr int kTile = 1 << kTileShift;    // slots per CTA of the tile kernel (2048: 128-thread CTAs, 8 per SM)
constexpr uint32_t kNearSpan = kTile;     // spans above this take the bucket path
constexpr int kFusedThreads = kTile / 16; // 16 slots per thread
constexpr int kTileVec = 4;               // = four int4 per thread (independent of the push path's scan shape)
static_assert(kFusedThreads * kTileVec * 4 == kTile, "tile kernel: threads x vectors x 4 slots must cover the tile");
static_assert(kTileShift >= 9 && kTileShift <= 12, "record format: 12-bit offset, 13-bit span code");
// Depth histogram of one tile, written by the tile kernel so that the statistics of large regions need not read the
// depth of the tiles that lie wholly inside them (k_stats_stream.cuh): kTileHistWords u16, [0] = anchor A, [1 + b] =
// slots of the tile with depth A + b (b < kTileHistBins).  A = kTileHistNone: some depth of the tile lies outside the
// window (or the tile's depth was rewritten afterwards), the tile is counted from the depth.
constexpr int kTileHistWords = 128;
constexpr int kTileHistBins = kTileHistWords - 1;
constexpr uint16_t kTileHistNone = 0xFFFF;
constexpr int kPrepThreads = 256;
constexpr int kPrepPer = 4;               // reads per thread
constexpr uint32_t kFarCapDefault = 1u << 26;

struct FusedArgs {
  ExpandArgs e;
  uint32_t* rec;              // [n] 4-byte records, see make_rec
  int64_t n_slots;
  int64_t n_tiles;
  int64_t tile_lo, tile_hi;   // tiles this pass writes (the whole slot space, or the batch's share when a file is streamed)
  int streaming;              // the pass is one batch of a streamed file (mcov_stream_push)
  int64_t* far_end;           // [far_cap] end slots of far reads
  uint32_t far_cap;
  int32_t* tile_agg;          // [cnt_pad] (#far starts - #far ends) per tile -> inclusive scan in place
  uint32_t* tile_cnt;         // [cnt_pad] far ends per tile -> inclusive scan in place (follows tile_agg)
  uint32_t* tile_cursor;      // [n_tiles] scatter cursors
  uint32_t* far_sorted;       // [far_cap] in-tile offsets bucketed by tile
  uint32_t* tile_first;       // [n_tiles+1] (a fused batch holds < 2^32 reads)
  int32_t* depth;
  union {                     // (one slot: the fused path and the push path never need both, and the layout stays)
    int32_t* tile_cap;        // fused: [n_tiles] max of depth[p-1]+starts[p] in the tile, written only when > max_depth
    int32_t* starts;          // push (k_expand<., true>): [n_slots] passing reads that start at each slot
  };
  uint16_t* tile_hist;        // [n_tiles][kTileHistWords] depth histograms of the tiles (k_tile_tma.cuh), nullptr: not written
  uint32_t* tile_heavy;       // [n_tiles] ids of the tiles with >= heavy_min reads (k_far_scatter; pc->n_heavy of them)
  uint32_t heavy_min;
  int32_t max_depth;          // htslib maxcnt (<= 0: cap disabled)
  int vec_ok;                 // SoA base pointers aligned for 128-bit loads
  const uint32_t* flag_lut;   // device, [128]: bit F of the table: a read with flag F (< 4096: the 12 bits BAM defines) passes the
                              // flag filter (kept out of the argument block: kernel parameters are copied at every launch)
};

// slot key of a read: contig offset + clamped position; reads without a valid
// contig sort after every slot
__device__ __forceinline__ int64_t slot_key(const ExpandArgs& a, int32_t t, int32_t p, int64_t n_slots, int64_t& len,
                                            int64_t& base) {
  if (t < 0 || t >= a.n_contigs) { len = 0; base = n_slots; return n_slots; }
  len = a.contig_len[t];
  base = a.contig_off[t];
  int64_t q = p < 0 ? 0 : (p > len ? len : (int64_t)p);
  return base + q;
}

__device__ __noinline__ unsigned long long warp_cigar_reflen_call(const uint32_t* p, uint32_t cnt, int lane) {
  return warp_cigar_reflen(p, cnt, lane);
}

// Rare path of k_fused_prep: some read of this warp is the first of a new tile.  Entered by the
// whole warp.  tl[r] = tile of read r (already clamped), prev = tile of the read before this thread's.
__device__ __noinline__ void prep_tile_boundaries(uint32_t* tile_first, int64_t i0, int nv, int64_t prev, int64_t t0,
                                                  int64_t t1, int64_t t2, int64_t t3, bool is_last, int64_t n,
                                                  int64_t last_tile, int lane) {
#pragma unroll 1
  for (int r = 0; r <= 4; ++r) {
    int64_t tcur = r == 0 ? t0 : r == 1 ? t1 : r == 2 ? t2 : t3;
    int64_t lo, hi, v;
    if (r < 4) {
      bool need = r < nv && tcur > prev;
      lo = need ? prev + 1 : 1; hi = need ? tcur : 0; v = i0 + r;
      if (r < nv && tcur > prev) prev = tcur;
    } else {                                   // the last read closes the table
      lo = is_last ? prev + 1 : 1; hi = is_last ? last_tile : 0; v = n;
    }
    bool big = (hi - lo) >= 8;
    if (!big) for (int64_t T = lo; T <= hi; ++T) tile_first[T] = (uint32_t)v;
    unsigned todo = __ballot_sync(0xffffffffu, big);
    while (todo) {                             // long gaps are written by the whole warp
      int src = __ffs(todo) - 1;
      todo &= todo - 1;
      int64_t l2 = __shfl_sync(0xffffffffu, lo, src), h2 = __shfl_sync(0xffffffffu, hi, src);
      int64_t v2 = __shfl_sync(0xffffffffu, v, src);
      for (int64_t T = l2 + lane; T <= h2; T += 32) tile_first[T] = (uint32_t)v2;
    }
  }
}

// Rare path: some read of this warp spans more than kNearSpan slots.  Entered by the whole warp.
__device__ __noinline__ void prep_far(const FusedArgs& f, uint32_t st0, uint32_t st1, uint32_t st2, uint32_t st3, int64_t e0,
                                      int64_t e1, int64_t e2, int64_t e3, unsigned farmask, int lane) {
  int nfar = __popc(farmask);
  int incl = nfar;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  int total = __shfl_sync(0xffffffffu, incl, 31);
  uint32_t base = 0;
  if (lane == 0) base = atomicAdd(&f.e.pc->n_far, (uint32_t)total);
  base = __shfl_sync(0xffffffffu, base, 0);
  uint32_t idx = base + (uint32_t)(incl - nfar);
#pragma unroll 1
  for (int r = 0; r < 4; ++r) {
    if (farmask & (1u << r)) {
      int64_t e = r == 0 ? e0 : r == 1 ? e1 : r == 2 ? e2 : e3;
      uint32_t st = r == 0 ? st0 : r == 1 ? st1 : r == 2 ? st2 : st3;
      if (idx < f.far_cap) {                      // (past the cap the pass is rejected: MCOV_ERR_RANGE)
        f.far_end[idx] = e;
        atomicAdd(f.tile_cnt + (e >> kTileShift), 1u);
        atomicAdd(f.tile_agg + st, 1);            // a far read is open from its start tile ...
        atomicAdd(f.tile_agg + (e >> kTileShift), -1);   // ... to its end tile
      }
      ++idx;
    }
  }
}

// Record written by k_fused_prep for the tile kernel, 4 bytes per read:
//   bits  0..11  offset of the start slot inside its tile (the tile itself follows from tile_first)
//   bits 12..24  span code: 0 = contributes nothing (filtered / empty), 1..kNearSpan = clipped span,
//                kRecFar = span above kNearSpan (its end comes from the far-end buckets)
constexpr uint32_t kRecFar = 0x1FFFu;
__device__ __forceinline__ uint32_t make_rec(uint32_t local, uint32_t span) {
  return local | ((span > kNearSpan ? kRecFar : span) << kTileShift);
}

struct PrepAcc { uint32_t n_pass, al32, max_span, unsorted; };

// General path of k_fused_prep for one warp iteration: contig changes inside the warp, negative
// positions, reads without a valid contig, the ragged tail, the first reads of the batch.  Entered
// by the whole warp.  All per-read arithmetic is 32-bit and contig relative: with base = contig
// offset, tb = base >> 12 and bo = base & 4095 the tile of position q is tb + ((bo + q) >> 12);
// 64-bit slot numbers are only formed for far reads.
__device__ __forceinline__ PrepAcc prep_general(const FusedArgs& f, int64_t i0, int nv, int32_t T0, int32_t T1, int32_t T2,
                                             int32_t T3, int32_t P0, int32_t P1, int32_t P2, int32_t P3, uint32_t R0,
                                             uint32_t R1, uint32_t R2, uint32_t R3, unsigned passm, int lane) {
  const ExpandArgs& a = f.e;
  const int64_t* __restrict__ g_coff = a.contig_off;
  const int32_t* __restrict__ g_clen = a.contig_len;
  const uint32_t n_contigs = (uint32_t)a.n_contigs;
  const int64_t n = a.n;
  const uint32_t last_tile = (uint32_t)f.n_tiles;             // tile_first has n_tiles+1 entries
  const uint32_t nslot_tb = (uint32_t)(f.n_slots >> kTileShift), nslot_bo = (uint32_t)(f.n_slots & (kTile - 1));
  const int32_t T[4] = {T0, T1, T2, T3}, P[4] = {P0, P1, P2, P3};
  const uint32_t reflen[4] = {R0, R1, R2, R3};
  PrepAcc acc = {0u, 0u, 0u, 0u};
  uint32_t span[4], tls[4], qq[4], loc[4];
  int32_t c_tid = INT_MIN;
  uint32_t c_len = 0, c_tb = nslot_tb, c_bo = nslot_bo;
  unsigned farmask = 0;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    if (T[r] != c_tid) {                        // contig change
      c_tid = T[r];
      if ((uint32_t)T[r] < n_contigs) {
        int64_t base = g_coff[T[r]];
        c_len = (uint32_t)g_clen[T[r]];
        c_tb = (uint32_t)(base >> kTileShift); c_bo = (uint32_t)base & (kTile - 1);
      } else { c_len = 0; c_tb = nslot_tb; c_bo = nslot_bo; }
    }
    uint32_t q = P[r] < 0 ? 0u : min((uint32_t)P[r], c_len);
    qq[r] = q;
    loc[r] = (c_bo + q) & (kTile - 1);
    tls[r] = min(c_tb + ((c_bo + q) >> kTileShift), last_tile);
    span[r] = 0;
    if ((passm >> r) & 1u) {
      // end = clamp(pos + reflen, 0, len), in 64 bits only for the (never negative in practice) sum
      int64_t e64 = (int64_t)P[r] + (int64_t)reflen[r];
      uint32_t e = e64 < 0 ? 0u : (e64 > (int64_t)c_len ? c_len : (uint32_t)e64);
      if (e > q) {
        span[r] = e - q;
        acc.n_pass += 1; acc.al32 += reflen[r];
        if (span[r] > kNearSpan) farmask |= 1u << r; else acc.max_span = max(acc.max_span, span[r]);
      }
    }
  }
  if (nv == kPrepPer) {
    *reinterpret_cast<uint4*>(f.rec + i0) =
        make_uint4(make_rec(loc[0], span[0]), make_rec(loc[1], span[1]), make_rec(loc[2], span[2]), make_rec(loc[3], span[3]));
  } else {
    for (int r = 0; r < nv; ++r) f.rec[i0 + r] = make_rec(loc[r], span[r]);
  }

  // ---- sortedness + tile boundaries (tile_first) -------------------------------------------------
  // "sorted" is judged on (contig, clamped position), i.e. on the slot keys the tile kernel relies on
  {
    uint32_t pt = __shfl_up_sync(0xffffffffu, (uint32_t)T[3], 1), pq = __shfl_up_sync(0xffffffffu, qq[3], 1);
    uint32_t ptile = __shfl_up_sync(0xffffffffu, tls[3], 1);
    bool has_prev = true;
    if (lane == 0) {
      has_prev = i0 > 0 && i0 - 1 < n;
      if (has_prev) {
        int32_t t0 = a.tid[i0 - 1], p0 = a.pos[i0 - 1];
        pt = (uint32_t)t0;
        if ((uint32_t)t0 < n_contigs) {
          int64_t base = g_coff[t0]; uint32_t len = (uint32_t)g_clen[t0];
          pq = p0 < 0 ? 0u : min((uint32_t)p0, len);
          ptile = min((uint32_t)(base >> kTileShift) + ((((uint32_t)base & (kTile - 1)) + pq) >> kTileShift), last_tile);
        } else { pq = 0; ptile = min(nslot_tb, last_tile); }
      }
    }
    // invalid contigs compare as the largest id (they sort last, like tid -1 in a BAM)
    uint32_t ut[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) ut[r] = (uint32_t)T[r] < n_contigs ? (uint32_t)T[r] : 0xffffffffu;
    if (pt >= n_contigs) pt = 0xffffffffu;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (r < nv) {
        uint32_t t0 = r ? ut[r - 1] : pt, q0 = r ? qq[r - 1] : pq;
        bool ok = (r == 0 && !has_prev) || ut[r] > t0 || (ut[r] == t0 && (ut[r] == 0xffffffffu || qq[r] >= q0));
        acc.unsorted |= ok ? 0u : 1u;
      }
    }
    const uint32_t tl_last = nv > 0 ? (nv == 4 ? tls[3] : nv == 3 ? tls[2] : nv == 2 ? tls[1] : tls[0]) : 0u;
    const bool bnd = nv > 0 && (!has_prev || tl_last > ptile);
    const bool is_last = nv > 0 && (i0 + nv == n);
    if (__any_sync(0xffffffffu, bnd || is_last))
      prep_tile_boundaries(f.tile_first, i0, nv, has_prev ? (int64_t)ptile : -1, tls[0], tls[1], tls[2], tls[3], is_last, n,
                           last_tile, lane);
  }

  // ---- far reads: end list, per-tile far-end counts, far-open aggregate ---------------------------
  if (__any_sync(0xffffffffu, farmask != 0)) {
    int64_t e64[4];                               // 64-bit end slots only here
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      int64_t base = ((farmask >> r) & 1u) ? g_coff[T[r]] : 0;
      e64[r] = base + qq[r] + span[r];
    }
    prep_far(f, tls[0], tls[1], tls[2], tls[3], e64[0], e64[1], e64[2], e64[3], farmask, lane);
  }
  return acc;
}

// Loads + filter + CIGAR reduction of the 4 reads of one thread (shared by both prep kernels).
struct PrepReads {
  int32_t T[4], P[4];
  uint32_t reflen[4];     // a read's reference length fits 32 bits (BAM positions are int32)
  unsigned passm;
  int nv;                 // valid reads of this thread
};

// OFF64: the CIGAR offsets are 64-bit (a batch of 2^32 or more ops: config C5 at full size).
template <bool OFF64>
__device__ __forceinline__ PrepReads prep_load_reduce(const FusedArgs& f, int64_t i0, int lane) {
  using off_t = typename std::conditional<OFF64, uint64_t, uint32_t>::type;
  const ExpandArgs& a = f.e;
  const int32_t* __restrict__ g_tid = a.tid;
  const int32_t* __restrict__ g_pos = a.pos;
  const uint16_t* __restrict__ g_flag = a.flag;
  const uint8_t* __restrict__ g_mapq = a.mapq;
  const off_t* __restrict__ g_off = OFF64 ? reinterpret_cast<const off_t*>(a.cig_off64) : reinterpret_cast<const off_t*>(a.cig_off);
  const uint32_t* __restrict__ g_cig = a.cig;
  const uint32_t n_contigs = (uint32_t)a.n_contigs;
  // pysam __advance_samtools + bam_plp_push's UNMAP drop (SURVEY.md Appendix A-2), branch-free:
  // pass <=> no dropped bit, a required bit (if any are required), mapq, not (paired and not proper)
  const uint32_t drop = (uint32_t)a.filt.flag_filter | 0x4u, req = a.filt.flag_require, minq = a.filt.min_mapq;
  const uint32_t req_none = req == 0 ? 1u : 0u, orph_mask = a.filt.ignore_orphans ? 3u : 0u;
  const int64_t n = a.n;
  PrepReads R;
  uint32_t F[4], Q[4];
  off_t O[5];
  R.nv = (int)min((int64_t)kPrepPer, max((int64_t)0, n - i0));
  if (R.nv == kPrepPer && f.vec_ok) {
    int4 t4 = *reinterpret_cast<const int4*>(g_tid + i0);
    int4 p4 = *reinterpret_cast<const int4*>(g_pos + i0);
    ushort4 f4 = *reinterpret_cast<const ushort4*>(g_flag + i0);
    uchar4 q4 = *reinterpret_cast<const uchar4*>(g_mapq + i0);
    if (OFF64) {
      const ulonglong2 oa = *reinterpret_cast<const ulonglong2*>(g_off + i0), ob = *reinterpret_cast<const ulonglong2*>(g_off + i0 + 2);
      O[0] = (off_t)oa.x; O[1] = (off_t)oa.y; O[2] = (off_t)ob.x; O[3] = (off_t)ob.y;
    } else {
      const uint4 o4 = *reinterpret_cast<const uint4*>(g_off + i0);
      O[0] = o4.x; O[1] = o4.y; O[2] = o4.z; O[3] = o4.w;
    }
    O[4] = g_off[i0 + 4];
    R.T[0] = t4.x; R.T[1] = t4.y; R.T[2] = t4.z; R.T[3] = t4.w;
    R.P[0] = p4.x; R.P[1] = p4.y; R.P[2] = p4.z; R.P[3] = p4.w;
    F[0] = f4.x; F[1] = f4.y; F[2] = f4.z; F[3] = f4.w;
    Q[0] = q4.x; Q[1] = q4.y; Q[2] = q4.z; Q[3] = q4.w;
  } else {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      bool v = r < R.nv;
      R.T[r] = v ? g_tid[i0 + r] : -1;
      R.P[r] = v ? g_pos[i0 + r] : 0;
      F[r] = v ? (uint32_t)g_flag[i0 + r] : 0x4u;
      Q[r] = v ? (uint32_t)g_mapq[i0 + r] : 0u;
    }
    // padding reads get an empty CIGAR: their offsets all equal cig_off[n]
#pragma unroll
    for (int r = 0; r <= 4; ++r) O[r] = (i0 <= n) ? g_off[min(i0 + r, n)] : (off_t)0;
  }
  unsigned passm = 0, coop = 0;
  uint32_t op0[4], nc[4];
  uint32_t nc_max = 0;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const bool p = (r < R.nv) & ((F[r] & drop) == 0u) & (((F[r] & req) | req_none) != 0u) & (Q[r] >= minq) &
                   ((F[r] & orph_mask) != 1u) & ((uint32_t)R.T[r] < n_contigs);
    nc[r] = (uint32_t)(O[r + 1] - O[r]);
    bool c = p && nc[r] > kThreadOps;
    passm |= p ? (1u << r) : 0u;
    coop |= c ? (1u << r) : 0u;
    if (!p || c) nc[r] = 0;                                           // ops this thread reduces itself
    nc_max = max(nc_max, nc[r]);
    op0[r] = nc[r] > 0 ? __ldg(g_cig + O[r]) : 0u;                    // four independent loads
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) R.reflen[r] = cigar_ref_len(op0[r]);
#pragma unroll 1
  for (uint32_t k = 1; k < nc_max; ++k) {                             // ops 2..4 (about 10 % of short reads)
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      uint32_t op = k < nc[r] ? __ldg(g_cig + O[r] + k) : 0u;
      R.reflen[r] += cigar_ref_len(op);
    }
  }
  // long CIGARs: the whole warp reduces one read at a time with 128-bit loads
  while (__any_sync(0xffffffffu, coop != 0)) {
    unsigned lanes = __ballot_sync(0xffffffffu, coop != 0);
    int src = __ffs(lanes) - 1;
    int r = __ffs(__shfl_sync(0xffffffffu, coop, src)) - 1;
    off_t ob = r == 0 ? O[0] : r == 1 ? O[1] : r == 2 ? O[2] : O[3];
    off_t oe = r == 0 ? O[1] : r == 1 ? O[2] : r == 2 ? O[3] : O[4];
    uint32_t cnt = (uint32_t)(oe - ob);
    ob = __shfl_sync(0xffffffffu, ob, src);
    cnt = __shfl_sync(0xffffffffu, cnt, src);
    unsigned long long v = warp_cigar_reflen_call(g_cig + ob, cnt, lane);
    if (lane == src) {
      uint32_t v32 = v > 0x7fffffffull ? 0x7fffffffu : (uint32_t)v;
      if (r == 0) R.reflen[0] = v32; else if (r == 1) R.reflen[1] = v32; else if (r == 2) R.reflen[2] = v32; else R.reflen[3] = v32;
      coop &= ~(1u << r);
    }
  }
  if (a.filt.reflen0_as_one) {                     // older htslib: a read that consumes no reference still occupies `pos`
#pragma unroll
    for (int r = 0; r < 4; ++r) if (((passm >> r) & 1u) && R.reflen[r] == 0u) R.reflen[r] = 1u;
  }
  R.passm = passm;
  return R;
}

// block-level reduction of the pass counters of a prep kernel (CONSUMERS_ONLY: the CTA has further warps
// that do not take part -- the kPrepThreads consumer warps meet at a named barrier)
template <bool CONSUMERS_ONLY = false>
__device__ __forceinline__ void prep_flush_counters(PassCounters* pc, uint32_t n_pass, unsigned long long aligned,
                                                    uint32_t unsorted, uint32_t max_span) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long np64 = warp_sum((unsigned long long)n_pass);
  aligned = warp_sum(aligned);
  unsorted = __any_sync(0xffffffffu, unsorted != 0);
  max_span = (uint32_t)warp_max((int)max_span);
  __shared__ unsigned long long s_np[kPrepThreads / 32], s_al[kPrepThreads / 32];
  __shared__ int s_un[kPrepThreads / 32];
  __shared__ uint32_t s_ms[kPrepThreads / 32];
  if (lane == 0) { s_np[warp] = np64; s_al[warp] = aligned; s_un[warp] = (int)unsorted; s_ms[warp] = max_span; }
  if (CONSUMERS_ONLY) named_bar_sync<1, kPrepThreads>(); else __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long np = 0, al = 0; int un = 0; uint32_t ms = 0;
    for (int k = 0; k < kPrepThreads / 32; ++k) { np += s_np[k]; al += s_al[k]; un |= s_un[k]; ms = max(ms, s_ms[k]); }
    if (np) atomicAdd(&pc->n_pass, np);
    if (al) atomicAdd(&pc->aligned_bases, al);
    if (un) atomicOr(&pc->unsorted, 1);
    if (ms) atomicMax(&pc->max_span, ms);
  }
}

// K1 of the push path (any read order): filter + CIGAR reduce + difference-array deltas, see
// k_expand.cuh.  Shares prep_load_reduce with the fused path (only f.e and f.vec_ok are read).
// STARTS: also count the passing reads that start at each slot (starts[slot] += 1), for the exact cap metric of
// mcov_begin_ex(MCOV_BEGIN_EXACT_CAP) into f.starts -- the same reads the fused path's tile kernel counts as starts.
template <bool OFF64, bool STARTS>
__global__ void __launch_bounds__(kPrepThreads, 4)
k_expand(const __grid_constant__ FusedArgs f) {
  const ExpandArgs& a = f.e;
  const int lane = threadIdx.x & 31;
  const int64_t n = a.n;
  const int64_t n_groups = (n + kPrepPer - 1) / kPrepPer;
  const int64_t g_round = (n_groups + 31) & ~(int64_t)31;     // whole warps iterate together
  const int64_t g_stride = (int64_t)gridDim.x * kPrepThreads;
  const int64_t* __restrict__ g_coff = a.contig_off;
  const int32_t* __restrict__ g_clen = a.contig_len;
  int32_t* __restrict__ delta = a.delta;
  unsigned long long aligned = 0;
  uint32_t n_pass = 0, unsorted = 0;
  int32_t c_tid = -1;                                         // contig constants, reloaded on change
  int64_t c_len = 0, c_base = 0;
#pragma unroll 1
  for (int64_t g = (int64_t)blockIdx.x * kPrepThreads + threadIdx.x; g < g_round; g += g_stride) {
    const int64_t i0 = g * kPrepPer;
    int32_t pvT = 0, pvP = 0;
    const bool has_prev = lane == 0 && i0 > 0 && i0 - 1 < n;
    if (has_prev) { pvT = a.tid[i0 - 1]; pvP = a.pos[i0 - 1]; }
    const PrepReads R = prep_load_reduce<OFF64>(f, i0, lane);
    // sortedness by (tid as unsigned: unplaced reads sort last, pos) -- informational (mcov_pass_info.sorted)
    {
      uint32_t pt = __shfl_up_sync(0xffffffffu, (uint32_t)R.T[3], 1);
      int32_t pp = __shfl_up_sync(0xffffffffu, R.P[3], 1);
      bool prev_ok = lane > 0 && i0 > 0;
      if (lane == 0) { pt = (uint32_t)pvT; pp = pvP; prev_ok = has_prev; }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        if (r < R.nv) {
          const uint32_t u1 = (uint32_t)R.T[r];
          if (prev_ok && (u1 < pt || (u1 == pt && R.P[r] < pp))) unsorted = 1;
          pt = u1; pp = R.P[r]; prev_ok = true;
        }
      }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if ((R.passm >> r) & 1u) {                              // (passing reads have a valid contig)
        if (R.T[r] != c_tid) { c_tid = R.T[r]; c_len = g_clen[c_tid]; c_base = g_coff[c_tid]; }
        int64_t s = R.P[r], e = (int64_t)R.P[r] + (int64_t)R.reflen[r];
        s = s < 0 ? 0 : (s > c_len ? c_len : s);
        e = e < 0 ? 0 : (e > c_len ? c_len : e);
        if (e > s) {                                          // reflen == 0 or entirely outside the contig: nothing
          atomicAdd(delta + c_base + s, 1);
          atomicAdd(delta + c_base + e, -1);
          if (STARTS) atomicAdd(f.starts + c_base + s, 1);
          n_pass += 1;
          aligned += R.reflen[r];
        }
      }
    }
  }
  prep_flush_counters(a.pc, n_pass, aligned, unsorted, 0u);
}

// The exact cap metric of an any-order pass, after the scan: max_p depth[p-1] + starts[p] over the slot space.  Every
// contig ends in a sentinel slot of depth 0 that no read starts at, so the maximum over the concatenation is the maximum
// within each contig with depth[-1] = 0.  Four slots per thread and step, 128-bit loads of both arrays.
__global__ void __launch_bounds__(256)
k_cap_exact(const int32_t* __restrict__ depth, const int32_t* __restrict__ starts, int64_t n_slots, PassCounters* pc) {
  const int64_t n_vec = n_slots >> 2;                            // (n_slots is a multiple of 4)
  int m = 0;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_vec; k += (int64_t)gridDim.x * blockDim.x) {
    const int4 d = __ldg(reinterpret_cast<const int4*>(depth) + k);
    const int4 s = __ldg(reinterpret_cast<const int4*>(starts) + k);
    const int prev = k ? __ldg(depth + 4 * k - 1) : 0;
    m = max(m, max(max(prev + s.x, d.x + s.y), max(d.y + s.z, d.z + s.w)));
  }
  m = warp_max(m);
  __shared__ int s_m[8];
  if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    int b = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) b = max(b, s_m[w]);
    if (b > 0) atomicMax(&pc->cap_metric, b);
  }
}

// Per-warp state of a prep kernel: pass counters and the constants of the warp's current contig
// (reloaded only when the contig changes).
struct PrepWarp {
  unsigned long long aligned;
  uint32_t n_pass, max_span, unsorted;
  int32_t w_tid;
  uint32_t w_len, w_tb, w_bo;
};

// Everything after the loads + filter + CIGAR reduction of one warp iteration (shared by both prep
// kernels): a warp-uniform FAST PATH takes the overwhelmingly common case -- all 128 reads of the
// warp (and the read before them, pvT/pvP on lane 0) lie in one valid contig at non-negative
// positions -- where the contig's constants live in uniform registers and nothing is 64-bit.  Near
// reads need no per-tile aggregate (see the file header), so the only cross-thread work is the tile
// border detection.  Any other warp iteration takes prep_general.
__device__ __forceinline__ void prep_emit(const FusedArgs& f, const int64_t i0, const PrepReads& R, const int32_t pvT,
                                          const int32_t pvP, const int lane, PrepWarp& W) {
  const ExpandArgs& a = f.e;
  const uint32_t n_contigs = (uint32_t)a.n_contigs;
  const int64_t n = a.n;
  const int32_t* T = R.T;
  const int32_t* P = R.P;
  const uint32_t* reflen = R.reflen;
  const unsigned passm = R.passm;

  const int32_t Tw = __shfl_sync(0xffffffffu, T[0], 0);
  bool simple = R.nv == kPrepPer && T[0] == Tw && T[1] == Tw && T[2] == Tw && T[3] == Tw && (P[0] | P[1] | P[2] | P[3]) >= 0;
  if (lane == 0) simple = simple && pvT == Tw && pvP >= 0;
  if (!(__all_sync(0xffffffffu, simple) && (uint32_t)Tw < n_contigs)) {
    const PrepAcc pa = prep_general(f, i0, R.nv, T[0], T[1], T[2], T[3], P[0], P[1], P[2], P[3], reflen[0], reflen[1],
                                    reflen[2], reflen[3], passm, lane);
    W.n_pass += pa.n_pass; W.aligned += pa.al32; W.max_span = max(W.max_span, pa.max_span); W.unsorted |= pa.unsorted;
    return;
  }
  if (Tw != W.w_tid) {                               // warp-uniform
    W.w_tid = Tw;
    const int64_t base = a.contig_off[Tw];
    W.w_len = (uint32_t)a.contig_len[Tw];
    W.w_tb = (uint32_t)(base >> kTileShift); W.w_bo = (uint32_t)base & (kTile - 1);
  }
  const uint32_t w_len = W.w_len, w_tb = W.w_tb, w_bo = W.w_bo;
  uint32_t q[4], sq[4], rc[4];
  uint32_t al32 = 0, n_pass = 0, max_span = W.max_span;
  unsigned farmask = 0;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    q[r] = min((uint32_t)P[r], w_len);
    const uint32_t e = min((uint32_t)P[r] + reflen[r], w_len);     // P >= 0 and reflen < 2^31: no wrap
    const uint32_t sp = ((passm >> r) & 1u) ? e - q[r] : 0u;
    sq[r] = w_bo + q[r];
    const bool far = sp > kNearSpan;
    rc[r] = (sq[r] & (kTile - 1)) | ((far ? kRecFar : sp) << kTileShift);
    n_pass += sp ? 1u : 0u;
    al32 += sp ? reflen[r] : 0u;
    farmask |= far ? (1u << r) : 0u;
    max_span = max(max_span, far ? 0u : sp);
  }
  W.aligned += al32; W.n_pass += n_pass; W.max_span = max_span;
  *reinterpret_cast<uint4*>(f.rec + i0) = make_uint4(rc[0], rc[1], rc[2], rc[3]);
  // sorted inside the contig <=> clamped positions never decrease
  uint32_t pq = __shfl_up_sync(0xffffffffu, q[3], 1);
  if (lane == 0) pq = min((uint32_t)pvP, w_len);
  W.unsorted |= (q[0] < pq || q[1] < q[0] || q[2] < q[1] || q[3] < q[2]) ? 1u : 0u;
  // tiles relative to the contig's first tile
  const uint32_t t3 = sq[3] >> kTileShift;
  uint32_t ptile = __shfl_up_sync(0xffffffffu, t3, 1);
  if (lane == 0) ptile = (w_bo + pq) >> kTileShift;
  const bool is_last = i0 + kPrepPer == n;
  if (__any_sync(0xffffffffu, t3 > ptile || is_last)) {
    // a tile border inside the warp's reads: the first read of every tile entered writes its index
    if (__any_sync(0xffffffffu, t3 - ptile > 4u || is_last)) {       // long gaps / end of batch: warp-cooperative
      prep_tile_boundaries(f.tile_first, i0, kPrepPer, (int64_t)(w_tb + ptile), w_tb + (sq[0] >> kTileShift),
                           w_tb + (sq[1] >> kTileShift), w_tb + (sq[2] >> kTileShift), w_tb + t3, is_last, n,
                           (uint32_t)f.n_tiles, lane);
    } else if (t3 > ptile) {
      uint32_t* __restrict__ tf = f.tile_first + w_tb;
      uint32_t prev = ptile;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const uint32_t tr = sq[r] >> kTileShift;
        for (uint32_t T2 = prev + 1; T2 <= tr; ++T2) tf[T2] = (uint32_t)(i0 + r);
        prev = max(prev, tr);
      }
    }
  }
  if (__any_sync(0xffffffffu, farmask != 0)) {
    const int64_t base = a.contig_off[Tw];
    int64_t e64[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) e64[r] = base + min((uint32_t)P[r] + reflen[r], w_len);
    prep_far(f, w_tb + (sq[0] >> kTileShift), w_tb + (sq[1] >> kTileShift), w_tb + (sq[2] >> kTileShift), w_tb + t3, e64[0],
             e64[1], e64[2], e64[3], farmask, lane);
  }
}

// First kernel of the fused path: 4 consecutive reads per thread, 128-bit SoA loads.
template <bool OFF64>
__global__ void __launch_bounds__(kPrepThreads, 4)
k_fused_prep(const __grid_constant__ FusedArgs f) {
  pdl_launch_dependents();                                    // k_scan_counts may take free slots as this grid drains
  const ExpandArgs& a = f.e;
  const int lane = threadIdx.x & 31;
  const int64_t n = a.n;
  const int64_t n_groups = (n + kPrepPer - 1) / kPrepPer;
  const int64_t g_round = (n_groups + 31) & ~(int64_t)31;     // whole warps iterate together
  const int64_t g_stride = (int64_t)gridDim.x * kPrepThreads;
  PrepWarp W = {0ull, 0u, 0u, 0u, -1, 0u, 0u, 0u};
#pragma unroll 1
  for (int64_t g = (int64_t)blockIdx.x * kPrepThreads + threadIdx.x; g < g_round; g += g_stride) {
    const int64_t i0 = g * kPrepPer;
    // the read before this warp's first one (lane 0 only): sortedness and tile border across warps
    int32_t pvT = -1, pvP = -1;
    if (lane == 0 && i0 > 0 && i0 - 1 < n) { pvT = a.tid[i0 - 1]; pvP = a.pos[i0 - 1]; }
    const PrepReads R = prep_load_reduce<OFF64>(f, i0, lane);
    prep_emit(f, i0, R, pvT, pvP, lane, W);
  }
  prep_flush_counters(a.pc, W.n_pass, W.aligned, W.unsorted, W.max_span);
}

// (A cp.async-staged version of this kernel -- every hot-loop load issued one to two iterations
// ahead into shared memory, 3+2 buffers, 54 KB per CTA -- was measured on B200 and is SLOWER:
// 79.3 vs 69.8 us on C2, 689 vs 570 us on C4 x0.1.  The kernel is bound by instruction issue and
// dependent-instruction latency (about 130 thread instructions per read), not by exposed HBM
// latency; the extra LDGSTS/LDS/DEPBAR instructions cost more than the overlap gains.  DESIGN.md 5.)

// bucket far ends by tile; tile_cnt holds the INCLUSIVE scan of the per-tile counts.  Because the
// scan runs over [tile_agg | tile_cnt] as one array and tile_agg sums to zero, tile_cnt's running
// sum starts from zero.
__global__ void k_far_scatter(FusedArgs f) {
  pdl_wait();
  pdl_launch_dependents();
  // tiles that hold very many reads (skewed abundance: a 4000x contig puts ~55 k reads into one tile,
  // 100x the average of config C3) are listed here so that the tile kernel can start with them
  for (int64_t T = f.tile_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; T < f.tile_hi; T += (int64_t)gridDim.x * blockDim.x) {
    if (f.tile_first[T + 1] - f.tile_first[T] >= f.heavy_min) f.tile_heavy[atomicAdd(&f.e.pc->n_heavy, 1u)] = (uint32_t)T;
  }
  uint32_t n_far = min(f.e.pc->n_far, f.far_cap);
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_far; k += gridDim.x * blockDim.x) {
    int64_t e = f.far_end[k];
    int64_t T = e >> kTileShift;
    uint32_t base = T > 0 ? f.tile_cnt[T - 1] : 0u;
    uint32_t p = atomicAdd(f.tile_cursor + T, 1u);
    f.far_sorted[base + p] = (uint32_t)(e - (T << kTileShift));
  }
}

// Exact replay of htslib's max_depth cap for the contigs where it can fire (SURVEY.md Appendix
// A-6; restated sequentially in oracle/coverage.c::orc_depth_plp).  For a whole-contig iterator the
// machine reduces to a recurrence over positions: with m(p) passing reads starting at p (file
// order) and D[p-1] the capped depth just before, the first
//     K(p) = max(1, min(m(p), max_depth - D[p-1]))
// of them are kept (the first read at a position is pushed while the iterator is still behind it
// and is never dropped; every later one is dropped once max_depth reads are buffered).  D depends
// on earlier decisions, so a contig is replayed by ONE thread, in place: the contig's slots are
// first cleared, kept reads add +1 at their end slot, and the running depth overwrites each slot
// as the walk passes it.  Only contigs flagged through tile_cap are replayed.
//
// The recurrence for one contig.  d[0 .. len] receives the capped depth (contig-relative positions; d[len] = sentinel 0).
// Only reads overlapping [rs, re) take part (rs = 0, re > len: every read of the contig -- the whole-contig iterator;
// else the reads `bam.fetch(ref, rs, re)` hands the per-region iterator pysam builds for pileup(ref, rs, re), reference
// metacov/cli.py:85-95 -> pileup.py:13).
__device__ void cap_replay_contig(const FusedArgs& f, const int c, int32_t* d, const int64_t rs, const int64_t re) {
  const int64_t base = f.e.contig_off[c];
  const int32_t len = f.e.contig_len[c];
  for (int32_t p = 0; p <= len; ++p) d[p] = 0;
  // Reads in file order from the first read of the tile holding the contig's first slot.  A
  // record stores its start relative to its tile; the tile follows from tile_first.
  int64_t T = base >> kTileShift;
  int64_t j = f.tile_first[T];
  const int64_t n = f.e.n;
  // contig-relative start of read j (advances T as j crosses tile borders); > len = past the contig
  auto rel = [&](int64_t jj) -> int64_t {
    while (T + 1 <= f.n_tiles && jj >= f.tile_first[T + 1]) ++T;
    return (T << kTileShift) + (int64_t)(f.rec[jj] & (kTile - 1)) - base;
  };
  while (j < n && rel(j) < 0) ++j;                  // reads of the previous contig sharing the tile
  int depth = 0;
  const int maxcnt = f.max_depth;
  int32_t p = 0;
  while (p < len) {
    // reads starting at p (sorted keys): keep the first K
    int kept = 0;
    bool first = true;
    while (j < n) {
      int64_t q = rel(j);
      if (q != p || q > len) break;
      uint32_t code = f.rec[j] >> kTileShift;
      ++j;
      if (code == 0) continue;                      // filtered / empty read
      int64_t span = code;
      if (code == kRecFar) {                        // long span: not in the record, reduce the CIGAR again
        int64_t rl = 0;
        const uint64_t o0 = f.e.cig_off64 ? f.e.cig_off64[j - 1] : f.e.cig_off[j - 1];
        const uint64_t o1 = f.e.cig_off64 ? f.e.cig_off64[j] : f.e.cig_off[j];
        for (uint64_t o = o0; o < o1; ++o) rl += cigar_ref_len(f.e.cig[o]);
        int64_t e = (int64_t)p + rl;
        span = (e > len ? len : e) - p;
      }
      if (!((int64_t)p + span > rs && (int64_t)p < re)) continue;     // not among the reads this iterator is given
      bool keep = first || (depth + kept) < maxcnt; // depth = D[p-1] = reads buffered from earlier positions
      first = false;
      if (keep) { ++kept; d[p + span] += 1; }
    }
    int32_t ends = d[p];
    depth += kept - ends;
    d[p] = depth;
    ++p;
    // no more reads in this contig: only the ends remain to be folded in
    if (j >= n || rel(j) > len) {
      for (; p < len; ++p) { depth -= d[p]; d[p] = depth; }
      break;
    }
  }
  d[len] = 0;                                       // sentinel slot
}

__global__ void k_cap_replay(FusedArgs f, uint8_t* __restrict__ contig_capped) {
  pdl_wait();                                       // the tile kernel is complete: cap_metric and tile_cap are final
  pdl_launch_dependents();
  // Launched after EVERY fused pass on the same stream, so whatever consumes the depth next
  // (statistics, copies, exports, pipelined or not) sees the capped depth; one load and out when
  // the cap cannot fire anywhere (always, in BASELINE's configs).
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= f.e.n_contigs || f.max_depth <= 0) return;
  if (f.e.pc->cap_metric <= f.max_depth) return;
  if (f.e.pc->unsorted || f.e.pc->n_far > f.far_cap) return;     // the pass is rejected by the verdict: nothing to replay
  if (f.streaming) { if (c == 0) f.e.pc->cap_unreplayed = 1u; return; }   // a contig's reads may lie in other batches: reported, not replayed
  {
    const int64_t b0 = f.e.contig_off[c];
    const int64_t T0 = b0 >> kTileShift, T1 = min((b0 + f.e.contig_len[c]) >> kTileShift, f.n_tiles - 1);
    bool hit = false;
    for (int64_t T = T0; T <= T1 && !hit; ++T) hit = f.tile_cap[T] > f.max_depth;
    if (!hit) return;
  }
  atomicAdd(&f.e.pc->cap_contigs, 1u);
  contig_capped[c] = 1;
  if (f.tile_hist) {                                // the histograms of the contig's tiles describe the uncapped depth
    const int64_t b0 = f.e.contig_off[c];
    const int64_t T1 = min((b0 + f.e.contig_len[c]) >> kTileShift, f.n_tiles - 1);
    for (int64_t T = b0 >> kTileShift; T <= T1; ++T) f.tile_hist[T * kTileHistWords] = kTileHistNone;
  }
  cap_replay_contig(f, c, f.depth + f.e.contig_off[c], 0, (int64_t)f.e.contig_len[c] + 1);
}

// Per-REGION replay (mcov_region_stats_run, regions that do not start at 0 inside a capped contig): pysam builds a fresh
// iterator per pileup(ref, start, end) call and gives it only the reads overlapping the region, so fewer reads are
// buffered when the pile is reached and a few more of it are kept than the whole-contig iterator keeps.  One thread per
// region; the capped depth of the region's contig under THAT iterator goes to scratch[off[k] .. off[k] + len].
__global__ void k_cap_replay_region(FusedArgs f, int n_reg, const int32_t* __restrict__ r_tid, const int32_t* __restrict__ r_start,
                                    const int32_t* __restrict__ r_end, const int64_t* __restrict__ scratch_off, int32_t* scratch) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_reg) return;
  cap_replay_contig(f, r_tid[k], scratch + scratch_off[k], r_start[k], r_end[k]);
}

// ---- compact host transport (mcov_depth_sorted_packed) ---------------------------------------------
// The PCIe link, not the GPU, bounds the end-to-end rate, so the host may ship a coordinate-sorted
// batch without the redundant columns: the contig of read i follows from a per-contig read-count
// prefix (instead of tid[R]), CIGAR offsets follow from u16 op counts (instead of u32 offsets), and
// mapq may be omitted when the filter does not look at it.  This kernel rebuilds tid[] and seeds the
// offset scan; k_scan_inplace turns the counts into cig_off[].
__global__ void k_unpack_reads(int64_t n, const int64_t* __restrict__ contig_read_start, int32_t n_contigs,
                               const uint16_t* __restrict__ ncig, int32_t* __restrict__ tid, uint32_t* __restrict__ cig_off,
                               int64_t off_len) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < off_len) cig_off[i] = (i >= 1 && i <= n) ? (uint32_t)ncig[i - 1] : 0u;      // entry 0 and the padding are 0
  if (i >= n) return;
  // contig of read i: largest c with contig_read_start[c] <= i; reads past the last contig are unplaced
  int32_t lo = 0, hi = n_contigs;
  if (i >= contig_read_start[n_contigs]) { tid[i] = -1; return; }
  while (hi - lo > 1) {
    int32_t mid = lo + ((hi - lo) >> 1);
    if (contig_read_start[mid] <= i) lo = mid; else hi = mid;
  }
  tid[i] = lo;
}

// ---- delta transport (mcov_depth_sorted_delta) ---------------------------------------------------------
// The end-to-end rate is PCIe-bound, so the host columns are narrowed further: positions as u16 differences
// to the previous read of the same contig (the first read of a contig: to 0), with the few differences that
// do not fit (or are negative: unsorted input travels faithfully) as (index, 32-bit difference) exceptions;
// u8 op counts; u16 ops (len << 4 | op with len < 4096: any short-read CIGAR).  7.3 bytes per read on config C2
// instead of 12.6.  Rebuilt here: differences widened + exceptions patched (k_delta_seed, k_delta_patch), ONE
// plain int32 prefix sum over the whole batch (wrap-around is harmless: only differences inside a contig are
// used), then pos[i] = S[i] - S[first read of the contig - 1] (k_delta_finish).
__global__ void k_delta_seed(int64_t n, const int64_t* __restrict__ contig_read_start, int32_t n_contigs,
                             const uint16_t* __restrict__ dpos, const uint8_t* __restrict__ ncig, int32_t* __restrict__ S,
                             int32_t* __restrict__ tid, uint32_t* __restrict__ cig_off, int64_t off_len) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < off_len) {
    cig_off[i] = (i >= 1 && i <= n) ? (uint32_t)ncig[i - 1] : 0u;      // entry 0 and the padding are 0
    S[i] = i < n ? (int32_t)dpos[i] : 0;
  }
  if (i >= n) return;
  int32_t lo = 0, hi = n_contigs;
  if (i >= contig_read_start[n_contigs]) { tid[i] = -1; return; }
  while (hi - lo > 1) {
    int32_t mid = lo + ((hi - lo) >> 1);
    if (contig_read_start[mid] <= i) lo = mid; else hi = mid;
  }
  tid[i] = lo;
}

__global__ void k_delta_patch(int64_t n_exc, const uint32_t* __restrict__ idx, const int32_t* __restrict__ delta, int64_t n,
                              int32_t* __restrict__ S) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n_exc && idx[k] < n) S[idx[k]] = delta[k];
}

__global__ void k_delta_finish(int64_t n, const int64_t* __restrict__ contig_read_start, int32_t n_contigs,
                               const int32_t* __restrict__ tid, const int32_t* __restrict__ S, int32_t* __restrict__ pos,
                               const uint16_t* __restrict__ cig16, uint32_t* __restrict__ cig, int64_t n_cig) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = i; k < n_cig; k += stride) cig[k] = cig16[k];
  for (; i < n; i += stride) {
    const int32_t t = tid[i];
    const int64_t first = contig_read_start[t >= 0 ? t : n_contigs];      // unplaced reads: one more segment
    pos[i] = (int32_t)((uint32_t)S[i] - (first > 0 ? (uint32_t)S[first - 1] : 0u));
  }
}

// ---- count_del = 0: only M = X positions count ------------------------------------------------------------
// The additive switch of mcov_filter (the reference reads `column.n`, which counts D / N positions too): a read is
// then one interval per run of M = X ops, so it goes through the any-order formulation -- +1 / -1 per run into the
// difference array, look-back scan afterwards.  One thread per read, ops walked serially: the generic path, not
// the tuned one.  Reads [i_begin, n) of the batch are expanded (a streamed batch skips its carried prefix).
__global__ void k_expand_runs(FusedArgs f, int64_t i_begin) {
  const ExpandArgs& a = f.e;
  unsigned long long np = 0, al = 0;
  for (int64_t i = i_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t t = a.tid[i];
    if (!read_passes(a.flag[i], a.mapq[i], a.filt) || (uint32_t)t >= (uint32_t)a.n_contigs) continue;
    const uint64_t o0 = a.cig_off64 ? a.cig_off64[i] : a.cig_off[i], o1 = a.cig_off64 ? a.cig_off64[i + 1] : a.cig_off[i + 1];
    const int64_t L = a.contig_len[t];
    int32_t* d = a.delta + a.contig_off[t];
    int64_t p = a.pos[i], counted = 0, consumed = 0;
    bool hit = false;
    for (uint64_t o = o0; o < o1; ++o) {
      const uint32_t op = a.cig[o], c = op & 15u;
      const int64_t ln = op >> 4;
      if (c == 0u || c == 7u || c == 8u) {
        const int64_t s = min(max(p, (int64_t)0), L), e = min(max(p + ln, (int64_t)0), L);
        if (e > s) { atomicAdd(d + s, 1); atomicAdd(d + e, -1); hit = true; }
        counted += ln; p += ln; consumed += ln;
      } else if (c == 2u || c == 3u) { p += ln; consumed += ln; }
    }
    if (consumed == 0 && a.filt.reflen0_as_one) {
      const int64_t s = a.pos[i];
      if (s >= 0 && s < L) { atomicAdd(d + s, 1); atomicAdd(d + s + 1, -1); hit = true; counted = 1; }
    }
    if (hit) { np += 1; al += (unsigned long long)counted; }
  }
  np = warp_sum(np); al = warp_sum(al);
  if ((threadIdx.x & 31) == 0) { if (np) atomicAdd(&a.pc->n_pass, np); if (al) atomicAdd(&a.pc->aligned_bases, al); }
}

// ---- streamed passes (mcov_stream_begin / mcov_stream_push) ---------------------------------------------
// A batch of a streamed file starts with n_carry reads that earlier batches have already counted (they are
// sent again because their intervals reach into this batch's tiles): their contribution to the pass counters
// is computed here and taken out again by k_stream_accumulate.
struct StreamAcc { unsigned long long n_pass, aligned_bases; int max_depth_seen, cap_metric; unsigned unsorted, cap_unreplayed, far_overflow, pad; };

__global__ void k_carry_counts(FusedArgs f, int64_t n_carry, unsigned long long* out /* [2]: n_pass, aligned */) {
  const ExpandArgs& a = f.e;
  unsigned long long np = 0, al = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_carry; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t t = a.tid[i];
    if (!read_passes(a.flag[i], a.mapq[i], a.filt) || (uint32_t)t >= (uint32_t)a.n_contigs) continue;
    const uint64_t o0 = a.cig_off64 ? a.cig_off64[i] : a.cig_off[i], o1 = a.cig_off64 ? a.cig_off64[i + 1] : a.cig_off[i + 1];
    int64_t rl = 0;
    for (uint64_t o = o0; o < o1; ++o) rl += cigar_ref_len(a.cig[o]);
    if (rl > 0x7fffffffll) rl = 0x7fffffffll;
    if (rl == 0 && a.filt.reflen0_as_one) rl = 1;
    const int64_t len = a.contig_len[t];
    int64_t s = a.pos[i], e = (int64_t)a.pos[i] + rl;
    s = s < 0 ? 0 : (s > len ? len : s);
    e = e < 0 ? 0 : (e > len ? len : e);
    if (e > s) { np += 1; al += (unsigned long long)rl; }
  }
  np = warp_sum(np); al = warp_sum(al);
  if ((threadIdx.x & 31) == 0) { if (np) atomicAdd(out, np); if (al) atomicAdd(out + 1, al); }
}

// one thread: totals of the stream so far += this batch's counters - its carried reads; the totals are then written
// back into the pass counters, so that every reader of PassCounters (verdict, mcov_pass_info_get) sees the stream.
__global__ void k_stream_accumulate(PassCounters* pc, StreamAcc* acc, const unsigned long long* carry, uint32_t far_cap) {
  acc->n_pass += pc->n_pass - carry[0];
  acc->aligned_bases += pc->aligned_bases - carry[1];
  acc->max_depth_seen = max(acc->max_depth_seen, pc->max_depth_seen);
  acc->cap_metric = max(acc->cap_metric, pc->cap_metric);
  acc->unsorted |= (unsigned)pc->unsorted;
  acc->cap_unreplayed |= pc->cap_unreplayed;
  acc->far_overflow |= pc->n_far > far_cap ? 1u : 0u;
  pc->n_pass = acc->n_pass; pc->aligned_bases = acc->aligned_bases;
  pc->max_depth_seen = acc->max_depth_seen; pc->cap_metric = acc->cap_metric;
  pc->unsorted = (int)acc->unsorted; pc->cap_unreplayed = acc->cap_unreplayed; pc->far_overflow = acc->far_overflow;
  pc->n_far = 0;
}

}  // namespace mcov
