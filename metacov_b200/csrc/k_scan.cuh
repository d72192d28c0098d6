// k_scan.cuh -- K2: single-pass prefix scan of the difference array (in place).
//
// Turns the +1/-1 deltas into per-base depth = the `column.n` the reference
// accumulates at metacov/pileup.py:16.  Segmentation is implicit: contig c
// owns len[c]+1 slots and every read's -1 lands inside its own contig's slots
// (ends clipped to the sentinel slot), so the running sum is 0 at every contig
// start and one plain scan over the concatenation is the segmented scan.
//
// Decoupled look-back (one pass, 4 B read + 4 B write per slot = 8*(L+C)
// algorithmic bytes).  Tile = 512 threads x 32 slots (64 KB), warp-striped
// L1-bypassing 128-bit loads/stores, tile id drawn as a ticket.
//
// Measured on B200, C2 (50 M slots; profiles/r01_o_scan_sweep.txt, r01_p_scan_variants.txt):
//   150.5 us  256 thr x 16 slots, atomic ticket for the tile id (first version)
//   109.7 us  this shape
//   118.8 us  + look-back by the whole CTA (512 predecessors per round instead of 32)
//   153.8 us  persistent CTAs, tiles i+1.. staged with cp.async while tile i is scanned (best of 7 shapes)
// ncu on this shape: 50 % of the stall samples sit at the barrier behind warp 0's look-back and
// 20 % on the tile's own loads -- a tile lives ~10 us, most of it waiting for its predecessors'
// aggregates, and neither a wider window nor prefetching shortens that wait.  The fused path
// (k_fused.cuh) exists because its tiles need no predecessor at all.
#pragma once
#include "common.cuh"

namespace mcov {

#ifndef MCOV_SCAN_VEC
#define MCOV_SCAN_VEC 8
#endif
#ifndef MCOV_SCAN_THREADS
#define MCOV_SCAN_THREADS 512
#endif
constexpr int kScanThreads = MCOV_SCAN_THREADS;
constexpr int kScanVec = MCOV_SCAN_VEC;                       // int4 per thread
constexpr int kScanTile = kScanThreads * kScanVec * 4;        // 16384 slots (64 KB)

// tile status word: [63:62] state, [31:0] value
constexpr unsigned long long kTileAggregate = 1ull << 62;
constexpr unsigned long long kTilePrefix = 2ull << 62;

// Look-back by warp 0: returns the exclusive prefix of tile `tile`.
__device__ __forceinline__ int scan_lookback(unsigned long long* status, int64_t tile, int lane) {
  int prefix = 0;
  int64_t t = tile - 1 - lane;
  while (true) {
    unsigned long long w = 0;
    unsigned st = 2;                       // tiles before 0 count as "prefix 0"
    if (t >= 0) {
      do {
        w = ld_acquire_u64(status + t);
        st = (unsigned)(w >> 62);
      } while (st == 0);
    }
    unsigned has_prefix = __ballot_sync(0xffffffffu, st == 2);
    int v = (t >= 0) ? (int)(uint32_t)w : 0;
    if (has_prefix) {
      int first = __ffs(has_prefix) - 1;   // nearest tile with a full prefix
      v = (lane <= first) ? v : 0;
      prefix += warp_sum(v);
      return prefix;
    }
    prefix += warp_sum(v);
    t -= 32;
  }
}

template <bool kMetrics>
__global__ void __launch_bounds__(kScanThreads)
k_scan_inplace(int32_t* __restrict__ data, int64_t n_slots, unsigned long long* status,
               PassCounters* pc) {
  __shared__ int s_warp[kScanThreads / 32];
  __shared__ int s_prefix;
  // A tile spins on its predecessors, so they must be running or done.  CTAs are dispatched in index order in practice
  // (CUB's decoupled look-back with static tile ids relies on the same), but nothing guarantees it -- least of all next
  // to programmatic dependent launches -- so the tile id is a TICKET drawn from a counter behind the status words: a
  // CTA only ever waits for tiles whose CTAs have started.  Cost: one L2 round trip per CTA (0.2 us on the three-tile
  // scan between prep and tile, nothing measurable on the 3 052 tiles of the push path).
  __shared__ unsigned s_tile;
  pdl_wait();
  if (threadIdx.x == 0) s_tile = atomicAdd(reinterpret_cast<unsigned*>(status + gridDim.x), 1u);
  __syncthreads();
  const int64_t tile = s_tile;
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = tile * kScanTile;
  int4* vp = reinterpret_cast<int4*>(data + base);
  const int64_t n_vec = (n_slots - base + 3) >> 2;             // buffer is padded to a multiple of 4

  int4 v[kScanVec];
  int run[kScanVec];
#pragma unroll
  for (int j = 0; j < kScanVec; ++j) {
    int idx = (warp * kScanVec + j) * 32 + lane;
    v[j] = (idx < n_vec) ? ld_na_int4(vp + idx) : make_int4(0, 0, 0, 0);
    v[j].y += v[j].x; v[j].z += v[j].y; v[j].w += v[j].z;
    run[j] = v[j].w;
  }
  // inclusive scan of each 32-lane run, then chain the 4 runs of this warp
  int carry = 0;
#pragma unroll
  for (int j = 0; j < kScanVec; ++j) {
    int x = run[j];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    int total = __shfl_sync(0xffffffffu, x, 31);
    run[j] = x - run[j] + carry;          // exclusive offset of this thread's int4
    carry += total;
  }
  if (lane == 31) s_warp[warp] = carry;
  __syncthreads();
  if (warp == 0) {
    int wv = (lane < kScanThreads / 32) ? s_warp[lane] : 0;
    int x = wv;
#pragma unroll
    for (int o = 1; o < kScanThreads / 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    int tile_sum = __shfl_sync(0xffffffffu, x, kScanThreads / 32 - 1);
    if (lane < kScanThreads / 32) s_warp[lane] = x - wv;      // exclusive warp offsets
    int prefix = 0;
    if (tile > 0) {
      if (lane == 0) st_release_u64(status + tile, kTileAggregate | (uint32_t)tile_sum);
      prefix = scan_lookback(status, tile, lane);
    }
    if (lane == 0) {
      st_release_u64(status + tile, kTilePrefix | (uint32_t)(prefix + tile_sum));
      s_prefix = prefix;
    }
  }
  __syncthreads();
  const int off = s_prefix + s_warp[warp];
  int mx = 0, pair = 0;
#pragma unroll
  for (int j = 0; j < kScanVec; ++j) {
    int idx = (warp * kScanVec + j) * 32 + lane;
    int o = off + run[j];  // exclusive prefix of this thread's int4
    int prev = o;                           // depth of the slot just before this int4
    v[j].x += o; v[j].y += o; v[j].z += o; v[j].w += o;
    mx = max(mx, max(max(v[j].x, v[j].y), max(v[j].z, v[j].w)));
    // upper bound of the cap metric: depth[p-1] + depth[p] >= depth[p-1] + starts[p]
    pair = max(pair, max(max(prev + v[j].x, v[j].x + v[j].y), max(v[j].y + v[j].z, v[j].z + v[j].w)));
    if (idx < n_vec) st_stream_int4(vp + idx, v[j]);
  }
  if (!kMetrics) return;
  mx = warp_max(mx);
  pair = warp_max(pair);
  __syncthreads();
  if (lane == 0) { s_warp[warp] = mx; }
  __shared__ int s_pair[kScanThreads / 32];
  if (lane == 0) s_pair[warp] = pair;
  __syncthreads();
  if (threadIdx.x == 0) {
    int m = 0, p2 = 0;
    for (int k = 0; k < kScanThreads / 32; ++k) { m = max(m, s_warp[k]); p2 = max(p2, s_pair[k]); }
    if (m > 0) atomicMax(&pc->max_depth_seen, m);
    if (p2 > 0) atomicMax(&pc->cap_metric, p2);
  }
}

}  // namespace mcov
