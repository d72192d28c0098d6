// k_stats.cuh -- K3/K4: per-region statistics of the depth array, one read of
// the depth per region.
//
// Replaces the seven reductions of `classic` (reference metacov/pileup.py:
// 18-26): min, max, sum, sum of squares (-> std), and the two order statistics
// the reference gets from `np.median` (pileup.py:21) and from
// `sorted(columns)[n//4 : n-n//4]` (pileup.py:24).  EVERYTHING is derived from
// an exact counting histogram of the depth values (one bin per value, kHistBins
// bins in shared memory), so the streaming loop does nothing but feed it:
//   sum = sum_b b*cnt[b], sumsq = sum_b b^2*cnt[b], min/max = first/last
//   non-empty bin, breadth = n - cnt[0], ranks by walking the running count.
// With htslib's default max_depth = 8000 a depth never reaches kHistBins =
// 8192, so one pass is exact.  A region holding a depth >= kHistBins-1 lands in
// the last bin, is flagged kStatOverflow and is finished exactly by the GPU
// radix-sort path (stats_sort.cu).
//
// Regions are arbitrary [start,end) slices and may overlap (reference
// cli.py:85-95 with tests/data/regions.blast7).  Regions longer than
// kSmallRegion slots go through the balanced stream of k_stats_stream.cuh; the
// others get one warp each (k_region_stats_warp), with one CTA each as the
// retry path (k_region_stats_small).
//
// HBM bytes per launch (algorithmic): 4 * sum(region lengths) + 64 * G.
#pragma once
#include "common.cuh"

namespace mcov {

constexpr int kStatThreads = 512;
constexpr int kHistBins = 8192;
constexpr int kStatValid = 1;      // mcov_region_stats.flags bit0
constexpr int kStatOverflow = 2;   // bit1

struct StatTask {
  int64_t slot;     // first slot of the region inside the depth array
  int32_t n;        // slots of the region inside its contig
  int32_t region;   // region index
};

struct StatArgs {
  const int32_t* depth;
  const StatTask* tasks;
  const int32_t* region_len;      // slots of the region inside its contig
  const int32_t* region_pad;      // positions of the region beyond the contig end: depth 0 there
  mcov_region_stats* out;         // device; every record is fully written by exactly one warp or CTA
  int32_t breadth_n;
};

// depth -> bin; anything outside [0, kHistBins-1) lands in the last bin (flagged as overflow)
__device__ __forceinline__ int hist_bin(int v) { return (unsigned)v < (unsigned)(kHistBins - 1) ? v : kHistBins - 1; }

struct WalkOut {
  long long sum, iq_sum, ge1, geN;
  unsigned long long sumsq;
  int mn, mx, med_lo, med_hi;
};

// Walk the bins [lo, hi] of a counting histogram held in shared memory (bins outside the range are
// not touched and may hold garbage); all THREADS threads participate, the result is valid on the
// first of them.  n = number of values the histogram describes.
// CONSUMERS_ONLY: the THREADS threads (an aligned group of threadIdx.x) are some of the warps of a warp-specialised CTA
// and meet at named barrier BAR.
// CLEAR: every thread zeroes the bins it walked, so [lo, hi] is zero again once all threads are past the walk's
// second barrier (bins outside it must be zero on entry).
template <int THREADS, bool CONSUMERS_ONLY = false, bool CLEAR = false, int BAR = 1>
__device__ __forceinline__ WalkOut hist_walk(uint32_t* hist, long long n, int breadth_n, int lo, int hi,
                                             unsigned long long* s_u64 /* [6][THREADS/32] */,
                                             int* s_i32 /* [4][THREADS/32] */, int* s_med /* 2 */) {
  constexpr int kW = THREADS / 32;
  const long long k1 = n / 4, k2 = n - n / 4;                // interquartile ranks [k1, k2)
  const long long m1 = (n - 1) / 2, m2 = n / 2;              // median pair
  const int t = threadIdx.x % THREADS, lane = t & 31, warp = t >> 5;
  const int per = (hi - lo + THREADS) / THREADS;             // bins per thread (>= 1)
  const int b0 = lo + t * per, b1 = min(b0 + per, hi + 1);   // this thread's bins [b0, b1)
  unsigned long long local = 0;
  for (int b = b0; b < b1; ++b) local += hist[b];
  // block exclusive scan of `local`
  unsigned long long x = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_u64[warp] = x;
  if (CONSUMERS_ONLY) named_bar_sync<BAR, THREADS>(); else __syncthreads();
  unsigned long long before = 0;
#pragma unroll
  for (int k = 0; k < kW; ++k) before += (k < warp) ? s_u64[k] : 0ull;
  long long c = (long long)(before + x - local);              // values sorted before bin b0
  long long sum = 0, iq = 0, ge1 = 0, geN = 0;
  unsigned long long sumsq = 0;
  int mn = INT_MAX, mx = INT_MIN;
  if (local) {
    for (int bb = b0; bb < b1; ++bb) {
      long long cn = hist[bb];
      if (cn) {
        long long b = bb;
        sum += b * cn;
        sumsq += (unsigned long long)(b * b) * (unsigned long long)cn;
        ge1 += b >= 1 ? cn : 0;
        geN += b >= breadth_n ? cn : 0;
        mn = min(mn, bb); mx = max(mx, bb);
        long long l2 = c > k1 ? c : k1, h2 = (c + cn) < k2 ? (c + cn) : k2;
        if (h2 > l2) iq += (h2 - l2) * b;
        if (c <= m1 && m1 < c + cn) s_med[0] = bb;
        if (c <= m2 && m2 < c + cn) s_med[1] = bb;
        c += cn;
        if (CLEAR) hist[bb] = 0u;
      }
    }
  }
  if (CONSUMERS_ONLY) named_bar_sync<BAR, THREADS>(); else __syncthreads();                                            // s_u64[0..kW) consumed, s_med written
  sum = warp_sum(sum); iq = warp_sum(iq); ge1 = warp_sum(ge1); geN = warp_sum(geN); sumsq = warp_sum(sumsq);
  mn = warp_min(mn); mx = warp_max(mx);
  if (lane == 0) {
    s_u64[0 * kW + warp] = (unsigned long long)sum; s_u64[1 * kW + warp] = (unsigned long long)iq;
    s_u64[2 * kW + warp] = (unsigned long long)ge1; s_u64[3 * kW + warp] = (unsigned long long)geN;
    s_u64[4 * kW + warp] = sumsq;
    s_i32[0 * kW + warp] = mn; s_i32[1 * kW + warp] = mx;
  }
  if (CONSUMERS_ONLY) named_bar_sync<BAR, THREADS>(); else __syncthreads();
  WalkOut w;
  w.sum = 0; w.iq_sum = 0; w.ge1 = 0; w.geN = 0; w.sumsq = 0; w.mn = INT_MAX; w.mx = INT_MIN;
  if (t == 0) {
    for (int k = 0; k < kW; ++k) {
      w.sum += (long long)s_u64[0 * kW + k]; w.iq_sum += (long long)s_u64[1 * kW + k];
      w.ge1 += (long long)s_u64[2 * kW + k]; w.geN += (long long)s_u64[3 * kW + k];
      w.sumsq += s_u64[4 * kW + k];
      w.mn = min(w.mn, s_i32[0 * kW + k]); w.mx = max(w.mx, s_i32[1 * kW + k]);
    }
  }
  w.med_lo = s_med[0];
  w.med_hi = s_med[1];
  return w;
}

__device__ __forceinline__ void write_stats(mcov_region_stats* out, const WalkOut& w) {
  mcov_region_stats r;
  r.sum = w.sum; r.sumsq = w.sumsq; r.iq_sum = w.iq_sum; r.n_ge1 = w.ge1; r.n_geN = w.geN;
  r.min = w.mn; r.max = w.mx; r.med_lo = w.med_lo; r.med_hi = w.med_hi; r.reserved = 0;
  r.flags = (w.mx >= kHistBins - 1) ? kStatOverflow : kStatValid;
  *out = r;
}

// One aligned vector of four depths -> four increments, and the running bin range of the thread.
// Plain +1 updates compile to ATOMS.POPC.INC, which the shared-memory unit sustains at a far higher
// rate than value-carrying ATOMS.ADD (measured: tools/ubench_hist.cu) -- so neighbours are
// deliberately NOT merged first.
__device__ __forceinline__ void hist_vec(uint32_t* s_hist, const int4& q, int& lo, int& hi) {
  const int b0 = hist_bin(q.x), b1 = hist_bin(q.y), b2 = hist_bin(q.z), b3 = hist_bin(q.w);
  atomicAdd(&s_hist[b0], 1u);
  atomicAdd(&s_hist[b1], 1u);
  atomicAdd(&s_hist[b2], 1u);
  atomicAdd(&s_hist[b3], 1u);
  lo = min(min(lo, b0), min(b1, min(b2, b3)));
  hi = max(max(hi, b0), max(b1, max(b2, b3)));
}

__device__ __forceinline__ void hist_partial(uint32_t* s_hist, const int4& q, int k0, int k1, int& lo, int& hi) {
  int v[4] = {q.x, q.y, q.z, q.w};
  for (int k = k0; k < k1; ++k) {
    const int b = hist_bin(v[k]);
    atomicAdd(&s_hist[b], 1u);
    lo = min(lo, b); hi = max(hi, b);
  }
}

struct RegionScratch {          // per split region of k_stats_stream; zero between runs (the CTA that walks the region resets it)
  uint32_t done;                // pieces that have merged their histogram
  uint32_t max_bin;             // highest non-empty bin
  uint32_t min_bin_inv;         // kHistBins-1 - lowest non-empty bin
  uint32_t pad;
};

// ---- small regions (<= kSmallRegion slots): one 256-thread CTA per region ---------------------------
// Hundreds of thousands of short contigs (config C3) make the fixed cost of clearing and walking
// 8192 bins dominate.  Here a first pass finds the region's min / max, only that bin range is cleared
// and walked, and the second pass (served by L1/L2) does the increments.
constexpr int kSmallThreads = 256;
constexpr int kSmallRegion = 8192;

// Runs over the retry list written by k_region_stats_warp (regions whose depth range does not fit
// a warp's window): retry[0] = count, retry[1..] = task indices.  Persistent: blocks stride over the list.
__global__ void __launch_bounds__(kSmallThreads, 6)
k_region_stats_small(StatArgs a, const uint32_t* __restrict__ retry) {
  __shared__ __align__(16) uint32_t s_hist[kHistBins];
  __shared__ unsigned long long s_u64[6 * (kSmallThreads / 32)];
  __shared__ int s_i32[4 * (kSmallThreads / 32)];
  __shared__ int s_med[2];
  const uint32_t n_retry = retry[0];
  for (uint32_t item = blockIdx.x; item < n_retry; item += gridDim.x) {
  const StatTask task = a.tasks[retry[1 + item]];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int g = task.region;
  const int pad = a.region_pad[g];
  const long long n_region = (long long)a.region_len[g] + pad;
  const int64_t s0 = task.slot, s1 = task.slot + task.n;
  const int64_t a0 = s0 & ~(int64_t)3;
  const int64_t nvec = ((s1 - a0) + 3) >> 2;
  const int4* vp = reinterpret_cast<const int4*>(a.depth + a0);
  // pass 1: min / max bin of the region
  int lo = pad > 0 ? 0 : kHistBins - 1, hi = 0;
  for (int64_t j = t; j < nvec; j += kSmallThreads) {
    int4 q = __ldg(vp + j);
    int v[4] = {q.x, q.y, q.z, q.w};
    int64_t e0 = a0 + (j << 2);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (e0 + k >= s0 && e0 + k < s1) { int b = hist_bin(v[k]); lo = min(lo, b); hi = max(hi, b); }
  }
  lo = warp_min(lo); hi = warp_max(hi);
  if (lane == 0) { s_i32[warp] = lo; s_i32[kSmallThreads / 32 + warp] = hi; }
  __syncthreads();
  lo = kHistBins - 1; hi = 0;
#pragma unroll
  for (int k = 0; k < kSmallThreads / 32; ++k) { lo = min(lo, s_i32[k]); hi = max(hi, s_i32[kSmallThreads / 32 + k]); }
  if (hi < lo) hi = lo;
  for (int b = lo + t; b <= hi; b += kSmallThreads) s_hist[b] = 0;
  __syncthreads();
  // pass 2: increments
  for (int64_t j = t; j < nvec; j += kSmallThreads) {
    int4 q = __ldg(vp + j);
    int v[4] = {q.x, q.y, q.z, q.w};
    int64_t e0 = a0 + (j << 2);
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (e0 + k >= s0 && e0 + k < s1) atomicAdd(&s_hist[hist_bin(v[k])], 1u);
  }
  if (pad > 0 && t == 0) atomicAdd(&s_hist[0], (uint32_t)pad);
  __syncthreads();
  WalkOut w = hist_walk<kSmallThreads>(s_hist, n_region, a.breadth_n, lo, hi, s_u64, s_i32, s_med);
  if (t == 0) write_stats(a.out + g, w);
  __syncthreads();
  }
}

// ---- small regions, first attempt: ONE WARP per region ------------------------------------------------
// 8 regions per CTA, each warp with a private window of kWarpBins one-value bins.  Everything is warp-synchronous
// (no block barrier).  The region is read from HBM ONCE: the window is anchored from the first 512 slots (their
// minimum less a margin; a region that begins where its contig begins starts at depth ~0, so the anchor is 0 for the
// whole-contig regions `metacov pileup` makes by default), every value is counted with its index clamped into the
// window, and the true minimum / maximum are tracked beside.  If they turn out to lie inside the window the counts are
// exact and the window is walked; if not (rare: the depth wanders by more than the window) the region is counted again
// from L2 with the window anchored at the now known minimum, and a region whose range does not fit any window is
// appended to the retry list for k_region_stats_small.
constexpr int kWarpBins = 1024;
constexpr int kWarpsPerCta = 8;
constexpr int kWarpAnchorMargin = 256;

__device__ __forceinline__ void warp_win_add1(uint32_t* win, const int v, const int wlo) {
  atomicAdd(&win[min((unsigned)(v - wlo), (unsigned)(kWarpBins - 1))], 1u);      // (a value below the window wraps and clamps too)
}
__device__ __forceinline__ void warp_win_add(uint32_t* win, const int4 q, const int wlo) {
  warp_win_add1(win, q.x, wlo); warp_win_add1(win, q.y, wlo); warp_win_add1(win, q.z, wlo); warp_win_add1(win, q.w, wlo);
}
__device__ __forceinline__ int min4(const int4 q) { return min(min(q.x, q.y), min(q.z, q.w)); }
__device__ __forceinline__ int max4(const int4 q) { return max(max(q.x, q.y), max(q.z, q.w)); }

__global__ void __launch_bounds__(kWarpsPerCta * 32)
k_region_stats_warp(StatArgs a, int64_t n_tasks, uint32_t* __restrict__ retry) {
  __shared__ __align__(16) uint32_t s_win[kWarpsPerCta][kWarpBins];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t wi = (int64_t)blockIdx.x * kWarpsPerCta + warp;
  if (wi >= n_tasks) return;
  const StatTask task = a.tasks[wi];
  const int g = task.region;
  const int pad = a.region_pad[g];
  const long long n = (long long)a.region_len[g] + pad;
  const int64_t s0 = task.slot, s1 = task.slot + task.n;
  const int64_t a0 = s0 & ~(int64_t)3;
  const int64_t nvec = ((s1 - a0) + 3) >> 2;
  const int4* vp = reinterpret_cast<const int4*>(a.depth + a0);
  uint32_t* win = s_win[warp];
  // full vectors [jf0, jf1); the first and last vector may hold slots of the neighbouring contigs
  const int64_t jf0 = (s0 != a0) ? 1 : 0, jf1 = ((a0 + (nvec << 2)) != s1) ? nvec - 1 : nvec;
  int vlo = INT_MAX, vhi = INT_MIN;                      // true range of the region's depth
  // the (at most two) partial vectors: lane 0 the head, lane 1 the tail
  int pv[4] = {0, 0, 0, 0};
  uint32_t inside = 0;                                    // which elements of pv belong to the region
  if (lane < 2 && nvec > 0 && ((lane == 0 && jf0 == 1) || (lane == 1 && jf1 == nvec - 1 && (nvec > 1 || jf0 == 0)))) {
    const int64_t j = lane == 0 ? 0 : nvec - 1;
    const int4 q = __ldg(vp + j);
    const int64_t e0 = a0 + (j << 2);
    pv[0] = q.x; pv[1] = q.y; pv[2] = q.z; pv[3] = q.w;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (e0 + k >= s0 && e0 + k < s1) { inside |= 1u << k; vlo = min(vlo, pv[k]); vhi = max(vhi, pv[k]); }
  }
  // first chunk: four independent 128-bit loads per lane in flight; the window is cleared under them
  int wlo = 0;
  {
    const int64_t j = jf0 + lane;
    const bool v0 = j < jf1, v1 = j + 32 < jf1, v2 = j + 64 < jf1, v3 = j + 96 < jf1;
    int4 q0 = make_int4(0, 0, 0, 0), q1 = q0, q2 = q0, q3 = q0;
    if (v0) q0 = __ldg(vp + j);
    if (v1) q1 = __ldg(vp + j + 32);
    if (v2) q2 = __ldg(vp + j + 64);
    if (v3) q3 = __ldg(vp + j + 96);
    uint4* w4 = reinterpret_cast<uint4*>(win);
#pragma unroll
    for (int k = 0; k < kWarpBins / 4 / 32; ++k) w4[k * 32 + lane] = make_uint4(0, 0, 0, 0);
    if (v0) { vlo = min(vlo, min4(q0)); vhi = max(vhi, max4(q0)); }
    if (v1) { vlo = min(vlo, min4(q1)); vhi = max(vhi, max4(q1)); }
    if (v2) { vlo = min(vlo, min4(q2)); vhi = max(vhi, max4(q2)); }
    if (v3) { vlo = min(vlo, min4(q3)); vhi = max(vhi, max4(q3)); }
    const int est = warp_min(vlo);
    wlo = (pad > 0 || est == INT_MAX) ? 0 : max(0, est - kWarpAnchorMargin);       // pad > 0: zeros are counted in bin 0
    __syncwarp();
    if (v0) warp_win_add(win, q0, wlo);
    if (v1) warp_win_add(win, q1, wlo);
    if (v2) warp_win_add(win, q2, wlo);
    if (v3) warp_win_add(win, q3, wlo);
#pragma unroll
    for (int k = 0; k < 4; ++k) if (inside & (1u << k)) warp_win_add1(win, pv[k], wlo);
  }
  for (int64_t jb = jf0 + 128; jb < jf1; jb += 128) {
    const int64_t j = jb + lane;
    const bool v0 = j < jf1, v1 = j + 32 < jf1, v2 = j + 64 < jf1, v3 = j + 96 < jf1;
    int4 q0 = make_int4(0, 0, 0, 0), q1 = q0, q2 = q0, q3 = q0;
    if (v0) q0 = __ldg(vp + j);
    if (v1) q1 = __ldg(vp + j + 32);
    if (v2) q2 = __ldg(vp + j + 64);
    if (v3) q3 = __ldg(vp + j + 96);
    if (v0) { vlo = min(vlo, min4(q0)); vhi = max(vhi, max4(q0)); warp_win_add(win, q0, wlo); }
    if (v1) { vlo = min(vlo, min4(q1)); vhi = max(vhi, max4(q1)); warp_win_add(win, q1, wlo); }
    if (v2) { vlo = min(vlo, min4(q2)); vhi = max(vhi, max4(q2)); warp_win_add(win, q2, wlo); }
    if (v3) { vlo = min(vlo, min4(q3)); vhi = max(vhi, max4(q3)); warp_win_add(win, q3, wlo); }
  }
  vlo = warp_min(vlo); vhi = warp_max(vhi);
  int lo, hi;
  if (vlo == INT_MAX) { lo = kHistBins - 1; hi = 0; }    // no slot inside the contig
  else { lo = hist_bin(vlo); hi = hist_bin(vhi); }       // hist_bin is monotone
  if (pad > 0) lo = 0;
  if (hi < lo) hi = lo;
  const int nb = hi - lo + 1;
  if (nb > kWarpBins || hi >= kHistBins - 1 || vlo < 0) {       // does not fit (or leaves the bin range): retry path
    if (lane == 0) { uint32_t k = atomicAdd(retry, 1u); retry[1 + k] = (uint32_t)wi; }
    return;
  }
  if (pad > 0 && lane == 0) atomicAdd(&win[0], (uint32_t)pad);      // pad > 0 => wlo == 0
  if (lo < wlo || hi > wlo + kWarpBins - 1) {
    // the guess missed: count again (served by L1/L2) with the window anchored at the minimum
    __syncwarp();
    uint4* w4 = reinterpret_cast<uint4*>(win);
#pragma unroll
    for (int k = 0; k < kWarpBins / 4 / 32; ++k) w4[k * 32 + lane] = make_uint4(0, 0, 0, 0);
    wlo = lo;
    __syncwarp();
    for (int64_t j = lane; j < nvec; j += 32) {
      int4 q = __ldg(vp + j);
      int v[4] = {q.x, q.y, q.z, q.w};
      int64_t e0 = a0 + (j << 2);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (e0 + k >= s0 && e0 + k < s1) atomicAdd(&win[v[k] - lo], 1u);
    }
    if (pad > 0 && lane == 0) atomicAdd(&win[0], (uint32_t)pad);
  }
  __syncwarp();
  win += lo - wlo;                                        // bin b of the walk below holds depth lo + b
  // walk the window: each lane a contiguous run of bins
  const long long k1 = n / 4, k2 = n - n / 4, m1 = (n - 1) / 2, m2 = n / 2;
  const int per = (nb + 31) / 32;
  const int b0 = lane * per, b1 = min(b0 + per, nb);
  unsigned long long local = 0;
  for (int b = b0; b < b1; ++b) local += win[b];
  unsigned long long x = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  long long c = (long long)(x - local);
  long long sum = 0, iq = 0, ge1 = 0, geN = 0;
  unsigned long long sumsq = 0;
  int mn = INT_MAX, mx = INT_MIN, ml = -1, mh = -1;
  for (int bb = b0; bb < b1; ++bb) {
    long long cn = win[bb];
    if (cn) {
      long long b = bb + lo;
      sum += b * cn;
      sumsq += (unsigned long long)(b * b) * (unsigned long long)cn;
      ge1 += b >= 1 ? cn : 0;
      geN += b >= a.breadth_n ? cn : 0;
      mn = min(mn, (int)b); mx = max(mx, (int)b);
      long long l2 = c > k1 ? c : k1, h2 = (c + cn) < k2 ? (c + cn) : k2;
      if (h2 > l2) iq += (h2 - l2) * b;
      if (c <= m1 && m1 < c + cn) ml = (int)b;
      if (c <= m2 && m2 < c + cn) mh = (int)b;
      c += cn;
    }
  }
  sum = warp_sum(sum); iq = warp_sum(iq); ge1 = warp_sum(ge1); geN = warp_sum(geN); sumsq = warp_sum(sumsq);
  mn = warp_min(mn); mx = warp_max(mx); ml = warp_max(ml); mh = warp_max(mh);
  if (lane == 0) {
    WalkOut w;
    w.sum = sum; w.iq_sum = iq; w.ge1 = ge1; w.geN = geN; w.sumsq = sumsq; w.mn = mn; w.mx = mx; w.med_lo = ml; w.med_hi = mh;
    write_stats(a.out + g, w);
  }
}

// ---- regions cut across devices (SURVEY.md 8(e)): partial histograms, merged, then finished -------
// When a contig is split between ranks, a region that straddles the cut cannot be finished from
// 64-byte records: the median and the interquartile sum need the merged multiset.  Each rank adds
// the exact counting histogram of ITS part to a [g][kHistBins] table (k_region_hist), the tables are
// summed across ranks (one all-reduce over NVLink) and k_hist_finish walks the merged histogram --
// the same hist_walk as the single-device kernels, so the records are identical.
struct HistTask {
  int64_t slot;     // first slot of the chunk
  int32_t n;        // slots in the chunk
  int32_t region;
  int32_t pad;      // zeros to add to bin 0 (positions beyond the contig end; first chunk of the region only)
  int32_t reserved;
};

__global__ void __launch_bounds__(kStatThreads, 4)
k_region_hist(const int32_t* __restrict__ depth, const HistTask* __restrict__ tasks, uint32_t* __restrict__ hist_out) {
  __shared__ __align__(16) uint32_t s_hist[kHistBins];
  __shared__ int s_rng[2 * (kStatThreads / 32)];
  const HistTask task = tasks[blockIdx.x];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  {
    uint4* h4 = reinterpret_cast<uint4*>(s_hist);
    for (int k = t; k < kHistBins / 4; k += kStatThreads) h4[k] = make_uint4(0, 0, 0, 0);
  }
  __syncthreads();
  const int64_t s0 = task.slot, s1 = task.slot + task.n;
  const int64_t a0 = s0 & ~(int64_t)3;
  const int64_t nvec = ((s1 - a0) + 3) >> 2;
  const int4* vp = reinterpret_cast<const int4*>(depth + a0);
  const int head = (int)(s0 - a0), tail = (int)((a0 + (nvec << 2)) - s1);
  const int64_t jf0 = head ? 1 : 0, jf1 = nvec - (tail ? 1 : 0);
  int lo = kHistBins, hi = -1;
  for (int64_t j = jf0 + t; j < jf1; j += kStatThreads) hist_vec(s_hist, __ldcs(vp + j), lo, hi);
  if (nvec > 0) {
    if (nvec == 1) { if (t == 0 && (head || tail)) hist_partial(s_hist, __ldcs(vp), head, 4 - tail, lo, hi); }
    else {
      if (t == 0 && head) hist_partial(s_hist, __ldcs(vp), head, 4, lo, hi);
      if (t == 32 && tail) hist_partial(s_hist, __ldcs(vp + nvec - 1), 0, 4 - tail, lo, hi);
    }
  }
  if (t == 0 && task.pad > 0) { atomicAdd(&s_hist[0], (uint32_t)task.pad); lo = 0; hi = max(hi, 0); }
  lo = warp_min(lo); hi = warp_max(hi);
  if (lane == 0) { s_rng[warp] = lo; s_rng[kStatThreads / 32 + warp] = hi; }
  __syncthreads();
  lo = kHistBins; hi = -1;
#pragma unroll
  for (int k = 0; k < kStatThreads / 32; ++k) { lo = min(lo, s_rng[k]); hi = max(hi, s_rng[kStatThreads / 32 + k]); }
  uint32_t* gh = hist_out + (int64_t)task.region * kHistBins;
  for (int b = lo + t; b <= hi; b += kStatThreads) {
    const uint32_t c = s_hist[b];
    if (c) atomicAdd(gh + b, c);
  }
}

// One CTA per region: statistics record from a complete counting histogram in global memory.
__global__ void __launch_bounds__(kStatThreads, 4)
k_hist_finish(const uint32_t* __restrict__ hist, mcov_region_stats* __restrict__ out, int32_t breadth_n) {
  __shared__ __align__(16) uint32_t s_hist[kHistBins];
  __shared__ unsigned long long s_u64[6 * (kStatThreads / 32)];
  __shared__ int s_i32[4 * (kStatThreads / 32)];
  __shared__ int s_med[2];
  __shared__ unsigned long long s_n;
  const int g = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const uint4* src = reinterpret_cast<const uint4*>(hist + (int64_t)g * kHistBins);
  unsigned long long n = 0;
  for (int k = t; k < kHistBins / 4; k += kStatThreads) {
    const uint4 v = src[k];
    reinterpret_cast<uint4*>(s_hist)[k] = v;
    n += (unsigned long long)v.x + v.y + v.z + v.w;
  }
  n = warp_sum(n);
  if (lane == 0) s_u64[warp] = n;
  if (t == 0) { s_med[0] = 0; s_med[1] = 0; }
  __syncthreads();
  if (t == 0) {
    unsigned long long tot = 0;
    for (int k = 0; k < kStatThreads / 32; ++k) tot += s_u64[k];
    s_n = tot;
  }
  __syncthreads();
  const long long total = (long long)s_n;
  __syncthreads();                                    // s_u64 is reused by hist_walk
  if (total == 0) {                                   // empty region: an all-zero record
    if (t == 0) { mcov_region_stats r; memset(&r, 0, sizeof(r)); out[g] = r; }
    return;
  }
  WalkOut w = hist_walk<kStatThreads>(s_hist, total, breadth_n, 0, kHistBins - 1, s_u64, s_i32, s_med);
  if (t == 0) write_stats(out + g, w);
}

// Fixed-window mean depth: one warp per window.
__global__ void k_window_sums(const int32_t* __restrict__ depth, const int64_t* __restrict__ win_slot,
                              const int32_t* __restrict__ win_n, int64_t n_win, long long* __restrict__ out) {
  int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (w >= n_win) return;
  const int32_t* p = depth + win_slot[w];
  int n = win_n[w];
  long long s = 0;
  for (int k = lane; k < n; k += 32) s += p[k];
  s = warp_sum(s);
  if (lane == 0) out[w] = s;
}

}  // namespace mcov
