// k_allele_rules.cuh -- the allele rules at one position (covered, present mask, consensus), the parameters they take
// and the pieces the allele kernels (k_alleles.cuh) and the compare kernels (k_compare.cuh) share.  The rules are
// restated in oracle/alleles.py.
#pragma once
#include <stdint.h>
#include "common.cuh"

namespace mcov {

struct AlleleParams {
  uint32_t min_cov, min_count;
  double min_freq;
  int32_t use_ref;
};

struct AlChunk { int64_t slot; int64_t n; };   // n positions from slot, all inside one contig

// The present mask (bit b: allele b present) and the consensus (0-3 = A C G T) of a covered position with counts c and
// dn their sum as a double.  These are the rules every allele and compare kernel shares (k_compare.cuh's signature is
// made of them).
struct AlRules { uint32_t mask, best; };

__device__ __forceinline__ AlRules allele_rules(const uint4 c, const double dn, const AlleleParams& P) {
  const double thr = __dmul_rn(P.min_freq, dn);
  const uint32_t v[4] = {c.x, c.y, c.z, c.w};
  uint32_t mask = 0, best = 0;
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    if (v[b] >= P.min_count && (double)v[b] >= thr) mask |= 1u << b;
    if (b > 0 && v[b] > v[best]) best = b;
  }
  return {mask, best};
}

__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

// A site tile's count: the sum of every thread's n over a CTA of kThreads, stored by thread 0 to tile_n[i] (s_w:
// kThreads / 32 ints of shared memory).  Every thread calls it; it ends with a barrier, so s_w may be used again.  tx is
// the kernel's threadIdx.x: read in the kernel, it keeps the range the kernel's __launch_bounds__ give it, which the
// kernel's slot arithmetic relies on (a read in here would not, and the kernel compiles to other instructions).
template <int kThreads>
__device__ __forceinline__ void store_tile_count(int n, int* s_w, int64_t* tile_n, int64_t i, const unsigned tx) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((tx & 31) == 0) s_w[tx >> 5] = n;
  __syncthreads();
  if (tx == 0) {
    int64_t tot = 0;
    for (int w = 0; w < kThreads / 32; ++w) tot += s_w[w];
    tile_n[i] = tot;
  }
  __syncthreads();
}

// The contig of slot s: the last contig whose offset is <= s.
__device__ __forceinline__ int32_t contig_of(const int64_t* contig_off, int32_t n_contigs, int64_t s) {
  int32_t lo = 0, hi = n_contigs - 1;
  while (lo < hi) { const int32_t m = (lo + hi + 1) >> 1; if (__ldg(contig_off + m) <= s) lo = m; else hi = m - 1; }
  return lo;
}

}  // namespace mcov
