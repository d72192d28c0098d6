// k_allele_rules.cuh -- the allele rules at one position (covered, present mask, consensus), the parameters they take
// and the pieces the allele kernels (k_alleles.cuh) and the compare kernels (k_compare.cuh) share.  They are restated
// in oracle/alleles.py.
#pragma once
#include <stdint.h>
#include <string>
#include "common.cuh"

namespace mcov {

struct AlleleParams {
  uint32_t min_cov, min_count;
  double min_freq;
  int32_t use_ref;
};

// Host helpers of the allele calls (alleles.cu), shared with the compare calls (compare.cu): the error text and code;
// the checked parameters or an error (MCOV_ERR_STATE without counts for the contig table); the grid of a grid-stride
// kernel over `items` work items, `per` of them a CTA.
int al_fail(mcov_ctx* ctx, int code, const std::string& what, cudaError_t e = cudaSuccess);
int al_check(mcov_ctx* ctx, const mcov_allele_params* p, AlleleParams* out, const char* who);
unsigned al_grid(const mcov_ctx* ctx, int64_t items, int per);

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

}  // namespace mcov
