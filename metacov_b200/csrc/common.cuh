// common.cuh -- shared device helpers and POD types for the coverage kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "metacov_b200.h"

namespace mcov {

constexpr int kStatValidBit = 1;     // mcov_region_stats.flags bit0: record valid
constexpr int kStatOverflowBit = 2;  // bit1: depth left the counting histogram, radix path used

// BAM CIGAR ops that consume reference: M(0) D(2) N(3) =(7) X(8)
// (htslib bam_cigar_type bit 1; SURVEY.md Appendix A-4).
constexpr uint32_t kRefConsumeMask = 0x18Du;

__host__ __device__ __forceinline__ uint32_t cigar_ref_len(uint32_t op) {
  return ((kRefConsumeMask >> (op & 15u)) & 1u) ? (op >> 4) : 0u;
}
// acc + cigar_ref_len(op), arranged for the pipes of the SM: the integer ALU pipe (logic, shifts,
// compares, selects: 16 lanes per clock) is what bounds the prep kernels (ncu: 72 % busy, FMA pipe
// 12 %), so the length extraction and the conditional add are done as IMAD.HI + IMAD on the FMA
// pipe; the mask lookup is one wrap-around shift of the table replicated into both half words.
__device__ __forceinline__ uint32_t cigar_ref_len_add(uint32_t acc, uint32_t op) {
  const uint32_t bit = ((kRefConsumeMask * 0x10001u) >> (op & 31u)) & 1u;
  return __umulhi(op, 0x10000000u) * bit + acc;
}

// Counters of one pass, device resident (mirrored to mcov_pass_info).
struct PassCounters {
  unsigned long long n_reads;
  unsigned long long n_pass;
  unsigned long long aligned_bases;
  int max_depth_seen;
  int cap_metric;
  int unsorted;          // set to 1 if any adjacent pair of reads is out of (tid,pos) order
  unsigned int ticket;   // dynamic tile id for the scan kernel
  unsigned int ticket2;  // dynamic tile tickets of the fused tile kernel (beyond the 3 static rounds)
  unsigned int max_span; // max clipped span of a near read (fused path)
  unsigned int n_far;    // reads whose span exceeds the near window (fused path)
  unsigned int n_heavy;  // tiles holding >= heavy_min reads (fused path: scheduled first)
  unsigned int cap_contigs;  // contigs replayed under htslib's max_depth cap (k_cap_replay)
  unsigned int cap_unreplayed;  // streamed pass: the cap can fire in a batch (a contig's reads are not all on the device)
  unsigned int far_overflow;    // streamed pass: a batch had more long-span reads than the bucket list holds
};

// pysam __advance_samtools predicate + bam_plp_push's own UNMAP drop
// (SURVEY.md Appendix A-2).
__device__ __forceinline__ bool read_passes(uint32_t flag, uint32_t mapq, const mcov_filter& f) {
  if (flag & f.flag_filter) return false;
  if (f.flag_require && !(flag & f.flag_require)) return false;
  if (mapq < f.min_mapq) return false;
  if (f.ignore_orphans && (flag & 0x1u) && !(flag & 0x2u)) return false;
  if (flag & 0x4u) return false;
  return true;
}

__device__ __forceinline__ int4 ld_stream_int4(const int4* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
// coherent variant for data the same kernel rewrites in place (no .nc)
__device__ __forceinline__ int4 ld_na_int4(const int4* p) {
  int4 r;
  asm volatile("ld.global.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ uint4 ld_stream_uint4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_int4(int4* p, const int4& v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Look-back status words carry state and value in ONE 64-bit word, so a relaxed (L1-bypassing)
// load/store pair is enough: nothing else has to be ordered with it.  (acquire/release at gpu scope
// would make ptxas emit CCTL.IVALL / MEMBAR around every poll.)
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization
// attribute may start while its predecessor in the stream drains; pdl_wait() blocks until the predecessor
// has completed and its writes are visible (a no-op for a normal launch), pdl_launch_dependents() lets the
// successor's CTAs take free slots from now on.  Removes the drain/launch/ramp gap between the short
// kernels of one step.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- TMA bulk copies behind mbarriers (sm_90+; SASS: UBLKCP / SYNCS) ----------------------------
// The streaming kernels stage their inputs with cp.async.bulk: ONE elected thread issues a
// multi-kilobyte global -> shared copy that completes on an mbarrier (complete_tx::bytes); the
// consumer threads wait on the barrier's phase parity and read shared memory.  No register is held
// while the copy is in flight and no per-thread load instruction is issued for the data.
// Addresses and sizes must be multiples of 16 bytes.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(arrivals) : "memory");
}
// makes the initialised barriers visible to the async proxy (the TMA unit); follow with a CTA barrier
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
// Producer-side wait: a producer is usually several stages ahead and would otherwise spin on the
// "empty" barrier -- a single thread, but every retry costs its scheduler a full issue slot (ncu: 6-12 %
// of the executed instructions of the first TMA kernels).  try_wait with a suspend-time hint parks the
// thread in hardware; the sleep between retries bounds what is left.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  for (;;) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(20000u) : "memory");
    if (ok) return;
    __nanosleep(256);
  }
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// same with an L2 eviction-priority hint (streams that are read once: evict_first)
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_1d_hint(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol) : "memory");
}
// named barrier over a subset of the CTA's warps (the consumer warps of a warp-specialised kernel)
template <int ID, int THREADS>
__device__ __forceinline__ void named_bar_sync() { asm volatile("bar.sync %0, %1;" :: "n"(ID), "n"(THREADS) : "memory"); }

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Reference length of one read whose ops are p[0, cnt), computed by a whole
// warp with 128-bit loads where alignment allows (long-read path, config C5:
// thousands of ops per read, the CIGAR stream is the dominant HBM traffic).
__device__ __forceinline__ unsigned long long warp_cigar_reflen(const uint32_t* __restrict__ p, uint32_t cnt, int lane) {
  unsigned long long acc = 0;
  // head: ops before the first 16-byte aligned one (< 4)
  uint32_t head = (uint32_t)((16u - (uint32_t)(reinterpret_cast<uintptr_t>(p) & 15u)) & 15u) >> 2;
  if (head > cnt) head = cnt;
  if ((uint32_t)lane < head) acc += cigar_ref_len(__ldg(p + lane));
  const uint32_t nvec = (cnt - head) >> 2;
  const uint4* v = reinterpret_cast<const uint4*>(p + head);
  uint32_t j = lane;
  // 4 independent 512-byte warp loads in flight
  for (; j + 96u < nvec; j += 128u) {
    uint4 q0 = ld_stream_uint4(v + j), q1 = ld_stream_uint4(v + j + 32u);
    uint4 q2 = ld_stream_uint4(v + j + 64u), q3 = ld_stream_uint4(v + j + 96u);
    acc += cigar_ref_len(q0.x) + cigar_ref_len(q0.y) + cigar_ref_len(q0.z) + cigar_ref_len(q0.w);
    acc += cigar_ref_len(q1.x) + cigar_ref_len(q1.y) + cigar_ref_len(q1.z) + cigar_ref_len(q1.w);
    acc += cigar_ref_len(q2.x) + cigar_ref_len(q2.y) + cigar_ref_len(q2.z) + cigar_ref_len(q2.w);
    acc += cigar_ref_len(q3.x) + cigar_ref_len(q3.y) + cigar_ref_len(q3.z) + cigar_ref_len(q3.w);
  }
  for (; j < nvec; j += 32u) {
    uint4 q = ld_stream_uint4(v + j);
    acc += cigar_ref_len(q.x) + cigar_ref_len(q.y) + cigar_ref_len(q.z) + cigar_ref_len(q.w);
  }
  const uint32_t k = head + (nvec << 2);      // tail (< 4 ops)
  if (k + (uint32_t)lane < cnt) acc += cigar_ref_len(__ldg(p + k + lane));
  return warp_sum(acc);
}

}  // namespace mcov
