// k_compare.cuh -- samples compared position by position through their allele signatures: one byte a slot made from a
// file's A / C / G / T counters with the rules of k_allele_rules.cuh (include/metacov_b200.h: mcov_allele_signature,
// mcov_compare_run, mcov_compare_sites; oracle/compare.py restates them).
//
//   k_allele_signature    one thread per slot (four in flight): 16 B of counters in, the signature byte out
//   k_compare_chunks      one warp per (chunk, pair), chunk-major: the pair's partial record over the chunk
//   k_compare_combine     one warp per (pair, region): the partials of the region's chunks, then a shuffle tree
//   k_compare_site_count  one CTA per (tile, pair), tile-major: the pair's sites in the tile
//   k_compare_site_write  one CTA per (tile, pair) that holds a site: its sites in slot order at the scanned offset
//
// Signature byte: 0x80 covered, bits 4-5 the consensus (0-3 = A C G T), bits 0-3 the present mask; 0 where not covered.
// The pair kernels read signatures as 4-byte words (n_slots is a multiple of 4, so is every contig's first slot) and
// count four positions a word with byte-wise masks and __popc; the bytes of a word outside a chunk are masked to 0,
// i.e. uncovered.  Chunk-major (tile-major) work items put the pairs of one chunk side by side, so the warps that run
// at one time share the chunk's signature bytes through L2: for S samples DRAM sees about S bytes a slot, not 2 per
// slot and pair.
#pragma once
#include <stdint.h>
#include "common.cuh"
#include "k_allele_rules.cuh"

namespace mcov {

constexpr int kSigThreads = 256;
constexpr int kSigUnroll = 4;            // loads in flight a thread
constexpr int kCmpThreads = 256;         // region kernels: 8 warps a CTA
constexpr int kCmpWarps = kCmpThreads / 32;
constexpr int kCmpChunk = 8192;          // positions a chunk (64 words a lane)
constexpr int kCmpTile = 8192;           // slots a site tile (8 words a thread)
constexpr int kCmpTileThreads = 256;
constexpr int kCmpTileWords = kCmpTile / 4;
constexpr int kCmpTileContigs = kCmpTile / 4 + 1;   // a contig spans at least 4 slots

struct CmpPart { uint32_t covered_a, covered_b, compared, con_snp, pop_snp, pad; };   // a chunk's counts for one pair

__device__ __forceinline__ uint32_t allele_signature(const uint4 c, const AlleleParams& P) {
  const uint64_t n = (uint64_t)c.x + c.y + c.z + c.w;
  if (n < P.min_cov) return 0;
  const AlRules ru = allele_rules(c, (double)n, P);
  return 0x80u | (ru.best << 4) | ru.mask;
}

__global__ void __launch_bounds__(kSigThreads)
k_allele_signature(const uint4* __restrict__ cnt, int64_t n_slots, AlleleParams P, uint8_t* __restrict__ out) {
  const int64_t step = (int64_t)gridDim.x * kSigThreads * kSigUnroll;
  for (int64_t s0 = (int64_t)blockIdx.x * kSigThreads * kSigUnroll + threadIdx.x; s0 < n_slots; s0 += step) {
    uint4 c[kSigUnroll];
#pragma unroll
    for (int k = 0; k < kSigUnroll; ++k) {
      const int64_t s = s0 + k * kSigThreads;
      c[k] = s < n_slots ? __ldg(cnt + s) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int k = 0; k < kSigUnroll; ++k) {
      const int64_t s = s0 + k * kSigThreads;
      if (s < n_slots) out[s] = (uint8_t)allele_signature(c[k], P);
    }
  }
}

constexpr uint32_t kSigLow = 0x01010101u;

// The allele set of each of four signature bytes: the present mask with the consensus' bit added.
__device__ __forceinline__ uint32_t sig_sets(const uint32_t s) {
  const uint32_t c0 = (s >> 4) & kSigLow, c1 = (s >> 5) & kSigLow;
  const uint32_t n0 = c0 ^ kSigLow, n1 = c1 ^ kSigLow;
  return (s & 0x0F0F0F0Fu) | (n1 & n0) | ((n1 & c0) << 1) | ((c1 & n0) << 2) | ((c1 & c0) << 3);
}

// Bit 0 of each byte: compared (covered in both), con_snp, pop_snp, for four positions.
struct CmpFlags { uint32_t compared, con, pop; };

__device__ __forceinline__ CmpFlags cmp_flags(const uint32_t a, const uint32_t b) {
  CmpFlags f;
  f.compared = (a & b & 0x80808080u) >> 7;
  const uint32_t dc = (a ^ b) >> 4;                             // consensus bits 0-1 of each byte (bits 2-3: the flag's)
  f.con = f.compared & (dc | (dc >> 1));
  const uint32_t x = sig_sets(a) & sig_sets(b);
  const uint32_t y = x | (x >> 2);
  f.pop = f.compared & ~(y | (y >> 1));
  f.con &= kSigLow; f.pop &= kSigLow;
  return f;
}

struct CmpRegionArgs {
  const uint8_t* const* sig;     // [2 * n_pairs] the signatures of sample a and sample b of each pair
  int64_t n_pairs;
  const AlChunk* chunks; int64_t n_chunks;
  CmpPart* part;                 // [n_chunks * n_pairs], chunk-major
};

__global__ void __launch_bounds__(kCmpThreads)
k_compare_chunks(CmpRegionArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kCmpWarps;
  const int64_t items = a.n_chunks * a.n_pairs;
  for (int64_t w = (int64_t)blockIdx.x * kCmpWarps + (threadIdx.x >> 5); w < items; w += nw) {
    const int64_t chunk = w / a.n_pairs, pair = w - chunk * a.n_pairs;
    const AlChunk ch = a.chunks[chunk];
    const uint32_t* pa = reinterpret_cast<const uint32_t*>(a.sig[2 * pair]);
    const uint32_t* pb = reinterpret_cast<const uint32_t*>(a.sig[2 * pair + 1]);
    const int64_t lo = ch.slot, hi = ch.slot + ch.n;
    const int64_t q0 = lo >> 2, q1 = (hi + 3) >> 2;
    uint32_t cov_a = 0, cov_b = 0, cmp = 0, con = 0, pop = 0;
    // four words in flight a lane; the head and tail words are masked to the chunk's bytes
    for (int64_t q = q0 + lane; q < q1; q += 128) {
      uint32_t va[4], vb[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t qq = q + 32 * u;
        va[u] = qq < q1 ? __ldg(pa + qq) : 0u;
        vb[u] = qq < q1 ? __ldg(pb + qq) : 0u;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int64_t s = 4 * (q + 32 * u);
        uint32_t m = 0xFFFFFFFFu;
        if (s < lo) m <<= 8 * (int)(lo - s);                                  // (lo - s <= 3)
        if (s + 4 > hi) m = s >= hi ? 0u : m & (0xFFFFFFFFu >> (8 * (int)(s + 4 - hi)));
        const uint32_t x = va[u] & m, y = vb[u] & m;
        const CmpFlags f = cmp_flags(x, y);
        cov_a += __popc(x & 0x80808080u); cov_b += __popc(y & 0x80808080u);
        cmp += __popc(f.compared); con += __popc(f.con); pop += __popc(f.pop);
      }
    }
    const long long ca = warp_sum_i64(cov_a), cb = warp_sum_i64(cov_b), cm = warp_sum_i64(cmp);
    const long long cs = warp_sum_i64(con), ps = warp_sum_i64(pop);
    if (lane == 0) {
      CmpPart p;
      p.covered_a = (uint32_t)ca; p.covered_b = (uint32_t)cb; p.compared = (uint32_t)cm;
      p.con_snp = (uint32_t)cs; p.pop_snp = (uint32_t)ps; p.pad = 0;
      a.part[w] = p;
    }
  }
}

// Record (pair, region r) = out[pair * g + r] from the partials of the region's chunks [first[r], first[r + 1]).
__global__ void __launch_bounds__(kCmpThreads)
k_compare_combine(const CmpPart* __restrict__ part, int64_t n_pairs, const int64_t* __restrict__ first,
                  const int64_t* __restrict__ length, int64_t g, mcov_compare_stats* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kCmpWarps;
  for (int64_t w = (int64_t)blockIdx.x * kCmpWarps + (threadIdx.x >> 5); w < g * n_pairs; w += nw) {
    const int64_t pair = w / g, r = w - pair * g;
    long long ca = 0, cb = 0, cm = 0, cs = 0, ps = 0;
    for (int64_t k = first[r] + lane; k < first[r + 1]; k += 32) {
      const CmpPart p = part[k * n_pairs + pair];
      ca += p.covered_a; cb += p.covered_b; cm += p.compared; cs += p.con_snp; ps += p.pop_snp;
    }
    ca = warp_sum_i64(ca); cb = warp_sum_i64(cb); cm = warp_sum_i64(cm); cs = warp_sum_i64(cs); ps = warp_sum_i64(ps);
    if (lane == 0) {
      mcov_compare_stats s;
      s.length = length[r]; s.covered_a = ca; s.covered_b = cb; s.compared = cm; s.con_snp = cs; s.pop_snp = ps;
      out[w] = s;
    }
  }
}

struct CmpSiteArgs {
  const uint8_t* const* sig;     // [2 * n_pairs] as CmpRegionArgs
  int64_t n_pairs, n_slots, n_tiles;
  const int64_t* contig_off; int32_t n_contigs;
  int64_t* tile_n;               // [n_pairs * n_tiles] sites of (pair, tile), pair-major (written by the count pass)
  const int64_t* tile_incl;      // their inclusive scan (read by the write pass): offsets in (pair, slot) order
  mcov_compare_site* sites;
};

__global__ void __launch_bounds__(kCmpTileThreads)
k_compare_site_count(CmpSiteArgs a) {
  __shared__ int s_w[kCmpTileThreads / 32];
  const int64_t n_words = a.n_slots >> 2;
  for (int64_t j = blockIdx.x; j < a.n_tiles * a.n_pairs; j += gridDim.x) {
    const int64_t t = j / a.n_pairs, pair = j - t * a.n_pairs;
    const uint32_t* pa = reinterpret_cast<const uint32_t*>(a.sig[2 * pair]);
    const uint32_t* pb = reinterpret_cast<const uint32_t*>(a.sig[2 * pair + 1]);
    const int64_t q0 = t * kCmpTileWords;
    int n = 0;
#pragma unroll
    for (int k = 0; k < kCmpTileWords / kCmpTileThreads; ++k) {
      const int64_t q = q0 + k * kCmpTileThreads + threadIdx.x;
      if (q < n_words) n += __popc(cmp_flags(__ldg(pa + q), __ldg(pb + q)).con);
    }
    store_tile_count<kCmpTileThreads>(n, s_w, a.tile_n, pair * a.n_tiles + t, threadIdx.x);
  }
}

// Thread k takes the tile's words [8k, 8k + 8), so that one block scan of the per-thread site counts gives every site
// its place in slot order.  The contigs the tile touches are found with one search over the offset table a tile; a
// site's contig is then looked up among them in shared memory.
__global__ void __launch_bounds__(kCmpTileThreads)
k_compare_site_write(CmpSiteArgs a) {
  constexpr int kPer = kCmpTileWords / kCmpTileThreads;
  __shared__ int64_t s_off[kCmpTileContigs];
  __shared__ int s_w[kCmpTileThreads / 32];
  __shared__ int32_t s_c[2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t n_words = a.n_slots >> 2;
  for (int64_t j = blockIdx.x; j < a.n_tiles * a.n_pairs; j += gridDim.x) {
    const int64_t t = j / a.n_pairs, pair = j - t * a.n_pairs;
    const int64_t nt = a.tile_n[pair * a.n_tiles + t];
    if (nt == 0) continue;                                   // (uniform over the CTA) tiles without a site are not read again
    const int64_t base = a.tile_incl[pair * a.n_tiles + t] - nt;
    const uint32_t* pa = reinterpret_cast<const uint32_t*>(a.sig[2 * pair]);
    const uint32_t* pb = reinterpret_cast<const uint32_t*>(a.sig[2 * pair + 1]);
    const int64_t s0 = t * kCmpTile, s1 = s0 + kCmpTile < a.n_slots ? s0 + kCmpTile : a.n_slots;
    if (threadIdx.x < 2) {
      // contig of the tile's first (thread 0) and last (thread 1) slot
      s_c[threadIdx.x] = contig_of(a.contig_off, a.n_contigs, threadIdx.x == 0 ? s0 : s1 - 1);
    }
    __syncthreads();
    const int32_t c0 = s_c[0], nc = s_c[1] - s_c[0] + 1;
    for (int i = threadIdx.x; i < nc; i += kCmpTileThreads) s_off[i] = __ldg(a.contig_off + c0 + i);
    const int64_t q0 = s0 / 4 + (int64_t)threadIdx.x * kPer;
    uint32_t va[kPer], vb[kPer], fl[kPer];
    int n = 0;
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int64_t q = q0 + k;
      va[k] = q < n_words ? __ldg(pa + q) : 0u;
      vb[k] = q < n_words ? __ldg(pb + q) : 0u;
      const CmpFlags f = cmp_flags(va[k], vb[k]);
      fl[k] = f.con | (f.pop << 1);
      n += __popc(f.con);
    }
    // exclusive block scan of n
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_w[warp] = incl;
    __syncthreads();
    int before = incl - n;
#pragma unroll
    for (int w = 0; w < kCmpTileThreads / 32; ++w) before += w < warp ? s_w[w] : 0;
    int64_t at = base + before;
    for (int k = 0; k < kPer; ++k) {
      if (fl[k] == 0) continue;
      const int64_t q = q0 + k;
      // the word's contig (every word lies in one contig: contigs start on 4-slot boundaries)
      int32_t lo = 0, hi = nc - 1;
      while (lo < hi) { const int32_t m = (lo + hi + 1) >> 1; if (s_off[m] <= 4 * q) lo = m; else hi = m - 1; }
      for (int b = 0; b < 4; ++b) {
        const uint32_t kind = (fl[k] >> (8 * b)) & 3u;
        if (!(kind & 1u)) continue;
        mcov_compare_site st;
        st.pair = (int32_t)pair; st.tid = c0 + lo; st.pos = (int32_t)(4 * q + b - s_off[lo]);
        st.sig_a = (uint8_t)(va[k] >> (8 * b)); st.sig_b = (uint8_t)(vb[k] >> (8 * b)); st.kind = (uint8_t)kind; st.pad = 0;
        a.sites[at++] = st;
      }
    }
    __syncthreads();
  }
}

}  // namespace mcov
