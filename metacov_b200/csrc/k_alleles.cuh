// k_alleles.cuh -- allele rules at every reference position from the A / C / G / T counters of mcov_base_counts
// ([slot][A C G T] uint32, k_basecount.cuh) and the reference store (one byte a slot, 0-3 = A C G T, 4 = unknown):
// coverage, present alleles, consensus, the per-site nucleotide diversity pi_p and the site kinds SNV / SUB / POPSUB
// (include/metacov_b200.h: mcov_allele_stats_run, mcov_allele_sites; oracle/alleles.py restates them).
//
//   k_ref_encode         ASCII reference of one contig -> codes in its slots
//   k_allele_chunks      one warp per chunk of kAlChunk positions of a region: the chunk's partial record
//   k_allele_combine     one warp per region: its chunks' partials, lanes strided over them, then a shuffle tree
//   k_allele_site_count  one CTA per tile of kAlTile slots: sites in the tile
//   k_allele_site_write  one CTA per tile that holds a site: the tile's sites in slot order at the tile's scanned offset
//
// pi is summed in a fixed order everywhere (a lane's positions in order, a fixed shuffle tree, chunks in a fixed
// order), with no float atomics: the same counts give bit-identical sums whatever the read order or the decoder.
// pi_p is computed with _rn intrinsics so that nothing is contracted into an FMA: it is bit-identical to numpy's.
#pragma once
#include <stdint.h>
#include "k_allele_rules.cuh"

namespace mcov {

constexpr int kAlThreads = 256;          // region kernels: 8 warps a CTA
constexpr int kAlWarps = kAlThreads / 32;
constexpr int kAlChunk = 2048;           // positions a chunk (64 a lane)
constexpr int kAlTile = 4096;            // slots a site tile
constexpr int kAlTileThreads = 256;
constexpr uint8_t kRefUnknown = 4;

struct AlPart {                                // a chunk's partial record (a region's record minus its length)
  int64_t covered, depth_sum;
  double pi_sum;
  int64_t snv, ref_covered, sub, popsub, pad;
};

// The rules at one position: kind bits 1 SNV, 2 SUB, 4 POPSUB; cons 0-3 (A C G T).  Only meaningful when covered.
struct AlPos {
  uint64_t n;
  double pi;
  uint32_t kind, cons;
  bool covered;
};

__device__ __forceinline__ AlPos allele_eval(const uint4 c, const uint32_t r, const AlleleParams& P) {
  AlPos o;
  o.n = (uint64_t)c.x + c.y + c.z + c.w;
  o.covered = o.n >= P.min_cov;
  o.pi = 0.0; o.kind = 0; o.cons = 0;
  if (!o.covered) return o;
  const double dn = (double)o.n;
  const AlRules ru = allele_rules(c, dn, P);
  const uint32_t mask = ru.mask, best = ru.best;
  const double fa = __ddiv_rn((double)c.x, dn), fc = __ddiv_rn((double)c.y, dn);
  const double fg = __ddiv_rn((double)c.z, dn), ft = __ddiv_rn((double)c.w, dn);
  o.pi = __dsub_rn(1.0, __dadd_rn(__dadd_rn(__dmul_rn(fa, fa), __dmul_rn(fc, fc)), __dadd_rn(__dmul_rn(fg, fg), __dmul_rn(ft, ft))));
  o.cons = best;
  uint32_t k = __popc(mask) >= 2 ? 1u : 0u;
  if (r < 4) {
    if (best != r) k |= 2u;
    if (mask != 0 && !((mask >> r) & 1u)) k |= 4u;
  }
  o.kind = k;
  return o;
}

__global__ void k_ref_encode(const uint8_t* __restrict__ ascii, int64_t n, uint8_t* __restrict__ dst) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t ch = ascii[i] & 0xDFu;                // upper case
    dst[i] = ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : kRefUnknown;
  }
}

struct AlRegionArgs {
  const uint4* cnt;              // [n_slots] A C G T
  const uint8_t* ref;            // [n_slots] codes (read only with P.use_ref)
  const AlChunk* chunks; int64_t n_chunks;
  AlPart* part;                  // [n_chunks]
  AlleleParams P;
};

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}

__global__ void __launch_bounds__(kAlThreads)
k_allele_chunks(AlRegionArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kAlWarps;
  for (int64_t w = (int64_t)blockIdx.x * kAlWarps + (threadIdx.x >> 5); w < a.n_chunks; w += nw) {
    const AlChunk ch = a.chunks[w];
    const uint4* cp = a.cnt + ch.slot;
    const uint8_t* rp = a.ref + ch.slot;
    const int n = (int)ch.n;
    uint32_t cov = 0, snv = 0, refc = 0, sub = 0, pop = 0;
    uint64_t dsum = 0;
    double pi = 0.0;
    // two loads in flight a lane; positions lane, lane + 32, ... in order
    for (int j = lane; j < n; j += 64) {
      const bool two = j + 32 < n;
      const uint4 c0 = __ldg(cp + j);
      const uint4 c1 = two ? __ldg(cp + j + 32) : make_uint4(0, 0, 0, 0);
      const uint32_t r0 = a.P.use_ref ? __ldg(rp + j) : kRefUnknown;
      const uint32_t r1 = (a.P.use_ref && two) ? __ldg(rp + j + 32) : kRefUnknown;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const AlPos o = allele_eval(u ? c1 : c0, u ? r1 : r0, a.P);
        dsum += o.n;
        if (o.covered) {
          const uint32_t r = u ? r1 : r0;
          cov += 1; pi = __dadd_rn(pi, o.pi);
          snv += o.kind & 1u; refc += r < 4; sub += (o.kind >> 1) & 1u; pop += (o.kind >> 2) & 1u;
        }
      }
    }
    const long long c_ = warp_sum_i64(cov), d_ = warp_sum_i64((long long)dsum), s_ = warp_sum_i64(snv);
    const long long rc_ = warp_sum_i64(refc), sb_ = warp_sum_i64(sub), pp_ = warp_sum_i64(pop);
    pi = warp_sum_f64(pi);
    if (lane == 0) {
      AlPart p;
      p.covered = c_; p.depth_sum = d_; p.pi_sum = pi; p.snv = s_; p.ref_covered = rc_; p.sub = sb_; p.popsub = pp_; p.pad = 0;
      a.part[w] = p;
    }
  }
}

// Region r's record from the partials of its chunks [first[r], first[r + 1]); length[r] = end - start.
__global__ void __launch_bounds__(kAlThreads)
k_allele_combine(const AlPart* __restrict__ part, const int64_t* __restrict__ first, const int64_t* __restrict__ length,
                 int64_t g, mcov_allele_stats* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kAlWarps;
  for (int64_t r = (int64_t)blockIdx.x * kAlWarps + (threadIdx.x >> 5); r < g; r += nw) {
    long long cov = 0, d = 0, snv = 0, refc = 0, sub = 0, pop = 0;
    double pi = 0.0;
    for (int64_t k = first[r] + lane; k < first[r + 1]; k += 32) {
      const AlPart p = part[k];
      cov += p.covered; d += p.depth_sum; pi = __dadd_rn(pi, p.pi_sum);
      snv += p.snv; refc += p.ref_covered; sub += p.sub; pop += p.popsub;
    }
    cov = warp_sum_i64(cov); d = warp_sum_i64(d); snv = warp_sum_i64(snv);
    refc = warp_sum_i64(refc); sub = warp_sum_i64(sub); pop = warp_sum_i64(pop);
    pi = warp_sum_f64(pi);
    if (lane == 0) {
      mcov_allele_stats s;
      s.length = length[r]; s.covered = cov; s.depth_sum = d; s.pi_sum = pi;
      s.snv = snv; s.ref_covered = refc; s.sub = sub; s.popsub = pop;
      out[r] = s;
    }
  }
}

struct AlSiteArgs {
  const uint4* cnt; const uint8_t* ref;
  int64_t n_slots, n_tiles;
  const int64_t* contig_off; int32_t n_contigs;
  int64_t* tile_n;               // sites a tile (written by the count pass)
  const int64_t* tile_incl;      // their inclusive scan (read by the write pass)
  mcov_allele_site* sites;
  AlleleParams P;
};

__device__ __forceinline__ uint32_t al_ref_at(const AlSiteArgs& a, int64_t s) { return a.P.use_ref ? __ldg(a.ref + s) : kRefUnknown; }

__global__ void __launch_bounds__(kAlTileThreads)
k_allele_site_count(AlSiteArgs a) {
  __shared__ int s_w[kAlTileThreads / 32];
  for (int64_t t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
    const int64_t s0 = t * kAlTile;
    int n = 0;
#pragma unroll 4
    for (int k = 0; k < kAlTile / kAlTileThreads; ++k) {
      const int64_t s = s0 + k * kAlTileThreads + threadIdx.x;
      if (s < a.n_slots) n += allele_eval(__ldg(a.cnt + s), al_ref_at(a, s), a.P).kind != 0;
    }
    store_tile_count<kAlTileThreads>(n, s_w, a.tile_n, t, threadIdx.x);
  }
}

__global__ void __launch_bounds__(kAlTileThreads)
k_allele_site_write(AlSiteArgs a) {
  __shared__ int s_w[kAlTileThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
    const int64_t nt = a.tile_n[t];
    if (nt == 0) continue;                                   // (uniform over the CTA) tiles without a site are not read again
    int64_t base = a.tile_incl[t] - nt;
    const int64_t s0 = t * kAlTile;
    for (int k = 0; k < kAlTile / kAlTileThreads; ++k) {
      const int64_t s = s0 + k * kAlTileThreads + threadIdx.x;
      uint4 c = make_uint4(0, 0, 0, 0);
      uint32_t r = kRefUnknown;
      AlPos o; o.kind = 0;
      if (s < a.n_slots) { c = __ldg(a.cnt + s); r = al_ref_at(a, s); o = allele_eval(c, r, a.P); }
      const unsigned bal = __ballot_sync(0xffffffffu, o.kind != 0);
      if (lane == 0) s_w[warp] = __popc(bal);
      __syncthreads();
      int before = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < kAlTileThreads / 32; ++w) { before += w < warp ? s_w[w] : 0; tot += s_w[w]; }
      if (o.kind != 0) {
        const int32_t lo = contig_of(a.contig_off, a.n_contigs, s);
        mcov_allele_site st;
        st.tid = lo; st.pos = (int32_t)(s - a.contig_off[lo]);
        st.cnt[0] = c.x; st.cnt[1] = c.y; st.cnt[2] = c.z; st.cnt[3] = c.w;
        st.ref = (uint8_t)(r < 4 ? "ACGT"[r] : 'N'); st.consensus = (uint8_t)"ACGT"[o.cons]; st.kind = (uint8_t)o.kind;
        for (int q = 0; q < 5; ++q) st.pad[q] = 0;
        a.sites[base + before + __popc(bal & ((1u << lane) - 1u))] = st;
      }
      base += tot;
      __syncthreads();
    }
  }
}

}  // namespace mcov
