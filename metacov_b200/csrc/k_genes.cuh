// k_genes.cuh -- codons of genes from the A / C / G / T counters of mcov_base_counts and the reference store
// (include/metacov_b200.h: mcov_gene_run; oracle/genes.py restates the rules).  A gene's codon span is cut on the host
// into chunks of whole codons, in genomic order.
//
//   k_gene_chunks      one warp per chunk, one lane per codon: the chunk's partial record and, with a site list, its
//                      number of site records
//   k_gene_combine     one warp per gene: its chunks' partials, lanes strided over them, then a shuffle tree
//   k_gene_site_write  one warp per chunk that holds a site record: the records of 32 codons at a time, placed by a warp
//                      scan of the lanes' record counts (at most 3 a codon) at the chunk's scanned offset
//
// Everything is integer: the same counts give the same records whatever the read order or the decoder.
#pragma once
#include <stdint.h>
#include "k_allele_rules.cuh"

namespace mcov {

constexpr int kGnThreads = 256;          // 8 warps a CTA
constexpr int kGnWarps = kGnThreads / 32;
constexpr int kGnChunk = 640;            // codons a chunk (20 a lane)

// n codons in genomic order from slot (contig tid, position pos) of gene `gene`; the i-th has codon index
// codon0 + dir * i (dir = the strand: on - the genomically first codon is the gene's last)
struct GnChunk {
  int64_t slot, gene;
  int32_t tid, pos, n, codon0, dir, pad;
};

struct GnPart {                          // a chunk's partial record (s_sites3 = 9 called - n_sites3)
  int64_t called, n3, snv_n, snv_s, snv_m, sub_n, sub_s, sub_m;
};

// The standard code indexed by A C G T codon codes (16 b0 + 4 b1 + b2, b0 the 5' base), and per codon n3: of its 9
// single-base changes, those that change the amino acid ('*' counts as one).
struct GnTables {
  char aa[64];
  uint8_t n3[64];
};

constexpr int gn_tcag(int b) { return b == 0 ? 2 : b == 1 ? 1 : b == 2 ? 3 : 0; }   // A C G T -> index in T C A G

constexpr GnTables gn_make_tables() {
  const char code[] = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";
  GnTables t{};
  for (int c = 0; c < 64; ++c) t.aa[c] = code[16 * gn_tcag(c >> 4) + 4 * gn_tcag((c >> 2) & 3) + gn_tcag(c & 3)];
  for (int c = 0; c < 64; ++c) {
    int n = 0;
    for (int sh = 0; sh <= 4; sh += 2)
      for (int x = 0; x < 4; ++x)
        if (x != ((c >> sh) & 3) && t.aa[(c & ~(3 << sh)) | (x << sh)] != t.aa[c]) ++n;
    t.n3[c] = (uint8_t)n;
  }
  return t;
}

__constant__ GnTables c_gn = gn_make_tables();

// The codon code, in gene orientation, of genomic bases g0 g1 g2 (on -: reversed and complemented).
__device__ __forceinline__ uint32_t gn_code(uint32_t g0, uint32_t g1, uint32_t g2, bool minus) {
  return minus ? ((3u - g2) << 4 | (3u - g1) << 2 | (3u - g0)) : (g0 << 4 | g1 << 2 | g2);
}

// code with genomic base j (0-2) of its codon replaced by b
__device__ __forceinline__ uint32_t gn_with(uint32_t code, int j, uint32_t b, bool minus) {
  const int sh = minus ? 2 * j : 4 - 2 * j;
  return (code & ~(3u << sh)) | ((minus ? 3u - b : b) << sh);
}

// One codon: called, and per genomic position j two bits each of kind (1 SNV, 2 SUB), consensus, minor allele, SNV
// type and SUB type (1 N, 2 S, 3 M); R the reference codon's code.  Only called codons have kinds.
struct GnCodon {
  bool called;
  uint32_t R, kind, cons, minor, snv_t, sub_t;
};

__device__ __forceinline__ GnCodon gn_eval(const uint4* c, const uint32_t* r, bool minus, const AlleleParams& P) {
  GnCodon o;
  o.called = false; o.R = 0; o.kind = 0; o.cons = 0; o.minor = 0; o.snv_t = 0; o.sub_t = 0;
  uint64_t n[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    n[j] = (uint64_t)c[j].x + c[j].y + c[j].z + c[j].w;
    if (n[j] < P.min_cov || r[j] > 3) return o;
  }
  o.called = true;
  o.R = gn_code(r[0], r[1], r[2], minus);
  int nsnv = 0, nsub = 0;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const AlRules ru = allele_rules(c[j], (double)n[j], P);
    const uint32_t v[4] = {c[j].x, c[j].y, c[j].z, c[j].w};
    uint32_t mi = ru.best == 0 ? 1u : 0u;                 // the largest other count, the first of equal ones
#pragma unroll
    for (uint32_t b = 0; b < 4; ++b)
      if (b != ru.best && v[b] > v[mi]) mi = b;
    const uint32_t k = (__popc(ru.mask) >= 2 ? 1u : 0u) | (ru.best != r[j] ? 2u : 0u);
    nsnv += k & 1u; nsub += k >> 1;
    o.kind |= k << (2 * j); o.cons |= ru.best << (2 * j); o.minor |= mi << (2 * j);
  }
  const char aa_ref = c_gn.aa[o.R];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const uint32_t k = (o.kind >> (2 * j)) & 3u;
    if (k == 0) continue;
    const char aa_major = c_gn.aa[gn_with(o.R, j, (o.cons >> (2 * j)) & 3u, minus)];
    if (k & 1u) {
      const char aa_minor = c_gn.aa[gn_with(o.R, j, (o.minor >> (2 * j)) & 3u, minus)];
      o.snv_t |= (nsnv >= 2 ? 3u : aa_major == aa_minor ? 2u : 1u) << (2 * j);
    }
    if (k & 2u) o.sub_t |= (nsub >= 2 ? 3u : aa_major == aa_ref ? 2u : 1u) << (2 * j);
  }
  return o;
}

// positions of a 2-bit-per-position field equal to v
__device__ __forceinline__ uint32_t gn_count(uint32_t f, uint32_t v) {
  return (((f & 3u) == v) ? 1u : 0u) + ((((f >> 2) & 3u) == v) ? 1u : 0u) + ((((f >> 4) & 3u) == v) ? 1u : 0u);
}

struct GnArgs {
  const uint4* cnt;              // [n_slots] A C G T
  const uint8_t* ref;            // [n_slots] codes
  const GnChunk* chunks; int64_t n_chunks;
  GnPart* part;                  // [n_chunks]
  int64_t* tile_n;               // [n_chunks] site records a chunk, or null: no site list
  const int64_t* tile_incl;      // their inclusive scan (read by the write pass)
  mcov_gene_site* sites;
  AlleleParams P;
};

__device__ __forceinline__ GnCodon gn_load_eval(const GnArgs& a, int64_t s, bool minus) {
  uint4 c[3];
  uint32_t r[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) { c[j] = __ldg(a.cnt + s + j); r[j] = __ldg(a.ref + s + j); }
  return gn_eval(c, r, minus, a.P);
}

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

__global__ void __launch_bounds__(kGnThreads)
k_gene_chunks(GnArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kGnWarps;
  for (int64_t w = (int64_t)blockIdx.x * kGnWarps + (threadIdx.x >> 5); w < a.n_chunks; w += nw) {
    const GnChunk ch = a.chunks[w];
    const bool minus = ch.dir < 0;
    uint32_t called = 0, n3 = 0, sn = 0, ss = 0, sm = 0, un = 0, us = 0, um = 0, recs = 0;
    for (int i = lane; i < ch.n; i += 32) {
      const GnCodon o = gn_load_eval(a, ch.slot + 3 * (int64_t)i, minus);
      if (!o.called) continue;
      called += 1; n3 += c_gn.n3[o.R];
      sn += gn_count(o.snv_t, 1); ss += gn_count(o.snv_t, 2); sm += gn_count(o.snv_t, 3);
      un += gn_count(o.sub_t, 1); us += gn_count(o.sub_t, 2); um += gn_count(o.sub_t, 3);
      recs += 3 - gn_count(o.kind, 0);
    }
    called = warp_sum_u32(called); n3 = warp_sum_u32(n3);
    sn = warp_sum_u32(sn); ss = warp_sum_u32(ss); sm = warp_sum_u32(sm);
    un = warp_sum_u32(un); us = warp_sum_u32(us); um = warp_sum_u32(um);
    if (a.tile_n) recs = warp_sum_u32(recs);
    if (lane == 0) {
      GnPart p;
      p.called = called; p.n3 = n3; p.snv_n = sn; p.snv_s = ss; p.snv_m = sm; p.sub_n = un; p.sub_s = us; p.sub_m = um;
      a.part[w] = p;
      if (a.tile_n) a.tile_n[w] = recs;
    }
  }
}

// Gene r's record from the partials of its chunks [first[r], first[r + 1]); length[r] = end - start, codons[r] = K.
__global__ void __launch_bounds__(kGnThreads)
k_gene_combine(const GnPart* __restrict__ part, const int64_t* __restrict__ first, const int64_t* __restrict__ length,
               const int64_t* __restrict__ codons, int64_t g, mcov_gene_stats* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kGnWarps;
  for (int64_t r = (int64_t)blockIdx.x * kGnWarps + (threadIdx.x >> 5); r < g; r += nw) {
    long long called = 0, n3 = 0, sn = 0, ss = 0, sm = 0, un = 0, us = 0, um = 0;
    for (int64_t k = first[r] + lane; k < first[r + 1]; k += 32) {
      const GnPart p = part[k];
      called += p.called; n3 += p.n3; sn += p.snv_n; ss += p.snv_s; sm += p.snv_m; un += p.sub_n; us += p.sub_s; um += p.sub_m;
    }
    called = warp_sum_i64(called); n3 = warp_sum_i64(n3);
    sn = warp_sum_i64(sn); ss = warp_sum_i64(ss); sm = warp_sum_i64(sm);
    un = warp_sum_i64(un); us = warp_sum_i64(us); um = warp_sum_i64(um);
    if (lane == 0) {
      mcov_gene_stats s;
      s.length = length[r]; s.codons = codons[r]; s.codons_called = called; s.n_sites3 = n3; s.s_sites3 = 9 * called - n3;
      s.snv_n = sn; s.snv_s = ss; s.snv_m = sm; s.sub_n = un; s.sub_s = us; s.sub_m = um; s.pad = 0;
      out[r] = s;
    }
  }
}

__global__ void __launch_bounds__(kGnThreads)
k_gene_site_write(GnArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kGnWarps;
  for (int64_t w = (int64_t)blockIdx.x * kGnWarps + (threadIdx.x >> 5); w < a.n_chunks; w += nw) {
    const int64_t nt = a.tile_n[w];
    if (nt == 0) continue;                                   // (uniform over the warp) chunks without a record
    int64_t base = a.tile_incl[w] - nt;
    const GnChunk ch = a.chunks[w];
    const bool minus = ch.dir < 0;
    for (int i0 = 0; i0 < ch.n; i0 += 32) {
      const int i = i0 + lane;
      GnCodon o;
      o.kind = 0;
      if (i < ch.n) o = gn_load_eval(a, ch.slot + 3 * (int64_t)i, minus);
      const uint32_t k = 3 - gn_count(o.kind, 0);
      uint32_t incl = k;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += y;
      }
      const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);
      if (k != 0) {
        int64_t at = base + incl - k;
        mcov_gene_site st;
        st.gene = ch.gene; st.tid = ch.tid; st.codon = ch.codon0 + ch.dir * i;
        const uint32_t R = o.R;
        st.ref_codon[0] = (uint8_t)"ACGT"[R >> 4]; st.ref_codon[1] = (uint8_t)"ACGT"[(R >> 2) & 3u];
        st.ref_codon[2] = (uint8_t)"ACGT"[R & 3u];
        st.aa_ref = (uint8_t)c_gn.aa[R];
        for (int j = 0; j < 3; ++j) {
          const uint32_t kj = (o.kind >> (2 * j)) & 3u;
          if (kj == 0) continue;
          const uint32_t cj = (o.cons >> (2 * j)) & 3u, mj = (o.minor >> (2 * j)) & 3u;
          const uint32_t tn = (o.snv_t >> (2 * j)) & 3u, tb = (o.sub_t >> (2 * j)) & 3u;
          st.pos = ch.pos + 3 * i + j;
          st.codon_pos = (uint8_t)(minus ? 2 - j : j);
          st.major = (uint8_t)"ACGT"[cj];
          st.minor = (kj & 1u) ? (uint8_t)"ACGT"[mj] : 0;
          st.aa_major = (uint8_t)c_gn.aa[gn_with(R, j, cj, minus)];
          st.aa_minor = (kj & 1u) ? (uint8_t)c_gn.aa[gn_with(R, j, mj, minus)] : 0;
          st.kind = (uint8_t)kj;
          st.snv_type = (uint8_t)"\0NSM"[tn];
          st.sub_type = (uint8_t)"\0NSM"[tb];
          a.sites[at++] = st;
        }
      }
      base += tot;
    }
  }
}

}  // namespace mcov
