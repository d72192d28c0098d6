// k_linkage.cuh -- linkage between nearby SNV sites from the reads and their mates (include/metacov_b200.h:
// mcov_linkage; oracle/linkage.py restates the rules).  The sites are an allele site list of the counts (k_alleles.cuh,
// use_reference 0: SNV sites only); the records are those k_bc_any counts, read through the same BcBamRec / BcSamRec.
//
//   k_link_sites        one thread per site: its slot, contig, major / minor allele and how many later sites of its
//                       contig lie within max_distance (one binary search)
//   k_link_obs<_, 0>    one warp per record: how many (unit, site, base) observations it makes
//   k_link_obs<_, 1>    the same walk, writing them at the record's scanned offset
//   k_link_unit_calls   one thread per observation sorted by (unit, site): the first of each (unit, site) run gets the
//                       unit's call there (0 major, 1 minor) or none, every other observation none
//   k_link_pairs        one thread per call: the later calls of its unit on its contig within max_distance, one
//                       atomicAdd each on the candidate pair's counter
//   k_link_pair_count   one CTA per tile of kLkTile candidate pairs: the pairs with at least min_reads units
//   k_link_pair_write   one CTA per tile that holds one: the tile's pairs in row order at the tile's scanned offset
//
// Candidate pairs: site i's partners are the sites i + 1 .. i + partners[i]; the pair (i, j) is row
// base[i] + (j - i - 1) of the counters, four uint32 a row (n_AB n_Ab n_aB n_ab, index 2 call_i + call_j).  Rows are in
// (site i, site j) order, which is (tid, pos_a, pos_b) order.
//
// An observation is 16 bytes sorted as one 128-bit key (name, sec), name the more significant word.  name: the unit's
// key -- read_name_key of QNAME, or the record's index in the file for a record named '*'.  sec, from the top:
//   bit 63                 1 for a '*' record (so that its index can never equal a name's key)
//   bits [63 - sb, 63)     the site's index in the site list (sb bits: enough for every index)
//   bits [61 - sb, 63 - sb) the base (0-3 = A C G T); in the unit-call output the call (0, 1; 3 = none)
//   below                  0, so that the sort covers bits [61 - sb, 128) only
// Sorting gives every unit's observations together, by site, and a site's bases of one unit together.
#pragma once
#include <stdint.h>
#include "k_allele_rules.cuh"
#include "k_basecount.cuh"

namespace mcov {

constexpr int kLkThreads = 256;
constexpr int kLkWarps = kLkThreads / 32;
constexpr int kLkTile = 4096;            // candidate pairs a tile
constexpr int kLkTileThreads = 256;

struct LkObs { uint64_t sec, name; };

__host__ __device__ __forceinline__ int lk_site_shift(int sb) { return 63 - sb; }
__host__ __device__ __forceinline__ uint64_t lk_sec(uint32_t star, uint64_t site, uint32_t code, int sb) {
  return ((uint64_t)star << 63) | (site << (63 - sb)) | ((uint64_t)code << (61 - sb));
}
__device__ __forceinline__ uint64_t lk_site(uint64_t sec, int sb) { return (sec << 1) >> (64 - sb); }
__device__ __forceinline__ uint32_t lk_code(uint64_t sec, int sb) { return (uint32_t)(sec >> (61 - sb)) & 3u; }
__device__ __forceinline__ bool lk_same_unit(const LkObs& a, const LkObs& b) { return a.name == b.name && (a.sec >> 63) == (b.sec >> 63); }

// Site i of the list: slot, contig, alleles (major | minor << 2) and partners (later sites of its contig at most
// max_distance after it).
__global__ void __launch_bounds__(kLkThreads)
k_link_sites(const mcov_allele_site* __restrict__ sites, int64_t n, const int64_t* __restrict__ contig_off, int32_t max_distance,
             int64_t* __restrict__ slot, int32_t* __restrict__ tid, uint8_t* __restrict__ allele, int64_t* __restrict__ partners) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const mcov_allele_site s = sites[i];
    const uint32_t major = s.consensus == 'A' ? 0 : s.consensus == 'C' ? 1 : s.consensus == 'G' ? 2 : 3;
    uint32_t minor = major == 0 ? 1 : 0;
#pragma unroll
    for (uint32_t b = 0; b < 4; ++b)
      if (b != major && s.cnt[b] > s.cnt[minor]) minor = b;           // (the first of equal counts stays)
    slot[i] = contig_off[s.tid] + s.pos;
    tid[i] = s.tid;
    allele[i] = (uint8_t)(major | (minor << 2));
    // the last site j >= i with (tid_j, pos_j) <= (tid, pos + max_distance)
    const int64_t lim = (int64_t)s.pos + max_distance;
    int64_t lo = i, hi = n - 1;
    while (lo < hi) {
      const int64_t m = (lo + hi + 1) >> 1;
      const int32_t mt = sites[m].tid;
      if (mt < s.tid || (mt == s.tid && (int64_t)sites[m].pos <= lim)) lo = m; else hi = m - 1;
    }
    partners[i] = lo - i;
  }
}

struct LkObsArgs {
  BcArgs bc;                     // the records [bc.i0, bc.n), their filter and error word (bc.cnt unused)
  const int64_t* slot; int64_t n_sites; int sb;
  int64_t* rec_n;                // count pass: the observations of record i at rec_n[i - bc.i0]
  const int64_t* rec_off;        // write pass: their exclusive scan
  LkObs* obs;                    // write pass: the batch's observations start here
};

// The unit key of record i and whether its QNAME is '*' (BAM: l_read_name 2 and a '*'; SAM: the field is one '*').
__device__ __forceinline__ uint64_t lk_name(const BcArgs& a, int64_t i, const BcBamRec&, bool* star) {
  const uint8_t* r = a.data + a.rec_off[i] + 4;
  const uint32_t l_name = r[8];
  *star = l_name == 2 && r[32] == '*';
  return read_name_key<1>(r, 32, l_name);
}
__device__ __forceinline__ uint64_t lk_name(const BcArgs& a, int64_t i, const BcSamRec&, bool* star) {
  const uint8_t* q = a.data + a.rec_off[i];
  const uint32_t n = a.aux[i].l_qname;
  *star = n == 1 && q[0] == '*';
  return read_name_key<0>(q, 0, n);
}

// Record i's observations, walked by one warp: the filter, SEQ / QUAL check and error word of bc_read, one binary
// search for the first site at or after the record's start, then the ops in order, the lanes taking 32 sites at a time
// from a cursor that every reference-consuming op moves past its end.  A site inside an M / = / X op is observed when
// the base there is A, C, G or T and passes the quality threshold.  Returns the count (every lane).
template <class Rec, bool kWrite>
__device__ __forceinline__ int64_t lk_read(const LkObsArgs& a, int64_t i, int lane) {
  const BcArgs& b = a.bc;
  const int32_t t = b.tid[i], p0 = b.pos[i];
  if ((uint32_t)t >= (uint32_t)b.n_contigs || p0 < 0 || (b.flag[i] & b.skip_flags)) return 0;
  const int32_t ls = b.l_seq[i];
  if (ls <= 0) return 0;
  const uint32_t c0 = b.cig_off[i], c1 = b.cig_off[i + 1];
  unsigned long long ql = 0;
  for (uint32_t k = c0 + lane; k < c1; k += 32) { const uint32_t c = b.cig[k]; if (bc_cons_query(c & 15u)) ql += c >> 4; }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) ql += __shfl_xor_sync(0xffffffffu, ql, s);
  const Rec R(b, i, ls);
  if (!R.ok || ql > (unsigned long long)ls) {
    if (!kWrite && lane == 0) atomicMin(b.err, ((unsigned long long)(b.rec_base + i) << 2) | (R.ok ? kBcErrQueryLong : kBcErrLeavesRecord));
    return 0;
  }
  if (b.qthr != 0 && !R.has_qual) return 0;
  const int64_t cbase = b.contig_off[t];
  const int64_t len = b.contig_len[t];
  int64_t k = 0, hi = a.n_sites;                                   // the first site with slot >= cbase + p0
  while (k < hi) { const int64_t m = (k + hi) >> 1; if (__ldg(a.slot + m) < cbase + p0) k = m + 1; else hi = m; }
  if (k == a.n_sites || __ldg(a.slot + k) >= cbase + len) return 0;
  uint64_t key = 0;
  uint32_t star = 0;
  int64_t out = 0;
  if (kWrite) {
    bool st = false;
    key = lk_name(b, i, R, &st);
    if (st) key = (uint64_t)(b.rec_base + i);
    star = st;
    out = a.rec_off[i - b.i0];
  }
  const unsigned lt = (1u << lane) - 1u;
  int64_t n = 0, q = 0, r = p0;
  for (uint32_t c = c0; c < c1 && r < len; ++c) {
    const uint32_t cg = b.cig[c], op = cg & 15u;
    const int64_t l = cg >> 4;
    if (bc_cons_ref(op)) {
      const int64_t A = cbase + r, B = cbase + (l < len - r ? r + l : len);
      const bool aligned = op == 0 || op == 7 || op == 8;
      for (;;) {
        const int64_t idx = k + lane;
        const int64_t s = idx < a.n_sites ? __ldg(a.slot + idx) : INT64_MAX;
        const bool in = s < B;
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        bool ok = false;
        uint32_t code = 0;
        if (aligned && in) {
          const int64_t qq = q + (s - A);
          const uint32_t bb = R.base(qq);
          ok = (bb == 1 || bb == 2 || bb == 4 || bb == 8) && (b.qthr == 0 || R.qv(qq) >= b.qthr);
          code = __ffs(bb) - 1;
        }
        const unsigned okb = __ballot_sync(0xffffffffu, ok);
        if (kWrite && ok) {
          LkObs o;
          o.name = key; o.sec = lk_sec(star, (uint64_t)idx, code, a.sb);
          a.obs[out + n + __popc(okb & lt)] = o;
        }
        n += __popc(okb);
        k += __popc(bal);
        if (bal != 0xffffffffu) break;
      }
    }
    if (bc_cons_query(op)) q += l;
    if (bc_cons_ref(op)) r += l;
  }
  return n;
}

template <class Rec, bool kWrite>
__global__ void __launch_bounds__(kLkThreads)
k_link_obs(LkObsArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kLkWarps;
  for (int64_t i = a.bc.i0 + (int64_t)blockIdx.x * kLkWarps + (threadIdx.x >> 5); i < a.bc.n; i += nw) {
    const int64_t n = lk_read<Rec, kWrite>(a, i, lane);
    if (!kWrite && lane == 0) a.rec_n[i - a.bc.i0] = n;
  }
}

// in[n] sorted -> out[n]: each observation with its code replaced by the call of its (unit, site) run if it starts one
// (all the run's bases equal -- the first and the last, as they are sorted -- and the major or the minor allele), else
// by 3.  *n_units gains the number of units (runs of one name and '*' bit).
__global__ void __launch_bounds__(kLkThreads)
k_link_unit_calls(const LkObs* __restrict__ in, int64_t n, const uint8_t* __restrict__ allele, int sb, LkObs* __restrict__ out,
                  unsigned long long* __restrict__ n_units) {
  const int sh = lk_site_shift(sb);
  const uint64_t code_mask = 3ull << (61 - sb);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j0 = (int64_t)blockIdx.x * blockDim.x; j0 < n; j0 += stride) {
    const int64_t j = j0 + threadIdx.x;
    bool unit_start = false;
    if (j < n) {
      const LkObs o = in[j];
      const LkObs p = j > 0 ? in[j - 1] : LkObs{~o.sec, ~o.name};
      unit_start = !lk_same_unit(o, p);
      uint32_t call = 3;
      if (unit_start || (o.sec >> sh) != (p.sec >> sh)) {
        int64_t e = j + 1;
        while (e < n && in[e].name == o.name && (in[e].sec >> sh) == (o.sec >> sh)) ++e;
        const uint32_t b0 = lk_code(o.sec, sb);
        if (b0 == lk_code(in[e - 1].sec, sb)) {
          const uint32_t al = allele[lk_site(o.sec, sb)];
          call = b0 == (al & 3u) ? 0u : b0 == (al >> 2) ? 1u : 3u;
        }
      }
      LkObs w = o;
      w.sec = (o.sec & ~code_mask) | ((uint64_t)call << (61 - sb));
      out[j] = w;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, unit_start);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(n_units, (unsigned long long)__popc(bal));
  }
}

struct LkPairArgs {
  const LkObs* calls; int64_t n_calls; int sb;
  const int64_t* slot; const int32_t* tid; const uint8_t* allele; const int64_t* base; int64_t n_sites;
  const int64_t* contig_off;
  int32_t max_distance; uint32_t min_reads;
  uint32_t* cnt;                 // [n_candidates][4]
  int64_t n_cand, n_tiles;
  int64_t* tile_n; const int64_t* tile_incl;
  mcov_linkage_pair* pairs;
};

__global__ void __launch_bounds__(kLkThreads)
k_link_pairs(LkPairArgs a) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n_calls; i += (int64_t)gridDim.x * blockDim.x) {
    const LkObs c = a.calls[i];
    const int64_t si = (int64_t)lk_site(c.sec, a.sb);
    const uint32_t ci = lk_code(c.sec, a.sb);
    const int64_t s0 = __ldg(a.slot + si);
    const int32_t t = __ldg(a.tid + si);
    const int64_t r0 = __ldg(a.base + si) - si - 1;          // + j: the row of the pair (si, j)
    for (int64_t j = i + 1; j < a.n_calls; ++j) {
      const LkObs d = a.calls[j];
      if (!lk_same_unit(c, d)) break;
      const int64_t sj = (int64_t)lk_site(d.sec, a.sb);
      if (__ldg(a.tid + sj) != t || __ldg(a.slot + sj) - s0 > a.max_distance) break;
      atomicAdd(a.cnt + (r0 + sj) * 4 + 2 * ci + lk_code(d.sec, a.sb), 1u);
    }
  }
}

__device__ __forceinline__ bool lk_reported(const LkPairArgs& a, int64_t row, uint4* c) {
  if (row >= a.n_cand) return false;
  *c = __ldg(reinterpret_cast<const uint4*>(a.cnt) + row);
  return (uint64_t)c->x + c->y + c->z + c->w >= a.min_reads;
}

__global__ void __launch_bounds__(kLkTileThreads)
k_link_pair_count(LkPairArgs a) {
  __shared__ int s_w[kLkTileThreads / 32];
  for (int64_t t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
    const int64_t r0 = t * kLkTile;
    int n = 0;
    uint4 c;
#pragma unroll 4
    for (int k = 0; k < kLkTile / kLkTileThreads; ++k) n += lk_reported(a, r0 + k * kLkTileThreads + threadIdx.x, &c);
    store_tile_count<kLkTileThreads>(n, s_w, a.tile_n, t, threadIdx.x);
  }
}

__global__ void __launch_bounds__(kLkTileThreads)
k_link_pair_write(LkPairArgs a) {
  __shared__ int s_w[kLkTileThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t t = blockIdx.x; t < a.n_tiles; t += gridDim.x) {
    const int64_t nt = a.tile_n[t];
    if (nt == 0) continue;                                   // (uniform over the CTA)
    int64_t out = a.tile_incl[t] - nt;
    const int64_t r0 = t * kLkTile;
    for (int k = 0; k < kLkTile / kLkTileThreads; ++k) {
      const int64_t row = r0 + k * kLkTileThreads + threadIdx.x;
      uint4 c;
      const bool rep = lk_reported(a, row, &c);
      const unsigned bal = __ballot_sync(0xffffffffu, rep);
      if (lane == 0) s_w[warp] = __popc(bal);
      __syncthreads();
      int before = 0, tot = 0;
#pragma unroll
      for (int w = 0; w < kLkTileThreads / 32; ++w) { before += w < warp ? s_w[w] : 0; tot += s_w[w]; }
      if (rep) {
        int64_t lo = 0, hi = a.n_sites - 1;                 // the site i whose rows hold `row`: the last base[i] <= row
        while (lo < hi) { const int64_t m = (lo + hi + 1) >> 1; if (__ldg(a.base + m) <= row) lo = m; else hi = m - 1; }
        const int64_t j = lo + 1 + (row - __ldg(a.base + lo));
        const int32_t tid = __ldg(a.tid + lo);
        const int64_t off = __ldg(a.contig_off + tid);
        const uint32_t ai = a.allele[lo], aj = a.allele[j];
        mcov_linkage_pair p;
        p.tid = tid; p.pos_a = (int32_t)(__ldg(a.slot + lo) - off); p.pos_b = (int32_t)(__ldg(a.slot + j) - off);
        p.major_a = (uint8_t)"ACGT"[ai & 3u]; p.minor_a = (uint8_t)"ACGT"[ai >> 2];
        p.major_b = (uint8_t)"ACGT"[aj & 3u]; p.minor_b = (uint8_t)"ACGT"[aj >> 2];
        p.n_AB = c.x; p.n_Ab = c.y; p.n_aB = c.z; p.n_ab = c.w;
        a.pairs[out + before + __popc(bal & ((1u << lane) - 1u))] = p;
      }
      out += tot;
      __syncthreads();
    }
  }
}

}  // namespace mcov
