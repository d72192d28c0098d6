// k_basecount.cuh -- A / C / G / T counts at every reference position (pysam's AlignmentFile.count_coverage) from the
// records of a device decode: the decoded columns (tid, pos, flag, l_seq, cig_off, cig) plus SEQ and QUAL read where
// the decoder left them -- the inflated BAM records or the SAM text.
//
//   k_bc_any      one warp per read, lanes over the query positions of each M / = / X op, one global atomicAdd per
//                 counted base.  Correct in any order, and the only kernel: a tiled variant for sorted input (a CTA
//                 counting the reads that start in a window of slots in shared memory, flushing the window with one
//                 add per non-zero counter) took 2.53 ms where this one takes 1.21 ms on the same sorted columns
//                 (DESIGN.md 3.14), and was removed.
//
// Counters: uint32 in the depth store's slot layout (contig_off + refpos), four per slot ([slot][A C G T]), so that the
// four counters of a position share one 16-byte sector.
#pragma once
#include <stdint.h>
#include "common.cuh"
#include "k_sam.cuh"

namespace mcov {

constexpr int kBcThreads = 256;
constexpr int kBcWarps = kBcThreads / 32;
constexpr uint32_t kBcSkipAll = 0x4u | 0x100u | 0x200u | 0x400u;  // read_callback="all": unmapped, secondary, QC fail, duplicate

// failure codes, low bits of the error word ((record << 2) | code; the smallest record wins)
enum BcErr { kBcErrQueryLong = 1, kBcErrLeavesRecord = 2 };

struct BcArgs {
  const int32_t* tid; const int32_t* pos; const uint16_t* flag; const int32_t* l_seq;
  const uint32_t* cig_off; const uint32_t* cig;
  const uint8_t* data;          // the inflated BAM stream or the SAM text
  const uint64_t* rec_off;      // where each record starts in `data`
  const SamAux* aux;            // SAM: field offsets of each line (SEQ at aux.seq_b)
  const int64_t* contig_off; const int32_t* contig_len; int32_t n_contigs;
  int64_t i0, n;                // the records [i0, n) are counted
  int64_t rec_base;             // added to a failing record's index in the error word (batches of a streamed file)
  uint32_t skip_flags;          // records with any of these flags are skipped
  int32_t qthr;                 // 0: every aligned base counts; else only with qualities and qual >= qthr
  uint32_t* cnt;                // [n_slots][4]
  unsigned long long* err;      // smallest (record << 2) | BcErr, ~0 = none
};

__device__ __forceinline__ uint32_t bc_ld16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
__device__ __forceinline__ uint32_t bc_ld32(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// A BAM record (SAM spec 4.2): SEQ behind the name and the ops, nt16 two per byte high nibble first, QUAL behind it;
// no qualities = first QUAL byte 0xFF.  `ok`: SEQ and QUAL lie inside the record.
struct BcBamRec {
  const uint8_t* seq; const uint8_t* qual; bool ok, has_qual;
  __device__ __forceinline__ BcBamRec(const BcArgs& a, int64_t i, int32_t l_seq) {
    const uint8_t* p = a.data + a.rec_off[i];
    const uint32_t bs = bc_ld32(p);
    const uint8_t* r = p + 4;
    const uint32_t l_name = r[8], n_op = bc_ld16(r + 12);
    seq = r + 32 + l_name + 4ull * n_op;
    qual = seq + (l_seq + 1) / 2;
    ok = 32ull + l_name + 4ull * n_op + (uint64_t)((l_seq + 1) / 2) + (uint64_t)l_seq <= bs;
    has_qual = ok && qual[0] != 0xFFu;
  }
  __device__ __forceinline__ uint32_t base(int64_t q) const { const uint32_t b = seq[q >> 1]; return (q & 1) ? (b & 15u) : (b >> 4); }
  __device__ __forceinline__ int qv(int64_t q) const { return qual[q]; }
};

// A SAM line: SEQ at aux.seq_b, QUAL one TAB behind it (the decoder checked it is '*' or l_seq long); no qualities = the
// QUAL field is exactly '*' (the byte behind it is a TAB, CR or LF -- or the zero padding behind the text -- whereas a
// quality byte is >= '!').  Bases through htslib's seq_nt16_table (case-insensitive), qualities the byte minus 33.
struct BcSamRec {
  const uint8_t* seq; const uint8_t* qual; bool ok, has_qual;
  __device__ __forceinline__ BcSamRec(const BcArgs& a, int64_t i, int32_t l_seq) {
    seq = a.data + a.rec_off[i] + a.aux[i].seq_b;
    qual = seq + l_seq + 1;
    ok = true;
    has_qual = !(qual[0] == '*' && (l_seq == 1 || qual[1] < 33u));
  }
  __device__ __forceinline__ uint32_t base(int64_t q) const { return sam_nt16(seq[q]); }
  __device__ __forceinline__ int qv(int64_t q) const { return (int)qual[q] - 33; }
};

// query bases an op consumes (M I S = X) / reference bases (M D N = X)
__device__ __forceinline__ bool bc_cons_query(uint32_t op) { return (0x193u >> op) & 1u; }
__device__ __forceinline__ bool bc_cons_ref(uint32_t op) { return (0x18Du >> op) & 1u; }

// The aligned pairs of read i (get_aligned_pairs(matches_only=True)) counted by one warp: the whole warp walks the ops,
// the lanes take the query positions of an M / = / X op.  Only A C G T (nt16 1 2 4 8) count; pairs at or past the
// contig's end are dropped.
template <class Rec>
__device__ __forceinline__ void bc_read(const BcArgs& a, int64_t i, int lane) {
  const int32_t t = a.tid[i], p0 = a.pos[i];
  if ((uint32_t)t >= (uint32_t)a.n_contigs || p0 < 0 || (a.flag[i] & a.skip_flags)) return;
  const int32_t ls = a.l_seq[i];
  if (ls <= 0) return;                                           // no SEQ: nothing to count
  const uint32_t c0 = a.cig_off[i], c1 = a.cig_off[i + 1];
  unsigned long long ql = 0;
  for (uint32_t k = c0 + lane; k < c1; k += 32) { const uint32_t c = a.cig[k]; if (bc_cons_query(c & 15u)) ql += c >> 4; }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) ql += __shfl_xor_sync(0xffffffffu, ql, s);
  const Rec R(a, i, ls);
  if (!R.ok || ql > (unsigned long long)ls) {                    // never read past SEQ or QUAL: the call fails instead
    if (lane == 0) atomicMin(a.err, ((unsigned long long)(a.rec_base + i) << 2) | (R.ok ? kBcErrQueryLong : kBcErrLeavesRecord));
    return;
  }
  if (a.qthr != 0 && !R.has_qual) return;
  const int64_t base = a.contig_off[t];
  const int64_t len = a.contig_len[t];
  int64_t q = 0, r = p0;
  for (uint32_t k = c0; k < c1 && r < len; ++k) {
    const uint32_t c = a.cig[k], op = c & 15u;
    const int64_t l = c >> 4;
    if (op == 0 || op == 7 || op == 8) {
      const int64_t m = l < len - r ? l : len - r;
      for (int64_t j = lane; j < m; j += 32) {
        const uint32_t b = R.base(q + j);
        if ((b == 1 || b == 2 || b == 4 || b == 8) && (a.qthr == 0 || R.qv(q + j) >= a.qthr))
          atomicAdd(a.cnt + (base + r + j) * 4 + (__ffs(b) - 1), 1u);
      }
    }
    if (bc_cons_query(op)) q += l;
    if (bc_cons_ref(op)) r += l;
  }
}

template <class Rec>
__global__ void __launch_bounds__(kBcThreads)
k_bc_any(BcArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * kBcWarps;
  for (int64_t i = a.i0 + (int64_t)blockIdx.x * kBcWarps + (threadIdx.x >> 5); i < a.n; i += nw) bc_read<Rec>(a, i, lane);
}

}  // namespace mcov
