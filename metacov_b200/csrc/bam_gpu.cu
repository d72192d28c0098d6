// bam_gpu.cu -- BGZF inflate and BAM record parsing on the GPU (SURVEY.md 8(f) row 3).
//
// From a BAM file the host decode -- zlib over every BGZF block, then a serial walk over the records --
// bounds the end-to-end rate of the coverage path by two orders of magnitude (bamio.cpp: ~0.3 s for the
// 10 M reads the kernels finish in 0.2 ms).  Here the COMPRESSED file goes over PCIe (3-4x fewer bytes
// than the SoA) and everything else happens on the device:
//
//   (inflate, B200, 4 173 blocks of a 1 M-read BAM: thread per block 127 ms; warp per block with lane-parallel
//   match copies 19.5 ms; + first-level Huffman tables 17.1 ms; + shared-memory output window of 16 / 8 / 4 / 2 KiB
//   25.6 / 19.1 / 13.0 / 11.6 ms -- the kernel is bound by instruction issue of the redundant symbol decode, so
//   resident warps matter more than the window size)
//
//   k_bgzf_inflate     one warp per BGZF block (independent raw-deflate streams of <= 64 KiB, SAM spec
//                      4.1; inflate.cuh: redundant symbol decode, lane-parallel match copies), optional
//                      CRC-32 check
//   k_bam_guess        BAM records are length-prefixed, so record starts form ONE chain from the end of
//                      the header -- serial by nature.  To walk it in parallel, a warp per 64 KiB chunk of
//                      the inflated stream looks for the first offset that parses as three plausible
//                      records in a row (the approach of Hadoop-BAM's record guesser) ...
//   k_bam_walk_count   ... then one thread per chunk walks the chain from its guessed start up to the next
//                      chunk's, counting records and CIGAR ops.  The host checks that every walk ENDS
//                      EXACTLY ON the next guessed start: a guess the true chain lands on is a true record
//                      start, so the union of the walks is the true chain -- exact, not heuristic.  A
//                      guess that is not hit is dropped and the two segments are walked again as one.
//   k_bam_walk_write   second walk: the SoA columns (tid, pos, flag, mapq, l_seq, isize, cig_off, cig) of
//                      reference scan.pyx:243-294 straight into device memory, ready for
//                      mcov_depth_sorted(..., MCOV_MEM_DEVICE).
//
// Replaces, for this path, `pysam.AlignmentFile` + `IteratorRowAll` (reference metacov/scan.pyx:204,
// 216; cli.py:56) -- like bamio.cpp, which stays the host decoder.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "bamfmt.h"
#include "ctx.cuh"
#include "inflate.cuh"

namespace mcov {

#ifndef MCOV_INFLATE_WINDOW
#define MCOV_INFLATE_WINDOW 2048              /* bytes of recent output mirrored in shared memory, per warp */
#endif
constexpr int kInflateThreads = 64;           // 2 warps per CTA
constexpr uint32_t kInflateWindow = MCOV_INFLATE_WINDOW;
static_assert((kInflateWindow & (kInflateWindow - 1)) == 0 && kInflateWindow >= 1024, "window: a power of two >= 1 KiB");
constexpr uint32_t kGuessChunk = 65536;
constexpr int kGuessChain = 3;

#ifndef MCOV_INFLATE_GROUP
#define MCOV_INFLATE_GROUP 32                 /* lanes that decode one BGZF block together (a power of two <= 32) */
#endif
constexpr int kInflateGroup = MCOV_INFLATE_GROUP;
constexpr int kInflateGroupsPerCta = kInflateThreads / kInflateGroup;
static_assert(kInflateGroup >= 1 && kInflateGroup <= 32 && (kInflateGroup & (kInflateGroup - 1)) == 0, "group: 1, 2, 4, ... 32 lanes");

// The symbol decode is redundant across the lanes of a group (that keeps its control flow uniform).  Smaller
// groups do NOT recover the redundant issue slots: groups of one warp sit at different points of their streams,
// the warp serialises them, and each group only gets slower -- measured 11.6 ms with whole warps, 20.3 ms with
// groups of 16, 34.9 ms with groups of 8 (same 1 M-read BAM).
__global__ void __launch_bounds__(kInflateThreads)
k_bgzf_inflate(const uint8_t* __restrict__ raw, const BgzfBlock* __restrict__ blocks, int64_t n_blocks, uint8_t* out,
               int verify_crc, int* __restrict__ status) {
  __shared__ uint16_t s_tabs[kInflateGroupsPerCta][kInfTabWords];                     // first-level Huffman tables, one set per group
  __shared__ uint8_t s_win[kInflateGroupsPerCta][kInflateWindow];                     // recent output, one window per group
  const int grp = threadIdx.x / kInflateGroup;
  const int64_t k = (int64_t)blockIdx.x * kInflateGroupsPerCta + grp;                 // one group per block
  const int lane = threadIdx.x & (kInflateGroup - 1);
  const unsigned gmask = (kInflateGroup == 32 ? 0xffffffffu : ((1u << kInflateGroup) - 1u)) << ((threadIdx.x & 31) & ~(kInflateGroup - 1));
  if (k >= n_blocks) return;
  const BgzfBlock b = blocks[k];
  int rc = b.ulen ? inflate_raw(raw + b.coff, b.clen, out + b.uoff, b.ulen, s_tabs[grp], lane, kInflateGroup, s_win[grp],
                               kInflateWindow - 1u, gmask) : 0;
  if (rc == 0 && verify_crc && b.ulen) {
    // lane-sliced CRC-32, folded left to right (inflate.cuh)
    uint32_t lo, hi;
    crc_slice(b.ulen, lane, kInflateGroup, lo, hi);
    const uint32_t mine = crc32_bytes(out + b.uoff + lo, hi - lo);
    const uint32_t op_full = crc_x8n(hi - lo);                  // (lanes with a full slice all compute the same factor)
    uint32_t crc = __shfl_sync(gmask, mine, 0, kInflateGroup);
    for (int j = 1; j < kInflateGroup; ++j) {
      const uint32_t cj = __shfl_sync(gmask, mine, j, kInflateGroup), opj = __shfl_sync(gmask, op_full, j, kInflateGroup);
      const uint32_t nj = __shfl_sync(gmask, hi - lo, j, kInflateGroup);
      if (nj) crc = crc_multmodp(opj, crc) ^ cj;
    }
    if (crc != b.crc) rc = 100;
  }
  if (lane == 0 && rc) { atomicCAS(status, 0, rc); atomicMax(status + 1, (int)min(k, (int64_t)0x7fffffff)); }   // first error code, a failing block
}

__device__ __forceinline__ uint32_t ld32u(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__device__ __forceinline__ uint32_t ld16u(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// Does a BAM alignment record plausibly start at offset p?  (SAM spec 4.2; every test is a necessary
// condition of a well-formed record.)  Returns the offset of the next record, or 0 if not plausible.
__device__ __forceinline__ uint64_t bam_plausible(const uint8_t* __restrict__ d, uint64_t p, uint64_t total, int32_t n_ref) {
  if (p + 36 > total) return 0;
  const uint32_t bs = ld32u(d + p);
  if (bs < 32u || bs > (1u << 28) || p + 4 + bs > total) return 0;
  const int32_t ref = (int32_t)ld32u(d + p + 4), pos = (int32_t)ld32u(d + p + 8);
  if (ref < -1 || ref >= n_ref || pos < -1) return 0;
  const uint32_t l_name = d[p + 12], n_op = ld16u(d + p + 16);
  const int32_t l_seq = (int32_t)ld32u(d + p + 20);
  const int32_t nref = (int32_t)ld32u(d + p + 24), npos = (int32_t)ld32u(d + p + 28);
  if (l_name < 1u || l_seq < 0 || nref < -1 || nref >= n_ref || npos < -1) return 0;
  const uint64_t need = 32ull + l_name + 4ull * n_op + (uint64_t)((l_seq + 1) >> 1) + (uint64_t)l_seq;
  if (need > bs) return 0;
  if (d[p + 36 + l_name - 1] != 0) return 0;              // the read name is NUL-terminated
  return p + 4 + bs;
}

// One warp per chunk: the first offset in [lo, hi) from which kGuessChain plausible records follow one
// another (a chain that reaches the end of the stream exactly also counts).
__global__ void __launch_bounds__(128)
k_bam_guess(const uint8_t* __restrict__ d, uint64_t total, uint64_t rec_begin, int32_t n_ref, int64_t n_chunks, long long* __restrict__ starts) {
  const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= n_chunks) return;
  uint64_t lo = (uint64_t)c * kGuessChunk, hi = min(lo + (uint64_t)kGuessChunk, total);
  long long found = -1;
  if (lo <= rec_begin && rec_begin < hi) { found = (long long)rec_begin; lo = hi; }      // the chain's known head
  if (hi <= rec_begin) lo = hi;                                                          // inside the header
  for (uint64_t p0 = lo; p0 < hi && found < 0; p0 += 32) {
    const uint64_t p = p0 + lane;
    bool ok = false;
    if (p < hi) {
      uint64_t q = p;
      ok = true;
      for (int k = 0; k < kGuessChain && q != total; ++k) {
        q = bam_plausible(d, q, total, n_ref);
        if (q == 0) { ok = false; break; }
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m) found = (long long)(p0 + (uint64_t)(__ffs(m) - 1));
  }
  if (lane == 0) starts[c] = found;
}

struct WalkSeg { uint64_t start, limit; uint64_t rec_base, cig_base; };
struct WalkOut { uint64_t end; uint32_t n_rec; uint32_t n_cig; int32_t err; int32_t pad; };

// One thread per segment: follow the record chain from seg.start until it reaches seg.limit.
__global__ void k_bam_walk_count(const uint8_t* __restrict__ d, uint64_t total, const WalkSeg* __restrict__ segs, int64_t n_seg,
                                 WalkOut* __restrict__ out, int allow_tail) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  const WalkSeg g = segs[s];
  uint64_t p = g.start;
  uint32_t n_rec = 0, n_cig = 0;
  int err = 0;
  while (p < g.limit) {
    if (p + 36 > total) { if (!allow_tail) err = 1; break; }      // (allow_tail: the record continues in the next chunk)
    const uint32_t bs = ld32u(d + p);
    const uint32_t l_name = d[p + 12], n_op = ld16u(d + p + 16);
    if (bs >= 32u && p + 4 + bs > total && allow_tail) break;
    if (bs < 32u || p + 4 + bs > total || 32ull + l_name + 4ull * n_op > bs) { err = 2; break; }
    ++n_rec;
    n_cig += n_op;
    p += 4ull + bs;
  }
  WalkOut o;
  o.end = p; o.n_rec = n_rec; o.n_cig = n_cig; o.err = err; o.pad = 0;
  out[s] = o;
}

struct SoaOut {
  int32_t* tid; int32_t* pos; uint16_t* flag; uint8_t* mapq; int32_t* l_seq; int32_t* isize; uint32_t* cig_off; uint32_t* cig;
  uint64_t* rec_off;      // where the record (its block_size field) starts in the inflated stream
};

__global__ void k_bam_walk_write(const uint8_t* __restrict__ d, const WalkSeg* __restrict__ segs, int64_t n_seg, SoaOut o) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_seg) return;
  const WalkSeg g = segs[s];
  uint64_t p = g.start, i = g.rec_base, co = g.cig_base;
  while (p < g.limit) {
    const uint8_t* r = d + p + 4;
    const uint32_t bs = ld32u(d + p);
    const uint32_t l_name = r[8], n_op = ld16u(r + 12);
    o.tid[i] = (int32_t)ld32u(r);
    o.pos[i] = (int32_t)ld32u(r + 4);
    o.mapq[i] = r[9];
    o.flag[i] = (uint16_t)ld16u(r + 14);
    o.l_seq[i] = (int32_t)ld32u(r + 16);
    o.isize[i] = (int32_t)ld32u(r + 28);
    o.cig_off[i] = (uint32_t)co;
    o.rec_off[i] = p;
    const uint8_t* c = r + 32 + l_name;
    for (uint32_t k = 0; k < n_op; ++k) o.cig[co + k] = ld32u(c + 4 * k);
    co += n_op;
    ++i;
    p += 4ull + bs;
  }
}

// Read names and SEQ, the parts of a record the coverage path never looks at but `pileup.experimental` and the k-mer
// histogram do.  One thread per record, straight from the inflated stream:
//   name_hash[i]  FNV-1a 64 of the read name (the key of the reference's mate dict, metacov/pileup.py:101-118);
//   kmer_code[i]  2-bit code of query_alignment_sequence[0:k_len] (pileup.py:109-110, 123): SEQ without the soft-clipped
//                 ends, first base most significant, A0 C1 G2 T3; -1 = shorter than k_len or another letter;
//   win[i][W]     the first (forward) / last (reverse strand, flag 0x10) win_bases bases, nt16 two per byte, high nibble
//                 first, missing bases 'N' (15): all of SEQ the k-mer histogram reads (scan.pyx:240-259, 513-520).
// Same definitions, bit for bit, as the host reader's mcov_bam_name_hash / mcov_bam_qas_kmer / mcov_bam_seq_windows.
__global__ void k_bam_names_seq(const uint8_t* __restrict__ d, const uint64_t* __restrict__ rec_off, int64_t n, int32_t k_len,
                                int32_t win_bases, uint64_t* __restrict__ name_hash, int32_t* __restrict__ kmer_code,
                                uint8_t* __restrict__ win, int* __restrict__ status) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t p = rec_off[i];
  const uint8_t* r = d + p + 4;
  const uint32_t bs = ld32u(d + p);
  const uint32_t l_name = r[8], n_op = ld16u(r + 12), flag = ld16u(r + 14);
  const int64_t l_seq = (int64_t)ld32u(r + 16);
  const uint8_t* cig = r + 32 + l_name;
  const uint8_t* sq = cig + 4ull * n_op;
  if (32ull + l_name + 4ull * n_op + (uint64_t)((l_seq + 1) / 2) > bs) { atomicExch(status + 2, 1); return; }   // SEQ leaves the record
  if (name_hash) {
    uint64_t h = 1469598103934665603ull;
    for (uint32_t k = 0; k + 1 < l_name; ++k) { h ^= r[32 + k]; h *= 1099511628211ull; }
    name_hash[i] = h == ~0ull ? h - 1 : h;                     // ~0 is the "no entry" key of the pair sort
  }
  auto base = [&](int64_t a) -> uint32_t { const uint32_t b = sq[a >> 1]; return (a & 1) ? (b & 15u) : (b >> 4); };
  if (kmer_code) {
    int64_t lo = 0, hi = l_seq;
    for (uint32_t k = 0; k < n_op; ++k) {                      // leading soft clips (hard clips hold no bases)
      const uint32_t c = ld32u(cig + 4 * k), op = c & 15u;
      if (op == 5) continue;
      if (op == 4) lo += c >> 4; else break;
    }
    for (uint32_t k = n_op; k > 0; --k) {
      const uint32_t c = ld32u(cig + 4 * (k - 1)), op = c & 15u;
      if (op == 5) continue;
      if (op == 4) hi -= c >> 4; else break;
    }
    int32_t code = hi - lo < k_len ? -1 : 0;
    for (int32_t j = 0; j < k_len && code >= 0; ++j) {
      const uint32_t b = base(lo + j);                         // "=ACMGRSVTWYHKDBN": A 1, C 2, G 4, T 8
      const int c = b == 1 ? 0 : b == 2 ? 1 : b == 4 ? 2 : b == 8 ? 3 : -1;
      code = c < 0 ? -1 : (code << 2) | c;
    }
    kmer_code[i] = code;
  }
  if (win) {
    const int W = (win_bases + 1) / 2;
    const bool rev = (flag & 0x10u) != 0;
    uint8_t* o = win + (size_t)i * W;
    for (int b2 = 0; b2 < W; ++b2) {
      uint32_t v = 0;
      for (int h = 0; h < 2; ++h) {
        const int j = 2 * b2 + h;
        uint32_t c = 15;
        if (j < win_bases) {
          const int64_t a = rev ? l_seq - win_bases + j : j;
          if (a >= 0 && a < l_seq) c = base(a);
        }
        v = (v << 4) | c;
      }
      o[b2] = (uint8_t)v;
    }
  }
}

// Streamed decode (mcov_bam_gpu_stream_depth): which reads of this batch must lead the next one.  The streamed depth
// pass wants every read that starts at or after the resend point (rt, rp) or reaches past it; in a sorted batch those
// form a SUFFIX plus a few earlier reads, and since resending more is harmless the whole suffix from the first such read
// is carried.  One thread per read; *first receives the smallest qualifying index (initialised to n).
__global__ void k_bam_carry_first(int64_t n, const int32_t* __restrict__ tid, const int32_t* __restrict__ pos,
                                  const uint32_t* __restrict__ cig_off, const uint32_t* __restrict__ cig, int32_t rt, int32_t rp,
                                  int32_t n_contigs, unsigned long long* __restrict__ first) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t t = (uint32_t)tid[i], r = (uint32_t)rt;
  if (t >= (uint32_t)n_contigs) return;                           // unplaced reads (tid -1, sorted last) never count: not carried
  bool take = t > r || (t == r && pos[i] >= rp);
  if (!take && t == r) {                                          // same contig, starts before the point: does it reach past it?
    long long e = pos[i];
    for (uint32_t k = cig_off[i]; k < cig_off[i + 1] && e <= rp; ++k) e += cigar_ref_len(cig[k]);
    take = e > rp;
  }
  if (take) atomicMin(first, (unsigned long long)i);
}
__global__ void k_bam_rebase_offsets(int64_t m, const uint32_t* __restrict__ src, uint32_t base, uint32_t* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < m) dst[i] = src[i] - base;
}

}  // namespace mcov

using namespace mcov;

#define CUB(call)                                                          \
  do {                                                                     \
    cudaError_t e__ = (call);                                              \
    if (e__ != cudaSuccess) { ctx->err = std::string("mcov_bam_decode_gpu: ") + #call + ": " + cudaGetErrorString(e__); return MCOV_ERR_CUDA; } \
  } while (0)

static int bfail(mcov_ctx* ctx, int code, const char* msg) { ctx->err = msg; return code; }

// Header of the inflated stream at B.data (read on the host) -> n_ref and the offset of the first alignment record.  Also
// the place where the inflate status is looked at.
static int bam_dev_header(mcov_ctx* ctx, uint64_t total, uint64_t* rec_begin_out, int32_t* n_ref_out) {
  mcov_ctx::BamDev& B = ctx->bam;
  cudaStream_t s = ctx->stream;
  int st[2] = {0, 0};
  std::vector<uint8_t> head;
  size_t want = (size_t)std::min<uint64_t>(total, 1u << 20);
  BamHeader h;
  for (;;) {
    head.resize(want);
    CUB(cudaMemcpyAsync(head.data(), B.data.p, want, cudaMemcpyDeviceToHost, s));
    CUB(cudaMemcpyAsync(st, B.status.p, sizeof(st), cudaMemcpyDeviceToHost, s));
    CUB(cudaStreamSynchronize(s));
    if (st[0]) {
      ctx->err = st[0] == 100 ? "mcov_bam_decode_gpu: CRC mismatch in a BGZF block" : "mcov_bam_decode_gpu: corrupt deflate stream in a BGZF block";
      return MCOV_ERR_IO;
    }
    const HeaderParse r = parse_bam_header(head.data(), want, false, h);
    if (r == HeaderParse::kOk) break;
    if (r == HeaderParse::kBad) { ctx->err = std::string("mcov_bam_decode_gpu: ") + h.bad; return MCOV_ERR_IO; }
    if (want >= total)
      return bfail(ctx, MCOV_ERR_IO, r == HeaderParse::kMoreText ? "mcov_bam_decode_gpu: truncated BAM header" : "mcov_bam_decode_gpu: truncated reference table");
    want = (size_t)std::min<uint64_t>(total, (uint64_t)want * 4);
  }
  *rec_begin_out = h.rec_begin; *n_ref_out = h.n_ref;
  return MCOV_OK;
}

// Record starts of the inflated stream B.data[0, total): guess per 64 KiB chunk, walk, verify the links (see the
// head of this file).  allow_tail: the stream may end inside a record (a chunk of a larger file): the chain then stops
// in front of it and *end_out is where that record begins; otherwise the chain must end exactly at `total`.
static int bam_dev_chain(mcov_ctx* ctx, uint64_t total, uint64_t rec_begin, int32_t n_ref, bool allow_tail,
                         std::vector<WalkSeg>& segs, std::vector<WalkOut>& wo, uint64_t* end_out) {
  mcov_ctx::BamDev& B = ctx->bam;
  cudaStream_t s = ctx->stream;
  const int64_t n_chunks = (int64_t)((total + kGuessChunk - 1) / kGuessChunk);
  CUB(B.starts.ensure((size_t)n_chunks * 8));
  MCOV_LAUNCH(ctx, kKBamGuess, (k_bam_guess<<<(unsigned)((n_chunks * 32 + 127) / 128), 128, 0, s>>>(
      B.data.as<uint8_t>(), total, rec_begin, n_ref, n_chunks, B.starts.as<long long>())));
  CUB(cudaGetLastError());
  std::vector<long long> starts((size_t)n_chunks);
  CUB(cudaMemcpyAsync(starts.data(), B.starts.p, (size_t)n_chunks * 8, cudaMemcpyDeviceToHost, s));
  CUB(cudaStreamSynchronize(s));
  std::vector<uint64_t> cand;
  if (rec_begin < total) cand.push_back(rec_begin);
  for (int64_t c = 0; c < n_chunks; ++c)
    if (starts[c] > (long long)rec_begin) cand.push_back((uint64_t)starts[c]);
  for (int round = 0;; ++round) {
    if (round > 64) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu: record chain could not be established");
    const int64_t ns = (int64_t)cand.size();
    segs.resize((size_t)ns);
    for (int64_t i = 0; i < ns; ++i) { segs[i].start = cand[i]; segs[i].limit = i + 1 < ns ? cand[i + 1] : total; segs[i].rec_base = 0; segs[i].cig_base = 0; }
    wo.resize((size_t)ns);
    if (ns == 0) break;
    CUB(B.segs.ensure((size_t)ns * sizeof(WalkSeg)));
    CUB(B.wout.ensure((size_t)ns * sizeof(WalkOut)));
    CUB(cudaMemcpyAsync(B.segs.p, segs.data(), (size_t)ns * sizeof(WalkSeg), cudaMemcpyHostToDevice, s));
    MCOV_LAUNCH(ctx, kKBamWalkCount, (k_bam_walk_count<<<(unsigned)((ns + 127) / 128), 128, 0, s>>>(
        B.data.as<uint8_t>(), total, B.segs.as<WalkSeg>(), ns, B.wout.as<WalkOut>(), allow_tail ? 1 : 0)));
    CUB(cudaGetLastError());
    CUB(cudaMemcpyAsync(wo.data(), B.wout.p, (size_t)ns * sizeof(WalkOut), cudaMemcpyDeviceToHost, s));
    CUB(cudaStreamSynchronize(s));
    // a walk must end exactly on the next start (the last one on the end of the stream); a start that is
    // not hit was a false guess: drop it and walk the merged segment again
    std::vector<uint64_t> keep;
    bool changed = false;
    keep.push_back(cand[0]);
    for (int64_t i = 0; i < ns; ++i) {
      if (wo[i].err) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu: malformed BAM record");
      if (i + 1 < ns) {
        if (wo[i].end == cand[i + 1]) keep.push_back(cand[i + 1]); else changed = true;
      } else if (wo[i].end != total && !allow_tail) {
        return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu: the last BAM record is truncated");
      }
    }
    if (!changed) break;
    // (dropping start i+1 changes where the merged walk ends, so later links are re-examined next round)
    cand.swap(keep);
  }
  *end_out = wo.empty() ? rec_begin : wo.back().end;
  return MCOV_OK;
}

// The columns of n records and `ops` CIGAR ops: sized, written from the records of `segs` (k_bam_walk_write) and closed
// with cig_off[n] = ops.  The rows in front of the segments' rec_base (reads carried into a chunk) are the caller's.
static cudaError_t bam_dev_columns(mcov_ctx* ctx, const std::vector<WalkSeg>& segs, uint64_t n, uint64_t ops, SoaOut& o) {
  mcov_ctx::BamDev& B = ctx->bam;
  cudaStream_t s = ctx->stream;
  const struct { DevBuf* buf; uint64_t bytes; } cols[] = {
      {&B.tid, (n + 4) * 4}, {&B.pos, (n + 4) * 4}, {&B.flag, (n + 4) * 2}, {&B.mapq, n + 4}, {&B.lseq, (n + 4) * 4},
      {&B.isize, (n + 4) * 4}, {&B.cig_off, (n + 5) * 4}, {&B.cig, (ops + 4) * 4}, {&B.rec_off, (n + 4) * 8}};
  cudaError_t e;
  for (const auto& c : cols)
    if ((e = c.buf->ensure((size_t)c.bytes)) != cudaSuccess) return e;
  o.tid = B.tid.as<int32_t>(); o.pos = B.pos.as<int32_t>(); o.flag = B.flag.as<uint16_t>(); o.mapq = B.mapq.as<uint8_t>();
  o.l_seq = B.lseq.as<int32_t>(); o.isize = B.isize.as<int32_t>(); o.cig_off = B.cig_off.as<uint32_t>(); o.cig = B.cig.as<uint32_t>();
  o.rec_off = B.rec_off.as<uint64_t>();
  if (!segs.empty()) {
    if ((e = cudaMemcpyAsync(B.segs.p, segs.data(), segs.size() * sizeof(WalkSeg), cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    MCOV_LAUNCH(ctx, kKBamWalkWrite, (k_bam_walk_write<<<(unsigned)((segs.size() + 127) / 128), 128, 0, s>>>(
        B.data.as<uint8_t>(), B.segs.as<WalkSeg>(), (int64_t)segs.size(), o)));
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  const uint32_t last = (uint32_t)ops;                   // (a pageable source is copied before the call returns)
  return cudaMemcpyAsync(o.cig_off + n, &last, 4, cudaMemcpyHostToDevice, s);
}

extern "C" int mcov_bam_decode_gpu(mcov_ctx* ctx, const void* file_bytes, int64_t n_bytes, int verify_crc, mcov_bam_dev* out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!file_bytes || n_bytes <= 0 || !out) return bfail(ctx, MCOV_ERR_ARG, "mcov_bam_decode_gpu: bad arguments");
  std::memset(out, 0, sizeof(*out));
  CUB(cudaSetDevice(ctx->device));
  ctx->bam.sam = false;
  cudaStream_t s = ctx->stream;
  const uint8_t* raw = static_cast<const uint8_t*>(file_bytes);
  std::vector<BgzfBlock> blocks;
  uint64_t total = 0;
  size_t used = 0;
  if (!bgzf_index(raw, (size_t)n_bytes, 0, false, blocks, total, used)) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu: not a valid BGZF file");
  if (total < 12) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu: not a valid BAM file");
  const int64_t nb = (int64_t)blocks.size();
  mcov_ctx::BamDev& B = ctx->bam;
  // compressed image + block table to the device, inflate
  CUB(B.raw.ensure((size_t)n_bytes));
  CUB(B.blocks.ensure((size_t)nb * sizeof(BgzfBlock)));
  CUB(B.data.ensure((size_t)total + 64));
  CUB(B.status.ensure(64));
  CUB(cudaMemcpyAsync(B.raw.p, raw, (size_t)n_bytes, cudaMemcpyHostToDevice, s));
  CUB(cudaMemcpyAsync(B.blocks.p, blocks.data(), (size_t)nb * sizeof(BgzfBlock), cudaMemcpyHostToDevice, s));
  CUB(cudaMemsetAsync(B.status.p, 0, 64, s));
  MCOV_LAUNCH(ctx, kKBgzfInflate, (k_bgzf_inflate<<<(unsigned)((nb + kInflateGroupsPerCta - 1) / kInflateGroupsPerCta), kInflateThreads, 0, s>>>(
      B.raw.as<uint8_t>(), B.blocks.as<BgzfBlock>(), nb, B.data.as<uint8_t>(), verify_crc, B.status.as<int>())));
  CUB(cudaGetLastError());
  uint64_t rec_begin = 0;
  int32_t n_ref = 0;
  { int hrc = bam_dev_header(ctx, total, &rec_begin, &n_ref); if (hrc) return hrc; }
  std::vector<WalkSeg> segs;
  std::vector<WalkOut> wo;
  { uint64_t chain_end = 0; int crc2 = bam_dev_chain(ctx, total, rec_begin, n_ref, false, segs, wo, &chain_end); if (crc2) return crc2; }
  // prefix sums -> where every segment writes
  uint64_t n_rec = 0, n_cig = 0;
  for (size_t i = 0; i < segs.size(); ++i) { segs[i].rec_base = n_rec; segs[i].cig_base = n_cig; n_rec += wo[i].n_rec; n_cig += wo[i].n_cig; }
  if (n_cig > 0xFFFFFFFFull) return bfail(ctx, MCOV_ERR_RANGE, "mcov_bam_decode_gpu: more than 2^32-1 CIGAR ops");
  B.n_rec = 0;
  SoaOut o;
  CUB(bam_dev_columns(ctx, segs, n_rec, n_cig, o));
  CUB(cudaStreamSynchronize(s));
  out->n_records = (int64_t)n_rec; out->n_cigar = (int64_t)n_cig; out->n_ref = n_ref;
  out->inflated_bytes = (int64_t)total; out->header_bytes = (int64_t)rec_begin; out->n_segments = (int64_t)segs.size();
  out->tid = o.tid; out->pos = o.pos; out->flag = o.flag; out->mapq = o.mapq; out->l_seq = o.l_seq; out->isize = o.isize;
  out->cig_off = o.cig_off; out->cig = o.cig; out->inflated = B.data.as<uint8_t>();
  B.n_rec = (int64_t)n_rec;
  return MCOV_OK;
}

int mcov_sam_gpu_names_seq(mcov_ctx* ctx, int32_t k_len, int32_t win_bases, uint64_t* d_hash, int32_t* d_kmer, uint8_t* d_win);   // sam_gpu.cu

extern "C" int mcov_bam_gpu_names_seq(mcov_ctx* ctx, int32_t k_len, int32_t win_bases, uint64_t* name_hash_out,
                                      int32_t* kmer_code_out, uint8_t* seq_win_out, int mem_kind) {
  if (!ctx) return MCOV_ERR_ARG;
  mcov_ctx::BamDev& B = ctx->bam;
  if (B.n_rec < 0 || !B.data.p) return bfail(ctx, MCOV_ERR_STATE, "mcov_bam_gpu_names_seq: no file decoded on this context");
  if ((kmer_code_out && (k_len <= 0 || k_len > 15)) || (seq_win_out && win_bases <= 0) ||
      (mem_kind != MCOV_MEM_HOST && mem_kind != MCOV_MEM_DEVICE))
    return bfail(ctx, MCOV_ERR_ARG, "mcov_bam_gpu_names_seq: bad arguments");
  const int64_t n = B.n_rec;
  if (n == 0 || (!name_hash_out && !kmer_code_out && !seq_win_out)) return MCOV_OK;
  CUB(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const size_t W = seq_win_out ? ((size_t)win_bases + 1) / 2 : 0;
  const bool dev = mem_kind == MCOV_MEM_DEVICE;
  uint64_t* d_hash = name_hash_out; int32_t* d_kmer = kmer_code_out; uint8_t* d_win = seq_win_out;
  if (!dev) {                                                  // results are produced on the device, then copied out
    if (name_hash_out) { CUB(B.name_hash.ensure((size_t)n * 8)); d_hash = B.name_hash.as<uint64_t>(); }
    if (kmer_code_out) { CUB(B.kmer.ensure((size_t)n * 4)); d_kmer = B.kmer.as<int32_t>(); }
    if (seq_win_out) { CUB(B.win.ensure((size_t)n * W)); d_win = B.win.as<uint8_t>(); }
  }
  CUB(cudaMemsetAsync(B.status.as<int>() + 2, 0, 4, s));
  if (B.sam) {                                                 // a SAM decode: the same outputs from the text
    const int src = mcov_sam_gpu_names_seq(ctx, k_len, win_bases, d_hash, d_kmer, d_win);
    if (src) return src;
  } else {
    MCOV_LAUNCH(ctx, kKBamNamesSeq, (k_bam_names_seq<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(
        B.data.as<uint8_t>(), B.rec_off.as<uint64_t>(), n, k_len, win_bases, d_hash, d_kmer, d_win, B.status.as<int>())));
  }
  CUB(cudaGetLastError());
  int bad = 0;
  CUB(cudaMemcpyAsync(&bad, B.status.as<int>() + 2, 4, cudaMemcpyDeviceToHost, s));
  if (!dev) {
    if (name_hash_out) CUB(cudaMemcpyAsync(name_hash_out, d_hash, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    if (kmer_code_out) CUB(cudaMemcpyAsync(kmer_code_out, d_kmer, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
    if (seq_win_out) CUB(cudaMemcpyAsync(seq_win_out, d_win, (size_t)n * W, cudaMemcpyDeviceToHost, s));
  }
  CUB(cudaStreamSynchronize(s));
  if (bad) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_gpu_names_seq: a record's SEQ leaves the record");
  return MCOV_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Streamed decode: a BAM of ANY size, chunk by chunk through the GPU decoder into the streamed depth pass.  Per chunk:
// the complete BGZF blocks of `chunk_bytes` of file go to the device and are inflated BEHIND the bytes of the record the
// previous chunk ended in (so every chunk's stream begins on a record border and its chain has a known head), the
// record chain is established as above but may stop in front of a record that continues in the next chunk, the columns
// are written behind the reads carried over from the previous batch, and the batch goes to mcov_stream_push from device
// memory.  The next chunk of the file is read (a host thread, into the other pinned buffer) while the GPU works.
// Replaces the `cnext()` loop of reference metacov/scan.pyx:653-667 over a file that is never held, for the coverage
// path, with the host doing nothing but read().
// ---------------------------------------------------------------------------------------------------------------------
#include <cstdio>
#include <future>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

// The whole-file decode straight from the file: the image is mapped (page cache, no copy into a host buffer of the
// caller's) and handed to mcov_bam_decode_gpu.
extern "C" int mcov_bam_decode_gpu_file(mcov_ctx* ctx, const char* path, int verify_crc, mcov_bam_dev* out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!path || !out) return bfail(ctx, MCOV_ERR_ARG, "mcov_bam_decode_gpu_file: bad arguments");
  const int fd = ::open(path, O_RDONLY);
  if (fd < 0) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu_file: cannot open the file");
  struct stat st;
  if (::fstat(fd, &st) != 0 || st.st_size <= 0) { ::close(fd); return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu_file: empty or unreadable file"); }
  void* map = ::mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
  ::close(fd);
  if (map == MAP_FAILED) return bfail(ctx, MCOV_ERR_IO, "mcov_bam_decode_gpu_file: cannot map the file");
  const int rc = mcov_bam_decode_gpu(ctx, map, (int64_t)st.st_size, verify_crc, out);
  ::munmap(map, (size_t)st.st_size);
  return rc;
}

// The chunk loop of the streamed decode: every chunk inflated, chained and written into columns behind the reads the
// sink carried, then handed to the sink.  The depth pass (mcov_bam_gpu_stream_depth) and the base counts
// (mcov_base_counts) are its two consumers.
int mcov::bam_gpu_chunks(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, int verify_crc, mcov_bam_gpu_stream_info* info,
                         const char* who, BamChunkSink& sink) {
  auto F = [&](int code, const char* why) { ctx->err = std::string(who) + ": " + why; return code; };
  if (chunk_bytes <= 0) chunk_bytes = 64ll << 20;
  chunk_bytes = std::max<int64_t>(chunk_bytes, 1 << 17);          // at least one BGZF block (<= 64 KiB) beside a leftover
  CUB(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  mcov_ctx::BamDev& B = ctx->bam;
  B.n_rec = -1;                                                   // (the whole-file decode's columns are gone after this)
  B.sam = false;
  FILE* fh = std::fopen(path, "rb");
  if (!fh) return F(MCOV_ERR_IO, "cannot open the file");
  struct Closer { FILE* f; ~Closer() { if (f) std::fclose(f); } } closer{fh};
  // a file smaller than the chunk: buffers no larger than the file needs.  The two host buffers are PINNED only for a long
  // stream (>= 1 GiB of file): pinning costs 0.6 - 2.4 ms per MB on these boxes (and as much again to free), which a short
  // file never earns back -- its chunks go through the driver's own staging (still faster than the inflate consumes them)
  long long fsz = -1;
  if (std::fseek(fh, 0, SEEK_END) == 0) {
    fsz = (long long)std::ftell(fh);
    if (fsz > 0 && fsz + 1 < chunk_bytes) chunk_bytes = std::max<int64_t>(fsz + 1, 1 << 17);
    std::rewind(fh);
  }
  static const bool force_pin = std::getenv("MCOV_STREAM_PIN") != nullptr;     // test / tuning hook: pinned buffers whatever the size
  const bool pin = force_pin || fsz >= (1ll << 30);
  // two pinned buffers: [leftover of an incomplete block | chunk_bytes of file]
  const size_t cap = (size_t)chunk_bytes + (1u << 17);
  CUB(B.pin[0].ensure(cap, pin)); CUB(B.pin[1].ensure(cap, pin));
  CUB(B.status.ensure(64));
  auto read_into = [fh](uint8_t* dst, size_t want) -> size_t { return std::fread(dst, 1, want, fh); };
  int rc = sink.begin(ctx);
  if (rc) return rc;
  int cur = 0;
  size_t left = 0;                                                // bytes of an incomplete block at the front of pin[cur]
  size_t got = read_into(B.pin[0].as<uint8_t>(), (size_t)chunk_bytes);
  bool eof = got < (size_t)chunk_bytes;
  uint64_t tail_len = 0;                                          // bytes of the record the previous chunk ended in (in B.tail)
  int64_t n_carry = 0, carry_ops = 0;
  int32_t n_ref = -1;
  bool first = true, pushed_last = false;
  std::vector<BgzfBlock> blocks;
  std::vector<WalkSeg> segs;
  std::vector<WalkOut> wo;
  while (!pushed_last) {
    uint8_t* raw = B.pin[cur].as<uint8_t>();
    const size_t have = left + got;
    // the next chunk of the file, behind the bytes this one will leave over (their number is known once the blocks are indexed)
    uint64_t total = 0;
    size_t consumed = 0;
    if (!bgzf_index(raw, have, tail_len, true, blocks, total, consumed)) return F(MCOV_ERR_IO, "not a valid BGZF file");
    if (eof && consumed != have) return F(MCOV_ERR_IO, "the file ends inside a BGZF block");
    if (!eof && consumed == 0) return F(MCOV_ERR_IO, "a BGZF block larger than the chunk");
    const size_t next_left = have - consumed;
    std::future<size_t> next_read;
    const bool was_eof = eof;
    if (!eof) {
      uint8_t* nxt = B.pin[cur ^ 1].as<uint8_t>();
      std::memcpy(nxt, raw + consumed, next_left);
      next_read = std::async(std::launch::async, read_into, nxt + next_left, (size_t)chunk_bytes);
    }
    const int64_t nb = (int64_t)blocks.size();
    int err_rc = MCOV_OK;
    do {                                                          // (one pass; `break` = leave with err_rc set, after joining the reader)
      // inflate behind the carried record bytes
      if (B.raw.ensure(consumed + 16) != cudaSuccess || B.blocks.ensure((size_t)std::max<int64_t>(nb, 1) * sizeof(BgzfBlock)) != cudaSuccess ||
          B.data.ensure((size_t)total + 64) != cudaSuccess) { err_rc = F(MCOV_ERR_NOMEM, "out of device memory"); break; }
      if (tail_len) cudaMemcpyAsync(B.data.p, B.tail.p, (size_t)tail_len, cudaMemcpyDeviceToDevice, s);
      if (consumed) cudaMemcpyAsync(B.raw.p, raw, consumed, cudaMemcpyHostToDevice, s);
      cudaMemsetAsync(B.status.p, 0, 64, s);
      if (nb) {
        cudaMemcpyAsync(B.blocks.p, blocks.data(), (size_t)nb * sizeof(BgzfBlock), cudaMemcpyHostToDevice, s);
        MCOV_LAUNCH(ctx, kKBgzfInflate, (k_bgzf_inflate<<<(unsigned)((nb + kInflateGroupsPerCta - 1) / kInflateGroupsPerCta), kInflateThreads, 0, s>>>(
            B.raw.as<uint8_t>(), B.blocks.as<BgzfBlock>(), nb, B.data.as<uint8_t>(), verify_crc, B.status.as<int>())));
      }
      if (cudaGetLastError() != cudaSuccess) { err_rc = F(MCOV_ERR_CUDA, "inflate launch failed"); break; }
      uint64_t rec_begin = 0;
      if (first) {
        if (total < 12) { err_rc = F(MCOV_ERR_IO, "not a valid BAM file"); break; }
        err_rc = bam_dev_header(ctx, total, &rec_begin, &n_ref);             // (a header that does not fit the first chunk reads as truncated)
        if (err_rc) break;
        if (n_ref != ctx->n_contigs) { err_rc = F(MCOV_ERR_ARG, "the context's contig table is not this file's"); break; }
        first = false;
      } else {
        int st2[2] = {0, 0};
        cudaMemcpyAsync(st2, B.status.p, sizeof(st2), cudaMemcpyDeviceToHost, s);
        if (cudaStreamSynchronize(s) != cudaSuccess) { err_rc = F(MCOV_ERR_CUDA, "inflate failed"); break; }
        if (st2[0]) { err_rc = F(MCOV_ERR_IO, st2[0] == 100 ? "CRC mismatch in a BGZF block" : "corrupt deflate stream in a BGZF block"); break; }
      }
      // the record chain of this chunk
      uint64_t chain_end = rec_begin;
      segs.clear(); wo.clear();
      if (total > rec_begin) { err_rc = bam_dev_chain(ctx, total, rec_begin, n_ref, !was_eof, segs, wo, &chain_end); if (err_rc) break; }
      // The chain may stop in front of a record that continues in the next chunk: the write pass must stop there too.  (Its
      // walk runs to the segment's limit; left at `total` it parsed the cut record -- with fewer than 36 of its bytes present
      // it took the op count from whatever lay behind the stream and wrote that many "ops" past the end of the op column.)
      if (!segs.empty()) segs.back().limit = chain_end;
      uint64_t n_rec = 0, n_cig = 0;
      for (size_t i = 0; i < segs.size(); ++i) { segs[i].rec_base = (uint64_t)n_carry + n_rec; segs[i].cig_base = (uint64_t)carry_ops + n_cig; n_rec += wo[i].n_rec; n_cig += wo[i].n_cig; }
      const uint64_t n_tot = (uint64_t)n_carry + n_rec, ops_tot = (uint64_t)carry_ops + n_cig;
      if (ops_tot > 0xFFFFFFF0ull || n_tot > 0x7FFFFFF0ull) { err_rc = F(MCOV_ERR_RANGE, "a chunk holds too many records; use a smaller chunk"); break; }
      // the bytes of the record this chunk ends in: kept for the front of the next chunk's stream
      const uint64_t new_tail = total - chain_end;
      if (new_tail) {
        if (B.tail2.ensure((size_t)new_tail) != cudaSuccess) { err_rc = F(MCOV_ERR_NOMEM, "out of device memory"); break; }
        cudaMemcpyAsync(B.tail2.p, B.data.as<uint8_t>() + chain_end, (size_t)new_tail, cudaMemcpyDeviceToDevice, s);
      }
      // columns: [carried reads | this chunk's]
      SoaOut o;
      const cudaError_t ce = bam_dev_columns(ctx, segs, n_tot, ops_tot, o);
      if (ce != cudaSuccess) { err_rc = ce == cudaErrorMemoryAllocation ? F(MCOV_ERR_NOMEM, "out of device memory") : F(MCOV_ERR_CUDA, "record walk failed"); break; }
      if (n_carry) {
        cudaMemcpyAsync(B.tid.p, B.c_tid.p, (size_t)n_carry * 4, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.pos.p, B.c_pos.p, (size_t)n_carry * 4, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.flag.p, B.c_flag.p, (size_t)n_carry * 2, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.mapq.p, B.c_mapq.p, (size_t)n_carry, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.cig_off.p, B.c_off.p, (size_t)n_carry * 4, cudaMemcpyDeviceToDevice, s);
        if (carry_ops) cudaMemcpyAsync(B.cig.p, B.c_cig.p, (size_t)carry_ops * 4, cudaMemcpyDeviceToDevice, s);
      }
      if (cudaStreamSynchronize(s) != cudaSuccess) { err_rc = F(MCOV_ERR_CUDA, "record walk failed"); break; }
      std::swap(B.tail, B.tail2);
      info->inflated_bytes += (int64_t)(total - tail_len);
      tail_len = new_tail;
      if (was_eof && tail_len) { err_rc = F(MCOV_ERR_IO, "the last BAM record is truncated"); break; }
      // the batch -> the consumer
      BamChunk bc;
      bc.n = (int64_t)n_tot; bc.n_carry = n_carry; bc.n_ops = (int64_t)ops_tot;
      bc.tid = o.tid; bc.pos = o.pos; bc.flag = o.flag; bc.mapq = o.mapq; bc.l_seq = o.l_seq; bc.cig_off = o.cig_off; bc.cig = o.cig;
      bc.data = B.data.as<uint8_t>(); bc.rec_off = o.rec_off; bc.last = was_eof;
      err_rc = sink.batch(ctx, bc, &n_carry, &carry_ops);
      if (err_rc) break;
      info->n_records += (int64_t)n_rec; info->n_chunks += 1; info->n_segments += (int64_t)segs.size();
      info->file_bytes += (int64_t)consumed;
      info->max_carry = std::max<int64_t>(info->max_carry, n_carry);
      if (was_eof) { pushed_last = true; break; }
    } while (false);
    if (next_read.valid()) {                                      // always join the reader before leaving or going on
      got = next_read.get();
      eof = got < (size_t)chunk_bytes;
      left = next_left;
      cur ^= 1;
    }
    if (err_rc) return err_rc;
  }
  return MCOV_OK;
}

namespace {

// The streamed depth pass as a consumer of the chunk loop: every batch goes to mcov_stream_push, and what the next batch
// must begin with is the suffix from the first read that starts at / reaches past the pass's resend point.
struct DepthSink : mcov::BamChunkSink {
  int32_t rt = -1, rp = 0;
  int begin(mcov_ctx* ctx) override { return mcov_stream_begin(ctx); }
  int batch(mcov_ctx* ctx, const BamChunk& b, int64_t* n_carry_out, int64_t* carry_ops_out) override {
    cudaStream_t s = ctx->stream;
    mcov_ctx::BamDev& B = ctx->bam;
    const int last = b.last ? 1 : 0;
    int rc = mcov_stream_push(ctx, b.n, b.n_carry, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, MCOV_MEM_DEVICE, last, &rt, &rp);
    if (rc) return rc;
    *n_carry_out = 0; *carry_ops_out = 0;
    if (last) return MCOV_OK;
    const uint64_t n_tot = (uint64_t)b.n, ops_tot = (uint64_t)b.n_ops;
    if (n_tot) {
      unsigned long long* d_first = reinterpret_cast<unsigned long long*>(B.status.as<int>() + 4);
      const unsigned long long init = n_tot;
      cudaMemcpyAsync(d_first, &init, 8, cudaMemcpyHostToDevice, s);
      k_bam_carry_first<<<(unsigned)((n_tot + 255) / 256), 256, 0, s>>>((int64_t)n_tot, b.tid, b.pos, b.cig_off, b.cig, rt, rp, ctx->n_contigs, d_first);
      unsigned long long j0 = n_tot;
      cudaMemcpyAsync(&j0, d_first, 8, cudaMemcpyDeviceToHost, s);
      if (cudaStreamSynchronize(s) != cudaSuccess) return bfail(ctx, MCOV_ERR_CUDA, "mcov_bam_gpu_stream_depth: carry selection failed");
      if (j0 < n_tot) {
        uint32_t o0 = 0;
        cudaMemcpyAsync(&o0, b.cig_off + j0, 4, cudaMemcpyDeviceToHost, s);
        cudaStreamSynchronize(s);
        const int64_t n_carry = (int64_t)(n_tot - j0), carry_ops = (int64_t)ops_tot - (int64_t)o0;
        const bool okm = B.c_tid.ensure((size_t)n_carry * 4) == cudaSuccess && B.c_pos.ensure((size_t)n_carry * 4) == cudaSuccess &&
                         B.c_flag.ensure((size_t)n_carry * 2) == cudaSuccess && B.c_mapq.ensure((size_t)n_carry) == cudaSuccess &&
                         B.c_off.ensure((size_t)n_carry * 4) == cudaSuccess && B.c_cig.ensure((size_t)std::max<int64_t>(carry_ops, 1) * 4) == cudaSuccess;
        if (!okm) return bfail(ctx, MCOV_ERR_NOMEM, "mcov_bam_gpu_stream_depth: out of device memory");
        cudaMemcpyAsync(B.c_tid.p, b.tid + j0, (size_t)n_carry * 4, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.c_pos.p, b.pos + j0, (size_t)n_carry * 4, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.c_flag.p, b.flag + j0, (size_t)n_carry * 2, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(B.c_mapq.p, b.mapq + j0, (size_t)n_carry, cudaMemcpyDeviceToDevice, s);
        k_bam_rebase_offsets<<<(unsigned)((n_carry + 255) / 256), 256, 0, s>>>(n_carry, b.cig_off + j0, o0, B.c_off.as<uint32_t>());
        if (carry_ops) cudaMemcpyAsync(B.c_cig.p, b.cig + o0, (size_t)carry_ops * 4, cudaMemcpyDeviceToDevice, s);
        *n_carry_out = n_carry; *carry_ops_out = carry_ops;
      }
    }
    if (cudaGetLastError() != cudaSuccess) return bfail(ctx, MCOV_ERR_CUDA, "mcov_bam_gpu_stream_depth: carry copy failed");
    return MCOV_OK;
  }
};

}  // namespace

extern "C" int mcov_bam_gpu_stream_depth(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, int verify_crc,
                                         mcov_bam_gpu_stream_info* info) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!path || !info) return bfail(ctx, MCOV_ERR_ARG, "mcov_bam_gpu_stream_depth: bad arguments");
  std::memset(info, 0, sizeof(*info));
  DepthSink sink;
  return bam_gpu_chunks(ctx, path, chunk_bytes, verify_crc, info, "mcov_bam_gpu_stream_depth", sink);
}

// The device decoder compiled for the host: lets the CPU test suite check inflate.cuh against zlib
// without a GPU (test hooks, not a product path).
extern "C" int mcov_inflate_host(const uint8_t* src, uint32_t clen, uint8_t* dst, uint32_t ulen) {
  if ((!src && clen) || (!dst && ulen)) return -1;
  uint16_t tabs[kInfTabWords];
  return inflate_raw(src, clen, dst, ulen, tabs);
}
extern "C" int mcov_inflate_host_win(const uint8_t* src, uint32_t clen, uint8_t* dst, uint32_t ulen, uint32_t window) {
  if ((!src && clen) || (!dst && ulen) || window < 1024 || (window & (window - 1))) return -1;
  uint16_t tabs[kInfTabWords];
  std::vector<uint8_t> win(window);
  return inflate_raw(src, clen, dst, ulen, tabs, 0, 1, win.data(), window - 1);
}
extern "C" uint32_t mcov_crc32_host(const uint8_t* p, uint32_t n) { return crc32_bytes(p, n); }
extern "C" uint32_t mcov_crc32_sliced_host(const uint8_t* p, uint32_t n, int nlanes) { return crc32_sliced_host(p, n, nlanes < 1 ? 1 : nlanes); }
