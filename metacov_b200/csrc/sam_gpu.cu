// sam_gpu.cu -- SAM text parsed on the GPU into the columns of a GPU-decoded BAM (mcov_bam_dev).
//
// The header (the '@' lines at the start of the file) is read on the host from the mapped image; the whole file goes to
// the device in chunks, and everything past the header is parsed there:
//
//   k_sam_nl_count    newlines per 32 KiB tile (16-byte loads, SWAR byte compare, popc), launched chunk by chunk behind
//                     the copy of each chunk; an exclusive scan of the tile counts (CUB) places every tile's lines
//   k_sam_nl_write    the position of every newline, in order: the line index (u64, files past 4 GiB)
//   k_sam_fields      one warp per line: lanes load 16 B each and ballots find the TABs, lanes 0-10 validate and convert
//                     the 11 mandatory fields at once (RNAME through a hash table of the @SQ names, exact compare), the
//                     warp counts and validates the CIGAR ops 32 bytes per step
//   k_sam_cigar       one warp per line again, behind a scan of the op counts: every op letter found by ballot takes the
//                     digits in front of it, and the op goes to its slot (a 100 KB CIGAR is 32 lanes' work, not one's)
//   k_sam_names_seq   read-name hashes, k-mer keys and SEQ windows (the outputs of k_bam_names_seq) from the text
//   k_sam_line_max    the longest line of a chunk of a stream, from its line index (mcov_sam_chunk_longest_line)
//
// A decode is a header part (sam_upload_header: the @SQ table) and a lines part (sam_decode_lines: everything above).  A
// file is one of each; a stream (mcov_sam_chunk_begin / mcov_sam_chunk_decode) is one header part and a lines part per
// chunk of whole lines, with indices local to the chunk.
//
// Validation failures do not stop the kernels: each one takes the smallest (record, field) with atomicMin, and the host
// reports that line.  The per-field rules live in k_sam.cuh, shared with the host-compiled test hook mcov_sam_parse_host.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <cub/device/device_scan.cuh>
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "ctx.cuh"
#include "k_sam.cuh"

namespace mcov {

constexpr int kSamThreads = 256;
constexpr int kSamRounds = 8;                                          // 16-byte loads per thread and tile
constexpr uint64_t kSamTile = (uint64_t)kSamThreads * 16 * kSamRounds; // 32 KiB
constexpr int kSamWarps = kSamThreads / 32;

// 16-bit mask of the bytes of v equal to c (exact SWAR zero-byte test per 32-bit word)
__device__ __forceinline__ uint32_t byte_eq_mask16(uint4 v, uint32_t c) {
  const uint32_t rep = c * 0x01010101u;
  const uint32_t w[4] = {v.x ^ rep, v.y ^ rep, v.z ^ rep, v.w ^ rep};
  uint32_t m = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t z = ~(((w[k] & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | w[k] | 0x7F7F7F7Fu);   // 0x80 in every zero byte
    m |= (((z >> 7) & 1u) | ((z >> 14) & 2u) | ((z >> 21) & 4u) | ((z >> 28) & 8u)) << (4 * k);
  }
  return m;
}

// newlines of the 16 bytes at q that lie in [lo, hi)
__device__ __forceinline__ uint32_t nl_mask(const uint8_t* __restrict__ d, uint64_t q, uint64_t lo, uint64_t hi) {
  if (q >= hi || q + 16 <= lo) return 0;
  uint32_t m = byte_eq_mask16(*reinterpret_cast<const uint4*>(d + q), '\n');
  if (q < lo) m &= 0xFFFFu << (uint32_t)(lo - q);
  if (hi - q < 16) m &= (1u << (uint32_t)(hi - q)) - 1u;
  return m;
}

// newlines in [lo, hi) of tiles [t0, t0 + gridDim.x)
__global__ void __launch_bounds__(kSamThreads)
k_sam_nl_count(const uint8_t* __restrict__ d, uint64_t lo, uint64_t hi, uint64_t t0, unsigned long long* __restrict__ cnt) {
  using BR = cub::BlockReduce<uint32_t, kSamThreads>;
  __shared__ typename BR::TempStorage tmp;
  const uint64_t t = t0 + blockIdx.x, base = t * kSamTile;
  uint32_t c = 0;
#pragma unroll
  for (int r = 0; r < kSamRounds; ++r) c += __popc(nl_mask(d, base + ((uint64_t)r * kSamThreads + threadIdx.x) * 16, lo, hi));
  const uint32_t tot = BR(tmp).Sum(c);
  if (threadIdx.x == 0) cnt[t] = tot;
}

// every newline of tile t at line_end[off[t] + k], in file order
__global__ void __launch_bounds__(kSamThreads)
k_sam_nl_write(const uint8_t* __restrict__ d, uint64_t lo, uint64_t hi, const unsigned long long* __restrict__ off,
               uint64_t* __restrict__ line_end) {
  using BS = cub::BlockScan<uint32_t, kSamThreads>;
  __shared__ typename BS::TempStorage tmp;
  const uint64_t t = blockIdx.x, base = t * kSamTile;
  uint64_t o = off[t];
  for (int r = 0; r < kSamRounds; ++r) {
    const uint64_t q = base + ((uint64_t)r * kSamThreads + threadIdx.x) * 16;
    uint32_t m = nl_mask(d, q, lo, hi), ex = 0, agg = 0;
    BS(tmp).ExclusiveSum((uint32_t)__popc(m), ex, agg);
    uint64_t k = o + ex;
    while (m) { line_end[k++] = q + (uint64_t)(__ffs(m) - 1); m &= m - 1u; }
    o += agg;
    __syncthreads();                                                   // (tmp is reused by the next round)
  }
}

struct SamOut {
  int32_t* tid; int32_t* pos; uint16_t* flag; uint8_t* mapq; int32_t* l_seq; int32_t* isize;
  uint64_t* rec_off; SamAux* aux; unsigned long long* ops;
};

__device__ __forceinline__ void sam_fail(unsigned long long* err, int64_t i, int code) {
  atomicMin(err, ((unsigned long long)i << 8) | (unsigned)code);
}

__device__ __forceinline__ bool is_digit(uint32_t c) { return c - '0' <= 9u; }

// One warp per line: TABs, the 11 mandatory fields, the op count of the CIGAR.
__global__ void __launch_bounds__(kSamThreads)
k_sam_fields(const uint8_t* __restrict__ d, uint64_t body, const uint64_t* __restrict__ line_end, int64_t n_rec,
             SamRefTable refs, SamOut o, unsigned long long* __restrict__ err) {
  __shared__ uint32_t s_tab[kSamWarps][12];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * kSamWarps + wid;
  if (i >= n_rec) return;
  const uint64_t start = i ? line_end[i - 1] + 1 : body;
  uint64_t end = line_end[i];
  if (end > start && d[end - 1] == '\r') --end;
  int code = -1;
  if (end == start) code = kErrFewFields;
  else if (end - start > 0xFFFFFFF0ull) code = kErrLineLong;
  else if (d[start] == '@') code = kErrHeaderAfter;
  uint32_t found = 0;
  if (code < 0) {
    for (uint64_t w = start & ~15ull; w < end && found < 11; w += 512) {
      const uint64_t q = w + 16 * (uint64_t)lane;
      uint32_t m = 0;
      if (q < end) {
        m = byte_eq_mask16(*reinterpret_cast<const uint4*>(d + q), '\t');
        if (q < start) m &= 0xFFFFu << (uint32_t)(start - q);
        if (end - q < 16) m &= (1u << (uint32_t)(end - q)) - 1u;
      }
      const uint32_t cnt = __popc(m);
      uint32_t incl = cnt;
#pragma unroll
      for (int s = 1; s < 32; s <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, incl, s); if (lane >= s) incl += v; }
      uint32_t idx = found + incl - cnt;
      while (m && idx < 11) { s_tab[wid][idx++] = (uint32_t)(q + (uint64_t)(__ffs(m) - 1) - start); m &= m - 1u; }
      found += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    if (found < 10) code = kErrFewFields;
  }
  if (code >= 0) {                                                     // (the whole warp takes this branch)
    if (lane == 0) { sam_fail(err, i, code); o.ops[i] = 0; o.rec_off[i] = start; o.aux[i] = SamAux{0, 0, 0, 0}; }
    return;
  }
  const uint32_t len = (uint32_t)(end - start);
  const uint8_t* L = d + start;
  auto fb = [&](int f) -> uint32_t { return f ? s_tab[wid][f - 1] + 1 : 0u; };
  auto fe = [&](int f) -> uint32_t { return (uint32_t)f < found ? s_tab[wid][f] : len; };
  // lanes 0-10: one field each
  int64_t v = 0;
  bool bad = false;
  if (lane < kSamFields && lane != kCigar) {
    const uint32_t b = fb(lane), n = fe(lane) - b;
    if (lane == kRname) {
      v = sam_is_star(L + b, n) ? -1 : sam_ref_lookup(refs, L + b, n);
      bad = n == 0 || (v < 0 && !sam_is_star(L + b, n));
    } else {
      const uint32_t sb = fb(kSeq), sn = fe(kSeq) - sb;
      bad = !sam_field_value(lane, L + b, n, sam_is_star(L + sb, sn) ? 0 : sn, &v);
    }
  }
  // the whole warp: CIGAR ops, 32 bytes per step
  const uint32_t cb = fb(kCigar), ce = fe(kCigar);
  uint32_t n_op = 0;
  bool cbad = ce == cb;
  if (!cbad && !sam_is_star(L + cb, ce - cb)) {
    uint32_t carry = 0;
    for (uint32_t w = cb; w < ce; w += 32) {
      const uint32_t q = w + lane;
      const uint32_t c = q < ce ? L[q] : 0u;
      uint32_t prev = __shfl_up_sync(0xffffffffu, c, 1);
      if (lane == 0) prev = carry;
      const bool isop = q < ce && sam_cigar_op(c) >= 0;
      if (q < ce && !isop && !is_digit(c)) cbad = true;
      if (isop && !is_digit(prev)) cbad = true;                        // every op has a length
      n_op += __popc(__ballot_sync(0xffffffffu, isop));
      carry = __shfl_sync(0xffffffffu, c, 31);
    }
    if (sam_cigar_op(L[ce - 1]) < 0) cbad = true;
  }
  const unsigned badm = __ballot_sync(0xffffffffu, bad) | (__any_sync(0xffffffffu, cbad) ? (1u << kCigar) : 0u);
  const int64_t flag = __shfl_sync(0xffffffffu, v, kFlag), tid = __shfl_sync(0xffffffffu, v, kRname);
  const int64_t pos = __shfl_sync(0xffffffffu, v, kPos), mapq = __shfl_sync(0xffffffffu, v, kMapq);
  const int64_t tlen = __shfl_sync(0xffffffffu, v, kTlen), lseq = __shfl_sync(0xffffffffu, v, kSeq);
  if (lane == 0) {
    if (badm) sam_fail(err, i, __ffs(badm) - 1);
    o.tid[i] = (int32_t)tid; o.pos[i] = (int32_t)pos; o.flag[i] = (uint16_t)flag; o.mapq[i] = (uint8_t)mapq;
    o.l_seq[i] = (int32_t)lseq; o.isize[i] = (int32_t)tlen; o.rec_off[i] = start;
    o.ops[i] = badm ? 0u : n_op;
    o.aux[i] = SamAux{fe(kQname), cb, ce, fb(kSeq)};
  }
}

// One warp per line: the ops of the CIGAR at their offsets (o.ops scanned), and the 32-bit offset column.
__global__ void __launch_bounds__(kSamThreads)
k_sam_cigar(const uint8_t* __restrict__ d, int64_t n_rec, const uint64_t* __restrict__ rec_off, const SamAux* __restrict__ aux,
            const unsigned long long* __restrict__ ops, uint32_t* __restrict__ cig_off, uint32_t* __restrict__ cig,
            unsigned long long* __restrict__ err) {
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * kSamWarps + wid;
  if (i >= n_rec) return;
  const uint64_t o0 = ops[i];
  if (lane == 0) cig_off[i] = (uint32_t)o0;
  if (ops[i + 1] == o0) return;                                        // no ops ('*', or a record that failed)
  const uint8_t* L = d + rec_off[i];
  const SamAux a = aux[i];
  uint64_t k0 = o0;
  bool bad = false;
  for (uint32_t w = a.cig_b; w < a.cig_e; w += 32) {
    const uint32_t q = w + lane;
    const int op = q < a.cig_e ? sam_cigar_op(L[q]) : -1;
    const unsigned m = __ballot_sync(0xffffffffu, op >= 0);
    if (op >= 0) {
      uint64_t len = 0, scale = 1;
      for (uint32_t p = q; p > a.cig_b && is_digit(L[p - 1]); --p) {
        const uint32_t c = L[p - 1] - '0';
        if (c && scale > kSamMaxOpLen) { bad = true; break; }          // a nonzero digit beyond the range
        len += c * scale;
        if (len > kSamMaxOpLen) { bad = true; break; }
        if (scale <= kSamMaxOpLen) scale *= 10;
      }
      cig[k0 + __popc(m & ((1u << lane) - 1u))] = (uint32_t)(len << 4) | (uint32_t)op;
    }
    k0 += __popc(m);
  }
  if (bad) sam_fail(err, i, kCigar);
}

__global__ void k_sam_names_seq(const uint8_t* __restrict__ d, const uint64_t* __restrict__ rec_off, const SamAux* __restrict__ aux,
                                const int32_t* __restrict__ l_seq, const uint16_t* __restrict__ flag, const uint32_t* __restrict__ cig_off,
                                const uint32_t* __restrict__ cig, int64_t n, int32_t k_len, int32_t win_bases,
                                uint64_t* __restrict__ name_hash, int32_t* __restrict__ kmer_code, uint8_t* __restrict__ win) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* L = d + rec_off[i];
  const SamAux a = aux[i];
  const uint32_t c0 = cig_off[i];
  sam_names_seq_one(L, a.l_qname, L + a.seq_b, l_seq[i], flag[i], cig + c0, cig_off[i + 1] - c0, k_len, win_bases,
                    name_hash ? name_hash + i : nullptr, kmer_code ? kmer_code + i : nullptr,
                    win ? win + (size_t)i * ((win_bases + 1) / 2) : nullptr);
}

// The index statistics of pysam's mapped / unmapped from decoded columns: placed records without 0x4, and the rest.
__global__ void __launch_bounds__(256)
k_dev_map_counts(const int32_t* __restrict__ tid, const uint16_t* __restrict__ flag, int64_t n, unsigned long long* __restrict__ out) {
  using BR = cub::BlockReduce<uint32_t, 256>;
  __shared__ typename BR::TempStorage tmp;
  uint32_t m = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    m += (tid[i] >= 0 && !(flag[i] & 4u)) ? 1u : 0u;
  const uint32_t tot = BR(tmp).Sum(m);
  if (threadIdx.x == 0 && tot) atomicAdd(out, (unsigned long long)tot);
}

// The longest line of a chunk, its LF included (a last line without one: up to the end of the text); from the line index.
__global__ void __launch_bounds__(256)
k_sam_line_max(const uint64_t* __restrict__ line_end, int64_t n_rec, uint64_t body, uint64_t n, unsigned long long* __restrict__ out) {
  using BR = cub::BlockReduce<unsigned long long, 256>;
  __shared__ typename BR::TempStorage tmp;
  unsigned long long m = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t start = i ? line_end[i - 1] + 1 : body;
    m = max(m, (unsigned long long)(min(line_end[i] + 1, n) - start));
  }
  const unsigned long long b = BR(tmp).Reduce(m, cub::Max());
  if (threadIdx.x == 0 && b) atomicMax(out, b);
}

// ---- host side ------------------------------------------------------------------------------------

// The header: the '@' lines in front of the first record.  References from @SQ SN:/LN:, in order.
struct SamHeader {
  uint64_t body = 0;                 // offset of the first record line
  int64_t lines = 0;                 // header lines
  std::vector<std::string> names;
  std::vector<int32_t> lens;
  std::string err;
};

static bool sam_parse_header(const uint8_t* d, uint64_t n, SamHeader& h) {
  uint64_t p = 0;
  std::vector<std::string> seen;
  while (p < n && d[p] == '@') {
    const uint8_t* nl = static_cast<const uint8_t*>(std::memchr(d + p, '\n', (size_t)(n - p)));
    const uint64_t e0 = nl ? (uint64_t)(nl - d) : n;
    uint64_t e = e0;
    if (e > p && d[e - 1] == '\r') --e;
    ++h.lines;
    if (e - p >= 4 && std::memcmp(d + p, "@SQ\t", 4) == 0) {
      std::string sn;
      bool has_sn = false, has_ln = false;
      uint64_t ln = 0;
      bool ln_ok = false;
      for (uint64_t f = p + 4; f <= e;) {
        uint64_t g = f;
        while (g < e && d[g] != '\t') ++g;
        if (g - f >= 3 && d[f] == 'S' && d[f + 1] == 'N' && d[f + 2] == ':') { sn.assign((const char*)d + f + 3, g - f - 3); has_sn = true; }
        if (g - f >= 3 && d[f] == 'L' && d[f + 1] == 'N' && d[f + 2] == ':') { has_ln = true; ln_ok = sam_dec_u(d + f + 3, (uint32_t)std::min<uint64_t>(g - f - 3, 64), 0x7FFFFFFFull, &ln) && ln >= 1; }
        f = g + 1;
      }
      char msg[160];
      if (!has_sn || sn.empty() || !has_ln || !ln_ok) {
        std::snprintf(msg, sizeof msg, "line %lld: @SQ needs SN and an LN in [1, 2^31-1]", (long long)h.lines);
        h.err = msg; return false;
      }
      h.names.push_back(sn);
      h.lens.push_back((int32_t)ln);
    }
    p = nl ? e0 + 1 : n;
  }
  // duplicate names
  std::vector<std::string> sorted = h.names;
  std::sort(sorted.begin(), sorted.end());
  for (size_t k = 1; k < sorted.size(); ++k)
    if (sorted[k] == sorted[k - 1]) { h.err = "duplicate @SQ name " + sorted[k]; return false; }
  h.body = p;
  return true;
}

// The @SQ name table (open addressing, at most half full): slots, name blob, name offsets
struct RefTableHost {
  std::vector<int32_t> slot;
  std::vector<uint8_t> names;
  std::vector<uint64_t> off;
  void build(const std::vector<std::string>& refs) {
    size_t cap = 2;
    while (cap < 2 * refs.size()) cap <<= 1;
    slot.assign(cap, -1);
    off.assign(1, 0);
    names.clear();
    for (size_t r = 0; r < refs.size(); ++r) {
      const std::string& s = refs[r];
      names.insert(names.end(), s.begin(), s.end());
      off.push_back(names.size());
      uint32_t k = sam_name_hash32((const uint8_t*)s.data(), (uint32_t)s.size()) & (uint32_t)(cap - 1);
      while (slot[k] >= 0) k = (k + 1) & (uint32_t)(cap - 1);
      slot[k] = (int32_t)r;
    }
    if (names.empty()) names.push_back(0);
  }
  SamRefTable view() const { return SamRefTable{slot.data(), (uint32_t)(slot.size() - 1), names.data(), off.data()}; }
};

static const char* sam_field_name(int f) {
  static const char* k[] = {"QNAME (1-254 bytes)", "FLAG (0-65535)", "RNAME (an @SQ name or *)", "POS (0-2^31-1)", "MAPQ (0-255)",
                            "CIGAR", "RNEXT", "PNEXT (0-2^31-1)", "TLEN (int32)", "SEQ", "QUAL (* or one per base)",
                            "fewer than 11 fields (or an empty line)", "a header line after a record", "a line of 4 GiB or more"};
  return f >= 0 && f <= kErrLineLong ? k[f] : "?";
}

static std::string sam_err_text(const char* fn, int64_t line, int f) {
  char msg[200];
  std::snprintf(msg, sizeof msg, "%s: line %lld: %s", fn, (long long)line, sam_field_name(f));
  return msg;
}

}  // namespace mcov

using namespace mcov;

#define SCU(call)                                                          \
  do {                                                                     \
    cudaError_t e__ = (call);                                              \
    if (e__ != cudaSuccess) { ctx->err = std::string("mcov_sam_decode_gpu: ") + #call + ": " + cudaGetErrorString(e__); return MCOV_ERR_CUDA; } \
  } while (0)

static int sfail(mcov_ctx* ctx, int code, const std::string& msg) { ctx->err = msg; return code; }

// The header part of a decode: the @SQ name table to the device (B.sam_ref), kept for the lines that follow.
static int sam_upload_header(mcov_ctx* ctx, const SamHeader& h) {
  mcov_ctx::BamDev& B = ctx->bam;
  RefTableHost rt;
  rt.build(h.names);
  const size_t tab_bytes = rt.slot.size() * 4, name_bytes = rt.names.size(), off_bytes = rt.off.size() * 8;
  SCU(B.sam_ref.ensure(tab_bytes + off_bytes + name_bytes + 16));
  uint8_t* refd = B.sam_ref.as<uint8_t>();
  cudaStream_t s = ctx->stream;
  SCU(cudaMemcpyAsync(refd, rt.slot.data(), tab_bytes, cudaMemcpyHostToDevice, s));
  SCU(cudaMemcpyAsync(refd + tab_bytes, rt.off.data(), off_bytes, cudaMemcpyHostToDevice, s));
  SCU(cudaMemcpyAsync(refd + tab_bytes + off_bytes, rt.names.data(), name_bytes, cudaMemcpyHostToDevice, s));
  B.sam_ref_mask = (uint32_t)(rt.slot.size() - 1);
  B.sam_tab_bytes = tab_bytes; B.sam_off_bytes = off_bytes;
  B.sam_n_ref = (int32_t)h.names.size();
  return MCOV_OK;
}

static SamRefTable sam_ref_view(const mcov_ctx::BamDev& B) {
  const uint8_t* refd = B.sam_ref.as<uint8_t>();
  return SamRefTable{reinterpret_cast<const int32_t*>(refd), B.sam_ref_mask, refd + B.sam_tab_bytes + B.sam_off_bytes,
                     reinterpret_cast<const uint64_t*>(refd + B.sam_tab_bytes)};
}

// The lines part of a decode: raw[body, n) holds whole record lines (the last one may lack its LF) and nothing after
// them; it goes to the device with raw[0, body), in copies of `chunk` bytes, and is parsed into the columns.  A malformed
// line is reported as line `line0` + its index + 1 (line0: the lines of the stream in front of raw[body]).
static int sam_decode_lines(mcov_ctx* ctx, const uint8_t* raw, uint64_t n, uint64_t body, uint64_t chunk, int64_t line0,
                            const char* who, mcov_bam_dev* out) {
  cudaStream_t s = ctx->stream;
  mcov_ctx::BamDev& B = ctx->bam;
  // the whole image to the device, chunk by chunk on the copy stream; the newline count of each chunk's tiles follows
  // its copy on the main stream
  const uint64_t n_tiles = (n + kSamTile - 1) / kSamTile;
  chunk = chunk > 0 ? chunk : (64ull << 20);
  chunk = (chunk + kSamTile - 1) / kSamTile * kSamTile;
  SCU(B.data.ensure((size_t)n + 64));
  SCU(B.status.ensure(64));
  SCU(B.sam_tiles.ensure((size_t)(n_tiles + 1) * 8));
  SCU(cudaMemsetAsync(B.data.as<uint8_t>() + n, 0, 64, s));
  SCU(cudaMemsetAsync(B.sam_tiles.p, 0, (size_t)(n_tiles + 1) * 8, s));
  unsigned long long* d_err = reinterpret_cast<unsigned long long*>(B.status.as<int>() + 8);
  SCU(cudaMemsetAsync(d_err, 0xFF, 8, s));
  cudaEvent_t ev = nullptr;
  SCU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  struct EvGuard { cudaEvent_t e; ~EvGuard() { if (e) cudaEventDestroy(e); } } evg{ev};
  SCU(cudaEventRecord(ev, s));                                         // earlier readers of B.data are done first
  SCU(cudaStreamWaitEvent(ctx->copy_stream, ev, 0));
  unsigned long long* tiles = B.sam_tiles.as<unsigned long long>();
  for (uint64_t c0 = 0; c0 < n; c0 += chunk) {
    const uint64_t c1 = std::min(n, c0 + chunk);
    SCU(cudaMemcpyAsync(B.data.as<uint8_t>() + c0, raw + c0, (size_t)(c1 - c0), cudaMemcpyHostToDevice, ctx->copy_stream));
    SCU(cudaEventRecord(ev, ctx->copy_stream));
    SCU(cudaStreamWaitEvent(s, ev, 0));
    const uint64_t t0 = c0 / kSamTile, t1 = (c1 + kSamTile - 1) / kSamTile;
    if (c1 > body)
      MCOV_LAUNCH(ctx, kKSamNlCount, (k_sam_nl_count<<<(unsigned)(t1 - t0), kSamThreads, 0, s>>>(B.data.as<uint8_t>(), body, n, t0, tiles)));
  }
  SCU(cudaGetLastError());
  size_t tb = 0;
  SCU(cub::DeviceScan::ExclusiveSum(nullptr, tb, tiles, tiles, (int64_t)(n_tiles + 1), s));
  SCU(B.sam_tmp.ensure(tb + 16));
  SCU(cub::DeviceScan::ExclusiveSum(B.sam_tmp.p, tb, tiles, tiles, (int64_t)(n_tiles + 1), s));
  unsigned long long n_nl = 0;
  SCU(cudaMemcpyAsync(&n_nl, tiles + n_tiles, 8, cudaMemcpyDeviceToHost, s));
  SCU(cudaStreamSynchronize(s));
  const bool tail = body < n && raw[n - 1] != '\n';                   // a last line without its newline
  const uint64_t n_rec = n_nl + (tail ? 1 : 0);
  SCU(B.sam_lines.ensure((size_t)(n_rec + 1) * 8));
  if (n_nl)
    MCOV_LAUNCH(ctx, kKSamNlWrite, (k_sam_nl_write<<<(unsigned)n_tiles, kSamThreads, 0, s>>>(B.data.as<uint8_t>(), body, n, tiles,
                                                                                         B.sam_lines.as<uint64_t>())));
  if (tail) SCU(cudaMemcpyAsync(B.sam_lines.as<uint64_t>() + n_nl, &n, 8, cudaMemcpyHostToDevice, s));
  // columns
  SCU(B.tid.ensure((n_rec + 4) * 4)); SCU(B.pos.ensure((n_rec + 4) * 4)); SCU(B.flag.ensure((n_rec + 4) * 2)); SCU(B.mapq.ensure(n_rec + 4));
  SCU(B.lseq.ensure((n_rec + 4) * 4)); SCU(B.isize.ensure((n_rec + 4) * 4)); SCU(B.cig_off.ensure((n_rec + 5) * 4));
  SCU(B.rec_off.ensure((n_rec + 4) * 8)); SCU(B.sam_aux.ensure((n_rec + 4) * sizeof(SamAux))); SCU(B.sam_ops.ensure((n_rec + 2) * 8));
  SamOut o;
  o.tid = B.tid.as<int32_t>(); o.pos = B.pos.as<int32_t>(); o.flag = B.flag.as<uint16_t>(); o.mapq = B.mapq.as<uint8_t>();
  o.l_seq = B.lseq.as<int32_t>(); o.isize = B.isize.as<int32_t>(); o.rec_off = B.rec_off.as<uint64_t>(); o.aux = B.sam_aux.as<SamAux>();
  o.ops = B.sam_ops.as<unsigned long long>();
  SCU(cudaMemsetAsync(o.ops + n_rec, 0, 8, s));
  if (n_rec)
    MCOV_LAUNCH(ctx, kKSamFields, (k_sam_fields<<<(unsigned)((n_rec + kSamWarps - 1) / kSamWarps), kSamThreads, 0, s>>>(
        B.data.as<uint8_t>(), body, B.sam_lines.as<uint64_t>(), (int64_t)n_rec, sam_ref_view(B), o, d_err)));
  SCU(cudaGetLastError());
  SCU(cub::DeviceScan::ExclusiveSum(nullptr, tb, o.ops, o.ops, (int64_t)(n_rec + 1), s));
  SCU(B.sam_tmp.ensure(tb + 16));
  SCU(cub::DeviceScan::ExclusiveSum(B.sam_tmp.p, tb, o.ops, o.ops, (int64_t)(n_rec + 1), s));
  unsigned long long hv[2] = {0, 0};                                   // error, op total
  SCU(cudaMemcpyAsync(&hv[0], d_err, 8, cudaMemcpyDeviceToHost, s));
  SCU(cudaMemcpyAsync(&hv[1], o.ops + n_rec, 8, cudaMemcpyDeviceToHost, s));
  SCU(cudaStreamSynchronize(s));
  if (hv[0] != kSamNoErr) return sfail(ctx, MCOV_ERR_IO, sam_err_text(who, line0 + (int64_t)(hv[0] >> 8) + 1, (int)(hv[0] & 255)));
  const uint64_t n_cig = hv[1];
  if (n_cig > 0xFFFFFFFFull) return sfail(ctx, MCOV_ERR_RANGE, std::string(who) + ": more than 2^32-1 CIGAR ops");
  SCU(B.cig.ensure((n_cig + 4) * 4));
  if (n_rec)
    MCOV_LAUNCH(ctx, kKSamCigar, (k_sam_cigar<<<(unsigned)((n_rec + kSamWarps - 1) / kSamWarps), kSamThreads, 0, s>>>(
        B.data.as<uint8_t>(), (int64_t)n_rec, o.rec_off, o.aux, o.ops, B.cig_off.as<uint32_t>(), B.cig.as<uint32_t>(), d_err)));
  SCU(cudaGetLastError());
  const uint32_t last = (uint32_t)n_cig;
  SCU(cudaMemcpyAsync(B.cig_off.as<uint32_t>() + n_rec, &last, 4, cudaMemcpyHostToDevice, s));
  SCU(cudaMemcpyAsync(&hv[0], d_err, 8, cudaMemcpyDeviceToHost, s));
  SCU(cudaStreamSynchronize(s));
  if (hv[0] != kSamNoErr) return sfail(ctx, MCOV_ERR_IO, sam_err_text(who, line0 + (int64_t)(hv[0] >> 8) + 1, (int)(hv[0] & 255)));
  out->n_records = (int64_t)n_rec; out->n_cigar = (int64_t)n_cig; out->n_ref = B.sam_n_ref;
  out->inflated_bytes = (int64_t)n; out->header_bytes = (int64_t)body; out->n_segments = 0;
  out->tid = o.tid; out->pos = o.pos; out->flag = o.flag; out->mapq = o.mapq; out->l_seq = o.l_seq; out->isize = o.isize;
  out->cig_off = B.cig_off.as<uint32_t>(); out->cig = B.cig.as<uint32_t>(); out->inflated = B.data.as<uint8_t>();
  B.n_rec = (int64_t)n_rec;
  B.sam = true;
  return MCOV_OK;
}

extern "C" int mcov_sam_decode_gpu(mcov_ctx* ctx, const void* bytes, int64_t n_bytes, int64_t chunk_bytes, mcov_bam_dev* out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!bytes || n_bytes <= 0 || !out || chunk_bytes < 0) return sfail(ctx, MCOV_ERR_ARG, "mcov_sam_decode_gpu: bad arguments");
  std::memset(out, 0, sizeof(*out));
  SCU(cudaSetDevice(ctx->device));
  mcov_ctx::BamDev& B = ctx->bam;
  B.n_rec = -1;                                                        // (the last decode's columns are overwritten below)
  B.sam = false;
  B.sam_chunked = false;
  const uint8_t* raw = static_cast<const uint8_t*>(bytes);
  SamHeader h;
  if (!sam_parse_header(raw, (uint64_t)n_bytes, h)) return sfail(ctx, MCOV_ERR_IO, "mcov_sam_decode_gpu: " + h.err);
  int rc = sam_upload_header(ctx, h);
  if (rc) return rc;
  return sam_decode_lines(ctx, raw, (uint64_t)n_bytes, h.body, (uint64_t)chunk_bytes, h.lines, "mcov_sam_decode_gpu", out);
}

extern "C" int mcov_sam_chunk_begin(mcov_ctx* ctx, const void* header_bytes, int64_t n, int32_t* n_ref) {
  if (!ctx) return MCOV_ERR_ARG;
  if ((!header_bytes && n) || n < 0) return sfail(ctx, MCOV_ERR_ARG, "mcov_sam_chunk_begin: bad arguments");
  SCU(cudaSetDevice(ctx->device));
  mcov_ctx::BamDev& B = ctx->bam;
  B.n_rec = -1;
  B.sam = false;
  B.sam_chunked = false;
  const uint8_t* raw = static_cast<const uint8_t*>(header_bytes);
  SamHeader h;
  if (!sam_parse_header(raw, (uint64_t)n, h)) return sfail(ctx, MCOV_ERR_IO, "mcov_sam_chunk_begin: " + h.err);
  if (h.body != (uint64_t)n) return sfail(ctx, MCOV_ERR_ARG, "mcov_sam_chunk_begin: the header holds a line that is not a header line");
  int rc = sam_upload_header(ctx, h);
  if (rc) return rc;
  B.sam_line0 = h.lines;
  B.sam_longest = 0;
  B.sam_chunked = true;
  if (n_ref) *n_ref = B.sam_n_ref;
  return MCOV_OK;
}

extern "C" int mcov_sam_chunk_decode(mcov_ctx* ctx, const void* bytes, int64_t n, int last, int64_t* consumed, mcov_bam_dev* out) {
  if (!ctx) return MCOV_ERR_ARG;
  if ((!bytes && n) || n < 0 || !consumed || !out) return sfail(ctx, MCOV_ERR_ARG, "mcov_sam_chunk_decode: bad arguments");
  mcov_ctx::BamDev& B = ctx->bam;
  if (!B.sam_chunked) return sfail(ctx, MCOV_ERR_STATE, "mcov_sam_chunk_decode: call mcov_sam_chunk_begin first");
  std::memset(out, 0, sizeof(*out));
  *consumed = 0;
  SCU(cudaSetDevice(ctx->device));
  const uint8_t* raw = static_cast<const uint8_t*>(bytes);
  uint64_t cut = (uint64_t)n;
  if (!last && n) {
    const void* nl = memrchr(raw, '\n', (size_t)n);
    cut = nl ? (uint64_t)(static_cast<const uint8_t*>(nl) - raw) + 1 : 0;
  }
  B.n_rec = -1;
  B.sam = false;
  ctx->ncig_key_ptr = nullptr;                                         // (the offset column is rewritten in place)
  if (cut == 0) { out->n_ref = B.sam_n_ref; return MCOV_OK; }
  const int rc = sam_decode_lines(ctx, raw, cut, 0, 0, B.sam_line0, "mcov_sam_chunk_decode", out);
  if (rc) return rc;
  B.sam_line0 += out->n_records;
  *consumed = (int64_t)cut;
  if (out->n_records) {                                                // (the line index of this chunk is still in sam_lines)
    cudaStream_t s = ctx->stream;
    unsigned long long* d_max = reinterpret_cast<unsigned long long*>(B.status.as<int>() + 12);
    SCU(cudaMemsetAsync(d_max, 0, 8, s));
    const int64_t grid = std::min<int64_t>((out->n_records + 255) / 256, (int64_t)std::max(ctx->n_sm, 1) * 4);
    MCOV_LAUNCH(ctx, kKSamLineMax, (k_sam_line_max<<<(unsigned)grid, 256, 0, s>>>(B.sam_lines.as<uint64_t>(), out->n_records, 0,
                                                                                  cut, d_max)));
    SCU(cudaGetLastError());
    unsigned long long m = 0;
    SCU(cudaMemcpyAsync(&m, d_max, 8, cudaMemcpyDeviceToHost, s));
    SCU(cudaStreamSynchronize(s));
    B.sam_longest = std::max<int64_t>(B.sam_longest, (int64_t)m);
  }
  return MCOV_OK;
}

extern "C" int mcov_sam_decode_gpu_file(mcov_ctx* ctx, const char* path, int64_t chunk_bytes, mcov_bam_dev* out) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!path || !out) return sfail(ctx, MCOV_ERR_ARG, "mcov_sam_decode_gpu_file: bad arguments");
  const int fd = ::open(path, O_RDONLY);
  if (fd < 0) return sfail(ctx, MCOV_ERR_IO, "mcov_sam_decode_gpu_file: cannot open the file");
  struct stat st;
  if (::fstat(fd, &st) != 0 || st.st_size <= 0) { ::close(fd); return sfail(ctx, MCOV_ERR_IO, "mcov_sam_decode_gpu_file: empty or unreadable file"); }
  void* map = ::mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
  ::close(fd);
  if (map == MAP_FAILED) return sfail(ctx, MCOV_ERR_IO, "mcov_sam_decode_gpu_file: cannot map the file");
  const int rc = mcov_sam_decode_gpu(ctx, map, (int64_t)st.st_size, chunk_bytes, out);
  ::munmap(map, (size_t)st.st_size);       // (every copy from the image has completed: the decode synchronised)
  return rc;
}

// mcov_bam_gpu_names_seq for a SAM decode: the same outputs, from the text (bam_gpu.cu dispatches here)
int mcov_sam_gpu_names_seq(mcov_ctx* ctx, int32_t k_len, int32_t win_bases, uint64_t* d_hash, int32_t* d_kmer, uint8_t* d_win) {
  mcov_ctx::BamDev& B = ctx->bam;
  const int64_t n = B.n_rec;
  MCOV_LAUNCH(ctx, kKSamNamesSeq, (k_sam_names_seq<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(
      B.data.as<uint8_t>(), B.rec_off.as<uint64_t>(), B.sam_aux.as<SamAux>(), B.lseq.as<int32_t>(), B.flag.as<uint16_t>(),
      B.cig_off.as<uint32_t>(), B.cig.as<uint32_t>(), n, k_len, win_bases, d_hash, d_kmer, d_win)));
  SCU(cudaGetLastError());
  return MCOV_OK;
}

extern "C" int mcov_bam_gpu_mapped(mcov_ctx* ctx, int64_t* mapped, int64_t* unmapped) {
  if (!ctx) return MCOV_ERR_ARG;
  if (!mapped || !unmapped) return sfail(ctx, MCOV_ERR_ARG, "mcov_bam_gpu_mapped: bad arguments");
  mcov_ctx::BamDev& B = ctx->bam;
  if (B.n_rec < 0 || !B.data.p) return sfail(ctx, MCOV_ERR_STATE, "mcov_bam_gpu_mapped: no file decoded on this context");
  SCU(cudaSetDevice(ctx->device));
  cudaStream_t s = ctx->stream;
  const int64_t n = B.n_rec;
  SCU(B.status.ensure(64));
  unsigned long long* d_cnt = reinterpret_cast<unsigned long long*>(B.status.as<int>() + 10);
  SCU(cudaMemsetAsync(d_cnt, 0, 8, s));
  if (n) {
    const int64_t grid = std::min<int64_t>((n + 255) / 256, (int64_t)std::max(ctx->n_sm, 1) * 8);
    MCOV_LAUNCH(ctx, kKMapCounts, (k_dev_map_counts<<<(unsigned)grid, 256, 0, s>>>(B.tid.as<int32_t>(), B.flag.as<uint16_t>(), n, d_cnt)));
    SCU(cudaGetLastError());
  }
  unsigned long long m = 0;
  SCU(cudaMemcpyAsync(&m, d_cnt, 8, cudaMemcpyDeviceToHost, s));
  SCU(cudaStreamSynchronize(s));
  *mapped = (int64_t)m;
  *unmapped = n - (int64_t)m;
  return MCOV_OK;
}

// ---- test hook: the same rules, line by line on the host ------------------------------------------------------------

extern "C" int mcov_sam_parse_host(const void* bytes, int64_t n_bytes, mcov_sam_host_cols* c, char* err, int err_len) {
  auto fail = [&](const std::string& m) { if (err && err_len > 0) std::snprintf(err, (size_t)err_len, "%s", m.c_str()); return MCOV_ERR_IO; };
  if (!c || (!bytes && n_bytes) || n_bytes < 0) return MCOV_ERR_ARG;
  const uint8_t* d = static_cast<const uint8_t*>(bytes);
  const uint64_t n = (uint64_t)n_bytes;
  c->fail_line = 0; c->fail_field = -1;
  SamHeader h;
  if (!sam_parse_header(d, n, h)) return fail("mcov_sam_parse_host: " + h.err);
  c->n_ref = (int32_t)h.names.size();
  c->header_bytes = (int64_t)h.body;
  RefTableHost rt;
  rt.build(h.names);
  const SamRefTable refs = rt.view();
  const bool fill = c->tid != nullptr;
  int64_t i = 0;
  uint64_t k_op = 0;
  std::vector<uint32_t> ops;
  for (uint64_t p = h.body; p < n; ++i) {
    const uint8_t* nl = static_cast<const uint8_t*>(std::memchr(d + p, '\n', (size_t)(n - p)));
    const uint64_t e0 = nl ? (uint64_t)(nl - d) : n;
    uint64_t e = e0;
    if (e > p && d[e - 1] == '\r') --e;
    const uint8_t* L = d + p;
    const uint32_t len = (uint32_t)(e - p);
    auto bad = [&](int f) { c->fail_line = h.lines + i + 1; c->fail_field = f; return fail(sam_err_text("mcov_sam_parse_host", c->fail_line, f)); };
    if (len == 0) return bad(kErrFewFields);
    if (L[0] == '@') return bad(kErrHeaderAfter);
    uint32_t tab[11], found = 0;
    for (uint32_t q = 0; q < len && found < 11; ++q) if (L[q] == '\t') tab[found++] = q;
    if (found < 10) return bad(kErrFewFields);
    auto fb = [&](int f) -> uint32_t { return f ? tab[f - 1] + 1 : 0u; };
    auto fe = [&](int f) -> uint32_t { return (uint32_t)f < found ? tab[f] : len; };
    int64_t v[kSamFields] = {0};
    const uint32_t sb = fb(kSeq), sn = fe(kSeq) - sb;
    const int64_t seq_len = sam_is_star(L + sb, sn) ? 0 : sn;
    for (int f = 0; f < kSamFields; ++f) {
      const uint32_t b = fb(f), m = fe(f) - b;
      if (f == kRname) {
        v[f] = sam_is_star(L + b, m) ? -1 : sam_ref_lookup(refs, L + b, m);
        if (m == 0 || (v[f] < 0 && !sam_is_star(L + b, m))) return bad(f);
      } else if (f == kCigar) {
        ops.clear();
        if (m == 0) return bad(f);
        if (sam_is_star(L + b, m)) continue;
        uint64_t val = 0;
        int nd = 0;
        for (uint32_t q = b; q < b + m; ++q) {
          const int op = sam_cigar_op(L[q]);
          if (op >= 0) {
            if (nd == 0 || val > kSamMaxOpLen) return bad(f);
            ops.push_back((uint32_t)(val << 4) | (uint32_t)op);
            val = 0; nd = 0;
          } else if (L[q] - (uint32_t)'0' <= 9u) {
            val = std::min<uint64_t>(val * 10 + (L[q] - '0'), kSamMaxOpLen + 1); ++nd;
          } else {
            return bad(f);
          }
        }
        if (nd) return bad(f);
      } else if (!sam_field_value(f, L + b, m, seq_len, &v[f])) {
        return bad(f);
      }
    }
    if (fill) {
      c->tid[i] = (int32_t)v[kRname]; c->pos[i] = (int32_t)v[kPos]; c->flag[i] = (uint16_t)v[kFlag]; c->mapq[i] = (uint8_t)v[kMapq];
      c->l_seq[i] = (int32_t)seq_len; c->isize[i] = (int32_t)v[kTlen]; c->cig_off[i] = (uint32_t)k_op;
      for (size_t k = 0; k < ops.size(); ++k) c->cig[k_op + k] = ops[k];
      sam_names_seq_one(L, fe(kQname), L + sb, seq_len, (uint32_t)v[kFlag], ops.data(), (uint32_t)ops.size(), c->k_len, c->win_bases,
                        c->name_hash ? c->name_hash + i : nullptr, c->kmer_code && c->k_len > 0 ? c->kmer_code + i : nullptr,
                        c->seq_win && c->win_bases > 0 ? c->seq_win + (size_t)i * ((c->win_bases + 1) / 2) : nullptr);
    }
    k_op += ops.size();
    p = nl ? e0 + 1 : n;
  }
  if (fill) c->cig_off[i] = (uint32_t)k_op;
  c->n_records = i;
  c->n_cigar = (int64_t)k_op;
  return MCOV_OK;
}

extern "C" int64_t mcov_sam_chunk_longest_line(const mcov_ctx* ctx) {
  return ctx && ctx->bam.sam_chunked ? ctx->bam.sam_longest : -1;
}
