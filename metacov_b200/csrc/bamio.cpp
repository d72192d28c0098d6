// bamio.cpp -- host BGZF / BAM / BAI decoder feeding the SoA packer.
//
// Replaces the pysam/htslib objects the reference opens at metacov/cli.py:56
// and :211 (`pysam.AlignmentFile`) and iterates at metacov/scan.pyx:204, 216
// (`IteratorRowAll` over raw `bam1_t`), reading exactly the fields the
// reference's getters read (scan.pyx:243-294: flag, pos, tid, l_qseq, isize)
// plus mapq and the CIGAR for the coverage kernels.  Formats: SAM spec v1
// section 4.1 (BGZF), 4.2 (BAM), 5.2 (BAI).  BGZF blocks are independent
// deflate streams, so they are inflated in parallel by a few host threads.
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "bamfmt.h"
#include "metacov_b200.h"

struct mcov_bam {
  std::string path;
  std::string text;
  std::vector<std::string> ref_name;
  std::vector<int32_t> ref_len;
  std::vector<uint8_t> raw;          // compressed file
  std::vector<uint8_t> data;         // inflated stream
  size_t rec_begin = 0;              // offset of the first alignment record in `data`
  bool loaded = false;
  std::vector<int32_t> tid, pos, lseq, isize;
  std::vector<uint16_t> flag;
  std::vector<uint8_t> mapq;
  std::vector<uint32_t> cig_off, cig;
  bool has_seq = false;
  std::vector<uint64_t> seq_off;     // byte offset of each record's packed SEQ
  std::vector<uint8_t> seq;          // nt16, two bases per byte, high nibble first (BAM encoding)
  std::vector<uint64_t> name_hash;   // FNV-1a 64 of the read name (filled with the SEQ pass)
};

using namespace mcov;

namespace {

int set_err(char* err, int errlen, const char* msg) {
  if (err && errlen > 0) std::snprintf(err, (size_t)errlen, "%s", msg);
  return MCOV_ERR_IO;
}

bool inflate_block(const uint8_t* src, size_t clen, uint8_t* dst, size_t ulen, uint32_t crc) {
  if (ulen == 0) return true;
  z_stream zs;
  std::memset(&zs, 0, sizeof(zs));
  if (inflateInit2(&zs, -15) != Z_OK) return false;
  zs.next_in = const_cast<Bytef*>(src);
  zs.avail_in = (uInt)clen;
  zs.next_out = dst;
  zs.avail_out = (uInt)ulen;
  int rc = inflate(&zs, Z_FINISH);
  bool ok = (rc == Z_STREAM_END) && zs.total_out == ulen;
  inflateEnd(&zs);
  if (ok) ok = ((uint32_t)crc32(crc32(0L, Z_NULL, 0), dst, (uInt)ulen) == crc);
  return ok;
}

// Inflates every block from raw to dst + its uoff on n_threads host threads (at most one per block); false when a
// block does not inflate to its ISIZE and CRC.
bool inflate_blocks(const uint8_t* raw, const std::vector<BgzfBlock>& blocks, uint8_t* dst, int n_threads) {
  const int nt = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(n_threads, 1), blocks.size()));
  std::atomic<size_t> next(0);
  std::atomic<bool> good(true);
  auto work = [&]() {
    for (;;) {
      const size_t k = next.fetch_add(1);
      if (k >= blocks.size() || !good.load()) break;
      const BgzfBlock& bl = blocks[k];
      if (!inflate_block(raw + bl.coff, bl.clen, dst + bl.uoff, bl.ulen, bl.crc)) good.store(false);
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nt; ++t) th.emplace_back(work);
  work();
  for (auto& t : th) t.join();
  return good.load();
}

// nothing may throw across the C ABI: allocation failures and anything else become status codes
template <typename F>
int guarded(F fn) {
  try { return fn(); }
  catch (const std::bad_alloc&) { return MCOV_ERR_NOMEM; }
  catch (...) { return MCOV_ERR_IO; }
}

// Calls f(i, r) for every record i of the inflated stream, r pointing behind its block_size; false when a record does
// not fit its block_size or the stream does not end where the last record does.
template <typename F>
bool each_record(const mcov_bam* b, F f) {
  const uint8_t* d = b->data.data();
  const size_t n = b->data.size();
  size_t p = b->rec_begin, i = 0;
  while (p + 4 <= n) {
    const uint32_t bs = rd32(d + p);
    if (bs < 32 || p + 4 + bs > n || !record_fits(d + p + 4, bs)) return false;
    f(i++, d + p + 4);
    p += 4 + bs;
  }
  return p == n;
}

}  // namespace

static int read_inflate(mcov_bam* b);
// read the file and inflate it into b->data; 0 ok, 1 cannot open, 2 short read, 3 bad BGZF, 4 bad BAM
static int read_inflate(mcov_bam* b) {
  FILE* fh = std::fopen(b->path.c_str(), "rb");
  if (!fh) return 1;
  std::fseek(fh, 0, SEEK_END);
  long sz = std::ftell(fh);
  std::fseek(fh, 0, SEEK_SET);
  b->raw.resize(sz > 0 ? (size_t)sz : 0);
  size_t got = b->raw.empty() ? 0 : std::fread(b->raw.data(), 1, b->raw.size(), fh);
  std::fclose(fh);
  if (got != b->raw.size()) return 2;
  std::vector<BgzfBlock> blocks;
  uint64_t total = 0;
  size_t used = 0;
  if (!bgzf_index(b->raw.data(), b->raw.size(), 0, false, blocks, total, used)) return 3;
  b->data.resize(total);
  unsigned hw = std::thread::hardware_concurrency();
  if (!inflate_blocks(b->raw.data(), blocks, b->data.data(), hw ? (int)hw : 4)) return 3;
  BamHeader h;
  if (parse_bam_header(b->data.data(), b->data.size(), true, h) != HeaderParse::kOk) return 4;
  b->text.swap(h.text); b->ref_name.swap(h.names); b->ref_len.swap(h.lens);
  b->rec_begin = h.rec_begin;
  std::vector<uint8_t>().swap(b->raw);
  return 0;
}

extern "C" {

int mcov_bam_open(mcov_bam** out, const char* path, char* err, int errlen) {
  if (!out || !path) return set_err(err, errlen, "mcov_bam_open: null argument");
  *out = nullptr;
  mcov_bam* b = new (std::nothrow) mcov_bam();
  if (!b) return set_err(err, errlen, "mcov_bam_open: out of memory");
  static const char* msg[] = {"", "mcov_bam_open: cannot open file", "mcov_bam_open: short read",
                              "mcov_bam_open: not a valid BGZF file", "mcov_bam_open: not a valid BAM file",
                              "mcov_bam_open: out of memory (a corrupt file may ask for more than the host has)"};
  int rc = 5;
  try { b->path = path; rc = read_inflate(b); }
  catch (const std::bad_alloc&) { rc = 5; }
  catch (...) { rc = 3; }
  if (rc) { delete b; return set_err(err, errlen, msg[rc]); }
  *out = b;
  return MCOV_OK;
}

void mcov_bam_close(mcov_bam* b) { delete b; }

int32_t mcov_bam_n_ref(const mcov_bam* b) { return b ? (int32_t)b->ref_name.size() : 0; }
const char* mcov_bam_ref_name(const mcov_bam* b, int32_t tid) {
  return (b && tid >= 0 && (size_t)tid < b->ref_name.size()) ? b->ref_name[tid].c_str() : nullptr;
}
int32_t mcov_bam_ref_len(const mcov_bam* b, int32_t tid) {
  return (b && tid >= 0 && (size_t)tid < b->ref_len.size()) ? b->ref_len[tid] : -1;
}
const char* mcov_bam_header_text(const mcov_bam* b) { return b ? b->text.c_str() : nullptr; }

int mcov_bam_index_stats(const mcov_bam* b, int64_t* mapped, int64_t* unmapped) {
  if (!b) return MCOV_ERR_ARG;
  return mcov_bai_stats(b->path.c_str(), mapped, unmapped);
}

int mcov_bai_stats(const char* bam_path, int64_t* mapped, int64_t* unmapped) {
  if (!bam_path || !mapped || !unmapped) return MCOV_ERR_ARG;
  const std::string path(bam_path);
  std::string cand[2] = {path + ".bai", path};
  if (cand[1].size() > 4 && cand[1].compare(cand[1].size() - 4, 4, ".bam") == 0) cand[1].replace(cand[1].size() - 4, 4, ".bai");
  FILE* fh = nullptr;
  for (auto& c : cand) { fh = std::fopen(c.c_str(), "rb"); if (fh) break; }
  if (!fh) return MCOV_ERR_IO;
  std::vector<uint8_t> d;
  uint8_t buf[65536];
  size_t k;
  while ((k = std::fread(buf, 1, sizeof(buf), fh)) > 0) d.insert(d.end(), buf, buf + k);
  std::fclose(fh);
  if (d.size() < 8 || std::memcmp(d.data(), "BAI\1", 4) != 0) return MCOV_ERR_IO;
  uint32_t n_ref = rd32(d.data() + 4);
  size_t p = 8;
  uint64_t m = 0, u = 0;
  for (uint32_t r = 0; r < n_ref; ++r) {
    if (p + 4 > d.size()) return MCOV_ERR_IO;
    uint32_t n_bin = rd32(d.data() + p);
    p += 4;
    for (uint32_t k2 = 0; k2 < n_bin; ++k2) {
      if (p + 8 > d.size()) return MCOV_ERR_IO;
      uint32_t bin = rd32(d.data() + p), n_chunk = rd32(d.data() + p + 4);
      p += 8;
      if (p + 16ull * n_chunk > d.size()) return MCOV_ERR_IO;
      if (bin == 37450 && n_chunk == 2) { m += rd64(d.data() + p + 16); u += rd64(d.data() + p + 24); }
      p += 16ull * n_chunk;
    }
    if (p + 4 > d.size()) return MCOV_ERR_IO;
    uint32_t n_intv = rd32(d.data() + p);
    p += 4 + 8ull * n_intv;
  }
  if (p + 8 <= d.size()) u += rd64(d.data() + p);     // n_no_coor
  *mapped = (int64_t)m;
  *unmapped = (int64_t)u;
  return MCOV_OK;
}

static int bam_load_impl(mcov_bam* b);
int mcov_bam_load(mcov_bam* b, int /*n_threads*/) {
  if (!b) return MCOV_ERR_ARG;
  if (b->loaded) return MCOV_OK;
  return guarded([&]() { return bam_load_impl(b); });
}
static int bam_load_impl(mcov_bam* b) {
  size_t n_rec = 0, n_cig = 0;
  if (!each_record(b, [&](size_t, const uint8_t* r) { n_cig += record_n_op(r); ++n_rec; })) return MCOV_ERR_IO;
  if (n_cig > 0xFFFFFFFFull) return MCOV_ERR_RANGE;
  b->tid.resize(n_rec); b->pos.resize(n_rec); b->lseq.resize(n_rec); b->isize.resize(n_rec);
  b->flag.resize(n_rec); b->mapq.resize(n_rec); b->cig_off.resize(n_rec + 1); b->cig.resize(n_cig);
  const RecordCols c{b->tid.data(), b->pos.data(), b->lseq.data(), b->isize.data(), b->flag.data(), b->mapq.data()};
  size_t co = 0;
  each_record(b, [&](size_t i, const uint8_t* r) { b->cig_off[i] = (uint32_t)co; co += copy_record(r, c, i, b->cig.data() + co); });
  b->cig_off[n_rec] = (uint32_t)co;
  std::vector<uint8_t>().swap(b->data);   // the SoA arrays are all that is kept
  b->loaded = true;
  return MCOV_OK;
}

int64_t mcov_bam_n_records(const mcov_bam* b) { return (b && b->loaded) ? (int64_t)b->tid.size() : -1; }
int64_t mcov_bam_n_cigar(const mcov_bam* b) { return (b && b->loaded) ? (int64_t)b->cig.size() : -1; }
const int32_t* mcov_bam_tid(const mcov_bam* b) { return (b && b->loaded) ? b->tid.data() : nullptr; }
const int32_t* mcov_bam_pos(const mcov_bam* b) { return (b && b->loaded) ? b->pos.data() : nullptr; }
const uint16_t* mcov_bam_flag(const mcov_bam* b) { return (b && b->loaded) ? b->flag.data() : nullptr; }
const uint8_t* mcov_bam_mapq(const mcov_bam* b) { return (b && b->loaded) ? b->mapq.data() : nullptr; }
const int32_t* mcov_bam_lseq(const mcov_bam* b) { return (b && b->loaded) ? b->lseq.data() : nullptr; }
const int32_t* mcov_bam_isize(const mcov_bam* b) { return (b && b->loaded) ? b->isize.data() : nullptr; }
const uint32_t* mcov_bam_cig_off(const mcov_bam* b) { return (b && b->loaded) ? b->cig_off.data() : nullptr; }
const uint32_t* mcov_bam_cig(const mcov_bam* b) { return (b && b->loaded) ? b->cig.data() : nullptr; }

// Packed SEQ of every record (needed by the k-mer histogram only).  Re-inflates the file when the
// record pass has already released it.
static int bam_load_seq_impl(mcov_bam* b);
int mcov_bam_load_seq(mcov_bam* b) {
  if (!b) return MCOV_ERR_ARG;
  if (b->has_seq) return MCOV_OK;
  return guarded([&]() { return bam_load_seq_impl(b); });
}
static int bam_load_seq_impl(mcov_bam* b) {
  if (b->data.empty()) { if (read_inflate(b)) return MCOV_ERR_IO; }
  size_t n_rec = 0, bytes = 0;
  if (!each_record(b, [&](size_t, const uint8_t* r) { bytes += ((size_t)rd32(r + 16) + 1) / 2; ++n_rec; })) return MCOV_ERR_IO;
  b->seq_off.resize(n_rec + 1);
  b->seq.resize(bytes);
  b->name_hash.resize(n_rec);
  size_t so = 0;
  each_record(b, [&](size_t i, const uint8_t* r) {
    const uint8_t l_read_name = r[8];
    const size_t nb = ((size_t)rd32(r + 16) + 1) / 2;
    b->seq_off[i] = so;
    uint64_t h = 1469598103934665603ull;                      // FNV-1a 64 over the name (without the NUL)
    for (unsigned k = 0; k + 1 < l_read_name; ++k) { h ^= r[32 + k]; h *= 1099511628211ull; }
    b->name_hash[i] = h == ~0ull ? h - 1 : h;                 // ~0 is the "no entry" key of the pair sort
    std::memcpy(b->seq.data() + so, r + 32 + l_read_name + 4u * record_n_op(r), nb);
    so += nb;
  });
  b->seq_off[n_rec] = so;
  b->has_seq = true;
  if (b->loaded) std::vector<uint8_t>().swap(b->data);
  return MCOV_OK;
}

// Per read a window of `win_bases` bases, re-packed two per byte (high nibble first) into
// out[n][(win_bases+1)/2]: forward reads contribute their FIRST win_bases bases, reverse reads
// (flag 0x10) their LAST win_bases, so that window base j is absolute base (l_seq - win_bases + j);
// missing bases are 'N' (15).  This is all the k-mer histogram needs (reference scan.pyx:240-259
// decodes the whole SEQ and undoes the mapper's reverse complement; only the read's first
// OFFSET+STEP*(NK-1)+K bases are ever looked at, scan.pyx:513-520).
static int bam_seq_windows_impl(const mcov_bam* b, int32_t win_bases, uint8_t* out);
int mcov_bam_seq_windows(const mcov_bam* b, int32_t win_bases, uint8_t* out) {
  if (!b || !out || win_bases <= 0) return MCOV_ERR_ARG;
  if (!b->has_seq || !b->loaded) return MCOV_ERR_ARG;
  return guarded([&]() { return bam_seq_windows_impl(b, win_bases, out); });
}
static int bam_seq_windows_impl(const mcov_bam* b, int32_t win_bases, uint8_t* out) {
  const size_t n = b->tid.size(), W = ((size_t)win_bases + 1) / 2;
  unsigned hw = std::thread::hardware_concurrency();
  int nt = (int)std::max(1u, std::min(hw ? hw : 4u, 32u));
  if (n < 4096) nt = 1;
  auto work = [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; ++i) {
      const uint8_t* s = b->seq.data() + b->seq_off[i];
      const int64_t l = b->lseq[i];
      const bool rev = (b->flag[i] & 0x10) != 0;
      uint8_t* o = out + i * W;
      std::memset(o, 0xff, W);
      for (int32_t j = 0; j < win_bases; ++j) {
        int64_t a = rev ? l - win_bases + j : j;
        uint8_t c = 15;
        if (a >= 0 && a < l) c = (a & 1) ? (s[a >> 1] & 15) : (s[a >> 1] >> 4);
        if (j & 1) o[j >> 1] = (uint8_t)((o[j >> 1] & 0xf0) | c);
        else o[j >> 1] = (uint8_t)((o[j >> 1] & 0x0f) | (c << 4));
      }
    }
  };
  std::vector<std::thread> th;
  size_t per = (n + nt - 1) / nt;
  for (int t = 1; t < nt; ++t) { size_t lo = t * per, hi = std::min(n, lo + per); if (lo < hi) th.emplace_back(work, lo, hi); }
  work(0, std::min(n, per));
  for (auto& t : th) t.join();
  return MCOV_OK;
}

// FNV-1a 64 hashes of the read names (`read.query_name`, reference metacov/pileup.py:101-118 joins
// mates through a dict keyed by it).  Valid after mcov_bam_load_seq.
const uint64_t* mcov_bam_name_hash(const mcov_bam* b) { return (b && b->has_seq) ? b->name_hash.data() : nullptr; }

// Per read the 2-bit code of the first k_len bases of `query_alignment_sequence` (SEQ as stored,
// without the soft-clipped ends; reference metacov/pileup.py:109-110, 123): first base most
// significant, A0 C1 G2 T3; -1 when the aligned part is shorter than k_len or holds another letter
// (a dict lookup with such a key raises KeyError in the reference).  k_len <= 15.
int mcov_bam_qas_kmer(const mcov_bam* b, int32_t k_len, int32_t* out) {
  if (!b || !out || k_len <= 0 || k_len > 15) return MCOV_ERR_ARG;
  if (!b->has_seq || !b->loaded) return MCOV_ERR_ARG;
  static const int8_t nt4[16] = {-1, 0, 1, -1, 2, -1, -1, -1, 3, -1, -1, -1, -1, -1, -1, -1};   // "=ACMGRSVTWYHKDBN"
  const size_t n = b->tid.size();
  for (size_t i = 0; i < n; ++i) {
    const uint8_t* s = b->seq.data() + b->seq_off[i];
    int64_t lo = 0, hi = b->lseq[i];
    const uint32_t c0 = b->cig_off[i], c1 = b->cig_off[i + 1];
    for (uint32_t k = c0; k < c1; ++k) {                      // leading soft clips (hard clips hold no bases)
      uint32_t op = b->cig[k] & 15u;
      if (op == 5) continue;
      if (op == 4) lo += b->cig[k] >> 4; else break;
    }
    for (uint32_t k = c1; k > c0; --k) {
      uint32_t op = b->cig[k - 1] & 15u;
      if (op == 5) continue;
      if (op == 4) hi -= b->cig[k - 1] >> 4; else break;
    }
    int32_t code = 0;
    if (hi - lo < k_len) code = -1;
    for (int32_t j = 0; j < k_len && code >= 0; ++j) {
      int64_t a = lo + j;
      int8_t c = nt4[(a & 1) ? (s[a >> 1] & 15) : (s[a >> 1] >> 4)];
      code = c < 0 ? -1 : (code << 2) | c;
    }
    out[i] = code;
  }
  return MCOV_OK;
}

}  // extern "C"

// ===========================================================================================================
// Streaming reader: the file is read, inflated and parsed in BATCHES straight into pinned SoA buffers (two sets:
// the GPU copies batch k from one set while batch k+1 is decoded into the other).  Replaces the record loop of
// reference metacov/scan.pyx:653-667 (`cnext()` over IteratorRowAll) for the coverage path: the file is never held,
// neither compressed nor inflated.  Each batch begins with the reads of earlier batches that the depth engine asked
// to see again (mcov_stream_push: everything that starts at or after the resend point or reaches past it).
// ===========================================================================================================
#include <cuda_runtime.h>

struct mcov_bam_stream {
  FILE* fh = nullptr;
  std::string text;
  std::vector<std::string> ref_name;
  std::vector<int32_t> ref_len;
  std::vector<uint8_t> raw;        // compressed bytes read but not yet inflated (an incomplete trailing block)
  std::vector<uint8_t> data;       // inflated bytes not yet parsed
  size_t data_pos = 0;
  bool eof = false, header_done = false, finished = false;
  int n_threads = 4;
  int64_t batch_reads = 1 << 21;
  int64_t cap_reads = 0, cap_ops = 0;
  struct Set {
    int32_t *tid = nullptr, *pos = nullptr, *lseq = nullptr, *isize = nullptr, *reflen = nullptr;
    uint16_t* flag = nullptr;
    uint8_t* mapq = nullptr;
    uint32_t *cig_off = nullptr, *cig = nullptr;
    int64_t n = 0, n_carry = 0, n_ops = 0;
    bool pinned = true;
  } set[2];
  int cur = 0;                     // set the NEXT batch is decoded into
  int32_t max_reflen = 1;
  int64_t n_records = 0;           // distinct records handed out so far
  std::vector<size_t> rec_off;     // scratch: record offsets of the batch being built
  std::string err;
  // transport blocks of the batches (mcov_bam_stream_next_block): two pinned buffers, like the SoA sets
  void* blk[2] = {nullptr, nullptr};
  int64_t blk_cap[2] = {0, 0};
  bool blk_pinned = true;
  int blk_cur = 0;
};

namespace {

constexpr size_t kStreamChunk = 32u << 20;     // compressed bytes per read() call

// Pinned memory when a CUDA device is there (true asynchronous H2D); without one (the CPU test suite checks the
// reader against the oracle's) plain aligned memory -- these are buffers, no compute path depends on which.
template <typename T>
bool pin_alloc(T*& p, size_t n, bool& pinned) {
  const size_t bytes = std::max<size_t>(n * sizeof(T), 64);
  if (pinned) {
    if (cudaHostAlloc(reinterpret_cast<void**>(&p), bytes, cudaHostAllocDefault) == cudaSuccess) return true;
    (void)cudaGetLastError();
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) == cudaSuccess && n_dev > 0) { p = nullptr; return false; }   // a device, but no pinned memory left
    (void)cudaGetLastError();
    pinned = false;
  }
  p = static_cast<T*>(std::aligned_alloc(64, (bytes + 63) & ~(size_t)63));
  return p != nullptr;
}

void stream_free_set(mcov_bam_stream::Set& s) {
  void* ps[] = {s.tid, s.pos, s.lseq, s.isize, s.reflen, s.flag, s.mapq, s.cig_off, s.cig};
  for (void* p : ps) if (p) { if (s.pinned) cudaFreeHost(p); else std::free(p); }
  s = mcov_bam_stream::Set();
}

bool stream_alloc_set(mcov_bam_stream::Set& s, int64_t reads, int64_t ops) {
  bool& pn = s.pinned;
  return pin_alloc(s.tid, reads, pn) && pin_alloc(s.pos, reads, pn) && pin_alloc(s.lseq, reads, pn) && pin_alloc(s.isize, reads, pn) &&
         pin_alloc(s.reflen, reads, pn) && pin_alloc(s.flag, reads, pn) && pin_alloc(s.mapq, reads, pn) && pin_alloc(s.cig_off, reads + 1, pn) &&
         pin_alloc(s.cig, ops + 4, pn);
}

// Read the next chunk of the file and inflate every complete BGZF block of it (in parallel) onto the end of `data`.
// Returns false on a malformed file.
struct StreamTimer {
  const char* what; std::chrono::steady_clock::time_point t0;
  explicit StreamTimer(const char* w) : what(w), t0(std::chrono::steady_clock::now()) {}
  ~StreamTimer() {
    static const bool on = std::getenv("MCOV_STREAM_DEBUG") != nullptr;
    if (on) std::fprintf(stderr, "[stream] %-10s %.1f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  }
};

bool stream_refill(mcov_bam_stream* s) {
  if (s->eof) return true;
  StreamTimer tm("refill");
  // drop what has been parsed
  if (s->data_pos > 0) { s->data.erase(s->data.begin(), s->data.begin() + (ptrdiff_t)s->data_pos); s->data_pos = 0; }
  // (the first read is small: opening a file should cost no more than its header)
  // (MCOV_STREAM_READ_BYTES: test hook -- small reads put a chunk border into every BGZF block and record of a small file)
  size_t chunk = kStreamChunk;
  if (const char* e = std::getenv("MCOV_STREAM_READ_BYTES")) { const long long v = std::atoll(e); if (v >= 1024) chunk = (size_t)v; }
  const size_t want = s->header_done ? chunk : std::min<size_t>(chunk, (size_t)256 << 10);
  const size_t old = s->raw.size();
  s->raw.resize(old + want);
  const size_t got = std::fread(s->raw.data() + old, 1, want, s->fh);
  s->raw.resize(old + got);
  if (got < want) s->eof = true;
  // inflate the complete blocks onto the end of `data`
  std::vector<BgzfBlock> blocks;
  uint64_t end = 0;
  size_t used = 0;
  if (!bgzf_index(s->raw.data(), s->raw.size(), s->data.size(), !s->eof, blocks, end, used)) return false;
  s->data.resize(end);
  if (!inflate_blocks(s->raw.data(), blocks, s->data.data(), s->n_threads)) return false;
  s->raw.erase(s->raw.begin(), s->raw.begin() + (ptrdiff_t)used);
  return true;
}

// header: magic, text, reference table; may span several chunks
int stream_parse_header(mcov_bam_stream* s) {
  for (;;) {
    BamHeader h;
    const HeaderParse r = parse_bam_header(s->data.data(), s->data.size(), true, h);
    if (r == HeaderParse::kOk) {
      s->text.swap(h.text); s->ref_name.swap(h.names); s->ref_len.swap(h.lens);
      s->data_pos = h.rec_begin;
      s->header_done = true;
      return 0;
    }
    if (r == HeaderParse::kBad || s->eof) return 4;
    if (!stream_refill(s)) return 3;
  }
}

}  // namespace

extern "C" {

int mcov_bam_stream_open(mcov_bam_stream** out, const char* path, int64_t batch_reads, int n_threads, char* err, int errlen) {
  if (!out || !path) return set_err(err, errlen, "mcov_bam_stream_open: null argument");
  *out = nullptr;
  mcov_bam_stream* s = new (std::nothrow) mcov_bam_stream();
  if (!s) return set_err(err, errlen, "mcov_bam_stream_open: out of memory");
  int rc = 0;
  try {
    s->fh = std::fopen(path, "rb");
    if (!s->fh) rc = 1;
    if (batch_reads > 0) s->batch_reads = batch_reads;
    unsigned hw = std::thread::hardware_concurrency();
    s->n_threads = n_threads > 0 ? n_threads : (hw ? (int)hw : 4);
    if (!rc && !stream_refill(s)) rc = 3;
    if (!rc) rc = stream_parse_header(s);
  } catch (const std::bad_alloc&) { rc = 5; }
  catch (...) { rc = 3; }
  static const char* msg[] = {"", "mcov_bam_stream_open: cannot open file", "", "mcov_bam_stream_open: not a valid BGZF file",
                              "mcov_bam_stream_open: not a valid BAM file", "mcov_bam_stream_open: out of memory"};
  if (rc) { if (s->fh) std::fclose(s->fh); delete s; return set_err(err, errlen, msg[rc]); }
  *out = s;
  return MCOV_OK;
}

void mcov_bam_stream_close(mcov_bam_stream* s) {
  if (!s) return;
  if (s->fh) std::fclose(s->fh);
  stream_free_set(s->set[0]); stream_free_set(s->set[1]);
  for (void* p : s->blk) if (p) { if (s->blk_pinned) cudaFreeHost(p); else std::free(p); }
  delete s;
}

int32_t mcov_bam_stream_n_ref(const mcov_bam_stream* s) { return s ? (int32_t)s->ref_name.size() : 0; }
const char* mcov_bam_stream_ref_name(const mcov_bam_stream* s, int32_t tid) {
  return (s && tid >= 0 && (size_t)tid < s->ref_name.size()) ? s->ref_name[tid].c_str() : nullptr;
}
int32_t mcov_bam_stream_ref_len(const mcov_bam_stream* s, int32_t tid) {
  return (s && tid >= 0 && (size_t)tid < s->ref_len.size()) ? s->ref_len[tid] : -1;
}
const char* mcov_bam_stream_header_text(const mcov_bam_stream* s) { return s ? s->text.c_str() : nullptr; }
const char* mcov_bam_stream_error(const mcov_bam_stream* s) { return s ? s->err.c_str() : "null stream"; }

static int stream_next_impl(mcov_bam_stream* s, int32_t resend_tid, int32_t resend_pos, mcov_bam_batch* out) {
  std::memset(out, 0, sizeof(*out));
  if (s->finished) return 0;
  mcov_bam_stream::Set& prev = s->set[s->cur ^ 1];
  // ---- walk the record chain of the new batch (serial: a length-prefixed list), refilling as needed ----
  s->rec_off.clear();
  int64_t new_ops = 0;
  bool at_end = false;
  StreamTimer tm_all("next");
  while ((int64_t)s->rec_off.size() < s->batch_reads) {
    const size_t avail = s->data.size() - s->data_pos;
    bool have = false;
    if (avail >= 4) {
      const uint32_t bs = rd32(s->data.data() + s->data_pos);
      if (bs < 32) { s->err = "record shorter than its fixed part"; return MCOV_ERR_IO; }
      if (avail >= 4 + (size_t)bs) {
        if (!record_fits(s->data.data() + s->data_pos + 4, bs)) { s->err = "record fields exceed block_size"; return MCOV_ERR_IO; }
        s->rec_off.push_back(s->data_pos);
        new_ops += record_n_op(s->data.data() + s->data_pos + 4);
        s->data_pos += 4 + (size_t)bs;
        have = true;
      }
    }
    if (have) continue;
    if (s->eof) {
      if (avail != 0) { s->err = "truncated record at the end of the file"; return MCOV_ERR_IO; }
      at_end = true;
      break;
    }
    // more data needed: the offsets collected so far move with the buffer
    const size_t shift = s->rec_off.empty() ? s->data_pos : s->rec_off.front();
    const size_t keep_pos = s->data_pos;
    s->data_pos = shift;                                     // keep the batch's records in the buffer
    if (!stream_refill(s)) { s->err = "BGZF block does not inflate"; return MCOV_ERR_IO; }
    for (size_t& o : s->rec_off) o -= shift;
    s->data_pos = keep_pos - shift;
  }
  if (!at_end && s->eof && s->data_pos == s->data.size()) at_end = true;
  const int64_t n_new = (int64_t)s->rec_off.size();
  StreamTimer tm_rest("carry+fill");
  // ---- carry: reads of the previous batch that start at or after the resend point or reach past it ----
  int64_t c_lo = prev.n;                                      // carry candidates are prev[c_lo, prev.n): a suffix in sorted order
  if (resend_tid >= 0 && prev.n > 0) {
    const int64_t reach = (int64_t)resend_pos - s->max_reflen;
    while (c_lo > 0) {
      const int32_t t = prev.tid[c_lo - 1];
      if (t >= 0 && (t < resend_tid || (t == resend_tid && prev.pos[c_lo - 1] < reach))) break;
      --c_lo;
    }
  }
  std::vector<int64_t> carry;
  int64_t carry_ops = 0;
  for (int64_t i = c_lo; i < prev.n && resend_tid >= 0; ++i) {
    const int32_t t = prev.tid[i];
    if (t < 0) continue;                                      // unplaced reads cover nothing: never needed again
    const bool need = t > resend_tid || (t == resend_tid && (prev.pos[i] >= resend_pos || (int64_t)prev.pos[i] + prev.reflen[i] > resend_pos));
    if (need) { carry.push_back(i); carry_ops += prev.cig_off[i + 1] - prev.cig_off[i]; }
  }
  const int64_t n = (int64_t)carry.size() + n_new, n_ops = carry_ops + new_ops;
  if (n_ops > 0xFFFFFFF0ll) { s->err = "more than 2^32 CIGAR ops in one batch: lower batch_reads"; return MCOV_ERR_RANGE; }
  // ---- (re)allocate both pinned sets when this batch does not fit ----
  if (n > s->cap_reads || n_ops > s->cap_ops) {
    const int64_t cr = std::max<int64_t>(n + n / 4, s->batch_reads + (s->batch_reads >> 2)), co = std::max<int64_t>(n_ops + n_ops / 4, 1024);
    mcov_bam_stream::Set fresh[2];
    if (!stream_alloc_set(fresh[0], cr, co) || !stream_alloc_set(fresh[1], cr, co)) {
      stream_free_set(fresh[0]); stream_free_set(fresh[1]);
      s->err = "pinned host memory exhausted";
      return MCOV_ERR_NOMEM;
    }
    // the previous batch is still needed for the carry: move it over
    mcov_bam_stream::Set& np = fresh[s->cur ^ 1];
    if (prev.n > 0) {
      std::memcpy(np.tid, prev.tid, prev.n * 4); std::memcpy(np.pos, prev.pos, prev.n * 4); std::memcpy(np.lseq, prev.lseq, prev.n * 4);
      std::memcpy(np.isize, prev.isize, prev.n * 4); std::memcpy(np.reflen, prev.reflen, prev.n * 4); std::memcpy(np.flag, prev.flag, prev.n * 2);
      std::memcpy(np.mapq, prev.mapq, prev.n); std::memcpy(np.cig_off, prev.cig_off, (prev.n + 1) * 4); std::memcpy(np.cig, prev.cig, prev.n_ops * 4);
    }
    np.n = prev.n; np.n_carry = prev.n_carry; np.n_ops = prev.n_ops;
    // (the caller must have finished with the old buffers: mcov_stream_push returns after its copies are done)
    stream_free_set(s->set[0]); stream_free_set(s->set[1]);
    s->set[0] = fresh[0]; s->set[1] = fresh[1];
    s->cap_reads = cr; s->cap_ops = co;
  }
  mcov_bam_stream::Set& cur = s->set[s->cur];
  mcov_bam_stream::Set& pv = s->set[s->cur ^ 1];
  // ---- carried reads first ----
  uint32_t co = 0;
  for (size_t k = 0; k < carry.size(); ++k) {
    const int64_t i = carry[k];
    cur.tid[k] = pv.tid[i]; cur.pos[k] = pv.pos[i]; cur.lseq[k] = pv.lseq[i]; cur.isize[k] = pv.isize[i]; cur.reflen[k] = pv.reflen[i];
    cur.flag[k] = pv.flag[i]; cur.mapq[k] = pv.mapq[i];
    const uint32_t nops = pv.cig_off[i + 1] - pv.cig_off[i];
    cur.cig_off[k] = co;
    std::memcpy(cur.cig + co, pv.cig + pv.cig_off[i], (size_t)nops * 4);
    co += nops;
  }
  const int64_t nc = (int64_t)carry.size();
  // ---- new reads: offsets serially (a prefix sum over the op counts), fields and ops in parallel ----
  const uint8_t* d = s->data.data();
  for (int64_t i = 0; i < n_new; ++i) { cur.cig_off[nc + i] = co; co += record_n_op(d + s->rec_off[(size_t)i] + 4); }
  cur.cig_off[n] = co;
  std::atomic<int32_t> mx(s->max_reflen);
  const RecordCols cols{cur.tid, cur.pos, cur.lseq, cur.isize, cur.flag, cur.mapq};
  auto fill = [&](int64_t lo, int64_t hi) {
    int32_t local_max = 1;
    for (int64_t i = lo; i < hi; ++i) {
      const int64_t k = nc + i;
      uint32_t* dst = cur.cig + cur.cig_off[k];
      const uint16_t n_op = copy_record(d + s->rec_off[(size_t)i] + 4, cols, (size_t)k, dst);
      int64_t rl = 0;
      for (uint16_t o = 0; o < n_op; ++o) { const uint32_t op = dst[o]; if ((0x18Du >> (op & 15u)) & 1u) rl += op >> 4; }
      const int32_t rl32 = rl > 0x7fffffff ? 0x7fffffff : (int32_t)rl;
      cur.reflen[k] = rl32;
      local_max = std::max(local_max, rl32);
    }
    int32_t seen = mx.load();
    while (local_max > seen && !mx.compare_exchange_weak(seen, local_max)) {}
  };
  {
    const int nt = n_new >= 65536 ? std::max(1, std::min(s->n_threads, 32)) : 1;
    const int64_t per = (n_new + nt - 1) / nt;
    std::vector<std::thread> th;
    for (int t = 1; t < nt; ++t) { const int64_t lo = t * per, hi = std::min(n_new, lo + per); if (lo < hi) th.emplace_back(fill, lo, hi); }
    fill(0, std::min(n_new, per));
    for (auto& t : th) t.join();
  }
  s->max_reflen = mx.load();
  cur.n = n; cur.n_carry = nc; cur.n_ops = co;
  s->n_records += n_new;
  out->n = n; out->n_carry = nc; out->n_cigar = co; out->last = at_end ? 1 : 0;
  out->tid = cur.tid; out->pos = cur.pos; out->flag = cur.flag; out->mapq = cur.mapq; out->l_seq = cur.lseq; out->isize = cur.isize;
  out->reflen = cur.reflen; out->cig_off = cur.cig_off; out->cig = cur.cig;
  s->cur ^= 1;
  if (at_end) s->finished = true;
  return 1;
}

int mcov_bam_stream_next(mcov_bam_stream* s, int32_t resend_tid, int32_t resend_pos, mcov_bam_batch* out) {
  if (!s || !out) return MCOV_ERR_ARG;
  try { return stream_next_impl(s, resend_tid, resend_pos, out); }
  catch (const std::bad_alloc&) { s->err = "out of memory"; return MCOV_ERR_NOMEM; }
  catch (...) { s->err = "unexpected failure"; return MCOV_ERR_IO; }
}

int64_t mcov_bam_stream_records(const mcov_bam_stream* s) { return s ? s->n_records : 0; }

// The next batch as a transport block (mcov_pack_block) in pinned memory owned by the stream: what
// mcov_stream_push_block / mcov_depth_sorted_block take with ONE host-to-device copy.  *block is NULL when the batch does
// not qualify for the block (a CIGAR of more than 127 ops: long reads) -- push its columns (*out) instead.
int mcov_bam_stream_next_block(mcov_bam_stream* s, int32_t resend_tid, int32_t resend_pos, int with_mapq,
                               const void** block, int64_t* bytes, mcov_bam_batch* out) {
  if (!s || !out || !block || !bytes) return MCOV_ERR_ARG;
  *block = nullptr; *bytes = 0;
  int rc = mcov_bam_stream_next(s, resend_tid, resend_pos, out);
  if (rc <= 0) return rc;
  try {
    const int32_t n_contigs = (int32_t)s->ref_len.size();
    if (n_contigs <= 0) return rc;
    const int64_t need = mcov_block_bound(out->n, out->n_cigar, n_contigs);
    const int k = s->blk_cur;
    s->blk_cur ^= 1;
    if (need > s->blk_cap[k]) {
      if (s->blk[k]) { if (s->blk_pinned) cudaFreeHost(s->blk[k]); else std::free(s->blk[k]); s->blk[k] = nullptr; s->blk_cap[k] = 0; }
      const int64_t want = need + need / 4;
      uint8_t* p = nullptr;
      if (!pin_alloc(p, (size_t)want, s->blk_pinned)) { s->err = "pinned host memory exhausted"; return MCOV_ERR_NOMEM; }
      s->blk[k] = p; s->blk_cap[k] = want;
    }
    int64_t nb = 0;
    const int prc = mcov_pack_block(out->n, out->n_carry, out->tid, out->pos, out->flag, with_mapq ? out->mapq : nullptr, out->cig_off,
                                    out->cig, n_contigs, s->blk[k], s->blk_cap[k], &nb, s->n_threads);
    if (prc == MCOV_OK) { *block = s->blk[k]; *bytes = nb; }
    else if (prc != MCOV_ERR_RANGE && prc != MCOV_ERR_ARG) { s->err = "transport block packing failed"; return prc; }
    // (MCOV_ERR_ARG: the file is not grouped by contig, i.e. not sorted -- the caller pushes the columns and gets the verdict)
    return rc;
  } catch (const std::bad_alloc&) { s->err = "out of memory"; return MCOV_ERR_NOMEM; }
  catch (...) { s->err = "unexpected failure"; return MCOV_ERR_IO; }
}

}  // extern "C"

// ===========================================================================================================
// BAM writer (bench / test support): SoA columns -> a BGZF-compressed BAM + the metadata-only BAI the coverage
// path reads (`mapped` / `unmapped`).  Read names are "r<index>", SEQ is pseudo-random ACGT (so that the file
// compresses like sequence data, not like padding), QUAL is 0xff (absent).  Blocks are deflated in parallel.
// The reference has no writer on this path; its fixtures were made by samtools.
// ===========================================================================================================
namespace {

inline void put32(std::vector<uint8_t>& v, uint32_t x) { v.push_back((uint8_t)x); v.push_back((uint8_t)(x >> 8)); v.push_back((uint8_t)(x >> 16)); v.push_back((uint8_t)(x >> 24)); }
inline void put16(std::vector<uint8_t>& v, uint16_t x) { v.push_back((uint8_t)x); v.push_back((uint8_t)(x >> 8)); }

int reg2bin(int64_t beg, int64_t end) {               // SAM spec 5.3
  --end;
  if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

bool bgzf_block(const uint8_t* src, size_t n, int level, std::vector<uint8_t>& out) {
  z_stream zs;
  std::memset(&zs, 0, sizeof(zs));
  if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) return false;
  std::vector<uint8_t> c(deflateBound(&zs, (uLong)n) + 64);
  zs.next_in = const_cast<Bytef*>(src); zs.avail_in = (uInt)n;
  zs.next_out = c.data(); zs.avail_out = (uInt)c.size();
  const int rc = deflate(&zs, Z_FINISH);
  const size_t clen = zs.total_out;
  deflateEnd(&zs);
  if (rc != Z_STREAM_END || clen + 26 > 65536) return false;
  const uint8_t head[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
  out.assign(head, head + 16);
  put16(out, (uint16_t)(clen + 25));
  out.insert(out.end(), c.begin(), c.begin() + (ptrdiff_t)clen);
  put32(out, (uint32_t)crc32(crc32(0L, Z_NULL, 0), src, (uInt)n));
  put32(out, (uint32_t)n);
  return true;
}

}  // namespace

extern "C" int mcov_bam_write(const char* path, int32_t n_ref, const char* const* ref_name, const int32_t* ref_len, int64_t n,
                              const int32_t* tid, const int32_t* pos, const uint16_t* flag, const uint8_t* mapq,
                              const uint32_t* cig_off, const uint32_t* cig, const int32_t* isize, int level, int n_threads) {
  if (!path || n_ref <= 0 || !ref_name || !ref_len || n < 0 || (n > 0 && (!tid || !pos || !flag || !mapq || !cig_off))) return MCOV_ERR_ARG;
  try {
    if (n_threads <= 0) { unsigned hw = std::thread::hardware_concurrency(); n_threads = hw ? (int)std::min(hw, 32u) : 4; }
    std::vector<uint8_t> head;
    std::string text = "@HD\tVN:1.4\tSO:coordinate\n";
    for (int32_t r = 0; r < n_ref; ++r) text += std::string("@SQ\tSN:") + ref_name[r] + "\tLN:" + std::to_string(ref_len[r]) + "\n";
    head.insert(head.end(), {'B', 'A', 'M', 1});
    put32(head, (uint32_t)text.size());
    head.insert(head.end(), text.begin(), text.end());
    put32(head, (uint32_t)n_ref);
    for (int32_t r = 0; r < n_ref; ++r) {
      const size_t l = std::strlen(ref_name[r]) + 1;
      put32(head, (uint32_t)l);
      head.insert(head.end(), ref_name[r], ref_name[r] + l);
      put32(head, (uint32_t)ref_len[r]);
    }
    // records are serialised by ranges of reads in parallel, then cut into BGZF payloads of <= 0xff00 bytes
    std::vector<std::vector<uint8_t>> part((size_t)n_threads);
    const int64_t per = (n + n_threads - 1) / std::max(n_threads, 1);
    auto ser = [&](int t) {
      std::vector<uint8_t>& v = part[(size_t)t];
      const int64_t a = t * per, b = std::min(n, a + per);
      if (a >= b) return;
      v.reserve((size_t)(b - a) * 260);
      for (int64_t i = a; i < b; ++i) {
        char name[24];
        const int ln = std::snprintf(name, sizeof(name), "r%lld", (long long)i) + 1;
        const uint32_t nc = cig_off[i + 1] - cig_off[i];
        int64_t ls = 0, rl = 0;
        for (uint32_t k = 0; k < nc; ++k) {
          const uint32_t op = cig[cig_off[i] + k], o = op & 15u, l = op >> 4;
          if (o == 0 || o == 1 || o == 4 || o == 7 || o == 8) ls += l;       // M I S = X consume the query
          if ((0x18Du >> o) & 1u) rl += l;
        }
        const size_t body = 32 + (size_t)ln + 4 * (size_t)nc + (size_t)(ls + 1) / 2 + (size_t)ls;
        put32(v, (uint32_t)body);
        put32(v, (uint32_t)tid[i]); put32(v, (uint32_t)pos[i]);
        v.push_back((uint8_t)ln); v.push_back(mapq[i]);
        const int64_t p0 = std::max<int64_t>(pos[i], 0);
        put16(v, tid[i] >= 0 ? (uint16_t)reg2bin(p0, p0 + std::max<int64_t>(rl, 1)) : (uint16_t)4680);
        put16(v, (uint16_t)nc); put16(v, flag[i]);
        put32(v, (uint32_t)ls); put32(v, 0xFFFFFFFFu); put32(v, 0xFFFFFFFFu); put32(v, isize ? (uint32_t)isize[i] : 0u);
        v.insert(v.end(), name, name + ln);
        const uint8_t* cp = reinterpret_cast<const uint8_t*>(cig + cig_off[i]);
        v.insert(v.end(), cp, cp + 4 * (size_t)nc);
        uint64_t x = 0x9E3779B97F4A7C15ull * (uint64_t)(i + 1);
        static const uint8_t nt[4] = {1, 2, 4, 8};
        for (int64_t k = 0; k < (ls + 1) / 2; ++k) {
          x ^= x << 13; x ^= x >> 7; x ^= x << 17;
          const uint8_t hi = nt[x & 3], lo = (2 * k + 1 < ls) ? nt[(x >> 2) & 3] : 0;
          v.push_back((uint8_t)((hi << 4) | lo));
        }
        v.insert(v.end(), (size_t)ls, (uint8_t)0xff);
      }
    };
    {
      std::vector<std::thread> th;
      for (int t = 1; t < n_threads; ++t) th.emplace_back(ser, t);
      ser(0);
      for (auto& t : th) t.join();
    }
    // one logical stream: header + parts; payload boundaries every 0xff00 bytes
    std::vector<const std::vector<uint8_t>*> segs;
    segs.push_back(&head);
    for (auto& p : part) if (!p.empty()) segs.push_back(&p);
    size_t total = 0;
    for (auto* sgm : segs) total += sgm->size();
    std::vector<uint8_t> stream;
    stream.reserve(total);
    for (auto* sgm : segs) stream.insert(stream.end(), sgm->begin(), sgm->end());
    for (auto& p : part) std::vector<uint8_t>().swap(p);
    const size_t kPay = 0xff00, n_blk = (total + kPay - 1) / kPay;
    std::vector<std::vector<uint8_t>> blk(n_blk);
    std::atomic<size_t> next(0);
    std::atomic<bool> good(true);
    auto comp = [&]() {
      for (;;) {
        const size_t k = next.fetch_add(1);
        if (k >= n_blk || !good.load()) break;
        const size_t a = k * kPay, len = std::min(kPay, total - a);
        if (!bgzf_block(stream.data() + a, len, level, blk[k])) good.store(false);
      }
    };
    {
      std::vector<std::thread> th;
      for (int t = 1; t < n_threads; ++t) th.emplace_back(comp);
      comp();
      for (auto& t : th) t.join();
    }
    if (!good.load()) return MCOV_ERR_IO;
    FILE* fh = std::fopen(path, "wb");
    if (!fh) return MCOV_ERR_IO;
    bool ok = true;
    for (auto& b : blk) ok = ok && std::fwrite(b.data(), 1, b.size(), fh) == b.size();
    static const uint8_t eof_blk[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    ok = ok && std::fwrite(eof_blk, 1, 28, fh) == 28;
    ok = (std::fclose(fh) == 0) && ok;
    if (!ok) return MCOV_ERR_IO;
    // metadata-only index: per reference one pseudo-bin 37450 with the mapped / unmapped counts
    std::vector<uint64_t> n_map((size_t)n_ref, 0), n_un((size_t)n_ref, 0);
    uint64_t no_coor = 0;
    for (int64_t i = 0; i < n; ++i) {
      if (tid[i] < 0 || tid[i] >= n_ref) { ++no_coor; continue; }
      if (flag[i] & 4) ++n_un[(size_t)tid[i]]; else ++n_map[(size_t)tid[i]];
    }
    std::vector<uint8_t> bai = {'B', 'A', 'I', 1};
    put32(bai, (uint32_t)n_ref);
    for (int32_t r = 0; r < n_ref; ++r) {
      put32(bai, 1); put32(bai, 37450); put32(bai, 2);
      for (uint64_t v : {(uint64_t)0, (uint64_t)0, n_map[(size_t)r], n_un[(size_t)r]}) { put32(bai, (uint32_t)v); put32(bai, (uint32_t)(v >> 32)); }
      put32(bai, 0);
    }
    put32(bai, (uint32_t)no_coor); put32(bai, (uint32_t)(no_coor >> 32));
    const std::string ipath = std::string(path) + ".bai";
    fh = std::fopen(ipath.c_str(), "wb");
    if (!fh) return MCOV_ERR_IO;
    ok = std::fwrite(bai.data(), 1, bai.size(), fh) == bai.size();
    ok = (std::fclose(fh) == 0) && ok;
    return ok ? MCOV_OK : MCOV_ERR_IO;
  } catch (const std::bad_alloc&) { return MCOV_ERR_NOMEM; }
  catch (...) { return MCOV_ERR_IO; }
}
