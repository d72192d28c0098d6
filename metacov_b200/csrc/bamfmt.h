// bamfmt.h -- the BGZF and BAM format rules (SAM spec v1 section 4.1 BGZF, 4.2 BAM) shared by the host readers
// (bamio.cpp) and the host side of the GPU decoder (bam_gpu.cu): little-endian reads, the BGZF block table, the BAM
// header and a record's fixed fields.  Plain host code: no CUDA, no zlib.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

namespace mcov {

inline uint16_t rd16(const uint8_t* p) { return (uint16_t)(p[0] | (p[1] << 8)); }
inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline uint64_t rd64(const uint8_t* p) { return (uint64_t)rd32(p) | ((uint64_t)rd32(p + 4) << 32); }

// One BGZF block: the deflate data at [coff, coff + clen) of the file inflates to the ulen bytes at uoff of the stream,
// whose CRC-32 is crc.  k_bgzf_inflate takes an array of these, so the layout is fixed.
struct BgzfBlock { uint64_t coff; uint64_t uoff; uint32_t clen; uint32_t ulen; uint32_t crc; uint32_t pad; };

// The BGZF blocks of raw[0, n) (gzip members with a 'BC' extra field holding BSIZE), their output placed from uoff0 on.
// partial: raw ends where a read of the file ended, so an incomplete last block is left for the next read; otherwise
// raw must be whole blocks.  Sets blocks, end (uoff0 + the inflated bytes) and used (the bytes the blocks take); false
// on a malformed block.
inline bool bgzf_index(const uint8_t* raw, size_t n, uint64_t uoff0, bool partial, std::vector<BgzfBlock>& blocks,
                       uint64_t& end, size_t& used) {
  blocks.clear();
  size_t off = 0;
  uint64_t uoff = uoff0;
  while (off + 18 <= n) {
    const uint8_t* h = raw + off;
    if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return false;
    const size_t xend = off + 12 + rd16(h + 10);
    if (xend > n) break;
    int bsize = -1;
    for (size_t p = off + 12; p + 4 <= xend; p += 4 + rd16(raw + p + 2))
      if (raw[p] == 'B' && raw[p + 1] == 'C' && rd16(raw + p + 2) == 2 && p + 6 <= xend) bsize = rd16(raw + p + 4);
    if (bsize < 0) return false;
    const size_t bend = off + (size_t)bsize + 1;
    if (bend > n) break;
    if (bend < xend + 8) return false;                       // no room for CRC32 and ISIZE
    BgzfBlock b;
    b.coff = xend;
    b.clen = (uint32_t)(bend - 8 - xend);
    b.crc = rd32(raw + bend - 8);
    b.ulen = rd32(raw + bend - 4);
    if (b.ulen > 65536u) return false;                       // a block inflates to at most 64 KiB
    b.uoff = uoff;
    b.pad = 0;
    uoff += b.ulen;
    blocks.push_back(b);
    off = bend;
  }
  end = uoff;
  used = off;
  return partial || off == n;
}

// The BAM header: magic, l_text, text, n_ref, reference table.
struct BamHeader {
  size_t rec_begin = 0;                  // where the first alignment record starts
  int32_t n_ref = 0;
  const char* bad = nullptr;             // kBad: what is wrong ("not a valid BAM file", "bad reference count")
  std::string text;                      // the text up to its first NUL; text, names and lens only when asked for
  std::vector<std::string> names;
  std::vector<int32_t> lens;
};
// kMoreText / kMoreRefs: the prefix ends in the magic, text or n_ref / in the reference table
enum class HeaderParse { kOk, kMoreText, kMoreRefs, kBad };

// The header at the front of d[0, n), a prefix of the inflated stream.
inline HeaderParse parse_bam_header(const uint8_t* d, size_t n, bool with_names, BamHeader& h) {
  if (n < 12) return HeaderParse::kMoreText;
  if (std::memcmp(d, "BAM\1", 4) != 0) { h.bad = "not a valid BAM file"; return HeaderParse::kBad; }
  const uint32_t l_text = rd32(d + 4);
  size_t p = 8 + (size_t)l_text;
  if (p + 4 > n) return HeaderParse::kMoreText;
  h.n_ref = (int32_t)rd32(d + p);
  if (h.n_ref < 0) { h.bad = "bad reference count"; return HeaderParse::kBad; }
  p += 4;
  h.names.clear();
  h.lens.clear();
  for (int32_t i = 0; i < h.n_ref; ++i) {
    if (p + 4 > n) return HeaderParse::kMoreRefs;
    const uint32_t l_name = rd32(d + p);                    // includes the NUL
    if (l_name == 0) { h.bad = "not a valid BAM file"; return HeaderParse::kBad; }
    if (p + 8 + (size_t)l_name > n) return HeaderParse::kMoreRefs;
    if (with_names) {
      h.names.emplace_back(reinterpret_cast<const char*>(d + p + 4), l_name - 1);
      h.lens.push_back((int32_t)rd32(d + p + 4 + l_name));
    }
    p += 8 + (size_t)l_name;
  }
  if (with_names) h.text.assign(reinterpret_cast<const char*>(d + 8), strnlen(reinterpret_cast<const char*>(d + 8), l_text));
  h.rec_begin = p;
  return HeaderParse::kOk;
}

// An alignment record (SAM spec 4.2); r points behind its block_size field.
inline uint16_t record_n_op(const uint8_t* r) { return rd16(r + 12); }

// fixed part + name + CIGAR + SEQ + QUAL of a record must fit its block_size
inline bool record_fits(const uint8_t* r, uint32_t bs) {
  const uint64_t l_read_name = r[8], n_op = record_n_op(r), l_seq = rd32(r + 16);
  return 32ull + l_read_name + 4ull * n_op + (l_seq + 1) / 2 + l_seq <= (uint64_t)bs;
}

// host columns a record's fixed fields go to
struct RecordCols { int32_t *tid, *pos, *l_seq, *isize; uint16_t* flag; uint8_t* mapq; };

// The fixed fields of the record at r into row i of c and its CIGAR to cig (record_fits holds); returns the op count.
inline uint16_t copy_record(const uint8_t* r, const RecordCols& c, size_t i, uint32_t* cig) {
  c.tid[i] = (int32_t)rd32(r);
  c.pos[i] = (int32_t)rd32(r + 4);
  c.mapq[i] = r[9];
  c.flag[i] = rd16(r + 14);
  c.l_seq[i] = (int32_t)rd32(r + 16);
  c.isize[i] = (int32_t)rd32(r + 28);
  const uint16_t n_op = record_n_op(r);
  std::memcpy(cig, r + 32 + r[8], 4u * n_op);
  return n_op;
}

}  // namespace mcov
