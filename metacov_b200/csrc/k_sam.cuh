// k_sam.cuh -- SAM text -> BAM columns: the per-field rules (SAM spec v1 1.4; the BAM encoding of htslib's sam_parse1),
// shared by the device parser (sam_gpu.cu) and its host-compiled test hook (mcov_sam_parse_host).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MCOV_HD __host__ __device__ __forceinline__
#else
#define MCOV_HD inline
#endif

namespace mcov {

// the 11 mandatory fields, and the error codes past them (low byte of a SamErr)
enum SamField { kQname = 0, kFlag, kRname, kPos, kMapq, kCigar, kRnext, kPnext, kTlen, kSeq, kQual, kSamFields };
enum SamErrKind { kErrFewFields = 11, kErrHeaderAfter = 12, kErrLineLong = 13 };
// a failure: (record index << 8) | field or kind; the smallest one wins (atomicMin), ~0 = none
constexpr unsigned long long kSamNoErr = ~0ull;

constexpr uint64_t kSamMaxOpLen = (1u << 28) - 1u;

struct SamAux { uint32_t l_qname, cig_b, cig_e, seq_b; };              // field offsets from the line start (device decode)

// unsigned decimal of [p, p + n) in [0, max]; false for an empty field, a non-digit or a value past max
MCOV_HD bool sam_dec_u(const uint8_t* p, uint32_t n, uint64_t max, uint64_t* v) {
  if (n == 0) return false;
  uint64_t x = 0;
  for (uint32_t k = 0; k < n; ++k) {
    const uint32_t c = (uint32_t)p[k] - '0';
    if (c > 9u) return false;
    x = x * 10u + c;
    if (x > max) return false;
  }
  *v = x;
  return true;
}

// signed decimal ([-]digits) in int32
MCOV_HD bool sam_dec_i32(const uint8_t* p, uint32_t n, int32_t* v) {
  const bool neg = n > 0 && p[0] == '-';
  uint64_t x = 0;
  if (!sam_dec_u(p + neg, n - neg, neg ? 0x80000000ull : 0x7FFFFFFFull, &x)) return false;
  *v = neg ? (int32_t)(0u - (uint32_t)x) : (int32_t)x;
  return true;
}

// CIGAR op letter -> BAM op code (MIDNSHP=X -> 0..8), -1 for any other byte
MCOV_HD int sam_cigar_op(uint32_t c) {
  switch (c) {
    case 'M': return 0; case 'I': return 1; case 'D': return 2; case 'N': return 3; case 'S': return 4;
    case 'H': return 5; case 'P': return 6; case '=': return 7; case 'X': return 8; default: return -1;
  }
}

// SEQ byte -> nt16 code of "=ACMGRSVTWYHKDBN" (case-insensitive); any other byte is 15 (N)
MCOV_HD uint32_t sam_nt16(uint32_t c) {
  c |= (c >= 'A' && c <= 'Z') ? 0x20u : 0u;
  switch (c) {
    case '=': return 0; case 'a': return 1; case 'c': return 2; case 'm': return 3; case 'g': return 4; case 'r': return 5;
    case 's': return 6; case 'v': return 7; case 't': return 8; case 'w': return 9; case 'y': return 10; case 'h': return 11;
    case 'k': return 12; case 'd': return 13; case 'b': return 14; default: return 15;
  }
}

MCOV_HD bool sam_is_star(const uint8_t* p, uint32_t n) { return n == 1 && p[0] == '*'; }

// FNV-1a 32 of a reference name: the slot of the @SQ name table
MCOV_HD uint32_t sam_name_hash32(const uint8_t* p, uint32_t n) {
  uint32_t h = 2166136261u;
  for (uint32_t k = 0; k < n; ++k) { h ^= p[k]; h *= 16777619u; }
  return h;
}

// The key of a read name: FNV-1a 64 of the name's bytes, with ~0 folded to ~0 - 1 (~0 is the "no entry" key of the pair
// sort of pileup.experimental).  The name is base[at, at + len - kNul): BAM's l_read_name counts a closing NUL that is
// not hashed (kNul 1), a SAM QNAME is len bytes (kNul 0).  The one definition of the key that joins mates:
// k_bam_names_seq, sam_names_seq_one and the linkage observations (k_linkage.cuh) all take it from here (the loop keeps
// the form each of the first two had, so that they compile as before); the host reader's mcov_bam_name_hash computes
// the same value.
template <uint32_t kNul>
MCOV_HD uint64_t read_name_key(const uint8_t* base, uint32_t at, uint32_t len) {
  uint64_t h = 1469598103934665603ull;
  for (uint32_t k = 0; k + kNul < len; ++k) { h ^= base[at + k]; h *= 1099511628211ull; }
  return h == ~0ull ? h - 1 : h;
}

// The @SQ names as an open-addressing table: slot -> tid (-1 empty), names in one blob at name_off[tid].
struct SamRefTable {
  const int32_t* slot; uint32_t mask;
  const uint8_t* names; const uint64_t* name_off;
};

// RNAME -> tid, exact byte compare; -1 = no such @SQ name
MCOV_HD int32_t sam_ref_lookup(const SamRefTable& t, const uint8_t* p, uint32_t n) {
  for (uint32_t s = sam_name_hash32(p, n) & t.mask;; s = (s + 1u) & t.mask) {
    const int32_t r = t.slot[s];
    if (r < 0) return -1;
    const uint64_t a = t.name_off[r], b = t.name_off[r + 1];
    if (b - a == n) {
      uint32_t k = 0;
      while (k < n && t.names[a + k] == p[k]) ++k;
      if (k == n) return r;
    }
  }
}

// One mandatory field other than CIGAR and RNAME (which need the op stream / the name table): validated and, where the
// columns keep it, converted into *v.  `seq_len` is l_seq (for QUAL).  false = the field breaks its rule.
MCOV_HD bool sam_field_value(int f, const uint8_t* p, uint32_t n, int64_t seq_len, int64_t* v) {
  uint64_t u = 0;
  int32_t s = 0;
  switch (f) {
    case kQname: *v = n; return n >= 1 && n <= 254;
    case kFlag: if (!sam_dec_u(p, n, 65535, &u)) return false; *v = (int64_t)u; return true;
    case kPos: case kPnext: if (!sam_dec_u(p, n, 0x7FFFFFFFull, &u)) return false; *v = (int64_t)u - 1; return true;
    case kMapq: if (!sam_dec_u(p, n, 255, &u)) return false; *v = (int64_t)u; return true;
    case kRnext: *v = 0; return n >= 1;
    case kTlen: if (!sam_dec_i32(p, n, &s)) return false; *v = s; return true;
    case kSeq: if (n == 0) return false; *v = sam_is_star(p, n) ? 0 : (int64_t)n; return true;
    case kQual: *v = 0; return n >= 1 && (sam_is_star(p, n) || (int64_t)n == seq_len);
    default: *v = 0; return n >= 1;
  }
}

// Names and SEQ of one record straight from its text, the outputs of k_bam_names_seq with the same definitions:
// FNV-1a 64 of QNAME (~0 folded to ~0-1), the 2-bit code of query_alignment_sequence[0:k_len] (soft clips of the decoded
// CIGAR skipped; -1 = no key) and the first / last win_bases bases as nt16 nibbles ('N' padded).
MCOV_HD void sam_names_seq_one(const uint8_t* qname, uint32_t l_qname, const uint8_t* seq, int64_t l_seq, uint32_t flag,
                               const uint32_t* cig, uint32_t n_op, int32_t k_len, int32_t win_bases, uint64_t* name_hash,
                               int32_t* kmer_code, uint8_t* win) {
  if (name_hash) *name_hash = read_name_key<0>(qname, 0, l_qname);
  if (kmer_code) {
    int64_t lo = 0, hi = l_seq;
    for (uint32_t k = 0; k < n_op; ++k) {
      const uint32_t c = cig[k], op = c & 15u;
      if (op == 5) continue;
      if (op == 4) lo += c >> 4; else break;
    }
    for (uint32_t k = n_op; k > 0; --k) {
      const uint32_t c = cig[k - 1], op = c & 15u;
      if (op == 5) continue;
      if (op == 4) hi -= c >> 4; else break;
    }
    int32_t code = hi - lo < k_len ? -1 : 0;
    for (int32_t j = 0; j < k_len && code >= 0; ++j) {
      const uint32_t b = sam_nt16(seq[lo + j]);
      const int c = b == 1 ? 0 : b == 2 ? 1 : b == 4 ? 2 : b == 8 ? 3 : -1;
      code = c < 0 ? -1 : (code << 2) | c;
    }
    *kmer_code = code;
  }
  if (win) {
    const int W = (win_bases + 1) / 2;
    const bool rev = (flag & 0x10u) != 0;
    for (int b2 = 0; b2 < W; ++b2) {
      uint32_t v = 0;
      for (int h = 0; h < 2; ++h) {
        const int j = 2 * b2 + h;
        uint32_t c = 15;
        if (j < win_bases) {
          const int64_t a = rev ? l_seq - win_bases + j : j;
          if (a >= 0 && a < l_seq) c = sam_nt16(seq[a]);
        }
        v = (v << 4) | c;
      }
      win[b2] = (uint8_t)v;
    }
  }
}

}  // namespace mcov
