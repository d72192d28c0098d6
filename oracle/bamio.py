"""Pure-Python BGZF / BAM / BAI decoder (oracle side; test infrastructure only).

Restates the on-disk formats of the SAM specification v1 section 4 (BGZF 4.1,
BAM 4.2, BAI 5.2).  The reference reaches these formats through pysam/htslib
(reference metacov/cli.py:56, 211; metacov/scan.pyx:204, 216, 243-294), which is
not vendored; this module is the independent restatement the product's C++
reader (metacov_b200/csrc/bamio.cpp) is checked against.
"""
import struct
import zlib
from collections import namedtuple

import numpy as np

CIGAR_OPS = "MIDNSHP=X"
# ops that consume reference: M(0) D(2) N(3) =(7) X(8)   (htslib bam_cigar_type & 2)
CONSUMES_REF = np.array([1, 0, 1, 1, 0, 0, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0], dtype=np.int64)
# ops that consume query: M(0) I(1) S(4) =(7) X(8)
CONSUMES_QRY = np.array([1, 1, 0, 0, 1, 0, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0], dtype=np.int64)
NT16 = "=ACMGRSVTWYHKDBN"

BamHeader = namedtuple("BamHeader", "text references lengths")


def bgzf_inflate(raw):
    """Concatenate the inflated payloads of all BGZF members in ``raw``."""
    out = []
    off = 0
    n = len(raw)
    while off < n:
        if raw[off:off + 4] != b"\x1f\x8b\x08\x04":
            raise ValueError("not a BGZF member at offset %d" % off)
        xlen = struct.unpack_from("<H", raw, off + 10)[0]
        # walk the extra subfields looking for 'BC'
        p = off + 12
        bsize = None
        while p < off + 12 + xlen:
            si1, si2, slen = struct.unpack_from("<BBH", raw, p)
            if si1 == 66 and si2 == 67 and slen == 2:
                bsize = struct.unpack_from("<H", raw, p + 4)[0]
            p += 4 + slen
        if bsize is None:
            raise ValueError("BGZF member without BC subfield")
        cdata = raw[off + 12 + xlen: off + bsize + 1 - 8]
        crc, isize = struct.unpack_from("<II", raw, off + bsize + 1 - 8)
        data = zlib.decompress(cdata, -15) if isize else b""
        if len(data) != isize or (zlib.crc32(data) & 0xFFFFFFFF) != crc:
            raise ValueError("BGZF block CRC/size mismatch")
        out.append(data)
        off += bsize + 1
    return b"".join(out)


class BamRecords:
    """All records of a BAM file as SoA numpy arrays (file order)."""

    def __init__(self):
        self.tid = self.pos = self.flag = self.mapq = None
        self.l_seq = self.isize = self.mtid = self.mpos = None
        self.cig_off = self.cig = None
        self.names = []
        self.seqs = []      # nt16 codes per read (np.uint8 arrays), as stored
        self.reflen = None  # sum of ref-consuming op lengths (htslib bam_cigar2rlen)

    def __len__(self):
        return len(self.tid)


def read_bam(path, want_seq=True):
    """Decode ``path`` -> (BamHeader, BamRecords)."""
    with open(path, "rb") as fh:
        data = bgzf_inflate(fh.read())
    if data[:4] != b"BAM\x01":
        raise ValueError("not a BAM file")
    l_text = struct.unpack_from("<i", data, 4)[0]
    text = data[8:8 + l_text].split(b"\0", 1)[0].decode()
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", data, p)[0]
    p += 4
    names, lens = [], []
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", data, p)[0]
        names.append(data[p + 4:p + 4 + l_name - 1].decode())
        lens.append(struct.unpack_from("<i", data, p + 4 + l_name)[0])
        p += 8 + l_name
    hdr = BamHeader(text, tuple(names), tuple(lens))

    tid, pos, flag, mapq, lseq, isz, mtid, mpos = [], [], [], [], [], [], [], []
    cig_off, cig, rnames, seqs = [0], [], [], []
    n = len(data)
    while p < n:
        (block_size, refid, ps, l_read_name, mq, _bin, n_cig, fl, l_seq,
         next_refid, next_pos, tlen) = struct.unpack_from("<iiiBBHHHiiii", data, p)
        q = p + 36
        rnames.append(data[q:q + l_read_name - 1].decode())
        q += l_read_name
        ops = np.frombuffer(data, dtype="<u4", count=n_cig, offset=q)
        q += 4 * n_cig
        if want_seq:
            packed = np.frombuffer(data, dtype=np.uint8, count=(l_seq + 1) // 2, offset=q)
            nt = np.empty(2 * len(packed), dtype=np.uint8)
            nt[0::2] = packed >> 4
            nt[1::2] = packed & 15
            seqs.append(nt[:l_seq].copy())
        tid.append(refid); pos.append(ps); flag.append(fl); mapq.append(mq)
        lseq.append(l_seq); isz.append(tlen); mtid.append(next_refid); mpos.append(next_pos)
        cig.append(ops)
        cig_off.append(cig_off[-1] + n_cig)
        p += 4 + block_size
    r = BamRecords()
    r.tid = np.asarray(tid, dtype=np.int32)
    r.pos = np.asarray(pos, dtype=np.int32)
    r.flag = np.asarray(flag, dtype=np.uint16)
    r.mapq = np.asarray(mapq, dtype=np.uint8)
    r.l_seq = np.asarray(lseq, dtype=np.int32)
    r.isize = np.asarray(isz, dtype=np.int32)
    r.mtid = np.asarray(mtid, dtype=np.int32)
    r.mpos = np.asarray(mpos, dtype=np.int32)
    r.cig_off = np.asarray(cig_off, dtype=np.int64)
    r.cig = (np.concatenate(cig) if cig else np.zeros(0, np.uint32)).astype(np.uint32)
    r.names = rnames
    r.seqs = seqs
    r.reflen = cigar_reflen(r.cig_off, r.cig)
    return hdr, r


def cigar_reflen(cig_off, cig):
    """Per-read reference length = sum of len(op) for op in {M,D,N,=,X}.

    htslib ``bam_cigar2rlen``; pysam ``reference_length`` (reference
    metacov/pileup.py:134,137 consumes it as ``read.reference_length``).
    """
    cig = np.asarray(cig, dtype=np.uint32)
    cig_off = np.asarray(cig_off, dtype=np.int64)
    contrib = (cig >> 4).astype(np.int64) * CONSUMES_REF[cig & 15]
    csum = np.concatenate(([0], np.cumsum(contrib)))
    return (csum[cig_off[1:]] - csum[cig_off[:-1]]).astype(np.int64)


def read_bai_stats(path, n_ref=None):
    """Per-reference (n_mapped, n_unmapped) from the BAI metadata pseudo-bin
    37450 and the trailing n_no_coor (SAM spec 5.2).  pysam's
    ``AlignmentFile.mapped`` / ``.unmapped`` (reference metacov/cli.py:73-75,
    214-216) are sums over these."""
    with open(path, "rb") as fh:
        d = fh.read()
    if d[:4] != b"BAI\x01":
        raise ValueError("not a BAI file")
    n = struct.unpack_from("<i", d, 4)[0]
    p = 8
    per_ref = []
    for _ in range(n):
        n_bin = struct.unpack_from("<i", d, p)[0]
        p += 4
        mapped = unmapped = 0
        for _b in range(n_bin):
            bin_id, n_chunk = struct.unpack_from("<Ii", d, p)
            p += 8
            if bin_id == 37450 and n_chunk == 2:
                # chunk 0 = (off_beg, off_end), chunk 1 = (n_mapped, n_unmapped)
                mapped, unmapped = struct.unpack_from("<QQ", d, p + 16)
            p += 16 * n_chunk
        n_intv = struct.unpack_from("<i", d, p)[0]
        p += 4 + 8 * n_intv
        per_ref.append((mapped, unmapped))
    n_no_coor = struct.unpack_from("<Q", d, p)[0] if p + 8 <= len(d) else 0
    return per_ref, n_no_coor


# --------------------------------------------------------------------------
# writers (test fixtures only): BGZF/BAM and a statistics-only BAI
# --------------------------------------------------------------------------

def _bgzf_block(payload):
    comp = zlib.compressobj(6, zlib.DEFLATED, -15)
    cdata = comp.compress(payload) + comp.flush()
    bsize = len(cdata) + 25
    head = struct.pack("<BBBBIBBHBBHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, 66, 67, 2, bsize)
    return head + cdata + struct.pack("<II", zlib.crc32(payload) & 0xFFFFFFFF, len(payload))


BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_compress(data, block=0xff00):
    out = [_bgzf_block(data[i:i + block]) for i in range(0, len(data), block)]
    out.append(BGZF_EOF)
    return b"".join(out)


def reg2bin(beg, end):
    """SAM spec 5.3."""
    end -= 1
    if beg >> 14 == end >> 14:
        return ((1 << 15) - 1) // 7 + (beg >> 14)
    if beg >> 17 == end >> 17:
        return ((1 << 12) - 1) // 7 + (beg >> 17)
    if beg >> 20 == end >> 20:
        return ((1 << 9) - 1) // 7 + (beg >> 20)
    if beg >> 23 == end >> 23:
        return ((1 << 6) - 1) // 7 + (beg >> 23)
    if beg >> 26 == end >> 26:
        return ((1 << 3) - 1) // 7 + (beg >> 26)
    return 0


def write_bam(path, references, lengths, tid, pos, flag, mapq, cig_off, cig, l_seq=None, isize=None,
              names=None, seqs=None, text=None, with_index=True, aux=None):
    """Write a BAM (and a BAI that carries only the metadata pseudo-bins) from SoA arrays.
    ``aux``: optional per-record bytes of encoded optional fields (SAM spec 4.2.4), appended after the qualities."""
    n = len(tid)
    if text is None:
        text = "@HD\tVN:1.4\tSO:coordinate\n" + "".join(
            "@SQ\tSN:%s\tLN:%d\n" % (r, l) for r, l in zip(references, lengths))
    tb = text.encode()
    parts = [b"BAM\x01", struct.pack("<i", len(tb)), tb, struct.pack("<i", len(references))]
    for r, l in zip(references, lengths):
        rb = r.encode() + b"\0"
        parts += [struct.pack("<i", len(rb)), rb, struct.pack("<i", l)]
    reflen = cigar_reflen(cig_off, cig)
    for i in range(n):
        name = (names[i] if names is not None else "r%d" % i).encode() + b"\0"
        ops = np.asarray(cig[int(cig_off[i]):int(cig_off[i + 1])], dtype="<u4")
        ls = int(l_seq[i]) if l_seq is not None else int(
            ((ops >> 4).astype(np.int64) * CONSUMES_QRY[ops & 15]).sum())
        if seqs is not None:
            nt = np.asarray(seqs[i], dtype=np.uint8)
            ls = len(nt)
        else:
            nt = np.full(ls, 1, dtype=np.uint8)        # all 'A'
        if len(nt) % 2:
            nt = np.concatenate([nt, [0]]).astype(np.uint8)
        packed = ((nt[0::2] << 4) | nt[1::2]).astype(np.uint8).tobytes()
        qual = b"\xff" * ls
        end = int(pos[i]) + max(int(reflen[i]), 1)
        body = struct.pack("<iiBBHHHiiii", int(tid[i]), int(pos[i]), len(name), int(mapq[i]),
                           reg2bin(max(int(pos[i]), 0), max(end, 1)) if tid[i] >= 0 else 4680,
                           len(ops), int(flag[i]), ls, -1, -1, int(isize[i]) if isize is not None else 0)
        body += name + ops.tobytes() + packed + qual + (aux[i] if aux is not None else b"")
        parts.append(struct.pack("<i", len(body)) + body)
    with open(path, "wb") as fh:
        fh.write(bgzf_compress(b"".join(parts)))
    if with_index:
        tid = np.asarray(tid); flag = np.asarray(flag)
        out = [b"BAI\x01", struct.pack("<i", len(references))]
        for c in range(len(references)):
            sel = tid == c
            n_un = int(np.sum(sel & ((flag & 4) != 0)))
            n_map = int(np.sum(sel)) - n_un
            out.append(struct.pack("<i", 1) + struct.pack("<Ii", 37450, 2) +
                       struct.pack("<QQQQ", 0, 0, n_map, n_un) + struct.pack("<i", 0))
        out.append(struct.pack("<Q", int(np.sum(tid < 0))))
        with open(path + ".bai", "wb") as fh:
            fh.write(b"".join(out))
