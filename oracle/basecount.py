"""pysam's ``AlignmentFile.count_coverage`` restated as a plain loop over records (SoA columns + SEQ + QUAL): the
reference the product's device counts (``metacov_b200.AlignmentFile.count_coverage``) are checked against.

Records are given as the decoded columns (tid, pos, flag, cig_off, cig) plus, per record, SEQ as nt16 codes
("=ACMGRSVTWYHKDBN" -> 0..15; an empty array for SEQ '*') and QUAL as Phred values (None for "no qualities": BAM's 0xff,
SAM's '*').  Test infrastructure only: the product never imports it.
"""
import numpy as np

SKIP_ALL = 0x4 | 0x100 | 0x200 | 0x400        # read_callback="all": unmapped, secondary, QC fail, duplicate
CONSUMES_QUERY = (0, 1, 4, 7, 8)             # M I S = X
CONSUMES_REF = (0, 2, 3, 7, 8)               # M D N = X
ALIGNED = (0, 7, 8)                          # M = X: the ops that make (qpos, refpos) pairs
BASE_INDEX = {1: 0, 2: 1, 4: 2, 8: 3}        # nt16 A C G T -> row of the result


def _mode(read_callback):
    if isinstance(read_callback, str) and read_callback in ("all", "nofilter"):
        return read_callback
    raise ValueError("read_callback must be 'all' or 'nofilter', got %r" % (read_callback,))


def full_counts(lengths, tid, pos, flag, cig_off, cig, seqs, quals, quality_threshold=15, read_callback="all"):
    """uint32 [4, length] per contig: A, C, G, T counts of every position over every record.  Raises IndexError
    naming the first counted record whose CIGAR consumes more query bases than its SEQ holds."""
    mode = _mode(read_callback)
    t = int(quality_threshold or 0)
    out = [np.zeros((4, int(l)), dtype=np.uint32) for l in lengths]
    for i in range(len(tid)):
        c, p = int(tid[i]), int(pos[i])
        if c < 0 or c >= len(lengths) or p < 0:
            continue                                         # not placed on a contig
        if mode == "all" and int(flag[i]) & SKIP_ALL:
            continue
        seq = np.asarray(seqs[i], dtype=np.uint8)
        if len(seq) == 0:
            continue                                         # no SEQ: nothing to count
        ops = [int(x) for x in cig[int(cig_off[i]):int(cig_off[i + 1])]]
        qlen = sum(o >> 4 for o in ops if o & 15 in CONSUMES_QUERY)
        if qlen > len(seq):
            raise IndexError("record %d: its CIGAR consumes %d query bases, SEQ holds %d" % (i, qlen, len(seq)))
        qual = quals[i]
        if t != 0 and qual is None:
            continue                                         # no qualities: nothing passes a threshold
        qual = None if qual is None else np.asarray(qual, dtype=np.int64)
        length = int(lengths[c])
        q, r = 0, p
        for o in ops:
            op, n = o & 15, o >> 4
            if op in ALIGNED:
                for j in range(n):
                    if r + j >= length:
                        break                                # past the contig's end
                    b = int(seq[q + j])
                    if b not in BASE_INDEX:
                        continue                             # '=', N and the IUPAC codes count nowhere
                    if t != 0 and not qual[q + j] >= t:
                        continue
                    out[c][BASE_INDEX[b], r + j] += 1
            if op in CONSUMES_QUERY:
                q += n
            if op in CONSUMES_REF:
                r += n
    return out


def interval(lengths, tid, start=None, stop=None):
    """pysam's interval rules: (start, stop) of contig ``tid`` or ValueError."""
    length = int(lengths[tid])
    start = 0 if start is None else int(start)
    stop = length if stop is None else min(int(stop), length)
    if start < 0:
        raise ValueError("start out of range (%d)" % start)
    if stop == start:
        raise ValueError("interval of size 0")
    if stop < start:
        raise ValueError("interval of size less than 0")
    return start, stop


def count_coverage(references, lengths, tid, pos, flag, cig_off, cig, seqs, quals, contig, start=None, stop=None,
                   quality_threshold=15, read_callback="all"):
    """The four uint32 arrays (A, C, G, T) of ``contig`` over [start, stop), index k = position start + k."""
    c = list(references).index(contig) if contig in references else None
    if c is None:
        raise KeyError(contig)
    start, stop = interval(lengths, c, start, stop)
    full = full_counts(lengths, tid, pos, flag, cig_off, cig, seqs, quals, quality_threshold, read_callback)[c]
    return tuple(full[k, start:stop].copy() for k in range(4))
