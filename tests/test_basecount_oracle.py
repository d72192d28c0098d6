"""The count_coverage restatement (oracle/basecount.py) against counts worked out by hand, one rule at a time: the op
kinds, qualities and their absence, the bases that count, the read filters, clipping at the interval and the contig
end, and the interval errors.  No GPU needed: these are the rules the device counts are checked against."""
import numpy as np
import pytest

from oracle import basecount
from oracle.bamio import CIGAR_OPS
import samio

REFS, LENS = ["c0", "c1"], [20, 10]


def _cigar(s):
    ops, num = [], ""
    for ch in s:
        if ch.isdigit():
            num += ch
        else:
            ops.append((int(num) << 4) | CIGAR_OPS.index(ch))
            num = ""
    return ops


def _records(recs):
    """(tid, pos, flag, CIGAR text, SEQ text or '*', QUAL text or '*') -> the oracle's columns (SEQ through the SAM
    decoder's nt16 table, QUAL minus 33)."""
    tid = np.array([r[0] for r in recs], np.int32)
    pos = np.array([r[1] for r in recs], np.int32)
    flag = np.array([r[2] for r in recs], np.uint16)
    ops = [_cigar(r[3]) if r[3] != "*" else [] for r in recs]
    cig_off = np.concatenate(([0], np.cumsum([len(o) for o in ops]))).astype(np.uint32)
    cig = np.array([x for o in ops for x in o], np.uint32)
    seqs = [np.array([samio._NT16_OF.get(c, 15) for c in r[4]] if r[4] != "*" else [], np.uint8) for r in recs]
    quals = [None if r[5] == "*" else [ord(c) - 33 for c in r[5]] for r in recs]
    return tid, pos, flag, cig_off, cig, seqs, quals


def _cc(recs, contig="c0", start=None, stop=None, t=15, cb="all"):
    return basecount.count_coverage(REFS, LENS, *_records(recs), contig, start, stop, quality_threshold=t, read_callback=cb)


def _at(counts, k):
    """{position: base} of the non-zero counts of one base row."""
    return {int(p): int(counts[k][p]) for p in np.nonzero(counts[k])[0]}


def test_every_op_kind():
    # q: GG|ACG|T|..|.|T|C|.|A ; ref: 2 3 4 (M), 5 6 (D), 7 (N), 8 (=), 9 (X); S, I, P and H make no pair
    r = (0, 2, 0, "2S3M1I2D1N1=1X1P1S1H", "GGACGTTCA", "*")
    a, c, g, t = _cc([r], t=0)
    assert _at((a, c, g, t), 0) == {2: 1}
    assert _at((a, c, g, t), 1) == {3: 1, 9: 1}
    assert _at((a, c, g, t), 2) == {4: 1}
    assert _at((a, c, g, t), 3) == {8: 1}
    assert all(len(x) == 20 and x.dtype == np.uint32 for x in (a, c, g, t))


def test_qualities():
    r_none = (0, 0, 0, "4M", "ACGT", "*")
    assert sum(int(x.sum()) for x in _cc([r_none], t=0)) == 4
    assert sum(int(x.sum()) for x in _cc([r_none], t=None)) == 4
    assert sum(int(x.sum()) for x in _cc([r_none], t=15)) == 0
    assert sum(int(x.sum()) for x in _cc([r_none], t=-1)) == 0          # (a negative threshold still needs qualities)
    r_q = (0, 0, 0, "4M", "ACGT", chr(33 + 10) + chr(33 + 15) + chr(33 + 30) + chr(33 + 14))
    a, c, g, t = _cc([r_q], t=15)
    assert (int(a[0]), int(c[1]), int(g[2]), int(t[3])) == (0, 1, 1, 0)
    assert sum(int(x.sum()) for x in _cc([r_q], t=-1)) == 4
    assert sum(int(x.sum()) for x in _cc([r_q], t=31)) == 0
    # one base and QUAL '*': no qualities, even though '*' would read as quality 9
    r1 = (0, 5, 0, "1M", "G", "*")
    assert int(_cc([r1], t=0)[2][5]) == 1 and int(_cc([r1], t=5)[2][5]) == 0


def test_bases():
    r = (0, 0, 0, "12M", "A=NRacgtMnYT", "*")
    a, c, g, t = _cc([r], t=0)
    assert _at((a, c, g, t), 0) == {0: 1, 4: 1}
    assert _at((a, c, g, t), 1) == {5: 1}
    assert _at((a, c, g, t), 2) == {6: 1}
    assert _at((a, c, g, t), 3) == {7: 1, 11: 1}
    # SEQ '*' counts nothing, and its CIGAR is not held against it
    assert sum(int(x.sum()) for x in _cc([(0, 0, 0, "5M", "*", "*")], t=0)) == 0


@pytest.mark.parametrize("f", [0x4, 0x100, 0x200, 0x400])
def test_filtered_flags(f):
    r = (0, 3, f, "2M", "AC", "*")
    assert sum(int(x.sum()) for x in _cc([r], t=0, cb="all")) == 0
    assert sum(int(x.sum()) for x in _cc([r], t=0, cb="nofilter")) == 2


@pytest.mark.parametrize("f", [0x1, 0x2, 0x10, 0x40, 0x800, 0x1 | 0x8])
def test_counted_flags(f):
    r = (0, 3, f, "2M", "AC", "*")
    assert sum(int(x.sum()) for x in _cc([r], t=0, cb="all")) == 2


def test_unplaced_records_never_count():
    recs = [(-1, 3, 0, "2M", "AC", "*"), (0, -1, 0, "2M", "AC", "*")]
    assert sum(int(x.sum()) for x in _cc(recs, t=0, cb="nofilter")) == 0


def test_clipping():
    r = (1, 7, 0, "5M", "ACGTA", "*")                                   # c1 is 10 long: positions 7 8 9 only
    a, c, g, t = _cc([r], contig="c1", t=0)
    assert (int(a[7]), int(c[8]), int(g[9]), int(t.sum())) == (1, 1, 1, 0)
    a, c, g, t = _cc([r], contig="c1", start=8, stop=9, t=0)
    assert len(a) == 1 and int(c[0]) == 1 and int(a.sum() + g.sum()) == 0
    a, c, g, t = _cc([r], contig="c1", start=8, stop=1000, t=0)          # stop clipped to the contig
    assert len(a) == 2 and int(c[0]) == 1 and int(g[1]) == 1


def test_interval_errors():
    r = [(0, 0, 0, "2M", "AC", "*")]
    with pytest.raises(ValueError, match="interval of size 0"):
        _cc(r, start=5, stop=5)
    with pytest.raises(ValueError, match="interval of size 0"):
        _cc(r, start=20)                                                # stop -> the contig length 20
    with pytest.raises(ValueError):
        _cc(r, start=6, stop=5)
    with pytest.raises(ValueError):
        _cc(r, start=-1, stop=5)
    with pytest.raises(KeyError):
        _cc(r, contig="nope")
    with pytest.raises(ValueError):
        _cc(r, cb="mapped")
    with pytest.raises(ValueError):
        _cc(r, cb=lambda read: True)


def test_cigar_longer_than_seq():
    good = (0, 0, 0, "2M", "AC", "*")
    bad = (0, 4, 0, "3M1I", "ACG", "*")
    with pytest.raises(IndexError, match="record 1"):
        _cc([good, bad], t=0)
    # a record that is not counted is not checked
    assert sum(int(x.sum()) for x in _cc([good, (0, 4, 0x400, "3M1I", "ACG", "*")], t=0)) == 2
