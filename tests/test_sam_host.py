"""SAM text rules of the GPU decoder (csrc/k_sam.cuh), CPU only, through the host-compiled test hook
mcov_sam_parse_host: against the Python restatement (tests/samio.py) on random lines with every edge the
rules name, one malformed file per rule, against the BAM host reader on the same records, and the format sniffing of
AlignmentFile."""
import ctypes as C

import numpy as np
import pytest

from helpers import load_soa
from oracle import bamio
import samio

COLS = ("tid", "pos", "flag", "mapq", "l_seq", "isize", "cig_off", "cig")


def host_parse(data, k_len=0, win_bases=0):
    """mcov_sam_parse_host over a file image -> (dict of the columns and name_hash / kmer_code / seq_win, the
    mcov_sam_host_cols, the error text); the dict is None when the hook refuses the file."""
    from metacov_b200 import _capi
    lib = _capi.lib
    buf = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(1, np.uint8)
    err = C.create_string_buffer(256)
    c = _capi.SamHostCols()
    rc = lib.mcov_sam_parse_host(buf.ctypes.data, len(data), C.byref(c), err, len(err))
    if rc != 0:
        return None, c, err.value.decode()
    n, m = c.n_records, c.n_cigar
    out = dict(tid=np.empty(n, np.int32), pos=np.empty(n, np.int32), flag=np.empty(n, np.uint16), mapq=np.empty(n, np.uint8),
               l_seq=np.empty(n, np.int32), isize=np.empty(n, np.int32), cig_off=np.empty(n + 1, np.uint32),
               cig=np.empty(max(m, 1), np.uint32), name_hash=np.empty(n, np.uint64), kmer_code=np.empty(n, np.int32),
               seq_win=np.empty((n, (win_bases + 1) // 2), np.uint8))
    for k, a in out.items():
        setattr(c, k, a.ctypes.data)
    c.k_len, c.win_bases = k_len, win_bases
    if not k_len:
        c.kmer_code = None
    if not win_bases:
        c.seq_win = None
    rc = lib.mcov_sam_parse_host(buf.ctypes.data, len(data), C.byref(c), err, len(err))
    assert rc == 0, err.value
    out["cig"] = out["cig"][:m]
    return out, c, ""


def fnv1a(b):
    h = 1469598103934665603
    for x in b:
        h = ((h ^ x) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h - 1 if h == 0xFFFFFFFFFFFFFFFF else h


def random_records(rng, n, n_ref=3):
    """Random records with the edges of the rules: '*' RNAME / CIGAR / SEQ / QUAL, lowercase and ambiguous bases,
    1- and 254-byte names, all ops, op lengths up to 2^28-1, extreme POS / TLEN / FLAG / MAPQ, optional fields with B:
    arrays.  Returns the keyword arguments of write_sam."""
    lengths = [int(x) for x in rng.integers(1000, 2 ** 31 - 1, n_ref)]
    refs = ["chr%d|x" % i for i in range(n_ref)]
    tid = rng.integers(-1, n_ref, n).astype(np.int32)
    pos = rng.integers(-1, 2 ** 31 - 1, n).astype(np.int32)
    pos[rng.random(n) < 0.1] = 2 ** 31 - 2
    flag = rng.integers(0, 65536, n).astype(np.uint16)
    mapq = rng.integers(0, 256, n).astype(np.uint8)
    isize = rng.integers(-2 ** 31, 2 ** 31, n, dtype=np.int64).astype(np.int32)
    cig, off, seqs, names, quals, aux = [], [0], [], [], [], []
    for i in range(n):
        k = int(rng.integers(0, 7))
        ops = [(int(rng.integers(0, 9)), int(rng.choice([0, 1, 9, 10, 99, 150, 12345, 2 ** 28 - 1]) if rng.random() < 0.2
                                                 else rng.integers(1, 200))) for _ in range(k)]
        cig += [(l << 4) | o for o, l in ops]
        off.append(len(cig))
        ls = int(rng.integers(0, 300)) if rng.random() < 0.9 else 0
        s = "".join(rng.choice(list("ACGTNacgtn=MRWSYKVHDBmrwsykvhdbXU."), ls).tolist())
        seqs.append(s)
        quals.append("*" if ls == 0 or rng.random() < 0.3 else "".join(chr(33 + int(q)) for q in rng.integers(0, 60, ls)))
        nl = int(rng.choice([1, 254, int(rng.integers(1, 60))]))
        names.append("".join(rng.choice(list("ABCxyz019:_/#!?~"), nl).tolist()))
        r = rng.random()
        aux.append("" if r < 0.3 else "NM:i:%d\tMD:Z:%dA0\tXB:B:i,1,-2,3\tZZ:B:f,1.5,2" % (i, i) if r < 0.7 else "RG:Z:g\t\tXA:A:q")
    mtid = rng.integers(-1, n_ref, n).astype(np.int32)
    mpos = rng.integers(-1, 2 ** 31 - 1, n).astype(np.int32)
    return dict(references=refs, lengths=lengths, tid=tid, pos=pos, flag=flag, mapq=mapq, cig_off=np.array(off, np.uint64),
                cig=np.array(cig, np.uint32), isize=isize, names=names, seqs=seqs, quals=quals, aux=aux, mtid=mtid, mpos=mpos)


def _check_against_oracle(data):
    got, c, err = host_parse(data)
    assert got is not None, err
    refs, lens, want, names, _seqs = samio.parse_sam(data)
    assert c.n_ref == len(refs) and c.n_records == len(names)
    for k in COLS:
        assert np.array_equal(got[k], want[k]), k
    assert got["name_hash"].tolist() == [fnv1a(x) for x in names]
    return got


@pytest.mark.parametrize("variant", ["plain", "crlf", "no_final_newline", "crlf_no_final_newline", "no_header"])
def test_host_hook_matches_restatement(tmp_path, variant):
    rng = np.random.default_rng(len(variant))
    kw = random_records(rng, 1500)
    if variant == "no_header":
        kw["text"] = ""
        kw["tid"][:] = -1
        kw["mtid"][:] = -1
    p = str(tmp_path / "r.sam")
    samio.write_sam(p, crlf="crlf" in variant, final_newline="no_final" not in variant, **kw)
    data = open(p, "rb").read()
    got = _check_against_oracle(data)
    assert len(got["tid"]) == 1500
    assert got["cig"].size and int((got["cig"] >> 4).max()) == 2 ** 28 - 1


def test_host_hook_long_cigar(tmp_path):
    """A record of 70 000 ops (more than BAM's 16-bit n_cigar_op field could hold without the CG tag) among short ones."""
    rng = np.random.default_rng(3)
    n = 5
    ops = [[(0, 10)], [(0, 3), (1, 1)] * 35000, [], [(4, 5), (0, 20)], [(0, 1)]]
    cig = [(l << 4) | o for r in ops for o, l in r]
    off = np.cumsum([0] + [len(r) for r in ops])
    p = str(tmp_path / "long.sam")
    samio.write_sam(p, ["c0"], [10 ** 6], np.zeros(n, np.int32), np.arange(n, dtype=np.int32) * 100, np.zeros(n, np.uint16),
                    rng.integers(0, 60, n).astype(np.uint8), off, np.array(cig, np.uint32))
    got = _check_against_oracle(open(p, "rb").read())
    assert np.diff(got["cig_off"]).tolist() == [1, 70000, 0, 2, 1]


GOOD = "r1\t0\tc0\t5\t30\t3M\t*\t0\t0\tACG\tIII"
BAD_LINES = [                       # (line text, field) -- each breaks one rule
    ("", 11), ("r1\t0\tc0\t5\t30\t3M\t*\t0\t0\tACG", 11), ("@CO\tlate header", 12),
    ("\t0\tc0\t5\t30\t3M\t*\t0\t0\tACG\tIII", 0), ("x" * 255 + "\t0\tc0\t5\t30\t3M\t*\t0\t0\tACG\tIII", 0),
    ("r1\t65536\tc0\t5\t30\t3M\t*\t0\t0\tACG\tIII", 1), ("r1\t-1\tc0\t5\t30\t3M\t*\t0\t0\tACG\tIII", 1),
    ("r1\t\tc0\t5\t30\t3M\t*\t0\t0\tACG\tIII", 1),
    ("r1\t0\tc9\t5\t30\t3M\t*\t0\t0\tACG\tIII", 2), ("r1\t0\tc\t5\t30\t3M\t*\t0\t0\tACG\tIII", 2),
    ("r1\t0\t\t5\t30\t3M\t*\t0\t0\tACG\tIII", 2),
    ("r1\t0\tc0\t2147483648\t30\t3M\t*\t0\t0\tACG\tIII", 3), ("r1\t0\tc0\t-5\t30\t3M\t*\t0\t0\tACG\tIII", 3),
    ("r1\t0\tc0\t5\t256\t3M\t*\t0\t0\tACG\tIII", 4), ("r1\t0\tc0\t5\t3x\t3M\t*\t0\t0\tACG\tIII", 4),
    ("r1\t0\tc0\t5\t30\t3Q\t*\t0\t0\tACG\tIII", 5), ("r1\t0\tc0\t5\t30\tM\t*\t0\t0\tACG\tIII", 5),
    ("r1\t0\tc0\t5\t30\t3M3\t*\t0\t0\tACG\tIII", 5), ("r1\t0\tc0\t5\t30\t268435456M\t*\t0\t0\tACG\tIII", 5),
    ("r1\t0\tc0\t5\t30\t\t*\t0\t0\tACG\tIII", 5), ("r1\t0\tc0\t5\t30\t3MM\t*\t0\t0\tACG\tIII", 5),
    ("r1\t0\tc0\t5\t30\t3M\t\t0\t0\tACG\tIII", 6), ("r1\t0\tc0\t5\t30\t3M\t*\t-1\t0\tACG\tIII", 7),
    ("r1\t0\tc0\t5\t30\t3M\t*\t0\t2147483648\tACG\tIII", 8), ("r1\t0\tc0\t5\t30\t3M\t*\t0\t-2147483649\tACG\tIII", 8),
    ("r1\t0\tc0\t5\t30\t3M\t*\t0\t0\t\tIII", 9), ("r1\t0\tc0\t5\t30\t3M\t*\t0\t0\tACG\tII", 10),
    ("r1\t0\tc0\t5\t30\t3M\t*\t0\t0\t*\tI", 10), ("r1\t0\tc0\t5\t30\t3M\t*\t0\t0\tACG\t", 10),
]
HEADER = "@HD\tVN:1.6\n@SQ\tSN:c0\tLN:1000\n@SQ\tSN:c1\tLN:2000\n"


def bad_file(line, field):
    """HEADER, three good lines, the bad line (line 7), a good line."""
    return (HEADER + (GOOD + "\n") * 3 + line + "\n" + GOOD + "\n").encode()


@pytest.mark.parametrize("line,field", BAD_LINES)
def test_malformed_line_names_line_and_field(line, field):
    data = bad_file(line, field)
    got, c, err = host_parse(data)
    assert got is None and c.fail_line == 7 and c.fail_field == field, (err, c.fail_line, c.fail_field)
    assert "line 7" in err
    with pytest.raises(samio.SamError) as e:
        samio.parse_sam(data)
    assert (e.value.line, e.value.field) == (7, field)


@pytest.mark.parametrize("header", ["@SQ\tSN:c0\n", "@SQ\tLN:5\n", "@SQ\tSN:c0\tLN:0\n", "@SQ\tSN:c0\tLN:2147483648\n",
                                    "@SQ\tSN:c0\tLN:5\n@SQ\tSN:c0\tLN:6\n"])
def test_malformed_header(header):
    data = (header + GOOD.replace("c0", "*") + "\n").encode()
    got, c, err = host_parse(data)
    assert got is None and "SQ" in err
    with pytest.raises(samio.SamError):
        samio.parse_sam(data)


def test_edge_values_decode():
    lines = ["q\t65535\t*\t0\t255\t*\t=\t2147483647\t-2147483648\t*\t*\tXX:B:c,1,2",
             "q\t0\tc1\t2147483647\t0\t0M1I268435455N\t*\t0\t2147483647\tA\t*",
             "q\t1\tc0\t1\t0\t00000000001M\t*\t0\t+0\tA\t*"]
    got, c, err = host_parse((HEADER + "\n".join(lines[:2]) + "\n").encode())
    assert got is not None, err
    assert got["tid"].tolist() == [-1, 1] and got["pos"].tolist() == [-1, 2 ** 31 - 2]
    assert got["flag"].tolist() == [65535, 0] and got["mapq"].tolist() == [255, 0]
    assert got["isize"].tolist() == [-2 ** 31, 2 ** 31 - 1] and got["l_seq"].tolist() == [0, 1]
    assert got["cig"].tolist() == [0, (1 << 4) | 1, ((2 ** 28 - 1) << 4) | 3]
    got, c, err = host_parse((HEADER + lines[2] + "\n").encode())
    assert got is None and c.fail_field == 8          # TLEN is [-]digits: no '+'
    got, c, err = host_parse((HEADER + lines[2].replace("+0", "0") + "\n").encode())
    assert got["cig"].tolist() == [1 << 4]            # leading zeros of an op length are fine


def _bam_and_sam(tmp_path, name, refs, lengths, b, **kw):
    pb, ps = str(tmp_path / (name + ".bam")), str(tmp_path / (name + ".sam"))
    bamio.write_bam(pb, refs, lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, **kw)
    samio.write_sam(ps, refs, lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, **kw)
    return pb, ps


def _compare_with_bam_reader(pb, ps):
    from metacov_b200 import AlignmentFile
    data = open(ps, "rb").read()
    with AlignmentFile(pb) as bam:
        s = bam.soa()
        for k in (1, 3, 7, 15):
            got = host_parse(data, k_len=k)[0]
            assert np.array_equal(got["kmer_code"], bam.qas_kmer_codes(k)), k
        for w in (1, 2, 56, 57, 300):
            got = host_parse(data, win_bases=w)[0]
            assert np.array_equal(got["seq_win"], bam.seq_windows(w)), w
        for c in COLS:
            assert np.array_equal(got[c], s[c]), c
        assert np.array_equal(got["name_hash"], bam.name_hashes())


def test_fixture_sam_equals_bam_reader(tmp_path):
    z, b = load_soa("fixture_soa.npz")
    so = z["seq_off"]
    seqs = [z["seq"][so[i]:so[i + 1]] for i in range(len(b.tid))]
    pb, ps = _bam_and_sam(tmp_path, "fixture", [str(x) for x in z["references"]], [int(x) for x in z["lengths"]], b,
                          isize=z["isize"], names=[str(x) for x in z["names"]], seqs=seqs)
    _compare_with_bam_reader(pb, ps)
    # the mate columns go to RNEXT / PNEXT (not stored): the same records
    ps2 = str(tmp_path / "fixture_mates.sam")
    samio.write_sam(ps2, [str(x) for x in z["references"]], [int(x) for x in z["lengths"]], b.tid, b.pos, b.flag, b.mapq,
                    b.cig_off, b.cig, isize=z["isize"], names=[str(x) for x in z["names"]], seqs=seqs,
                    mtid=z["mtid"], mpos=z["mpos"])
    _compare_with_bam_reader(pb, ps2)


def test_random_set_sam_equals_bam_reader(tmp_path):
    from metacov_b200 import ReadBatch
    rng = np.random.default_rng(77)
    n = 3000
    tid = np.sort(rng.integers(-1, 2, n)).astype(np.int32)
    pos = np.where(tid >= 0, rng.integers(0, 39000, n), -1).astype(np.int32)
    flag = (rng.integers(0, 2, n) * 0x10 + rng.choice([0x40, 0x80, 0x4], n)).astype(np.uint16)
    cig, off, seqs, names = [], [0], [], []
    for i in range(n):
        ops = []
        if rng.random() < 0.2: ops.append((5, int(rng.integers(1, 9))))
        if rng.random() < 0.4: ops.append((4, int(rng.integers(1, 30))))
        ops.append((0, int(rng.integers(1, 120))))
        if rng.random() < 0.3: ops += [(1, int(rng.integers(1, 5))), (0, int(rng.integers(1, 60)))]
        if rng.random() < 0.4: ops.append((4, int(rng.integers(1, 30))))
        qlen = 0 if i % 97 == 0 else sum(l for o, l in ops if o in (0, 1, 4))
        cig += [(l << 4) | o for o, l in ops]
        off.append(len(cig))
        seqs.append(rng.choice(np.array([1, 2, 4, 8, 15, 1, 2, 4, 8, 3, 0, 13], np.uint8), qlen))
        names.append("r%d/%s" % (i // 2, "x" * int(rng.integers(0, 40))))
    b = ReadBatch(tid, pos, flag, rng.integers(0, 61, n).astype(np.uint8), np.array(off, np.uint32), np.array(cig, np.uint32))
    pb, ps = _bam_and_sam(tmp_path, "rand", ["c0", "c1"], [40000, 30000], b, isize=rng.integers(-600, 600, n).astype(np.int32),
                          names=names, seqs=seqs)
    _compare_with_bam_reader(pb, ps)
    # lowercase letters are the same bases
    pl = str(tmp_path / "lower.sam")
    samio.write_sam(pl, ["c0", "c1"], [40000, 30000], b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig,
                    isize=rng.integers(-600, 600, n).astype(np.int32), names=names,
                    seqs=["".join(bamio.NT16[c] for c in s).lower() for s in seqs])
    a, _, _ = host_parse(open(ps, "rb").read(), k_len=7, win_bases=57)
    l, _, _ = host_parse(open(pl, "rb").read(), k_len=7, win_bases=57)
    assert np.array_equal(a["kmer_code"], l["kmer_code"]) and np.array_equal(a["seq_win"], l["seq_win"])


def test_format_sniffing(tmp_path):
    from metacov_b200.alignmentfile import is_sam_text
    z, b = load_soa("fixture_soa.npz")
    pb, ps = _bam_and_sam(tmp_path, "f", [str(x) for x in z["references"]], [int(x) for x in z["lengths"]], b)
    assert is_sam_text(ps) and not is_sam_text(pb) and not is_sam_text(pb + ".bai")
    headerless = tmp_path / "nohdr.sam"
    headerless.write_text("\n".join(open(ps).read().splitlines()[3:]) + "\n")
    assert is_sam_text(str(headerless))
    long_first = tmp_path / "long.sam"                   # a first record far longer than the first read
    long_first.write_text("r\t0\t*\t0\t0\t*\t*\t0\t0\t" + "A" * 300000 + "\t*\n")
    assert is_sam_text(str(long_first))
    (tmp_path / "empty").write_bytes(b"")
    (tmp_path / "garbage").write_bytes(b"not a bam file at all" * 10)
    (tmp_path / "fewtabs").write_text("a\tb\tc\n" + "x\t" * 20 + "\n")
    (tmp_path / "at").write_text("@not a header\n")
    for name in ("empty", "garbage", "fewtabs", "at", "missing"):
        assert not is_sam_text(str(tmp_path / name)), name
