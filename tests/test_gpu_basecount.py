"""AlignmentFile.count_coverage on the GPU (csrc/basecount.cu) against the restatement of pysam's rules
(oracle/basecount.py): seeded read sets with every op kind, long reads, reads past the contig end, SEQ / QUAL '*' and a
pile of 20 000 reads on one position; BAM against SAM, sorted against shuffled (and the kernel that ran), the three decode
modes, the depth as an independent cross-check, the depth left untouched, and the errors."""
import gzip
import io
import os
import struct
import zlib

import numpy as np
import pytest

from oracle import bamio, basecount
import samio

pytestmark = pytest.mark.gpu

REFS = ["c0", "c1", "c2"]
LENS = [3000, 500, 60000]
LETTERS = "ACGTACGTACGTacgtN=RYMKW"


def _gen(seed, n=3000, acgt_only=False, unpaired=False, pile=20000, long_reads=4):
    """Records (tid, pos, flag, ops, SEQ letters, Phred list or None), coordinate-sorted."""
    rng = np.random.default_rng(seed)
    recs = []
    flags = [0, 16, 0x4, 0x100, 0x400] if unpaired else [0, 16, 0x4, 0x100, 0x200, 0x400, 0x800, 1 | 2 | 0x40, 1 | 0x80 | 0x10, 1 | 8 | 0x40]
    letters = "ACGT" if acgt_only else LETTERS

    def seq_qual(qlen, no_seq_p=0.03, no_qual_p=0.2):
        if qlen == 0 or (not acgt_only and rng.random() < no_seq_p):
            return "", None
        s = "".join(letters[k] for k in rng.integers(0, len(letters), qlen))
        if rng.random() < no_qual_p:
            return s, None
        q = [int(x) for x in rng.integers(0, 46, qlen)]
        if qlen == 1 and q[0] == 9:
            q[0] = 10                                      # (SAM reads a lone '*' as "no qualities")
        return s, q

    for _ in range(n):
        if rng.random() < 0.04:
            tid, pos = -1, -1
        else:
            tid = int(rng.integers(0, len(LENS)))
            pos = int(rng.integers(max(LENS[tid] - 60, 0), LENS[tid])) if rng.random() < 0.1 else int(rng.integers(0, LENS[tid]))
        ops = []
        for _k in range(int(rng.integers(1, 8))):
            op = "MMMMIDNSHP=X"[int(rng.integers(0, 12))]
            ops.append((int(rng.integers(1, 31)) << 4) | bamio.CIGAR_OPS.index(op))
        qlen = sum(o >> 4 for o in ops if (o & 15) in basecount.CONSUMES_QUERY)
        s, q = seq_qual(qlen)
        recs.append((tid, pos, int(rng.choice(flags)), ops, s, q))
    for k in range(long_reads):                            # > 127 ops, ~50 kb
        ops = []
        for _j in range(40):
            ops += [(1200 << 4) | 0, (1 << 4) | 1, (2 << 4) | 2, (10 << 4) | 8]
        qlen = sum(o >> 4 for o in ops if (o & 15) in basecount.CONSUMES_QUERY)
        s, q = seq_qual(qlen, 0, 0.25 * (k == 3))
        recs.append((2, int(rng.integers(0, 12000)), 0, ops, s, q))
    for _ in range(pile):                                  # contention: 20 000 reads on the same ten positions
        s, q = seq_qual(10, 0.0, 0.1)
        recs.append((1, 100, int(rng.choice([0, 16])), [(10 << 4) | 0], s, q))
    recs.sort(key=lambda r: (r[0] & 0xFFFFFFFF, r[1]))
    return recs


def _columns(recs):
    tid = np.array([r[0] for r in recs], np.int32)
    pos = np.array([r[1] for r in recs], np.int32)
    flag = np.array([r[2] for r in recs], np.uint16)
    mapq = np.full(len(recs), 30, np.uint8)
    cig_off = np.concatenate(([0], np.cumsum([len(r[3]) for r in recs]))).astype(np.uint32)
    cig = np.array([o for r in recs for o in r[3]], np.uint32)
    nt16 = [np.array([samio._NT16_OF[c] for c in r[4]], np.uint8) for r in recs]
    quals = [r[5] for r in recs]
    return tid, pos, flag, mapq, cig_off, cig, nt16, quals


def _set_bam_quals(path, quals):
    """Put per-record Phred qualities (None = none, 0xff) into a BAM that ``bamio.write_bam`` wrote (it writes none):
    inflate, walk the records (SAM spec 4.2), overwrite each QUAL, compress again."""
    data = bytearray(gzip.decompress(open(path, "rb").read()))
    l_text = struct.unpack_from("<i", data, 4)[0]
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", data, p)[0]
    p += 4
    for _ in range(n_ref):
        p += 8 + struct.unpack_from("<i", data, p)[0]
    for q in quals:
        bs = struct.unpack_from("<i", data, p)[0]
        l_name, n_op, l_seq = data[p + 12], struct.unpack_from("<H", data, p + 16)[0], struct.unpack_from("<i", data, p + 20)[0]
        if q is not None:
            assert len(q) == l_seq
            o = p + 36 + l_name + 4 * n_op + (l_seq + 1) // 2
            data[o:o + l_seq] = bytes(q)
        p += 4 + bs
    assert p == len(data)
    with open(path, "wb") as fh:
        fh.write(bamio.bgzf_compress(bytes(data)))


def _write(recs, d, name):
    tid, pos, flag, mapq, cig_off, cig, nt16, quals = _columns(recs)
    pb, ps = str(d / (name + ".bam")), str(d / (name + ".sam"))
    bamio.write_bam(pb, REFS, LENS, tid, pos, flag, mapq, cig_off, cig, seqs=nt16, with_index=False)
    _set_bam_quals(pb, quals)
    samio.write_sam(ps, REFS, LENS, tid, pos, flag, mapq, cig_off, cig, seqs=[r[4] for r in recs],
                    quals=["*" if r[5] is None else "".join(chr(33 + x) for x in r[5]) for r in recs])
    return pb, ps


_ORACLE = {}


def _oracle(key, recs, t, cb):
    k = (key, int(t or 0), cb)
    if k not in _ORACLE:
        tid, pos, flag, _mapq, cig_off, cig, nt16, quals = _columns(recs)
        _ORACLE[k] = basecount.full_counts(LENS, tid, pos, flag, cig_off, cig, nt16, quals, t, cb)
    return _ORACLE[k]


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("basecount")
    recs = _gen(7)
    rng = np.random.default_rng(8)
    shuf = [recs[i] for i in rng.permutation(len(recs))]
    pb, ps = _write(recs, d, "sorted")
    ub, us = _write(shuf, d, "shuffled")
    return dict(recs=recs, bam=pb, sam=ps, bam_shuf=ub, sam_shuf=us, dir=d)


def _all_counts(af, t, cb):
    return [np.stack(af.count_coverage(c, quality_threshold=t, read_callback=cb)) for c in REFS]


def _kernels(af, fn):
    eng = af._count_engine()
    eng.profile(True)
    fn()
    got = set(eng.profile_read())
    eng.profile(False)
    return got


@pytest.mark.parametrize("fmt", ["bam", "sam"])
@pytest.mark.parametrize("cb", ["all", "nofilter"])
@pytest.mark.parametrize("t", [0, 15, 30, None])
def test_matches_oracle(files, fmt, cb, t):
    from metacov_b200 import AlignmentFile
    ref = _oracle("sorted", files["recs"], t, cb)
    rng = np.random.default_rng(zlib.crc32(repr((fmt, cb, t)).encode()))
    with AlignmentFile(files[fmt], decode="gpu") as af:
        got = _all_counts(af, t, cb)
        for c in range(len(REFS)):
            assert np.array_equal(got[c], ref[c]), (REFS[c], fmt, t, cb)
            for _ in range(6):
                a = int(rng.integers(0, LENS[c]))
                b = int(rng.integers(a + 1, LENS[c] + 50))
                cc = af.count_coverage(REFS[c], a, b, quality_threshold=t, read_callback=cb)
                e = min(b, LENS[c])
                assert all(x.dtype == np.uint32 and len(x) == e - a for x in cc)
                assert np.array_equal(np.stack(cc), ref[c][:, a:e])
    assert int(sum(r.sum() for r in ref)) > 50000


def test_bam_equals_sam_and_sorted_equals_shuffled(files):
    from metacov_b200 import AlignmentFile
    for t, cb in ((15, "all"), (0, "nofilter")):
        out = {}
        for k in ("bam", "sam", "bam_shuf", "sam_shuf"):
            with AlignmentFile(files[k], decode="gpu") as af:
                ran = _kernels(af, lambda: af.count_coverage("c0", quality_threshold=t, read_callback=cb))
                # one kernel for every read order, and nothing of the depth path runs
                assert ran == {"k_bc_any"}, (k, ran)
                out[k] = _all_counts(af, t, cb)
        for k in ("sam", "bam_shuf", "sam_shuf"):
            for c in range(len(REFS)):
                assert np.array_equal(out[k][c], out["bam"][c]), (k, c)


@pytest.mark.parametrize("name", ["bam", "bam_shuf"])
def test_decode_modes(files, name):
    from metacov_b200 import AlignmentFile
    res = []
    for decode, kw in (("gpu", {}), ("host", {}), ("gpu-stream", {"gpu_chunk_bytes": 1 << 17})):
        with AlignmentFile(files[name], decode=decode, **kw) as af:
            assert af.decode == decode
            res.append([_all_counts(af, t, cb) for t, cb in ((15, "all"), (0, "nofilter"))])
    ref = [_oracle("sorted", files["recs"], t, cb) for t, cb in ((15, "all"), (0, "nofilter"))]
    assert os.path.getsize(files[name]) > 4 * (1 << 17)          # (the chunks cut records)
    for r in res:
        for j in range(2):
            for c in range(len(REFS)):
                assert np.array_equal(r[j][c], ref[j][c]), (name, j, c)


def test_equals_depth_for_acgt_unpaired_reads(tmp_path):
    from metacov_b200 import AlignmentFile
    recs = _gen(11, n=2000, acgt_only=True, unpaired=True, pile=3000)
    pb, ps = _write(recs, tmp_path, "acgt")
    for p in (pb, ps):
        with AlignmentFile(p, decode="gpu") as af:
            af.set_pileup_filter(count_del=False, max_depth=0)
            for c in REFS:
                s = np.stack(af.count_coverage(c, quality_threshold=0)).sum(axis=0)
                d = af.count_coverage_depth(c)
                assert s.sum() > 0 and np.array_equal(s.astype(np.int64), d.astype(np.int64)), (p, c)


def test_depth_and_statistics_unchanged(files):
    from metacov_b200 import AlignmentFile
    for decode in ("gpu", "host"):
        with AlignmentFile(files["bam"], decode=decode) as af:
            eng = af.coverage_engine()
            tid = np.arange(len(REFS), dtype=np.int32)

            def snap():
                return ([af.count_coverage_depth(c) for c in REFS],
                        eng.region_stats(tid, np.zeros_like(tid), np.array(LENS, np.int32)))
            d0, s0 = snap()
            af.count_coverage("c2", quality_threshold=30)
            af.count_coverage("c1", read_callback="nofilter")
            d1, s1 = snap()
            for a, b in zip(d0, d1):
                assert np.array_equal(a, b)
            for k in s0.dtype.names:
                assert np.array_equal(s0[k], s1[k]), k


def test_errors_leave_the_file_usable(files, tmp_path, monkeypatch):
    from metacov_b200 import AlignmentFile
    good = files["recs"][:50]
    ref = _oracle("sorted", files["recs"], 15, "all")
    with AlignmentFile(io.BytesIO(open(files["sam"], "rb").read())) as s:
        with pytest.raises(ValueError, match="read once"):
            s.count_coverage("c0")
    with AlignmentFile(files["bam"], decode="gpu") as af:
        for bad in (lambda r: True, "mapped", None):
            with pytest.raises(ValueError):
                af.count_coverage("c0", read_callback=bad)
        with pytest.raises(ValueError, match="interval of size 0"):
            af.count_coverage("c0", 10, 10)
        with pytest.raises(ValueError, match="interval of size 0"):
            af.count_coverage("c0", 3000)
        with pytest.raises(ValueError):
            af.count_coverage("c0", 10, 5)
        with pytest.raises(ValueError):
            af.count_coverage("c0", -1, 5)
        with pytest.raises(KeyError):
            af.count_coverage("nope")
        monkeypatch.setenv("MCOV_BC_FREE_BYTES", "1000")
        with pytest.raises(MemoryError, match=r"need \d+ bytes of device memory, \d+ are free"):
            af.count_coverage("c0")
        monkeypatch.delenv("MCOV_BC_FREE_BYTES")
        assert np.array_equal(np.stack(af.count_coverage("c2")), ref[2])
    # a CIGAR that consumes more query bases than SEQ holds: the first such record is named, in every decode mode
    recs = list(good)
    recs[20] = (0, 5, 0, [(4 << 4) | 0, (3 << 4) | 4], "ACGTAC", None)
    recs[30] = (0, 9, 0, [(9 << 4) | 0], "ACGT", None)
    recs[40] = (0, 9, 0x400, [(9 << 4) | 0], "ACGT", None)             # (filtered: not counted, not checked)
    recs.sort(key=lambda r: (r[0] & 0xFFFFFFFF, r[1]))
    first = min(i for i, r in enumerate(recs) if r[2] == 0 and r[1] in (5, 9) and r[0] == 0 and r[4] in ("ACGTAC", "ACGT"))
    pb, ps = _write(recs, tmp_path, "long_cigar")
    for p, decode in ((pb, "gpu"), (ps, "gpu"), (pb, "host"), (pb, "gpu-stream")):
        with AlignmentFile(p, decode=decode) as af:
            with pytest.raises(IndexError, match="record %d " % first):
                af.count_coverage("c0", quality_threshold=0)
            with pytest.raises(IndexError):
                af.count_coverage("c0", quality_threshold=0)        # (no counts were kept)
            d = af.count_coverage_depth("c0")                       # the file stays usable
            assert d.sum() > 0
