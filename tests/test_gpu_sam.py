"""SAM text decoded on the GPU (mcov_sam_decode_gpu, csrc/sam_gpu.cu) against the BAM decoders on the same records:
columns, read names and SEQ, depth, the AlignmentFile protocol and the CLI; chunk borders everywhere; long-read lines
with more than 65 535 ops; malformed files naming their line."""
import csv

import numpy as np
import pytest
from click.testing import CliRunner

from helpers import load_json, load_soa, write_fixture_bam
from oracle import bamio, cport
import samio

pytestmark = pytest.mark.gpu

COLS = ("tid", "pos", "flag", "mapq", "l_seq", "isize", "cig_off", "cig")


def _fixture_args():
    z, b = load_soa("fixture_soa.npz")
    so = z["seq_off"]
    n = len(b.tid)
    return z, b, dict(isize=z["isize"], names=[str(x) for x in z["names"]], l_seq=z["l_seq"],
                      seqs=[z["seq"][so[i]:so[i + 1]] for i in range(n)])


@pytest.fixture(scope="module")
def fixture_pair(tmp_path_factory):
    d = tmp_path_factory.mktemp("sam")
    z, b, kw = _fixture_args()
    pb = write_fixture_bam(str(d / "fixture.bam"))
    ps = str(d / "fixture.sam")
    aux = ["AM:C:%d\tXT:A:%s\tRG:Z:lane%d" % (int(z["mapq"][i]), "U" if z["mapq"][i] else "R", i % 11 * 7) for i in range(len(b.tid))]
    samio.write_sam(ps, [str(x) for x in z["references"]], z["lengths"].tolist(), b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig,
                    mtid=z["mtid"], mpos=z["mpos"], aux=aux, **kw)
    return pb, ps


def _device_columns(soa):
    return {c: soa.to_host(c) for c in COLS}


def test_fixture_sam_equals_bam(fixture_pair):
    from metacov_b200 import AlignmentFile, pileup
    pb, ps = fixture_pair
    gold = load_json("fixture_classic.json")
    with AlignmentFile(pb, decode="gpu") as bam, AlignmentFile(ps) as sam:
        assert sam.format == "sam" and sam.decode == "gpu" and not sam.has_index()
        assert sam.references == bam.references and sam.lengths == bam.lengths
        assert sam.text.startswith("@HD\tVN:1.4") and sam.text.count("\n@SQ\t") == 2
        hs, ss = bam.soa(), sam.soa()
        for c in COLS:
            assert np.array_equal(hs[c], ss[c]), c
        assert (sam.mapped, sam.unmapped) == (3979, 133) == (gold["mapped"], gold["unmapped"])
        for row in gold["classic"]:
            assert pileup.classic(sam, row["ref"], row["start"], row["end"]) == row["result"], row
        assert [(c.pos, c.n) for c in sam.pileup("ref1", 0, 425)] == [(c.pos, c.n) for c in bam.pileup("ref1", 0, 425)]
        assert np.array_equal(sam.name_hashes(), bam.name_hashes())
        for k in (1, 4, 7, 15):
            assert np.array_equal(sam.qas_kmer_codes(k), bam.qas_kmer_codes(k)), k
        for w in (1, 7, 56, 101, 400):
            assert np.array_equal(sam.seq_windows(w), bam.seq_windows(w)), w
        assert sam._h is None
    with pytest.raises(ValueError):
        AlignmentFile(ps, decode="gpu-stream")
    for mode in ("host", "auto"):
        with AlignmentFile(ps, decode=mode) as sam:
            assert sam.decode == "gpu"
    old = AlignmentFile.SAM_DECODE_FOOTPRINT
    AlignmentFile.SAM_DECODE_FOOTPRINT = 1 << 50
    try:
        with pytest.raises(OSError, match="BAM input streams"):
            AlignmentFile(ps)
    finally:
        AlignmentFile.SAM_DECODE_FOOTPRINT = old


def _random_set(rng, n=6000):
    """The read set of test_gpu_bamgpu.test_names_and_seq_on_the_device: clips, both strands, ambiguity codes, empty SEQ."""
    from metacov_b200 import ReadBatch
    lengths = np.array([40000, 30000], np.int32)
    tid = np.sort(rng.integers(0, 2, n)).astype(np.int32)
    pos = np.zeros(n, np.int32)
    for c in range(2):
        m = tid == c
        pos[m] = np.sort(rng.integers(0, lengths[c] - 400, m.sum()))
    flag = (rng.integers(0, 2, n) * 0x10 + rng.integers(0, 2, n) * 0x1 + rng.integers(0, 2, n) * 0x2 +
            rng.choice([0x40, 0x80], n)).astype(np.uint16)
    cig, off, seqs, names = [], [0], [], []
    for i in range(n):
        ops = []
        if rng.random() < 0.2: ops.append((5, int(rng.integers(1, 9))))
        if rng.random() < 0.4: ops.append((4, int(rng.integers(1, 30))))
        ops.append((0, int(rng.integers(1, 120))))
        if rng.random() < 0.3: ops += [(1, int(rng.integers(1, 5))), (0, int(rng.integers(1, 60)))]
        if rng.random() < 0.3: ops += [(2, int(rng.integers(1, 5))), (0, int(rng.integers(1, 60)))]
        if rng.random() < 0.4: ops.append((4, int(rng.integers(1, 30))))
        if rng.random() < 0.2: ops.append((5, int(rng.integers(1, 9))))
        qlen = 0 if i % 97 == 0 else sum(l for o, l in ops if o in (0, 1, 4))
        cig += [(l << 4) | o for o, l in ops]
        off.append(len(cig))
        seqs.append(rng.choice(np.array([1, 2, 4, 8, 15, 1, 2, 4, 8, 1, 2, 4, 8, 3], np.uint8), qlen))
        names.append("r%d/%s" % (i // 2, "x" * int(rng.integers(0, 40))))
    b = ReadBatch(tid, pos, flag, np.full(n, 30, np.uint8), np.array(off, np.uint32), np.array(cig, np.uint32))
    return b, lengths, dict(isize=rng.integers(-600, 600, n).astype(np.int32), names=names, seqs=seqs)


def test_names_seq_experimental_and_scan(tmp_path):
    from metacov_b200 import AlignmentFile, pileup
    from metacov_b200 import scan as mscan
    b, lengths, kw = _random_set(np.random.default_rng(77))
    n = len(b.tid)
    pb, ps = str(tmp_path / "seq.bam"), str(tmp_path / "seq.sam")
    for w, p in ((bamio.write_bam, pb), (samio.write_sam, ps)):
        w(p, ["c0", "c1"], lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, **kw)
    with AlignmentFile(pb, decode="gpu") as bam, AlignmentFile(ps) as sam:
        assert np.array_equal(sam.name_hashes(), bam.name_hashes())
        for k in (1, 3, 7, 15):
            assert np.array_equal(sam.qas_kmer_codes(k), bam.qas_kmer_codes(k)), k
        for w in (1, 2, 56, 57, 300):
            assert np.array_equal(sam.seq_windows(w), bam.seq_windows(w)), w
        kc = [{}, {}]
        rr = np.random.default_rng(5)
        for r in range(2):
            for code in range(4 ** 3):
                if rr.random() < 0.8:
                    kc[r]["".join("ACGT"[(code >> (2 * (2 - j))) & 3] for j in range(3))] = float(rr.uniform(0.5, 2.0))
        for ref, s0, e0 in (("c0", 0, 4000), ("c1", 1000, 9000)):
            assert pileup.experimental(bam, kc, 3, None, ref, s0, e0) == pileup.experimental(sam, kc, 3, None, ref, s0, e0)
        rows = []
        for f in (bam, sam):
            kh = mscan.KmerHist(3, 4, 3, 1)
            mscan.scan_reads(f, None, [kh])
            rows.append(kh.counts.copy())
        assert np.array_equal(rows[0], rows[1]) and rows[0].sum() > 0
        for maxreads in (0, 37):
            res = []
            for f in (bam, sam):
                bf = mscan.ByFlag([mscan.IsizeHist(), mscan.KmerHist(3, 4, 3, 1)], [mscan.Flags["Readdir"], mscan.Flags["IsRead1"]])
                nrec = mscan.scan_reads(f, None, bf, maxreads=maxreads)
                res.append((nrec, [[list(map(str, r)) for r in bf.get_rows(i)] for i in range(2)]))
            assert res[0][0] == res[1][0] == (maxreads or n)
            assert res[0][1] == res[1][1]
        assert sam._h is None and bam._h is None


def _depth_check(eng, soa, batch, lengths):
    from metacov_b200 import bamgpu
    bamgpu.depth_sorted(eng, soa)
    d, off, info = cport.depth(batch, lengths, mode="diff")
    assert eng.pass_info()["n_pass"] == info["n_pass"]
    for c in range(len(lengths)):
        assert np.array_equal(eng.copy_depth(c), d[off[c]:off[c] + lengths[c]]), c


def _records_equal(soa, batch, isize=None):
    got = _device_columns(soa)
    for c in ("tid", "pos", "flag", "mapq", "cig"):
        assert np.array_equal(got[c], np.asarray(getattr(batch, c))), c
    assert np.array_equal(got["cig_off"].astype(np.int64), np.asarray(batch.cig_off).astype(np.int64))
    if isize is not None:
        assert np.array_equal(got["isize"], isize)


def test_c2_sample_and_chunk_borders(tmp_path):
    """~200 k short reads with full QUAL and two optional fields: records and depth equal the generating columns, and
    chunk sizes that put copy borders at every place in a line give identical columns."""
    from metacov_b200 import CoverageEngine, bamgpu, synth
    w = synth.c2(0.02)
    hb, isz = synth.generate_host(w)
    n = len(hb.tid)
    rng = np.random.default_rng(2)
    letters = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n * 150)].tobytes().decode()
    seqs = [letters[i * 150:(i + 1) * 150] for i in range(n)]
    p = str(tmp_path / "c2.sam")
    samio.write_sam(p, ["c%d" % c for c in range(w.n_contigs)], [int(x) for x in w.contig_len], hb.tid, hb.pos, hb.flag, hb.mapq,
                    hb.cig_off, hb.cig, isize=isz, seqs=seqs, quals=["I" * 150] * n, aux=["NM:i:0\tAS:i:%d" % (i % 150) for i in range(n)])
    lengths = [int(x) for x in w.contig_len]
    with CoverageEngine(lengths) as eng:
        soa = bamgpu.decode_sam(eng, p)
        assert soa.n_records == n
        _records_equal(soa, hb, isz)
        base = _device_columns(soa)
        _depth_check(eng, soa, hb, lengths)
        data = open(p, "rb").read()
        assert len(data) > 8 << 20
        for chunk in (1, 40_000, 1 << 20, 3 << 20, 0):
            s2 = bamgpu.decode_sam(eng, data, chunk_bytes=chunk)
            got = _device_columns(s2)
            for c in COLS:
                assert np.array_equal(got[c], base[c]), (chunk, c)


def test_long_reads_and_65536_ops(tmp_path):
    """C5-like long reads (lines of 100 KB and more), three of them with more than 65 535 ops."""
    from metacov_b200 import CoverageEngine, ReadBatch, bamgpu, synth
    w = synth.c5(0.0005)
    hb, isz = synth.generate_host(w)
    cig, off = [np.asarray(hb.cig)], np.asarray(hb.cig_off).astype(np.int64)
    lens = np.diff(off)
    ops = [np.asarray(hb.cig[off[i]:off[i + 1]]) for i in range(len(hb.tid))]
    for i in (5, 700, 1900):
        ops[i] = np.array([(3 << 4) | 0, (1 << 4) | 1] * 35000, np.uint32)          # 70 000 ops
    cig = np.concatenate(ops).astype(np.uint32)
    off = np.concatenate(([0], np.cumsum([len(o) for o in ops]))).astype(np.uint32)
    b = ReadBatch(hb.tid, hb.pos, hb.flag, hb.mapq, off, cig)
    lengths = [int(x) for x in w.contig_len]
    p = str(tmp_path / "c5.sam")
    samio.write_sam(p, ["c%d" % c for c in range(w.n_contigs)], lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, isize=isz)
    assert max(len(l) for l in open(p, "rb")) > 100_000 and int(lens.max()) > 0
    with CoverageEngine(lengths) as eng:
        soa = bamgpu.decode_sam(eng, p)
        _records_equal(soa, b, isz)
        assert soa.to_host("l_seq")[700] == 35000 * 4
        _depth_check(eng, soa, b, lengths)


def test_unsorted_sam_takes_the_push_path(tmp_path):
    from metacov_b200 import AlignmentFile, ReadBatch, synth
    w = synth.c2(0.002)
    hb, _ = synth.generate_host(w)
    perm = np.arange(len(hb.tid)); perm[10], perm[15000] = perm[15000], perm[10]
    ub = ReadBatch(hb.tid[perm], hb.pos[perm], hb.flag[perm], hb.mapq[perm], np.arange(len(perm) + 1, dtype=np.uint32),
                   np.full(len(perm), 100 << 4, np.uint32))
    refs, lengths = ["c%d" % c for c in range(w.n_contigs)], [int(x) for x in w.contig_len]
    pb, ps = str(tmp_path / "u.bam"), str(tmp_path / "u.sam")
    bamio.write_bam(pb, refs, lengths, ub.tid, ub.pos, ub.flag, ub.mapq, ub.cig_off, ub.cig)
    samio.write_sam(ps, refs, lengths, ub.tid, ub.pos, ub.flag, ub.mapq, ub.cig_off, ub.cig)
    with AlignmentFile(pb) as bam, AlignmentFile(ps) as sam:
        for c in range(len(lengths)):
            assert np.array_equal(sam.count_coverage_depth(refs[c]), bam.count_coverage_depth(refs[c])), c
        assert sam.coverage_engine().pass_info()["sorted"] == 0


def test_malformed_files_name_their_line(tmp_path):
    from test_sam_host import BAD_LINES, bad_file
    from metacov_b200 import AlignmentFile, CoverageEngine, McovError, bamgpu
    good = bad_file("r2\t16\tc1\t9\t0\t1S2M\t=\t5\t-4\tAcG\t*", None)
    with CoverageEngine([1000, 2000]) as eng:
        for line, field in BAD_LINES:
            with pytest.raises(McovError, match="line 7"):
                bamgpu.decode_sam(eng, bad_file(line, field))
            soa = bamgpu.decode_sam(eng, good)                 # the context survives
            assert soa.n_records == 5 and soa.to_host("tid").tolist() == [0, 0, 0, 1, 0]
        for header in ("@SQ\tSN:c0\n", "@SQ\tSN:c0\tLN:5\n@SQ\tSN:c0\tLN:6\n"):
            with pytest.raises(McovError, match="SQ"):
                bamgpu.decode_sam(eng, (header + "r\t0\t*\t0\t0\t*\t*\t0\t0\t*\t*\n").encode())
    p = tmp_path / "bad.sam"
    p.write_bytes(bad_file("r1\t0\tc9\t5\t30\t3M\t*\t0\t0\tACG\tIII", 2))
    with pytest.raises(OSError, match="line 7: RNAME"):
        AlignmentFile(str(p))


def test_cli_scan_and_pileup(fixture_pair, tmp_path):
    from test_gpu_cli import BLAST7
    from metacov_b200.cli import pileup as pileup_cmd, scan as scan_cmd
    pb, ps = fixture_pair
    outs = {}
    for name, path in (("bam", pb), ("sam", ps)):
        d = tmp_path / name
        d.mkdir()
        res = CliRunner().invoke(scan_cmd, [path, "-o", str(d / "k.csv"), "-I", str(d / "i.csv"), "-g", "Mapped", "-g", "IsRead1"])
        assert res.exit_code == 0, res.output
        rb = d / "r.blast7"
        rb.write_text(BLAST7)
        for tag, extra in (("hdr", []), ("blast", ["-rb", str(rb)]), ("kmer", ["-k", str(d / "k.csv")]),
                           ("bg", ["-bg", str(d / "cov.bedgraph"), "-w", "100", "-wo", str(d / "win.csv")])):
            res = CliRunner().invoke(pileup_cmd, ["-b", path, "-o", str(d / (tag + ".csv"))] + extra)
            assert res.exit_code == 0, res.output
        outs[name] = {f.name: f.read_text() for f in sorted(d.iterdir()) if f.suffix != ".blast7"}
    assert outs["sam"] == outs["bam"]
    assert len(list(csv.reader(outs["sam"]["blast.csv"].splitlines()))) == 5
