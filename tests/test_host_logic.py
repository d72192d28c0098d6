"""Host-side logic of the product package, CPU only: float finishing of `classic`, the BAM
reader, the synthetic generator, region parsing."""
import io

import numpy as np
import pytest

from helpers import load_soa, write_fixture_bam
from oracle import bamio, classic as oc


def int_stats(d):
    """Exact integer statistics of a depth vector (what mcov_region_stats carries)."""
    d = np.asarray(d, dtype=np.int64)
    n = len(d)
    s = np.sort(d)
    q = n // 4
    return {"sum": int(d.sum()), "sumsq": int((d * d).sum()), "iq_sum": int(s[q:n - q].sum()),
            "min": int(d.min()), "max": int(d.max()), "med_lo": int(s[(n - 1) // 2]), "med_hi": int(s[n // 2])}


@pytest.mark.parametrize("seed", range(12))
def test_finish_classic_matches_numpy_reductions(seed):
    """finish_classic (integer moments) vs the reference's numpy reductions (pileup.py:18-26):
    ints identical, floats within 1e-6 relative before rounding, rounded values to the cent."""
    from metacov_b200.pileup import finish_classic
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 5000))
    d = rng.integers(0, [3, 50, 600, 8000][seed % 4], n)
    if seed % 3 == 0:
        d = np.sort(d)
    got = finish_classic(int_stats(d), n)
    want = oc.stats_from_columns(d.astype(np.float64))
    for k in ("min", "max", "med", "sum"):
        assert got[k] == want[k] and isinstance(got[k], int)
    for k in ("std", "avg", "q23"):
        assert isinstance(got[k], np.floating)
        assert abs(got[k] - want[k]) <= 0.01 + 1e-9
    assert got["avg"] == want["avg"] and got["q23"] == want["q23"]
    raw_std = np.std(d.astype(np.float64))
    exact = np.sqrt((n * int((d.astype(object) ** 2).sum()) - int(d.sum()) ** 2) / (n * n))
    assert abs(raw_std - exact) <= 1e-6 * max(raw_std, 1e-300)


def test_native_bam_reader_roundtrip(tmp_path):
    """csrc/bamio.cpp against the oracle's pure-Python reader on a BAM the oracle writer made."""
    from metacov_b200 import AlignmentFile
    z, b = load_soa("synth_small_soa.npz")
    refs = [str(x) for x in z["references"]]
    path = str(tmp_path / "t.bam")
    isize = (np.arange(len(b.tid)) % 700 - 350).astype(np.int32)
    bamio.write_bam(path, refs, z["lengths"].tolist(), b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, isize=isize)
    hdr, recs = bamio.read_bam(path)
    with AlignmentFile(path) as af:
        assert af.references == tuple(refs) == hdr.references
        assert af.lengths == tuple(z["lengths"].tolist())
        s = af.soa()
        for k, want in (("tid", b.tid), ("pos", b.pos), ("flag", b.flag), ("mapq", b.mapq), ("cig", b.cig),
                        ("isize", isize), ("l_seq", recs.l_seq)):
            assert np.array_equal(s[k], want), k
        assert np.array_equal(s["cig_off"], b.cig_off)
        un = (b.flag & 4) != 0
        assert af.mapped == int(np.sum(~un & (b.tid >= 0))) and af.unmapped == int(np.sum(un))
        assert af.get_tid("ctgC") == 2 and af.get_tid("nope") == -1
    with pytest.raises(OSError):
        AlignmentFile(str(tmp_path / "missing.bam"))
    bad = tmp_path / "bad.bam"
    bad.write_bytes(b"not a bam file at all, definitely")
    with pytest.raises(OSError):
        AlignmentFile(str(bad))


def test_native_bam_reader_on_reference_fixture(tmp_path):
    from metacov_b200 import AlignmentFile
    z, b = load_soa("fixture_soa.npz")
    with AlignmentFile(write_fixture_bam(str(tmp_path / "bbmap.sorted.bam"))) as af:
        assert af.references == ("ref1", "ref2") and af.lengths == (425, 575)
        assert (af.mapped, af.unmapped) == (3979, 133)
        s = af.soa()
        assert len(af) == 4112
        for k in ("tid", "pos", "flag", "mapq", "cig", "isize", "l_seq"):
            assert np.array_equal(s[k], z[k]), k
        assert np.array_equal(s["cig_off"], b.cig_off)


def test_synth_generator_shapes_and_sortedness():
    from metacov_b200 import synth
    for w in (synth.c2(0.005), synth.c3(0.0005), synth.c5(0.001, span_min=2000, span_max=6000)):
        b, isz, rl = synth.generate_host(w, want_reflen=True)
        key = b.tid.astype(np.int64) * (1 << 32) + b.pos
        assert np.all(np.diff(key) >= 0), w.name
        assert np.array_equal(rl, bamio.cigar_reflen(b.cig_off, b.cig))
        assert np.all(b.pos + rl <= w.contig_len[b.tid])
        assert np.all(np.bincount(b.tid, minlength=w.n_contigs) == np.diff(w.read_start))
        # any window of reads can be re-derived on its own (counter-based generator)
        lo, n = w.n_reads // 3, min(1000, w.n_reads - w.n_reads // 3)
        b2, isz2 = synth.generate_host(w, i0=lo, n=n)
        assert np.array_equal(b2.pos, b.pos[lo:lo + n]) and np.array_equal(b2.flag, b.flag[lo:lo + n])
        o = b.cig_off.astype(np.int64)
        assert np.array_equal(b2.cig, b.cig[o[lo]:o[lo + n]])


def test_native_seq_windows(tmp_path):
    """csrc/bamio.cpp: packed SEQ and the per-read k-mer windows (first bases of forward reads,
    last bases of reverse reads)."""
    from metacov_b200 import AlignmentFile
    z, b = load_soa("fixture_soa.npz")
    so = z["seq_off"]
    n = 300
    seqs = [z["seq"][so[i]:so[i + 1]] for i in range(n)]
    path = str(tmp_path / "s.bam")
    o = b.cig_off.astype(np.int64)
    bamio.write_bam(path, ["ref1", "ref2"], [425, 575], b.tid[:n], b.pos[:n], b.flag[:n], b.mapq[:n],
                    (o[:n + 1] - o[0]).astype(np.uint32), b.cig[o[0]:o[n]], seqs=seqs)
    P = 23
    with AlignmentFile(path) as af:
        win = af.seq_windows(P)
        assert win.shape == (n, (P + 1) // 2)
        assert np.array_equal(af.soa()["l_seq"], np.array([len(s) for s in seqs]))
        for i in range(n):
            nib = np.empty(2 * win.shape[1], np.uint8)
            nib[0::2] = win[i] >> 4
            nib[1::2] = win[i] & 15
            s = seqs[i]
            if b.flag[i] & 0x10:
                want = [s[len(s) - P + j] if len(s) - P + j >= 0 else 15 for j in range(P)]
            else:
                want = [s[j] if j < len(s) else 15 for j in range(P)]
            assert nib[:P].tolist() == [int(x) for x in want], i


def test_load_kmerhist_both_csv_dialects():
    """`load_kmerhist` (reference pileup.py:29-35): k-mer -> n0 / mean(n1..) per read number, unmapped and
    all-N rows dropped; the read-number column is `R` in the layout the reference was written for and
    `IsRead1` at the reference's HEAD (SURVEY.md Appendix C-8)."""
    import io
    from metacov_b200 import pileup
    rows = [("AAC", [10, 2, 4, 6], "Mapped", "R1"), ("AAC", [9, 3, 3, 3], "Mapped", "R2"), ("ACG", [0, 1, 1, 1], "Mapped", "R1"),
            ("NNN", [5, 5, 5, 5], "Mapped", "R1"), ("TTT", [7, 1, 1, 1], "Unmapped", "R1"), ("GGA", [8, 4, 4, 4], "Mapped", "R2")]
    want = [{"AAC": 10 / 4.0, "ACG": 0.0}, {"AAC": 9 / 3.0, "GGA": 2.0}]
    for rcol in ("R", "IsRead1"):
        csv_text = "kmer,n0,n1,n2,n3,Mapped,%s\n" % rcol + "".join(
            "%s,%s,%s,%s\n" % (k, ",".join(str(x) for x in n), m, r) for k, n, m, r in rows)
        got = pileup.load_kmerhist(io.StringIO(csv_text), k_len=3)
        assert [dict((k, float(v)) for k, v in d.items()) for d in got] == want, rcol


def test_native_bam_reader_rejects_malformed_sizes(tmp_path):
    """Sizes read from the file are validated before anything is allocated from them (a corrupt
    ISIZE or l_seq must end in an error code / OSError, never in an exception crossing the C ABI)."""
    import ctypes as C
    import struct
    import zlib
    from metacov_b200 import AlignmentFile, _capi
    z, b = load_soa("synth_small_soa.npz")
    refs = [str(x) for x in z["references"]]
    good = str(tmp_path / "good.bam")
    bamio.write_bam(good, refs, z["lengths"].tolist(), b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig)
    raw = bytearray(open(good, "rb").read())
    # (1) ISIZE of the first BGZF block claims 1 GiB
    bsize = struct.unpack_from("<H", raw, 16)[0] + 1
    bad1 = bytearray(raw)
    struct.pack_into("<I", bad1, bsize - 4, 1 << 30)
    p1 = str(tmp_path / "isize.bam")
    open(p1, "wb").write(bad1)
    with pytest.raises(OSError):
        AlignmentFile(p1)
    # (2) a record whose l_seq does not fit its block_size
    data = bytearray(bamio.bgzf_inflate(bytes(raw)))
    hdr, recs = bamio.read_bam(good)
    p = 12 + struct.unpack_from("<i", data, 4)[0]
    for _ in refs:
        p += 8 + struct.unpack_from("<i", data, p)[0]
    struct.pack_into("<i", data, p + 4 + 16, 0x7fffff00)          # l_seq of the first record
    p2 = str(tmp_path / "lseq.bam")
    open(p2, "wb").write(bamio.bgzf_compress(bytes(data)))
    h = C.c_void_p()
    err = C.create_string_buffer(256)
    assert _capi.lib.mcov_bam_open(C.byref(h), p2.encode(), err, 256) == 0
    assert _capi.lib.mcov_bam_load(h, 0) == _capi.MCOV_ERR_IO
    assert _capi.lib.mcov_bam_load_seq(h) == _capi.MCOV_ERR_IO
    _capi.lib.mcov_bam_close(h)


def test_finish_classic_many_equals_the_per_record_version():
    """pileup.finish_classic_many (numpy over all regions) returns exactly what finish_classic returns record by record --
    values, value types, NaN for a q23 without an interquartile range -- including regions whose integer moments leave the
    range float64 holds exactly (those take the scalar path)."""
    from metacov_b200 import _capi
    from metacov_b200.pileup import finish_classic, finish_classic_many
    rng = np.random.default_rng(7)
    g = 4000
    st = np.zeros(g, dtype=_capi.REGION_STATS_DTYPE)
    n = rng.integers(1, 60000, g)
    dm = np.where(rng.random(g) < 0.8, rng.integers(0, 200, g), rng.integers(0, 9000, g))
    st["sum"] = n * dm + rng.integers(0, 50, g)
    st["sumsq"] = n * (dm.astype(np.int64) ** 2) + rng.integers(0, 99999, g)
    iqn = n - 2 * (n // 4)
    st["iq_sum"] = iqn * dm + rng.integers(0, 7, g)
    st["max"] = dm * 2
    st["med_lo"] = dm
    st["med_hi"] = dm + rng.integers(0, 3, g)
    n[:20] = 90_000_000                                  # beyond the exact range
    st["sumsq"][:20] = 1 << 60
    n[20:40] = rng.integers(1, 4, 20)                    # 1..3 slots: iq range of 1 or 2
    got = finish_classic_many(st, n)
    assert finish_classic_many(st[:0], n[:0]) == []
    for i in range(g):
        want = finish_classic(st[i], n[i])
        assert set(got[i]) == set(want)
        for k, v in want.items():
            assert type(got[i][k]) is type(v), (i, k)
            assert got[i][k] == v or (v != v and got[i][k] != got[i][k]), (i, k, got[i][k], v)
