"""The oracle pinned against the committed golden vectors (made by the reference's own
classic(), oracle/make_golden.py) and its formulations against each other.  CPU only."""
import hashlib
import os

import numpy as np
import pytest

from helpers import assert_classic_equal, fake_bam, load_json, load_soa, regions_of, write_fixture_bam
from oracle import bamio, classic as oc, cport
from oracle.pysam_boundary import FakeAlignmentFile, PileupFilter, plp_columns


def test_fixture_known_answers_appendix_b():
    """SURVEY.md Appendix B: record counts, flags, BAI stats, depth sha1s."""
    z, b = load_soa("fixture_soa.npz")
    gold = load_json("fixture_classic.json")
    assert len(b.tid) == 4112 == gold["n_records"]
    assert gold["mapped"] == 3979 and gold["unmapped"] == 133
    assert int(PileupFilter().passes(b.flag, b.mapq).sum()) == 3350
    d = oc.depth_diffarray(b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, z["lengths"])
    assert int(d[0].sum()) == 121714 and int(d[1].sum()) == 166182
    assert hashlib.sha1(d[0].astype("<i4").tobytes()).hexdigest() == "11ed20e88c63aa6c8ee4c7a7b002e66f5b1b69aa"
    assert hashlib.sha1(d[1].astype("<i4").tobytes()).hexdigest() == "d3075eb38351dde7ace91e8975de6333040f5373"
    for c, name in enumerate(gold["references"]):
        assert np.array_equal(d[c], np.load(os.path.join(os.path.dirname(__file__), "golden", "fixture_depth_%s.npy" % name)))


@pytest.mark.parametrize("soa,js", [("fixture_soa.npz", "fixture_classic.json"),
                                    ("synth_small_soa.npz", "synth_small_classic.json")])
def test_python_oracle_matches_reference_golden(soa, js):
    z, _ = load_soa(soa)
    bam = fake_bam(z)
    for row in load_json(js)["classic"]:
        got = oc.classic(bam, row["ref"], row["start"], row["end"])
        assert got == row["result"], row
        assert isinstance(got["min"], int) and isinstance(got["std"], np.floating)


@pytest.mark.parametrize("soa,js", [("fixture_soa.npz", "fixture_classic.json"),
                                    ("synth_small_soa.npz", "synth_small_classic.json")])
def test_c_oracle_matches_reference_golden(soa, js):
    from metacov_b200.pileup import finish_classic
    z, b = load_soa(soa)
    gold = load_json(js)
    d_diff, off, _ = cport.depth(b, z["lengths"], mode="diff")
    d_plp, _, info = cport.depth(b, z["lengths"], mode="plp")
    d_par, _, _ = cport.depth(b, z["lengths"], mode="par", threads=3)
    assert info["dropped_by_cap"] == 0
    assert np.array_equal(d_diff, d_plp) and np.array_equal(d_diff, d_par)
    tid, st, en = regions_of(gold, z["references"])
    stats = cport.region_stats(d_diff, off, z["lengths"], tid, st, en, threads=2)
    for row, rec, a, e in zip(gold["classic"], stats, st, en):
        assert_classic_equal(finish_classic(rec, e - a), row["result"], row)


def test_plp_engine_cap_semantics():
    """htslib maxcnt: only reads starting exactly at the column being assembled are dropped,
    once 8000 reads are buffered (SURVEY.md Appendix A-6)."""
    reads = [(0, 100, 200)] * 9000 + [(0, 150, 250)] * 10
    cols = {p: n for _, p, n in plp_columns(iter(reads), 8000)}
    assert cols[100] == 8000 and cols[149] == 8000
    # the first read at 150 arrives while the iterator is still at 100 (never capped); by the time
    # the other nine arrive the iterator sits at 150 with 8001 reads buffered: all dropped
    assert cols[150] == 8001
    assert cols[200] == 1 and 250 not in cols
    # reads arriving one position apart are never capped
    reads = [(0, p, p + 20000) for p in range(9000)]
    cols = {p: n for _, p, n in plp_columns(iter(reads), 8000)}
    assert cols[8999] == 9000
    # cap disabled
    reads = [(0, 5, 10)] * 9000
    assert {p: n for _, p, n in plp_columns(iter(reads), 1 << 60)}[5] == 9000
    # reflen 0 contributes nothing
    assert list(plp_columns(iter([(0, 5, 5), (0, 7, 9)]), 8000)) == [(0, 7, 1), (0, 8, 1)]
    with pytest.raises(ValueError):
        list(plp_columns(iter([(0, 9, 12), (0, 3, 5)]), 8000))


def test_cap_c_vs_python_and_idle_condition():
    from metacov_b200.engine import ReadBatch
    rng = np.random.default_rng(7)
    n = 15000
    pos = np.sort(np.r_[np.full(9000, 300), rng.integers(0, 900, n - 9000)]).astype(np.int32)
    b = ReadBatch(np.zeros(n, np.int32), pos, np.zeros(n, np.uint16), np.full(n, 30, np.uint8),
                  np.arange(n + 1, dtype=np.uint32), np.full(n, 80 << 4, np.uint32))
    d_diff, off, _ = cport.depth(b, [1000], mode="diff")
    d_plp, _, info = cport.depth(b, [1000], mode="plp")
    assert info["dropped_by_cap"] > 0 and d_plp.max() <= 8000 < d_diff.max()
    z = dict(references=np.array(["c"]), lengths=np.array([1000], np.int32), tid=b.tid, pos=b.pos, flag=b.flag,
             mapq=b.mapq, cig_off=b.cig_off, cig=b.cig)
    cols = oc.depth_columns(fake_bam(z), "c", 0, 1000)
    assert np.array_equal(cols.astype(np.int32), d_plp[:1000])
    starts = np.bincount(pos, minlength=1000)
    assert not oc.cap_is_idle(d_diff[:1000], starts, 8000)
    assert oc.cap_is_idle(d_diff[:1000], starts, 20000)


def test_isize_known_answers_appendix_b():
    z, _ = load_soa("fixture_soa.npz")
    hist, cnt, mx = cport.isize_hist(z["flag"], z["isize"], (), 1024)
    assert mx == 248 and hist[0, 0] == 762 and int(cnt[0]) == 4112
    assert hashlib.sha1(hist[0, :249].astype("<u4").tobytes()).hexdigest() == "1f9e912d7107e60feebf927217016199cc4a1448"
    # ByFlag(-g Mapped -g IsRead1): group index = bits MSB first (scan.pyx:414-418)
    _, cnt, _ = cport.isize_hist(z["flag"], z["isize"], (0x4, 0x40), 1024)
    # n = (unmapped<<1)|read1 -> (Mapped,R2)=0 (Mapped,R1)=1 (Unmapped,R2)=2 (Unmapped,R1)=3
    assert cnt.tolist() == [1996, 1983, 60, 73]


def test_bam_reader_on_reference_fixture(tmp_path):
    path = write_fixture_bam(str(tmp_path / "bbmap.sorted.bam"))
    hdr, recs = bamio.read_bam(path)
    z, b = load_soa("fixture_soa.npz")
    assert hdr.references == ("ref1", "ref2") and hdr.lengths == (425, 575)
    assert np.array_equal(recs.tid, b.tid) and np.array_equal(recs.cig, b.cig)
    per_ref, n_no_coor = bamio.read_bai_stats(path + ".bai")
    assert per_ref == [(1694, 38), (2285, 91)] and n_no_coor == 4


def test_kmer_hist_known_answers():
    """scan.pyx:491-533 restated; Appendix B: 3666 fixture reads are long enough for the default
    KmerHist (K=7, NK=8, STEP=7, OFFSET=0)."""
    from oracle import scanstats
    z, _ = load_soa("fixture_soa.npz")
    so = z["seq_off"]
    seqs = [z["seq"][so[i]:so[i + 1]] for i in range(len(z["tid"]))]
    h = scanstats.kmer_hist(z["flag"], seqs, 7, 8, 7, 0)
    assert h.shape == (1, 4 ** 7 + 1, 8)
    assert (h[0].sum(axis=0) == 3666).all()
    assert hashlib.sha1(h.tobytes()).hexdigest() == "ed8186021fd049fba4cb4cfadadff9103651b2d9"
    # a reverse-strand read is reverse-complemented back before its k-mers are taken
    fwd = np.array([1, 2, 4, 8, 1, 1, 2, 2], np.uint8)            # ACGTAACC
    hf = scanstats.kmer_hist([0], [fwd], 2, 2, 3, 0)
    assert hf[0, 0 | (1 << 2), 0] == 1 and hf[0, 3 | (0 << 2), 1] == 1          # "AC" at 0, "TA" at 3
    hr = scanstats.kmer_hist([16], [fwd], 2, 2, 3, 0)             # read = revcomp = GGTTACGT
    assert hr[0, 2 | (2 << 2), 0] == 1 and hr[0, 3 | (0 << 2), 1] == 1          # "GG" at 0, "TA" at 3
    hn = scanstats.kmer_hist([0], [np.array([1, 15, 1, 1, 1, 1], np.uint8)], 2, 2, 3, 0)
    assert hn[0, 16, 0] == 1 and hn[0, 0, 1] == 1                # an N sends the k-mer to row 4**K
