"""The drop-in Python API and CLI on the GPU, against the committed golden vectors (reference
tests/test_cli.py runs the same commands but only asserts exit_code == 0)."""
import csv
import io
import os

import numpy as np
import pytest
from click.testing import CliRunner

from helpers import load_json, load_soa, write_fixture_bam
from oracle import cport
from test_dropin_surface import BLAST7

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def fixture_bam(tmp_path_factory):
    """The reference fixture rebuilt from tests/golden/fixture_soa.npz (helpers.write_fixture_bam)."""
    return write_fixture_bam(str(tmp_path_factory.mktemp("bam") / "fixture.bam"))


def test_classic_api_matches_golden(fixture_bam):
    from metacov_b200 import AlignmentFile, pileup
    gold = load_json("fixture_classic.json")
    with AlignmentFile(fixture_bam) as bam:
        assert bam.mapped == gold["mapped"] and bam.unmapped == gold["unmapped"]
        for row in gold["classic"]:
            got = pileup.classic(bam, row["ref"], row["start"], row["end"])
            assert got == row["result"], row
            assert list(got) == ["min", "max", "med", "std", "avg", "q23", "sum"]
            assert isinstance(got["min"], int) and isinstance(got["sum"], int) and isinstance(got["std"], np.floating)
        with pytest.raises(ValueError):
            pileup.classic(bam, "ref1", 5, 5)                  # np.amin of an empty vector (pileup.py:19)
        # pysam protocol: columns of a region
        cols = {c.pos: c.n for c in bam.pileup("ref1", 0, 425)}
        want = np.load(os.path.join(os.path.dirname(__file__), "golden", "fixture_depth_ref1.npy"))
        assert all(cols.get(p, 0) == want[p] for p in range(425))
    with pytest.raises(TypeError):
        pileup.classic(object(), "ref1", 0, 5)                 # foreign bam objects: no CPU fallback


def run_pileup(args):
    from metacov_b200.cli import pileup
    res = CliRunner().invoke(pileup, args)
    assert res.exit_code == 0, res.output
    return res


def test_cli_pileup_blast7_and_header_regions(fixture_bam, tmp_path):
    gold = load_json("fixture_classic.json")["classic"]
    rb = tmp_path / "regions.blast7"
    rb.write_text(BLAST7)
    out = tmp_path / "out.csv"
    run_pileup(["-b", fixture_bam, "-rb", str(rb), "-o", str(out)])
    rows = list(csv.DictReader(open(out)))
    assert list(rows[0]) == ["sacc", "start", "end", "avg", "max", "med", "min", "q23", "std", "sum"]
    # regions.blast7 rows are golden rows 2..5 (the last one written reversed: 575..301)
    assert [(r["sacc"], r["start"], r["end"]) for r in rows] == [("ref1", "1", "425"), ("ref2", "1", "575"),
                                                                  ("ref2", "1", "300"), ("ref2", "575", "301")]
    for r, g in zip(rows, gold[2:6]):
        for k, v in g["result"].items():
            assert float(r[k]) == float(v), (r, g)
        assert r["sum"] == str(g["result"]["sum"]) and r["avg"] == str(np.float64(g["result"]["avg"]))
    # regions from the BAM header (reference test_pileup2)
    out2 = tmp_path / "out2.csv"
    run_pileup(["-b", fixture_bam, "-o", str(out2)])
    rows = list(csv.DictReader(open(out2)))
    assert [(r["sacc"], r["start"], r["end"]) for r in rows] == [("ref1", "0", "425"), ("ref2", "0", "575")]
    for r, g in zip(rows, gold[0:2]):
        for k, v in g["result"].items():
            assert float(r[k]) == float(v)
    # CSV regions
    rc = tmp_path / "regions.csv"
    rc.write_text("sequence_id,start,end\nref2,301,575\n")
    out3 = tmp_path / "out3.csv"
    run_pileup(["-b", fixture_bam, "-rc", str(rc), "-o", str(out3)])
    row = list(csv.DictReader(open(out3)))[0]
    assert float(row["q23"]) == gold[5]["result"]["q23"] and row["min"] == "5"


def test_scan_api_and_cli(fixture_bam, tmp_path):
    from metacov_b200 import AlignmentFile, scan
    from metacov_b200.cli import scan as scan_cmd
    z, _ = load_soa("fixture_soa.npz")
    # API: ByFlag(IsizeHist) over every record
    calls = []
    with AlignmentFile(fixture_bam) as af:
        counters = scan.ByFlag([scan.IsizeHist()], [scan.Flags["Mapped"], scan.Flags["IsRead1"]])
        n = scan.scan_reads(af, None, counters, 1000, lambda: calls.append(1))
    assert n == 4112 and len(calls) == 4
    rh, rc, rmx = cport.isize_hist(z["flag"], z["isize"], (0x4, 0x40), 1024)
    for g, p in enumerate(counters.processors):
        h = p.processors[0]
        nz = np.nonzero(rh[g])[0]
        assert h.max_isize == (int(nz[-1]) if len(nz) else 0)
        assert np.array_equal(h.counts[:h.max_isize + 1], rh[g][:h.max_isize + 1])
        assert h.counts.dtype == np.uint32 and len(h.counts) in (128, 256, 512)
    # ungrouped list + maxreads
    with AlignmentFile(fixture_bam) as af:
        h = scan.IsizeHist()
        assert scan.scan_reads(af, None, [h], maxreads=1000) == 1000
    r1, _, _ = cport.isize_hist(z["flag"][:1000], z["isize"][:1000], (), 1024)
    assert np.array_equal(h.counts[:h.max_isize + 1], r1[0][:h.max_isize + 1])
    # CLI
    out = tmp_path / "isize.csv"
    res = CliRunner().invoke(scan_cmd, [fixture_bam, "-I", str(out), "-g", "Mapped"])
    assert res.exit_code == 0, res.output
    rows = list(csv.reader(open(out)))
    assert rows[0] == ["n", "count", "Mapped"]
    r2, _, _ = cport.isize_hist(z["flag"], z["isize"], (0x4,), 1024)
    mapped_rows = [r for r in rows[1:] if r[2] == "Mapped"]
    assert len(mapped_rows) == 249 and int(mapped_rows[0][1]) == int(r2[0][0]) and int(mapped_rows[210][1]) == int(r2[0][210])
    # out-of-scope options fail loudly instead of computing something else
    res = CliRunner().invoke(scan_cmd, [fixture_bam, "-b", str(tmp_path / "b.csv")])
    assert res.exit_code != 0 and "outside the GPU hot path" in res.output


def test_kmer_hist_api_and_cli(fixture_bam, tmp_path):
    """KmerHist on the GPU against the restated scan.pyx:491-533 (oracle/scanstats.py)."""
    from metacov_b200 import AlignmentFile, scan
    from metacov_b200.cli import scan as scan_cmd
    from oracle import scanstats
    z, _ = load_soa("fixture_soa.npz")
    so = z["seq_off"]
    seqs = [z["seq"][so[i]:so[i + 1]] for i in range(len(z["tid"]))]
    for K, NK, STEP, OFFSET, gf in ((7, 8, 7, 0, ()), (3, 5, 2, 4, (0x10, 0x40)), (5, 3, 9, 1, (0x4,))):
        with AlignmentFile(fixture_bam) as af:
            flags = [f for f in scan.Flags.values() if f.flag in gf]
            flags.sort(key=lambda f: gf.index(f.flag))
            counters = scan.ByFlag([scan.KmerHist(K, NK, STEP, OFFSET), scan.IsizeHist()], flags)
            assert scan.scan_reads(af, None, counters) == 4112
        want = scanstats.kmer_hist(z["flag"], seqs, K, NK, STEP, OFFSET, gf)
        for g, p in enumerate(counters.processors):
            assert np.array_equal(p.processors[0].counts, want[g]), (K, NK, STEP, OFFSET, g)
    # CLI: reference tests/test_cli.py:22-29 runs `scan X.bam -o out1.csv`
    out = tmp_path / "kmers.csv"
    res = CliRunner().invoke(scan_cmd, [fixture_bam, "-o", str(out), "-I", str(tmp_path / "i.csv")])
    assert res.exit_code == 0, res.output
    rows = list(csv.reader(open(out)))
    want = scanstats.kmer_hist(z["flag"], seqs, 7, 8, 7, 0)[0]
    assert rows[0] == ["kmer"] + ["n%d" % i for i in range(8)] and rows[1][0] == "NNNNNNN" and len(rows) == 4 ** 7 + 2
    assert [int(x) for x in rows[1][1:]] == want[4 ** 7].tolist()
    assert rows[2][0] == "AAAAAAA" and [int(x) for x in rows[2][1:]] == want[0].tolist()
    k = 0b01_00_11_10_00_01_11                      # low bits first: T C A G T A C  (11 01 00 10 11 00 01)
    assert rows[2 + k][0] == scan.kmer_base2_to_ascii(k, 7) and [int(x) for x in rows[2 + k][1:]] == want[k].tolist()
    assert sum(1 for _ in open(tmp_path / "i.csv")) == 250


def test_cli_pileup_with_kmer_histogram(fixture_bam, tmp_path):
    """reference tests/test_cli.py:47-56 (`scan X.bam -o k.csv` then `pileup -k k.csv`): the scan CSV
    feeds load_kmerhist, `experimental` adds its 13 columns to every row (cli.py:93-95)."""
    from metacov_b200 import pileup
    from metacov_b200.cli import pileup as pileup_cmd, scan as scan_cmd
    from oracle import experimental as oexp
    from helpers import assert_experimental_equal, fake_bam
    kcsv = tmp_path / "kmers.csv"
    res = CliRunner().invoke(scan_cmd, [fixture_bam, "-o", str(kcsv), "-g", "Mapped", "-g", "IsRead1"])
    assert res.exit_code == 0, res.output
    gold = load_json("fixture_experimental.json")
    fa = tmp_path / "ref.fa"
    with open(fa, "w") as fh:
        for name, seq in gold["fasta"].items():
            fh.write(">%s some description\n" % name)
            for i in range(0, len(seq), 60):
                fh.write(seq[i:i + 60] + "\n")
    out = tmp_path / "cov.csv"
    res = CliRunner().invoke(pileup_cmd, ["-b", fixture_bam, "-k", str(kcsv), "-f", str(fa), "-o", str(out)])
    assert res.exit_code == 0, res.output
    rows = list(csv.DictReader(open(out)))
    assert len(rows) == 2 and rows[0]["sacc"] == "ref1"
    keys = {"cov", "covc", "den", "denc", "cov2", "cf", "ambig", "improper", "nzef", "gc", "ecor", "wnf", "cov3"}
    assert keys | {"min", "max", "med", "std", "avg", "q23", "sum", "sacc", "start", "end"} == set(rows[0])
    # the same numbers from the oracle with the k-mer ratios the CSV yields
    with open(kcsv) as fh:
        k_cor = pileup.load_kmerhist(fh)
    assert len(k_cor) == 2 and len(k_cor[0]) > 100
    z, _ = load_soa("fixture_soa.npz")
    obam = fake_bam(z)
    for row, (ref, ln) in zip(rows, zip(obam.references, obam.lengths)):
        with np.errstate(all="ignore"):
            _, want = oexp.experimental(obam.recs, obam.references, k_cor, 7, gold["fasta"][ref], ref, 0, ln)
        got = {k: float(row[k]) for k in keys}
        assert_experimental_equal(got, {k: float(v) for k, v in want.items()}, ref)


def _numpy_runs(depth_by_contig):
    """Run-length form of per-contig depth vectors, the plain way (test oracle of mcov_depth_runs)."""
    rows = []
    for t, d in enumerate(depth_by_contig):
        if len(d) == 0:
            continue
        cut = np.flatnonzero(np.diff(d)) + 1
        st = np.concatenate(([0], cut))
        en = np.concatenate((cut, [len(d)]))
        rows += [(t, int(s), int(e), int(d[s])) for s, e in zip(st, en)]
    return rows


def test_depth_runs_match_numpy_rle():
    """mcov_depth_runs on the fixture, on a synthetic set with empty / tiny contigs, and on a scaled C2
    shard (runs crossing the 8192-slot chunks of the export kernels), against numpy on the oracle depth."""
    from metacov_b200 import CoverageEngine, synth
    cases = []
    z, fb = load_soa("fixture_soa.npz")
    cases.append((fb, z["lengths"]))
    z2, sb = load_soa("synth_small_soa.npz")
    cases.append((sb, z2["lengths"]))
    w = synth.c2(0.003)
    hb, _ = synth.generate_host(w)
    cases.append((hb, w.contig_len))
    w5 = synth.c5(0.0005)                                   # long reads: long flat runs across many chunks
    h5, _ = synth.generate_host(w5)
    cases.append((h5, w5.contig_len))
    for batch, lengths in cases:
        d, off, _ = cport.depth(batch, lengths, mode="diff")
        want = _numpy_runs([d[off[c]:off[c] + lengths[c]] for c in range(len(lengths))])
        with CoverageEngine(lengths) as eng:
            eng.compute_depth(batch)
            runs = eng.depth_runs()
            got = list(zip(runs["tid"].tolist(), runs["start"].tolist(), runs["end"].tolist(), runs["depth"].tolist()))
            assert got == want
            # a contig sub-range and the zero filter
            if len(lengths) > 1:
                sub = eng.depth_runs(1, 2)
                assert [r for r in want if r[0] == 1] == list(zip(sub["tid"].tolist(), sub["start"].tolist(),
                                                                  sub["end"].tolist(), sub["depth"].tolist()))
            nz = eng.depth_runs(skip_zero=True)
            assert len(nz) == sum(1 for r in want if r[3] != 0) and int(((nz["end"] - nz["start"]).astype(np.int64) * nz["depth"]).sum()) == int(d.astype(np.int64).sum())
            assert len(eng.depth_runs(0, 0)) == 0


def test_cli_bedgraph_and_windows(fixture_bam, tmp_path):
    """Additive outputs of `metacov pileup`: --bedgraph (runs of equal non-zero depth) and --window."""
    bg, wo, out = tmp_path / "cov.bedgraph", tmp_path / "win.csv", tmp_path / "cov.csv"
    run_pileup(["-b", fixture_bam, "-o", str(out), "-bg", str(bg), "-w", "100", "-wo", str(wo)])
    ref1 = np.load(os.path.join(os.path.dirname(__file__), "golden", "fixture_depth_ref1.npy"))
    ref2 = np.load(os.path.join(os.path.dirname(__file__), "golden", "fixture_depth_ref2.npy"))
    names = ["ref1", "ref2"]
    want = ["%s\t%d\t%d\t%d" % (names[t], s, e, d) for t, s, e, d in _numpy_runs([ref1, ref2]) if d != 0]
    assert bg.read_text().splitlines() == want
    rows = list(csv.DictReader(io.StringIO(wo.read_text())))
    exp = []
    for name, d in zip(names, (ref1, ref2)):
        for p in range(0, len(d), 100):
            exp.append({"sacc": name, "start": str(p), "end": str(min(p + 100, len(d))),
                        "avg": str(round(float(np.mean(d[p:p + 100])), 2))})
    assert rows == exp
    from metacov_b200.cli import pileup
    assert CliRunner().invoke(pileup, ["-b", fixture_bam, "-w", "100"]).exit_code != 0      # --window without --window-out
