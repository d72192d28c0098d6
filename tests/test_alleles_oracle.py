"""The allele rules of oracle/alleles.py against cases worked out by hand, ``alleles.derive`` and the argument errors of
``metacov alleles`` that are raised before any GPU work (no GPU needed)."""
import math
import os

import numpy as np
import pytest

from oracle import alleles as oa


def one(a, c, g, t, ref=None, **kw):
    """The rules at one position: (covered, present mask, consensus letter, pi, kind)."""
    e = oa.evaluate(np.array([[a], [c], [g], [t]], np.uint32), ref, **kw)
    mask = sum(1 << b for b in range(4) if e["present"][b, 0])
    return bool(e["covered"][0]), mask, "ACGT"[int(e["consensus"][0])], float(e["pi"][0]), int(e["kind"][0])


def test_consensus_ties_go_to_the_first_of_acgt():
    assert one(3, 3, 0, 0)[2] == "A"
    assert one(0, 2, 2, 2)[2] == "C"
    assert one(0, 0, 4, 4)[2] == "G"
    assert one(0, 0, 1, 9)[2] == "T"
    # a tie with the reference: the consensus is the earlier letter, so SUB depends on which one the reference is
    assert one(0, 3, 3, 0, "c")[4] & oa.SUB == 0
    assert one(0, 3, 3, 0, "G")[4] & oa.SUB != 0


def test_min_freq_boundary_at_equality():
    # 0.05 * 20.0 rounds to exactly 1.0 in float64: n_b = 1 is present
    assert 0.05 * 20.0 == 1.0
    assert one(19, 1, 0, 0, min_count=1, min_freq=0.05)[1] == 0b11
    assert one(19, 1, 0, 0, min_count=1, min_freq=0.05)[4] == oa.SNV
    assert one(19, 1, 0, 0, min_count=1, min_freq=0.0500001)[1] == 0b01
    assert one(0, 0, 0, 5, min_count=1, min_freq=1.0)[1] == 0b1000
    assert one(0, 0, 1, 4, min_count=1, min_freq=0.0)[1] == 0b1100


def test_min_coverage_edge():
    cov, mask, _c, pi, kind = one(2, 2, 0, 0, min_coverage=5, min_count=1)
    assert (cov, pi, kind) == (False, 0.0, 0)                 # N = min_coverage - 1: nothing is defined there
    cov, mask, _c, pi, kind = one(3, 2, 0, 0, min_coverage=5, min_count=1)
    assert cov and kind == oa.SNV and pi == 1.0 - ((0.6 * 0.6 + 0.4 * 0.4) + (0.0 + 0.0))


def test_min_count_against_min_freq():
    # min_freq alone would admit C (2 / 5 = 0.4), min_count = 3 does not
    assert one(3, 2, 0, 0, min_count=3)[1] == 0b01
    # min_count alone would admit C (2 >= 2), min_freq does not (2 < 0.05 * 100)
    assert one(98, 2, 0, 0, min_count=2)[1] == 0b01
    assert one(95, 5, 0, 0, min_count=2)[1] == 0b11


def test_reference_bases():
    counts = np.array([[0] * 7, [0] * 7, [0] * 7, [10] * 7], np.uint32)      # consensus T everywhere, only T present
    e = oa.evaluate(counts, "acgtNRy")
    assert e["ref"].tolist() == [0, 1, 2, 3, 4, 4, 4]
    assert e["kind"].tolist() == [oa.SUB | oa.POPSUB] * 3 + [0, 0, 0, 0]
    assert oa.ref_codes(b"AcGtn-*", 7).tolist() == [0, 1, 2, 3, 4, 4, 4]


def test_no_reference_gives_snv_only():
    rng = np.random.default_rng(1)
    counts = rng.integers(0, 12, (4, 5000)).astype(np.uint32)
    e = oa.evaluate(counts, None)
    assert set(np.unique(e["kind"]).tolist()) == {0, oa.SNV}
    assert (e["ref"] == 4).all()


def test_pi_values():
    assert one(5, 5, 0, 0)[3] == 0.5
    assert one(10, 0, 0, 0)[3] == 0.0
    assert one(0, 0, 0, 7)[3] == 0.0
    assert one(5, 5, 5, 5)[3] == 0.75


def test_popsub_needs_a_present_allele():
    # consensus = reference (A wins the tie), no allele reaches min_count: the reference is not present, but neither is
    # anything else, so the position is neither SUB nor POPSUB
    cov, mask, cons, _pi, kind = one(1, 1, 1, 1, "A", min_coverage=4, min_count=2)
    assert cov and mask == 0 and cons == "A" and kind == 0
    # with the reference allele short of min_count and another present, POPSUB comes with SUB
    assert one(1, 4, 0, 0, "A", min_count=2)[4] == oa.SUB | oa.POPSUB
    # and the present allele being the reference: neither
    assert one(1, 4, 0, 0, "C", min_count=2)[4] == 0


def test_popsub_implies_sub():
    """Under these rules a reference that is not present while another allele is has a smaller count than it."""
    rng = np.random.default_rng(2)
    counts = rng.integers(0, 9, (4, 20000)).astype(np.uint32)
    ref = "".join("ACGTN"[k] for k in rng.integers(0, 5, 20000))
    for kw in (dict(), dict(min_count=1, min_freq=0.3), dict(min_coverage=1, min_count=3, min_freq=0.0)):
        k = oa.evaluate(counts, ref, **kw)["kind"]
        assert ((k & oa.POPSUB) != 0).sum() > 100
        assert (k[(k & oa.POPSUB) != 0] & oa.SUB).all()


def test_parameters_checked():
    for kw in (dict(min_coverage=0), dict(min_count=0), dict(min_freq=-0.1), dict(min_freq=1.5), dict(min_freq=float("nan"))):
        with pytest.raises(ValueError):
            oa.evaluate(np.zeros((4, 1), np.uint32), None, **kw)


def test_region_stats():
    counts = np.array([[10, 5, 0, 1, 0], [0, 5, 0, 1, 0], [0, 0, 0, 1, 0], [0, 0, 9, 2, 0]], np.uint32)
    r = oa.region_stats(counts, "AAGTN", 0, 8)
    # positions past the contig end (5, 6, 7) add to the length only
    assert r == dict(length=8, covered=4, depth_sum=34, pi_sum=math.fsum([0.0, 0.5, 0.0, 1.0 - ((0.2 * 0.2 + 0.2 * 0.2) + (0.2 * 0.2 + 0.4 * 0.4))]),
                     snv=1, ref_covered=4, sub=1, popsub=1)
    assert oa.region_stats(counts, None, 2, 2)["length"] == 0
    assert oa.region_stats(counts, None, 1, 3)["ref_covered"] == 0


def test_derive_divisions_by_zero_give_nan():
    from metacov_b200._capi import ALLELE_STATS_DTYPE
    from metacov_b200.alleles import DERIVED, derive
    s = np.zeros(3, ALLELE_STATS_DTYPE)
    s[0] = (1000, 800, 24000, 8.0, 4, 600, 6, 3)
    s[1] = (100, 0, 0, 0.0, 0, 0, 0, 0)
    d = derive(s)
    assert sorted(d) == sorted(DERIVED)
    assert d["breadth"][0] == 0.8 and d["depth"][0] == 24.0 and d["pi"][0] == 0.01
    assert d["snv_per_kbp"][0] == 5.0
    assert d["con_ani"][0] == pytest.approx(0.99, abs=1e-15) and d["pop_ani"][0] == pytest.approx(0.995, abs=1e-15)
    assert d["breadth"][1] == 0.0 and d["depth"][1] == 0.0
    for k in ("pi", "snv_per_kbp", "con_ani", "pop_ani"):
        assert np.isnan(d[k][1]), k
    assert all(np.isnan(d[k][2]) for k in DERIVED)
    one_rec = derive(s[0])
    assert float(one_rec["breadth"]) == 0.8


def test_cli_argument_errors(tmp_path):
    from click.testing import CliRunner
    from metacov_b200.cli import main
    bam = tmp_path / "x.bam"
    bam.write_bytes(b"not read")
    run = CliRunner().invoke
    r = run(main, ["alleles", "-b", "-"], input=b"@HD\tVN:1.6\n")
    assert r.exit_code == 2 and "piped stream" in r.output
    fifo = str(tmp_path / "fifo")
    os.mkfifo(fifo)
    r = run(main, ["alleles", "-b", fifo])
    assert r.exit_code == 2 and "piped stream" in r.output
    for bad in (["--min-coverage", "0"], ["--min-count", "0"], ["--min-freq", "1.5"], ["--min-freq", "-0.1"],
                ["--read-callback", "mapped"], ["--bam-decode", "cpu"]):
        r = run(main, ["alleles", "-b", str(bam)] + bad)
        assert r.exit_code == 2, (bad, r.output)
    rb, rc = tmp_path / "r.blast7", tmp_path / "r.csv"
    rb.write_text("# BLAST\n")
    rc.write_text("sacc,start,end\n")
    r = run(main, ["alleles", "-b", str(bam), "-rb", str(rb), "-rc", str(rc)])
    assert r.exit_code == 2 and "Only one of" in r.output
    r = run(main, ["alleles", "-b", str(bam), "-f", str(tmp_path / "missing.fa")])
    assert r.exit_code == 2
