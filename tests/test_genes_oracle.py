"""The gene rules restated in oracle/genes.py, on the CPU: the codon tables, hand-built counts on + and - genes (SNVs
synonymous, nonsynonymous, stop-gaining and multiple; substitutions N / S / M; phases 1 and 2), trailing bases, genes
without a codon, uncovered positions and N references, overlapping genes, ``alleles.derive_genes``, and the Prodigal
and GFF3 readers of ``metacov_b200.genes``."""
import math

import numpy as np
import pytest

from oracle import genes as og

COMP = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
# codons 0-6: ATG GCT TTA TGG AAA CCC GGG, then a trailing base
REF = "ATGGCTTTATGGAAACCCGGGA"
# position -> {base: count}; every other position holds its reference base 10 times
ALT = {
    0: {"A": 6, "C": 4},      # ATG / CTG: SNV N
    5: {"T": 6, "C": 4},      # GCT / GCC: SNV S (third position)
    6: {"T": 6, "C": 4},      # TTA: two SNVs, both M
    8: {"A": 6, "G": 4},
    10: {"G": 6, "A": 4},     # TGG / TAG: SNV N, a stop gain
    12: {"G": 10},            # AAA -> GAA: SUB N
    17: {"A": 10},            # CCC -> CCA: SUB S
    18: {"A": 10},            # GGG -> AGT: two SUBs, both M
    20: {"T": 10},
}
PARAMS = dict(min_coverage=5, min_freq=0.05, min_count=2)


def _counts(ref, alt):
    c = np.zeros((4, len(ref)), np.uint32)
    for p, ch in enumerate(ref):
        for b, n in alt.get(p, {ch: 10} if ch in "ACGT" else {}).items():
            c["ACGT".index(b), p] = n
    return c


def _revcomp(ref, alt):
    n = len(ref)
    rref = "".join(COMP[ch] for ch in reversed(ref))
    ralt = {n - 1 - p: {COMP[b]: v for b, v in d.items()} for p, d in alt.items()}
    return rref, ralt


def _run(ref, alt, gene_list, **kw):
    p = dict(PARAMS)
    p.update(kw)
    return og.genes([_counts(ref, alt)], [ref], gene_list, **p)


def test_codon_tables():
    aa, n3, s3 = og.codon_table()
    assert len(aa) == len(n3) == len(s3) == 64
    assert all(a + b == 9 for a, b in zip(n3, s3))

    def code(s):
        return 16 * "ACGT".index(s[0]) + 4 * "ACGT".index(s[1]) + "ACGT".index(s[2])
    for codon, want_s3 in (("ATG", 0), ("TGG", 0), ("GCT", 3), ("TTA", 2), ("TAA", 2)):
        assert s3[code(codon)] == want_s3, codon
    for codon, letter in (("ATG", "M"), ("TGG", "W"), ("TAA", "*"), ("TAG", "*"), ("TGA", "*"), ("TTT", "F"),
                          ("GGG", "G"), ("AAA", "K"), ("CCA", "P"), ("AGT", "S")):
        assert aa[code(codon)] == letter, codon
    assert sorted(set(aa)) == sorted(set(og.STANDARD_CODE))


WANT = dict(length=22, codons=7, codons_called=7, snv_n=2, snv_s=1, snv_m=2, sub_n=1, sub_s=1, sub_m=2)
# (codon_pos, ref codon, major, minor, aa_ref, aa_major, aa_minor, kind, snv_type, sub_type) at each + position
WANT_SITES = {
    0: (0, 0, "ATG", "A", "C", "M", "M", "L", 1, "N", ""),
    5: (1, 2, "GCT", "T", "C", "A", "A", "A", 1, "S", ""),
    6: (2, 0, "TTA", "T", "C", "L", "L", "L", 1, "M", ""),
    8: (2, 2, "TTA", "A", "G", "L", "L", "L", 1, "M", ""),
    10: (3, 1, "TGG", "G", "A", "W", "W", "*", 1, "N", ""),
    12: (4, 0, "AAA", "G", "", "K", "E", "", 2, "", "N"),
    17: (5, 2, "CCC", "A", "", "P", "P", "", 2, "", "S"),
    18: (6, 0, "GGG", "A", "", "G", "R", "", 2, "", "M"),
    20: (6, 2, "GGG", "T", "", "G", "G", "", 2, "", "M"),
}


def _n3(codons):
    aa, n3, _ = og.codon_table()
    return sum(n3[16 * "ACGT".index(c[0]) + 4 * "ACGT".index(c[1]) + "ACGT".index(c[2])] for c in codons)


def test_plus_gene_known_answers():
    recs, sites = _run(REF, ALT, [(0, 0, 22, 1, 0)])
    r = recs[0]
    for k, v in WANT.items():
        assert r[k] == v, k
    n3 = _n3(["ATG", "GCT", "TTA", "TGG", "AAA", "CCC", "GGG"])
    assert (r["n_sites3"], r["s_sites3"]) == (n3, 63 - n3)
    assert [s[2] for s in sites] == sorted(WANT_SITES)
    for s in sites:
        assert s[:2] == (0, 0)
        assert s[3:] == WANT_SITES[s[2]], s


def test_minus_gene_is_the_mirror():
    """The reverse complement of the contig on the - strand: the same records, codons and amino acids; positions
    mirrored, alleles complemented, in ascending position order."""
    rref, ralt = _revcomp(REF, ALT)
    # the - gene reads from its end: [0, 22) would read the trailing base first; [1, 23) of a contig with one more base
    recs, sites = _run("C" + rref, {p + 1: d for p, d in ralt.items()}, [(0, 1, 23, -1, 0)])
    assert recs[0] == dict(_run(REF, ALT, [(0, 0, 22, 1, 0)])[0][0])
    want = sorted((22 - p, v) for p, v in WANT_SITES.items())
    assert [s[2] for s in sites] == [p for p, _ in want]
    for s, (p, v) in zip(sites, want):
        codon, cpos, rc, ma, mi, ar, am, an, kind, st, bt = v
        assert s[3:] == (codon, cpos, rc, COMP[ma], COMP[mi] if mi else "", ar, am, an, kind, st, bt), s


@pytest.mark.parametrize("phase", [1, 2])
def test_phase(phase):
    base, _ = _run(REF, ALT, [(0, 0, 22, 1, 0)])
    pad = "CA"[:phase]
    recs, sites = _run(pad + REF, {p + phase: d for p, d in ALT.items()}, [(0, 0, 22 + phase, 1, phase)])
    assert {k: v for k, v in recs[0].items() if k != "length"} == {k: v for k, v in base[0].items() if k != "length"}
    assert [s[2] - phase for s in sites] == sorted(WANT_SITES)
    rref, ralt = _revcomp(REF, ALT)
    recs, sites = _run("C" + rref + pad, {p + 1: d for p, d in ralt.items()}, [(0, 1, 23 + phase, -1, phase)])
    assert {k: v for k, v in recs[0].items() if k != "length"} == {k: v for k, v in base[0].items() if k != "length"}
    assert [s[2] for s in sites] == sorted(22 - p for p in WANT_SITES)


def test_trailing_bases_and_genes_without_codons():
    recs, _ = _run(REF, ALT, [(0, 0, 21, 1, 0), (0, 0, 22, 1, 0), (0, 0, 2, 1, 0), (0, 0, 4, 1, 2), (0, 20, 22, -1, 0)])
    assert recs[0]["codons"] == recs[1]["codons"] == 7
    assert {k: v for k, v in recs[0].items() if k != "length"} == {k: v for k, v in recs[1].items() if k != "length"}
    for r, length in zip(recs[2:], (2, 4, 2)):
        assert r == dict(dict.fromkeys(og.RECORD_FIELDS, 0), length=length)


def test_uncovered_position_and_unknown_reference_drop_their_codon():
    alt = dict(ALT)
    alt[13] = {"A": 2}                                     # under min_coverage: codon 4 (SUB N) is not called
    ref = REF[:16] + "N" + REF[17:]                        # codon 5 (SUB S) has an unknown reference base
    recs, sites = _run(ref, alt, [(0, 0, 22, 1, 0)])
    r = recs[0]
    assert r["codons_called"] == 5 and r["sub_n"] == 0 and r["sub_s"] == 0 and r["sub_m"] == 2
    n3 = _n3(["ATG", "GCT", "TTA", "TGG", "GGG"])
    assert (r["n_sites3"], r["s_sites3"]) == (n3, 45 - n3)
    assert [s[2] for s in sites] == [0, 5, 6, 8, 10, 18, 20]


def test_overlapping_genes_list_a_position_once_each():
    gl = [(0, 0, 22, 1, 0), (0, 3, 12, 1, 0), (0, 0, 22, 1, 0)]
    recs, sites = _run(REF, ALT, gl)
    assert recs[0] == recs[2]
    assert recs[1]["codons"] == 3 and (recs[1]["snv_s"], recs[1]["snv_m"], recs[1]["snv_n"]) == (1, 2, 1)
    assert [(s[0], s[2]) for s in sites] == ([(0, p) for p in sorted(WANT_SITES)] + [(1, p) for p in (5, 6, 8, 10)]
                                             + [(2, p) for p in sorted(WANT_SITES)])
    assert [s[3] for s in sites if s[0] == 1] == [0, 1, 1, 2]


def test_bad_genes():
    for g in [(0, 0, 23, 1, 0), (0, -1, 10, 1, 0), (0, 5, 5, 1, 0), (1, 0, 3, 1, 0), (0, 0, 9, 0, 0), (0, 0, 9, 1, 3)]:
        with pytest.raises(ValueError):
            _run(REF, ALT, [g])
    with pytest.raises(ValueError):
        og.genes([_counts(REF, ALT)], None, [(0, 0, 9, 1, 0)])


def test_derive_genes():
    from metacov_b200 import _capi
    from metacov_b200.alleles import derive_genes
    rec = np.zeros(4, _capi.GENE_STATS_DTYPE)
    rec["n_sites3"] = [21, 0, 21, 27]
    rec["s_sites3"] = [6, 9, 0, 0]
    rec["snv_n"] = [7, 3, 1, 0]
    rec["snv_s"] = [1, 0, 2, 0]
    rec["sub_n"] = [14, 0, 0, 9]
    rec["sub_s"] = [0, 2, 0, 0]
    d = derive_genes(rec)
    assert list(d) == ["N_sites", "S_sites", "pN", "pS", "pn_ps", "dN", "dS", "dn_ds"]
    assert d["N_sites"].tolist() == [7.0, 0.0, 7.0, 9.0] and d["S_sites"].tolist() == [2.0, 3.0, 0.0, 0.0]
    assert d["pN"][0] == 1.0 and d["pS"][0] == 0.5 and d["pn_ps"][0] == 2.0
    assert d["dN"][0] == 2.0 and d["dS"][0] == 0.0 and math.isnan(d["dn_ds"][0])      # dS = 0
    assert math.isnan(d["pN"][1]) and math.isnan(d["pn_ps"][1]) and d["pS"][1] == 0.0    # N_sites = 0
    assert math.isnan(d["pS"][2]) and math.isnan(d["pn_ps"][2]) and math.isnan(d["dS"][2])   # S_sites = 0
    assert d["dN"][3] == 1.0 and math.isnan(d["dn_ds"][3])


def test_read_prodigal(tmp_path):
    from metacov_b200.genes import read_genes
    p = tmp_path / "genes.fna"
    p.write_text(">ctg_a_1 # 3 # 101 # 1 # ID=1_1;partial=00;start_type=ATG\nATGAAA\nTAA\n"
                 ">ctg_a_12 # 200 # 499 # -1 # ID=1_12;partial=00\nATG\n"
                 ">k141_7_3 # 1 # 30 # 1 # ID=2_3\nATG\n")
    t = read_genes(str(p))
    assert t.name == ["ctg_a_1", "ctg_a_12", "k141_7_3"] and t.contig == ["ctg_a", "ctg_a", "k141_7"]
    assert t.start.tolist() == [2, 199, 0] and t.end.tolist() == [101, 499, 30]
    assert t.strand.tolist() == [1, -1, 1] and t.phase.tolist() == [0, 0, 0]
    for bad in (">ctg_1 # 3 # 101\n", ">ctg # 3 # 101 # 1 # x\n", ">ctg_1 # three # 101 # 1 # x\n",
                ">ctg_1 # 3 # 101 # + # x\n", ">ctg_1 # 0 # 101 # 1 # x\n", ">ctg_1 # 30 # 10 # 1 # x\n"):
        p.write_text(">ok_1 # 1 # 3 # 1 # x\nATG\n" + bad)
        with pytest.raises(ValueError, match=r"genes.fna:3"):
            read_genes(str(p))


def test_read_gff3(tmp_path):
    from metacov_b200.genes import read_genes
    p = tmp_path / "genes.gff"
    lines = ["##gff-version 3", "# a comment",
             "c1\tProdigal\tgene\t1\t90\t.\t+\t.\tID=g1",
             "c1\tProdigal\tCDS\t1\t90\t.\t+\t0\tID=cds1;Parent=g1",
             "c2 desc\tx\tCDS\t10\t300\t12.5\t-\t2\tName=foo",
             "c1\tx\tmRNA\t5\t50\t.\t+\t.\tID=m1",
             "c1\tx\tCDS\t100\t200\t.\t-\t1\tID=cds3",
             "##FASTA", ">c1", "ACGT"]
    p.write_text("\n".join(lines) + "\n")
    t = read_genes(str(p))
    assert t.name == ["cds1", "c2 desc:10-300", "cds3"] and t.contig == ["c1", "c2 desc", "c1"]
    assert t.start.tolist() == [0, 9, 99] and t.end.tolist() == [90, 300, 200]
    assert t.strand.tolist() == [1, -1, -1] and t.phase.tolist() == [0, 2, 1]
    for bad in ("c1\tx\tCDS\t1\t90\t.\t+\t0", "c1\tx\tCDS\tone\t90\t.\t+\t0\tID=a", "c1\tx\tCDS\t1\t90\t.\t.\t0\tID=a",
                "c1\tx\tCDS\t1\t90\t.\t+\t.\tID=a", "c1\tx\tCDS\t0\t90\t.\t+\t0\tID=a", "c1\tx\tCDS\t9\t8\t.\t+\t0\tID=a"):
        p.write_text("##gff-version 3\nc1\tx\tCDS\t1\t3\t.\t+\t0\tID=ok\n" + bad + "\n")
        with pytest.raises(ValueError, match=r"genes.gff:3"):
            read_genes(str(p))
