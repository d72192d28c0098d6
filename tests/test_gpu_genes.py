"""Genes on the GPU (csrc/genes.cu) against oracle/genes.py: seeded two-strain reads over a reference with fixed
differences and N bases, genes on both strands in every phase (one ending at its contig's end, overlapping ones, some
without a codon); invariance over decoders; what the call leaves alone; the errors; a contig across slot 2^31; and
``metacov genes``."""
import ctypes as C
import csv
import io
import math

import numpy as np
import pytest

from oracle import basecount
from oracle import genes as og
from test_gpu_basecount import LENS, REFS, _columns, _write

pytestmark = pytest.mark.gpu

PARAMS = dict(min_coverage=5, min_freq=0.05, min_count=2)
INT_FIELDS = og.RECORD_FIELDS


def _two_strain(seed, lens, coverage=24, read_len=100, var=0.08, minor=0.35, err=0.01):
    """(records of test_gpu_basecount's form, the strain-a bases per contig, the reference FASTA per contig): strain b
    differs from strain a at a fraction ``var`` of positions and is carried by ``minor`` of the reads; the FASTA differs
    from strain a at 2 % of positions (substitutions) and has 0.5 % N."""
    rng = np.random.default_rng(seed)
    recs, strain_a, fasta = [], [], []
    for t, n in enumerate(lens):
        a = rng.integers(0, 4, n)
        b = a.copy()
        v = rng.random(n) < var
        b[v] = (b[v] + rng.integers(1, 4, int(v.sum()))) % 4
        f = np.array(list("ACGT"))[a]
        s = rng.random(n) < 0.02
        f[s] = np.array(list("ACGT"))[(a[s] + rng.integers(1, 4, int(s.sum()))) % 4]
        f[rng.random(n) < 0.005] = "N"
        strain_a.append(a)
        fasta.append("".join(f.tolist()))
        for _ in range(int(n * coverage / read_len)):
            p = int(rng.integers(0, n - read_len + 1))
            src = b if rng.random() < minor else a
            bases = src[p:p + read_len].copy()
            e = rng.random(read_len) < err
            bases[e] = (bases[e] + rng.integers(1, 4, int(e.sum()))) % 4
            flag = int(rng.choice([0, 16, 0, 16, 0x400, 0x100]))
            qual = None if rng.random() < 0.1 else [int(q) for q in rng.integers(2, 41, read_len)]
            recs.append((t, p, flag, [(read_len << 4) | 0], "".join("ACGT"[k] for k in bases), qual))
    recs.sort(key=lambda r: (r[0], r[1]))
    return recs, strain_a, fasta


def _gene_list(lens, seed):
    """Genes tiling about 88 % of each contig on both strands in every phase, one ending at each contig's end,
    overlapping genes and genes without a codon."""
    rng = np.random.default_rng(seed)
    out = []
    for t, n in enumerate(lens):
        p = 0
        while p < n:
            ln = int(rng.integers(150, 1200))
            if p + ln > n:
                ln = n - p
            if rng.random() < 0.88 and ln > 0:
                out.append((t, p, p + ln, int(rng.choice([1, -1])), int(rng.integers(0, 3))))
            p += ln + int(rng.integers(0, 60))
        out.append((t, n - 301, n, -1, 1))                           # ending at the contig's end
        out.append((t, n - 300, n, 1, 0))
        out.append((t, 10, 12, 1, 0))                                 # shorter than a codon
        out.append((t, 10, 14, -1, 2))
        if n > 2000:
            out.append((t, 400, 1400, 1, 2))                          # overlapping the tiles
            out.append((t, 400, 1400, 1, 2))
    return out


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("genes")
    recs, _a, fasta = _two_strain(41, LENS)
    pb, ps = _write(recs, d, "genes")
    fa = str(d / "ref.fa")
    with open(fa, "w") as fh:
        for n, s in zip(REFS, fasta):
            fh.write(">%s description\n" % n)
            for a in range(0, len(s), 70):
                fh.write(s[a:a + 70] + "\n")
    return dict(recs=recs, bam=pb, sam=ps, fasta=fa, seqs=fasta, genes=_gene_list(LENS, 42), dir=d)


def _table(gene_list):
    from metacov_b200.genes import GeneTable
    return GeneTable(["g%d" % k for k in range(len(gene_list))], [REFS[g[0]] for g in gene_list],
                     *[np.array([g[i] for g in gene_list], np.int64) for i in range(1, 5)])


_ORACLE = {}


def _oracle(f, t, cb, **params):
    key = (t, cb, tuple(sorted(params.items())))
    if key not in _ORACLE:
        tid, pos, flag, _mapq, cig_off, cig, nt16, quals = _columns(f["recs"])
        counts = basecount.full_counts(LENS, tid, pos, flag, cig_off, cig, nt16, quals, t, cb)
        _ORACLE[key] = og.genes(counts, f["seqs"], f["genes"], **(params or PARAMS))
    return _ORACLE[key]


def _site_rows(sites):
    cols = [sites[k].tolist() for k in ("gene", "tid", "pos", "codon", "codon_pos")]
    let = [[x.decode() for x in sites[k].tolist()] for k in ("ref_codon", "major", "minor", "aa_ref", "aa_major",
                                                                "aa_minor")]
    return [tuple(a) + tuple(b) + (k, st.decode(), bt.decode()) for a, b, k, st, bt in
            zip(zip(*cols), zip(*let), sites["kind"].tolist(), sites["snv_type"].tolist(), sites["sub_type"].tolist())]


def _check(records, sites, want):
    recs, want_sites = want
    assert len(records) == len(recs)
    for k, r in enumerate(recs):
        assert {f: int(records[f][k]) for f in INT_FIELDS} == r, k
    assert int(records["pad"].max(initial=0)) == 0
    assert _site_rows(sites) == want_sites


@pytest.mark.parametrize("fmt", ["bam", "sam"])
@pytest.mark.parametrize("cb", ["all", "nofilter"])
@pytest.mark.parametrize("t", [0, 15])
def test_matches_oracle(files, fmt, cb, t):
    from metacov_b200 import AlignmentFile, FastaFile
    want = _oracle(files, t, cb)
    with AlignmentFile(files[fmt], decode="gpu") as af:
        records, stats, sites = af.gene_stats(_table(files["genes"]), FastaFile(files["fasta"]), quality_threshold=t,
                                              read_callback=cb, sites=True, **PARAMS)
        _check(records, sites, want)
        g = files["genes"]
        st = af.allele_stats([REFS[x[0]] for x in g], [x[1] for x in g], [x[2] for x in g],
                             fasta=FastaFile(files["fasta"]), quality_threshold=t, read_callback=cb, **PARAMS)
        assert stats.tobytes() == st.tobytes()
        again, _stats, none = af.gene_stats(_table(g), FastaFile(files["fasta"]), quality_threshold=t, read_callback=cb,
                                            **PARAMS)
        assert none is None and again.tobytes() == records.tobytes()
    long_genes = records["length"] >= 600
    for f in ("snv_n", "snv_s", "snv_m", "sub_n", "sub_s"):
        assert (records[f][long_genes] > 0).mean() > 0.8, f
    assert records["sub_m"].sum() > 0 and len(sites) > 2000
    ends = [k for k, x in enumerate(files["genes"]) if x[2] == LENS[x[0]]]
    assert len(ends) >= 6 and all(records["codons_called"][k] > 0 for k in ends)
    assert (records["codons_called"] < records["codons"]).any()          # N bases and uncovered positions drop codons


def test_other_parameters(files):
    from metacov_b200 import AlignmentFile, FastaFile
    params = dict(min_coverage=3, min_freq=0.2, min_count=3)
    with AlignmentFile(files["bam"], decode="gpu") as af:
        records, _stats, sites = af.gene_stats(_table(files["genes"]), FastaFile(files["fasta"]), quality_threshold=15,
                                               sites=True, **params)
    _check(records, sites, _oracle(files, 15, "all", **params))


def test_identical_across_decoders(files):
    from metacov_b200 import AlignmentFile, FastaFile
    runs = {}
    for decode, kw in (("gpu", {}), ("gpu-stream", {"gpu_chunk_bytes": 1 << 17}), ("host", {})):
        with AlignmentFile(files["bam"], decode=decode, **kw) as af:
            r, s, sites = af.gene_stats(_table(files["genes"]), FastaFile(files["fasta"]), sites=True)
            runs[decode] = (r.tobytes(), s.tobytes(), sites.tobytes())
    assert runs["gpu"] == runs["gpu-stream"] == runs["host"]


def test_depth_counts_and_lists_left_alone(files):
    from metacov_b200 import AlignmentFile, FastaFile, _capi
    from metacov_b200._capi import lib
    fa = FastaFile(files["fasta"])
    with AlignmentFile(files["bam"], decode="gpu") as af:
        eng = af.coverage_engine()
        ceng = af._count_engine()
        tid = np.arange(3, dtype=np.int32)
        sites0 = af.allele_sites(fasta=fa, min_count=1)
        import torch
        sig = [ceng.allele_signature()]
        sig.append(sig[0].clone())
        every = sig[1][::97]                                   # another consensus at some covered slots
        sig[1][::97] = torch.where(every >= 0x80, every ^ 0x10, every)
        cmp0 = ceng.compare_sites(sig, [[0, 1]])
        link0, _info = af.linkage(min_reads=2)
        lists = ((lib.mcov_allele_sites_read, sites0), (lib.mcov_compare_sites_read, cmp0), (lib.mcov_linkage_read, link0))
        assert len(sites0) and len(cmp0) and len(link0)

        def snap():
            out = [af.count_coverage_depth(c).tobytes() for c in REFS]
            out.append(eng.region_stats(tid, np.zeros_like(tid), np.array(LENS, np.int32)).tobytes())
            out.append(eng.pass_info())
            out += [np.stack(af.count_coverage(c)).tobytes() for c in REFS]
            for read, ref in lists:
                got = np.zeros_like(ref)
                ceng._check(read(ceng._ctx, 0, len(ref), _capi.ptr(got)))
                out.append(got.tobytes())
            return out
        s0 = snap()
        af.gene_stats(_table(files["genes"]), fa, sites=True)
        af.gene_stats(_table(files["genes"][:5]), fa, min_coverage=1, min_count=1, min_freq=0.0, sites=True)
        assert snap() == s0
        assert af.allele_sites(fasta=fa, min_count=1).tobytes() == sites0.tobytes()


def test_errors(files, tmp_path, monkeypatch):
    from metacov_b200 import AlignmentFile, CoverageEngine, FastaFile, McovError, _capi
    from metacov_b200._capi import lib
    fa = FastaFile(files["fasta"])
    good = _table(files["genes"])
    with AlignmentFile(io.BytesIO(open(files["sam"], "rb").read())) as s:
        with pytest.raises(ValueError, match="read once"):
            s.gene_stats(good, fa)
    with AlignmentFile(files["bam"], decode="gpu") as af:
        eng = af._count_engine()
        with pytest.raises(KeyError):
            af.gene_stats(_table([(0, 0, 30, 1, 0)])._replace(contig=["nope"]), fa)
        n = eng.launch_count()
        for bad in ([(0, 0, LENS[0] + 1, 1, 0)], [(0, 5, 5, 1, 0)], [(0, -1, 30, 1, 0)], [(0, 0, 30, 0, 0)],
                    [(0, 0, 30, 1, 3)]):
            with pytest.raises(ValueError):
                af.gene_stats(_table(bad), fa)
        for bad in (dict(min_coverage=0), dict(min_count=0), dict(min_freq=1.5), dict(read_callback="mapped")):
            with pytest.raises(ValueError):
                af.gene_stats(good, fa, **bad)
        with pytest.raises(ValueError):
            af.gene_stats(good, None)
        assert eng.launch_count() == n                                    # nothing ran
        want, _stats, want_sites = af.gene_stats(good, fa, sites=True)
        # the C level: MCOV_ERR_ARG for bad genes and parameters, the context usable afterwards
        p = eng._allele_params(5, 0.05, 2, True)
        out = np.zeros(1, _capi.GENE_STATS_DTYPE)
        cnt = C.c_int64(0)

        def run(gene, params=p):
            cols = [np.array([x], np.int32) for x in gene]
            return lib.mcov_gene_run(eng._ctx, 1, *[_capi.ptr(x) for x in cols], C.byref(params), _capi.ptr(out),
                                     C.byref(cnt))
        for gene in ((3, 0, 30, 1, 0), (0, -1, 30, 1, 0), (0, 30, 30, 1, 0), (0, 0, LENS[0] + 1, 1, 0),
                     (0, 0, 30, 2, 0), (0, 0, 30, -1, -1), (0, 0, 30, 1, 3)):
            assert run(gene) == _capi.MCOV_ERR_ARG, gene
        for field, v in (("use_reference", 0), ("min_coverage", 0), ("min_count", 0), ("min_freq", 1.5)):
            q = eng._allele_params(5, 0.05, 2, True)
            setattr(q, field, v)
            assert run((0, 0, 30, 1, 0), q) == _capi.MCOV_ERR_ARG
        rec = np.zeros(1, _capi.GENE_SITE_DTYPE)
        assert lib.mcov_gene_sites_read(eng._ctx, 0, 1, _capi.ptr(rec)) == _capi.MCOV_ERR_STATE   # (dropped)
        assert run((0, LENS[0] - 3, LENS[0], -1, 0)) == _capi.MCOV_OK                           # the contig's end
        r, _s, sites = af.gene_stats(good, fa, sites=True)
        assert r.tobytes() == want.tobytes() and sites.tobytes() == want_sites.tobytes()
        assert lib.mcov_gene_sites_read(eng._ctx, len(sites), 1, _capi.ptr(rec)) == _capi.MCOV_ERR_ARG
        # records without a list keep the last list readable
        eng.gene_stats([0], [0], [30], [1], [0])
        got = np.zeros(len(sites), _capi.GENE_SITE_DTYPE)
        eng._check(lib.mcov_gene_sites_read(eng._ctx, 0, len(sites), _capi.ptr(got)))
        assert got.tobytes() == sites.tobytes()
    # the list does not fit: MemoryError naming the file and the byte counts, then a good call
    with AlignmentFile(files["bam"], decode="gpu") as af:
        monkeypatch.setenv("MCOV_GENE_FREE_BYTES", "1000")
        with pytest.raises(MemoryError, match=r"genes.bam.*needs? \d+ bytes of device memory, \d+ are free"):
            af.gene_stats(good, fa, sites=True)
        monkeypatch.delenv("MCOV_GENE_FREE_BYTES")
        r, _s, sites = af.gene_stats(good, fa, sites=True)
        assert r.tobytes() == want.tobytes() and sites.tobytes() == want_sites.tobytes()
    # without counts, and without a reference: MCOV_ERR_STATE
    with CoverageEngine(LENS) as eng:
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng.gene_stats([0], [0], [30], [1], [0])
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng._check(lib.mcov_gene_sites_read(eng._ctx, 0, 0, None))
    with AlignmentFile(files["bam"], decode="gpu") as af:
        eng = af._count_engine()
        af.count_coverage("c0")
        eng.set_reference(0, files["seqs"][0])
        with pytest.raises(McovError, match="contig 1 has no reference"):
            eng.gene_stats([0], [0], [30], [1], [0])


def test_cli(files, tmp_path):
    from click.testing import CliRunner
    from metacov_b200 import AlignmentFile, FastaFile
    from metacov_b200.alleles import derive, derive_genes
    from metacov_b200.cli import main
    gl = files["genes"][:40]
    gff = tmp_path / "genes.gff"
    with open(gff, "w") as fh:
        fh.write("##gff-version 3\n")
        for k, (t, a, b, s, ph) in enumerate(gl):
            if b - a >= 1:
                fh.write("%s\tsim\tCDS\t%d\t%d\t.\t%s\t%d\tID=g%d\n" % (REFS[t], a + 1, b, "+" if s > 0 else "-", ph, k))
            fh.write("%s\tsim\tgene\t%d\t%d\t.\t+\t.\tID=x%d\n" % (REFS[t], a + 1, b, k))
    out, sites_out = tmp_path / "g.csv", tmp_path / "s.tsv"
    r = CliRunner().invoke(main, ["genes", "-b", files["bam"], "-f", files["fasta"], "-g", str(gff), "-o", str(out),
                                  "--sites-out", str(sites_out), "-q", "0"], catch_exceptions=False)
    assert r.exit_code == 0, r.output
    with AlignmentFile(files["bam"], decode="gpu") as af:
        records, stats, sites = af.gene_stats(_table(gl), FastaFile(files["fasta"]), quality_threshold=0, sites=True)
    rows = list(csv.DictReader(open(out)))
    ints = [f for f in INT_FIELDS]
    d, dg = derive(stats), derive_genes(records)
    assert list(rows[0]) == ["name", "contig", "start", "end", "strand"] + ints + sorted(d) + list(dg)
    assert len(rows) == len(gl)
    for k, row in enumerate(rows):
        t, a, b, s, _ph = gl[k]
        assert [row["name"], row["contig"], row["start"], row["end"], row["strand"]] == \
            ["g%d" % k, REFS[t], str(a), str(b), "+" if s > 0 else "-"]
        assert [int(row[f]) for f in ints] == [int(records[f][k]) for f in ints]
        for name, v in list(d.items()) + list(dg.items()):
            x = float(row[name])
            assert (math.isnan(x) and math.isnan(v[k])) or x == float(v[k]), (name, row)
    lines = open(sites_out).read().splitlines()
    assert lines[0].split("\t") == ["gene", "contig", "pos", "codon", "codon_pos", "ref_codon", "major", "minor",
                                    "aa_ref", "aa_major", "aa_minor", "snv", "sub", "snv_type", "sub_type"]
    assert len(lines) - 1 == len(sites) > 100
    for line, row in zip(lines[1:], _site_rows(sites)):
        g, t, p, c, cp, rc, ma, mi, ar, am, an, k, st, bt = row
        assert line.split("\t") == ["g%d" % g, REFS[t], str(p), str(c), str(cp), rc, ma, mi or ".", ar, am, an or ".",
                                    str(k & 1), str(k >> 1), st or ".", bt or "."]
    r = CliRunner().invoke(main, ["genes", "-b", "-", "-f", files["fasta"], "-g", str(gff), "-o", str(out)],
                           input=open(files["sam"]).read())
    assert r.exit_code != 0 and "piped stream" in r.output


def test_contig_across_slot_2_31(tmp_path):
    """A contig of 2.14 x 10^9 and one of 2 x 10^7 that crosses slot 2^31: genes around that slot and at the second
    contig's end against the oracle on the counts of their windows (34 GB of counters)."""
    import samio
    from metacov_b200 import AlignmentFile
    L0, L1 = 2_140_000_000, 20_000_000
    refs, lens = ["big0", "big1"], [L0, L1]
    off1 = (L0 + 1 + 3) & ~3
    px = (1 << 31) - off1                                     # position of contig 1 at slot 2^31
    windows = [(px - 3000, px + 3000), (L1 - 3000, L1)]
    rng = np.random.default_rng(43)
    letters = np.frombuffer(b"ACGT", np.uint8)
    fasta1 = letters[rng.integers(0, 4, L1)]
    recs = []
    for a, b in windows:
        w = rng.integers(0, 4, b - a)                          # strain a; strain b differs at 8 % of positions
        alt = w.copy()
        v = rng.random(b - a) < 0.08
        alt[v] = (alt[v] + 1) % 4
        for _ in range((b - a) * 20 // 100):
            p = int(rng.integers(0, b - a - 100 + 1))
            src = alt if rng.random() < 0.35 else w
            recs.append((1, a + p, 0, [(100 << 4) | 0], "".join("ACGT"[k] for k in src[p:p + 100]), None))
        ref = letters[w]
        m = rng.random(b - a) < 0.02                           # fixed differences from the reads
        ref[m] = letters[(w[m] + 2) % 4]
        fasta1[a:b] = ref
    recs.sort(key=lambda r: r[1])
    tid, pos, flag, mapq, cig_off, cig, nt16, _q = _columns(recs)
    pb = str(tmp_path / "big.sam")                            # (SAM: a BAM bin cannot hold positions past 2^29)
    samio.write_sam(pb, refs, lens, tid, pos, flag, mapq, cig_off, cig, seqs=[r[4] for r in recs])
    genes = [(1, px - 2500, px + 2400, 1, 1), (1, px - 1000, px + 2990, -1, 2), (1, px - 7, px + 8, 1, 0),
             (1, L1 - 2900, L1, -1, 0), (1, L1 - 2000, L1, 1, 2), (0, 0, 3000, 1, 0)]
    params = dict(min_coverage=5, min_freq=0.05, min_count=2)
    with AlignmentFile(pb, decode="gpu") as af:
        eng = af._count_engine()
        af.count_coverage("big1", 0, 1, quality_threshold=0)
        assert int(eng.n_slots) > (1 << 31) + 1000
        eng.set_reference(0, b"A" * L0)
        eng.set_reference(1, fasta1.tobytes())
        tidc, a_, b_, s_, ph_ = (np.array([g[i] for g in genes], np.int64) for i in range(5))
        records, sites = eng.gene_stats(tidc, a_, b_, s_, ph_, sites=True, **params)
        want_recs, want_sites = [], []
        for k, (t, a, b, s, ph) in enumerate(genes):
            if t == 0:
                want_recs.append(dict(dict.fromkeys(INT_FIELDS, 0), length=3000, codons=1000))
                continue
            wa, wb = next(w for w in windows if w[0] <= a and b <= w[1])
            cnt = np.stack(af.count_coverage("big1", wa, wb, quality_threshold=0))
            r, st = og.genes([cnt], [fasta1[wa:wb].tobytes().decode()], [(0, a - wa, b - wa, s, ph)], **params)
            want_recs += r
            want_sites += [(k, 1, p + wa) + x[3:] for x in st for p in [x[2]]]
        for k, r in enumerate(want_recs):
            assert {f: int(records[f][k]) for f in INT_FIELDS} == r, k
        assert _site_rows(sites) == want_sites
        assert records["snv_n"][:2].min() > 0 and records["sub_n"][:2].min() > 0
        assert any(p < px for _g, _t, p, *_x in want_sites) and any(p >= px for _g, _t, p, *_x in want_sites)
