"""Allele statistics and sites on the GPU (csrc/alleles.cu) against oracle/alleles.py: the seeded read sets of
test_gpu_basecount.py with a reference FASTA of lowercase, N and IUPAC bases; invariance over formats, read orders and
decode modes; C2- and C3-shaped tables of 5 x 10^7 slots; a table of more than 2^31 slots; what the calls leave alone;
the errors; and ``metacov alleles``."""
import csv
import io
import math
import os
import sys

import numpy as np
import pytest

from oracle import alleles as oa
from oracle import basecount
from test_gpu_basecount import LENS, REFS, _columns, _gen, _write

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAMS = [dict(), dict(min_coverage=1, min_freq=0.0, min_count=1), dict(min_coverage=20, min_freq=0.3, min_count=5),
          dict(min_coverage=3, min_freq=0.2, min_count=2)]
INT_FIELDS = ("length", "covered", "depth_sum", "snv", "ref_covered", "sub", "popsub")


def _fasta_seqs(seed):
    rng = np.random.default_rng(seed)
    letters = "ACGTACGTacgtNNRYKMSWn"
    return [("".join(letters[k] for k in rng.integers(0, len(letters), n))) for n in LENS]


def _write_fasta(path, names, seqs):
    with open(path, "w") as fh:
        for n, s in zip(names, seqs):
            fh.write(">%s some description\n" % n)
            for a in range(0, len(s), 61):
                fh.write(s[a:a + 61] + "\n")


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("alleles")
    recs = _gen(17)
    rng = np.random.default_rng(18)
    shuf = [recs[i] for i in rng.permutation(len(recs))]
    pb, ps = _write(recs, d, "sorted")
    ub, us = _write(shuf, d, "shuffled")
    seqs = _fasta_seqs(19)
    fa = str(d / "ref.fa")
    _write_fasta(fa, REFS, seqs)
    return dict(recs=recs, bam=pb, sam=ps, bam_shuf=ub, sam_shuf=us, fasta=fa, seqs=seqs, dir=d)


_COUNTS = {}


def _counts(recs, t, cb):
    k = (id(recs), t, cb)
    if k not in _COUNTS:
        tid, pos, flag, _mapq, cig_off, cig, nt16, quals = _columns(recs)
        _COUNTS[k] = basecount.full_counts(LENS, tid, pos, flag, cig_off, cig, nt16, quals, t, cb)
    return _COUNTS[k]


def _regions(rng):
    """Whole contigs, overlapping, empty, past the contig end, starting past it, and random ones."""
    reg = [(c, 0, LENS[c]) for c in range(3)]
    reg += [(0, 100, 900), (0, 500, 1500), (0, 700, 700), (1, 90, 130), (1, 95, 105), (1, 400, 700), (1, 600, 800),
            (2, 59000, 70000), (2, 0, 1), (2, 12000, 52000)]
    for _ in range(30):
        c = int(rng.integers(0, 3))
        a = int(rng.integers(0, LENS[c]))
        reg.append((c, a, a + int(rng.integers(0, 5000))))
    return reg


def _check_stats(got, counts, seqs, reg, params):
    for k, (c, a, b) in enumerate(reg):
        ref = oa.region_stats(counts[c], None if seqs is None else seqs[c], a, b, **params)
        for f in INT_FIELDS:
            assert int(got[f][k]) == ref[f], (f, c, a, b, params)
        assert abs(float(got["pi_sum"][k]) - ref["pi_sum"]) <= 1e-12 * abs(ref["pi_sum"]), (c, a, b, params)


def _check_sites(got, counts, seqs, params):
    ref = oa.sites(counts, seqs, **params)
    assert len(got) == len(ref)
    rows = list(zip(got["tid"].tolist(), got["pos"].tolist(), got["A"].tolist(), got["C"].tolist(), got["G"].tolist(),
                    got["T"].tolist(), [x.decode() for x in got["ref"].tolist()],
                    [x.decode() for x in got["consensus"].tolist()], got["kind"].tolist()))
    assert rows == ref
    return len(ref)


@pytest.mark.parametrize("fmt", ["bam", "sam"])
@pytest.mark.parametrize("cb", ["all", "nofilter"])
@pytest.mark.parametrize("t", [0, 15])
def test_matches_oracle(files, fmt, cb, t):
    from metacov_b200 import AlignmentFile, FastaFile
    counts = _counts(files["recs"], t, cb)
    rng = np.random.default_rng(len(fmt) * 7 + t + len(cb))
    reg = _regions(rng)
    fa = FastaFile(files["fasta"])
    n_sites = {}
    with AlignmentFile(files[fmt], decode="gpu") as af:
        for params in PARAMS:
            for fasta, seqs in ((None, None), (fa, files["seqs"])):
                kw = dict(fasta=fasta, quality_threshold=t, read_callback=cb, **params)
                got = af.allele_stats([REFS[c] for c, _, _ in reg], [a for _, a, _ in reg], [b for _, _, b in reg], **kw)
                _check_stats(got, counts, seqs, reg, params)
                n_sites[(len(n_sites), fasta is None)] = _check_sites(af.allele_sites(**kw), counts, seqs, params)
                whole = af.allele_stats(**kw)                        # defaults: whole contigs
                _check_stats(whole, counts, seqs, [(c, 0, LENS[c]) for c in range(3)], params)
    assert max(n_sites.values()) > 1000


def _snapshot(af, fa):
    out = []
    for params in PARAMS[:2]:
        for t, cb in ((15, "all"), (0, "nofilter")):
            kw = dict(fasta=fa, quality_threshold=t, read_callback=cb, **params)
            out.append(af.allele_stats(**kw).tobytes())
            out.append(af.allele_stats(["c0", "c1", "c2", "c1"], [10, 0, 100, 90], [2500, 900, 60000, 120], **kw).tobytes())
            out.append(af.allele_sites(**kw).tobytes())
    return out


def test_bit_identical_over_formats_orders_and_decoders(files):
    from metacov_b200 import AlignmentFile, FastaFile
    fa = FastaFile(files["fasta"])
    runs = {}
    for name in ("bam", "sam", "bam_shuf", "sam_shuf"):
        with AlignmentFile(files[name], decode="gpu") as af:
            runs[name] = _snapshot(af, fa)
            assert _snapshot(af, fa) == runs[name]                  # the same call twice
    for decode, kw in (("host", {}), ("gpu-stream", {"gpu_chunk_bytes": 1 << 17})):
        for name in ("bam", "bam_shuf"):
            with AlignmentFile(files[name], decode=decode, **kw) as af:
                runs[name + "_" + decode] = _snapshot(af, fa)
    for k, v in runs.items():
        assert v == runs["bam"], k


def test_depth_counts_and_verdict_left_alone(files):
    from metacov_b200 import AlignmentFile, FastaFile
    fa = FastaFile(files["fasta"])
    for decode in ("gpu", "host"):
        with AlignmentFile(files["bam"], decode=decode) as af:
            eng = af.coverage_engine()
            tid = np.arange(3, dtype=np.int32)

            def snap():
                return ([af.count_coverage_depth(c) for c in REFS],
                        eng.region_stats(tid, np.zeros_like(tid), np.array(LENS, np.int32)), eng.pass_info())
            d0, s0, p0 = snap()
            af.allele_stats(fasta=fa)
            af.allele_sites(fasta=fa, min_coverage=1, min_count=1, min_freq=0.0)
            ceng = af._count_engine()
            n = ceng.launch_count()
            c1 = [np.stack(af.count_coverage(c, quality_threshold=15)) for c in REFS]
            assert ceng.launch_count() == n                          # the same pair: no recount
            d1, s1, p1 = snap()
            for a, b in zip(c1, _counts(files["recs"], 15, "all")):
                assert np.array_equal(a, b)
            for a, b in zip(d0, d1):
                assert np.array_equal(a, b)
            assert s0.tobytes() == s1.tobytes() and p0 == p1
            af.allele_stats(quality_threshold=0)                     # another pair recounts
            assert ceng.launch_count() > n


def test_errors(files, tmp_path, monkeypatch):
    import ctypes as C
    from metacov_b200 import AlignmentFile, CoverageEngine, FastaFile, McovError, _capi
    from metacov_b200._capi import lib
    good = FastaFile(files["fasta"])
    missing, wrong = str(tmp_path / "missing.fa"), str(tmp_path / "wrong.fa")
    _write_fasta(missing, REFS[:2], files["seqs"][:2])
    _write_fasta(wrong, REFS, files["seqs"][:2] + [files["seqs"][2][:-1]])
    with AlignmentFile(io.BytesIO(open(files["sam"], "rb").read())) as s:
        with pytest.raises(ValueError, match="read once"):
            s.allele_stats()
        with pytest.raises(ValueError, match="read once"):
            s.allele_sites()
    with AlignmentFile(files["bam"], decode="gpu") as af:
        with pytest.raises(ValueError, match="'c2' is not in the reference FASTA"):
            af.allele_stats(fasta=FastaFile(missing))
        with pytest.raises(ValueError, match="'c2' is 59999 long in the reference FASTA and 60000"):
            af.allele_sites(fasta=FastaFile(wrong))
        for bad in (dict(min_coverage=0), dict(min_count=0), dict(min_freq=1.01), dict(min_freq=-1e-9),
                    dict(min_freq=float("nan")), dict(min_coverage=2.5), dict(read_callback="mapped")):
            with pytest.raises(ValueError):
                af.allele_stats(**bad)
            with pytest.raises(ValueError):
                af.allele_sites(**bad)
        for reg in ((["c0"], [-1], [10]), (["c0"], [10], [5]), (["c0", "c1"], [0], [5])):
            with pytest.raises(ValueError):
                af.allele_stats(*reg)
        with pytest.raises(KeyError):
            af.allele_stats(["nope"])
        # the C level: bad parameters and regions are MCOV_ERR_ARG, with the file still usable afterwards
        eng = af._count_engine()
        p = _capi.AlleleParams(min_coverage=5, min_count=2, min_freq=0.05, use_reference=0)
        out = np.zeros(1, _capi.ALLELE_STATS_DTYPE)
        one = np.zeros(1, np.int32)
        for field, v in (("min_coverage", 0), ("min_count", 0), ("min_freq", 1.5), ("use_reference", 2)):
            q = _capi.AlleleParams(min_coverage=5, min_count=2, min_freq=0.05, use_reference=0)
            setattr(q, field, v)
            assert lib.mcov_allele_stats_run(eng._ctx, 1, _capi.ptr(one), _capi.ptr(one), _capi.ptr(one), C.byref(q),
                                             _capi.ptr(out)) == _capi.MCOV_ERR_ARG
        for t, a, b in ((3, 0, 1), (0, -1, 1), (0, 5, 4)):
            arr = [np.array([x], np.int32) for x in (t, a, b)]
            assert lib.mcov_allele_stats_run(eng._ctx, 1, *[_capi.ptr(x) for x in arr], C.byref(p),
                                             _capi.ptr(out)) == _capi.MCOV_ERR_ARG
        n = C.c_int64(0)
        assert lib.mcov_allele_sites_read(eng._ctx, 0, 1 << 40, _capi.ptr(out)) in (_capi.MCOV_ERR_ARG, _capi.MCOV_ERR_STATE)
        assert lib.mcov_set_reference(eng._ctx, 0, b"ACGT", 4) == _capi.MCOV_ERR_ARG      # not the contig's length
        # the reference store does not fit: MemoryError naming both byte counts, nothing kept
        af2 = AlignmentFile(files["bam"], decode="gpu")
        monkeypatch.setenv("MCOV_REF_FREE_BYTES", "1000")
        with pytest.raises(MemoryError, match=r"needs \d+ bytes of device memory, \d+ are free"):
            af2.allele_stats(fasta=good)
        monkeypatch.delenv("MCOV_REF_FREE_BYTES")
        counts = _counts(files["recs"], 15, "all")
        _check_stats(af2.allele_stats(fasta=good), counts, files["seqs"], [(c, 0, LENS[c]) for c in range(3)], {})
        af2.close()
        _check_stats(af.allele_stats(fasta=good), counts, files["seqs"], [(c, 0, LENS[c]) for c in range(3)], {})
    # before any counts, and with use_reference without a reference: MCOV_ERR_STATE
    with CoverageEngine(LENS) as eng:
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng.allele_stats([0], [0], [10])
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng.allele_sites()
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng._check(lib.mcov_allele_sites_read(eng._ctx, 0, 0, None))
    with AlignmentFile(files["bam"], decode="gpu") as af:
        eng = af._count_engine()
        af.count_coverage("c0")
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng.allele_stats([0], [0], [10], use_reference=True)
        eng.set_reference(0, files["seqs"][0])
        with pytest.raises(McovError, match="contig 1 has no reference"):
            eng.allele_sites(use_reference=True)
        assert len(eng.allele_sites()) > 0


def _invoke(args):
    from click.testing import CliRunner
    from metacov_b200.cli import main
    r = CliRunner().invoke(main, args, catch_exceptions=False)
    assert r.exit_code == 0, r.output
    return r


def test_cli(files, tmp_path):
    from metacov_b200 import AlignmentFile, FastaFile
    from metacov_b200.alleles import derive
    rb = tmp_path / "r.blast7"
    rb.write_text("# BLASTN 2.2.31+\n# Fields: query acc., subject acc., % identity, alignment length, mismatches, gap opens, "
                  "q. start, q. end, s. start, s. end, evalue, bit score\n"
                  "q1\tc0\t99.0\t800\t0\t0\t1\t800\t100\t900\t0.0\t1000\n"
                  "q2\tc2\t99.0\t800\t0\t0\t1\t800\t52000\t12000\t0.0\t1000\n"
                  "q3\tc1\t99.0\t800\t0\t0\t1\t800\t400\t700\t0.0\t1000\n")
    for fasta in (None, files["fasta"]):
        for regions in (None, str(rb)):
            out, sites = tmp_path / "r.csv", tmp_path / "s.tsv"
            args = ["alleles", "-b", files["bam"], "-o", str(out), "--sites-out", str(sites), "--min-count", "3"]
            args += ["-f", fasta] if fasta else []
            args += ["-rb", regions] if regions else []
            _invoke(args)
            with AlignmentFile(files["bam"], decode="gpu") as af:
                fa = FastaFile(fasta) if fasta else None
                reg = [("c0", 100, 900), ("c2", 12000, 52000), ("c1", 400, 700)] if regions else [(c, 0, n) for c, n in zip(REFS, LENS)]
                st = af.allele_stats([r[0] for r in reg], [r[1] for r in reg], [r[2] for r in reg], fasta=fa, min_count=3)
                want = derive(st)
                want_sites = af.allele_sites(fasta=fa, min_count=3)
            rows = list(csv.DictReader(open(out)))
            assert list(rows[0]) == ["sacc", "start", "end", "breadth", "con_ani", "depth", "pi", "pop_ani", "snv_per_kbp"]
            assert len(rows) == len(reg)
            for k, row in enumerate(rows):
                assert row["sacc"] == reg[k][0]
                for name, v in want.items():
                    x = float(row[name])
                    assert (math.isnan(x) and math.isnan(v[k])) or x == float(v[k]), (name, row)
            if regions:
                assert (rows[1]["start"], rows[1]["end"]) == ("52000", "12000")       # echoed as given
            lines = open(sites).read().splitlines()
            assert lines[0].split("\t") == ["contig", "pos", "ref", "A", "C", "G", "T", "consensus", "snv", "sub", "popsub"]
            assert len(lines) - 1 == len(want_sites) > 100
            for line, s in zip(lines[1:], want_sites):
                f = line.split("\t")
                k = int(s["kind"])
                assert f == [REFS[s["tid"]], str(s["pos"]), s["ref"].decode(), str(s["A"]), str(s["C"]), str(s["G"]),
                             str(s["T"]), s["consensus"].decode(), str(k & 1), str((k >> 1) & 1), str((k >> 2) & 1)]
            if fasta is None:
                assert all(l.split("\t")[2] == "N" for l in lines[1:])


def _bench_module():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_alleles
    return bench_alleles


def _check_against_own_counts(af, eng, refs, params):
    """GPU records and sites against the oracle applied to the GPU's own counts (only the allele kernels under test)."""
    lens = [int(l) for l in af.lengths]
    st = af.allele_stats(**params)
    sites = af.allele_sites(**params)
    k = 0
    for c in range(len(lens)):
        cnt = eng.copy_base_counts(c)
        ref = None if refs is None else refs[c]
        r = oa.region_stats(cnt, ref, 0, lens[c], **{x: params[x] for x in ("min_coverage", "min_freq", "min_count")})
        for f in INT_FIELDS:
            assert int(st[f][c]) == r[f], (c, f)
        assert abs(float(st["pi_sum"][c]) - r["pi_sum"]) <= 1e-12 * abs(r["pi_sum"])
        e = oa.evaluate(cnt, ref, **{x: params[x] for x in ("min_coverage", "min_freq", "min_count")})
        pos = np.nonzero(e["kind"])[0]
        got = sites[k:k + len(pos)]
        assert (got["tid"] == c).all() and np.array_equal(got["pos"], pos), c
        assert np.array_equal(got["kind"], e["kind"][pos])
        for b, name in enumerate("ACGT"):
            assert np.array_equal(got[name], cnt[b, pos])
        assert np.array_equal(got["consensus"], np.frombuffer(b"ACGT", "S1")[e["consensus"][pos]])
        assert np.array_equal(got["ref"], np.frombuffer(b"ACGTN", "S1")[e["ref"][pos]])
        k += len(pos)
    assert k == len(sites)
    return st, sites


@pytest.mark.parametrize("shape", ["c2", "c3"])
def test_scale_5e7_slots(tmp_path, shape):
    from metacov_b200 import AlignmentFile, FastaFile, synth
    ba = _bench_module()
    lengths = synth.c2(1.0).contig_len if shape == "c2" else synth.c3(0.045).contig_len
    assert int(np.asarray(lengths, np.int64).sum()) >= 5e7
    pb, pf, _n = ba.write_workload(str(tmp_path), shape, lengths, 6.0, 23)
    fa = FastaFile(pf)
    with AlignmentFile(pb, decode="gpu") as af:
        eng = af._count_engine()
        refs = [fa.fetch(n) for n in af.references]
        params = dict(min_coverage=3, min_freq=0.1, min_count=2)
        st, sites = _check_against_own_counts(af, eng, refs, dict(fasta=fa, **params))
        assert int(eng.n_slots) >= 5e7
        assert st["snv"].sum() > 50000 and (sites["kind"] & 2).any() and (sites["kind"] & 4).any()


def test_more_than_2_31_slots(tmp_path):
    """Two contigs of 1.5 x 10^9: reads near the end of the second and across slot 2^31; 48 GB of
    counters."""
    import samio
    from metacov_b200 import AlignmentFile
    L = 1_500_000_000
    refs, lens = ["big0", "big1"], [L, L]
    off1 = (L + 1 + 3) & ~3
    px = (1 << 31) - off1                                   # position of contig 1 at slot 2^31
    rng = np.random.default_rng(29)
    recs = []
    for base in (px - 120, L - 400):
        for _ in range(300):
            p = base + int(rng.integers(0, 250))
            s = "".join("ACGT"[k] if rng.random() < 0.3 else "ACGT"[(p + j) % 4] for j, k in enumerate(rng.integers(0, 4, 150)))
            recs.append((1, p, 0, [(150 << 4) | 0], s, None))
    recs.sort(key=lambda r: r[1])
    tid, pos, flag, mapq, cig_off, cig, nt16, _q = _columns(recs)
    pb = str(tmp_path / "big.sam")                          # (SAM: a BAM bin cannot hold positions past 2^29)
    samio.write_sam(pb, refs, lens, tid, pos, flag, mapq, cig_off, cig, seqs=[r[4] for r in recs])
    windows = [(px - 1000, px + 1000), (L - 2000, L)]
    params = dict(quality_threshold=0, min_coverage=5, min_freq=0.05, min_count=2)
    with AlignmentFile(pb, decode="gpu") as af:
        eng = af._count_engine()
        assert int(eng.n_slots) > (1 << 31) + 1000
        reg = [("big0", 0, L), ("big1", 0, L), ("big1", px - 1000, px + 1000), ("big1", px - 3, px + 2),
               ("big1", L - 2000, L + 500), ("big1", px + 5000, px + 6000)]
        st = af.allele_stats([r[0] for r in reg], [r[1] for r in reg], [r[2] for r in reg], **params)
        sites = af.allele_sites(**params)
        # the GPU's counts in the two windows equal the count rules applied to the reads shifted into them
        win = []
        for a, b in windows:
            got = np.stack(af.count_coverage("big1", a, b, quality_threshold=0))
            sel = [i for i, r in enumerate(recs) if a <= r[1] < b]
            want = basecount.full_counts([b - a], np.zeros(len(sel), np.int32), pos[sel] - a, flag[sel],
                                         np.concatenate(([0], np.cumsum(np.diff(cig_off)[sel]))).astype(np.uint32),
                                         cig[np.concatenate([np.arange(cig_off[i], cig_off[i + 1]) for i in sel])],
                                         [nt16[i] for i in sel], [None] * len(sel), 0, "all")[0]
            assert np.array_equal(got, want) and got.sum() > 0
            win.append(got)
        op = {k: params[k] for k in ("min_coverage", "min_freq", "min_count")}
        w0 = oa.region_stats(win[0], None, 0, 2000, **op)
        w1 = oa.region_stats(win[1], None, 0, 2000, **op)
        both = {f: w0[f] + w1[f] for f in INT_FIELDS}
        for f in INT_FIELDS:
            assert int(st[f][0]) == (L if f == "length" else 0)
            assert int(st[f][1]) == (L if f == "length" else both[f]), f
            assert int(st[f][2]) == w0[f], f
            assert int(st[f][4]) == (2500 if f == "length" else w1[f]), f
            assert int(st[f][5]) == (1000 if f == "length" else 0), f
        assert abs(float(st["pi_sum"][1]) - math.fsum([w0["pi_sum"], w1["pi_sum"]])) <= 1e-12 * float(st["pi_sum"][1])
        assert abs(float(st["pi_sum"][2]) - w0["pi_sum"]) <= 1e-12 * w0["pi_sum"]
        assert int(st["length"][3]) == 5 and int(st["covered"][3]) == 5
        want = [(1, a + p) + t[2:] for (a, _b), w in zip(windows, win) for t in oa.sites([w], None, **op)
                for p in [t[1]]]
        rows = list(zip(sites["tid"].tolist(), sites["pos"].tolist(), sites["A"].tolist(), sites["C"].tolist(),
                        sites["G"].tolist(), sites["T"].tolist(), [x.decode() for x in sites["ref"].tolist()],
                        [x.decode() for x in sites["consensus"].tolist()], sites["kind"].tolist()))
        assert rows == want and len(rows) > 100
        assert any(r[1] < px for r in rows) and any(px <= r[1] < px + 1000 for r in rows)
