"""Samples compared on the GPU (csrc/compare.cu) against oracle/compare.py: signatures of the seeded read sets of
test_gpu_basecount.py; all pairs of three samples over the region mix of test_gpu_alleles.py; the known answer of pure
strains from tools/bench_alleles.two_strain; invariance over formats, read orders, decode modes, pair batching and file
order; one counter store at a time; a table of more than 2^31 slots; the errors; and ``metacov compare``."""
import csv
import io
import math
import os
import sys

import numpy as np
import pytest

from oracle import basecount
from oracle import compare as oc
from test_gpu_alleles import PARAMS, _regions
from test_gpu_basecount import LENS, REFS, _columns, _gen, _write

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("length", "covered_a", "covered_b", "compared", "con_snp", "pop_snp")
SEEDS = (31, 32, 33)


def _bench_alleles():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_alleles
    return bench_alleles


@pytest.fixture(scope="module")
def samples(tmp_path_factory):
    """Three seeded read sets (BAM and SAM); the first also shuffled."""
    d = tmp_path_factory.mktemp("compare")
    out = []
    for k, seed in enumerate(SEEDS):
        recs = _gen(seed, n=6000)
        pb, ps = _write(recs, d, "s%d" % k)
        out.append(dict(recs=recs, bam=pb, sam=ps))
    rng = np.random.default_rng(34)
    recs = out[0]["recs"]
    out[0]["bam_shuf"], out[0]["sam_shuf"] = _write([recs[i] for i in rng.permutation(len(recs))], d, "s0_shuf")
    return out


_COUNTS = {}


def _counts(recs, t=15, cb="all"):
    k = (id(recs), t, cb)
    if k not in _COUNTS:
        tid, pos, flag, _mapq, cig_off, cig, nt16, quals = _columns(recs)
        _COUNTS[k] = basecount.full_counts(LENS, tid, pos, flag, cig_off, cig, nt16, quals, t, cb)
    return _COUNTS[k]


def _oracle_sigs(recs, t=15, cb="all", **params):
    return [oc.signature(c, **params) for c in _counts(recs, t, cb)]


@pytest.mark.parametrize("fmt", ["bam", "sam"])
@pytest.mark.parametrize("cb", ["all", "nofilter"])
@pytest.mark.parametrize("t", [0, 15])
def test_signature_matches_oracle(samples, fmt, cb, t):
    import torch
    from metacov_b200 import AlignmentFile
    s = samples[0]
    with AlignmentFile(s[fmt], decode="gpu") as af:
        eng = af._count_engine()
        n_covered = 0
        for params in PARAMS:
            sig = af.allele_signature(quality_threshold=t, read_callback=cb, **params)
            assert sig.dtype == torch.uint8 and sig.is_cuda and sig.numel() == int(eng.n_slots)
            got = sig.cpu().numpy()
            inside = np.zeros(len(got), bool)
            for c, want in enumerate(_oracle_sigs(s["recs"], t, cb, **params)):
                o = eng.contig_offset(c)
                assert np.array_equal(got[o:o + LENS[c]], want), (c, params)
                inside[o:o + LENS[c]] = True
                n_covered += int((want != 0).sum())
            assert not got[~inside].any()                  # padding and end slots
    assert n_covered > 10000


def _check_stats(stats, sigs, pairs, reg):
    assert stats.shape == (len(pairs), len(reg))
    for p, (a, b) in enumerate(pairs):
        for k, (c, lo, hi) in enumerate(reg):
            want = oc.pair_region(sigs[a][c], sigs[b][c], lo, hi)
            got = {f: int(stats[f][p, k]) for f in FIELDS}
            assert got == want, (a, b, c, lo, hi)


def _site_rows(sites):
    return list(zip(*(sites[f].tolist() for f in ("pair", "tid", "pos", "sig_a", "sig_b", "kind"))))


def _want_sites(sigs, pairs):
    return [r for p, (a, b) in enumerate(pairs) for r in oc.pair_sites(sigs[a], sigs[b], p)]


@pytest.mark.parametrize("params", [PARAMS[0], PARAMS[1], PARAMS[3]])
def test_stats_and_sites_match_oracle(samples, params):
    from metacov_b200.compare import compare
    reg = _regions(np.random.default_rng(35))
    sigs = [_oracle_sigs(s["recs"], **params) for s in samples]
    res = compare([s["bam"] for s in samples], [REFS[c] for c, _, _ in reg], [a for _, a, _ in reg],
                  [b for _, _, b in reg], sites=True, **params)
    assert res.pairs.tolist() == [[0, 1], [0, 2], [1, 2]]
    _check_stats(res.stats, sigs, res.pairs.tolist(), reg)
    want = _want_sites(sigs, res.pairs.tolist())
    assert _site_rows(res.sites) == want and len(want) > 50
    assert any(r[5] == 3 for r in want) and any(r[5] == 1 for r in want)
    whole = compare([s["sam"] for s in samples], **params)          # defaults: whole contigs, all pairs
    _check_stats(whole.stats, sigs, whole.pairs.tolist(), [(c, 0, LENS[c]) for c in range(3)])
    assert whole.sites is None


def _depth(tid, pos, lengths, span):
    out = []
    for c, n in enumerate(lengths):
        d = np.zeros(n + span + 1, np.int64)
        p = pos[tid == c]
        np.add.at(d, p, 1)
        np.add.at(d, np.minimum(p + span, n + span), -1)
        out.append(np.cumsum(d)[:n])
    return out


def test_known_answer_pure_strains(tmp_path):
    """err = 0: pure strain A against pure strain B differs, by consensus and by population, exactly at the covered
    variant positions; each pure strain against itself nowhere."""
    from metacov_b200.compare import compare
    ba = _bench_alleles()
    lengths, seed, cov = [40000, 7000, 300], 41, 12.0
    paths = []
    for minor in (0.0, 1.0, 0.5):
        cols, refs = ba.two_strain(lengths, cov, seed, minor=minor, err=0.0)
        p = str(tmp_path / ("m%g.bam" % minor))
        ba.write_bam_fast(p, lengths, *cols)
        paths.append(p)
    # the variant positions two_strain drew (the same generator, the same draws)
    rng = np.random.Generator(np.random.PCG64(seed))
    total = int(sum(lengths))
    rng.integers(0, 4, total, dtype=np.uint8)               # (the reference)
    var = np.unique(rng.integers(0, total, int(total * 0.01)))
    off = np.concatenate(([0], np.cumsum(lengths)))
    depth = _depth(cols[0], cols[1], lengths, ba.L_SEQ)
    covered = np.concatenate([d >= 5 for d in depth])
    n_var = int(covered[var].sum())
    assert n_var > 100
    res = compare(paths + [paths[0]], pairs=[(0, 1), (1, 0), (0, 2), (0, 3)], sites=True)      # A, B, mix, A again
    st = res.stats
    for c in range(len(lengths)):
        want_cov = int(covered[off[c]:off[c + 1]].sum())
        assert int(st["compared"][0, c]) == int(st["covered_a"][0, c]) == int(st["covered_b"][0, c]) == want_cov
        want = int(covered[var[(var >= off[c]) & (var < off[c + 1])]].sum())
        assert int(st["con_snp"][0, c]) == int(st["pop_snp"][0, c]) == want
        for f in ("length", "compared", "con_snp", "pop_snp"):                  # (B, A) mirrors (A, B)
            assert int(st[f][1, c]) == int(st[f][0, c])
        assert int(st["con_snp"][3, c]) == int(st["pop_snp"][3, c]) == 0        # pure A against itself
        assert int(st["compared"][3, c]) == want_cov
        # the 50 / 50 mix shares an allele with pure A wherever both alleles are called
        assert int(st["pop_snp"][2, c]) <= int(st["con_snp"][2, c])
    sites0 = res.sites[res.sites["pair"] == 0]
    slot = off[sites0["tid"]] + sites0["pos"]
    assert np.array_equal(np.sort(slot), var[covered[var]]) and (sites0["kind"] == 3).all()
    # pure B against itself
    same = compare([paths[1], paths[1]])
    assert int(same.stats["con_snp"].sum()) == int(same.stats["pop_snp"].sum()) == 0


def _snapshot(paths, decode="auto", **kw):
    from metacov_b200.compare import compare
    res = compare(paths, ["c0", "c2", "c1", "c2"], [10, 0, 90, 59000], [2500, 60000, 120, 70000], sites=True,
                  decode=decode, **kw)
    return res.stats.tobytes(), res.sites.tobytes()


def test_invariance(samples):
    from metacov_b200 import AlignmentFile
    from metacov_b200.compare import compare
    kw = dict(min_coverage=1, min_freq=0.0, min_count=1)
    rest = [samples[1]["bam"], samples[2]["sam"]]
    base = _snapshot([samples[0]["bam"]] + rest, **kw)
    for name in ("sam", "bam_shuf", "sam_shuf"):
        assert _snapshot([samples[0][name]] + rest, **kw) == base, name
    for decode in ("host", "gpu", "gpu-stream"):
        assert _snapshot([samples[0]["bam"], samples[1]["bam"], samples[2]["bam"]], decode=decode, **kw) == \
            _snapshot([samples[0]["bam"], samples[1]["bam"], samples[2]["bam"]], **kw), decode
    # open files as well as paths
    with AlignmentFile(samples[0]["bam"], decode="host") as af:
        assert _snapshot([af] + rest, **kw) == base
    # one call for every pair == one call per pair
    paths = [s["bam"] for s in samples]
    reg = _regions(np.random.default_rng(36))
    args = ([REFS[c] for c, _, _ in reg], [a for _, a, _ in reg], [b for _, _, b in reg])
    allp = compare(paths, *args, sites=True, **kw)
    for p, (a, b) in enumerate(allp.pairs.tolist()):
        one = compare(paths, *args, pairs=[(a, b)], sites=True, **kw)
        assert one.stats.tobytes() == allp.stats[p:p + 1].tobytes()
        mine = allp.sites[allp.sites["pair"] == p].copy()
        mine["pair"] = 0
        assert one.sites.tobytes() == mine.tobytes()
    # file order: the pairs of the reversed list are the same pairs with a and b swapped
    rev = compare(paths[::-1], *args, pairs=[(2, 1), (2, 0), (1, 0)], sites=True, **kw)
    assert rev.stats.tobytes() == allp.stats.tobytes()
    assert rev.sites.tobytes() == allp.sites.tobytes()
    sw = compare(paths, *args, pairs=[(1, 0), (2, 0), (2, 1)], sites=True, **kw)
    for f in ("length", "compared", "con_snp", "pop_snp"):
        assert np.array_equal(sw.stats[f], allp.stats[f])
    assert np.array_equal(sw.stats["covered_a"], allp.stats["covered_b"])
    assert np.array_equal(sw.sites["sig_a"], allp.sites["sig_b"]) and np.array_equal(sw.sites["pos"], allp.sites["pos"])


def test_allele_and_compare_calls_share_an_engine(samples):
    """The allele and compare calls of one engine share their region and site scratch but keep separate site lists:
    building the compare list leaves the allele list readable, and a compare pass in between leaves allele_stats
    bit-identical."""
    from metacov_b200 import AlignmentFile, _capi
    from metacov_b200._capi import lib
    kw = dict(min_coverage=1, min_freq=0.0, min_count=1)
    with AlignmentFile(samples[1]["bam"], decode="gpu") as af:
        other = af.allele_signature(**kw)
    reg = _regions(np.random.default_rng(37))
    tid, lo, hi = (np.array([r[k] for r in reg]) for k in range(3))
    with AlignmentFile(samples[0]["bam"], decode="gpu") as af:
        sigs, pairs = [af.allele_signature(**kw), other], [(0, 1)]
        eng = af._count_engine()
        sites = eng.allele_sites(**kw)
        csites = eng.compare_sites(sigs, pairs)
        first = eng.allele_stats(tid, lo, hi, **kw)
        cstats = eng.compare_stats(sigs, pairs, tid, lo, hi)
        again = eng.allele_stats(tid, lo, hi, **kw)
        assert len(sites) > 50 and len(csites) > 50 and int(cstats["con_snp"].sum()) > 0
        assert again.tobytes() == first.tobytes()
        for read, want, dtype in ((lib.mcov_allele_sites_read, sites, _capi.ALLELE_SITE_DTYPE),
                                  (lib.mcov_compare_sites_read, csites, _capi.COMPARE_SITE_DTYPE)):
            got = np.zeros(len(want), dtype=dtype)
            eng._check(read(eng._ctx, 0, len(want), _capi.ptr(got)))
            assert got.tobytes() == want.tobytes()


def test_one_counter_store_at_a_time(samples, monkeypatch):
    """compare counts a file only after the engine of every file counted before it is closed."""
    from metacov_b200 import CoverageEngine
    from metacov_b200.compare import compare
    counted = []
    real = CoverageEngine.base_counts

    def spy(self, *a, **k):
        assert all(e._ctx is None for e in counted if e is not self), "two counter stores held at once"
        counted.append(self)
        return real(self, *a, **k)

    monkeypatch.setattr(CoverageEngine, "base_counts", spy)
    for decode in ("gpu", "host"):
        counted.clear()
        compare([s["bam"] for s in samples] + [samples[0]["sam"]], sites=True, decode=decode)
        assert len(counted) == 4 and all(e._ctx is None for e in counted)


def test_more_than_2_31_slots(tmp_path):
    """Two files on two contigs of 1.5 x 10^9: reads across slot 2^31 and near the end of the second contig."""
    import samio
    from metacov_b200 import AlignmentFile
    from metacov_b200.compare import compare
    L = 1_500_000_000
    refs, lens = ["big0", "big1"], [L, L]
    off1 = (L + 1 + 3) & ~3
    px = (1 << 31) - off1                                   # position of contig 1 at slot 2^31
    windows = [(px - 1000, px + 1000), (L - 2000, L)]
    paths = []
    for seed in (51, 52):
        rng = np.random.default_rng(seed)
        recs = []
        for base in (px - 120, L - 400):
            for _ in range(300):
                p = base + int(rng.integers(0, 250))
                # the second file's strain differs from the first's at every seventh position
                s = "".join("ACGT"[k] if rng.random() < 0.3 else "ACGT"[(p + j + (seed == 52 and (p + j) % 7 == 0)) % 4]
                            for j, k in enumerate(rng.integers(0, 4, 150)))
                recs.append((1, p, 0, [(150 << 4) | 0], s, None))
        recs.sort(key=lambda r: r[1])
        tid, pos, flag, mapq, cig_off, cig, _nt16, _q = _columns(recs)
        pb = str(tmp_path / ("big%d.sam" % seed))               # (SAM: a BAM bin cannot hold positions past 2^29)
        samio.write_sam(pb, refs, lens, tid, pos, flag, mapq, cig_off, cig, seqs=[r[4] for r in recs])
        paths.append(pb)
    params = dict(quality_threshold=0, min_coverage=5, min_freq=0.05, min_count=2)
    op = {k: params[k] for k in ("min_coverage", "min_freq", "min_count")}
    win_sigs = []                                           # [file][window] signatures of the GPU's counts there
    for pb in paths:
        with AlignmentFile(pb, decode="gpu") as af:
            win_sigs.append([oc.signature(np.stack(af.count_coverage("big1", a, b, quality_threshold=0)), **op)
                             for a, b in windows])
    reg = [("big0", 0, L), ("big1", 0, L), ("big1", px - 1000, px + 1000), ("big1", L - 2000, L + 500),
           ("big1", px - 3, px + 2), ("big1", px + 5000, px + 6000)]
    res = compare(paths, [r[0] for r in reg], [r[1] for r in reg], [r[2] for r in reg], sites=True, **params)
    st = res.stats
    w = [oc.pair_region(win_sigs[0][k], win_sigs[1][k], 0, 2000) for k in range(2)]
    assert w[0]["compared"] > 100 and w[1]["compared"] > 100 and w[0]["con_snp"] > 10
    for f in FIELDS:
        assert int(st[f][0, 0]) == (L if f == "length" else 0), f
        assert int(st[f][0, 1]) == (L if f == "length" else w[0][f] + w[1][f]), f
        assert int(st[f][0, 2]) == w[0][f], f
        assert int(st[f][0, 3]) == (2500 if f == "length" else w[1][f]), f
        assert int(st[f][0, 5]) == (1000 if f == "length" else 0), f
    assert int(st["length"][0, 4]) == 5 and int(st["compared"][0, 4]) == 5
    want = [(0, 1, a + p, x, y, k) for (a, _b), k_ in zip(windows, range(2))
            for (_pair, _t, p, x, y, k) in oc.pair_sites([win_sigs[0][k_]], [win_sigs[1][k_]])]
    assert _site_rows(res.sites) == want
    assert any(r[2] < px for r in want) and any(px <= r[2] < px + 1000 for r in want)


def test_errors(samples, tmp_path):
    import ctypes as C
    import torch
    from metacov_b200 import AlignmentFile, CoverageEngine, McovError, _capi
    from metacov_b200._capi import lib
    from metacov_b200.compare import compare
    paths = [s["bam"] for s in samples]
    with pytest.raises(ValueError, match="at least two files"):
        compare(paths[:1])
    for bad in ([(0, 0)], [(0, 3)], [(-1, 1)], []):
        with pytest.raises(ValueError, match="pairs"):
            compare(paths, pairs=bad)
    with pytest.raises(ValueError):
        compare(paths, min_count=0)
    # differing headers: the first file and contig that differ are named
    import samio
    other = str(tmp_path / "other.sam")
    recs = samples[1]["recs"]
    tid, pos, flag, mapq, cig_off, cig, _nt16, _q = _columns(recs)
    samio.write_sam(other, REFS, [LENS[0], LENS[1] + 1, LENS[2]], tid, pos, flag, mapq, cig_off, cig,
                    seqs=[r[4] for r in recs])
    with pytest.raises(ValueError, match=r"other\.sam: contig 1 is 'c1' of length 501, and 'c1' of length 500 in"):
        compare(paths[:2] + [other])
    # a piped input
    with AlignmentFile(io.BytesIO(open(samples[0]["sam"], "rb").read())) as s:
        with pytest.raises(ValueError, match="read once"):
            s.allele_signature()
        with pytest.raises(ValueError, match="read once"):
            compare([paths[0], s])
    with CoverageEngine(LENS) as eng:
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):          # no counts
            eng.allele_signature()
        p = _capi.AlleleParams(min_coverage=5, min_count=2, min_freq=0.05, use_reference=1)
        out = torch.zeros(int(eng.n_slots), dtype=torch.uint8, device="cuda")
        assert lib.mcov_allele_signature(eng._ctx, C.byref(p), _capi.ptr(out)) == _capi.MCOV_ERR_ARG
    with AlignmentFile(paths[0], decode="gpu") as af:
        eng = af._count_engine()
        sig = af.allele_signature()
        sig2 = af.allele_signature(min_count=1)
        p = _capi.AlleleParams(min_coverage=5, min_count=2, min_freq=0.05, use_reference=1)
        assert lib.mcov_allele_signature(eng._ctx, C.byref(p), _capi.ptr(sig)) == _capi.MCOV_ERR_ARG
        p.use_reference = 0
        host = np.zeros(int(eng.n_slots), np.uint8)
        assert lib.mcov_allele_signature(eng._ctx, C.byref(p), _capi.ptr(host)) == _capi.MCOV_ERR_ARG
        g = np.zeros(1, np.int32)
        for bad in (sig.cpu(), sig.to(torch.int32), sig[:-4], sig[::2], sig.view(-1, 4)):
            with pytest.raises(ValueError, match="signature 1"):
                eng.compare_stats([sig2, bad], [(0, 1)], g, g, g + 10)
            with pytest.raises(ValueError, match="signature 1"):
                eng.compare_sites([sig2, bad], [(0, 1)])
        for pairs in ([(0, 0)], [(0, 2)], []):
            with pytest.raises(ValueError, match="pairs"):
                eng.compare_stats([sig, sig2], pairs, g, g, g + 10)
        with pytest.raises(ValueError, match="at least two"):
            eng.compare_sites([sig], [(0, 0)])
        # the C level: MCOV_ERR_ARG, the context usable afterwards
        tab = (C.c_void_p * 2)(sig.data_ptr(), sig2.data_ptr())
        out = np.zeros(1, _capi.COMPARE_STATS_DTYPE)
        n = C.c_int64(0)
        for pr in ((0, 0), (0, 2), (-1, 1)):
            pa = np.array(pr, np.int32)
            assert lib.mcov_compare_run(eng._ctx, 2, tab, 1, _capi.ptr(pa), 1, _capi.ptr(g), _capi.ptr(g),
                                        _capi.ptr(g + 10), _capi.ptr(out)) == _capi.MCOV_ERR_ARG
            assert lib.mcov_compare_sites(eng._ctx, 2, tab, 1, _capi.ptr(pa), C.byref(n)) == _capi.MCOV_ERR_ARG
        pa = np.array([0, 1], np.int32)
        assert lib.mcov_compare_run(eng._ctx, 1, tab, 1, _capi.ptr(pa), 1, _capi.ptr(g), _capi.ptr(g),
                                    _capi.ptr(g + 10), _capi.ptr(out)) == _capi.MCOV_ERR_ARG
        htab = (C.c_void_p * 2)(sig.data_ptr(), host.ctypes.data)
        assert lib.mcov_compare_sites(eng._ctx, 2, htab, 1, _capi.ptr(pa), C.byref(n)) == _capi.MCOV_ERR_ARG
        for t, a, b in ((3, 0, 1), (0, -1, 1), (0, 5, 4)):
            arr = [np.array([x], np.int32) for x in (t, a, b)]
            assert lib.mcov_compare_run(eng._ctx, 2, tab, 1, _capi.ptr(pa), 1, *[_capi.ptr(x) for x in arr],
                                        _capi.ptr(out)) == _capi.MCOV_ERR_ARG
        assert lib.mcov_compare_sites_read(eng._ctx, 0, 1, _capi.ptr(out)) in (_capi.MCOV_ERR_ARG, _capi.MCOV_ERR_STATE)
        st = eng.compare_stats([sig, sig2], [(0, 1)], g, g, g + 3000)
        assert int(st["length"][0, 0]) == 3000 and int(st["compared"][0, 0]) > 0
        assert len(eng.compare_sites([sig, sig2], [(0, 1)])) >= 0
    with CoverageEngine(LENS) as eng:
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng._check(lib.mcov_compare_sites_read(eng._ctx, 0, 0, None))


def _invoke(args):
    from click.testing import CliRunner
    from metacov_b200.cli import main
    r = CliRunner().invoke(main, args, catch_exceptions=False)
    assert r.exit_code == 0, r.output
    return r


def test_cli(samples, tmp_path):
    from metacov_b200.alleles import derive_compare
    from metacov_b200.compare import compare
    rc = tmp_path / "r.csv"
    rc.write_text("sacc,start,end\nc0,100,900\nc2,52000,12000\nc1,400,700\n")
    paths = [s["bam"] for s in samples]
    for regions in (None, str(rc)):
        out, sites = tmp_path / "c.csv", tmp_path / "s.tsv"
        args = ["compare"] + [x for p in paths for x in ("-b", p)] + ["-o", str(out), "--sites-out", str(sites),
                                                                      "--min-count", "3"]
        args += ["-rc", regions] if regions else []
        _invoke(args)
        reg = [("c0", 100, 900), ("c2", 12000, 52000), ("c1", 400, 700)] if regions else list(zip(REFS, [0] * 3, LENS))
        want = compare(paths, [r[0] for r in reg], [r[1] for r in reg], [r[2] for r in reg], sites=True, min_count=3)
        der = derive_compare(want.stats)
        rows = list(csv.DictReader(open(out)))
        assert list(rows[0]) == ["sacc", "start", "end", "sample_a", "sample_b", "compared", "con_ani", "con_snps",
                                 "covered_a", "covered_b", "percent_compared", "pop_ani", "pop_snps"]
        assert len(rows) == 3 * len(reg)
        for k, row in enumerate(rows):
            r, p = divmod(k, 3)
            a, b = want.pairs[p]
            assert (row["sacc"], row["sample_a"], row["sample_b"]) == (reg[r][0], paths[a], paths[b])
            for name, f in (("compared", "compared"), ("con_snps", "con_snp"), ("pop_snps", "pop_snp"),
                            ("covered_a", "covered_a"), ("covered_b", "covered_b")):
                assert int(row[name]) == int(want.stats[f][p, r]), (name, row)
            for name, v in der.items():
                x = float(row[name])
                assert (math.isnan(x) and math.isnan(v[p, r])) or x == float(v[p, r]), (name, row)
        if regions:
            assert (rows[3]["start"], rows[3]["end"]) == ("52000", "12000")       # echoed as given
        lines = open(sites).read().splitlines()
        assert lines[0].split("\t") == ["sample_a", "sample_b", "contig", "pos", "cons_a", "cons_b", "alleles_a",
                                        "alleles_b", "con_snp", "pop_snp"]
        assert len(lines) - 1 == len(want.sites) > 20
        for line, s in zip(lines[1:], want.sites):
            f = line.split("\t")
            a, b = want.pairs[s["pair"]]
            sets = oc.allele_sets(np.array([s["sig_a"], s["sig_b"]], np.uint8))
            letters = ["".join(ch for i, ch in enumerate("ACGT") if x >> i & 1) for x in sets.tolist()]
            assert f == [paths[a], paths[b], REFS[s["tid"]], str(s["pos"]), "ACGT"[(s["sig_a"] >> 4) & 3],
                         "ACGT"[(s["sig_b"] >> 4) & 3], letters[0], letters[1], "1", str((s["kind"] >> 1) & 1)]
