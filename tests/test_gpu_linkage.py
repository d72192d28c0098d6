"""Linkage on the GPU (csrc/linkage.cu) against oracle/linkage.py: seeded paired read sets of two and three strains with
errors, every flag kind (supplementary pieces included), reads with and without qualities, '*' names, reads past the
contig end and long reads; one output over formats, read orders and decode modes (the streamed one with mates in
different chunks); what the call leaves alone; the errors; ``metacov linkage``; a table of more than 2^31 slots."""
import io

import numpy as np
import pytest

from oracle import bamio
from oracle import linkage as ol
import samio
from test_gpu_basecount import _columns, _set_bam_quals

pytestmark = pytest.mark.gpu

REFS = ["c0", "c1 second contig", "c2"]
LENS = [3000, 700, 20000]
PARAMS = dict(min_coverage=3, min_freq=0.05, min_count=2, max_distance=600, min_reads=3)
FLAGS = [0x1 | 0x2 | 0x40, 0x1 | 0x2 | 0x80 | 0x10, 0x1 | 0x40 | 0x10, 0x1 | 0x80]
ODD_FLAGS = [0x100, 0x200, 0x400, 0x800, 0x4, 0x1 | 0x8 | 0x40]


def _gen(seed, n_strains, n_frag=2500, long_reads=3, one_name=False):
    """Records (tid, pos, flag, ops, SEQ letters, Phred list or None, name), coordinate-sorted: fragments of
    `n_strains` strains over a random reference, two mates each (inserts 300-500), sometimes a supplementary piece."""
    rng = np.random.default_rng(seed)
    ref = [rng.integers(0, 4, n) for n in LENS]
    strains = []
    for _s in range(n_strains):
        st = []
        for r in ref:
            x = r.copy()
            var = rng.random(len(x)) < 0.03
            x[var] = (x[var] + rng.integers(1, 4, int(var.sum()))) % 4
            st.append(x)
        strains.append(st)
    weights = np.array([0.6, 0.3, 0.1][:n_strains]) / sum([0.6, 0.3, 0.1][:n_strains])
    recs = []

    def read(tid, pos, strain, qlen, name, flag, complex_ops):
        ops = [(qlen << 4) | 0]
        if complex_ops:
            ops = []
            left = qlen
            while left > 0:
                op = "MMMMIDNS=X"[int(rng.integers(0, 10))]
                n = int(min(left, rng.integers(1, 40))) if op in "MIS=X" else int(rng.integers(1, 20))
                ops.append((n << 4) | bamio.CIGAR_OPS.index(op))
                if op in "MIS=X":
                    left -= n
        seq = []
        r = pos
        for o in ops:
            op, n = o & 15, o >> 4
            for j in range(n if op in (0, 1, 4, 7, 8) else 0):
                if op in (0, 7, 8):
                    b = int(strains[strain][tid][r + j]) if r + j < LENS[tid] else int(rng.integers(0, 4))
                else:
                    b = int(rng.integers(0, 4))
                if rng.random() < 0.01:
                    b = (b + int(rng.integers(1, 4))) % 4
                seq.append("ACGTN"[4 if rng.random() < 0.002 else b])
            if op in (0, 2, 3, 7, 8):
                r += n
        q = None if rng.random() < 0.2 else [int(x) for x in rng.integers(2, 42, len(seq))]
        recs.append((tid, pos, flag, ops, "".join(seq), q, name))

    for f in range(n_frag):
        tid = int(rng.choice(len(LENS), p=np.array(LENS) / sum(LENS)))
        strain = int(rng.choice(n_strains, p=weights))
        ins = int(rng.integers(300, 501))
        start = int(rng.integers(0, max(LENS[tid] - ins // 2, 1)))       # some fragments run past the contig end
        name = "*" if rng.random() < 0.03 else ("frag%d" % f if not one_name else "same")
        l1, l2 = int(rng.integers(100, 151)), int(rng.integers(100, 151))
        cx = rng.random() < 0.1
        odd = rng.random() < 0.1
        f1 = int(rng.choice(ODD_FLAGS)) if odd else FLAGS[int(rng.integers(0, 2)) * 2]
        read(tid, start, strain, l1, name, f1, cx)
        if rng.random() < 0.9:
            read(tid, min(start + ins - l2, LENS[tid] - 1), strain, l2, name, FLAGS[1] if not odd else f1, cx)
        if rng.random() < 0.03:
            read(tid, start + 10, strain, 60, name, 0x800 | 0x1 | 0x40, False)
    for k in range(long_reads):                                         # long reads, > 127 ops
        tid = 2
        pos = int(rng.integers(0, 8000))
        ops = []
        for _j in range(40):
            ops += [(200 << 4) | 0, (1 << 4) | 1, (2 << 4) | 2, (10 << 4) | 8]
        seq = []
        r = pos
        for o in ops:
            op, n = o & 15, o >> 4
            if op in (0, 8):
                seq += ["ACGT"[int(strains[0][tid][r + j])] for j in range(n)]
            elif op == 1:
                seq += ["A"] * n
            if op in (0, 2, 8):
                r += n
        recs.append((tid, pos, 0, ops, "".join(seq), None if k == 2 else [30] * len(seq), "long%d" % k))
    # unplaced records
    for k in range(20):
        recs.append((-1, -1, 0x4, [], "ACGT", None, "un%d" % k))
    recs.sort(key=lambda r: (r[0] & 0xFFFFFFFF, r[1]))
    return recs


def _write(recs, d, name):
    tid, pos, flag, mapq, cig_off, cig, nt16, quals = _columns(recs)
    names = [r[6] for r in recs]
    pb, ps = str(d / (name + ".bam")), str(d / (name + ".sam"))
    bamio.write_bam(pb, REFS, LENS, tid, pos, flag, mapq, cig_off, cig, seqs=nt16, names=names, with_index=False)
    _set_bam_quals(pb, quals)
    samio.write_sam(ps, REFS, LENS, tid, pos, flag, mapq, cig_off, cig, seqs=[r[4] if r[4] else "*" for r in recs],
                    names=names, quals=["*" if r[5] is None else "".join(chr(33 + x) for x in r[5]) for r in recs])
    return pb, ps


_ORACLE = {}


def _oracle(recs, t, cb, **kw):
    params = dict(PARAMS)
    params.update(kw)
    k = (id(recs), t, cb, tuple(sorted(params.items())))
    if k not in _ORACLE:
        tid, pos, flag, _mapq, cig_off, cig, nt16, quals = _columns(recs)
        _ORACLE[k] = ol.linkage(LENS, tid, pos, flag, cig_off, cig, nt16, quals, [r[6].encode() for r in recs],
                                quality_threshold=t, read_callback=cb, **params)
    return _ORACLE[k]


def _rows(pairs):
    return list(zip(pairs["tid"].tolist(), pairs["pos_a"].tolist(), pairs["pos_b"].tolist(),
                    *[[x.decode() for x in pairs[k].tolist()] for k in ("major_a", "minor_a", "major_b", "minor_b")],
                    pairs["n_AB"].tolist(), pairs["n_Ab"].tolist(), pairs["n_aB"].tolist(), pairs["n_ab"].tolist()))


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("linkage")
    out = {}
    for ns in (2, 3):
        recs = _gen(40 + ns, ns)
        rng = np.random.default_rng(50 + ns)
        shuf = [recs[i] for i in rng.permutation(len(recs))]
        pb, ps = _write(recs, d, "s%d" % ns)
        ub, us = _write(shuf, d, "u%d" % ns)
        out[ns] = dict(recs=recs, bam=pb, sam=ps, bam_shuf=ub, sam_shuf=us)
    out["dir"] = d
    return out


@pytest.mark.parametrize("ns", [2, 3])
@pytest.mark.parametrize("fmt", ["bam", "sam"])
@pytest.mark.parametrize("cb", ["all", "nofilter"])
@pytest.mark.parametrize("t", [0, 15])
def test_matches_oracle(files, ns, fmt, cb, t):
    from metacov_b200 import AlignmentFile
    f = files[ns]
    want, info = _oracle(f["recs"], t, cb)
    with AlignmentFile(f[fmt], decode="gpu") as af:
        got, ginfo = af.linkage(quality_threshold=t, read_callback=cb, **PARAMS)
    assert _rows(got) == want
    assert ginfo == info
    assert len(want) > 100 and info["n_units"] > 1000


def test_other_parameters(files):
    from metacov_b200 import AlignmentFile
    f = files[3]
    with AlignmentFile(f["bam"], decode="gpu") as af:
        for kw in (dict(max_distance=1, min_reads=1), dict(max_distance=100000, min_reads=1, min_freq=0.2),
                   dict(max_distance=450, min_reads=10, min_count=3, min_coverage=10)):
            want, info = _oracle(f["recs"], 15, "all", **kw)
            got, ginfo = af.linkage(**dict(PARAMS, **kw))
            assert _rows(got) == want, kw
            assert ginfo == info, kw
        # the defaults
        got, _ = af.linkage()
        want, _ = _oracle(f["recs"], 15, "all", min_coverage=5, min_freq=0.05, min_count=2, max_distance=1000,
                          min_reads=20)
        assert _rows(got) == want


def test_one_unit(tmp_path):
    """Every record under one name: one unit, whatever its size."""
    from metacov_b200 import AlignmentFile
    recs = _gen(61, 2, n_frag=600, one_name=True)
    pb, _ps = _write(recs, tmp_path, "one")
    want, info = _oracle(recs, 0, "all", min_reads=1, min_freq=0.02)
    with AlignmentFile(pb, decode="gpu") as af:
        got, ginfo = af.linkage(quality_threshold=0, **dict(PARAMS, min_reads=1, min_freq=0.02))
    assert _rows(got) == want and ginfo == info
    assert info["n_units"] <= 1 + sum(1 for r in recs if r[6] == "*")


def test_identical_over_formats_orders_and_decoders(files):
    from metacov_b200 import AlignmentFile
    f = files[2]
    runs = {}
    for name in ("bam", "sam", "bam_shuf", "sam_shuf"):
        with AlignmentFile(f[name], decode="gpu") as af:
            runs[name] = af.linkage(**PARAMS)
            again = af.linkage(**PARAMS)
            assert again[0].tobytes() == runs[name][0].tobytes() and again[1] == runs[name][1]
    for decode, kw in (("host", {}), ("gpu-stream", {"gpu_chunk_bytes": 1 << 17})):
        for name in ("bam", "bam_shuf"):
            with AlignmentFile(f[name], decode=decode, **kw) as af:
                runs[name + "_" + decode] = af.linkage(**PARAMS)
    for k, (pairs, info) in runs.items():
        assert pairs.tobytes() == runs["bam"][0].tobytes(), k
        assert info == runs["bam"][1], k


def test_depth_counts_and_sites_left_alone(files):
    from metacov_b200 import AlignmentFile
    f = files[2]
    for decode in ("gpu", "host"):
        with AlignmentFile(f["bam"], decode=decode) as af:
            eng = af.coverage_engine()
            tid = np.arange(3, dtype=np.int32)

            def snap():
                return ([af.count_coverage_depth(c).tobytes() for c in REFS],
                        eng.region_stats(tid, np.zeros_like(tid), np.array(LENS, np.int32)).tobytes(), eng.pass_info(),
                        [np.stack(af.count_coverage(c)).tobytes() for c in REFS],
                        af.allele_sites(min_count=1).tobytes(), af.allele_stats().tobytes())
            s0 = snap()
            ceng = af._count_engine()
            sites0 = ceng.allele_sites(min_count=1)
            af.linkage(**PARAMS)
            af.linkage(min_reads=1, max_distance=5)
            assert ceng.allele_sites(min_count=1).tobytes() == sites0.tobytes()
            from metacov_b200 import _capi
            got = np.zeros(len(sites0), _capi.ALLELE_SITE_DTYPE)
            ceng._check(_capi.lib.mcov_allele_sites_read(ceng._ctx, 0, len(sites0), _capi.ptr(got)))
            assert got.tobytes() == sites0.tobytes()
            assert snap() == s0


def test_errors(files, tmp_path, monkeypatch):
    import ctypes as C
    from metacov_b200 import AlignmentFile, CoverageEngine, McovError, _capi
    from metacov_b200._capi import lib
    f = files[2]
    with AlignmentFile(io.BytesIO(open(f["sam"], "rb").read())) as s:
        with pytest.raises(ValueError, match="read once"):
            s.linkage()
    with AlignmentFile(f["bam"], decode="gpu") as af:
        eng = af._count_engine()
        n = eng.launch_count()
        for bad in (dict(max_distance=0), dict(max_distance=100001), dict(max_distance=1.5), dict(min_reads=0),
                    dict(min_reads=2.5), dict(min_coverage=0), dict(min_count=0), dict(min_freq=1.5),
                    dict(read_callback="mapped")):
            with pytest.raises(ValueError):
                af.linkage(**bad)
        assert eng.launch_count() == n                                   # nothing ran
        want = _rows(af.linkage(**PARAMS)[0])
        # the C level: bad parameters are MCOV_ERR_ARG, the file stays usable
        out = C.c_int64(0)
        for field, v in (("max_distance", 0), ("max_distance", 100001), ("min_reads", 0)):
            p = eng._linkage_params(5, 0.05, 2, 1000, 20)
            setattr(p, field, v)
            assert lib.mcov_linkage(eng._ctx, None, 0, C.byref(p), C.byref(out), None) == _capi.MCOV_ERR_ARG
        p = eng._linkage_params(5, 0.05, 2, 1000, 20)
        p.sites.use_reference = 1
        assert lib.mcov_linkage(eng._ctx, None, 0, C.byref(p), C.byref(out), None) == _capi.MCOV_ERR_ARG
        rec = np.zeros(1, _capi.LINKAGE_PAIR_DTYPE)
        assert lib.mcov_linkage_read(eng._ctx, 0, 1, _capi.ptr(rec)) == _capi.MCOV_ERR_STATE   # (the failed call dropped it)
        got, info = af.linkage(**PARAMS)
        assert lib.mcov_linkage_read(eng._ctx, len(got), 1, _capi.ptr(rec)) == _capi.MCOV_ERR_ARG
        # no SNV sites: an empty result
        empty, info = af.linkage(min_coverage=10 ** 6)
        assert len(empty) == 0 and info["n_sites"] == 0 and info["n_candidates"] == 0
    # the NOMEM hook: MemoryError naming the file and the byte counts, nothing kept, then a good call; resident and
    # streamed records
    for decode in ("gpu", "host"):
        with AlignmentFile(f["bam"], decode=decode) as af:
            monkeypatch.setenv("MCOV_LINK_FREE_BYTES", "1000")
            with pytest.raises(MemoryError, match=r"s2.bam.*needs? \d+ bytes of device memory, \d+ are free"):
                af.linkage(**PARAMS)
            monkeypatch.delenv("MCOV_LINK_FREE_BYTES")
            assert _rows(af.linkage(**PARAMS)[0]) == want
    # later checks: a hook above the site buffers trips the candidate counters (resident records) and, with few
    # candidates and a streamed file of several chunks, the growth of the observation buffer across chunks
    _pairs, info = _oracle(f["recs"], 15, "all")
    with AlignmentFile(f["bam"], decode="gpu") as af:
        monkeypatch.setenv("MCOV_LINK_FREE_BYTES", str(16 * info["n_candidates"] // 2))
        with pytest.raises(MemoryError, match=r"s2.bam.*candidate pairs: need \d+ bytes of device memory, \d+ are free"):
            af.linkage(**PARAMS)
        monkeypatch.delenv("MCOV_LINK_FREE_BYTES")
        assert _rows(af.linkage(**PARAMS)[0]) == want
    near = dict(PARAMS, max_distance=1, min_reads=1)
    with AlignmentFile(f["bam"], decode="gpu-stream", gpu_chunk_bytes=1 << 17) as af:
        monkeypatch.setenv("MCOV_LINK_FREE_BYTES", str(16 * info["n_observations"] // 2))
        with pytest.raises(MemoryError, match=r"s2.bam.*observations: growing their buffer needs \d+ bytes"):
            af.linkage(**near)
        monkeypatch.delenv("MCOV_LINK_FREE_BYTES")
        assert _rows(af.linkage(**near)[0]) == _oracle(f["recs"], 15, "all", max_distance=1, min_reads=1)[0]
    # without counts, and without a decoded file: MCOV_ERR_STATE
    with CoverageEngine(LENS) as eng:
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng.linkage()
        with pytest.raises(McovError, match="MCOV_ERR_STATE"):
            eng._check(lib.mcov_linkage_read(eng._ctx, 0, 0, None))
        eng.base_counts(15, _capi.MCOV_BC_ALL, path=f["bam"])
        with pytest.raises(McovError, match="no file decoded"):
            eng.linkage()
        assert _rows(eng.linkage(path=f["bam"], **PARAMS)[0]) == want


def test_cli(files, tmp_path):
    from click.testing import CliRunner
    from metacov_b200 import AlignmentFile
    from metacov_b200.alleles import derive_linkage
    from metacov_b200.cli import main
    f = files[3]
    out = tmp_path / "l.tsv"
    r = CliRunner().invoke(main, ["linkage", "-b", f["bam"], "-o", str(out), "--max-distance", "600", "--min-reads", "3",
                                  "--min-coverage", "3", "-q", "0"], catch_exceptions=False)
    assert r.exit_code == 0, r.output
    with AlignmentFile(f["bam"], decode="gpu") as af:
        pairs, _ = af.linkage(quality_threshold=0, **PARAMS)
    d = derive_linkage(pairs)
    lines = open(out).read().splitlines()
    assert lines[0].split("\t") == ["contig", "pos_a", "pos_b", "distance", "major_a", "minor_a", "major_b", "minor_b",
                                    "n_AB", "n_Ab", "n_aB", "n_ab", "total", "r2", "d_prime"]
    assert len(lines) - 1 == len(pairs) > 100
    for line, row, r2, dp in zip(lines[1:], _rows(pairs), d["r2"].tolist(), d["d_prime"].tolist()):
        x = line.split("\t")
        t, pa, pb = row[:3]
        assert x[:13] == [REFS[t].split()[0], str(pa), str(pb), str(pb - pa), *row[3:7], *map(str, row[7:]),
                          str(sum(row[7:]))]
        for got, want in ((x[13], r2), (x[14], dp)):
            assert (got == "nan" and want != want) or float(got) == want
    r = CliRunner().invoke(main, ["linkage", "-b", "-", "-o", str(out)], input=open(f["sam"]).read())
    assert r.exit_code != 0 and "piped stream" in r.output


def test_more_than_2_31_slots(tmp_path):
    """Two contigs of 1.5 x 10^9: paired reads around slot 2^31 and near the end of the second contig."""
    from metacov_b200 import AlignmentFile
    L = 1_500_000_000
    refs, lens = ["big0", "big1"], [L, L]
    off1 = (L + 1 + 3) & ~3
    px = (1 << 31) - off1                                   # position of contig 1 at slot 2^31
    rng = np.random.default_rng(31)
    base = {}

    def ref_at(p):
        return "ACGT"[(p * 2654435761 >> 7) % 4]
    var = {p: "ACGT"[("ACGT".index(ref_at(p)) + 1) % 4] for a in (px - 600, L - 1500) for p in range(a, a + 1200, 37)}
    recs = []
    for k in range(400):
        a = (px - 600) if k % 2 else (L - 1500)
        strain = rng.random() < 0.4
        p1 = a + int(rng.integers(0, 500))
        ins = int(rng.integers(300, 501))
        for p, fl in ((p1, 0x41), (min(p1 + ins - 150, L - 150), 0x91)):
            s = "".join(var[q] if (strain and q in var) else ref_at(q) for q in range(p, p + 150))
            recs.append((1, p, fl, [(150 << 4) | 0], s, None, "f%d" % k))
    recs.sort(key=lambda r: r[1])
    tid, pos, flag, mapq, cig_off, cig, nt16, _q = _columns(recs)
    ps = str(tmp_path / "big.sam")                          # (SAM: a BAM bin cannot hold positions past 2^29)
    samio.write_sam(ps, refs, lens, tid, pos, flag, mapq, cig_off, cig, seqs=[r[4] for r in recs],
                    names=[r[6] for r in recs])
    params = dict(min_coverage=5, min_freq=0.05, min_count=2, max_distance=500, min_reads=5)
    with AlignmentFile(ps, decode="gpu") as af:
        eng = af._count_engine()
        got, info = af.linkage(quality_threshold=0, **params)
        assert int(eng.n_slots) > (1 << 31) + 1000
    # the oracle on the reads shifted into two small windows of a small contig each
    rows = []
    for w0 in (px - 2000, L - 3000):
        sel = [r for r in recs if w0 <= r[1] < w0 + 3000]
        sh = [(0, r[1] - w0) + r[2:] for r in sel]
        t2, p2, f2, _m, co, cg, n2, q2 = _columns(sh)
        want, _ = ol.linkage([3000], t2, p2, f2, co, cg, n2, q2, [r[6].encode() for r in sh], quality_threshold=0,
                             **params)
        rows += [(1, w[1] + w0, w[2] + w0) + tuple(w[3:]) for w in want]
    assert _rows(got) == rows and len(rows) > 50
    assert any(r[1] < px < r[2] for r in rows) and any(r[2] > L - 1500 for r in rows)
