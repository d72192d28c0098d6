"""The linkage rules restated in oracle/linkage.py, on the CPU: known answers (perfect linkage, independent sites,
mates that link sites beyond one read, disagreeing mates, third alleles, '*' names), the max_distance / min_reads
boundaries and contig borders, the major / minor alleles at SNV sites over random counts, the read-name key against the
host BAM reader, and ``alleles.derive_linkage``."""
import math

import numpy as np
import pytest

from oracle import alleles as oa
from oracle import bamio
from oracle import linkage as ol

NT16 = {"A": 1, "C": 2, "G": 4, "T": 8, "N": 15}
LENS = [2000, 2000]


def _cols(recs):
    """recs: (name, tid, pos, SEQ letters[, flag[, ops]]) -> the oracle's record arguments (no qualities)."""
    tid = np.array([r[1] for r in recs], np.int32)
    pos = np.array([r[2] for r in recs], np.int32)
    flag = np.array([r[4] if len(r) > 4 else 0 for r in recs], np.uint16)
    ops = [r[5] if len(r) > 5 else [(len(r[3]) << 4) | 0] for r in recs]
    cig_off = np.concatenate(([0], np.cumsum([len(o) for o in ops]))).astype(np.uint32)
    cig = np.array([o for x in ops for o in x], np.uint32)
    seqs = [np.array([NT16[c] for c in r[3]], np.uint8) for r in recs]
    names = [r[0].encode() for r in recs]
    return tid, pos, flag, cig_off, cig, seqs, [None] * len(recs), names


def _run(recs, **kw):
    params = dict(quality_threshold=0, min_coverage=1, min_freq=0.0, min_count=1, max_distance=1000, min_reads=1)
    params.update(kw)
    return ol.linkage(LENS, *_cols(recs), **params)


def _read(base, pos, alleles, length=100):
    """SEQ of `length` bases over `base` (a string of the reference) from pos, with {refpos: letter} put in."""
    s = list(base[pos:pos + length])
    for p, ch in alleles.items():
        if pos <= p < pos + length:
            s[p - pos] = ch
    return "".join(s)


REF = "".join("ACGT"[(i * 7 + i // 5) % 4] for i in range(2000))
S, T = 30, 80          # two sites, both inside one 100 bp read from 0


def _hap(name, a, b, pos=0, tid=0, length=100):
    return (name, tid, pos, _read(REF, pos, {S: a, T: b}, length))


def test_perfect_linkage():
    recs = [_hap("u%d" % k, "A", "C") for k in range(12)] + [_hap("v%d" % k, "G", "T") for k in range(8)]
    pairs, info = _run(recs)
    assert len(pairs) == 1
    t, pa, pb, ma, na, mb, nb, AB, Ab, aB, ab = pairs[0]
    assert (t, pa, pb, ma, na, mb, nb) == (0, S, T, "A", "G", "C", "T")
    assert (AB, Ab, aB, ab) == (12, 0, 0, 8)
    assert info == dict(n_sites=2, n_observations=40, n_units=20, n_candidates=1)
    from metacov_b200.alleles import derive_linkage
    arr = np.array([(AB, Ab, aB, ab, pa, pb)], dtype=[("n_AB", "u4"), ("n_Ab", "u4"), ("n_aB", "u4"), ("n_ab", "u4"),
                                                      ("pos_a", "i4"), ("pos_b", "i4")])
    d = derive_linkage(arr)
    assert d["r2"][0] == 1.0 and d["d_prime"][0] == 1.0 and d["distance"][0] == T - S


def test_independent_sites():
    recs = []
    for a, b, n in (("A", "C", 9), ("A", "T", 6), ("G", "C", 3), ("G", "T", 2)):
        recs += [_hap("%s%s%d" % (a, b, k), a, b) for k in range(n)]
    pairs, _ = _run(recs)
    assert pairs == [(0, S, T, "A", "G", "C", "T", 9, 6, 3, 2)]


def test_mates_link_beyond_one_read():
    far = 400
    recs = []
    for k in range(10):
        a, b = ("A", "C") if k < 6 else ("G", "T")
        recs.append(("p%d" % k, 0, 0, _read(REF, 0, {S: a, far: b}), 0x41))
        recs.append(("p%d" % k, 0, far - 50, _read(REF, far - 50, {S: a, far: b}), 0x81))
    pairs, info = _run(recs)
    assert pairs == [(0, S, far, "A", "G", "C", "T", 6, 0, 0, 4)]
    assert info["n_units"] == 10
    # the same reads under different names link nothing
    pairs, _ = _run([(r[0] + ("a" if i % 2 else "b"),) + r[1:] for i, r in enumerate(recs)])
    assert pairs == []


def test_disagreeing_mates_and_third_alleles():
    recs = [_hap("u%d" % k, "A", "C") for k in range(10)] + [_hap("v%d" % k, "G", "T") for k in range(10)]
    # w: R1 says A at S, R2 (overlapping) says G at S; both say C at T -> no call at S for w
    recs += [("w", 0, 0, _read(REF, 0, {S: "A", T: "C"})), ("w", 0, 10, _read(REF, 10, {S: "G", T: "C"}))]
    # x: a third allele at S (T, seen once) -> no call at S; y: agreeing mates count once
    recs += [_hap("x", "T", "C"), ("y", 0, 0, _read(REF, 0, {S: "A", T: "T"})), ("y", 0, 20, _read(REF, 20, {S: "A", T: "T"}))]
    pairs, info = _run(recs, min_count=2)
    assert pairs == [(0, S, T, "A", "G", "C", "T", 10, 1, 0, 10)]
    assert info["n_units"] == 23


def test_star_names_never_merge():
    recs = []
    for k in range(5):
        recs.append(("*", 0, 0, _read(REF, 0, {S: "A"}, 50)))            # covers S only
        recs.append(("*", 0, 60, _read(REF, 60, {T: "C"}, 50)))          # covers T only
    recs += [_hap("u%d" % k, "G", "T") for k in range(5)]
    pairs, info = _run(recs)
    assert pairs == [(0, S, T, "A", "G", "C", "T", 0, 0, 0, 5)]
    assert info["n_units"] == 15
    named = [("n%d" % (i // 2),) + r[1:] for i, r in enumerate(recs[:10])] + recs[10:]
    assert _run(named)[0] == [(0, S, T, "A", "G", "C", "T", 5, 0, 0, 5)]


def test_max_distance_contigs_and_min_reads():
    N = 200
    recs = []
    for k in range(6):
        a, b = ("A", "C") if k % 2 else ("G", "T")
        recs.append(("m%d" % k, 0, 0, _read(REF, 0, {S: a, S + N: b}, 300)))
        recs.append(("m%d" % k, 1, 0, _read(REF, 0, {S: a}, 300)))       # the mate on contig 1: same unit, no pair across
    for md, want in ((N, 1), (N - 1, 0), (N + 1, 1)):
        pairs, info = _run(recs, max_distance=md)
        assert len(pairs) == want, md
        assert info["n_candidates"] == want
    for mr, want in ((6, 1), (7, 0)):
        assert len(_run(recs, max_distance=N, min_reads=mr)[0]) == want


def test_skipped_records_and_qualities():
    recs = [_hap("u%d" % k, "A", "C") for k in range(4)] + [_hap("v%d" % k, "G", "T") for k in range(4)]
    recs += [_hap("d%d" % k, "A", "T") + (0x400,) for k in range(3)]     # duplicates: skipped under "all"
    assert _run(recs, min_count=2)[0] == [(0, S, T, "A", "G", "C", "T", 4, 0, 0, 4)]
    # counted, the duplicates make T the major allele at the second site
    assert _run(recs, min_count=2, read_callback="nofilter")[0] == [(0, S, T, "A", "G", "T", "C", 3, 4, 4, 0)]
    # a threshold: records without qualities give nothing
    assert _run(recs, quality_threshold=15)[0] == []


def test_major_minor_present_over_random_counts():
    rng = np.random.default_rng(5)
    for trial in range(40):
        c = rng.integers(0, 40, (4, 3000)) * (rng.random((4, 3000)) < 0.6)
        params = dict(min_coverage=int(rng.integers(1, 10)), min_freq=float(rng.random() * 0.3),
                      min_count=int(rng.integers(1, 6)))
        sl = ol.sites([c], **params)
        e = oa.evaluate(c, None, **params)
        assert [s[1] for s in sl] == np.nonzero(e["kind"] & 1)[0].tolist()
        for _t, p, major, minor in sl:
            assert major != minor
            assert e["present"][major, p] and e["present"][minor, p], (trial, p)
            assert major == int(np.argmax(c[:, p]))
            others = [b for b in range(4) if b != major]
            assert minor == others[int(np.argmax(c[others, p]))]


def test_name_key_matches_host_reader(tmp_path):
    from metacov_b200 import AlignmentFile
    names = ["r1", "*", "a" * 254, "SRR123.4/1", "x y", "é"]
    n = len(names)
    pb = str(tmp_path / "names.bam")
    bamio.write_bam(pb, ["c0"], [100], np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint16),
                    np.full(n, 30, np.uint8), np.arange(n + 1, dtype=np.uint32), np.full(n, (10 << 4), np.uint32),
                    names=names, seqs=[np.full(10, 1, np.uint8)] * n, with_index=False)
    with AlignmentFile(pb, decode="host") as af:
        assert af.name_hashes().tolist() == [ol.name_key(x.encode()) for x in names]
    assert ol.name_key(b"") == 1469598103934665603


def test_bad_params():
    for kw in (dict(max_distance=0), dict(max_distance=100001), dict(max_distance=2.5), dict(min_reads=0),
               dict(min_coverage=0), dict(min_freq=1.5)):
        with pytest.raises(ValueError):
            _run([_hap("u", "A", "C")], **kw)


def test_derive_linkage():
    from metacov_b200.alleles import derive_linkage
    dt = [("pos_a", "i4"), ("pos_b", "i4"), ("n_AB", "u4"), ("n_Ab", "u4"), ("n_aB", "u4"), ("n_ab", "u4")]
    recs = np.array([(10, 25, 9, 2, 3, 6),       # D > 0
                     (0, 1, 1, 7, 4, 8),         # D < 0
                     (5, 9, 0, 0, 0, 0),         # no units
                     (5, 9, 4, 0, 3, 0),         # p_B = 1: r2 and D' divide by zero
                     (5, 9, 4, 4, 4, 4)],        # D = 0
                    dtype=dt)
    d = derive_linkage(recs)
    for k, r in enumerate(recs):
        ab, a_b, ab_, ab2 = (float(r[x]) for x in ("n_AB", "n_Ab", "n_aB", "n_ab"))
        tot = ab + a_b + ab_ + ab2
        assert d["distance"][k] == r["pos_b"] - r["pos_a"]
        if tot == 0:
            assert math.isnan(d["r2"][k]) and math.isnan(d["d_prime"][k])
            continue
        pa, pb = (ab + a_b) / tot, (ab + ab_) / tot
        D = ab / tot - pa * pb
        den = pa * (1 - pa) * pb * (1 - pb)
        dmax = min(pa * (1 - pb), (1 - pa) * pb) if D > 0 else min(pa * pb, (1 - pa) * (1 - pb))
        assert (math.isnan(d["r2"][k]) if den == 0 else math.isclose(d["r2"][k], D * D / den, rel_tol=1e-12))
        assert (math.isnan(d["d_prime"][k]) if dmax == 0 else math.isclose(d["d_prime"][k], abs(D) / dmax, rel_tol=1e-12,
                                                                            abs_tol=1e-15))
    assert d["d_prime"][0] > 0.1 and d["d_prime"][1] > 0.1 and d["d_prime"][4] == 0 and d["r2"][4] == 0
    assert math.isnan(d["r2"][3])
