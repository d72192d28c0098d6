"""The comparison rules of oracle/compare.py worked by hand, their invariants over random counts, derive_compare and the
CLI's argument errors; no GPU."""
import math

import numpy as np
import pytest

from oracle import compare as oc


def _counts(*cols):
    return np.array(cols, dtype=np.uint32).T          # columns (A, C, G, T) -> [4, n]


def test_signature_by_hand():
    c = _counts((10, 0, 0, 0),        # A only
                (5, 5, 0, 0),         # tie A / C: consensus A, both present
                (0, 0, 3, 1),         # N = 4 < 5: not covered
                (1, 1, 1, 3),         # N = 6: only T reaches min_count 2 -> mask T, consensus T
                (0, 0, 0, 0))
    sig = oc.signature(c, min_coverage=5, min_freq=0.05, min_count=2)
    assert sig.tolist() == [0x80 | 0x01, 0x80 | 0x03, 0, 0x80 | (3 << 4) | 0x08, 0]
    # min_count above every count: covered with an empty present mask, the consensus still set
    sig = oc.signature(_counts((6, 4, 0, 0), (0, 0, 2, 9)), min_coverage=5, min_count=100)
    assert sig.tolist() == [0x80, 0x80 | (3 << 4)]
    assert oc.allele_sets(sig).tolist() == [0x01, 0x08]
    # min_freq: 1 of 30 reads is below 0.05
    assert oc.signature(_counts((29, 1, 0, 0)), min_count=1).tolist() == [0x81]
    assert oc.signature(_counts((29, 1, 0, 0)), min_count=1, min_freq=0.0).tolist() == [0x83]


def test_pair_rules_by_hand():
    A, C, G, T = 0, 1, 2, 3

    def s(cons, mask):
        return 0x80 | (cons << 4) | mask

    a = np.array([s(A, 1), s(A, 1), s(A, 0b0011), s(A, 0), s(G, 0), 0, s(T, 8)], np.uint8)
    b = np.array([s(A, 1), s(C, 2), s(C, 0b0011), s(C, 0), s(G, 4), s(A, 1), 0], np.uint8)
    cov_a, cov_b, cmp_, con, pop = oc.pair_flags(a, b)
    assert cmp_.tolist() == [1, 1, 1, 1, 1, 0, 0]
    assert con.tolist() == [0, 1, 1, 1, 0, 0, 0]
    # {A} vs {C}: disjoint; {A, C} vs {A, C}: shared; empty masks fall back to the consensus: {A} vs {C}
    assert pop.tolist() == [0, 1, 0, 1, 0, 0, 0]
    r = oc.pair_region(a, b, 0, 10)
    assert r == dict(length=10, covered_a=6, covered_b=6, compared=5, con_snp=3, pop_snp=2)
    assert oc.pair_region(a, b, 2, 2)["length"] == 0 and oc.pair_region(a, b, 9, 12)["compared"] == 0
    assert oc.pair_sites([a], [b], pair=4) == [(4, 0, 1, int(a[1]), int(b[1]), 3), (4, 0, 2, int(a[2]), int(b[2]), 1),
                                                (4, 0, 3, int(a[3]), int(b[3]), 3)]


def _random_counts(rng, n):
    c = rng.integers(0, 12, (4, n)).astype(np.uint32)
    c[:, rng.random(n) < 0.2] = 0
    hot = rng.random(n) < 0.3
    c[rng.integers(0, 4, n)[hot], np.nonzero(hot)[0]] += rng.integers(5, 60, int(hot.sum())).astype(np.uint32)
    return c


@pytest.mark.parametrize("params", [dict(), dict(min_coverage=1, min_freq=0.0, min_count=1),
                                    dict(min_coverage=20, min_freq=0.3, min_count=5), dict(min_count=1000)])
def test_invariants_over_random_counts(params):
    rng = np.random.default_rng(5)
    a, b = _random_counts(rng, 20000), _random_counts(rng, 20000)
    sa, sb = oc.signature(a, **params), oc.signature(b, **params)
    _ca, _cb, cmp_, con, pop = oc.pair_flags(sa, sb)
    assert not (pop & ~con).any()                       # a pop_snp is always a con_snp
    assert (oc.allele_sets(sa)[(sa & 0x80) != 0] != 0).all()
    assert con.any()
    # a against itself: nothing differs, every covered position is compared
    r = oc.pair_region(sa, sa, 0, len(sa))
    assert r["con_snp"] == r["pop_snp"] == 0 and r["compared"] == r["covered_a"] == r["covered_b"]
    # (a, b) mirrors (b, a)
    ab, ba = oc.pair_region(sa, sb, 100, 19000), oc.pair_region(sb, sa, 100, 19000)
    assert (ab["covered_a"], ab["covered_b"]) == (ba["covered_b"], ba["covered_a"])
    assert all(ab[k] == ba[k] for k in ("length", "compared", "con_snp", "pop_snp"))
    s_ab, s_ba = oc.pair_sites([sa], [sb]), oc.pair_sites([sb], [sa])
    assert [(t, p, x, y, k) for _, t, p, x, y, k in s_ab] == [(t, p, y, x, k) for _, t, p, x, y, k in s_ba]
    assert len(s_ab) == int(con.sum())


def test_derive_compare():
    from metacov_b200.alleles import COMPARE_DERIVED, derive_compare
    from metacov_b200._capi import COMPARE_STATS_DTYPE
    s = np.zeros(3, COMPARE_STATS_DTYPE)
    s["length"] = [100, 0, 50]
    s["compared"] = [80, 0, 0]
    s["con_snp"] = [4, 0, 0]
    s["pop_snp"] = [1, 0, 0]
    d = derive_compare(s)
    assert sorted(d) == sorted(COMPARE_DERIVED)
    assert d["con_ani"][0] == 1 - 4 / 80 and d["pop_ani"][0] == 1 - 1 / 80 and d["percent_compared"][0] == 0.8
    for k in ("con_ani", "pop_ani", "percent_compared"):
        assert math.isnan(d[k][1])
    assert math.isnan(d["con_ani"][2]) and d["percent_compared"][2] == 0.0


def test_cli_argument_errors(tmp_path):
    from click.testing import CliRunner
    from metacov_b200.cli import main
    p = tmp_path / "x.sam"
    p.write_text("@SQ\tSN:c0\tLN:10\n")
    r = CliRunner().invoke(main, ["compare", "-b", str(p)])
    assert r.exit_code == 2 and "at least two files" in r.output
    r = CliRunner().invoke(main, ["compare", "-b", str(p), "-b", "-"])
    assert r.exit_code == 2 and "piped stream" in r.output


def test_site_records_have_no_undefined_bytes():
    """Every byte of a site record is a field, so a masked copy of a site list has the bytes of its source."""
    from metacov_b200._capi import COMPARE_SITE_DTYPE
    assert sum(COMPARE_SITE_DTYPE[k].itemsize for k in COMPARE_SITE_DTYPE.names) == COMPARE_SITE_DTYPE.itemsize == 16
    a = np.zeros(3000, COMPARE_SITE_DTYPE)
    a["pair"] = np.arange(3000) % 3
    a["kind"] = 1
    for _ in range(20):
        junk = np.full(1 << 16, 0x5A, np.uint8)
        del junk
        b = a[a["pair"] == 1].copy()
        assert b.tobytes() == a[1::3].tobytes()
