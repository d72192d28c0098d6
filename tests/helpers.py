"""Shared test helpers (tests may use oracle/; the product package may not)."""
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def load_soa(name):
    from metacov_b200.engine import ReadBatch
    z = np.load(os.path.join(GOLD, name), allow_pickle=False)
    batch = ReadBatch(z["tid"], z["pos"], z["flag"], z["mapq"], z["cig_off"].astype(np.uint32), z["cig"])
    return z, batch


def write_fixture_bam(path):
    """The reference's fixture BAM (tests/data/bbmap.sorted.bam, 4 112 reads on ref1 / ref2), rebuilt by the oracle's
    writer from the columns decoded from it (golden/fixture_soa.npz): names, sequences, insert sizes.  Qualities are
    0xff and the optional fields (AM:C, XT:A, RG:Z, of varying length) are SYNTHETIC stand-ins, not the fixture's:
    they only give every record an optional-field block for the readers to step over.  The BAI carries only the
    metadata pseudo-bins.  Writes path + ".bai" too."""
    from oracle import bamio
    z = np.load(os.path.join(GOLD, "fixture_soa.npz"), allow_pickle=False)
    so = z["seq_off"]
    n = len(z["tid"])
    aux = [b"AMC" + bytes([int(z["mapq"][i])]) + b"XTA" + (b"U" if z["mapq"][i] else b"R") +
           b"RGZ" + b"lane%d\0" % (i % 11 * 7) for i in range(n)]
    bamio.write_bam(path, [str(x) for x in z["references"]], z["lengths"].tolist(), z["tid"], z["pos"], z["flag"],
                    z["mapq"], z["cig_off"], z["cig"], l_seq=z["l_seq"], isize=z["isize"], names=[str(x) for x in z["names"]],
                    seqs=[z["seq"][so[i]:so[i + 1]] for i in range(n)], aux=aux)
    return path


def load_json(name):
    with open(os.path.join(GOLD, name)) as fh:
        return json.load(fh)


def fake_bam(z):
    """oracle FakeAlignmentFile over a golden SoA npz."""
    from oracle import bamio
    from oracle.pysam_boundary import FakeAlignmentFile
    r = bamio.BamRecords()
    r.tid, r.pos, r.flag, r.mapq = z["tid"], z["pos"], z["flag"], z["mapq"]
    r.cig_off = z["cig_off"].astype(np.int64)
    r.cig = z["cig"]
    n = len(r.tid)
    r.l_seq = z["l_seq"] if "l_seq" in z else np.zeros(n, np.int32)
    r.isize = z["isize"] if "isize" in z else np.zeros(n, np.int32)
    r.names = list(z["names"]) if "names" in z else [""] * n
    if "seq" in z:
        so = z["seq_off"]
        r.seqs = [z["seq"][so[i]:so[i + 1]] for i in range(n)]
    else:
        r.seqs = [np.zeros(0, np.uint8)] * n
    r.reflen = bamio.cigar_reflen(r.cig_off, r.cig)
    hdr = bamio.BamHeader("", tuple(str(x) for x in z["references"]), tuple(int(x) for x in z["lengths"]))
    return FakeAlignmentFile(hdr, r)


def regions_of(gold, references):
    refs = [str(x) for x in references]
    tid = [refs.index(r["ref"]) for r in gold["classic"]]
    start = [r["start"] for r in gold["classic"]]
    end = [r["end"] for r in gold["classic"]]
    return tid, start, end


def assert_classic_equal(got, want, where=""):
    """Bit-exact for the integer outputs; floats: 1e-6 relative before rounding is the
    north_star contract, after the reference's round(.,2) they must agree to the cent."""
    for k in ("min", "max", "med", "sum"):
        assert int(got[k]) == int(want[k]), (where, k, got[k], want[k])
    for k in ("std", "avg", "q23"):
        assert abs(float(got[k]) - float(want[k])) <= 0.01 + 1e-9, (where, k, got[k], want[k])
    for k in ("avg", "q23"):
        assert float(got[k]) == float(want[k]), (where, k, got[k], want[k])


def exp_value(v):
    """Golden JSON stores nan / inf as strings."""
    return float(v) if isinstance(v, str) else v


def assert_experimental_equal(got, want, where=""):
    """``experimental`` outputs.  Integer-derived keys must be identical; keys made of float sums
    (north_star: 1e-6 relative) are compared before rounding where possible, and to one unit of
    the reference's round(., 3) after it."""
    import math
    assert set(got) == set(want), (where, sorted(got), sorted(want))
    for k in ("den", "ambig", "improper", "nzef", "gc", "cov2"):
        g, w = float(got[k]), exp_value(want[k])
        assert g == w or (math.isnan(g) and math.isnan(w)), (where, k, got[k], want[k])
    for k in ("cov", "covc"):
        g, w = float(got[k]), exp_value(want[k])
        if math.isnan(w) or math.isinf(w):          # k-mer ratios of 0/0 or x/0 propagate (garbage in, same garbage out)
            assert (math.isnan(g) and math.isnan(w)) or g == w, (where, k, g, w)
        else:
            assert abs(g - w) <= 1e-9 * max(1.0, abs(w)), (where, k, g, w)
    for k in ("denc", "cf", "wnf", "ecor", "cov3"):
        g, w = float(got[k]), exp_value(want[k])
        if math.isnan(w) or math.isinf(w):
            assert (math.isnan(g) and math.isnan(w)) or g == w, (where, k, g, w)
        else:
            assert abs(g - w) <= 0.001 + 1e-6 * abs(w) + 1e-9, (where, k, g, w)
