"""The linkage rules of ``AlignmentFile.linkage`` (include/metacov_b200.h, mcov_linkage) restated as plain loops over
decoded records: the reference the device pairs are checked against.  Test infrastructure only: the product never
imports it.

Records are given as in ``oracle/basecount.py`` (columns tid, pos, flag, cig_off, cig; SEQ as nt16 codes; QUAL as Phred
values or None) plus each record's QNAME as bytes.

Sites.  The SNV sites (kind bit 1) of the counts for (quality_threshold, read_callback) under (min_coverage, min_freq,
min_count), exactly the kind-1 sites of ``allele_sites`` without a reference.  The major allele is the consensus (the
largest count, ties to the first of A C G T), the minor allele the largest count among the other three (same tie rule).

Units.  The records the counts count, grouped by the FNV-1a 64 of QNAME with ~0 folded to ~0 - 1 (``name_key``): mates
and supplementary pieces are one unit, and so are two names whose keys collide (odds of about 2^-64 for a pair of
names; for a file of n names about n^2 / 2^65).  A record named '*' is a unit of its own.

Calls.  A record gives a base at a site when the site is the reference position of one of its M / = / X pairs, the base
is A, C, G or T and, with a non-zero threshold, its quality is at least the threshold.  A unit calls 0 (major) or 1
(minor) at a site when all its bases there are that allele; a disagreement or a third allele is no call.

Pairs.  Sites s < t of one contig with 0 < pos_t - pos_s <= max_distance; each unit with calls at both adds one to
n[call_s][call_t]: n_AB, n_Ab, n_aB, n_ab (upper case = major).  Listed when the total is at least min_reads, in
(tid, pos_a, pos_b) order.  Every field is an integer or a letter.
"""
from collections import defaultdict

import numpy as np

from . import alleles as oa
from . import basecount

ACGT = "ACGT"


def name_key(name):
    """FNV-1a 64 of a read name's bytes, ~0 folded to ~0 - 1 (the key the decoders give ``pileup.experimental``)."""
    h = 1469598103934665603
    for b in bytes(name):
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h - 1 if h == 0xFFFFFFFFFFFFFFFF else h


def check_params(max_distance=1000, min_reads=20, **allele_params):
    oa.check_params(**allele_params)
    if int(max_distance) != max_distance or not 1 <= max_distance <= 100000:
        raise ValueError("max_distance must be an integer in [1, 100000]")
    if int(min_reads) != min_reads or min_reads < 1:
        raise ValueError("min_reads must be an integer >= 1")


def site_alleles(counts):
    """(major, minor) allele codes (0-3) of count columns [4, n]: the consensus and the largest of the other three."""
    c = np.asarray(counts, dtype=np.int64).reshape(4, -1)
    major = np.argmax(c, axis=0)
    other = c.copy()
    other[major, np.arange(c.shape[1])] = -1
    return major, np.argmax(other, axis=0)


def sites(counts_per_contig, min_coverage=5, min_freq=0.05, min_count=2):
    """The SNV sites in (tid, pos) order: list of (tid, pos, major, minor)."""
    out = []
    for t, c in enumerate(counts_per_contig):
        e = oa.evaluate(c, None, min_coverage=min_coverage, min_freq=min_freq, min_count=min_count)
        pos = np.nonzero(e["kind"] & oa.SNV)[0]
        major, minor = site_alleles(np.asarray(c)[:, pos])
        out += [(t, int(p), int(a), int(b)) for p, a, b in zip(pos.tolist(), major.tolist(), minor.tolist())]
    return out


def observations(lengths, tid, pos, flag, cig_off, cig, seqs, quals, names, site_list, quality_threshold=15,
                 read_callback="all"):
    """Every (unit, site index, base code) a counted record gives, in record order.  A unit is the name's key, or
    ("*", record index) for a record named '*'."""
    mode = basecount._mode(read_callback)
    t = int(quality_threshold or 0)
    index = {(s[0], s[1]): k for k, s in enumerate(site_list)}
    out = []
    for i in range(len(tid)):
        c, p = int(tid[i]), int(pos[i])
        if c < 0 or c >= len(lengths) or p < 0:
            continue
        if mode == "all" and int(flag[i]) & basecount.SKIP_ALL:
            continue
        seq = np.asarray(seqs[i], dtype=np.uint8)
        if len(seq) == 0:
            continue
        ops = [int(x) for x in cig[int(cig_off[i]):int(cig_off[i + 1])]]
        if sum(o >> 4 for o in ops if o & 15 in basecount.CONSUMES_QUERY) > len(seq):
            raise IndexError("record %d: its CIGAR consumes more query bases than SEQ holds" % i)
        qual = quals[i]
        if t != 0 and qual is None:
            continue
        unit = ("*", i) if bytes(names[i]) == b"*" else name_key(names[i])
        length = int(lengths[c])
        q, r = 0, p
        for o in ops:
            op, n = o & 15, o >> 4
            if op in basecount.ALIGNED:
                for j in range(n):
                    if r + j >= length:
                        break
                    k = index.get((c, r + j))
                    if k is None:
                        continue
                    b = int(seq[q + j])
                    if b not in basecount.BASE_INDEX or (t != 0 and not qual[q + j] >= t):
                        continue
                    out.append((unit, k, basecount.BASE_INDEX[b]))
            if op in basecount.CONSUMES_QUERY:
                q += n
            if op in basecount.CONSUMES_REF:
                r += n
    return out


def unit_calls(obs, site_list):
    """{unit: sorted list of (site index, call)} from the observations."""
    bases = defaultdict(set)
    for unit, k, b in obs:
        bases[(unit, k)].add(b)
    calls = defaultdict(list)
    for (unit, k), bs in bases.items():
        if len(bs) != 1:
            continue
        b = next(iter(bs))
        _t, _p, major, minor = site_list[k]
        if b == major:
            calls[unit].append((k, 0))
        elif b == minor:
            calls[unit].append((k, 1))
    for v in calls.values():
        v.sort()
    return calls


def candidates(site_list, max_distance):
    """Number of site pairs s < t of one contig with pos_t - pos_s <= max_distance."""
    n = 0
    by_contig = defaultdict(list)
    for t, p, _a, _b in site_list:
        by_contig[t].append(p)
    for ps in by_contig.values():
        ps = np.asarray(ps, dtype=np.int64)
        n += int((np.searchsorted(ps, ps + max_distance, side="right") - np.arange(1, len(ps) + 1)).sum())
    return n


def linkage(lengths, tid, pos, flag, cig_off, cig, seqs, quals, names, quality_threshold=15, read_callback="all",
            min_coverage=5, min_freq=0.05, min_count=2, max_distance=1000, min_reads=20):
    """(pairs, info): pairs a list of (tid, pos_a, pos_b, major_a, minor_a, major_b, minor_b, n_AB, n_Ab, n_aB, n_ab)
    with the alleles as letters, in (tid, pos_a, pos_b) order; info the dict n_sites, n_observations, n_units,
    n_candidates of ``mcov_linkage_info``."""
    check_params(max_distance, min_reads, min_coverage=min_coverage, min_freq=min_freq, min_count=min_count)
    counts = basecount.full_counts(lengths, tid, pos, flag, cig_off, cig, seqs, quals, quality_threshold, read_callback)
    sl = sites(counts, min_coverage, min_freq, min_count)
    obs = observations(lengths, tid, pos, flag, cig_off, cig, seqs, quals, names, sl, quality_threshold, read_callback)
    calls = unit_calls(obs, sl)
    n = defaultdict(lambda: [0, 0, 0, 0])
    for cl in calls.values():
        for x, (s, cs) in enumerate(cl):
            ts, ps = sl[s][0], sl[s][1]
            for t, ct in cl[x + 1:]:
                if sl[t][0] != ts or sl[t][1] - ps > max_distance:
                    break
                n[(s, t)][2 * cs + ct] += 1
    pairs = []
    for (s, t) in sorted(n):
        v = n[(s, t)]
        if sum(v) >= min_reads:
            a, b = sl[s], sl[t]
            pairs.append((a[0], a[1], b[1], ACGT[a[2]], ACGT[a[3]], ACGT[b[2]], ACGT[b[3]], v[0], v[1], v[2], v[3]))
    info = dict(n_sites=len(sl), n_observations=len(obs), n_units=len({u for u, _k, _b in obs}),
                n_candidates=candidates(sl, max_distance))
    return pairs, info
