"""The comparison rules of ``metacov_b200.compare`` (include/metacov_b200.h, mcov_allele_signature / mcov_compare_*)
restated over count arrays with numpy, on top of ``oracle.alleles.evaluate``: the reference the device results are
checked against.  Test infrastructure only: the product never imports it.

Signature of a position (one byte): 0x80 covered (N >= min_coverage), bits 4-5 the consensus (0-3 = A C G T, ties to
the first), bits 0-3 the present mask (n_b >= min_count and n_b >= min_freq * N); 0x00 where not covered.

For a pair (a, b) at a position: compared = covered in both; the allele set of a sample is its present mask OR the bit
of its consensus; con_snp = compared and the consensuses differ; pop_snp = compared and the allele sets are disjoint.
"""
import numpy as np

from . import alleles as oa

CON_SNP, POP_SNP = 1, 2


def signature(counts, min_coverage=5, min_freq=0.05, min_count=2):
    """uint8 [n] signatures of counts [4, n]."""
    e = oa.evaluate(counts, None, min_coverage=min_coverage, min_freq=min_freq, min_count=min_count)
    mask = np.zeros(len(e["covered"]), np.uint8)
    for b in range(4):
        mask |= (e["present"][b].astype(np.uint8) << b)
    sig = 0x80 | (e["consensus"].astype(np.uint8) << 4) | mask
    return np.where(e["covered"], sig, 0).astype(np.uint8)


def allele_sets(sig):
    """The allele set of each signature byte: present mask | (1 << consensus)."""
    s = np.asarray(sig, np.uint8)
    return (s & 0x0F) | (np.uint8(1) << ((s >> 4) & 3)).astype(np.uint8)


def pair_flags(sig_a, sig_b):
    """(covered_a, covered_b, compared, con_snp, pop_snp) as bool arrays of two signature arrays."""
    a, b = np.asarray(sig_a, np.uint8), np.asarray(sig_b, np.uint8)
    cov_a, cov_b = (a & 0x80) != 0, (b & 0x80) != 0
    compared = cov_a & cov_b
    con = compared & (((a >> 4) & 3) != ((b >> 4) & 3))
    pop = compared & ((allele_sets(a) & allele_sets(b)) == 0)
    return cov_a, cov_b, compared, con, pop


def pair_region(sig_a, sig_b, start, end):
    """The record of region [start, end) of one contig (signatures of the contig's positions): positions past the
    contig end are not covered."""
    n = len(sig_a)
    lo, hi = min(start, n), min(end, n)
    cov_a, cov_b, cmp_, con, pop = pair_flags(sig_a[lo:hi], sig_b[lo:hi])
    return dict(length=int(end - start), covered_a=int(cov_a.sum()), covered_b=int(cov_b.sum()),
                compared=int(cmp_.sum()), con_snp=int(con.sum()), pop_snp=int(pop.sum()))


def pair_sites(sigs_a, sigs_b, pair=0):
    """Every con_snp position of a pair, by (tid, pos): a list of (pair, tid, pos, sig_a, sig_b, kind) with kind
    CON_SNP | POP_SNP bits.  sigs_a / sigs_b: one signature array per contig."""
    out = []
    for t, (a, b) in enumerate(zip(sigs_a, sigs_b)):
        _ca, _cb, _cmp, con, pop = pair_flags(a, b)
        for p in np.nonzero(con)[0].tolist():
            out.append((pair, t, p, int(a[p]), int(b[p]), CON_SNP | (POP_SNP if pop[p] else 0)))
    return out
