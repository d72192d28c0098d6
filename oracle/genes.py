"""The gene rules of ``AlignmentFile.gene_stats`` (include/metacov_b200.h, mcov_gene_run) restated with numpy on top of
``oracle/alleles.evaluate``: the reference the device records and site lists are checked against.  Test infrastructure
only: the product never imports it.

A gene is (tid, start, end, strand +1 / -1, phase 0-2), 0-based half-open.  Its codons are read from its 5' end after
``phase`` bases (from ``start`` on +, back from ``end`` on -), K = (end - start - phase) // 3 of them; on - the bases are
complemented.  A codon is called when its three positions are covered and their reference bases known.  Over called
codons: n3 / s3 (Nei-Gojobori in thirds, '*' an amino acid), SNV positions typed by the major and minor allele, SUB
positions by the reference and the consensus, M for a codon with two or more of the kind.
"""
import numpy as np

from . import alleles as oa

# The standard code in TCAG order (first base slowest)
STANDARD_CODE = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
_TCAG = "TCAG"
SNV, SUB = 1, 2
RECORD_FIELDS = ("length", "codons", "codons_called", "n_sites3", "s_sites3", "snv_n", "snv_s", "snv_m",
                 "sub_n", "sub_s", "sub_m")


def codon_table():
    """(aa, n3, s3): 64 entries each, indexed by the codon's A C G T codes (16 b0 + 4 b1 + b2, b0 the 5' base)."""
    aa = []
    for c in range(64):
        b = ("ACGT"[c >> 4], "ACGT"[(c >> 2) & 3], "ACGT"[c & 3])
        aa.append(STANDARD_CODE[16 * _TCAG.index(b[0]) + 4 * _TCAG.index(b[1]) + _TCAG.index(b[2])])
    n3 = []
    for c in range(64):
        n = 0
        for p in range(3):
            sh = 4 - 2 * p
            for x in range(4):
                if x != (c >> sh) & 3 and aa[(c & ~(3 << sh)) | (x << sh)] != aa[c]:
                    n += 1
        n3.append(n)
    return aa, n3, [9 - n for n in n3]


AA, N3, S3 = codon_table()


def _code(bases):
    return 16 * int(bases[0]) + 4 * int(bases[1]) + int(bases[2])


def check_gene(lengths, tid, start, end, strand, phase):
    if not 0 <= tid < len(lengths):
        raise ValueError("gene on contig %d of %d" % (tid, len(lengths)))
    if not 0 <= start < end <= int(lengths[tid]):
        raise ValueError("gene [%d, %d) outside contig %d of length %d" % (start, end, tid, int(lengths[tid])))
    if strand not in (1, -1):
        raise ValueError("strand must be +1 or -1, got %r" % (strand,))
    if phase not in (0, 1, 2):
        raise ValueError("phase must be 0, 1 or 2, got %r" % (phase,))


def genes(counts_per_contig, refs, gene_list, min_coverage=5, min_freq=0.05, min_count=2):
    """(records, sites): a dict of RECORD_FIELDS per gene, and every (gene, classified position) as a tuple (gene, tid,
    pos, codon, codon_pos, ref codon letters, major, minor, aa_ref, aa_major, aa_minor, kind, snv_type, sub_type) in
    (gene, pos) order; letters are str, '' where a field does not apply (minor and aa_minor off SNV positions, a type
    of the other kind)."""
    if refs is None:
        raise ValueError("the gene rules need a reference")
    lengths = [np.asarray(c).shape[1] for c in counts_per_contig]
    evals = {}
    records, sites = [], []
    for g, (tid, start, end, strand, phase) in enumerate(gene_list):
        check_gene(lengths, tid, start, end, strand, phase)
        if tid not in evals:
            evals[tid] = oa.evaluate(counts_per_contig[tid], refs[tid], min_coverage, min_freq, min_count)
        e = evals[tid]
        c = np.asarray(counts_per_contig[tid], dtype=np.int64)
        k_codons = max(end - start - phase, 0) // 3
        rec = dict.fromkeys(RECORD_FIELDS, 0)
        rec["length"], rec["codons"] = end - start, k_codons
        rows = []
        for k in range(k_codons):
            # genomic positions of codon positions 0, 1, 2 (5' to 3')
            if strand == 1:
                pos = [start + phase + 3 * k + j for j in range(3)]
            else:
                pos = [end - phase - 3 * k - 1 - j for j in range(3)]
            if not all(e["covered"][p] and e["ref"][p] < 4 for p in pos):
                continue

            def orient(b):
                return int(b) if strand == 1 else 3 - int(b)
            ref_codon = [orient(e["ref"][p]) for p in pos]
            r_code = _code(ref_codon)
            rec["codons_called"] += 1
            rec["n_sites3"] += N3[r_code]
            rec["s_sites3"] += S3[r_code]
            snv = [bool(e["kind"][p] & oa.SNV) for p in pos]
            sub = [bool(e["kind"][p] & oa.SUB) for p in pos]
            for j, p in enumerate(pos):
                if not (snv[j] or sub[j]):
                    continue
                major = int(e["consensus"][p])
                others = c[:, p].copy()
                others[major] = -1
                minor = int(np.argmax(others))                    # (ties: the first of A C G T)
                with_major = list(ref_codon)
                with_major[j] = orient(major)
                with_minor = list(ref_codon)
                with_minor[j] = orient(minor)
                aa_major = AA[_code(with_major)]
                snv_type = sub_type = ""
                if snv[j]:
                    snv_type = "M" if sum(snv) >= 2 else ("S" if aa_major == AA[_code(with_minor)] else "N")
                    rec["snv_" + snv_type.lower()] += 1
                if sub[j]:
                    sub_type = "M" if sum(sub) >= 2 else ("S" if aa_major == AA[r_code] else "N")
                    rec["sub_" + sub_type.lower()] += 1
                rows.append((g, tid, p, k, j, "".join("ACGT"[b] for b in ref_codon), "ACGT"[major],
                             "ACGT"[minor] if snv[j] else "", AA[r_code], aa_major,
                             AA[_code(with_minor)] if snv[j] else "", (SNV if snv[j] else 0) | (SUB if sub[j] else 0),
                             snv_type, sub_type))
        records.append(rec)
        sites.extend(sorted(rows, key=lambda r: r[2]))
    return records, sites
