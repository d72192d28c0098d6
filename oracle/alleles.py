"""The allele rules of ``AlignmentFile.allele_stats`` / ``allele_sites`` (include/metacov_b200.h, mcov_allele_*)
restated over count arrays with numpy: the reference the device results are checked against.  Test infrastructure
only: the product never imports it.

Counts are uint32 [4, n] (A, C, G, T rows, as ``count_coverage`` / ``basecount.full_counts`` give them); a reference is
a str / bytes of the same length or None (unknown everywhere).
"""
import math

import numpy as np

SNV, SUB, POPSUB = 1, 2, 4
UNKNOWN = 4


def ref_codes(seq, n):
    """A C G T (any case) -> 0..3, anything else (N, IUPAC codes) -> 4; None -> all 4."""
    if seq is None:
        return np.full(n, UNKNOWN, np.uint8)
    b = np.frombuffer(seq.encode("ascii") if isinstance(seq, str) else bytes(seq), np.uint8) & 0xDF
    if len(b) != n:
        raise ValueError("reference of %d bases for %d positions" % (len(b), n))
    out = np.full(n, UNKNOWN, np.uint8)
    for code, ch in enumerate(b"ACGT"):
        out[b == ch] = code
    return out


def check_params(min_coverage=5, min_freq=0.05, min_count=2):
    if int(min_coverage) != min_coverage or min_coverage < 1:
        raise ValueError("min_coverage must be an integer >= 1")
    if int(min_count) != min_count or min_count < 1:
        raise ValueError("min_count must be an integer >= 1")
    if not 0.0 <= float(min_freq) <= 1.0:
        raise ValueError("min_freq must be in [0, 1]")


def evaluate(counts, ref=None, min_coverage=5, min_freq=0.05, min_count=2):
    """Per position: dict of N (int64), covered (bool), present (bool [4, n]), consensus (0-3, valid where covered),
    pi (float64, 0 where not covered), ref (codes) and kind (SNV | SUB | POPSUB bits, 0 where not covered)."""
    check_params(min_coverage, min_freq, min_count)
    c = np.asarray(counts, dtype=np.int64).reshape(4, -1)
    n = c.shape[1]
    r = ref_codes(ref, n) if (ref is None or isinstance(ref, (str, bytes))) else np.asarray(ref, np.uint8)
    N = c[0] + c[1] + c[2] + c[3]
    covered = N >= min_coverage
    dN = N.astype(np.float64)
    thr = float(min_freq) * dN                                        # one float64 multiply
    present = (c >= min_count) & (c.astype(np.float64) >= thr)
    consensus = np.argmax(c, axis=0)                                  # (ties: the first maximum, A C G T order)
    with np.errstate(invalid="ignore", divide="ignore"):
        f = c.astype(np.float64) / dN
        pi = 1.0 - ((f[0] * f[0] + f[1] * f[1]) + (f[2] * f[2] + f[3] * f[3]))
    pi = np.where(covered, pi, 0.0)
    npres = present.sum(axis=0)
    known = r < 4
    ref_present = np.zeros(n, bool)
    for b in range(4):
        ref_present |= (r == b) & present[b]
    kind = (np.where(npres >= 2, SNV, 0) | np.where(known & (consensus != r), SUB, 0)
            | np.where(known & (npres >= 1) & ~ref_present, POPSUB, 0))
    kind = np.where(covered, kind, 0).astype(np.uint8)
    return dict(N=N, covered=covered, present=present, consensus=consensus, pi=pi, ref=r, kind=kind)


def region_stats(counts, ref, start, end, **params):
    """The record of region [start, end) of one contig (counts [4, length]): positions past the contig end have zero
    counts.  pi_sum is math.fsum over the covered positions' pi."""
    c = np.asarray(counts)
    length = c.shape[1]
    a, b = min(start, length), min(end, length)
    e = evaluate(c[:, a:b], None if ref is None else ref[a:b], **params)
    cov = e["covered"]
    return dict(length=int(end - start), covered=int(cov.sum()), depth_sum=int(e["N"].sum()),
                pi_sum=math.fsum(e["pi"][cov].tolist()), snv=int(((e["kind"] & SNV) != 0).sum()),
                ref_covered=int((cov & (e["ref"] < 4)).sum()), sub=int(((e["kind"] & SUB) != 0).sum()),
                popsub=int(((e["kind"] & POPSUB) != 0).sum()))


def sites(counts_per_contig, refs=None, **params):
    """Every position with kind != 0, by (tid, pos): a list of (tid, pos, A, C, G, T, ref letter, consensus letter,
    kind)."""
    out = []
    for t, c in enumerate(counts_per_contig):
        e = evaluate(c, None if refs is None else refs[t], **params)
        c = np.asarray(c, dtype=np.int64)
        for p in np.nonzero(e["kind"])[0].tolist():
            out.append((t, p, int(c[0, p]), int(c[1, p]), int(c[2, p]), int(c[3, p]), "ACGTN"[int(e["ref"][p])],
                        "ACGT"[int(e["consensus"][p])], int(e["kind"][p])))
    return out
