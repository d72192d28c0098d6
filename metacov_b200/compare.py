"""Samples compared on the GPU (DESIGN.md §3.16): per region and pair of alignment files, the positions covered in both
and how many of them differ by consensus (con_snp) or share no allele (pop_snp) -- inStrain's conANI / popANI
questions, with the fixed allele calls of ``AlignmentFile.allele_stats``.

A file is reduced to its signature, one byte a reference slot (``AlignmentFile.allele_signature``), and the pairs are
compared from the signatures.  Files are taken one at a time (decode, count, signature, close), so a comparison of S
files holds one file's counters and S bytes a slot of signatures, never S counter stores."""
import collections

import numpy as np

from . import samstream
from .alignmentfile import AlignmentFile, BamStream, _check_read_callback, is_sam_text
from .engine import CoverageEngine

CompareResult = collections.namedtuple("CompareResult", "pairs stats sites")
CompareResult.__doc__ = """pairs: int32 [n_pairs, 2] file indices (a, b); stats: ``_capi.COMPARE_STATS_DTYPE`` records
[n_pairs, g] (length, covered_a, covered_b, compared, con_snp, pop_snp); sites: ``_capi.COMPARE_SITE_DTYPE`` records in
(pair, tid, pos) order with ``sites=True``, else None."""


def all_pairs(n):
    """Every (i, j) with i < j of n files, in lexicographic order."""
    return np.array([(i, j) for i in range(n) for j in range(i + 1, n)], dtype=np.int32).reshape(-1, 2)


def read_references(path):
    """(names, lengths) of an alignment file's references from its header alone (no record is decoded)."""
    if is_sam_text(path):
        with open(path, "rb") as fh:
            head, _ = samstream.read_header(fh)
        refs = samstream.header_refs(head.decode())
        return tuple(r for r, _ in refs), tuple(n for _, n in refs)
    with BamStream(path) as bs:
        return bs.references, bs.lengths


def _header_mismatch(name, refs, lens, name0, refs0, lens0):
    """ValueError naming file `name` and the first contig where its header differs from `name0`'s."""
    for k in range(max(len(refs), len(refs0))):
        if k >= len(refs) or k >= len(refs0) or refs[k] != refs0[k] or int(lens[k]) != int(lens0[k]):
            mine = "%r of length %d" % (refs[k], int(lens[k])) if k < len(refs) else "no contig"
            theirs = "%r of length %d" % (refs0[k], int(lens0[k])) if k < len(refs0) else "no contig"
            return ValueError("%s: contig %d is %s, and %s in %s: every file of a comparison needs the same reference "
                              "names and lengths in the same order" % (name, k, mine, theirs, name0))
    return None


def compare(files, contigs=None, starts=None, stops=None, pairs=None, sites=False, decode="auto", quality_threshold=15,
            read_callback="all", min_coverage=5, min_freq=0.05, min_count=2):
    """Compare two or more alignment files -> ``CompareResult(pairs, stats, sites)``.

    ``files``: paths or open ``AlignmentFile``s (a path is opened with ``decode`` and closed once its signature is
    made; an open file is left open).  Every file needs the same reference names and lengths in the same order, else
    ValueError naming the first file and contig that differ.  Regions as in ``AlignmentFile.allele_stats`` (default:
    every contig whole).  ``pairs``: [n, 2] file indices, default every i < j.  The allele parameters are those of
    ``allele_stats`` and apply to every file.  ``alleles.derive_compare(stats)`` gives con_ani, pop_ani and
    percent_compared.  A piped stream raises ValueError: a signature needs every record of a file."""
    files = list(files)
    if len(files) < 2:
        raise ValueError("compare needs at least two files, got %d" % len(files))
    pairs = all_pairs(len(files)) if pairs is None else np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    if len(pairs) == 0 or pairs.min() < 0 or pairs.max() >= len(files) or (pairs[:, 0] == pairs[:, 1]).any():
        raise ValueError("pairs must be one or more pairs of two different file indices of 0 .. %d" % (len(files) - 1))
    pairs = pairs.astype(np.int32)
    _check_read_callback(read_callback)
    CoverageEngine._allele_params(min_coverage, min_freq, min_count, False)      # (ValueError before any work)
    kw = dict(quality_threshold=quality_threshold, read_callback=read_callback, min_coverage=min_coverage,
              min_freq=min_freq, min_count=min_count)
    sigs, first, last, own_last = [], None, None, False
    try:
        for k, f in enumerate(files):
            own = not isinstance(f, AlignmentFile)
            af = AlignmentFile(f, decode=decode) if own else f
            try:
                if first is None:
                    first = (af.filename, af.references, af.lengths)
                else:
                    err = _header_mismatch(af.filename, af.references, af.lengths, *first)
                    if err is not None:
                        raise err
                sigs.append(af.allele_signature(**kw))
            except BaseException:
                if own:
                    af.close()
                raise
            if k == len(files) - 1:
                last, own_last = af, own
            elif own:
                af.close()                                    # (its counters go before the next file is counted)
        tid, start, stop = last._regions(contigs, starts, stops)
        eng = last._count_engine()
        stats = eng.compare_stats(sigs, pairs, tid, start, stop)
        site_list = eng.compare_sites(sigs, pairs) if sites else None
    finally:
        if own_last:
            last.close()
    return CompareResult(pairs, stats, site_list)
