"""Gene tables for ``AlignmentFile.gene_stats`` and ``metacov genes``: Prodigal's nucleotide FASTA and GFF3 CDS lines."""
from typing import List, NamedTuple

import numpy as np


class GeneTable(NamedTuple):
    """Genes as columns: name and contig (str lists), start / end (0-based half-open), strand (+1 / -1) and phase (0-2)
    as int64 arrays."""
    name: List[str]
    contig: List[str]
    start: np.ndarray
    end: np.ndarray
    strand: np.ndarray
    phase: np.ndarray


def _int(text, what, where):
    try:
        return int(text)
    except ValueError:
        raise ValueError("%s: %s %r is not an integer" % (where, what, text)) from None


def _prodigal(line, where):
    """``>name # start # end # strand # ...``: contig = name without its trailing ``_<n>``, phase 0."""
    f = [x.strip() for x in line[1:].split("#")]
    if len(f) < 4 or not f[0]:
        raise ValueError("%s: not a Prodigal header (>name # start # end # strand # ...)" % where)
    name = f[0].split()[0]
    contig, sep, n = name.rpartition("_")
    if not sep or not contig or not n.isdigit():
        raise ValueError("%s: gene name %r does not end in _<n>" % (where, name))
    start, end = _int(f[1], "start", where), _int(f[2], "end", where)
    strand = {"1": 1, "-1": -1, "+1": 1}.get(f[3])
    if strand is None:
        raise ValueError("%s: strand %r is not 1 or -1" % (where, f[3]))
    return name, contig, start, end, strand, 0


def _gff_cds(line, where):
    f = line.rstrip("\r\n").split("\t")
    if len(f) != 9:
        raise ValueError("%s: a GFF3 line has 9 tab-separated columns, this one %d" % (where, len(f)))
    if f[2] != "CDS":
        return None
    start, end = _int(f[3], "start", where), _int(f[4], "end", where)
    strand = {"+": 1, "-": -1}.get(f[6])
    if strand is None:
        raise ValueError("%s: CDS strand %r is not + or -" % (where, f[6]))
    if f[7] not in ("0", "1", "2"):
        raise ValueError("%s: CDS phase %r is not 0, 1 or 2" % (where, f[7]))
    name = None
    for attr in f[8].split(";"):
        key, _, value = attr.strip().partition("=")
        if key == "ID" and value:
            name = value
    if name is None:
        name = "%s:%d-%d" % (f[0], start, end)
    return name, f[0], start, end, strand, int(f[7])


def read_genes(path):
    """The genes of a Prodigal nucleotide FASTA (headers ``>name # start # end # strand # ...``, sequence lines
    skipped) or of a GFF3 file (its ``CDS`` lines; other feature types, comments and a trailing ``##FASTA`` section are
    skipped), told apart by the first line that is not empty or a comment.  Coordinates are 1-based inclusive in both
    and come back 0-based half-open.  A malformed line, or one with start < 1 or end < start, raises ValueError naming
    it."""
    rows = []
    kind = None
    with open(path) as fh:
        for no, line in enumerate(fh, 1):
            where = "%s:%d" % (path, no)
            s = line.strip()
            if not s:
                continue
            if kind is None:
                if s.startswith("#") and not s.startswith("##FASTA"):
                    continue
                kind = "fasta" if s.startswith(">") else "gff"
            if kind == "fasta":
                if not s.startswith(">"):
                    continue
                row = _prodigal(s, where)
            else:
                if s.startswith("##FASTA"):
                    break
                if s.startswith("#"):
                    continue
                row = _gff_cds(line, where)
                if row is None:
                    continue
            if row[2] < 1 or row[3] < row[2]:
                raise ValueError("%s: need 1 <= start <= end, got %d..%d" % (where, row[2], row[3]))
            rows.append(row)
    return GeneTable([r[0] for r in rows], [r[1] for r in rows],
                     np.array([r[2] - 1 for r in rows], np.int64), np.array([r[3] for r in rows], np.int64),
                     np.array([r[4] for r in rows], np.int64), np.array([r[5] for r in rows], np.int64))
