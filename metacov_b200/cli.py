"""``metacov`` command line on the B200 path.

Keeps the commands, options and CSV formats of reference metacov/cli.py
(`pileup` cli.py:35-109, `scan` cli.py:112-285) so that existing invocations
keep working; the work behind them runs on the GPU.  What is not carried over
is out of the hot-path scope and fails with a clear message instead of being
silently approximated: FASTQ input and `-b/-M` of `scan`, and the `simulate`
command (SURVEY.md 2, 8(f)).  `pileup -k` (the `experimental` coverage model,
reference metacov/pileup.py:38-173) runs on the GPU like `classic`.
"""
import csv
import logging
import sys

import click

from . import pileup as _pileup
from . import scan as _scan
from . import util
from .alignmentfile import AlignmentFile
from .alleles import derive, derive_compare, derive_genes, derive_linkage
from .compare import compare as _compare, read_references
from .samstream import is_stream
from .fasta import FastaFile
from .genes import read_genes

logging.basicConfig(level=logging.INFO, format="[%(relativeCreated)6.1f %(funcName)s]  %(message)s",
                    datefmt="%I:%M:%S")
log = logging.getLogger(__name__)


@click.group()
def main():
    """
    MetaCov estimates abundance values from the stacking depth of
    reads mapped to a reference.
    """


@main.command()
@click.option("--bamfile", "-b", type=click.File("rb"), required=True,
              help="Input BAM (sorted, indexed) or SAM file; '-' or a pipe (e.g. <(minimap2 -a ...)) reads SAM text as it "
                   "is written, in any read order.")
@click.option("--reference-fasta", "-f", type=click.File("rb"))
@click.option("--regionfile-blast7", "-rb", type=click.File("r"), help="Input Region file in BLAST7 format")
@click.option("--regionfile-csv", "-rc", type=click.File("r"), help="Input Region file in CSV format")
@click.option("--kmer-histogram", "-k", type=click.File("r"), help="Kmer Histogram produced with metacov scan")
@click.option("--kmer-length", "-K", type=int, default=7, help="Length of k-mer")
@click.option("--outfile", "-o", type=click.File("w"), default="-", help="Output CSV (default STDOUT)")
@click.option("--bedgraph", "-bg", type=click.File("w"), metavar="FILE",
              help="Also write the per-base depth as bedGraph (runs of equal depth; zero-depth runs omitted). "
                   "Not in the reference: additive.")
@click.option("--window", "-w", type=click.IntRange(1), metavar="N",
              help="Also write the mean depth of fixed windows of N bp to --window-out. Not in the reference: additive.")
@click.option("--window-out", "-wo", type=click.File("w"), metavar="FILE", help="Output CSV of --window (sacc,start,end,avg)")
@click.option("--bam-decode", type=click.Choice(["host", "gpu", "gpu-stream", "auto"]), default="auto", show_default=True,
              help="Where the BAM file is inflated and parsed: host threads (zlib), the GPU (whole file / streamed in chunks), or "
                   "auto = the GPU, streamed when the file does not fit it. Applies to BAM only: SAM text is always parsed whole "
                   "on the GPU (gpu-stream is refused for it). Not in the reference: additive.")
def pileup(bamfile, reference_fasta, regionfile_blast7, regionfile_csv, kmer_histogram, kmer_length, outfile,
           bedgraph=None, window=None, window_out=None, bam_decode="auto"):
    """
    Compute fold coverage values
    """
    if (window is None) != (window_out is None):
        raise click.UsageError("--window and --window-out go together")
    source = "-" if _is_stdin(bamfile) else bamfile.name
    if kmer_histogram and is_stream(source):
        raise click.UsageError("-k/--kmer-histogram (the experimental model) fetches reads per region, which a piped "
                               "stream cannot give; write the alignments to a sorted file for it")
    bam = AlignmentFile(source, decode=bam_decode)
    fasta = FastaFile(reference_fasta.name) if reference_fasta else None          # cli.py:59
    regions = util.make_region_iterator(regionfile_blast7, regionfile_csv, bam)
    try:
        mapped, unmapped = bam.mapped, bam.unmapped
        log.info("Number of reads:\n  total:    {total}\n  mapped:   {mapped} ({mappct}%)\n  unmapped: {unmapped}\n"
                 "".format(mapped=mapped, unmapped=unmapped, total=mapped + unmapped,
                           mappct=mapped / (mapped + unmapped) * 100))
    except (AttributeError, ValueError, ZeroDivisionError):
        log.error("BAM file not indexed!?")

    name2ref = {word.split()[0]: word for word in bam.references}
    # The reference piles every region up from scratch (cli.py:85-95); here the depth of the
    # whole file exists once on the GPU and all regions are answered by one kernel launch.
    hits = list(regions)
    refs, starts, ends = [], [], []
    for hit in hits:
        refs.append(name2ref[hit.sacc])
        # blast uses end<start for the reverse strand; the sorted pair is used verbatim as
        # 0-based half-open (cli.py:89, SURVEY.md Appendix C-1)
        start, end = sorted((int(hit.sstart), int(hit.send)))
        starts.append(start)
        ends.append(end)
    # cli.py:81 -- the k-mer length option is not passed on to the loader (its default 7 applies)
    k_cor = _pileup.load_kmerhist(kmer_histogram) if kmer_histogram else None
    with click.progressbar(file=sys.stderr, length=0, label="Calculating coverages"):
        results = _pileup.classic_many(bam, refs, starts, ends) if hits else []
        if k_cor is not None and hits:                                            # cli.py:93-95
            for result, extra in zip(results, _pileup.experimental_many(bam, k_cor, kmer_length, fasta, refs, starts, ends)):
                result.update(extra)
    writer = None
    for hit, result in zip(hits, results):
        if writer is None:
            writer = csv.DictWriter(outfile, fieldnames=["sacc", "start", "end"] + sorted(result.keys()))
            writer.writeheader()
        result.update({"sacc": hit.sacc, "start": hit.sstart, "end": hit.send})
        writer.writerow(result)
    if bedgraph is not None:
        write_bedgraph(bam, bedgraph)
    if window is not None:
        write_windows(bam, window, window_out)
    bam.close()


def _is_stdin(f):
    """click.File gives standard input for '-' (named "<stdin>", or unnamed under a test runner)."""
    name = getattr(f, "name", None)
    return not isinstance(name, str) or name in ("<stdin>", "-")


def write_bedgraph(bam, out):
    """Per-base depth as bedGraph lines `name<TAB>start<TAB>end<TAB>depth` (0-based half-open), one per
    run of equal non-zero depth; the runs come from the GPU (mcov_depth_runs)."""
    names = [ref.split()[0] for ref in bam.references]
    runs = bam.coverage_engine().depth_runs(skip_zero=True)
    for t, s, e, d in zip(runs["tid"].tolist(), runs["start"].tolist(), runs["end"].tolist(), runs["depth"].tolist()):
        out.write("%s\t%d\t%d\t%d\n" % (names[t], s, e, d))


def write_windows(bam, window, out):
    """Mean depth of fixed windows (the last window of a contig may be shorter): CSV sacc,start,end,avg."""
    means = bam.coverage_engine().window_means(window)
    w = csv.writer(out)
    w.writerow(["sacc", "start", "end", "avg"])
    k = 0
    for ref, ln in zip(bam.references, bam.lengths):
        for p in range(0, ln, window):
            w.writerow([ref.split()[0], p, min(p + window, ln), round(float(means[k]), 2)])
            k += 1


@main.command()
@click.option("--readfile-type", "-t", type=click.Choice(["bam", "fq"]),
              help="Override filename based detection of readfile type.")
@click.option("--max-reads", "-m", type=click.IntRange(1), metavar="N", help="Only consider the first N reads.")
@click.option("--group-by", "-g", type=click.Choice(list(_scan.Flags.keys())), multiple=True, metavar="FLAG",
              help="Group output by BAM flag. May be specified multiple times. "
                   "FLAG can be one of {}".format(list(_scan.Flags.keys())))
@click.option("--reference-fasta", "-f", type=click.File("rb"), metavar="FILE",
              help="Fasta file reads where mapped to. Required for boffset. File may be bgzip'ed, but not gzip'ed.")
@click.option("--out-basehist", "-b", type=click.File("w", lazy=False), metavar="FILE",
              help="Compute histogram of base counts by position in read.")
@click.option("--boffset", "-bo", type=click.IntRange(0, 200), default=0, metavar="N", show_default=True,
              help="Include N bases prior to read start in base histogram. Requires reference fasta file.")
@click.option("--out-kmerhist", "-o", type=click.File("w", lazy=False), metavar="FILE",
              help="Compute histogram of kmers in reads")
@click.option("-k", type=click.IntRange(2, 12), default=7, metavar="N", show_default=True, help="Length of kmers")
@click.option("--step", "-s", type=click.IntRange(1, 100), default=7, metavar="N", show_default=True,
              help="Step between sampled kmers")
@click.option("--offset", "-O", type=click.IntRange(-100, 100), default=0, metavar="N", show_default=True,
              help="Offset of first sampled kmer")
@click.option("--number", "-n", type=click.IntRange(1, 100), default=8, metavar="N", show_default=True,
              help="Numer of sampled kmers")
@click.option("--out-mirrorhist", "-M", type=click.File("w", lazy=False), metavar="FILE",
              help="Compute histogram of mismatches against palindrome")
@click.option("--mirror-offset", "-MO", type=click.IntRange(-100, 100), default=4, metavar="N", show_default=True,
              help="Offset of palindrome center from read start")
@click.option("--mirror-length", "-Ml", type=click.IntRange(1, 50), default=10, metavar="N", show_default=True,
              help="Palindrome length is 2N+1")
@click.option("--out-isizehist", "-I", type=click.File("w", lazy=False), metavar="FILE",
              help="Compute histogram of insert sizes.")
@click.option("--bam-decode", type=click.Choice(["host", "gpu", "gpu-stream", "auto"]), default="auto", show_default=True,
              help="Where the BAM file is inflated and parsed (see `pileup`); with the GPU the accumulators run on the "
                   "device-resident columns. Applies to BAM only: SAM text is always parsed on the GPU. Not in the "
                   "reference: additive.")
@click.argument("readfile", nargs=-1, required=True, metavar="READFILE...  ('-' or a pipe: SAM text as it is written)")
def scan(readfile, readfile_type, out_basehist, boffset, out_kmerhist, k, number, step, offset, max_reads,
         reference_fasta, out_mirrorhist, mirror_offset, mirror_length, out_isizehist, group_by, bam_decode="auto"):
    """
    Gather read statistics
    """
    if not readfile_type and is_stream(readfile[0]):
        readfile_type = "bam"                           # (a stream is read as SAM text)
    if not readfile_type:
        for ext, ft in ((".bam", "bam"), (".sam", "bam"), (".fq", "fq"), (".fq.gz", "fq"), (".fastq", "fq"),
                        (".fastq.gz", "fq")):
            if readfile[0].endswith(ext):
                readfile_type = ft
                break
    if not readfile_type:
        raise click.UsageError("Couldn't guess input format. Please supply -t")
    if readfile_type != "fq" and len(readfile) > 1:
        raise click.UsageError("Multiple input files only supported for fastq")
    if len(readfile) > 2:
        raise click.UsageError("At most two fastq files allowed (fwd and rev)")
    if readfile_type != "bam" and reference_fasta:
        raise click.UsageError("Reference fasta can only be used with mapped (bam/sam) reads")
    if readfile_type != "bam":
        raise click.UsageError("FASTQ input is outside the GPU hot path of this build (unmapped reads carry "
                               "no coverage); use the reference implementation for it")
    for opt, name in ((out_basehist, "-b/--out-basehist"), (out_mirrorhist, "-M/--out-mirrorhist")):
        if opt:
            raise click.UsageError(name + " needs the reference FASTA and is outside the GPU hot path of this build")

    update_every = 100000
    if max_reads and max_reads > 0 and max_reads / 100 < update_every:
        update_every = int(max_reads + 50 / 100)        # sic (reference cli.py:205-206)

    infile = AlignmentFile(readfile[0], decode=bam_decode)
    if infile.piped:
        length = max_reads or 0                         # (the counts of a stream are known once it has been read)
    else:
        log.info("mapped = {}, unmapped = {}, total = {}".format(infile.mapped, infile.unmapped,
                                                                 infile.mapped + infile.unmapped))
        length = infile.mapped + infile.unmapped
    if max_reads and 0 < max_reads < length:
        length = max_reads

    counters = []
    if out_kmerhist:
        counters.append(_scan.KmerHist(k, number, step, offset))
    if out_isizehist:
        counters.append(_scan.IsizeHist())
    counters = _scan.ByFlag(counters, [_scan.Flags[flag] for flag in group_by])

    with click.progressbar(length=length, label="Scanning reads", show_pos=True) as bar:
        with infile:
            nreads = _scan.scan_reads(infile, None, counters, update_every, lambda: bar.update(update_every),
                                      max_reads)
            if infile.piped:
                log.info("mapped = {}, unmapped = {}, total = {}".format(infile.mapped, infile.unmapped,
                                                                         infile.mapped + infile.unmapped))
        bar.update(update_every)
    log.info("Processed {} reads".format(nreads))

    n = 0
    if out_kmerhist:
        csv.writer(out_kmerhist).writerows(counters.get_rows(n))
        n += 1       # (the reference forgets this increment, cli.py:273-280; harmless there without -M)
    if out_isizehist:
        csv.writer(out_isizehist).writerows(counters.get_rows(n))
        n += 1


def _allele_rule_options():
    """The allele rules' options (counts, present alleles, coverage) and --bam-decode, which `alleles`, `compare`,
    `linkage` and `genes` share, in this order behind their own."""
    return [
        click.option("--quality-threshold", "-q", type=int, default=15, show_default=True,
                     help="Count a base only with a quality of at least this (0: every base)."),
        click.option("--read-callback", type=click.Choice(["all", "nofilter"]), default="all", show_default=True,
                     help="all: skip unmapped, secondary, QC-fail and duplicate reads; nofilter: count every "
                          "placed read."),
        click.option("--min-coverage", type=click.IntRange(1), default=5, show_default=True),
        click.option("--min-freq", type=click.FloatRange(0, 1), default=0.05, show_default=True),
        click.option("--min-count", type=click.IntRange(1), default=2, show_default=True),
        click.option("--bam-decode", type=click.Choice(["host", "gpu", "gpu-stream", "auto"]), default="auto",
                     show_default=True, help="Where the BAM file is inflated and parsed (see `pileup`).")]


def _apply(options):
    def apply(f):
        for option in reversed(options):
            f = option(f)
        return f
    return apply


def _allele_options(sites_help):
    """The options `alleles` and `compare` share, in this order behind their own; ``sites_help``: --sites-out's help."""
    return _apply([
        click.option("--regionfile-blast7", "-rb", type=click.File("r"), help="Input Region file in BLAST7 format"),
        click.option("--regionfile-csv", "-rc", type=click.File("r"), help="Input Region file in CSV format"),
        click.option("--outfile", "-o", type=click.File("w"), default="-", help="Output CSV (default STDOUT)"),
        click.option("--sites-out", type=click.File("w"), metavar="FILE", help=sites_help)] + _allele_rule_options())


def _refuse_stream(path, option="-b/--bamfile"):
    if is_stream(path):
        raise click.UsageError(option + ": the allele counts need every record of a file; a piped stream cannot give "
                               "them (write the alignments to a file)")


def _hit_columns(hits, references):
    """(refs, starts, ends) of region hits: the full reference name of each hit's contig and its 0-based interval."""
    name2ref = {word.split()[0]: word for word in references}
    refs, starts, ends = [], [], []
    for hit in hits:
        refs.append(name2ref[hit.sacc])
        start, end = sorted((int(hit.sstart), int(hit.send)))      # (as `pileup`: blast's reverse strand has end < start)
        starts.append(start)
        ends.append(end)
    return refs, starts, ends


@main.command()
@click.option("--bamfile", "-b", type=click.Path(dir_okay=False, allow_dash=True), required=True,
              help="Input BAM or SAM file (any read order, no index needed). Not a pipe: the counts need every record.")
@click.option("--reference-fasta", "-f", type=click.Path(exists=True, dir_okay=False),
              help="Reference the reads were mapped to: enables SUB / POPSUB, con_ani and pop_ani.")
@_allele_options("Also write every site as TSV: contig pos ref A C G T consensus snv sub popsub (pos 0-based).")
def alleles(bamfile, reference_fasta, regionfile_blast7, regionfile_csv, outfile, sites_out, quality_threshold,
            read_callback, min_coverage, min_freq, min_count, bam_decode):
    """
    Allele statistics per region from the A/C/G/T counts on the GPU: breadth, depth, nucleotide diversity (pi), SNVs
    per kbp and, with a reference, consensus and population ANI.  Not in the reference: additive.
    """
    _refuse_stream(bamfile)
    regions = None
    if regionfile_blast7 or regionfile_csv:
        regions = util.make_region_iterator(regionfile_blast7, regionfile_csv, None)
    bam = AlignmentFile(bamfile, decode=bam_decode)
    fasta = FastaFile(reference_fasta) if reference_fasta else None
    if regions is None:
        regions = util.get_regions_from_bam(bam)
    hits = list(regions)
    refs, starts, ends = _hit_columns(hits, bam.references)
    kw = dict(fasta=fasta, quality_threshold=quality_threshold, read_callback=read_callback,
              min_coverage=min_coverage, min_freq=min_freq, min_count=min_count)
    if hits:
        derived = derive(bam.allele_stats(refs, starts, ends, **kw))
        writer = csv.DictWriter(outfile, fieldnames=["sacc", "start", "end"] + sorted(derived))
        writer.writeheader()
        for k, hit in enumerate(hits):
            row = {name: float(v[k]) for name, v in derived.items()}
            row.update({"sacc": hit.sacc, "start": hit.sstart, "end": hit.send})
            writer.writerow(row)
    if sites_out is not None:
        write_sites(bam, bam.allele_sites(**kw), sites_out)
    bam.close()


def write_sites(bam, sites, out):
    """Sites as TSV lines: contig (first word of its name), 0-based position, reference base (N: unknown), the A C G T
    counts, the consensus and the SNV / SUB / POPSUB flags as 0 / 1."""
    names = [ref.split()[0] for ref in bam.references]
    out.write("contig\tpos\tref\tA\tC\tG\tT\tconsensus\tsnv\tsub\tpopsub\n")
    kind = sites["kind"]
    cols = [sites[k].tolist() for k in ("tid", "pos", "A", "C", "G", "T")]
    for (t, p, a, c, g, tt), r, cons, k in zip(zip(*cols), sites["ref"].tolist(), sites["consensus"].tolist(), kind.tolist()):
        out.write("%s\t%d\t%s\t%d\t%d\t%d\t%d\t%s\t%d\t%d\t%d\n" % (names[t], p, r.decode(), a, c, g, tt, cons.decode(),
                                                                    k & 1, (k >> 1) & 1, (k >> 2) & 1))


@main.command()
@click.option("--bamfile", "-b", "bamfiles", type=click.Path(dir_okay=False, allow_dash=True), multiple=True, required=True,
              help="Input BAM or SAM file, two or more times (any read order, no index; every file with the same "
                   "reference names and lengths). Not a pipe: the counts need every record.")
@_allele_options("Also write every con_snp site of every pair as TSV: sample_a sample_b contig pos cons_a cons_b "
                 "alleles_a alleles_b con_snp pop_snp (pos 0-based; alleles: the present alleles plus the consensus).")
def compare(bamfiles, regionfile_blast7, regionfile_csv, outfile, sites_out, quality_threshold, read_callback,
            min_coverage, min_freq, min_count, bam_decode):
    """
    Compare samples per region and pair on the GPU: positions covered in both, consensus and population ANI (conANI /
    popANI) from the A/C/G/T counts of each file.  Not in the reference: additive.
    """
    if len(bamfiles) < 2:
        raise click.UsageError("-b/--bamfile: a comparison needs at least two files")
    for f in bamfiles:
        _refuse_stream(f, "-b/--bamfile " + f)
    names, lengths = read_references(bamfiles[0])
    if regionfile_blast7 or regionfile_csv:
        hits = list(util.make_region_iterator(regionfile_blast7, regionfile_csv, None))
    else:
        hits = [util.Region(n, name, 0, length) for n, (name, length) in enumerate(zip(names, lengths))]
    refs, starts, ends = _hit_columns(hits, names)
    res = _compare(bamfiles, refs, starts, ends, sites=sites_out is not None, decode=bam_decode,
                   quality_threshold=quality_threshold, read_callback=read_callback, min_coverage=min_coverage,
                   min_freq=min_freq, min_count=min_count)
    derived = derive_compare(res.stats)
    cols = {"compared": res.stats["compared"], "con_snps": res.stats["con_snp"], "covered_a": res.stats["covered_a"],
            "covered_b": res.stats["covered_b"], "pop_snps": res.stats["pop_snp"]}
    cols.update(derived)
    writer = csv.DictWriter(outfile, fieldnames=["sacc", "start", "end", "sample_a", "sample_b"] + sorted(cols))
    writer.writeheader()
    for k, hit in enumerate(hits):
        for p, (a, b) in enumerate(res.pairs.tolist()):
            row = {name: (int(v[p, k]) if v.dtype.kind == "i" else float(v[p, k])) for name, v in cols.items()}
            row.update({"sacc": hit.sacc, "start": hit.sstart, "end": hit.send, "sample_a": bamfiles[a],
                        "sample_b": bamfiles[b]})
            writer.writerow(row)
    if sites_out is not None:
        write_compare_sites(names, bamfiles, res.pairs, res.sites, sites_out)


@main.command()
@click.option("--bamfile", "-b", type=click.Path(dir_okay=False, allow_dash=True), required=True,
              help="Input BAM or SAM file (any read order, no index needed; mates share a read name). Not a pipe: the "
                   "linkage needs every record.")
@click.option("--outfile", "-o", type=click.File("w"), default="-", help="Output TSV (default STDOUT)")
@click.option("--max-distance", type=click.IntRange(1, 100000), default=1000, show_default=True,
              help="Link SNV sites at most this many bases apart.")
@click.option("--min-reads", type=click.IntRange(1), default=20, show_default=True,
              help="List a pair of sites when at least this many read pairs (or reads) call both.")
@_apply(_allele_rule_options())
def linkage(bamfile, outfile, max_distance, min_reads, quality_threshold, read_callback, min_coverage, min_freq, min_count,
            bam_decode):
    """
    Linkage between nearby SNV sites on the GPU: for each pair of SNV sites that enough reads and their mates span, the
    four haplotype counts, r2 and D' (inStrain's linkage table with fixed allele calls).  Not in the reference:
    additive.
    """
    _refuse_stream(bamfile)
    with AlignmentFile(bamfile, decode=bam_decode) as bam:
        pairs, _info = bam.linkage(quality_threshold=quality_threshold, read_callback=read_callback,
                                   min_coverage=min_coverage, min_freq=min_freq, min_count=min_count,
                                   max_distance=max_distance, min_reads=min_reads)
        write_linkage(bam.references, pairs, outfile)


def write_linkage(references, pairs, out):
    """Linkage pairs as TSV lines: contig (first word of its name), both 0-based positions, their distance, the major
    and minor allele of each site, the four haplotype counts (upper case = major), their total, r2 and D'."""
    names = [ref.split()[0] for ref in references]
    derived = derive_linkage(pairs)
    out.write("contig\tpos_a\tpos_b\tdistance\tmajor_a\tminor_a\tmajor_b\tminor_b\tn_AB\tn_Ab\tn_aB\tn_ab\ttotal\tr2"
              "\td_prime\n")
    cols = [pairs[k].tolist() for k in ("tid", "pos_a", "pos_b", "major_a", "minor_a", "major_b", "minor_b", "n_AB", "n_Ab",
                                        "n_aB", "n_ab")]
    for (t, pa, pb, ma, na, mb, nb, c0, c1, c2, c3), r2, dp in zip(zip(*cols), derived["r2"].tolist(),
                                                                  derived["d_prime"].tolist()):
        out.write("%s\t%d\t%d\t%d\t%s\t%s\t%s\t%s\t%d\t%d\t%d\t%d\t%d\t%r\t%r\n" % (
            names[t], pa, pb, pb - pa, ma.decode(), na.decode(), mb.decode(), nb.decode(), c0, c1, c2, c3,
            c0 + c1 + c2 + c3, r2, dp))


@main.command()
@click.option("--bamfile", "-b", type=click.Path(dir_okay=False, allow_dash=True), required=True,
              help="Input BAM or SAM file (any read order, no index needed). Not a pipe: the counts need every record.")
@click.option("--reference-fasta", "-f", type=click.Path(exists=True, dir_okay=False), required=True,
              help="Reference the reads were mapped to.")
@click.option("--genes", "-g", "gene_file", type=click.Path(exists=True, dir_okay=False), required=True,
              help="Genes: Prodigal's nucleotide FASTA (genes.fna) or GFF3 (its CDS lines).")
@click.option("--outfile", "-o", type=click.File("w"), default="-", help="Output CSV (default STDOUT)")
@click.option("--sites-out", type=click.File("w"), metavar="FILE",
              help="Also write every SNV / SUB position of a called codon as TSV (pos 0-based).")
@_apply(_allele_rule_options())
def genes(bamfile, reference_fasta, gene_file, outfile, sites_out, quality_threshold, read_callback, min_coverage,
          min_freq, min_count, bam_decode):
    """
    Profile genes on the GPU: codons called, expected N and S sites, SNVs and substitutions typed synonymous (S),
    nonsynonymous (N) or multiple (M), pN/pS and dN/dS, with the allele statistics of each gene (inStrain's gene_info
    with fixed allele calls).  Not in the reference: additive.
    """
    _refuse_stream(bamfile)
    table = read_genes(gene_file)
    with AlignmentFile(bamfile, decode=bam_decode) as bam:
        records, stats, sites = bam.gene_stats(
            table, FastaFile(reference_fasta), quality_threshold=quality_threshold, read_callback=read_callback,
            min_coverage=min_coverage, min_freq=min_freq, min_count=min_count, sites=sites_out is not None)
    ints = [f for f in records.dtype.names if f != "pad"]
    derived = derive(stats)
    derived_genes = derive_genes(records)
    writer = csv.writer(outfile)
    writer.writerow(["name", "contig", "start", "end", "strand"] + ints + sorted(derived) + list(derived_genes))
    for k in range(len(records)):
        writer.writerow([table.name[k], table.contig[k], int(table.start[k]), int(table.end[k]),
                         "+" if table.strand[k] > 0 else "-"] + [int(records[f][k]) for f in ints]
                        + [float(derived[n][k]) for n in sorted(derived)] + [float(v[k]) for v in derived_genes.values()])
    if sites is not None:
        write_gene_sites(table, sites, sites_out)


def write_gene_sites(table, sites, out):
    """Gene sites as TSV lines: gene name, contig, 0-based position, codon index and position in it (from the 5' end),
    the reference codon, major and minor allele (genomic orientation), the amino acids of the reference codon and with
    the major / minor allele, the SNV / SUB flags as 0 / 1 and the SNV / SUB types N S M ('.' where none applies)."""
    out.write("gene\tcontig\tpos\tcodon\tcodon_pos\tref_codon\tmajor\tminor\taa_ref\taa_major\taa_minor\tsnv\tsub"
              "\tsnv_type\tsub_type\n")
    cols = [sites[k].tolist() for k in ("gene", "pos", "codon", "codon_pos", "kind")]
    letters = [[x.decode() or "." for x in sites[k].tolist()] for k in ("ref_codon", "major", "minor", "aa_ref", "aa_major",
                                                                        "aa_minor", "snv_type", "sub_type")]
    for (g, p, c, cp, k), (rc, ma, mi, ar, am, an, st, bt) in zip(zip(*cols), zip(*letters)):
        out.write("%s\t%s\t%d\t%d\t%d\t%s\t%s\t%s\t%s\t%s\t%s\t%d\t%d\t%s\t%s\n" % (
            table.name[g], table.contig[g], p, c, cp, rc, ma, mi, ar, am, an, k & 1, (k >> 1) & 1, st, bt))


def _alleles_of(sig):
    """Letters of a signature byte's allele set: the present alleles plus the consensus, in A C G T order."""
    bits = (sig & 0x0F) | (1 << ((sig >> 4) & 3))
    return "".join(ch for b, ch in enumerate("ACGT") if bits >> b & 1)


def write_compare_sites(references, samples, pairs, sites, out):
    """Compare sites as TSV lines: the two samples as given, contig (first word of its name), 0-based position, both
    consensus bases, both allele sets as letters (e.g. AG) and the con_snp / pop_snp flags as 0 / 1."""
    names = [ref.split()[0] for ref in references]
    out.write("sample_a\tsample_b\tcontig\tpos\tcons_a\tcons_b\talleles_a\talleles_b\tcon_snp\tpop_snp\n")
    pairs = pairs.tolist()
    cols = [sites[k].tolist() for k in ("pair", "tid", "pos", "sig_a", "sig_b", "kind")]
    for p, t, pos, sa, sb, k in zip(*cols):
        a, b = pairs[p]
        out.write("%s\t%s\t%s\t%d\t%s\t%s\t%s\t%s\t%d\t%d\n" % (
            samples[a], samples[b], names[t], pos, "ACGT"[(sa >> 4) & 3], "ACGT"[(sb >> 4) & 3], _alleles_of(sa),
            _alleles_of(sb), k & 1, (k >> 1) & 1))


if __name__ == "__main__":
    main()
