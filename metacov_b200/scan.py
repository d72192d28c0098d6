"""Drop-in for ``metacov.scan`` on the B200 path (read statistics of a BAM).

Mirrors the surface of reference metacov/scan.pyx: ``Flag`` / ``Flags`` /
``FLAG_*`` (scan.pyx:76-133), ``ReadProcessor`` / ``ReadProcessorList``
(345-376), ``ByFlag`` (380-420), ``IsizeHist`` (581-620), ``KmerHist``
(491-533) and ``scan_reads`` (623-672), each accumulator with ``__copy__``,
``.counts`` and ``.get_rows()``.

The reference walks the file one record at a time under the GIL
(scan.pyx:653-667); here the records are decoded once into SoA arrays and every
accumulator is filled by one CUDA kernel over all records (order does not
matter for a histogram).  GPU-backed: ``ByFlag`` grouping, ``IsizeHist`` (flag
and isize only) and ``KmerHist`` (per-read SEQ windows).  ``BaseHist`` /
``MirrorHist`` need a reference FASTA and are out of scope (SURVEY.md 2 /
Appendix C-9).
"""
from copy import copy
from itertools import islice

import numpy as np

from .alignmentfile import AlignmentFile
from .engine import CoverageEngine


class Flag:
    def __init__(self, flag, name_true, name_false, name_col):
        self.flag = int(flag)
        self.name_true = name_true
        self.name_false = name_false
        self.name_col = name_col

    def __repr__(self):
        return "Flag(0x%x, %r, %r, %r)" % (self.flag, self.name_true, self.name_false, self.name_col)


# the eleven BAM flag bits with the labels of scan.pyx:86-106 (note: FLAG_MAPPED wraps
# BAM_FUNMAP, so its *true* label is "Unmapped"; Appendix C-7)
FLAG_PAIRED = Flag(0x1, "Paired", "Unpaired", "Paired")
FLAG_PROPER_PAIR = Flag(0x2, "Paired", "Unpaired", "PairedProperly")
FLAG_MAPPED = Flag(0x4, "Unmapped", "Mapped", "Mapped")
FLAG_MMAPPED = Flag(0x8, "Unmapped", "Mapped", "MateMapped")
FLAG_REVERSE = Flag(0x10, "Reverse", "Forward", "Readdir")
FLAG_MREVERSE = Flag(0x20, "Reverse", "Forward", "MateReaddir")
FLAG_READ1 = Flag(0x40, "R1", "R2", "IsRead1")
FLAG_READ2 = Flag(0x80, "R2", "R1", "IsRead2")
FLAG_SECONDARY = Flag(0x100, "Secondary", "Primary", "Alignment")
FLAG_QCFAIL = Flag(0x200, "Fail", "Pass", "QC")
FLAG_DUP = Flag(0x400, "Duplicate", "Singleton", "Duplicate")

Flags = {f.name_col: f for f in (FLAG_PAIRED, FLAG_PROPER_PAIR, FLAG_MAPPED, FLAG_MMAPPED, FLAG_REVERSE,
                                 FLAG_MREVERSE, FLAG_READ1, FLAG_READ2, FLAG_SECONDARY, FLAG_QCFAIL, FLAG_DUP)}


class ReadProcessor:
    """Base class of the read-statistics accumulators."""

    def set_max_readlen(self, rlen):
        pass

    def process_read(self, rlen, read, flags, it):
        print("ArgHHH")          # scan.pyx:350-352: the base class is not meant to be fed

    # -- GPU path: fill this accumulator from all records at once ------------------------------
    def _accumulate(self, ctx, group_flags, targets):
        raise NotImplementedError(
            "%s is not GPU-backed in this build (scope: SURVEY.md 8(f))" % type(self).__name__)


class ReadProcessorList(ReadProcessor):
    """Fan-out over several accumulators (scan.pyx:355-376)."""

    def __init__(self, processors):
        self.processors = processors
        for p in processors:
            assert isinstance(p, ReadProcessor)

    def __copy__(self):
        return ReadProcessorList([copy(p) for p in self.processors])

    def set_max_readlen(self, rlen):
        for p in self.processors:
            p.set_max_readlen(rlen)

    def get_rows(self, i):
        return self.processors[i].get_rows()

    def _merge(self, other):
        for p, q in zip(self.processors, other.processors):
            p._merge(q)

    def _accumulate(self, ctx, group_flags, targets):
        # targets: the copies of this list, one per ByFlag group (or just [self])
        for i, p in enumerate(self.processors):
            p._accumulate(ctx, group_flags, [t.processors[i] for t in targets])


class ByFlag(ReadProcessorList):
    """2**len(flags) copies of an accumulator (list); a read goes to copy
    n = its bits of the selected flags, first selected flag = most significant
    (scan.pyx:380-420)."""

    def __init__(self, processor, flags):
        if isinstance(processor, list):
            processor = ReadProcessorList(processor)
        assert isinstance(processor, ReadProcessor)
        self.nflags = len(flags)
        self.flags = flags
        super().__init__([copy(processor) for _ in range(2 ** self.nflags)])

    def __copy__(self):
        return ByFlag(copy(self.processors[0]), list(self.flags))

    def get_rows(self, i):
        tag_head = [f.name_col for f in reversed(self.flags)]
        yield next(iter(self.processors[0].get_rows(i))) + tag_head
        for n, processor in enumerate(self.processors):
            tag = [f.name_true if (1 << m) & n else f.name_false for m, f in enumerate(reversed(self.flags))]
            for row in islice(processor.get_rows(i), 1, None):
                yield row + tag

    def _accumulate(self, ctx, group_flags, targets):
        if group_flags:
            raise NotImplementedError("nested ByFlag")
        gf = [f.flag for f in self.flags]
        self.processors[0]._accumulate(ctx, gf, self.processors)


class IsizeHist(ReadProcessor):
    """counts[abs(isize)] += 1 for every read; isize counts only for PROPER_PAIR
    reads, everything else lands in bin 0 (scan.pyx:267-271, 581-620)."""

    def __init__(self):
        self._counts_data = np.zeros(128, dtype=np.uint32)
        self.max_isize = 0

    def __copy__(self):
        return IsizeHist()

    @property
    def counts(self):
        return self._counts_data

    def get_rows(self):
        yield ["n", "count"]
        for i in range(self.max_isize + 1):
            yield [i, self._counts_data[i]]

    def _ingest(self, row):
        nz = np.nonzero(row)[0]
        self.max_isize = int(nz[-1]) if len(nz) else 0
        asize = 128
        while asize <= self.max_isize:        # the reference doubles its array (scan.pyx:603-608)
            asize *= 2
        data = np.zeros(asize, dtype=np.uint32)
        m = min(asize, len(row))
        data[:m] = row[:m]
        self._counts_data = data

    def _merge(self, other):
        """Add the counts of another IsizeHist (tables of any widths): the rows one call over both sets of reads gives."""
        a, b = self._counts_data, other._counts_data
        row = np.zeros(max(len(a), len(b)), dtype=np.uint32)
        row[:len(a)] += a
        row[:len(b)] += b
        self._ingest(row)

    def _accumulate(self, ctx, group_flags, targets):
        hist, _, _ = ctx["engine"].isize_hist(ctx["flag"], ctx["isize"], group_flags)
        for g, t in enumerate(targets):
            t._ingest(hist[g])


class KmerHist(ReadProcessor):
    """k-mer histogram at NK sampled read positions (scan.pyx:491-533): reads shorter than
    OFFSET+STEP*NK are skipped; the k-mer at read position OFFSET+i*STEP is counted in
    counts[kmer, i], first base in the low bits, any N -> row 4**K."""

    def __init__(self, K, NK, STEP, OFFSET):
        self.K, self.NK, self.STEP, self.OFFSET = K, NK, STEP, OFFSET
        self._counts_data = np.zeros((4 ** K + 1, NK), dtype=np.uint32)

    def __copy__(self):
        return KmerHist(self.K, self.NK, self.STEP, self.OFFSET)

    @property
    def counts(self):
        return self._counts_data

    def get_rows(self):
        yield ["kmer"] + ["n{}".format(i) for i in range(self.NK)]
        yield ["N" * self.K] + list(self.counts[4 ** self.K])
        for i in range(4 ** self.K):
            yield [kmer_base2_to_ascii(i, self.K)] + list(self._counts_data[i])

    def _merge(self, other):
        self._counts_data = self._counts_data + other._counts_data

    def _accumulate(self, ctx, group_flags, targets):
        if self.OFFSET < 0:
            raise ValueError("KmerHist: a negative OFFSET reads outside the read in the reference "
                             "(SURVEY.md Appendix C-9); not supported")
        win_bases = self.OFFSET + (self.NK - 1) * self.STEP + self.K
        if "device_soa" in ctx:
            win = ctx["device_soa"].seq_windows_device(win_bases)      # (rows beyond maxreads are simply not looked at)
        else:
            win = ctx["infile"].seq_windows(win_bases)[:len(ctx["flag"])]
        hist = ctx["engine"].kmer_hist(ctx["flag"], ctx["l_seq"], win, win_bases, self.K, self.NK, self.STEP,
                                       self.OFFSET, group_flags)
        for g, t in enumerate(targets):
            t._counts_data = hist[g].copy()


class BaseHist(ReadProcessor):
    """Out of scope (needs the reference FASTA; undefined without it, Appendix C-9)."""

    def __init__(self, start_pos):
        self.start_pos = start_pos

    def __copy__(self):
        return BaseHist(self.start_pos)


class MirrorHist(ReadProcessor):
    """Out of scope (needs the reference FASTA)."""

    def __init__(self, OFFSET=4, N=10):
        self.OFFSET, self.N = OFFSET, N

    def __copy__(self):
        return MirrorHist(self.OFFSET, self.N)


def kmer_base2_to_ascii(kmer, l):
    """2 bits per base, first base in the low bits (scan.pyx:70-72)."""
    return "".join("ACGT"[(kmer >> n) & 3] for n in range(0, 2 * l, 2))


def scan_reads(infile, fasta, counters, progress_interval=10000000, progress_cb=None, maxreads=0):
    """Drop-in for ``metacov.scan.scan_reads`` (scan.pyx:623-672): every record of
    the file (mapped or not) feeds the counters; returns the number of records.

    progress_cb keeps its cadence (once per progress_interval records), delivered
    at batch granularity."""
    if not isinstance(infile, AlignmentFile):
        raise Exception("meh")               # scan.pyx:642 (FASTQ input is out of scope here)
    if isinstance(counters, list):
        processor = ReadProcessorList(counters)
    elif isinstance(counters, ReadProcessor):
        processor = counters
    else:
        raise Exception("mah")               # scan.pyx:649
    processor.set_max_readlen(50)
    if infile.piped:
        n = _scan_pipe(infile, processor, maxreads)
        if progress_cb:
            for _ in range(n // max(int(progress_interval), 1)):
                progress_cb()
        return n
    gpu = getattr(infile, "_gpu", None)
    if gpu is not None:
        # a file decoded on the GPU: flag / isize / l_seq (and, for KmerHist, the SEQ windows) stay where the decoder left
        # them, the accumulators run on the decoder's own engine, and only the histograms come back
        engine, dsoa = gpu
        n = int(dsoa.n_records)
        if maxreads and n > maxreads:
            n = int(maxreads)
        ctx = {"engine": engine, "infile": infile, "flag": dsoa.device_view("flag", n), "isize": dsoa.device_view("isize", n),
               "l_seq": dsoa.device_view("l_seq", n), "device_soa": dsoa}
        processor._accumulate(ctx, [], [processor])
        if n:
            processor.set_max_readlen(max(50, int(dsoa.to_host("l_seq")[:n].max())))
        if progress_cb:
            for _ in range(n // max(int(progress_interval), 1)):
                progress_cb()
        return n
    soa = infile.soa()
    n = len(soa["flag"])
    if maxreads and n > maxreads:
        n = int(maxreads)
    lengths = infile.lengths if len(infile.lengths) else (1,)
    with CoverageEngine(lengths, device=getattr(infile, "_device", 0)) as engine:
        ctx = {"engine": engine, "infile": infile, "flag": soa["flag"][:n], "isize": soa["isize"][:n],
               "l_seq": soa["l_seq"][:n]}
        processor._accumulate(ctx, [], [processor])
    if n:
        processor.set_max_readlen(max(50, int(soa["l_seq"][:n].max())))
    if progress_cb:
        for _ in range(n // max(int(progress_interval), 1)):
            progress_cb()
    return n


def _scan_pipe(infile, processor, maxreads):
    """``scan_reads`` over a piped SAM stream: the accumulators run on the device columns of every chunk as it is decoded,
    and the chunks' histograms are added up.  ``maxreads`` ends the read after that many records."""
    infile._pipe_claim("scan_reads")
    state = {"n": 0, "rlen": 0}

    def per_chunk(dsoa, n):
        target = processor if state["n"] == 0 else copy(processor)
        ctx = {"engine": dsoa._engine, "infile": infile, "flag": dsoa.device_view("flag", n), "isize": dsoa.device_view("isize", n),
               "l_seq": dsoa.device_view("l_seq", n), "device_soa": dsoa}
        target._accumulate(ctx, [], [target])
        if target is not processor:
            processor._merge(target)
        if n:
            state["rlen"] = max(state["rlen"], int(dsoa.to_host("l_seq")[:n].max()))
        state["n"] += n

    infile._pipe_pass(per_chunk, stop_after=int(maxreads or 0))
    if state["n"]:
        processor.set_max_readlen(max(50, state["rlen"]))
    return state["n"]
