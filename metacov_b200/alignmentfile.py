"""``AlignmentFile``: the subset of the pysam object protocol the coverage path
consumes, backed by the native BGZF/BAM/BAI reader (csrc/bamio.cpp) and the
CUDA depth engine.

Protocol provided (reference call sites): constructor from a path
(metacov/cli.py:56, 211); context manager (cli.py:258); ``references`` /
``lengths`` (util.py:67-68, cli.py:80); ``mapped`` / ``unmapped``
(cli.py:73-75, 214-216); ``pileup(ref, start, end)`` yielding objects with
``.pos`` / ``.n`` (pileup.py:13-16); ``count_coverage(contig, start, stop,
quality_threshold, read_callback)``, the A / C / G / T counts per position
(pysam's signature; computed on the GPU, csrc/basecount.cu).
"""
import ctypes as C
import os

import numpy as np

from . import _capi, samstream
from ._capi import McovError, lib
from .engine import CoverageEngine, ReadBatch


def _view(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=n)


class PileupColumn:
    """Stand-in for pysam.PileupColumn (only ``pos`` and ``n`` are read by the
    reference, pileup.py:14-16)."""
    __slots__ = ("reference_id", "pos", "n")

    def __init__(self, tid, pos, n):
        self.reference_id = tid
        self.pos = pos
        self.n = n

    reference_pos = property(lambda self: self.pos)
    nsegments = property(lambda self: self.n)


class BamStream:
    """The streaming host reader (csrc/bamio.cpp, mcov_bam_stream_*): batches of a BAM decoded into pinned SoA
    buffers, each led by the reads the depth engine asked to see again.  Iterate with ``next_batch(resend)``."""

    def __init__(self, filename, batch_reads=1 << 21, threads=0):
        self._h = C.c_void_p()
        err = C.create_string_buffer(256)
        rc = lib.mcov_bam_stream_open(C.byref(self._h), str(filename).encode(), int(batch_reads), int(threads), err, len(err))
        if rc != 0:
            self._h = None
            raise OSError("%s: %s" % (filename, err.value.decode()))
        n = lib.mcov_bam_stream_n_ref(self._h)
        self.references = tuple(lib.mcov_bam_stream_ref_name(self._h, i).decode() for i in range(n))
        self.lengths = tuple(lib.mcov_bam_stream_ref_len(self._h, i) for i in range(n))
        self.text = lib.mcov_bam_stream_header_text(self._h).decode()

    def next_batch(self, resend=(-1, 0)):
        """(ReadBatch of pinned numpy views, n_carry, last, extra columns) or None after the last batch."""
        b = _capi.BamBatch()
        rc = lib.mcov_bam_stream_next(self._h, int(resend[0]), int(resend[1]), C.byref(b))
        if rc < 0:
            raise McovError(rc, lib.mcov_bam_stream_error(self._h).decode())
        if rc == 0:
            return None
        n = b.n
        batch = ReadBatch(_view(b.tid, n, np.int32), _view(b.pos, n, np.int32), _view(b.flag, n, np.uint16),
                          _view(b.mapq, n, np.uint8), _view(b.cig_off, n + 1, np.uint32), _view(b.cig, b.n_cigar, np.uint32))
        extra = dict(l_seq=_view(b.l_seq, n, np.int32), isize=_view(b.isize, n, np.int32), reflen=_view(b.reflen, n, np.int32))
        return batch, int(b.n_carry), bool(b.last), extra

    def next_block(self, resend=(-1, 0), with_mapq=False):
        """Like ``next_batch`` plus the batch as a transport block: (block or None, ReadBatch, n_carry, last, extra)."""
        b = _capi.BamBatch()
        blk, nb = C.c_void_p(), C.c_int64(0)
        rc = lib.mcov_bam_stream_next_block(self._h, int(resend[0]), int(resend[1]), 1 if with_mapq else 0,
                                            C.byref(blk), C.byref(nb), C.byref(b))
        if rc < 0:
            raise McovError(rc, lib.mcov_bam_stream_error(self._h).decode())
        if rc == 0:
            return None
        n = b.n
        batch = ReadBatch(_view(b.tid, n, np.int32), _view(b.pos, n, np.int32), _view(b.flag, n, np.uint16),
                          _view(b.mapq, n, np.uint8), _view(b.cig_off, n + 1, np.uint32), _view(b.cig, b.n_cigar, np.uint32))
        extra = dict(l_seq=_view(b.l_seq, n, np.int32), isize=_view(b.isize, n, np.int32), reflen=_view(b.reflen, n, np.int32))
        block = (blk.value, nb.value) if blk.value else None
        return block, batch, int(b.n_carry), bool(b.last), extra

    @property
    def n_records(self):
        return lib.mcov_bam_stream_records(self._h)

    def close(self):
        if getattr(self, "_h", None):
            lib.mcov_bam_stream_close(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
        return False


def stream_depth(engine, stream):
    """Per-base depth of a whole sorted BAM through the streamed fused path: batch k+1 is decoded on the host while
    the GPU works on batch k.  Returns the number of batches.  Raises McovError(MCOV_ERR_UNSORTED) -- at the first
    synchronising call on the engine -- when the file is not coordinate-sorted."""
    engine.stream_begin()
    resend = (-1, 0)
    k = 0
    while True:
        item = stream.next_block(resend, with_mapq=engine.filter.min_mapq > 0)
        if item is None:
            if k == 0:
                engine.stream_push(ReadBatch(*[np.zeros(0, d) for d in (np.int32, np.int32, np.uint16, np.uint8)],
                                             np.zeros(1, np.uint32), np.zeros(0, np.uint32)), 0, last=True)
            break
        block, batch, n_carry, last, _ = item
        # the transport block (one narrow host-to-device copy) when the batch qualifies, else its columns
        if block is not None and len(batch.tid):
            rt = engine.stream_push_block(block, last=last)
        else:
            rt = engine.stream_push(batch, n_carry=n_carry, last=last)
        if len(batch.tid):
            resend = rt
        k += 1
        if last:
            break
    return k


def is_sam_text(filename):
    """The format decision of ``AlignmentFile``: SAM text when the file does not start with the gzip magic and its first
    line is a header line ('@' + two letters + TAB) or has at least 11 TAB-separated fields.  Everything else (BAM, an
    empty file, an index, garbage) is left to the BAM readers, which reject what is not BAM."""
    try:
        fh = open(filename, "rb")
    except OSError:
        return False
    with fh:
        line = fh.read(1 << 16)
        if not line or line[:2] == b"\x1f\x8b":
            return False
        while b"\n" not in line and line.count(b"\t") < 10:        # (a long first record: read on to its tenth TAB)
            more = fh.read(1 << 20)
            if not more:
                break
            line += more
    line = line.split(b"\n", 1)[0]
    if len(line) >= 4 and line[:1] == b"@" and line[1:3].isalpha() and line[3:4] == b"\t":
        return True
    return line.count(b"\t") >= 10


def _check_read_callback(read_callback):
    if callable(read_callback) or read_callback not in ("all", "nofilter"):
        raise ValueError("read_callback must be 'all' or 'nofilter' (a callable is not supported: the counts are "
                         "computed on the GPU), got %r" % (read_callback,))


class AlignmentFile:
    def __init__(self, filename, mode="rb", device=0, decode="host", **kw):
        """decode="host": BGZF inflate and record parsing by the native host reader (csrc/bamio.cpp), streamed batch by
        batch; decode="gpu": the compressed file goes to the device and is inflated and parsed there (csrc/bam_gpu.cu) --
        the coverage path then never holds the records on the host, and the file is decoded ~10x faster than 16 host
        cores manage (tools/bench_bam.py), but the compressed image, the inflated stream and the columns must fit the
        device; decode="gpu-stream": the file is read in chunks (``gpu_chunk_bytes``, default 64 MiB) and every chunk is
        inflated, parsed and pushed into the streamed depth pass on the device (mcov_bam_gpu_stream_depth) -- any file size,
        the host only reads; accessors that need every record on the host (soa(), read names) open the host reader on
        demand; decode="auto": "gpu" when the whole file fits the device (file size x GPU_DECODE_FOOTPRINT below the free
        device memory), else "gpu-stream".

        The format comes from the content (``is_sam_text``).  SAM text is always parsed whole on the device
        (csrc/sam_gpu.cu): "host", "gpu" and "auto" all do that and ``decode`` reads "gpu"; "gpu-stream" is refused, and a
        file whose decode does not fit the free device memory raises OSError.

        A stream -- "-" (standard input), a binary file object, or a path that is not a regular file (a FIFO, the
        /dev/fd/N of a pipe) -- is read once, as SAM text, in chunks of whole lines (``gpu_chunk_bytes``, default 64 MiB):
        ``piped`` is True and ``decode`` reads "gpu-stream".  Its header is read by the constructor.  The first consumer
        reads the records: the depth (``coverage_engine`` and everything built on it, ``mapped`` / ``unmapped``
        included) or ``scan_reads``; the other kind, and the accessors that need every record (``soa``, ``len``, read
        names, SEQ), raise ValueError.  Gzip data on a stream (BAM) raises OSError: BAM is read from a file path.
        ``mapped`` / ``unmapped`` of a stream count the records read: all of them after the depth pass, and after a
        ``scan_reads`` that ``maxreads`` stopped, every record of the chunks read up to that point.  The host buffers are
        pageable; ``pinned_buffers=True`` makes them page-locked (tools/bench_pipe.py compares the two)."""
        if "w" in mode:
            raise ValueError("metacov_b200.AlignmentFile is read-only")
        if decode not in ("host", "gpu", "gpu-stream", "auto"):
            raise ValueError("decode must be 'host', 'gpu', 'gpu-stream' or 'auto'")
        self.piped = False
        self._pipe = None
        if samstream.is_stream(filename):
            self._open_pipe(filename, device, kw)
            return
        self.format = "sam" if is_sam_text(filename) else "bam"
        if self.format == "sam":
            if decode == "gpu-stream":
                raise ValueError("%s: SAM text is not streamed; use decode='gpu' (or BAM input)" % filename)
            self._check_sam_fits(filename, device)
            decode = "gpu"
        if decode == "auto":
            decode = "gpu" if self._fits_device(filename, device) else "gpu-stream"
        self._gpu_chunk_bytes = int(kw.get("gpu_chunk_bytes", 64 << 20))
        self.gpu_stream_info = None
        self.decode = decode
        self.filename = filename
        self._gpu = None
        self._device = device
        self._soa = None
        self._engine = None
        self._filter_kw = None
        self._index_stats = None
        self._batch_reads = int(kw.get("batch_reads", 1 << 21))     # records per batch of the streamed depth pass
        self.stream_batches = 0
        self._h = None
        self._stream = None
        self._bc_eng = None                                 # count_coverage of a file that is not resident on the device
        self._bc_key = None                                 # (threshold, mode) of the counts held
        self._ref_fasta = None                              # the FASTA whose sequences the count engine holds
        if decode == "gpu":
            self._open_gpu(filename, device)
            return
        # host decode: only the header is read here (streaming reader: the first blocks of the file); the records are
        # streamed batch by batch by coverage_engine(), or loaded whole by soa() for the callers that need every column
        self._stream = BamStream(filename, batch_reads=self._batch_reads)
        self.references, self.lengths, self.text = self._stream.references, self._stream.lengths, self._stream.text
        self.nreferences = len(self.references)
        self._tid = {name: i for i, name in enumerate(self.references)}

    def _open_pipe(self, source, device, kw):
        """A stream: the header now, the records by the first consumer (``_pipe_pass``)."""
        src, head, rest, owned = samstream.open_stream(source)
        self.format = "sam"
        self.piped = True
        self.decode = "gpu-stream"
        self.filename = source if isinstance(source, str) else getattr(source, "name", "<stream>")
        self._device = device
        self._gpu_chunk_bytes = int(kw.get("gpu_chunk_bytes", 64 << 20))
        self.gpu_stream_info = None
        self.pipe_info = None
        self.stream_batches = 0
        self._gpu = self._soa = self._engine = self._filter_kw = self._index_stats = None
        self._h = self._stream = None
        self._bc_eng = self._bc_key = self._ref_fasta = None
        self._pipe_consumer = None
        self._pipe_read = False
        self._pipe_reader = None
        self._pipe_pinned = bool(kw.get("pinned_buffers", False))
        self.text = head.decode()
        refs = samstream.header_refs(self.text)
        eng = CoverageEngine([1], device=device)
        try:
            n_ref = C.c_int32(0)
            keep = np.frombuffer(head, dtype=np.uint8) if head else None
            rc = lib.mcov_sam_chunk_begin(eng._ctx, keep.ctypes.data if keep is not None else None, len(head), C.byref(n_ref))
            if rc != 0:
                raise OSError("%s: %s" % (self.filename, lib.mcov_last_error(eng._ctx).decode()))
        except BaseException:
            eng.close()
            if owned is not None:
                owned.close()
            raise
        self.references = tuple(r for r, _ in refs)
        self.lengths = tuple(l for _, l in refs)
        self.nreferences = len(refs)
        self._tid = {name: i for i, name in enumerate(self.references)}
        if self.lengths:
            eng.set_contigs(self.lengths)
        self._pipe_eng = eng
        self._pipe = (src, rest, owned)

    def _pipe_claim(self, consumer):
        """The stream goes to its first consumer; a second kind of consumer cannot have it."""
        if self._pipe_consumer is None:
            self._pipe_consumer = consumer
        elif self._pipe_consumer != consumer:
            raise ValueError("%s: a piped SAM stream is read once, and it has been read by %s; %s needs the records again "
                             "(write the stream to a file to use both)" % (self.filename, self._pipe_consumer, consumer))

    def _no_records(self, what):
        if self.piped:
            raise ValueError("%s: %s needs every record, and a piped SAM stream is read once by the depth pass or "
                             "scan_reads without keeping its records (write it to a file instead)" % (self.filename, what))

    def _pipe_pass(self, per_chunk, stop_after=0):
        """Read the stream: every chunk is decoded on the device (``mcov_sam_chunk_decode``) and ``per_chunk(dsoa, n)``
        sees its columns (n: the records of the chunk to use; ``stop_after`` > 0 ends the read after that many records).
        Counts records and mapped / unmapped (BAI definitions) of the chunks read."""
        from . import bamgpu
        if self._pipe_read:
            raise ValueError("%s: the piped SAM stream has been read already (by a pass that did not complete)" % self.filename)
        self._pipe_read = True
        src, rest, _owned = self._pipe
        eng = self._pipe_eng
        reader = samstream.ChunkReader(src, rest, self._gpu_chunk_bytes, pinned=self._pipe_pinned)
        self._pipe_reader = reader
        tot = {"records": 0, "mapped": 0, "unmapped": 0}

        def decode(view, last):
            raw, used = _capi.BamDev(), C.c_int64(0)
            a = np.frombuffer(view, dtype=np.uint8)
            try:
                rc = lib.mcov_sam_chunk_decode(eng._ctx, a.ctypes.data if len(a) else None, len(a), 1 if last else 0,
                                               C.byref(used), C.byref(raw))
            finally:
                del a
            if rc != 0:
                raise OSError("%s: %s" % (self.filename, lib.mcov_last_error(eng._ctx).decode()))
            assert used.value == len(view), (used.value, len(view))
            if raw.n_records == 0:
                return True
            dsoa = bamgpu.DeviceSoA(eng, raw, "sam")
            n = raw.n_records
            if stop_after:
                n = min(n, stop_after - tot["records"])
            per_chunk(dsoa, n)
            m, u = dsoa.mapped_counts()
            tot["records"] += raw.n_records
            tot["mapped"] += m
            tot["unmapped"] += u
            return not (stop_after and tot["records"] >= stop_after)

        reader.run(decode)
        self._index_stats = (tot["mapped"], tot["unmapped"])
        self.pipe_info = dict(records=tot["records"], longest_line=int(lib.mcov_sam_chunk_longest_line(eng._ctx)),
                              **reader.info())
        self.stream_batches = reader.chunks
        return tot["records"]

    def _pipe_depth(self):
        """The depth of a stream: one any-order pass with the exact cap verdict (``mcov_begin_ex``)."""
        self._pipe_claim("the depth pass")
        eng = self._pipe_eng
        if self._filter_kw:
            eng.set_filter(**self._filter_kw)
        eng.begin(exact_cap=True)

        def push(dsoa, n):
            r = dsoa.raw
            eng._check(lib.mcov_push_reads(eng._ctx, n, r.tid, r.pos, r.flag, r.mapq, r.cig_off, r.cig, _capi.MEM_DEVICE))

        self._pipe_pass(push)
        eng.finalize()
        info = eng.pass_info()
        md = eng.filter.max_depth
        if md > 0 and info["cap_metric"] > md:
            from .pileup import DepthCapError
            raise DepthCapError(
                "%s: depth[p-1]+starts[p] reaches %d > max_depth=%d: htslib's pileup would drop reads here, and a piped "
                "stream cannot be read again to replay its cap; write the input to a coordinate-sorted file instead, or "
                "raise max_depth via set_pileup_filter(max_depth=...) before the first use" % (self.filename, info["cap_metric"], md))
        self._engine = eng
        return eng

    # device bytes per byte of BAM that a GPU decode needs: the image itself, the inflated stream (BAM records deflate
    # ~4-5x), the SoA columns, and as much again for the depth arrays and scratch of the pass that follows
    GPU_DECODE_FOOTPRINT = 12

    @classmethod
    def _fits_device(cls, filename, device):
        import torch
        try:
            size = os.path.getsize(filename)
            free, _total = torch.cuda.mem_get_info(device)
        except (OSError, RuntimeError):
            return False
        return size * cls.GPU_DECODE_FOOTPRINT < free

    # device bytes per byte of SAM text that the decode holds: the text (1), and per line -- 23 bytes at the least -- its
    # end (8), the columns (23), the record offset (8), the field offsets (16) and the op count (8): 63 / 23 < 2.8; each
    # CIGAR op (4 bytes, at least 2 of text) stays below that ratio.  With DevBuf's 1/8 growth margin: 1.125 x 3.8 < 4.3,
    # rounded up to leave room for the depth pass that follows.
    SAM_DECODE_FOOTPRINT = 5

    @classmethod
    def _check_sam_fits(cls, filename, device):
        import torch
        try:
            size = os.path.getsize(filename)
            free, _total = torch.cuda.mem_get_info(device)
        except (OSError, RuntimeError):
            return                                          # (no size or no device: the decode itself reports it)
        if size * cls.SAM_DECODE_FOOTPRINT >= free:
            raise OSError("%s: a SAM file of %d bytes needs about %d bytes of device memory to decode, %d are free; "
                          "SAM is decoded whole on the device, while BAM input streams (decode='gpu-stream')"
                          % (filename, size, size * cls.SAM_DECODE_FOOTPRINT, free))

    def _open_gpu(self, filename, device):
        from . import bamgpu
        self._h = None
        eng = CoverageEngine([1], device=device)            # the contig table follows once the header is decoded
        try:
            # (the library maps the file: no host copy of the image)
            if self.format == "sam":
                dsoa = bamgpu.decode_sam(eng, os.fspath(filename))
            else:
                dsoa = bamgpu.decode(eng, os.fspath(filename))
            self.text, refs = dsoa.header()
        except McovError as e:
            eng.close()
            raise OSError("%s: %s" % (filename, e))
        except BaseException:
            eng.close()
            raise
        self.references = tuple(r for r, _ in refs)
        self.lengths = tuple(l for _, l in refs)
        self.nreferences = len(refs)
        self._tid = {name: i for i, name in enumerate(self.references)}
        eng.set_contigs(self.lengths)
        self._gpu = (eng, dsoa)

    def _host_handle(self):
        """The host reader's handle (a GPU-decoded file never needs it: columns, read names and SEQ all come from
        the device, bamgpu.DeviceSoA)."""
        if self._h is None:
            self._open_host(self.filename, header=False)
        return self._h

    def _open_host(self, filename, header=True):
        self._h = C.c_void_p()
        err = C.create_string_buffer(256)
        rc = lib.mcov_bam_open(C.byref(self._h), str(filename).encode(), err, len(err))
        if rc != 0:
            self._h = None
            # pysam raises OSError/ValueError for unreadable files
            raise OSError("%s: %s" % (filename, err.value.decode()))
        if not header:
            return
        n = lib.mcov_bam_n_ref(self._h)
        self.references = tuple(lib.mcov_bam_ref_name(self._h, i).decode() for i in range(n))
        self.lengths = tuple(lib.mcov_bam_ref_len(self._h, i) for i in range(n))
        self.nreferences = n
        self.text = lib.mcov_bam_header_text(self._h).decode()
        self._tid = {name: i for i, name in enumerate(self.references)}

    # -- lifetime ---------------------------------------------------------
    def close(self):
        if getattr(self, "_pipe", None) is not None:
            if self._engine is self._pipe_eng:
                self._engine = None
            self._pipe_eng.close()
            owned = self._pipe[2]
            if owned is not None:
                if self._pipe_reader is not None:
                    self._pipe_reader.release(owned.close)   # (after an early stop: once the reader thread is out)
                else:
                    owned.close()
            self._pipe = None
        if getattr(self, "_engine", None) is not None:
            self._engine.close()
            self._engine = None
        if getattr(self, "_gpu", None) is not None:
            self._gpu[0].close()                            # (the same engine, if the depth was computed)
            self._gpu = None
        if getattr(self, "_bc_eng", None) is not None:
            self._bc_eng.close()
            self._bc_eng = None
        if getattr(self, "_h", None):
            lib.mcov_bam_close(self._h)
            self._h = None
        if getattr(self, "_stream", None) is not None:
            self._stream.close()
            self._stream = None
        self._soa = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
        return False

    # -- header / index ---------------------------------------------------
    def get_tid(self, reference):
        return self._tid.get(reference, -1)

    def get_reference_name(self, tid):
        return self.references[tid]

    def _idx(self):
        if self._index_stats is None and self.piped:
            self.coverage_engine()                          # (counted while the stream is read)
        if self._index_stats is None and self.format == "sam":
            self._index_stats = self._gpu[1].mapped_counts()      # (SAM has no index: counted from the decoded columns)
        if self._index_stats is None:
            m, u = C.c_int64(0), C.c_int64(0)
            rc = lib.mcov_bai_stats(str(self.filename).encode(), C.byref(m), C.byref(u))
            if rc != 0:
                raise ValueError("mapping information not recorded in index or index not available")
            self._index_stats = (m.value, u.value)
        return self._index_stats

    @property
    def mapped(self):
        return self._idx()[0]

    @property
    def unmapped(self):
        return self._idx()[1]

    def has_index(self):
        if self.format == "sam":
            return False
        try:
            self._idx()
            return True
        except ValueError:
            return False

    # -- records ----------------------------------------------------------
    def soa(self):
        """Every record of the file as SoA numpy views (file order; the arrays
        the reference reads field by field at scan.pyx:243-294)."""
        self._no_records("soa()")
        if self._soa is None and self._gpu is not None:
            self._soa = {c: self._gpu[1].to_host(c) for c, _ in self._gpu[1].COLS}
        if self._soa is None:
            self._host_handle()
            rc = lib.mcov_bam_load(self._h, 0)
            if rc != 0:
                raise McovError(rc, "BAM record decode failed")
            n = lib.mcov_bam_n_records(self._h)
            nc = lib.mcov_bam_n_cigar(self._h)
            self._soa = dict(
                tid=_view(lib.mcov_bam_tid(self._h), n, np.int32),
                pos=_view(lib.mcov_bam_pos(self._h), n, np.int32),
                flag=_view(lib.mcov_bam_flag(self._h), n, np.uint16),
                mapq=_view(lib.mcov_bam_mapq(self._h), n, np.uint8),
                l_seq=_view(lib.mcov_bam_lseq(self._h), n, np.int32),
                isize=_view(lib.mcov_bam_isize(self._h), n, np.int32),
                cig_off=_view(lib.mcov_bam_cig_off(self._h), n + 1, np.uint32),
                cig=_view(lib.mcov_bam_cig(self._h), nc, np.uint32),
            )
        return self._soa

    def seq_windows(self, win_bases):
        """uint8[n, (win_bases+1)//2]: per read the first (forward) / last (reverse) win_bases bases,
        nt16 two per byte -- the part of SEQ the k-mer histogram looks at."""
        self._no_records("seq_windows()")
        if self._gpu is not None:                       # decoded on the GPU: SEQ is read there too
            return self._gpu[1].names_seq(win_bases=win_bases)["seq_win"]
        n = len(self.soa()["tid"])
        rc = lib.mcov_bam_load_seq(self._host_handle())
        if rc != 0:
            raise McovError(rc, "BAM SEQ decode failed")
        out = np.empty((n, (win_bases + 1) // 2), dtype=np.uint8)
        rc = lib.mcov_bam_seq_windows(self._host_handle(), int(win_bases), _capi.ptr(out))
        if rc != 0:
            raise McovError(rc, "mcov_bam_seq_windows failed")
        return out

    def __len__(self):
        self._no_records("len()")
        return len(self.soa()["tid"])

    # -- pileup.experimental ------------------------------------------------
    def name_hashes(self):
        """uint64[n]: FNV-1a of every read name (the key of the reference's mate dict, pileup.py:101)."""
        self._no_records("name_hashes()")
        if self._gpu is not None:
            return self._gpu[1].names_seq(name_hash=True)["name_hash"]
        n = len(self.soa()["tid"])
        rc = lib.mcov_bam_load_seq(self._host_handle())
        if rc != 0:
            raise McovError(rc, "BAM SEQ decode failed")
        return _view(lib.mcov_bam_name_hash(self._host_handle()), n, np.uint64)

    def qas_kmer_codes(self, k_len):
        """int32[n]: code of ``read.query_alignment_sequence[0:k_len]`` (pileup.py:109, 123), -1 = no key."""
        self._no_records("qas_kmer_codes()")
        if self._gpu is not None:
            return self._gpu[1].names_seq(k_len=k_len)["kmer_code"]
        n = len(self.soa()["tid"])
        rc = lib.mcov_bam_load_seq(self._host_handle())
        if rc != 0:
            raise McovError(rc, "BAM SEQ decode failed")
        out = np.empty(n, dtype=np.int32)
        rc = lib.mcov_bam_qas_kmer(self._host_handle(), int(k_len), _capi.ptr(out))
        if rc != 0:
            raise McovError(rc, "mcov_bam_qas_kmer failed")
        return out

    def _fetch_index(self):
        """Per-contig record ranges and the longest reference span: what stands in for the BAI when
        a region's candidate records are looked up (``bam.fetch`` needs a sorted, indexed file)."""
        if getattr(self, "_fidx", None) is None:
            s = self.soa()
            # (contig, position) as one sortable key; unplaced reads (tid -1 -> 2^32-1) sort last
            key = (s["tid"].view(np.uint32).astype(np.int64) << 31) | s["pos"].astype(np.int64).clip(0)
            if len(key) > 1 and np.any(key[1:] < key[:-1]):
                raise ValueError("fetch called on bamfile without index")          # pysam's message
            ut = s["tid"].view(np.uint32)
            cstart = np.searchsorted(ut, np.arange(self.nreferences + 1, dtype=np.uint32), side="left")
            consumes = np.array([1, 0, 1, 1, 0, 0, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0], dtype=np.int64)   # M D N = X
            per_op = (s["cig"] >> 4).astype(np.int64) * consumes[s["cig"] & 15]
            csum = np.concatenate(([0], np.cumsum(per_op)))
            reflen = csum[s["cig_off"][1:]] - csum[s["cig_off"][:-1]]
            self._fidx = (cstart, int(max(reflen.max(initial=0), 1)))
        return self._fidx

    def experimental_stats(self, refs, starts, ends, k_len, kc_val, kc_has):
        """``mcov_exp_stats`` records of the regions (the read loop of pileup.py:90-146 on the GPU)."""
        self._no_records("experimental_stats()")
        s = self.soa()
        cstart, max_span = self._fetch_index()
        pos = s["pos"]
        g = len(refs)
        lb = np.zeros(g, dtype=np.int64)
        ub = np.zeros(g, dtype=np.int64)
        for i, (ref, s0, e0) in enumerate(zip(refs, starts, ends)):
            tid = self._tid[ref]                                             # KeyError for unknown contigs, like pysam
            c0, c1 = int(cstart[tid]), int(cstart[tid + 1])
            lb[i] = c0 + np.searchsorted(pos[c0:c1], s0 - max_span, side="right")
            ub[i] = c0 + np.searchsorted(pos[c0:c1], e0, side="left")
            ub[i] = max(ub[i], lb[i])
        hashes = self.name_hashes()
        codes = self.qas_kmer_codes(k_len) if kc_val is not None else np.full(len(pos), -1, dtype=np.int32)
        eng = self.coverage_engine()
        out = np.zeros(g, dtype=_capi.EXP_STATS_DTYPE)
        # batches bounded by the scratch they need: (region, read) entries and last-writer slots
        i = 0
        while i < g:
            j, ent, slots = i, 0, 0
            while j < g and (j == i or (ent + ub[j] - lb[j] < (1 << 30) and slots + ends[j] - starts[j] < (1 << 29))):
                ent += int(ub[j] - lb[j]); slots += int(ends[j] - starts[j]); j += 1
            # only the reads the batch's regions can touch travel to the device: [lo, hi) of the file order (a single region
            # of a 10 M-read file is a few thousand reads, not 266 MB of columns)
            lo, hi = int(lb[i:j].min()), int(ub[i:j].max())
            hi = max(hi, lo)
            o0, o1 = int(s["cig_off"][lo]), int(s["cig_off"][hi])
            sub = {"pos": s["pos"][lo:hi], "flag": s["flag"][lo:hi], "cig": s["cig"][o0:o1],
                   "cig_off": (s["cig_off"][lo:hi + 1] - np.uint32(o0)).astype(np.uint32)}
            out[i:j] = eng.experimental_stats(sub, hashes[lo:hi], codes[lo:hi], k_len, kc_val, kc_has,
                                              np.asarray(starts[i:j], dtype=np.int32), np.asarray(ends[i:j], dtype=np.int32),
                                              lb[i:j] - lo, ub[i:j] - lo)
            i = j
        return out

    # -- coverage ---------------------------------------------------------
    def set_pileup_filter(self, **kw):
        """Override pysam's implicit pileup arguments (flag_filter, flag_require,
        min_mapq, ignore_orphans, max_depth); invalidates the cached depth.  A piped stream takes it before its
        records are read only."""
        if self.piped and self._pipe_consumer is not None:
            raise ValueError("%s: set_pileup_filter after the piped stream has been read: its depth cannot be computed "
                             "again; set the filter before the first use" % self.filename)
        self._filter_kw = kw
        if self._engine is not None:
            if self._gpu is None:
                self._engine.close()                        # (a GPU-decoded file keeps its engine: it owns the columns)
            self._engine = None

    def coverage_engine(self):
        """The per-base depth of the whole file, computed once on the GPU."""
        if self.piped:
            return self._engine if self._engine is not None else self._pipe_depth()
        if self._engine is None and self._gpu is not None:
            eng, path = self._gpu_depth()
        elif self._engine is None and self._soa is None:
            # host decode, records not loaded: stream the file in batches (never held in memory); a file that is not
            # coordinate-sorted, or one where htslib's max_depth cap fires, takes the whole-file path below
            eng = CoverageEngine(self.lengths, device=self._device, filt=self._filter_kw)
            path = None
            if self.decode == "gpu-stream":
                # chunks of the file through the GPU decoder into the streamed pass; a file it cannot take (not sorted, the
                # max_depth cap fires) falls through to the host paths below, which know what to do with it
                from . import bamgpu
                try:
                    self.gpu_stream_info = bamgpu.stream_depth(eng, self.filename, chunk_bytes=self._gpu_chunk_bytes)
                    eng.pass_info()
                    path = "fused"
                    self.stream_batches = self.gpu_stream_info["n_chunks"]
                except McovError as e:
                    if e.code not in (_capi.MCOV_ERR_UNSORTED, _capi.MCOV_ERR_RANGE, _capi.MCOV_ERR_STATE):
                        eng.close()
                        raise
            if path is None and self.decode != "gpu-stream":    # (what the GPU stream refused, the host stream would refuse too)
                try:
                    st, self._stream = self._stream, None       # the reader opened for the header, not yet advanced
                    if st is None:
                        st = BamStream(self.filename, batch_reads=self._batch_reads)
                    with st:
                        self.stream_batches = stream_depth(eng, st)
                    eng.pass_info()                              # delivers the verdict of the stream
                    path = "fused"
                except McovError as e:
                    if e.code not in (_capi.MCOV_ERR_UNSORTED, _capi.MCOV_ERR_RANGE, _capi.MCOV_ERR_STATE):
                        eng.close()
                        raise
            if path is None:
                s = self.soa()
                path = eng.compute_depth(ReadBatch(s["tid"], s["pos"], s["flag"], s["mapq"], s["cig_off"], s["cig"]))
        elif self._engine is None:
            s = self.soa()
            eng = CoverageEngine(self.lengths, device=self._device, filt=self._filter_kw)
            path = eng.compute_depth(ReadBatch(s["tid"], s["pos"], s["flag"], s["mapq"], s["cig_off"], s["cig"]))
        if self._engine is None:
            info = eng.pass_info()
            md = eng.filter.max_depth
            # the fused (sorted) path replays htslib's cap exactly on the GPU; the any-order path cannot
            # (the cap is only defined for sorted input), so it refuses rather than return uncapped numbers
            if path != "fused" and md > 0 and info["cap_metric"] > md:
                if self._gpu is None:
                    eng.close()
                from .pileup import DepthCapError
                raise DepthCapError(
                    "depth[p-1]+starts[p] reaches %d > max_depth=%d: htslib's pileup would drop reads here "
                    "(order-dependent cap); raise max_depth via set_pileup_filter(max_depth=...)"
                    % (info["cap_metric"], md))
            self._engine = eng
        return self._engine

    def _gpu_depth(self):
        """Depth straight from the device-resident columns of a GPU-decoded file."""
        from . import bamgpu
        eng, dsoa = self._gpu
        if self._filter_kw:
            eng.set_filter(**self._filter_kw)
        try:
            bamgpu.depth_sorted(eng, dsoa)
            return eng, "fused"
        except McovError as e:
            if e.code not in (_capi.MCOV_ERR_UNSORTED, _capi.MCOV_ERR_RANGE):
                raise
        r = dsoa.raw
        eng.begin()
        eng._check(lib.mcov_push_reads(eng._ctx, dsoa.n_records, r.tid, r.pos, r.flag, r.mapq, r.cig_off, r.cig, _capi.MEM_DEVICE))
        eng.finalize()
        return eng, "push"

    def pileup(self, contig=None, start=None, stop=None, **kw):
        """Columns with n > 0 inside [start, stop) (pysam also emits columns
        outside the region when truncate=False; the reference discards them,
        pileup.py:14-15)."""
        tid = self._tid[contig]
        start = 0 if start is None else max(int(start), 0)
        stop = self.lengths[tid] if stop is None else min(int(stop), self.lengths[tid])
        d = self.coverage_engine().copy_depth(tid, start, stop) if stop > start else np.zeros(0, np.int32)
        for off in np.nonzero(d)[0]:
            yield PileupColumn(tid, start + int(off), int(d[off]))

    def count_coverage_depth(self, contig, start=None, stop=None):
        """Per-base depth as an int32 array (additive helper)."""
        tid = self._tid[contig]
        return self.coverage_engine().copy_depth(tid, 0 if start is None else start, stop)

    def count_coverage(self, contig, start=None, stop=None, quality_threshold=15, read_callback="all"):
        """pysam's ``count_coverage``: four ``numpy.uint32`` arrays (A, C, G, T), each ``stop - start`` long, index k =
        position start + k, counted on the GPU over the whole file once per (threshold, read_callback) and sliced.

        ``start`` None -> 0, ``stop`` None -> the contig length (a larger ``stop`` is clipped to it); an empty or
        negative interval or a negative ``start`` raises ValueError, an unknown contig KeyError.  ``read_callback``
        "all" skips records flagged 0x4, 0x100, 0x200 or 0x400, "nofilter" none; anything else, a callable included,
        raises ValueError.  Every (qpos, refpos) pair of an M / = / X op counts where the base is A, C, G or T and,
        with ``quality_threshold`` (None = 0) non-zero, the read has qualities and the base's quality is at least the
        threshold.  No MAPQ, orphan or max_depth filter; ``set_pileup_filter`` does not apply.  A record whose CIGAR
        consumes more query bases than its SEQ holds raises IndexError naming it, as pysam does; counters that do not fit
        the free device memory raise MemoryError.

        Deliberate differences from pysam: the file need not be coordinate-sorted or indexed (pysam's ``fetch`` needs
        both); under "nofilter", a record flagged unmapped that carries a CIGAR counts by its CIGAR everywhere, where
        pysam's ``fetch`` returns it only for intervals that contain its POS.  Files decoded on the device count from
        the resident records; others (``decode="host"`` / ``"gpu-stream"``) go through the GPU decoder chunk by chunk.
        The depth and its statistics are left as they were.  A piped stream raises ValueError."""
        self._no_records("count_coverage()")
        _check_read_callback(read_callback)
        tid = self._tid[contig]                             # KeyError for unknown contigs, like pysam
        length = int(self.lengths[tid])
        start = 0 if start is None else int(start)
        stop = length if stop is None else min(int(stop), length)
        if start < 0:
            raise ValueError("start out of range (%d)" % start)
        if stop == start:
            raise ValueError("interval of size 0")
        if stop < start:
            raise ValueError("interval of size less than 0")
        eng = self._counted(quality_threshold, read_callback)
        c = eng.copy_base_counts(tid, start, stop)
        return c[0], c[1], c[2], c[3]

    def _counted(self, quality_threshold, read_callback):
        """The count engine holding the counts of (threshold, read_callback): counted now unless they are held."""
        t = max(min(int(quality_threshold or 0), 2 ** 31 - 1), -2 ** 31)
        mode = _capi.MCOV_BC_NOFILTER if read_callback == "nofilter" else _capi.MCOV_BC_ALL
        eng = self._count_engine()
        if self._bc_key != (t, mode):
            self._bc_key = None
            try:
                if self._gpu is not None:
                    eng.base_counts(t, mode)
                else:
                    eng.base_counts(t, mode, path=self.filename, chunk_bytes=self._gpu_chunk_bytes)
            except McovError as e:
                if e.code == _capi.MCOV_ERR_IO and "consumes more query bases" in str(e):
                    raise IndexError("%s: %s" % (self.filename, e))         # (pysam's error there)
                self._raise_nomem(e)
                if e.code == _capi.MCOV_ERR_IO:
                    raise OSError("%s: %s" % (self.filename, e))
                raise
            self._bc_key = (t, mode)
        return eng

    def allele_stats(self, contigs=None, starts=None, stops=None, fasta=None, quality_threshold=15, read_callback="all",
                     min_coverage=5, min_freq=0.05, min_count=2):
        """Allele statistics of regions from the A / C / G / T counts of ``count_coverage`` (same counts, same cache):
        a structured array (``_capi.ALLELE_STATS_DTYPE``) with one record per region -- length, covered, depth_sum,
        pi_sum, snv, ref_covered, sub, popsub; ``alleles.derive`` turns it into breadth, depth, pi, SNVs per kbp and the
        consensus / population ANI.  The rules are those of ``mcov_allele_stats_run`` (include/metacov_b200.h).

        Regions: ``contigs`` (names; default every contig), ``starts`` (default 0) and ``stops`` (default the contig
        length), 0-based half-open; they may overlap and reach past the contig end.  ``fasta`` (a ``FastaFile``, or
        anything with ``references`` and ``fetch``) gives the reference bases for SUB / POPSUB: each contig is looked up
        by the first word of its name and must have the contig's length, else ValueError naming it; a FASTA is sent to
        the GPU once per file.  Without it the reference is unknown everywhere.  Bad parameters or regions raise
        ValueError, an unknown contig KeyError, a piped stream ValueError."""
        eng, use_ref = self._allele_engine("allele_stats()", fasta, quality_threshold, read_callback,
                                           min_coverage, min_freq, min_count)
        tid, start, stop = self._regions(contigs, starts, stops)
        return eng.allele_stats(tid, start, stop, min_coverage, min_freq, min_count, use_reference=use_ref)

    def _regions(self, contigs, starts, stops):
        """(tid, start, stop) int64 arrays of regions given as in ``allele_stats``: ValueError for bad regions,
        KeyError for an unknown contig."""
        if contigs is None:
            contigs = self.references
        elif isinstance(contigs, str):
            contigs = [contigs]
        tid = np.array([self._tid[c] for c in contigs], dtype=np.int64)
        lengths = np.asarray(self.lengths, dtype=np.int64)
        start = np.zeros(len(tid), np.int64) if starts is None else np.asarray(starts, dtype=np.int64).reshape(-1)
        stop = lengths[tid] if stops is None else np.asarray(stops, dtype=np.int64).reshape(-1)
        if not len(start) == len(stop) == len(tid):
            raise ValueError("contigs, starts and stops differ in length")
        if len(tid) and (start.min() < 0 or (stop < start).any() or stop.max() >= 2 ** 31):
            raise ValueError("regions need 0 <= start <= stop < 2^31")
        return tid, start, stop

    def allele_sites(self, fasta=None, quality_threshold=15, read_callback="all", min_coverage=5, min_freq=0.05,
                     min_count=2):
        """Every site -- a covered position where two or more alleles are present (SNV, kind bit 1) or, with ``fasta``,
        where the consensus differs from the reference (SUB, 2) or the reference base is not present (POPSUB, 4) -- in
        (tid, pos) order: a structured array (``_capi.ALLELE_SITE_DTYPE``: tid pos A C G T ref consensus kind).
        Arguments as in ``allele_stats``."""
        eng, use_ref = self._allele_engine("allele_sites()", fasta, quality_threshold, read_callback,
                                           min_coverage, min_freq, min_count)
        return eng.allele_sites(min_coverage, min_freq, min_count, use_reference=use_ref)

    def allele_signature(self, quality_threshold=15, read_callback="all", min_coverage=5, min_freq=0.05, min_count=2):
        """The signature of every slot of the count engine's table from the counts of ``count_coverage`` (same counts,
        same cache): a CUDA ``torch.uint8`` tensor of ``n_slots`` bytes, 0x80 covered, bits 4-5 the consensus (0-3 =
        A C G T), bits 0-3 the present mask, 0 where not covered.  It is what ``compare`` keeps of a file.  Arguments as
        in ``allele_stats``; a piped stream raises ValueError."""
        eng, _ = self._allele_engine("allele_signature()", None, quality_threshold, read_callback,
                                     min_coverage, min_freq, min_count)
        return eng.allele_signature(min_coverage, min_freq, min_count)

    def _allele_engine(self, what, fasta, quality_threshold, read_callback, min_coverage, min_freq, min_count):
        """The count engine with the counts of (threshold, read_callback) and, given a FASTA, its reference."""
        self._no_records(what)
        _check_read_callback(read_callback)
        CoverageEngine._allele_params(min_coverage, min_freq, min_count, False)      # (ValueError before any work)
        eng = self._counted(quality_threshold, read_callback)
        if fasta is not None and self._ref_fasta is not fasta:
            self._ref_fasta = None
            names = set(fasta.references)
            for tid, name in enumerate(self.references):
                key = (name.split() or [name])[0]
                if key not in names:
                    raise ValueError("%s: contig %r is not in the reference FASTA" % (self.filename, name))
                seq = fasta.fetch(key)
                if len(seq) != int(self.lengths[tid]):
                    raise ValueError("%s: contig %r is %d long in the reference FASTA and %d in the alignments"
                                     % (self.filename, name, len(seq), int(self.lengths[tid])))
                try:
                    eng.set_reference(tid, seq)
                except McovError as e:
                    self._raise_nomem(e)
                    raise
            self._ref_fasta = fasta
        return eng, fasta is not None

    def _raise_nomem(self, e):
        """MemoryError naming the file for an McovError of device memory that does not fit (MCOV_ERR_NOMEM)."""
        if e.code == _capi.MCOV_ERR_NOMEM:
            raise MemoryError("%s: %s" % (self.filename, e))

    def _count_engine(self):
        """The engine that counts: a device-decoded file's own (it holds the records); else one of the counts' own."""
        if self._gpu is not None:
            return self._gpu[0]
        if self._bc_eng is None:
            self._bc_eng = CoverageEngine(self.lengths, device=self._device)
        return self._bc_eng
