"""BAM and SAM decode on the GPU (SURVEY.md 8(f) row 3): the compressed file goes to the device, BGZF blocks are
inflated and the records parsed there (csrc/bam_gpu.cu), and the SoA columns stay in HBM for the coverage
kernels.  Replaces, for this path, ``pysam.AlignmentFile`` + ``IteratorRowAll`` (reference
metacov/scan.pyx:204, 216; cli.py:56) without the host decode of ``alignmentfile.AlignmentFile``.

    eng = CoverageEngine(lengths)
    soa = bamgpu.decode(eng, "reads.bam")        # device-resident columns, owned by the engine's context
    soa = bamgpu.decode_sam(eng, "reads.sam")    # (the same columns from SAM text)
    bamgpu.depth_sorted(eng, soa)                # per-base depth straight from them
"""
import ctypes as C
import os

import numpy as np

from . import _capi, samstream
from ._capi import lib


class DevView:
    """A device pointer with a length: quacks like a CUDA tensor for the engine's pointer-taking calls."""
    is_cuda = True

    def __init__(self, ptr, n):
        self._ptr, self._n = int(ptr or 0), int(n)
        self.shape = (self._n,)

    def data_ptr(self):
        return self._ptr

    def __len__(self):
        return self._n


class DeviceSoA:
    """Device pointers of a decoded BAM or SAM (``mcov_bam_dev``; ``format`` "bam" or "sam"); valid until the next decode
    on the same engine."""

    COLS = (("tid", np.int32), ("pos", np.int32), ("flag", np.uint16), ("mapq", np.uint8), ("l_seq", np.int32),
            ("isize", np.int32), ("cig_off", np.uint32), ("cig", np.uint32))

    def __init__(self, engine, raw, format="bam"):
        self._engine = engine
        self.raw = raw
        self.format = format
        self.n_records, self.n_cigar, self.n_ref = raw.n_records, raw.n_cigar, raw.n_ref
        self.inflated_bytes, self.header_bytes, self.n_segments = raw.inflated_bytes, raw.header_bytes, raw.n_segments

    def _len(self, name):
        return self.n_cigar if name == "cig" else (self.n_records + 1 if name == "cig_off" else self.n_records)

    def device_view(self, name, n=None):
        """One column as a device-resident view (``DevView``: pointer + length, what the engine's calls take for
        device memory) -- valid until the next decode on the same engine."""
        return DevView(getattr(self.raw, name), self._len(name) if n is None else int(n))

    def to_host(self, name):
        """One column copied to a numpy array (tests, accessors)."""
        dt = dict(self.COLS)[name]
        out = np.empty(self._len(name), dtype=dt)
        self._engine._check(lib.mcov_copy_to_host(self._engine._ctx, getattr(self.raw, name), _capi.ptr(out), out.nbytes))
        return out

    def seq_windows_device(self, win_bases):
        """The k-mer histogram's view of SEQ left ON THE DEVICE: a torch uint8 tensor [n, (win_bases+1)//2]."""
        import torch
        n = self.n_records
        out = torch.empty((n, (win_bases + 1) // 2), dtype=torch.uint8, device="cuda:%d" % self._engine.device)
        if n:
            self._engine._check(lib.mcov_bam_gpu_names_seq(self._engine._ctx, 0, int(win_bases), None, None, out.data_ptr(),
                                                           _capi.MEM_DEVICE))
        return out

    def names_seq(self, name_hash=False, k_len=0, win_bases=0):
        """Read names and SEQ computed on the device from the inflated stream (``mcov_bam_gpu_names_seq``): a dict with
        ``name_hash`` uint64[n] (FNV-1a of query_name), ``kmer_code`` int32[n] (query_alignment_sequence[0:k_len], -1 = no
        key) and ``seq_win`` uint8[n, (win_bases+1)//2] (the k-mer histogram's view of SEQ), whichever were asked for."""
        n = self.n_records
        out = {}
        if name_hash:
            out["name_hash"] = np.empty(n, dtype=np.uint64)
        if k_len:
            out["kmer_code"] = np.empty(n, dtype=np.int32)
        if win_bases:
            out["seq_win"] = np.empty((n, (win_bases + 1) // 2), dtype=np.uint8)
        p = lambda k: _capi.ptr(out[k]) if k in out and n else None
        self._engine._check(lib.mcov_bam_gpu_names_seq(self._engine._ctx, int(k_len), int(win_bases), p("name_hash"),
                                                       p("kmer_code"), p("seq_win"), _capi.MEM_HOST))
        return out

    def mapped_counts(self):
        """(mapped, unmapped) counted on the device from the columns, with the BAI metadata definitions
        (``mcov_bam_gpu_mapped``)."""
        m, u = C.c_int64(0), C.c_int64(0)
        self._engine._check(lib.mcov_bam_gpu_mapped(self._engine._ctx, C.byref(m), C.byref(u)))
        return m.value, u.value

    def header(self):
        """(text, [(name, length)]) parsed from the inflated stream's header (SAM spec 4.2), or from the '@' lines of a
        SAM file (text: those lines as in the file; references: @SQ SN / LN in order)."""
        buf = np.empty(self.header_bytes, dtype=np.uint8)
        if buf.nbytes:
            self._engine._check(lib.mcov_copy_to_host(self._engine._ctx, self.raw.inflated, _capi.ptr(buf), buf.nbytes))
        b = buf.tobytes()
        if self.format == "sam":
            text = b.decode()
            return text, samstream.header_refs(text)
        l_text = int.from_bytes(b[4:8], "little")
        text = b[8:8 + l_text].split(b"\0")[0].decode()
        p = 8 + l_text
        n_ref = int.from_bytes(b[p:p + 4], "little")
        p += 4
        refs = []
        for _ in range(n_ref):
            ln = int.from_bytes(b[p:p + 4], "little")
            name = b[p + 4:p + 4 + ln - 1].decode()
            refs.append((name, int.from_bytes(b[p + 4 + ln:p + 8 + ln], "little")))
            p += 8 + ln
        return text, refs


def decode(engine, source, verify_crc=True):
    """Decode a BAM on the GPU.  ``source``: a path, ``bytes`` or a uint8 numpy array / pinned torch tensor
    holding the file image.  Returns a ``DeviceSoA``."""
    keep = None
    if isinstance(source, (str, os.PathLike)):              # a path: the library maps the file itself
        raw = _capi.BamDev()
        engine._check(lib.mcov_bam_decode_gpu_file(engine._ctx, os.fsencode(source), 1 if verify_crc else 0, C.byref(raw)))
        return DeviceSoA(engine, raw)
    if isinstance(source, bytes):
        keep = np.frombuffer(source, dtype=np.uint8)
        ptr, n = keep.ctypes.data, keep.nbytes
    elif hasattr(source, "data_ptr"):
        keep = source
        ptr, n = source.data_ptr(), source.numel() * source.element_size()
    else:
        keep = np.ascontiguousarray(source, dtype=np.uint8)
        ptr, n = keep.ctypes.data, keep.nbytes
    raw = _capi.BamDev()
    engine._check(lib.mcov_bam_decode_gpu(engine._ctx, ptr, n, 1 if verify_crc else 0, C.byref(raw)))
    del keep
    return DeviceSoA(engine, raw)


def decode_sam(engine, source, chunk_bytes=0):
    """Parse a SAM text file on the GPU into the same device-resident columns as ``decode`` (csrc/sam_gpu.cu).
    ``source``: a path, ``bytes`` or a uint8 numpy array / pinned torch tensor holding the file image; ``chunk_bytes``: the
    size of the copies the newline count overlaps (0 = 64 MiB).  Returns a ``DeviceSoA`` of format "sam"."""
    raw = _capi.BamDev()
    if isinstance(source, (str, os.PathLike)):
        engine._check(lib.mcov_sam_decode_gpu_file(engine._ctx, os.fsencode(source), int(chunk_bytes), C.byref(raw)))
        return DeviceSoA(engine, raw, "sam")
    if isinstance(source, bytes):
        keep = np.frombuffer(source, dtype=np.uint8)
        ptr, n = keep.ctypes.data, keep.nbytes
    elif hasattr(source, "data_ptr"):
        keep = source
        ptr, n = source.data_ptr(), source.numel() * source.element_size()
    else:
        keep = np.ascontiguousarray(source, dtype=np.uint8)
        ptr, n = keep.ctypes.data, keep.nbytes
    engine._check(lib.mcov_sam_decode_gpu(engine._ctx, ptr, n, int(chunk_bytes), C.byref(raw)))
    del keep
    return DeviceSoA(engine, raw, "sam")


def depth_sorted(engine, soa, wait=True):
    """Per-base depth of every contig from device-resident columns (fused sorted path)."""
    fn = lib.mcov_depth_sorted if wait else lib.mcov_depth_sorted_async
    r = soa.raw
    engine._check(fn(engine._ctx, soa.n_records, r.tid, r.pos, r.flag, r.mapq, r.cig_off, r.cig, _capi.MEM_DEVICE))


def stream_depth(engine, path, chunk_bytes=64 << 20, verify_crc=True):
    """Per-base depth of a coordinate-sorted BAM of any size: the file goes through the GPU decoder chunk by chunk into the
    streamed depth pass (``mcov_bam_gpu_stream_depth``); the engine's contig table must be the file's.  Returns the
    decoder's counters (records, chunks, bytes)."""
    info = _capi.BamGpuStreamInfo()
    engine._check(lib.mcov_bam_gpu_stream_depth(engine._ctx, str(path).encode(), int(chunk_bytes), 1 if verify_crc else 0,
                                                C.byref(info)))
    return {k: getattr(info, k) for k, _ in info._fields_}
