"""Host-side driver of the CUDA coverage path (thin layer over the C-ABI).

One ``CoverageEngine`` = one ``mcov_ctx`` = one GPU.  It owns the per-base
depth of every contig of one BAM (the quantity reference metacov/pileup.py:
10-16 rebuilds per region) and answers region queries from it.
"""
import ctypes as C
import os
from collections import namedtuple

import numpy as np

from . import _capi
from ._capi import McovError, lib

ReadBatch = namedtuple("ReadBatch", "tid pos flag mapq cig_off cig")
ReadBatch.__doc__ = """SoA of mapped reads: the bam1_t fields the coverage path needs.

tid:int32[n] pos:int32[n] flag:uint16[n] mapq:uint8[n] cig_off:uint32[n+1]
cig:uint32[cig_off[n]] (BAM encoding len<<4|op).  numpy arrays (host) or torch
tensors (host or CUDA).  A batch of 2^32 or more ops carries 64-bit offsets
(numpy uint64/int64, torch int64) and takes the *_wide entry points."""

RUNS_DTYPE = np.dtype([("tid", "<i4"), ("start", "<i4"), ("end", "<i4"), ("depth", "<i4")])

_DT = dict(tid=np.int32, pos=np.int32, flag=np.uint16, mapq=np.uint8, cig_off=np.uint32, cig=np.uint32)


def _is_torch(a):
    return hasattr(a, "data_ptr") and hasattr(a, "is_cuda")


def _mem_kind(batch):
    kinds = set()
    for name, a in zip(ReadBatch._fields, batch):
        if _is_torch(a):
            kinds.add(_capi.MEM_DEVICE if a.is_cuda else _capi.MEM_HOST)
            if not a.is_contiguous():
                raise ValueError("ReadBatch.%s must be contiguous" % name)
        else:
            kinds.add(_capi.MEM_HOST)
    if len(kinds) != 1:
        raise ValueError("ReadBatch mixes host and device arrays")
    return kinds.pop()


def _is_wide(batch):
    """True when the batch carries 64-bit CIGAR offsets."""
    o = batch.cig_off
    if _is_torch(o):
        return o.element_size() == 8
    return np.asarray(o).dtype.itemsize == 8


def _canon(batch):
    """numpy members -> contiguous arrays of the ABI dtypes; torch members are
    checked, not converted."""
    out = []
    wide = _is_wide(batch)
    for name, a in zip(ReadBatch._fields, batch):
        if _is_torch(a):
            import torch
            want = {np.int32: torch.int32, np.uint16: (torch.uint16, torch.int16),
                    np.uint8: torch.uint8, np.uint32: (torch.uint32, torch.int32)}[_DT[name]]
            if name == "cig_off" and wide:
                want = (torch.int64, torch.uint64)
            want = want if isinstance(want, tuple) else (want,)
            if a.dtype not in want:
                raise TypeError("ReadBatch.%s: dtype %s, expected %s" % (name, a.dtype, want[0]))
            out.append(a)
        else:
            out.append(np.ascontiguousarray(a, dtype=np.uint64 if (name == "cig_off" and wide) else _DT[name]))
    return ReadBatch(*out)


class CoverageEngine:
    def __init__(self, lengths, device=0, stream=None, filt=None):
        self._ctx = C.c_void_p()
        rc = lib.mcov_create(C.byref(self._ctx), int(device), stream)
        if rc != 0:
            self._ctx = None
            raise McovError(rc, "mcov_create failed: no usable CUDA device %d (there is no CPU fallback)" % device)
        self.device = int(device)
        self.lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        self._check(lib.mcov_set_contigs(self._ctx, len(self.lengths), _capi.ptr(self.lengths)))
        self.n_slots = lib.mcov_n_slots(self._ctx)
        self.filter = _capi.Filter()
        lib.mcov_default_filter(C.byref(self.filter))
        if filt is not None:
            self.set_filter(**filt)
        self._keep = None
        self._pinned = None

    def set_contigs(self, lengths):
        """Replace the contig table (any depth computed so far is dropped)."""
        self.lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        self._check(lib.mcov_set_contigs(self._ctx, len(self.lengths), _capi.ptr(self.lengths)))
        self.n_slots = lib.mcov_n_slots(self._ctx)

    # -- plumbing ---------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise McovError(rc, lib.mcov_last_error(self._ctx).decode())

    def close(self):
        if getattr(self, "_ctx", None):
            lib.mcov_destroy(self._ctx)
            self._ctx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
        return False

    def set_filter(self, flag_filter=None, flag_require=None, min_mapq=None, ignore_orphans=None, max_depth=None,
                   count_del=None, reflen0_as_one=None):
        f = self.filter
        if flag_filter is not None:
            f.flag_filter = flag_filter
        if flag_require is not None:
            f.flag_require = flag_require
        if min_mapq is not None:
            f.min_mapq = min_mapq
        if ignore_orphans is not None:
            f.ignore_orphans = 1 if ignore_orphans else 0
        if max_depth is not None:
            f.max_depth = max_depth
        if count_del is not None:
            f.count_del = 1 if count_del else 0
        if reflen0_as_one is not None:
            f.reflen0_as_one = 1 if reflen0_as_one else 0
        self._check(lib.mcov_set_filter(self._ctx, C.byref(f)))

    def contig_offset(self, tid):
        return lib.mcov_contig_offset(self._ctx, int(tid))

    def bind_depth(self, tensor):
        """Use a caller-owned CUDA int32 tensor (>= n_slots elements) as the depth store."""
        self._keep = tensor
        self._check(lib.mcov_bind_depth(self._ctx, tensor.data_ptr(), tensor.numel()))

    # -- depth ------------------------------------------------------------
    def begin(self, exact_cap=False):
        """Start an any-order pass.  exact_cap: the pass reports the exact cap metric max depth[p-1]+starts[p]
        (mcov_begin_ex, MCOV_BEGIN_EXACT_CAP) instead of an upper bound of it."""
        if exact_cap:
            self._check(lib.mcov_begin_ex(self._ctx, _capi.MCOV_BEGIN_EXACT_CAP))
        else:
            self._check(lib.mcov_begin(self._ctx))

    def push(self, batch):
        b = _canon(batch)
        n = len(b.tid)
        fn = lib.mcov_push_reads_wide if _is_wide(b) else lib.mcov_push_reads
        self._check(fn(self._ctx, n, *[_capi.ptr(x) for x in b], _mem_kind(b)))

    def finalize(self):
        self._check(lib.mcov_finalize(self._ctx))

    def depth_sorted(self, batch, wait=True):
        """Fused path; raises McovError(MCOV_ERR_UNSORTED) on unsorted input.  With
        wait=False the call only enqueues the work and the verdict is raised by the next
        synchronising call (region_stats / copy_depth / pass_info)."""
        b = _canon(batch)
        n = len(b.tid)
        if _is_wide(b):
            self._check(lib.mcov_depth_sorted_wide(self._ctx, n, *[_capi.ptr(x) for x in b], _mem_kind(b), 1 if wait else 0))
            return
        fn = lib.mcov_depth_sorted if wait else lib.mcov_depth_sorted_async
        self._check(fn(self._ctx, n, *[_capi.ptr(x) for x in b], _mem_kind(b)))

    # -- streaming: successive batches of a coordinate-sorted file -------------
    def stream_begin(self):
        """Start a streamed pass (mcov_stream_begin)."""
        self._check(lib.mcov_stream_begin(self._ctx))

    def stream_push(self, batch, n_carry=0, last=False):
        """Add the next batch (file order) of a streamed pass; the batch begins with ``n_carry`` reads
        re-sent from earlier batches (see mcov_stream_push).  Returns the resend point (tid, pos): the
        next batch must begin with every earlier read that starts at or after it or reaches past it."""
        b = _canon(batch)
        if _is_wide(b):
            raise ValueError("stream_push takes 32-bit CIGAR offsets (a batch is far below 2^32 ops)")
        rt, rp = C.c_int32(-1), C.c_int32(0)
        self._check(lib.mcov_stream_push(self._ctx, len(b.tid), int(n_carry), *[_capi.ptr(x) for x in b], _mem_kind(b),
                                         1 if last else 0, C.byref(rt), C.byref(rp)))
        return rt.value, rp.value

    def stream_resend_point(self, last_tid, last_pos):
        rt, rp = C.c_int32(-1), C.c_int32(0)
        self._check(lib.mcov_stream_resend_point(self._ctx, int(last_tid), int(last_pos), C.byref(rt), C.byref(rp)))
        return rt.value, rp.value

    def depth_sorted_block(self, block, wait=True):
        """Fused path from a transport block (``pack_block`` / the streaming reader): one host-to-device copy."""
        buf, nbytes = block
        self._check(lib.mcov_depth_sorted_block(self._ctx, _capi.ptr(buf), int(nbytes), 1 if wait else 0))

    def block_unpack(self, block):
        """The SoA columns a transport block widens into on the device, copied back (``mcov_block_unpack``):
        dict with tid, pos, flag, mapq, cig_off (n + 1), cig."""
        import struct
        buf, nbytes = block
        raw = buf.numpy() if _is_torch(buf) else np.asarray(buf)
        n, _n_carry, n_cigar = struct.unpack_from("<qqq", raw[:32].tobytes(), 8)
        out = {"tid": np.empty(n, np.int32), "pos": np.empty(n, np.int32), "flag": np.empty(n, np.uint16),
               "mapq": np.empty(n, np.uint8), "cig_off": np.empty(n + 1, np.uint32), "cig": np.empty(n_cigar, np.uint32)}
        self._check(lib.mcov_block_unpack(self._ctx, _capi.ptr(buf), int(nbytes), *[_capi.ptr(out[k]) for k in
                                                                                  ("tid", "pos", "flag", "mapq", "cig_off", "cig")]))
        return out

    def stream_push_block(self, block, last=False):
        """One batch of a streamed pass as a transport block; returns the resend point like ``stream_push``."""
        buf, nbytes = block
        rt, rp = C.c_int32(-1), C.c_int32(0)
        self._check(lib.mcov_stream_push_block(self._ctx, buf if isinstance(buf, int) else _capi.ptr(buf), int(nbytes),
                                               1 if last else 0, C.byref(rt), C.byref(rp)))
        return rt.value, rp.value

    def depth_sorted_packed(self, packed, wait=True):
        """Fused path from the compact host transport (see ``pack_batch``)."""
        self._check(lib.mcov_depth_sorted_packed(
            self._ctx, packed["n"], _capi.ptr(packed["contig_read_start"]), _capi.ptr(packed["pos"]),
            _capi.ptr(packed["flag"]), _capi.ptr(packed["mapq"]) if packed.get("mapq") is not None else None,
            _capi.ptr(packed["n_cigar"]), _capi.ptr(packed["cig"]), packed["n_cig_total"], 1 if wait else 0))

    def depth_sorted_delta(self, packed, wait=True):
        """Fused path from the delta host transport (see ``pack_batch_delta``)."""
        n_exc = len(packed["exc_index"]) if not _is_torch(packed["exc_index"]) else packed["exc_index"].numel()
        self._check(lib.mcov_depth_sorted_delta(
            self._ctx, packed["n"], _capi.ptr(packed["contig_read_start"]), _capi.ptr(packed["dpos"]), n_exc,
            _capi.ptr(packed["exc_index"]) if n_exc else None, _capi.ptr(packed["exc_delta"]) if n_exc else None,
            _capi.ptr(packed["flag"]), _capi.ptr(packed["mapq"]) if packed.get("mapq") is not None else None,
            _capi.ptr(packed["n_cigar"]), _capi.ptr(packed["cig"]), packed["n_cig_total"], 1 if wait else 0))

    def compute_depth(self, batch):
        """Per-base depth of all contigs from one batch: the fused sorted path,
        or clear + expand + scan when the reads are not coordinate-sorted (or
        carry more long-span reads than the fused path buckets).  Both run on
        the GPU."""
        try:
            self.depth_sorted(batch)
            return "fused"
        except McovError as e:
            if e.code not in (_capi.MCOV_ERR_UNSORTED, _capi.MCOV_ERR_RANGE):
                raise
        self.begin()
        self.push(batch)
        self.finalize()
        return "push"

    def pass_info(self):
        info = _capi.PassInfo()
        self._check(lib.mcov_pass_info_get(self._ctx, C.byref(info)))
        return {k: getattr(info, k) for k, _ in _capi.PassInfo._fields_ if k != "reserved"}

    def copy_depth(self, tid, start=0, end=None):
        end = int(self.lengths[tid]) if end is None else int(end)
        out = np.empty(max(end - int(start), 0), dtype=np.int32)
        self._check(lib.mcov_copy_depth(self._ctx, int(tid), int(start), end, _capi.ptr(out)))
        return out

    def depth_ptr(self):
        return lib.mcov_depth_ptr(self._ctx)

    def sync(self):
        """Wait for everything enqueued on the engine's stream."""
        self._check(lib.mcov_sync(self._ctx))

    # -- A / C / G / T counts -------------------------------------------------
    def base_counts(self, quality_threshold=15, mode=_capi.MCOV_BC_ALL, path=None, chunk_bytes=0):
        """A / C / G / T counts at every position of every contig (``mcov_base_counts``): of the file last decoded on this
        engine (``bamgpu.decode`` / ``decode_sam``), or of the BAM at ``path`` through the streamed decoder.  ``mode``:
        MCOV_BC_ALL or MCOV_BC_NOFILTER.  The depth is left as it was."""
        p = os.fsencode(path) if path is not None else None
        self._check(lib.mcov_base_counts(self._ctx, p, int(chunk_bytes), int(quality_threshold), int(mode)))

    def copy_base_counts(self, tid, start=0, end=None):
        """uint32 [4, end - start]: the A, C, G and T counts of [start, end) of contig ``tid`` (``base_counts`` first)."""
        end = int(self.lengths[tid]) if end is None else int(end)
        out = np.empty((4, max(end - int(start), 0)), dtype=np.uint32)
        self._check(lib.mcov_copy_base_counts(self._ctx, int(tid), int(start), end, _capi.ptr(out)))
        return out

    # -- alleles (from the counts of base_counts) ---------------------------------------------------------------------
    def set_reference(self, tid, seq):
        """The reference of contig ``tid`` (str or bytes, exactly the contig's length) for ``use_reference=True``."""
        b = seq.encode("ascii") if isinstance(seq, str) else bytes(seq)
        self._check(lib.mcov_set_reference(self._ctx, int(tid), b, len(b)))

    @staticmethod
    def _allele_params(min_coverage, min_freq, min_count, use_reference):
        p = _capi.AlleleParams()
        for name, v, lo in (("min_coverage", min_coverage, 1), ("min_count", min_count, 1)):
            if int(v) != v or not lo <= int(v) < 2 ** 32:
                raise ValueError("%s must be an integer >= %d, got %r" % (name, lo, v))
        if not 0.0 <= float(min_freq) <= 1.0:
            raise ValueError("min_freq must be in [0, 1], got %r" % (min_freq,))
        p.min_coverage, p.min_count, p.min_freq = int(min_coverage), int(min_count), float(min_freq)
        p.use_reference = 1 if use_reference else 0
        return p

    @staticmethod
    def _region_columns(tid, start, end):
        """(tid, start, end) as contiguous int32 arrays of one length g, and g; else ValueError."""
        tid = np.ascontiguousarray(tid, dtype=np.int32)
        start = np.ascontiguousarray(start, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        if not (len(start) == len(end) == len(tid)):
            raise ValueError("tid/start/end lengths differ")
        return tid, start, end, len(tid)

    def allele_stats(self, tid, start, end, min_coverage=5, min_freq=0.05, min_count=2, use_reference=False):
        """Allele statistics of g regions (``mcov_allele_stats_run``) -> structured array ``_capi.ALLELE_STATS_DTYPE``
        (length, covered, depth_sum, pi_sum, snv, ref_covered, sub, popsub).  Needs ``base_counts`` first, and with
        ``use_reference`` a ``set_reference`` of every contig."""
        tid, start, end, g = self._region_columns(tid, start, end)
        p = self._allele_params(min_coverage, min_freq, min_count, use_reference)
        out = np.zeros(g, dtype=_capi.ALLELE_STATS_DTYPE)
        self._check(lib.mcov_allele_stats_run(self._ctx, g, _capi.ptr(tid), _capi.ptr(start), _capi.ptr(end), C.byref(p),
                                              _capi.ptr(out)))
        return out

    def allele_sites(self, min_coverage=5, min_freq=0.05, min_count=2, use_reference=False):
        """Every site (a covered position of kind SNV, SUB or POPSUB) in (tid, pos) order -> structured array
        ``_capi.ALLELE_SITE_DTYPE`` (tid pos A C G T ref consensus kind)."""
        p = self._allele_params(min_coverage, min_freq, min_count, use_reference)
        n = C.c_int64(0)
        self._check(lib.mcov_allele_sites(self._ctx, C.byref(p), C.byref(n)))
        out = np.zeros(n.value, dtype=_capi.ALLELE_SITE_DTYPE)
        self._check(lib.mcov_allele_sites_read(self._ctx, 0, n.value, _capi.ptr(out)))
        return out

    # -- comparisons (signatures of base_counts, then pairs of signatures) --------------------------------------------
    def allele_signature(self, min_coverage=5, min_freq=0.05, min_count=2):
        """The signature of every slot (``mcov_allele_signature``) -> CUDA ``torch.uint8`` tensor of ``n_slots``: 0x80
        covered, bits 4-5 the consensus, bits 0-3 the present mask, 0 where not covered.  Needs ``base_counts`` first."""
        import torch
        p = self._allele_params(min_coverage, min_freq, min_count, False)
        dev = torch.device("cuda", self.device)
        out = torch.empty(int(self.n_slots), dtype=torch.uint8, device=dev)
        torch.cuda.current_stream(dev).synchronize()         # (the tensor's memory may still be read by earlier work)
        self._check(lib.mcov_allele_signature(self._ctx, C.byref(p), _capi.ptr(out)))
        return out

    def _compare_args(self, signatures, pairs):
        """(ctypes pointer table, pairs as int32 [n, 2]) after checking every tensor and pair, else ValueError."""
        import torch
        sigs = list(signatures)
        if len(sigs) < 2:
            raise ValueError("a comparison needs at least two signatures, got %d" % len(sigs))
        for i, s in enumerate(sigs):
            if not isinstance(s, torch.Tensor) or s.device.type != "cuda" or s.device.index != self.device:
                raise ValueError("signature %d must be a CUDA tensor on device %d" % (i, self.device))
            if s.dtype != torch.uint8 or s.dim() != 1 or not s.is_contiguous() or s.numel() != int(self.n_slots):
                raise ValueError("signature %d must be a contiguous torch.uint8 vector of n_slots = %d, got %s %s"
                                 % (i, int(self.n_slots), s.dtype, tuple(s.shape)))
        pairs = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
        if len(pairs) == 0:
            raise ValueError("pairs must hold at least one pair of signatures")
        if pairs.min() < 0 or pairs.max() >= len(sigs) or (pairs[:, 0] == pairs[:, 1]).any():
            raise ValueError("pairs must index two different signatures of 0 .. %d" % (len(sigs) - 1))
        tab = (C.c_void_p * len(sigs))(*[s.data_ptr() for s in sigs])
        torch.cuda.current_stream(torch.device("cuda", self.device)).synchronize()   # (the signatures are written)
        return tab, np.ascontiguousarray(pairs, dtype=np.int32), sigs

    def compare_stats(self, signatures, pairs, tid, start, end):
        """Every pair's records over g regions (``mcov_compare_run``) -> structured array
        ``_capi.COMPARE_STATS_DTYPE`` of shape [n_pairs, g] (length, covered_a, covered_b, compared, con_snp,
        pop_snp).  ``signatures``: tensors of ``allele_signature`` made under this contig table; ``pairs``: [n, 2]
        indices into them."""
        tab, pairs, _keep = self._compare_args(signatures, pairs)
        tid, start, end, g = self._region_columns(tid, start, end)
        out = np.zeros((len(pairs), g), dtype=_capi.COMPARE_STATS_DTYPE)
        self._check(lib.mcov_compare_run(self._ctx, len(tab), tab, len(pairs), _capi.ptr(pairs), g, _capi.ptr(tid),
                                         _capi.ptr(start), _capi.ptr(end), _capi.ptr(out)))
        return out

    def compare_sites(self, signatures, pairs):
        """Every con_snp position of every pair in (pair, tid, pos) order (``mcov_compare_sites``) -> structured array
        ``_capi.COMPARE_SITE_DTYPE`` (pair tid pos sig_a sig_b kind; kind 1 con_snp, 2 pop_snp)."""
        tab, pairs, _keep = self._compare_args(signatures, pairs)
        n = C.c_int64(0)
        self._check(lib.mcov_compare_sites(self._ctx, len(tab), tab, len(pairs), _capi.ptr(pairs), C.byref(n)))
        out = np.zeros(n.value, dtype=_capi.COMPARE_SITE_DTYPE)
        self._check(lib.mcov_compare_sites_read(self._ctx, 0, n.value, _capi.ptr(out)))
        return out

    # -- accounting ---------------------------------------------------------
    def launch_count(self):
        return lib.mcov_launch_count(self._ctx)

    def profile(self, on=True):
        self._check(lib.mcov_profile_enable(self._ctx, 1 if on else 0))

    def profile_read(self):
        """{kernel name: (launches, total_ms)} of the CUDA-event timing since profile(True)."""
        arr = (_capi.KernelTime * 48)()
        n = lib.mcov_profile_read(self._ctx, arr, 48)
        if n < 0:
            self._check(n)
        return {arr[i].name.decode(): (arr[i].launches, arr[i].total_ms) for i in range(n)}

    # -- statistics -------------------------------------------------------
    def region_stats(self, tid, start, end, breadth_n=1):
        """Exact integer statistics of g regions -> structured array
        (``_capi.REGION_STATS_DTYPE``)."""
        tid = np.ascontiguousarray(tid, dtype=np.int32)
        start = np.ascontiguousarray(start, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        g = len(tid)
        if not (len(start) == len(end) == g):
            raise ValueError("tid/start/end lengths differ")
        out = self._stats_buffer(g)
        self._check(lib.mcov_region_stats_run(self._ctx, g, _capi.ptr(tid), _capi.ptr(start), _capi.ptr(end),
                                              int(breadth_n), _capi.ptr(out)))
        return out

    def _stats_buffer(self, g):
        """Result records land in a pinned host buffer owned by the engine and reused between calls
        (the returned array is a view: copy it to keep it across the next region_stats call)."""
        if g <= 1024:
            return np.zeros(g, dtype=_capi.REGION_STATS_DTYPE)
        if self._pinned is None or self._pinned.numel() < g * 64:
            import torch
            self._pinned = torch.empty(g * 64 + 64, dtype=torch.uint8).pin_memory()
        return self._pinned.numpy()[:g * 64].view(_capi.REGION_STATS_DTYPE)

    def region_stats_submit(self, tid, start, end, breadth_n=1, slot=0):
        """Pipelined statistics: enqueue the kernels and the copy-back into staging slot 0/1 and
        return at once, so that the next depth pass can be enqueued before these results are
        waited for.  ``region_stats_collect(ticket)`` returns the records."""
        tid = np.ascontiguousarray(tid, dtype=np.int32)
        start = np.ascontiguousarray(start, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        self._check(lib.mcov_region_stats_submit(self._ctx, len(tid), _capi.ptr(tid), _capi.ptr(start), _capi.ptr(end),
                                                 int(breadth_n), int(slot)))
        return (int(slot), len(tid))

    def region_stats_collect(self, ticket, copy=True):
        """Records of a submitted slot.  copy=False returns a zero-copy view of the engine's pinned
        staging slot (valid until the next submit on that slot): what a pipeline with hundreds of
        thousands of regions wants."""
        slot, g = ticket
        if copy:
            out = np.zeros(g, dtype=_capi.REGION_STATS_DTYPE)
            self._check(lib.mcov_region_stats_collect(self._ctx, slot, _capi.ptr(out)))
            return out
        view, n = C.c_void_p(), C.c_int64()
        self._check(lib.mcov_region_stats_collect_view(self._ctx, slot, C.byref(view), C.byref(n)))
        if n.value == 0:
            return np.zeros(0, dtype=_capi.REGION_STATS_DTYPE)
        raw = (C.c_uint8 * (n.value * 64)).from_address(view.value)
        return np.frombuffer(raw, dtype=_capi.REGION_STATS_DTYPE)

    def region_stats_enqueue(self, tid, start, end, out, breadth_n=1):
        """Asynchronous: write len(tid) records into the CUDA uint8 tensor ``out`` (>= 64 bytes per
        region) on the engine's stream; no synchronisation (see mcov_region_stats_enqueue)."""
        tid = np.ascontiguousarray(tid, dtype=np.int32)
        start = np.ascontiguousarray(start, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        if out.numel() * out.element_size() < 64 * len(tid):
            raise ValueError("output tensor too small")
        self._check(lib.mcov_region_stats_enqueue(self._ctx, len(tid), _capi.ptr(tid), _capi.ptr(start),
                                                  _capi.ptr(end), int(breadth_n), out.data_ptr()))

    def region_hist_enqueue(self, tid, start, end, hist):
        """Regions cut across devices: ADD the exact counting histogram of this engine's part of each
        region to ``hist`` (CUDA int32/uint32 tensor [g, 8192], zeroed by the caller); see
        mcov_region_hist_enqueue and sharding.ShardedCoverage."""
        tid = np.ascontiguousarray(tid, dtype=np.int32)
        start = np.ascontiguousarray(start, dtype=np.int32)
        end = np.ascontiguousarray(end, dtype=np.int32)
        if hist.numel() < _capi.HIST_BINS * len(tid) or hist.element_size() != 4 or not hist.is_contiguous():
            raise ValueError("hist must be a contiguous 4-byte tensor of g x %d bins" % _capi.HIST_BINS)
        self._check(lib.mcov_region_hist_enqueue(self._ctx, len(tid), _capi.ptr(tid), _capi.ptr(start), _capi.ptr(end),
                                                 hist.data_ptr()))

    def hist_stats_enqueue(self, hist, g, out, breadth_n=1):
        """Statistics records of g regions from complete (merged) counting histograms -> CUDA uint8
        tensor ``out`` (>= 64 bytes per region); no synchronisation."""
        if out.numel() * out.element_size() < 64 * g:
            raise ValueError("output tensor too small")
        self._check(lib.mcov_hist_stats_enqueue(self._ctx, int(g), hist.data_ptr(), int(breadth_n), out.data_ptr()))

    def experimental_stats(self, soa, name_hash, kmer_code, k_len, kc_val, kc_has, r_start, r_end, r_lb, r_ub):
        """One ``mcov_experimental_run`` call -> EXP_STATS_DTYPE records."""
        n = len(soa["pos"])
        g = len(r_start)
        out = np.zeros(g, dtype=_capi.EXP_STATS_DTYPE)
        r_start = np.ascontiguousarray(r_start, dtype=np.int32)
        r_end = np.ascontiguousarray(r_end, dtype=np.int32)
        r_lb = np.ascontiguousarray(r_lb, dtype=np.int64)
        r_ub = np.ascontiguousarray(r_ub, dtype=np.int64)
        name_hash = np.ascontiguousarray(name_hash, dtype=np.uint64)
        kmer_code = np.ascontiguousarray(kmer_code, dtype=np.int32)
        if kc_val is not None:
            kc_val = np.ascontiguousarray(kc_val, dtype=np.float64)
            kc_has = np.ascontiguousarray(kc_has, dtype=np.uint8)
        self._check(lib.mcov_experimental_run(
            self._ctx, n, _capi.ptr(soa["pos"]), _capi.ptr(soa["flag"]), _capi.ptr(soa["cig_off"]), _capi.ptr(soa["cig"]),
            _capi.ptr(name_hash), _capi.ptr(kmer_code), int(k_len) if kc_val is not None else 0,
            _capi.ptr(kc_val), _capi.ptr(kc_has), g, _capi.ptr(r_start), _capi.ptr(r_end), _capi.ptr(r_lb), _capi.ptr(r_ub),
            _capi.ptr(out)))
        return out

    def exp_revsum(self, cor_rev, w):
        """cor_revsum of reference pileup.py:78-83 (mcov_exp_revsum)."""
        cor_rev = np.ascontiguousarray(cor_rev, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        out = np.zeros(len(cor_rev), dtype=np.float64)
        self._check(lib.mcov_exp_revsum(self._ctx, len(cor_rev), _capi.ptr(cor_rev), len(w), _capi.ptr(w), _capi.ptr(out)))
        return out

    def kmer_hist(self, flag, l_seq, seq_win, win_bases, K, NK, STEP, OFFSET, group_flags=()):
        """ByFlag-grouped k-mer histogram -> uint32[groups, 4**K + 1, NK] (see mcov_kmer_hist)."""
        gf = np.ascontiguousarray(group_flags, dtype=np.uint16)
        dev = _is_torch(flag) and flag.is_cuda               # device-resident columns (a GPU-decoded file): no copies
        if not dev:
            flag = np.ascontiguousarray(flag, dtype=np.uint16)
            l_seq = np.ascontiguousarray(l_seq, dtype=np.int32)
            seq_win = np.ascontiguousarray(seq_win, dtype=np.uint8)
        n = len(flag)
        win_bytes = seq_win.shape[1] if len(seq_win.shape) == 2 else (win_bases + 1) // 2
        hist = np.zeros((1 << len(gf), 4 ** K + 1, NK), dtype=np.uint32)
        self._check(lib.mcov_kmer_hist_mem(self._ctx, n, _capi.ptr(flag), _capi.ptr(l_seq), _capi.ptr(seq_win),
                                           _capi.MEM_DEVICE if dev else _capi.MEM_HOST, win_bytes,
                                           win_bases, K, NK, STEP, OFFSET, len(gf), _capi.ptr(gf) if len(gf) else None,
                                           _capi.ptr(hist)))
        return hist

    def depth_runs(self, tid0=0, tid1=None, skip_zero=False):
        """Run-length form of the per-base depth of contigs [tid0, tid1): structured array
        (tid, start, end, depth), one record per maximal run of equal depth -- the rows of a
        bedGraph file (mcov_depth_runs)."""
        tid1 = len(self.lengths) if tid1 is None else int(tid1)
        n = C.c_int64()
        self._check(lib.mcov_depth_runs(self._ctx, int(tid0), tid1, C.byref(n)))
        n = n.value
        cols = [np.empty(n, dtype=np.int32) for _ in range(4)]
        self._check(lib.mcov_depth_runs_read(self._ctx, 0, n, *[_capi.ptr(c) for c in cols]))
        out = np.empty(n, dtype=RUNS_DTYPE)
        for name, c in zip(RUNS_DTYPE.names, cols):
            out[name] = c
        return out[out["depth"] != 0] if skip_zero else out

    def window_means(self, window):
        n_out = int(sum((int(l) + window - 1) // window for l in self.lengths))
        out = np.empty(n_out, dtype=np.float64)
        self._check(lib.mcov_window_means(self._ctx, int(window), _capi.ptr(out), n_out))
        return out

    # -- read-statistics scan --------------------------------------------
    def isize_hist(self, flag, isize, group_flags=(), n_bins=1024):
        """ByFlag-grouped |isize| histogram.  Returns (hist[groups, bins], group_counts, max_isize);
        the table is regrown until it covers max_isize (reference IsizeHist doubles its array,
        scan.pyx:603-608)."""
        gf = np.ascontiguousarray(group_flags, dtype=np.uint16)
        groups = 1 << len(gf)
        kind = _capi.MEM_DEVICE if (_is_torch(flag) and flag.is_cuda) else _capi.MEM_HOST
        if not _is_torch(flag):
            flag = np.ascontiguousarray(flag, dtype=np.uint16)
            isize = np.ascontiguousarray(isize, dtype=np.int32)
        n = len(flag)
        while True:
            hist = np.zeros((groups, n_bins), dtype=np.uint32)
            cnt = np.zeros(groups, dtype=np.uint64)
            mx = C.c_int32(0)
            self._check(lib.mcov_isize_hist(self._ctx, n, _capi.ptr(flag), _capi.ptr(isize), kind, len(gf),
                                            _capi.ptr(gf) if len(gf) else None, n_bins, _capi.ptr(hist),
                                            _capi.ptr(cnt), C.addressof(mx)))
            if mx.value < n_bins:
                return hist, cnt, mx.value
            while n_bins <= mx.value:
                n_bins *= 2


def _offsets_u32(cig_off, who):
    """cig_off as uint32 -- refusing, instead of truncating, 64-bit offsets that do not fit (a batch of 2^32 or more
    ops travels through the *_wide entry points as plain columns)."""
    a = cig_off.cpu().numpy() if _is_torch(cig_off) else np.asarray(cig_off)
    a = np.ascontiguousarray(a)
    if a.dtype.itemsize == 4:
        return a.view(np.uint32)
    if len(a) and (int(a.max()) > 0xFFFFFFFF or int(a.min()) < 0):
        raise ValueError("%s: the batch holds 2^32 or more CIGAR ops (64-bit offsets): it does not qualify for the narrow "
                         "transports; use depth_sorted / push with the wide offsets" % who)
    return a.astype(np.uint32)


def pack_batch(batch, n_contigs, with_mapq=False, pinned=False):
    """Compact host transport of a coordinate-sorted ``ReadBatch`` (numpy or CPU torch members):
    per-contig read prefix instead of ``tid``, u16 op counts instead of u32 offsets, ``mapq`` only
    on request.  Raises ValueError if the batch is not grouped by contig.  With ``pinned`` the
    arrays are torch pinned tensors (true asynchronous H2D)."""
    def as_np(a, dt):
        if _is_torch(a):
            a = a.cpu().numpy()
        return np.ascontiguousarray(a).view(dt) if np.dtype(a.dtype).itemsize == np.dtype(dt).itemsize else np.ascontiguousarray(a, dtype=dt)
    tid = as_np(batch.tid, np.int32)
    n = len(tid)
    placed = tid[(tid >= 0) & (tid < n_contigs)]
    if len(placed) and (np.any(np.diff(placed) < 0) or np.any(tid[:len(placed)] != placed)):
        raise ValueError("pack_batch: reads are not grouped by contig (unplaced reads must come last)")
    crs = np.zeros(n_contigs + 1, dtype=np.int64)
    np.cumsum(np.bincount(placed, minlength=n_contigs), out=crs[1:])
    off = _offsets_u32(batch.cig_off, "pack_batch").astype(np.int64)
    ncig = np.diff(off)
    if len(ncig) and ncig.max() > 65535:
        raise ValueError("pack_batch: a CIGAR has more than 65535 ops")
    out = {"n": n, "contig_read_start": crs, "pos": as_np(batch.pos, np.int32), "flag": as_np(batch.flag, np.uint16),
           "mapq": as_np(batch.mapq, np.uint8) if with_mapq else None, "n_cigar": ncig.astype(np.uint16),
           "cig": as_np(batch.cig, np.uint32), "n_cig_total": int(off[-1]) if len(off) else 0}
    if pinned:
        import torch
        for k in ("contig_read_start", "pos", "flag", "mapq", "n_cigar", "cig"):
            if out[k] is not None:
                t = torch.from_numpy(out[k].view({8: np.int64, 4: np.int32, 2: np.int16, 1: np.uint8}[out[k].dtype.itemsize]))
                out[k] = t.pin_memory()
    return out


def pack_batch_delta(batch, n_contigs, with_mapq=False, pinned=False):
    """Delta transport of a coordinate-sorted ``ReadBatch`` (see mcov_depth_sorted_delta): u16 position
    differences inside each contig (+ exceptions), u8 op counts, u16 ops.  Raises ValueError when the batch
    does not qualify (a CIGAR of more than 255 ops, an op longer than 4095, reads not grouped by contig);
    ``pack_batch`` is the fallback."""
    base = pack_batch(batch, n_contigs, with_mapq=with_mapq, pinned=False)
    n = base["n"]
    ncig, cig, pos, crs = base["n_cigar"], base["cig"], base["pos"], base["contig_read_start"]
    if len(ncig) and int(ncig.max()) > 255:
        raise ValueError("pack_batch_delta: a CIGAR has more than 255 ops")
    if len(cig) and int(cig.max()) > 0xFFFF:
        raise ValueError("pack_batch_delta: an op is longer than 4095")
    d = np.empty(n, dtype=np.int64)
    if n:
        d[0] = pos[0]
        np.subtract(pos[1:], pos[:-1], out=d[1:], dtype=np.int64)
        firsts = np.unique(np.concatenate((crs[:-1], crs[-1:])))        # first read of every contig and of the unplaced tail
        firsts = firsts[firsts < n]
        d[firsts] = pos[firsts]
    exc = np.nonzero((d < 0) | (d > 0xFFFF))[0]
    dpos = d.astype(np.uint16)
    dpos[exc] = 0
    out = {"n": n, "contig_read_start": crs, "dpos": dpos, "exc_index": exc.astype(np.uint32), "exc_delta": d[exc].astype(np.int32),
           "flag": base["flag"], "mapq": base["mapq"], "n_cigar": ncig.astype(np.uint8), "cig": cig.astype(np.uint16),
           "n_cig_total": base["n_cig_total"]}
    if pinned:
        import torch
        for k in ("contig_read_start", "dpos", "exc_index", "exc_delta", "flag", "mapq", "n_cigar", "cig"):
            if out[k] is not None:
                t = torch.from_numpy(out[k].view({8: np.int64, 4: np.int32, 2: np.int16, 1: np.uint8}[out[k].dtype.itemsize]))
                out[k] = t.pin_memory()
    return out


def pack_block(batch, n_contigs, with_mapq=False, n_carry=0, pinned=False, threads=0):
    """Transport block of a coordinate-sorted ``ReadBatch`` (numpy or CPU torch members) -- the format the native
    decoder hands to the GPU (mcov_pack_block: u8 position differences + exceptions, flag dictionary, CIGAR
    dictionary + explicit ops; ONE buffer, one host-to-device copy).  Returns (buffer, n_bytes); the buffer is a
    pinned torch uint8 tensor with ``pinned`` else a numpy array.  Raises ValueError when the batch does not qualify
    (a CIGAR of more than 127 ops, reads not grouped by contig): ``pack_batch`` / the plain columns are the fallback."""
    def as_np(a, dt):
        if _is_torch(a):
            a = a.cpu().numpy()
        a = np.ascontiguousarray(a)
        return a.view(dt) if a.dtype.itemsize == np.dtype(dt).itemsize else a.astype(dt)
    tid, pos = as_np(batch.tid, np.int32), as_np(batch.pos, np.int32)
    flag, mapq = as_np(batch.flag, np.uint16), as_np(batch.mapq, np.uint8)
    off, cig = _offsets_u32(batch.cig_off, "pack_block"), as_np(batch.cig, np.uint32)
    n = len(tid)
    cap = lib.mcov_block_bound(n, int(off[-1]) if n else 0, int(n_contigs))
    if pinned:
        import torch
        buf = torch.empty(cap + 16, dtype=torch.uint8).pin_memory()
    else:
        buf = np.empty(cap + 16, dtype=np.uint8)
    nb = C.c_int64(0)
    rc = lib.mcov_pack_block(n, int(n_carry), _capi.ptr(tid), _capi.ptr(pos), _capi.ptr(flag), _capi.ptr(mapq) if with_mapq else None,
                             _capi.ptr(off), _capi.ptr(cig), int(n_contigs), _capi.ptr(buf), cap, C.byref(nb), int(threads))
    if rc != 0:
        raise ValueError("pack_block: the batch does not qualify for the transport block (status %d)" % rc)
    return buf, nb.value


def packed_bytes(packed):
    tot = 0
    for k in ("contig_read_start", "pos", "dpos", "exc_index", "exc_delta", "flag", "mapq", "n_cigar", "cig"):
        a = packed.get(k)
        if a is not None:
            tot += a.numel() * a.element_size() if _is_torch(a) else a.nbytes
    return int(tot)
