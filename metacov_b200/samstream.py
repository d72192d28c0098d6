"""SAM text from a stream (stdin, a pipe, a FIFO, a binary file object): the host side of reading an aligner's output as
it is written.

A stream is read once, front to back.  ``open_stream`` sniffs the format from its first bytes and reads the header (every
'@' line in front of the first record); ``ChunkReader`` then hands the records to a decoder in chunks of whole lines,
read by a thread into one of two host buffers while the caller decodes the other (csrc/sam_gpu.cu,
``mcov_sam_chunk_decode``).  Nothing here needs a GPU: the decoder is a callable.
"""
import io
import os
import queue
import stat
import sys
import threading

import numpy as np

GZIP_MAGIC = b"\x1f\x8b"


def is_stream(source):
    """True for what ``AlignmentFile`` reads as a stream: "-" (stdin), a binary file object, or a path that is not a
    regular file (a FIFO, /dev/fd/N of a pipe, a character device)."""
    if isinstance(source, str) and source == "-":
        return True
    if hasattr(source, "read"):
        return True
    try:
        return not stat.S_ISREG(os.stat(source).st_mode)
    except (OSError, TypeError, ValueError):
        return False


class _Source:
    """Reads of a binary handle into caller buffers.  Standard input and a path opened here are read through their file
    descriptor, without Python's buffering or its lock, so that a reader thread left blocked on a pipe never holds up
    the caller; a file object of the caller's is read through its own ``readinto``."""

    def __init__(self, handle, use_fd=False):
        self.handle = handle
        self._raw = None
        if use_fd:
            try:
                self._raw = io.FileIO(handle.fileno(), "rb", closefd=False)
            except (AttributeError, OSError, io.UnsupportedOperation, ValueError):
                self._raw = None

    def readinto(self, mv):
        if self._raw is not None:
            return self._raw.readinto(mv) or 0
        if hasattr(self.handle, "readinto"):
            return self.handle.readinto(mv) or 0
        b = self.handle.read(len(mv))
        mv[:len(b)] = b
        return len(b)

    def read(self, n):
        buf = bytearray(n)
        k = self.readinto(memoryview(buf))
        del buf[k:]
        return bytes(buf)


def open_stream(source):
    """(reader, header bytes, bytes read past the header, handle to close or None).  Raises OSError for input that is
    not SAM text: gzip data (BAM or BGZF-compressed SAM must be given as a file path) and anything else."""
    owned = None
    if isinstance(source, str) and source == "-":
        stdin = sys.stdin.buffer if hasattr(sys.stdin, "buffer") else sys.stdin
        src = _Source(stdin, use_fd=True)
    elif hasattr(source, "read"):
        src = _Source(source)
    else:
        owned = open(source, "rb", buffering=0)
        src = _Source(owned, use_fd=True)
    try:
        head, rest = read_header(src)
    except BaseException:
        if owned is not None:
            owned.close()
        raise
    return src, head, rest, owned


def sniff(first):
    """The format of a stream from its first bytes: "sam", "gzip" or None (empty or something else)."""
    if first[:2] == GZIP_MAGIC:
        return "gzip"
    line = first.split(b"\n", 1)[0]
    if len(line) >= 4 and line[:1] == b"@" and line[1:3].isalpha() and line[3:4] == b"\t":
        return "sam"
    if line.count(b"\t") >= 10:
        return "sam"
    return None


def read_header(src, piece=1 << 16):
    """Read the stream up to its first record line: (header bytes, the bytes read past them).  The format is sniffed from
    the first bytes of the same reads, which are kept."""
    data = bytearray()
    eof = False

    def more():
        nonlocal eof
        b = src.read(piece)
        if not b:
            eof = True
        data.extend(b)

    while not eof and len(data) < 2:
        more()
    if not data:
        raise OSError("empty input: no SAM header and no records")
    if bytes(data[:2]) == GZIP_MAGIC:
        raise OSError("gzip-compressed input on a stream: BAM (or BGZF-compressed SAM) must be given as a file path; "
                      "a stream is read as SAM text")
    # the first line decides (a long first record: read on to its tenth TAB)
    while not eof and b"\n" not in data and data.count(b"\t") < 10:
        more()
    if sniff(bytes(data[:data.find(b"\n") if b"\n" in data else len(data)])) != "sam":
        raise OSError("input stream is not SAM text (neither a header line nor a record of 11 TAB-separated fields "
                      "starts it)")
    # header: '@' lines in front of the first record
    p = 0
    while True:
        if p < len(data) and data[p:p + 1] != b"@":
            break
        nl = data.find(b"\n", p)
        if nl < 0:
            if eof:
                p = len(data)
                break
            more()
            continue
        p = nl + 1
        if p == len(data) and not eof:
            more()
        if p >= len(data) and eof:
            break
    return bytes(data[:p]), bytes(data[p:])


def header_refs(text):
    """[(name, length)] of the @SQ lines of a SAM header, in order (the decoder validates them)."""
    refs = []
    for line in text.splitlines():
        if line.startswith("@SQ\t"):
            tags = dict(t.split(":", 1) for t in line.split("\t")[1:] if ":" in t)
            if "SN" in tags and "LN" in tags:
                refs.append((tags["SN"], int(tags["LN"])))
    return refs


def _pageable(nbytes):
    return np.empty(nbytes, dtype=np.uint8)


def _pinned(nbytes):
    """Page-locked host memory (torch's pinned allocator) as a numpy array (whose base, the tensor, keeps it alive)."""
    import torch
    return torch.empty(nbytes, dtype=torch.uint8, pin_memory=True).numpy()


def _last_lf(a, n):
    """1 + the index of the last LF in a[:n], 0 if there is none (searched from the end, 64 KiB at a time)."""
    e = n
    while e > 0:
        b = max(0, e - (1 << 16))
        hit = np.flatnonzero(a[b:e] == 10)
        if len(hit):
            return b + int(hit[-1]) + 1
        e = b
    return 0


class ChunkReader:
    """The records of a stream in chunks of whole lines.  A reader thread fills one of two host buffers with
    ``readinto`` while the caller decodes the other; the bytes behind a buffer's last LF move to the front of the next
    buffer, and a buffer that holds no complete line doubles, so lines of any length pass.  ``run(decode)`` calls
    ``decode(memoryview, last)`` with each chunk (whole lines, the last chunk possibly without a final LF) until the stream
    ends or ``decode`` returns False.  ``pinned``: page-locked buffers instead of pageable ones."""

    def __init__(self, src, first=b"", chunk_bytes=64 << 20, pinned=False):
        self.src = src
        self.chunk = max(int(chunk_bytes), 1)
        self._first = first
        self._alloc = _pinned if pinned else _pageable
        self.bytes = 0                   # record bytes handed to the decoder
        self.chunks = 0
        self._stop = threading.Event()
        self._thread = None
        self._lock = threading.Lock()
        self._done = False
        self._at_exit = []

    def _wait(self, q):
        while True:
            try:
                return q.get(timeout=0.1)
            except queue.Empty:
                if self._stop.is_set():
                    return None

    def _grown(self, buf, need, keep):
        """A buffer of at least `need` bytes holding buf[:keep]."""
        if len(buf) >= need:
            return buf
        nb = self._alloc(need)
        nb[:keep] = buf[:keep]
        return nb

    def _fill(self, free, ready):
        try:
            carry = np.frombuffer(self._first, dtype=np.uint8)
            while not self._stop.is_set():
                buf = self._wait(free)
                if buf is None:
                    return
                buf = self._grown(buf, max(self.chunk, 2 * len(carry)), 0)
                buf[:len(carry)] = carry
                n, eof = len(carry), False
                while True:
                    mv = memoryview(buf)
                    while n < len(buf):
                        k = self.src.readinto(mv[n:])
                        if self._stop.is_set():
                            return
                        if k == 0:
                            eof = True
                            break
                        n += k
                    mv.release()
                    cut = n if eof else _last_lf(buf, n)
                    if cut or eof:
                        break
                    buf = self._grown(buf, 2 * len(buf), n)            # no complete line: the buffer doubles
                carry = buf[cut:n].copy()
                ready.put((buf, cut, eof))
                if eof:
                    return
        except BaseException as e:                                     # delivered to the caller
            ready.put(e)
        finally:
            with self._lock:
                self._done = True
                at_exit, self._at_exit = self._at_exit, []
            for fn in at_exit:
                fn()

    def run(self, decode):
        free, ready = queue.Queue(), queue.Queue()
        free.put(self._alloc(self.chunk))
        free.put(self._alloc(self.chunk))
        self._thread = threading.Thread(target=self._fill, args=(free, ready), name="sam-stream-reader", daemon=True)
        self._thread.start()
        eof = False
        try:
            while True:
                item = ready.get()
                if isinstance(item, BaseException):
                    raise item
                buf, cut, eof = item
                self.bytes += cut
                self.chunks += 1
                with memoryview(buf) as mv:
                    view = mv[:cut]
                    go = decode(view, eof)
                    view.release()
                if eof or go is False:
                    break
                free.put(buf)
        finally:
            self._stop.set()
        if eof:
            self._thread.join()

    def release(self, fn):
        """Run `fn` (closing the handle the reader reads) once the reader thread cannot read any more: now if it has
        ended, else when it does.  A thread left blocked on a pipe after an early stop then never reads through a
        descriptor that has been closed, and perhaps reused, under it."""
        self._stop.set()
        with self._lock:
            if not self._done and self._thread is not None:
                self._at_exit.append(fn)
                return
        fn()

    def info(self):
        return {"chunks": self.chunks, "bytes": self.bytes}
