"""SAM text read from a stream (a pipe, stdin, a binary file object): AlignmentFile's piped path against the same SAM read
as a regular file and against the C oracle; the exact max_depth verdict of the any-order pass (mcov_begin_ex) against the
fused path's; scan_reads and the CLI on a stream.  The host logic of the stream reader (sniffing, header split, tail
carry, buffer growth) is checked without a device."""
import io
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from helpers import load_json, load_soa
from oracle import bamio, cport
import samio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pipe_from(data, seed=0, max_piece=1 << 20):
    """A pipe fed with `data` by a writer thread in random pieces of 1 B .. max_piece; returns the read end as a binary
    file object."""
    r, w = os.pipe()
    rng = np.random.default_rng(seed)

    def writer():
        try:
            p = 0
            while p < len(data):
                k = int(min(len(data) - p, rng.integers(1, max_piece + 1) if rng.random() < 0.7 else rng.integers(1, 64)))
                os.write(w, data[p:p + k])
                p += k
        except OSError:
            pass
        finally:
            os.close(w)

    threading.Thread(target=writer, daemon=True).start()
    return os.fdopen(r, "rb", buffering=0)


# ---- host logic (no device) --------------------------------------------------------------------------------------------

def _header(n_sq=2):
    return ("@HD\tVN:1.6\tSO:unsorted\n" + "".join("@SQ\tSN:c%d\tLN:%d\n" % (i, 1000 + i) for i in range(n_sq))).encode()


def _lines(n, rng, long_every=0):
    out = []
    for i in range(n):
        ln = int(rng.integers(0, 40)) if not (long_every and i % long_every == 0) else 5000
        out.append(("r%d\t0\tc0\t%d\t60\t10M\t*\t0\t0\t%s\t*\tXA:Z:%s\n" % (i, i + 1, "A" * 10, "x" * ln)).encode())
    return b"".join(out)


def test_sniff_and_header_split():
    from metacov_b200 import samstream
    head, body = _header(3), _lines(5, np.random.default_rng(1))
    src = samstream._Source(io.BytesIO(head + body))
    h, rest = samstream.read_header(src, piece=7)
    assert h == head and rest + src.read(1 << 20) == body
    assert samstream.header_refs(h.decode()) == [("c0", 1000), ("c1", 1001), ("c2", 1002)]
    # no header; header only; header without a final LF
    h, rest = samstream.read_header(samstream._Source(io.BytesIO(body)), piece=3)
    assert h == b"" and rest.startswith(body[:3])
    h, rest = samstream.read_header(samstream._Source(io.BytesIO(head)), piece=5)
    assert (h, rest) == (head, b"")
    h, rest = samstream.read_header(samstream._Source(io.BytesIO(head[:-1])), piece=5)
    assert (h, rest) == (head[:-1], b"")
    with pytest.raises(OSError, match="empty input"):
        samstream.read_header(samstream._Source(io.BytesIO(b"")))
    with pytest.raises(OSError, match="file path"):
        samstream.read_header(samstream._Source(io.BytesIO(b"\x1f\x8b\x08\x04" + bytes(100))))
    with pytest.raises(OSError, match="not SAM"):
        samstream.read_header(samstream._Source(io.BytesIO(b"hello\tworld\n")))
    assert samstream.is_stream("-") and samstream.is_stream(io.BytesIO(b""))
    assert not samstream.is_stream(os.path.join(ROOT, "README.md"))
    r, w = os.pipe()
    try:
        assert samstream.is_stream("/dev/fd/%d" % r)
    finally:
        os.close(r)
        os.close(w)


@pytest.mark.parametrize("chunk", [1, 7, 64, 1000, 1 << 20])
@pytest.mark.parametrize("final_lf", [True, False])
def test_chunk_reader_whole_lines(chunk, final_lf):
    """A fake decoder sees whole lines only, in order, every byte once; buffers that hold no line grow."""
    from metacov_b200 import samstream
    rng = np.random.default_rng(chunk)
    body = _lines(300, rng, long_every=50).replace(b"\n", b"\r\n", 20)
    if not final_lf:
        body = body[:-1]
    f = _pipe_from(body, seed=chunk, max_piece=3000)
    got = []

    def decode(view, last):
        b = bytes(view)
        assert last or b.endswith(b"\n") or b == b""
        got.append(b)
        return True

    rd = samstream.ChunkReader(samstream._Source(f), b"", chunk)
    rd.run(decode)
    f.close()
    assert b"".join(got) == body
    assert rd.info()["bytes"] == len(body)


def test_last_lf_and_release():
    from metacov_b200 import samstream
    a = np.frombuffer(b"x" * 70000 + b"\n" + b"y" * 200000, dtype=np.uint8)
    assert samstream._last_lf(a, len(a)) == 70001 and samstream._last_lf(a, 70000) == 0 and samstream._last_lf(a, 0) == 0
    # a reader stopped early on a pipe whose writer is still alive: the handle is closed only once the thread is out
    r, w = os.pipe()
    f = os.fdopen(r, "rb", buffering=0)
    os.write(w, _lines(50, np.random.default_rng(5)))
    rd = samstream.ChunkReader(samstream._Source(f), b"", 64)
    rd.run(lambda v, last: False)
    closed = threading.Event()
    rd.release(lambda: (f.close(), closed.set()))
    os.write(w, b"x" * 4096)                                   # (wakes a thread blocked in read)
    os.close(w)
    assert closed.wait(10) and f.closed


def test_chunk_reader_stops_early():
    from metacov_b200 import samstream
    body = _lines(2000, np.random.default_rng(3))
    f = _pipe_from(body, max_piece=500)
    seen = []
    rd = samstream.ChunkReader(samstream._Source(f), b"", 256)
    rd.run(lambda v, last: seen.append(len(v)) or len(seen) < 3)
    assert len(seen) == 3
    f.close()


# ---- on the device -----------------------------------------------------------------------------------------------------

def _fixture_sam(path, crlf=False, final_newline=True):
    z, b = load_soa("fixture_soa.npz")
    so = z["seq_off"]
    n = len(b.tid)
    aux = ["AM:C:%d\tRG:Z:lane%d" % (int(z["mapq"][i]), i % 11 * 7) for i in range(n)]
    samio.write_sam(path, [str(x) for x in z["references"]], z["lengths"].tolist(), b.tid, b.pos, b.flag, b.mapq, b.cig_off,
                    b.cig, mtid=z["mtid"], mpos=z["mpos"], aux=aux, isize=z["isize"], names=[str(x) for x in z["names"]],
                    l_seq=z["l_seq"], seqs=[z["seq"][so[i]:so[i + 1]] for i in range(n)], crlf=crlf,
                    final_newline=final_newline)
    return path


def _same_depth(a, b):
    assert a.references == b.references and a.lengths == b.lengths
    for r, ln in zip(a.references, a.lengths):
        assert np.array_equal(a.count_coverage_depth(r, 0, ln), b.count_coverage_depth(r, 0, ln)), r
    assert a.coverage_engine().pass_info()["n_pass"] == b.coverage_engine().pass_info()["n_pass"]
    assert (a.mapped, a.unmapped) == (b.mapped, b.unmapped)


@pytest.mark.gpu
@pytest.mark.parametrize("crlf,final_lf", [(False, True), (True, True), (False, False)])
def test_fixture_through_a_pipe(tmp_path, crlf, final_lf):
    from metacov_b200 import AlignmentFile, pileup
    ps = _fixture_sam(str(tmp_path / "f.sam"), crlf=crlf, final_newline=final_lf)
    data = open(ps, "rb").read()
    gold = load_json("fixture_classic.json")
    with AlignmentFile(ps) as ref:
        for k, chunk in enumerate((701, 4096, 65536, 64 << 20)):
            with AlignmentFile(_pipe_from(data, seed=k, max_piece=5000), gpu_chunk_bytes=chunk, pinned_buffers=k == 2) as s:
                assert s.piped and s.format == "sam" and s.decode == "gpu-stream" and not s.has_index()
                assert s.references == ref.references and s.text == ref.text
                _same_depth(s, ref)
                for row in gold["classic"]:
                    assert pileup.classic(s, row["ref"], row["start"], row["end"]) == row["result"], row
                assert s.pipe_info["records"] == 4112 and s.pipe_info["bytes"] + len(s.text.encode()) == len(data)
                assert s.pipe_info["chunks"] >= (2 if chunk < len(data) else 1)
                assert s.pipe_info["longest_line"] == max(len(l) + 1 for l in data.split(b"\n") if not l.startswith(b"@"))


@pytest.mark.gpu
def test_every_offset_inside_a_line(tmp_path):
    """Chunk sizes 1..40 around short lines put the border at every offset of a line, and between CR and LF."""
    from metacov_b200 import AlignmentFile
    lengths = [500, 300]
    rng = np.random.default_rng(9)
    n = 120
    tid = rng.integers(0, 2, n).astype(np.int32)
    pos = rng.integers(0, 250, n).astype(np.int32)
    cig = np.array([(int(rng.integers(1, 40)) << 4) for _ in range(n)], np.uint32)
    off = np.arange(n + 1, dtype=np.uint32)
    flag = np.zeros(n, np.uint16)
    mapq = np.full(n, 30, np.uint8)
    ps = str(tmp_path / "s.sam")
    samio.write_sam(ps, ["a", "b"], lengths, tid, pos, flag, mapq, off, cig, crlf=True)
    data = open(ps, "rb").read()
    d, doff, _ = cport.depth(_batch(tid, pos, flag, mapq, off, cig), lengths, mode="diff")
    for chunk in range(1, 41):
        with AlignmentFile(io.BytesIO(data), gpu_chunk_bytes=chunk) as s:
            for c, r in enumerate(("a", "b")):
                assert np.array_equal(s.count_coverage_depth(r, 0, lengths[c]), d[doff[c]:doff[c] + lengths[c]]), (chunk, r)


def _batch(tid, pos, flag, mapq, off, cig):
    from metacov_b200 import ReadBatch
    return ReadBatch(np.asarray(tid, np.int32), np.asarray(pos, np.int32), np.asarray(flag, np.uint16),
                     np.asarray(mapq, np.uint8), np.asarray(off, np.uint32), np.asarray(cig, np.uint32))


def _pile(depth, length=3000, seed=0):
    """`depth` reads of 100M stacked at one position plus background reads, shuffled (aligner order)."""
    rng = np.random.default_rng(seed)
    n_bg = 2000
    pos = np.r_[np.full(depth, 1000), rng.integers(0, length - 150, n_bg)].astype(np.int32)
    n = len(pos)
    tid = np.zeros(n, np.int32)
    cig = np.full(n, 100 << 4, np.uint32)
    perm = rng.permutation(n)
    return _batch(tid, pos[perm], np.zeros(n, np.uint16), np.full(n, 30, np.uint8), np.arange(n + 1, dtype=np.uint32), cig)


@pytest.mark.gpu
def test_unsorted_input_and_the_exact_verdict(tmp_path):
    from metacov_b200 import AlignmentFile
    from metacov_b200.pileup import DepthCapError
    # shuffled reads give the sorted file's depth
    z, b = load_soa("fixture_soa.npz")
    n = len(b.tid)
    perm = np.random.default_rng(4).permutation(n)
    lens = np.diff(b.cig_off.astype(np.int64))
    cig = np.concatenate([b.cig[b.cig_off[i]:b.cig_off[i + 1]] for i in perm]).astype(np.uint32)
    off = np.r_[0, np.cumsum(lens[perm])].astype(np.uint32)
    refs, lengths = [str(x) for x in z["references"]], z["lengths"].tolist()
    pu, pso = str(tmp_path / "u.sam"), str(tmp_path / "s.sam")
    samio.write_sam(pu, refs, lengths, b.tid[perm], b.pos[perm], b.flag[perm], b.mapq[perm], off, cig)
    samio.write_sam(pso, refs, lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig)
    with AlignmentFile(pso) as ref, AlignmentFile(_pipe_from(open(pu, "rb").read()), gpu_chunk_bytes=9000) as s:
        _same_depth(s, ref)
    # a 5 000-deep pile in aligner order: the bound (about 2x the depth) would refuse it, the exact metric does not
    for depth, ok in ((5000, True), (12000, False)):
        pb = _pile(depth)
        p = str(tmp_path / ("p%d.sam" % depth))
        samio.write_sam(p, ["c"], [3000], pb.tid, pb.pos, pb.flag, pb.mapq, pb.cig_off, pb.cig)
        d, doff, info = cport.depth(pb, [3000], mode="diff")
        with AlignmentFile(_pipe_from(open(p, "rb").read()), gpu_chunk_bytes=50000) as s:
            if ok:
                assert np.array_equal(s.count_coverage_depth("c", 0, 3000), d[:3000])
                assert s.coverage_engine().pass_info()["cap_metric"] <= 8000
            else:
                with pytest.raises(DepthCapError, match="cannot be read again"):
                    s.count_coverage_depth("c", 0, 3000)
                with pytest.raises(ValueError):
                    s.count_coverage_depth("c", 0, 3000)
        if not ok:
            with AlignmentFile(_pipe_from(open(p, "rb").read())) as s:
                s.set_pileup_filter(max_depth=0)
                assert np.array_equal(s.count_coverage_depth("c", 0, 3000), d[:3000])
                with pytest.raises(ValueError, match="set_pileup_filter"):
                    s.set_pileup_filter(max_depth=100)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 4, 7, 10, 13, 22, 25, 31])
def test_exact_metric_equals_the_fused_one(seed):
    """mcov_begin_ex(EXACT_CAP) + push of the reads in any order reports the fused path's cap_metric on the sorted order."""
    import test_gpu_fuzz
    from metacov_b200 import CoverageEngine
    batch, _isize, lengths, _r, filt = test_gpu_fuzz._case(seed)
    filt = dict(filt, max_depth=3, count_del=1)
    n = len(batch.tid)
    with CoverageEngine(lengths, filt=filt) as eng:
        assert eng.compute_depth(batch) == "fused"
        fused = eng.pass_info()
        rng = np.random.default_rng(seed)
        perm = rng.permutation(n)
        lens = np.diff(batch.cig_off.astype(np.int64))
        cig = np.concatenate([batch.cig[batch.cig_off[i]:batch.cig_off[i + 1]] for i in perm] + [np.zeros(0, np.uint32)])
        sh = _batch(batch.tid[perm], batch.pos[perm], batch.flag[perm], batch.mapq[perm],
                    np.r_[0, np.cumsum(lens[perm])], cig)
        eng.begin(exact_cap=True)
        eng.push(sh)
        eng.finalize()
        exact = eng.pass_info()
        eng.begin()
        eng.push(sh)
        eng.finalize()
        bound = eng.pass_info()
        # a filter switched to count_del = 0 inside an exact pass: its starts would miss the reads pushed after it, so the
        # pass keeps the bound -- the metric of the same pushes in a plain pass
        infos = []
        for exact_cap in (True, False):
            eng.set_filter(count_del=1)
            eng.begin(exact_cap=exact_cap)
            eng.push(sh)
            eng.set_filter(count_del=0)
            eng.push(sh)
            eng.finalize()
            infos.append(eng.pass_info())
    assert exact["cap_metric"] == fused["cap_metric"], (seed, exact, fused)
    assert bound["cap_metric"] >= exact["cap_metric"]
    assert exact["n_pass"] == fused["n_pass"]
    assert infos[0] == infos[1]


@pytest.mark.gpu
def test_chunk_decode_abi():
    """mcov_sam_chunk_decode on pieces that end inside a line: it consumes through the last LF, reports 0 for a piece
    without one, takes everything with `last`, counts lines across chunks for errors and for the longest line."""
    import ctypes as C
    from metacov_b200 import CoverageEngine, McovError, _capi, bamgpu
    from metacov_b200._capi import lib
    head = _header(2)
    body = _lines(40, np.random.default_rng(8), long_every=13).replace(b"\tc0\t", b"\tc1\t", 7)[:-1]   # (no final LF)
    lines = body.split(b"\n")
    with CoverageEngine([1000, 1001]) as eng:
        n_ref = C.c_int32(0)
        eng._check(lib.mcov_sam_chunk_begin(eng._ctx, head, len(head), C.byref(n_ref)))
        assert n_ref.value == 2

        def decode(b, last):
            raw, used = _capi.BamDev(), C.c_int64(0)
            eng._check(lib.mcov_sam_chunk_decode(eng._ctx, b, len(b), 1 if last else 0, C.byref(used), C.byref(raw)))
            return used.value, bamgpu.DeviceSoA(eng, raw, "sam") if raw.n_records else None

        got_pos, p, piece = [], 0, 1000
        while True:
            chunk = body[p:p + piece]
            last = p + piece >= len(body)
            used, soa = decode(chunk, last)
            assert used == (len(chunk) if last else chunk.rfind(b"\n") + 1)
            if soa is not None:
                got_pos += soa.to_host("pos").tolist()
            p += used
            if last:
                break
            piece = 1000 if used else 2 * piece                        # (no complete line in the piece: a longer one)
        assert got_pos == [int(l.split(b"\t")[3]) - 1 for l in lines]
        assert lib.mcov_sam_chunk_longest_line(eng._ctx) == max([len(l) + 1 for l in lines[:-1]] + [len(lines[-1])])
        # a piece without an LF: nothing consumed; a malformed line names its line of the whole stream; the context goes on
        assert decode(b"r9\t0\tc0\t5", False)[0] == 0
        bad = lines[0].split(b"\t")
        bad[1] = b"x"
        with pytest.raises(McovError, match="line %d: FLAG" % (3 + len(lines) + 2)):
            decode(lines[0] + b"\n" + b"\t".join(bad) + b"\n", False)
        eng._check(lib.mcov_sam_chunk_begin(eng._ctx, head, len(head), None))
        used, soa = decode(body, True)
        assert used == len(body) and soa.n_records == len(lines)
        eng.begin()
        r = soa.raw
        eng._check(lib.mcov_push_reads(eng._ctx, soa.n_records, r.tid, r.pos, r.flag, r.mapq, r.cig_off, r.cig, _capi.MEM_DEVICE))
        eng.finalize()
        assert eng.pass_info()["n_pass"] == len(lines)


@pytest.mark.gpu
def test_long_header_and_long_lines(tmp_path):
    from metacov_b200 import AlignmentFile
    # 30 000 @SQ lines across many chunks
    refs = ["contig_%05d_%s" % (i, "q" * 20) for i in range(30000)]
    lengths = [200 + i % 50 for i in range(30000)]
    rng = np.random.default_rng(2)
    n = 3000
    tid = rng.integers(0, 30000, n).astype(np.int32)
    pos = rng.integers(0, 150, n).astype(np.int32)
    b = _batch(tid, pos, np.zeros(n, np.uint16), np.full(n, 20, np.uint8), np.arange(n + 1), np.full(n, 40 << 4, np.uint32))
    p = str(tmp_path / "h.sam")
    samio.write_sam(p, refs, lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig)
    with AlignmentFile(p) as ref, AlignmentFile(_pipe_from(open(p, "rb").read()), gpu_chunk_bytes=1 << 16) as s:
        assert len(s.references) == 30000
        for t in np.unique(tid)[:50]:
            r = refs[t]
            assert np.array_equal(s.count_coverage_depth(r), ref.count_coverage_depth(r))
        assert (s.mapped, s.unmapped) == (ref.mapped, ref.unmapped)
    # lines over 100 KB and 70 000-op CIGARs, longer than the chunk (buffer growth)
    n = 12
    ops = []
    off = [0]
    for i in range(n):
        k = 70000 if i % 3 == 0 else 5
        o = np.where(np.arange(k) % 2 == 0, (3 << 4) | 0, (1 << 4) | 2).astype(np.uint32)
        ops.append(o)
        off.append(off[-1] + k)
    cig = np.concatenate(ops)
    pos = np.sort(rng.integers(0, 1000, n)).astype(np.int32)
    b = _batch(np.zeros(n, np.int32), pos, np.zeros(n, np.uint16), np.full(n, 20, np.uint8), np.array(off), cig)
    p = str(tmp_path / "l.sam")
    samio.write_sam(p, ["big"], [400000], b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig)
    d, doff, _ = cport.depth(b, [400000], mode="diff")
    with AlignmentFile(_pipe_from(open(p, "rb").read()), gpu_chunk_bytes=40000) as s:
        assert np.array_equal(s.count_coverage_depth("big"), d[:400000])
        assert s.pipe_info["longest_line"] > 100000


@pytest.mark.gpu
def test_errors(tmp_path):
    from metacov_b200 import AlignmentFile
    from metacov_b200 import scan as mscan
    ps = _fixture_sam(str(tmp_path / "f.sam"))
    lines = open(ps, "rb").read().split(b"\n")
    n_head = sum(1 for l in lines if l.startswith(b"@"))
    bad = list(lines)
    k = n_head + 3000                                          # a record far into the stream: the third chunk or later
    f = bad[k].split(b"\t")
    f[4] = b"999"
    bad[k] = b"\t".join(f)
    with AlignmentFile(_pipe_from(b"\n".join(bad)), gpu_chunk_bytes=100000) as s:
        with pytest.raises(OSError, match="line %d: MAPQ" % (k + 1)):
            s.count_coverage_depth("ref1")
        assert s.pipe_info is None
        # the context that failed stays usable: a new stream on the same engine decodes and gives the file's depth
        from metacov_b200 import _capi, bamgpu
        from metacov_b200._capi import lib
        import ctypes as C
        eng = s._pipe_eng
        good = open(ps, "rb").read()
        head = b"".join(l + b"\n" for l in lines[:n_head])
        eng._check(lib.mcov_sam_chunk_begin(eng._ctx, head, len(head), None))
        raw, used = _capi.BamDev(), C.c_int64(0)
        eng._check(lib.mcov_sam_chunk_decode(eng._ctx, good[len(head):], len(good) - len(head), 1, C.byref(used), C.byref(raw)))
        assert raw.n_records == 4112
        eng.begin(exact_cap=True)
        eng._check(lib.mcov_push_reads(eng._ctx, raw.n_records, raw.tid, raw.pos, raw.flag, raw.mapq, raw.cig_off, raw.cig,
                                       _capi.MEM_DEVICE))
        eng.finalize()
        with AlignmentFile(ps) as ok:
            for t, r in enumerate(ok.references):
                assert np.array_equal(eng.copy_depth(t), ok.count_coverage_depth(r)), r
    with pytest.raises(OSError, match="empty input"):
        AlignmentFile(_pipe_from(b""))
    head = b"\n".join(l for l in lines if l.startswith(b"@")) + b"\n"
    with AlignmentFile(_pipe_from(head)) as s:
        assert s.references == ("ref1", "ref2")
        assert not s.count_coverage_depth(s.references[0]).any()
        assert (s.mapped, s.unmapped) == (0, 0)
    bam = os.path.join(str(tmp_path), "x.bam")
    from helpers import write_fixture_bam
    write_fixture_bam(bam)
    with pytest.raises(OSError, match="file path"):
        AlignmentFile(_pipe_from(open(bam, "rb").read()))
    # one consumer; record accessors
    with AlignmentFile(_pipe_from(open(ps, "rb").read())) as s:
        s.count_coverage_depth("ref1")
        with pytest.raises(ValueError, match="read once"):
            mscan.scan_reads(s, None, [mscan.IsizeHist()])
        for acc in (lambda: s.soa(), lambda: len(s), lambda: s.name_hashes(), lambda: s.qas_kmer_codes(3),
                    lambda: s.seq_windows(8), lambda: s.experimental_stats([], [], [], 3, None, None)):
            with pytest.raises(ValueError, match="read once"):
                acc()
    with AlignmentFile(_pipe_from(open(ps, "rb").read())) as s:
        mscan.scan_reads(s, None, [mscan.IsizeHist()])
        with pytest.raises(ValueError, match="scan_reads"):
            s.count_coverage_depth("ref1")


@pytest.mark.gpu
def test_scan_reads_on_a_stream(tmp_path):
    from metacov_b200 import AlignmentFile
    from metacov_b200 import scan as mscan
    ps = _fixture_sam(str(tmp_path / "f.sam"))
    data = open(ps, "rb").read()
    for maxreads in (0, 37, 2500):
        res = []
        for src in (ps, _pipe_from(data)):
            with AlignmentFile(src, gpu_chunk_bytes=20000) as f:
                bf = mscan.ByFlag([mscan.IsizeHist(), mscan.KmerHist(3, 4, 3, 1)], [mscan.Flags["Readdir"], mscan.Flags["IsRead1"]])
                nrec = mscan.scan_reads(f, None, bf, maxreads=maxreads)
                res.append((nrec, [[list(map(str, r)) for r in bf.get_rows(i)] for i in range(2)]))
                if not maxreads:
                    res[-1] += ((f.mapped, f.unmapped),)
        assert res[0] == res[1], maxreads
        assert res[0][0] == (maxreads or 4112)


def _cli_outputs(tmp_path, tag, args, stdin_data=None, runner=False):
    d = tmp_path / tag
    d.mkdir()
    full = [a.replace("{d}", str(d)) for a in args]
    if runner:
        from click.testing import CliRunner
        from metacov_b200.cli import main
        res = CliRunner().invoke(main, full, input=stdin_data)
        assert res.exit_code == 0, (res.output, res.exception)
    else:
        env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
        p = subprocess.run([sys.executable, "-m", "metacov_b200.cli"] + full, input=stdin_data, cwd=str(d), env=env,
                           capture_output=True)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
    return {f: open(os.path.join(str(d), f), "rb").read() for f in sorted(os.listdir(str(d)))}


@pytest.mark.gpu
def test_cli_on_a_pipe(tmp_path):
    from click.testing import CliRunner
    from metacov_b200.cli import pileup as pileup_cmd
    ps = _fixture_sam(str(tmp_path / "f.sam"))
    data = open(ps, "rb").read()
    from test_gpu_cli import BLAST7
    rb = tmp_path / "r.blast7"
    rb.write_text(BLAST7)
    args = ["pileup", "-b", "SRC", "-rb", str(rb), "-o", "{d}/o.csv", "-bg", "{d}/o.bg", "-w", "25", "-wo", "{d}/w.csv"]
    ref = _cli_outputs(tmp_path, "file", [a.replace("SRC", ps) for a in args])
    assert ref["o.csv"].count(b"\n") == 5 and len(ref["o.bg"]) > 0
    assert _cli_outputs(tmp_path, "pipe", [a.replace("SRC", "-") for a in args], stdin_data=data) == ref
    assert _cli_outputs(tmp_path, "runner", [a.replace("SRC", "-") for a in args], stdin_data=data, runner=True) == ref
    hargs = ["pileup", "-b", "SRC", "-o", "{d}/o.csv"]
    assert _cli_outputs(tmp_path, "hp", [a.replace("SRC", "-") for a in hargs], stdin_data=data) == \
        _cli_outputs(tmp_path, "hf", [a.replace("SRC", ps) for a in hargs])
    sargs = ["scan", "SRC", "-o", "{d}/k.csv", "-I", "{d}/i.csv", "-g", "Mapped", "-g", "IsRead1"]
    sref = _cli_outputs(tmp_path, "sfile", [a.replace("SRC", ps) for a in sargs])
    assert _cli_outputs(tmp_path, "spipe", [a.replace("SRC", "-") for a in sargs], stdin_data=data) == sref
    assert _cli_outputs(tmp_path, "spipe_t", [a.replace("SRC", "-") for a in sargs] + ["-t", "bam"], stdin_data=data) == sref
    assert _cli_outputs(tmp_path, "srun", [a.replace("SRC", "-") for a in sargs], stdin_data=data, runner=True) == sref
    kh = tmp_path / "k.csv"
    kh.write_bytes(sref["k.csv"])
    res = CliRunner().invoke(pileup_cmd, ["-b", "-", "-k", str(kh)], input=data)
    assert res.exit_code == 2 and "piped" in res.output
