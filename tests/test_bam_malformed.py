"""Malformed BAM files, one table of edits to a valid file: the whole-file host reader (mcov_bam_open + mcov_bam_load),
the streaming host reader (BamStream) and, on a GPU, the device decoder (bamgpu.decode, bamgpu.stream_depth) all return
an error for every case, and none lets an exception cross the C ABI."""
import ctypes as C
import struct

import pytest

from helpers import load_soa
from oracle import bamio


def _refs_at(data):
    """Offset of the first reference entry of an inflated BAM stream."""
    return 12 + struct.unpack_from("<i", data, 4)[0]


def _records_at(data):
    p = _refs_at(data)
    for _ in range(struct.unpack_from("<i", data, p - 4)[0]):
        p += 8 + struct.unpack_from("<i", data, p)[0]
    return p


def _patch(b, off, fmt, value):
    out = bytearray(b)
    struct.pack_into(fmt, out, off, value)
    return bytes(out)


def _block1_end(raw):
    return struct.unpack_from("<H", raw, 16)[0] + 1                # BSIZE + 1 of the first BGZF block


def _empty_first_name(data):
    """The first reference entry rewritten as l_name = 0 with no name bytes (its l_ref kept)."""
    p = _refs_at(data)
    l_name = struct.unpack_from("<i", data, p)[0]
    return data[:p] + struct.pack("<i", 0) + data[p + 4 + l_name:]


# name -> (edit of (compressed file, inflated stream), what the GPU decoder says)
CASES = {
    "gzip_magic": (lambda raw, data: b"\x1e" + raw[1:], "not a valid BGZF file"),
    "no_bc_field": (lambda raw, data: raw[:12] + b"XY" + raw[14:], "not a valid BGZF file"),
    "bsize_past_eof": (lambda raw, data: _patch(raw, len(raw) - 28 + 16, "<H", 1000), "not a valid BGZF file"),
    "isize_over_64k": (lambda raw, data: _patch(raw, _block1_end(raw) - 4, "<I", 65537), "not a valid BGZF file"),
    "crc_mismatch": (lambda raw, data: _patch(raw, _block1_end(raw) - 8, "<I", struct.unpack_from("<I", raw, _block1_end(raw) - 8)[0] ^ 1),
                     "CRC mismatch"),
    "trailing_bytes": (lambda raw, data: raw + b"these bytes follow the BGZF EOF block", "not a valid BGZF file"),
    "cut_in_text": (lambda raw, data: bamio.bgzf_compress(data[:8 + struct.unpack_from("<i", data, 4)[0] // 2]), "truncated BAM header"),
    "cut_in_ref_table": (lambda raw, data: bamio.bgzf_compress(data[:_refs_at(data) + 6]), "truncated reference table"),
    "empty_ref_name": (lambda raw, data: bamio.bgzf_compress(_empty_first_name(data)), "not a valid BAM file"),
    "l_seq_past_block_size": (lambda raw, data: bamio.bgzf_compress(_patch(data, _records_at(data) + 4 + 16, "<i", 0x7fffff00)), None),
}


def _good(tmp_path):
    z, b = load_soa("fixture_soa.npz")
    refs, lengths = [str(x) for x in z["references"]], [int(x) for x in z["lengths"]]
    path = str(tmp_path / "good.bam")
    bamio.write_bam(path, refs, lengths, b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig)
    return path, lengths


def _case_file(tmp_path, name):
    good, lengths = _good(tmp_path)
    raw = open(good, "rb").read()
    path = str(tmp_path / (name + ".bam"))
    open(path, "wb").write(CASES[name][0](raw, bamio.bgzf_inflate(raw)))
    return path, lengths


def _stream_all(path):
    from metacov_b200.alignmentfile import BamStream
    with BamStream(path, batch_reads=1000, threads=3) as st:
        while True:
            item = st.next_batch()
            if item is None or item[2]:
                break


def test_the_unedited_file_reads(tmp_path):
    from metacov_b200 import AlignmentFile
    path, _ = _good(tmp_path)
    with AlignmentFile(path) as bam:
        n = len(bam)
    assert n > 0
    _stream_all(path)


@pytest.mark.parametrize("name", sorted(CASES))
def test_host_readers_reject(tmp_path, monkeypatch, name):
    from metacov_b200 import McovError, _capi
    path, _ = _case_file(tmp_path, name)
    h = C.c_void_p()
    err = C.create_string_buffer(256)
    rc = _capi.lib.mcov_bam_open(C.byref(h), path.encode(), err, 256)
    if name == "l_seq_past_block_size":                            # the header is fine: the record pass fails
        assert rc == 0
        assert _capi.lib.mcov_bam_load(h, 0) == _capi.MCOV_ERR_IO
        _capi.lib.mcov_bam_close(h)
    else:
        assert rc == _capi.MCOV_ERR_IO and err.value.startswith(b"mcov_bam_open: not a valid B")
    for read_bytes in (None, "1024"):                              # 1024: a read border inside every block and record
        if read_bytes is None:
            monkeypatch.delenv("MCOV_STREAM_READ_BYTES", raising=False)
        else:
            monkeypatch.setenv("MCOV_STREAM_READ_BYTES", read_bytes)
        with pytest.raises((OSError, McovError)):
            _stream_all(path)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_decoder_rejects(tmp_path, name):
    from metacov_b200 import CoverageEngine, McovError, bamgpu
    path, lengths = _case_file(tmp_path, name)
    why = CASES[name][1]
    with CoverageEngine(lengths) as eng:
        if why is None:                       # the device decoder reads SEQ only when asked for it
            soa = bamgpu.decode(eng, path)
            with pytest.raises(McovError, match="SEQ leaves the record"):
                soa.names_seq(win_bases=8)
        else:
            with pytest.raises(McovError, match=why):
                bamgpu.decode(eng, path)
            with pytest.raises(McovError, match="the file ends inside a BGZF block" if name == "bsize_past_eof" else why):
                bamgpu.stream_depth(eng, path)
        good, _ = _good(tmp_path)
        assert bamgpu.decode(eng, good).n_records > 0              # the context survives the error


@pytest.mark.gpu
def test_alignment_file_rejects_an_empty_reference_name(tmp_path):
    """A reference whose l_name is 0 is not a valid BAM file, whichever decoder reads the header (the table above runs
    the case through bamgpu.decode and bamgpu.stream_depth)."""
    from metacov_b200 import AlignmentFile
    path, _ = _case_file(tmp_path, "empty_ref_name")
    for decode in ("gpu", "host", "gpu-stream"):
        with pytest.raises(OSError, match="not a valid BAM file"):
            AlignmentFile(path, decode=decode)
