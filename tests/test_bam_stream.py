"""The streaming host reader (csrc/bamio.cpp, mcov_bam_stream_*): batches of a BAM decoded into SoA buffers.
CPU part: the batches put together are the file (against the oracle's pure-Python reader), and the reads a
batch repeats from earlier ones are exactly those the resend rule of mcov_stream_push names.  GPU part: a
BAM streamed in >= 4 batches gives the depth of the one-shot pass bit for bit."""
import os

import numpy as np
import pytest

from helpers import load_soa, write_fixture_bam
from oracle import bamio, cport


def _write_synth_bam(tmp_path, scale=0.004, seed=None):
    from metacov_b200 import synth
    w = synth.c2(scale) if seed is None else synth.c2(scale, seed=seed)
    b, isize = synth.generate_host(w)
    refs = ["c%d" % c for c in range(w.n_contigs)]
    path = str(tmp_path / "synth.bam")
    bamio.write_bam(path, refs, w.contig_len.tolist(), b.tid, b.pos, b.flag, b.mapq, b.cig_off, b.cig, isize=isize)
    return path, w, b


def test_stream_batches_are_the_file(tmp_path):
    from metacov_b200.alignmentfile import BamStream
    paths = [_write_synth_bam(tmp_path)[0], write_fixture_bam(str(tmp_path / "bbmap.sorted.bam"))]
    for path in paths:
        hdr, recs = bamio.read_bam(path)
        for batch_reads in (997, 1 << 20):
            cols = {k: [] for k in ("tid", "pos", "flag", "mapq", "cig", "l_seq", "isize", "reflen", "ncig")}
            with BamStream(path, batch_reads=batch_reads, threads=3) as st:
                assert st.references == tuple(hdr.references) and st.lengths == tuple(hdr.lengths)
                n_batches = 0
                while True:
                    item = st.next_batch()                       # no resend point: nothing is repeated
                    if item is None:
                        break
                    b, n_carry, last, extra = item
                    assert n_carry == 0 and len(b.tid) <= batch_reads
                    for k in ("tid", "pos", "flag", "mapq", "cig"):
                        cols[k].append(np.array(getattr(b, k)))
                    cols["ncig"].append(np.diff(b.cig_off.astype(np.int64)))
                    for k in ("l_seq", "isize", "reflen"):
                        cols[k].append(np.array(extra[k]))
                    n_batches += 1
                    if last:
                        break
                assert st.next_batch() is None and st.n_records == len(recs.tid)
            assert n_batches == max(1, -(-len(recs.tid) // batch_reads)) or n_batches == len(recs.tid) // batch_reads + 1
            got = {k: np.concatenate(v) for k, v in cols.items()}
            for k, want in (("tid", recs.tid), ("pos", recs.pos), ("flag", recs.flag), ("mapq", recs.mapq), ("cig", recs.cig),
                            ("l_seq", recs.l_seq), ("isize", recs.isize), ("reflen", recs.reflen),
                            ("ncig", np.diff(np.asarray(recs.cig_off, dtype=np.int64)))):
                assert np.array_equal(got[k], np.asarray(want)), (path, batch_reads, k)


def test_stream_carry_follows_the_resend_rule(tmp_path):
    """A batch is led by every earlier read that starts at or after the resend point or reaches past it (file order)."""
    from metacov_b200.alignmentfile import BamStream
    path, w, b = _write_synth_bam(tmp_path, scale=0.006)
    hdr, recs = bamio.read_bam(path)
    tid, pos, reflen = np.asarray(recs.tid, np.int64), np.asarray(recs.pos, np.int64), np.asarray(recs.reflen, np.int64)
    rng = np.random.default_rng(5)
    with BamStream(path, batch_reads=7000, threads=2) as st:
        done = 0
        resend = (-1, 0)
        while True:
            item = st.next_batch(resend)
            assert item is not None
            bt, n_carry, last, extra = item
            if resend[0] >= 0:
                rt, rp = resend
                need = (tid[:done] > rt) | ((tid[:done] == rt) & ((pos[:done] >= rp) | (pos[:done] + reflen[:done] > rp)))
                idx = np.nonzero(need)[0]
                assert n_carry == len(idx)
                assert np.array_equal(bt.pos[:n_carry], pos[idx]) and np.array_equal(bt.tid[:n_carry], tid[idx])
                o = bt.cig_off.astype(np.int64)
                ro = np.asarray(recs.cig_off, dtype=np.int64)
                for k in rng.choice(n_carry, min(n_carry, 50), replace=False) if n_carry else []:
                    assert np.array_equal(bt.cig[o[k]:o[k + 1]], recs.cig[ro[idx[k]]:ro[idx[k] + 1]])
            else:
                assert n_carry == 0
            n_new = len(bt.tid) - n_carry
            assert np.array_equal(bt.pos[n_carry:], pos[done:done + n_new])
            done += n_new
            if last:
                break
            # a resend point a little behind the batch's last read, never moving backwards
            lt, lp = int(bt.tid[-1]), int(bt.pos[-1])
            cand = (lt, max(0, lp - int(rng.integers(0, 900))))
            resend = max(resend, cand)
        assert done == len(tid)


@pytest.mark.gpu
def test_bam_streamed_in_batches_equals_one_shot(tmp_path):
    """AlignmentFile streams the file through mcov_stream_push (here in >= 4 batches); depth, pass counters and
    `classic` records equal the whole-file pass and the C oracle."""
    from metacov_b200 import AlignmentFile, CoverageEngine, ReadBatch
    path, w, b = _write_synth_bam(tmp_path, scale=0.01)
    want, off, info = cport.depth(b, w.contig_len, mode="diff")
    with AlignmentFile(path, batch_reads=20000) as af:
        eng = af.coverage_engine()
        assert af.stream_batches >= 4
        for c in range(w.n_contigs):
            assert np.array_equal(eng.copy_depth(c), want[off[c]:off[c] + w.contig_len[c]]), c
        pi = eng.pass_info()
        assert pi["n_reads"] == len(b.tid) and pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"]
        tid = np.arange(w.n_contigs, dtype=np.int32)
        st = eng.region_stats(tid, np.zeros_like(tid), w.contig_len).copy()
    with CoverageEngine(w.contig_len) as one:
        one.depth_sorted(b)
        assert one.region_stats(tid, np.zeros_like(tid), w.contig_len).tobytes() == st.tobytes()
    # the reads of the reference fixture (golden SoA, written back to a BAM by the oracle's writer), three batches
    z, fb = load_soa("fixture_soa.npz")
    fpath = str(tmp_path / "fixture.bam")
    bamio.write_bam(fpath, [str(x) for x in z["references"]], z["lengths"].tolist(), fb.tid, fb.pos, fb.flag, fb.mapq, fb.cig_off, fb.cig)
    with AlignmentFile(fpath, batch_reads=1500) as af:
        eng = af.coverage_engine()
        assert af.stream_batches == 3
        fw, foff, _ = cport.depth(fb, np.asarray(af.lengths, np.int32), mode="diff")
        for c in range(2):
            assert np.array_equal(eng.copy_depth(c), fw[foff[c]:foff[c] + af.lengths[c]])


def test_stream_reader_with_small_file_reads(tmp_path, monkeypatch):
    """The streaming host reader reads the file in pieces (32 MB in production); MCOV_STREAM_READ_BYTES makes the pieces
    small, so that their borders cut the BGZF blocks and records of a small file everywhere.  Whatever the piece and batch
    sizes, the batches put together are the file (columns of the oracle's reader)."""
    from metacov_b200.alignmentfile import BamStream
    path = _write_synth_bam(tmp_path, scale=0.002)[0]
    hdr, recs = bamio.read_bam(path)
    size = os.path.getsize(path)
    rng = np.random.default_rng(3)
    for trial in range(14):
        piece = int(rng.integers(1024, max(2048, size // 2)))
        batch_reads = int(rng.integers(200, 9000))
        monkeypatch.setenv("MCOV_STREAM_READ_BYTES", str(piece))
        cols = {k: [] for k in ("tid", "pos", "flag", "mapq", "cig", "ncig")}
        with BamStream(path, batch_reads=batch_reads, threads=2) as st:
            assert st.references == tuple(hdr.references)
            while True:
                item = st.next_batch()
                if item is None:
                    break
                b, n_carry, last, extra = item
                assert n_carry == 0
                for k in ("tid", "pos", "flag", "mapq", "cig"):
                    cols[k].append(np.array(getattr(b, k)))
                cols["ncig"].append(np.diff(b.cig_off.astype(np.int64)))
                if last:
                    break
            assert st.n_records == len(recs.tid), (piece, batch_reads)
        got = {k: np.concatenate(v) for k, v in cols.items()}
        for k, want in (("tid", recs.tid), ("pos", recs.pos), ("flag", recs.flag), ("mapq", recs.mapq), ("cig", recs.cig),
                        ("ncig", np.diff(np.asarray(recs.cig_off, dtype=np.int64)))):
            assert np.array_equal(got[k], np.asarray(want)), (piece, batch_reads, k)
