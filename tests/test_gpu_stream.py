"""Streamed fused pass (mcov_stream_begin / mcov_stream_push): a coordinate-sorted read set pushed in several
batches -- each batch led by the reads the previous call asked to see again -- must give, bit for bit, the depth,
the pass counters and the statistics of the one-shot pass (and of the C oracle).  The reference streams records
and never holds the file (metacov/scan.pyx:653-667; pileup.py:13 iterates htslib's streaming pileup)."""
import numpy as np
import pytest

from oracle import cport

pytestmark = pytest.mark.gpu


def sub_batch(b, idx):
    from metacov_b200 import ReadBatch
    o = b.cig_off.astype(np.int64)
    n_ops = (o[idx + 1] - o[idx]) if len(idx) else np.zeros(0, np.int64)
    off = np.zeros(len(idx) + 1, np.int64)
    np.cumsum(n_ops, out=off[1:])
    cig = np.concatenate([b.cig[o[i]:o[i + 1]] for i in idx]) if len(idx) else np.zeros(0, np.uint32)
    return ReadBatch(b.tid[idx], b.pos[idx], b.flag[idx], b.mapq[idx], off.astype(np.uint32), cig.astype(np.uint32))


def push_in_batches(eng, b, reflen, cuts):
    """Push reads [cuts[k], cuts[k+1]) as batch k, led by the carry the previous push asked for."""
    eng.stream_begin()
    carry = np.zeros(0, np.int64)
    sizes = []
    for k in range(len(cuts) - 1):
        idx = np.concatenate([carry, np.arange(cuts[k], cuts[k + 1], dtype=np.int64)])
        last = k == len(cuts) - 2
        rt, rp = eng.stream_push(sub_batch(b, idx), n_carry=len(carry), last=last)
        sizes.append((len(carry), len(idx)))
        t, p = b.tid[idx].astype(np.int64), b.pos[idx].astype(np.int64)
        t = np.where(t < 0, np.iinfo(np.int64).max, t)               # unplaced reads sort last
        keep = (t > rt) | ((t == rt) & ((p >= rp) | (p + reflen[idx] > rp)))
        carry = idx[keep]
    return sizes


@pytest.mark.parametrize("wl,scale,n_batches", [("c2", 0.02, 5), ("c3", 0.002, 7), ("c5", 0.004, 6)])
def test_streamed_batches_equal_one_shot(wl, scale, n_batches):
    from metacov_b200 import CoverageEngine, synth
    w = synth.WORKLOADS[wl](scale)
    b, _, reflen = synth.generate_host(w, want_reflen=True)
    n = len(b.tid)
    rng = np.random.default_rng(11)
    cuts = np.r_[0, np.sort(rng.choice(np.arange(1, n), n_batches - 1, replace=False)), n]
    want, off, info = cport.depth(b, w.contig_len, mode="diff")
    tid = np.arange(w.n_contigs, dtype=np.int32)
    with CoverageEngine(w.contig_len) as eng:
        eng.depth_sorted(b)
        ref_stats = eng.region_stats(tid, np.zeros_like(tid), w.contig_len).copy()
        ref_info = eng.pass_info()
        sizes = push_in_batches(eng, b, reflen, cuts)
        assert len(sizes) == n_batches and all(c < m for c, m in sizes[1:])
        st = eng.region_stats(tid, np.zeros_like(tid), w.contig_len)            # delivers the verdict of the stream
        for c in range(w.n_contigs):
            assert np.array_equal(eng.copy_depth(c), want[off[c]:off[c] + w.contig_len[c]]), c
        assert st.tobytes() == ref_stats.tobytes()
        pi = eng.pass_info()
        for k in ("n_reads", "n_pass", "aligned_bases", "max_depth_seen", "sorted"):
            assert pi[k] == ref_info[k], (k, pi[k], ref_info[k])
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"]
        # a batch that ends inside the tile where the previous one ended (no new tile becomes final) is fine too
        sizes = push_in_batches(eng, b, reflen, np.r_[0, n // 2, n // 2 + 1, n // 2 + 2, n])
        assert np.array_equal(eng.copy_depth(0), want[off[0]:off[0] + w.contig_len[0]])
        assert eng.pass_info()["n_pass"] == info["n_pass"]


def test_stream_rejects_misuse():
    from metacov_b200 import CoverageEngine, McovError, synth
    w = synth.c2(0.004)
    b, _, reflen = synth.generate_host(w, want_reflen=True)
    n = len(b.tid)
    with CoverageEngine(w.contig_len) as eng:
        with pytest.raises(McovError):
            eng.stream_push(b, last=True)                                 # no stream_begin
        eng.stream_begin()
        eng.stream_push(sub_batch(b, np.arange(n // 2, n)), last=False)
        with pytest.raises(McovError):                                    # a batch that ends before the previous one
            eng.stream_push(sub_batch(b, np.arange(0, n // 4)), last=False)


def test_stream_cap_verdict_reaches_every_consumer():
    """Where htslib's max_depth cap fires in a streamed pass, the pass cannot be replayed exactly (the pile's contig
    may be spread over batches) and its depth is not the capped one.  Every call that delivers the verdict of such a
    pass must refuse it with MCOV_ERR_STATE, the pipelined statistics included."""
    from metacov_b200 import CoverageEngine, McovError, ReadBatch, _capi
    rng = np.random.default_rng(23)
    lengths = np.array([20000], np.int32)
    pos = np.sort(np.r_[np.full(400, 9000), rng.integers(0, 19900, 3000)]).astype(np.int32)     # a pile 400 deep
    n = len(pos)
    reflen = np.full(n, 100, np.int64)
    b = ReadBatch(np.zeros(n, np.int32), pos, np.zeros(n, np.uint16), np.full(n, 30, np.uint8),
                  np.arange(n + 1, dtype=np.uint32), reflen.astype(np.uint32) << 4)
    cuts = np.r_[0, n // 3, 2 * n // 3, n]
    tid, start, end = np.zeros(1, np.int32), np.zeros(1, np.int32), lengths

    def refused(call):
        with pytest.raises(McovError) as ei:
            call()
        assert ei.value.code == _capi.MCOV_ERR_STATE

    with CoverageEngine(lengths) as eng:
        eng.set_filter(max_depth=100)
        push_in_batches(eng, b, reflen, cuts)
        refused(lambda: eng.region_stats(tid, start, end))
        push_in_batches(eng, b, reflen, cuts)
        refused(eng.pass_info)
        for copy in (True, False):
            push_in_batches(eng, b, reflen, cuts)
            ticket = eng.region_stats_submit(tid, start, end, slot=0)
            refused(lambda: eng.region_stats_collect(ticket, copy=copy))
