"""Parity of the CUDA path (through the C-ABI) against the oracle and the committed golden
vectors.  Integer results bit-exact; floats to the cent after the reference's round(.,2)
(1e-6 relative before rounding is checked in test_host_logic)."""
import os

import numpy as np
import pytest

from helpers import assert_classic_equal, load_json, load_soa, regions_of
from oracle import cport

pytestmark = pytest.mark.gpu


def engine_for(lengths, **filt):
    from metacov_b200 import CoverageEngine
    return CoverageEngine(lengths, filt=filt or None)


def full_depth(eng):
    return [eng.copy_depth(c) for c in range(len(eng.lengths))]


def oracle_depth(batch, lengths, mode="diff", **filt):
    d, off, info = cport.depth(batch, lengths, filt=cport.default_filter(**filt) if filt else None, mode=mode)
    return [d[off[c]:off[c] + lengths[c]] for c in range(len(lengths))], d, off, info


@pytest.mark.parametrize("soa,js", [("fixture_soa.npz", "fixture_classic.json"),
                                    ("synth_small_soa.npz", "synth_small_classic.json")])
@pytest.mark.parametrize("path", ["fused", "push"])
def test_golden_depth_and_classic(soa, js, path):
    from metacov_b200.pileup import finish_classic
    z, b = load_soa(soa)
    gold = load_json(js)
    lengths = z["lengths"]
    with engine_for(lengths) as eng:
        if path == "fused":
            eng.depth_sorted(b)
        else:
            eng.begin(); eng.push(b); eng.finalize()
        want, _, _, info = oracle_depth(b, lengths)
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c]), (path, c)
        pi = eng.pass_info()
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"]
        assert pi["sorted"] == 1
        tid, st, en = regions_of(gold, z["references"])
        stats = eng.region_stats(tid, st, en)
        for row, rec, a, e in zip(gold["classic"], stats, st, en):
            assert rec["flags"] & 1
            assert_classic_equal(finish_classic(rec, e - a), row["result"], (path, row))


def test_fixture_depth_known_answers():
    import hashlib
    z, b = load_soa("fixture_soa.npz")
    with engine_for(z["lengths"]) as eng:
        assert eng.compute_depth(b) == "fused"
        d = full_depth(eng)
        assert hashlib.sha1(d[0].astype("<i4").tobytes()).hexdigest() == "11ed20e88c63aa6c8ee4c7a7b002e66f5b1b69aa"
        assert hashlib.sha1(d[1].astype("<i4").tobytes()).hexdigest() == "d3075eb38351dde7ace91e8975de6333040f5373"
        assert eng.pass_info()["n_pass"] == 3350


@pytest.mark.parametrize("wl,scale", [("c2", 0.02), ("c3", 0.002), ("c5", 0.004)])
@pytest.mark.parametrize("path", ["fused", "push"])
def test_synthetic_configs_bit_exact(wl, scale, path):
    """Scaled-down BASELINE configs: depth bit-exact against the C oracle, region stats equal."""
    from metacov_b200 import synth
    w = synth.WORKLOADS[wl](scale)
    b, _ = synth.generate_host(w)
    lengths = w.contig_len
    with engine_for(lengths) as eng:
        if path == "fused":
            eng.depth_sorted(b)
        else:
            eng.begin()
            # several pushes: batches split at arbitrary read boundaries
            n = len(b.tid)
            cuts = [0, n // 3, n // 3 + 1, n]
            o = b.cig_off.astype(np.int64)
            for lo, hi in zip(cuts[:-1], cuts[1:]):
                from metacov_b200 import ReadBatch
                eng.push(ReadBatch(b.tid[lo:hi], b.pos[lo:hi], b.flag[lo:hi], b.mapq[lo:hi],
                                   (o[lo:hi + 1] - o[lo]).astype(np.uint32), b.cig[o[lo]:o[hi]]))
            eng.finalize()
        want, dflat, off, info = oracle_depth(b, lengths)
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c]), (wl, path, c)
        pi = eng.pass_info()
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"]
        assert pi["max_depth_seen"] == int(dflat.max())
        # whole-contig regions plus random sub-ranges (overlapping)
        rng = np.random.default_rng(3)
        nc = len(lengths)
        tid = np.r_[np.arange(nc), rng.integers(0, nc, 64)].astype(np.int32)
        a = np.r_[np.zeros(nc, np.int64), [rng.integers(0, lengths[t]) for t in tid[nc:]]]
        e = np.r_[lengths.astype(np.int64), [rng.integers(a[nc + k] + 1, lengths[t] + 1) for k, t in enumerate(tid[nc:])]]
        got = eng.region_stats(tid, a, e, breadth_n=10)
        ref = cport.region_stats(dflat, off, lengths, tid, a, e, breadth_n=10)
        for k in ("sum", "sumsq", "iq_sum", "n_ge1", "n_geN", "min", "max", "med_lo", "med_hi"):
            assert np.array_equal(got[k], ref[k]), (wl, path, k)


def test_exact_cap_metric_fused():
    """cap_metric of the fused path = max_p depth[p-1] + starts[p] (htslib no-op condition)."""
    from metacov_b200 import synth
    w = synth.c3(0.001)
    b, _ = synth.generate_host(w)
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted(b)
        pi = eng.pass_info()
        want, dflat, off, _ = oracle_depth(b, w.contig_len)
        ok = cport.default_filter()
        from oracle.pysam_boundary import PileupFilter
        passing = PileupFilter().passes(b.flag, b.mapq)
        from oracle import bamio
        rl = bamio.cigar_reflen(b.cig_off, b.cig)
        passing &= rl > 0
        best = 0
        for c in range(w.n_contigs):
            sel = passing & (b.tid == c)
            starts = np.bincount(b.pos[sel], minlength=w.contig_len[c] + 1)[:w.contig_len[c]]
            prev = np.r_[0, want[c][:-1]]
            best = max(best, int((prev + starts).max()))
        assert pi["cap_metric"] == best
        eng.begin(); eng.push(b); eng.finalize()
        assert eng.pass_info()["cap_metric"] >= best      # push path: upper bound


def test_unsorted_input_falls_to_push_path_on_gpu():
    from metacov_b200 import McovError, ReadBatch, _capi
    z, b = load_soa("synth_small_soa.npz")
    perm = np.random.default_rng(5).permutation(len(b.tid))
    o = b.cig_off.astype(np.int64)
    ncig = np.diff(o)[perm]
    cig = np.concatenate([b.cig[o[i]:o[i + 1]] for i in perm]) if len(b.cig) else b.cig
    sb = ReadBatch(b.tid[perm], b.pos[perm], b.flag[perm], b.mapq[perm],
                   np.r_[0, np.cumsum(ncig)].astype(np.uint32), cig.astype(np.uint32))
    with engine_for(z["lengths"]) as eng:
        with pytest.raises(McovError) as ei:
            eng.depth_sorted(sb)
        assert ei.value.code == _capi.MCOV_ERR_UNSORTED
        assert eng.compute_depth(sb) == "push"
        assert eng.pass_info()["sorted"] == 0
        want, _, _, _ = oracle_depth(b, z["lengths"])
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c])


def test_filters_and_edge_cases():
    from metacov_b200 import McovError, ReadBatch
    z, b = load_soa("synth_small_soa.npz")
    lengths = z["lengths"]
    for filt in (dict(ignore_orphans=0), dict(flag_filter=0x4), dict(min_mapq=30), dict(flag_require=0x10),
                 dict(flag_filter=0, ignore_orphans=0)):
        with engine_for(lengths, **filt) as eng:
            eng.depth_sorted(b)
            want, _, _, _ = oracle_depth(b, lengths, **filt)
            for c, d in enumerate(full_depth(eng)):
                assert np.array_equal(d, want[c]), filt
    with engine_for(lengths) as eng:
        # empty input: all-zero depth, stats of zeros
        empty = ReadBatch(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.uint16), np.zeros(0, np.uint8),
                          np.zeros(1, np.uint32), np.zeros(0, np.uint32))
        eng.depth_sorted(empty)
        assert all(int(d.sum()) == 0 for d in full_depth(eng))
        st = eng.region_stats([0, 2], [0, 10], [lengths[0], 11])
        assert st["sum"].tolist() == [0, 0] and st["max"].tolist() == [0, 0] and (st["flags"] & 1).all()
        # zero-length region -> zeros, no crash; bad regions -> MCOV_ERR_ARG
        assert eng.region_stats([0], [5], [5])["flags"][0] == 0
        with pytest.raises(McovError):
            eng.region_stats([7], [0], [5])
        with pytest.raises(McovError):
            eng.region_stats([0], [9], [5])
    # calls out of order
    with engine_for(lengths) as eng:
        with pytest.raises(McovError):
            eng.finalize()
        with pytest.raises(McovError):
            eng.region_stats([0], [0], [5])
        with pytest.raises(McovError):
            eng.push(b)


def test_region_beyond_contig_end_counts_zeros():
    """pileup.py:10-11: the vector is end-start long whatever the contig length."""
    z, b = load_soa("fixture_soa.npz")
    with engine_for(z["lengths"]) as eng:
        eng.depth_sorted(b)
        _, dflat, off, _ = oracle_depth(b, z["lengths"])
        tid, a, e = [0, 1, 1], [400, 0, 575], [500, 2000, 600]
        got = eng.region_stats(tid, a, e)
        ref = cport.region_stats(dflat, off, z["lengths"], tid, a, e)
        for k in ("sum", "sumsq", "iq_sum", "n_ge1", "min", "max", "med_lo", "med_hi"):
            assert np.array_equal(got[k], ref[k]), k


def test_large_regions_multi_chunk_and_window_means():
    """A region longer than one chunk merges partial histograms through the global pool."""
    from metacov_b200 import synth
    w = synth.Workload("big", [300_000, 70_000], [60_000, 9_000], seed=11)
    b, _ = synth.generate_host(w)
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted(b)
        want, dflat, off, _ = oracle_depth(b, w.contig_len)
        tid, a, e = [0, 0, 1, 0], [0, 5, 0, 100_000], [300_000, 299_999, 70_000, 100_001]
        got = eng.region_stats(tid, a, e)
        ref = cport.region_stats(dflat, off, w.contig_len, tid, a, e)
        for k in ("sum", "sumsq", "iq_sum", "n_ge1", "min", "max", "med_lo", "med_hi"):
            assert np.array_equal(got[k], ref[k]), k
        wm = eng.window_means(1000)
        exp = np.concatenate([[d[i:i + 1000].mean() for i in range(0, len(d), 1000)] for d in want])
        assert np.allclose(wm, exp, rtol=0, atol=1e-12)


def test_histogram_overflow_uses_gpu_radix_path():
    """Depth beyond the counting histogram (needs max_depth raised): exact order statistics."""
    from metacov_b200 import ReadBatch
    n = 20000
    rng = np.random.default_rng(2)
    pos = np.sort(np.r_[np.full(12000, 100), rng.integers(0, 900, n - 12000)]).astype(np.int32)
    b = ReadBatch(np.zeros(n, np.int32), pos, np.zeros(n, np.uint16), np.full(n, 30, np.uint8),
                  np.arange(n + 1, dtype=np.uint32), np.full(n, 100 << 4, np.uint32))
    with engine_for([1000], max_depth=0) as eng:
        eng.depth_sorted(b)
        pi = eng.pass_info()
        assert pi["max_depth_seen"] > 8191 and pi["cap_metric"] > 8000
        _, dflat, off, _ = oracle_depth(b, np.array([1000], np.int32))
        tid, a, e = [0, 0, 0], [0, 90, 0], [1000, 250, 1500]
        got = eng.region_stats(tid, a, e)
        ref = cport.region_stats(dflat, off, np.array([1000], np.int32), tid, a, e)
        assert (got["flags"] & 2).all()
        for k in ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi"):
            assert np.array_equal(got[k], ref[k]), k


def test_isize_hist_byflag():
    z, _ = load_soa("fixture_soa.npz")
    with engine_for(z["lengths"]) as eng:
        for gf in ((), (0x4, 0x40), (0x10, 0x1, 0x80)):
            hist, cnt, mx = eng.isize_hist(z["flag"], z["isize"], gf, n_bins=64)   # forces a regrow
            rh, rc, rmx = cport.isize_hist(z["flag"], z["isize"], gf, hist.shape[1])
            assert mx == rmx == 248 and np.array_equal(hist, rh) and np.array_equal(cnt, rc)


def test_device_resident_inputs_match_host_inputs():
    import torch
    from metacov_b200 import synth
    w = synth.c2(0.01)
    hb, hisz = synth.generate_host(w)
    db, disz = synth.generate_device(w, 0)
    for name, h, d in zip(hb._fields, hb, db):
        hv = np.asarray(h)
        dv = d.cpu().numpy().view(hv.dtype)
        assert np.array_equal(hv, dv), name
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted(db)
        want, _, _, _ = oracle_depth(hb, w.contig_len)
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c])
        # torch-owned depth buffer
        buf = torch.zeros(eng.n_slots, dtype=torch.int32, device="cuda")
        eng.bind_depth(buf)
        eng.depth_sorted(db)
        torch.cuda.synchronize()
        o = eng.contig_offset(3)
        assert np.array_equal(buf[o:o + int(w.contig_len[3])].cpu().numpy(), want[3])


def region_iterator_stats(b, lengths, t, a, e):
    """The reference's numbers for regions of a pass where max_depth may fire: one htslib iterator per
    region, fed the reads overlapping it (bam.pileup(ref, start, end), pileup.py:13); columns outside
    [start, end) are discarded (pileup.py:14-15).  Single-op reads only (reflen = cigar >> 4)."""
    from metacov_b200 import ReadBatch
    rows = []
    tid = np.asarray(b.tid); pos = np.asarray(b.pos).astype(np.int64); rl = (np.asarray(b.cig) >> 4).astype(np.int64)
    for ti, ai, ei in zip(t, a, e):
        m = np.flatnonzero((tid == ti) & (pos < ei) & (pos + rl > ai))
        sub = ReadBatch(tid[m], np.asarray(b.pos)[m], np.asarray(b.flag)[m], np.asarray(b.mapq)[m],
                        np.arange(len(m) + 1, dtype=np.uint32), np.asarray(b.cig)[m])
        d, off, _ = cport.depth(sub, lengths, mode="plp")
        rows.append(cport.region_stats(d, off, lengths, [ti], [ai], [ei]))
    return np.concatenate(rows)


def test_max_depth_cap_replayed_exactly():
    """Where htslib's maxcnt fires, the fused path replays the affected contigs and must equal the
    sequential htslib machine (oracle orc_depth_plp), statistics included."""
    from metacov_b200 import ReadBatch
    rng = np.random.default_rng(9)
    lengths = np.array([3000, 1500, 2500], np.int32)
    tid, pos = [], []
    # contig 0: a 12 000-deep stack at 300 plus background and a second pile at 310; contig 1: shallow;
    # contig 2: ramp that crosses 8000 gradually (never capped: reads arrive at distinct positions)
    for c, ps in ((0, np.r_[np.full(12000, 300), np.full(3000, 310), rng.integers(0, 2800, 4000)]),
                  (1, rng.integers(0, 1400, 2000)),
                  (2, np.r_[np.repeat(np.arange(100, 1100), 9), rng.integers(0, 2300, 500)])):
        ps = np.sort(ps)
        tid += [c] * len(ps); pos += ps.tolist()
    n = len(tid)
    rl = rng.integers(60, 140, n)
    rl[np.array(tid) == 2] = 1200
    b = ReadBatch(np.array(tid, np.int32), np.array(pos, np.int32), np.zeros(n, np.uint16), np.full(n, 30, np.uint8),
                  np.arange(n + 1, dtype=np.uint32), (rl.astype(np.uint32) << 4))
    want, off, info = cport.depth(b, lengths, mode="plp")
    assert info["dropped_by_cap"] > 0
    with engine_for(lengths) as eng:
        eng.depth_sorted(b)
        pi = eng.pass_info()
        assert pi["cap_metric"] > 8000 and pi["cap_contigs"] >= 1
        for c in range(3):
            assert np.array_equal(eng.copy_depth(c), want[off[c]:off[c] + lengths[c]]), c
        # whole-contig regions read the replayed store; a region inside a capped contig gets its own iterator
        # (only the reads overlapping it), which keeps MORE of a pile once the reads that ended before the region
        # no longer occupy the buffer: [320, 420) starts behind the pile at 300 / 310
        t, a, e = [0, 1, 2, 0, 0, 0, 2], [0, 0, 0, 250, 320, 2990, 1000], [3000, 1500, 2500, 400, 420, 3100, 1800]
        got = eng.region_stats(t, a, e)
        ref = region_iterator_stats(b, lengths, t, a, e)
        whole = cport.region_stats(want, off, lengths, t, a, e)
        keys = ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi")
        for k in keys:
            assert np.array_equal(got[k], ref[k]), (k, got[k], ref[k], whole[k])
        assert any(not np.array_equal(ref[k], whole[k]) for k in keys)      # (the two iterators do differ here)
        # the pipelined form has no reads left to replay from: it refuses regions that start inside a contig ...
        from metacov_b200 import McovError
        eng.depth_sorted(b, wait=False)
        tk = eng.region_stats_submit(t, a, e, slot=0)
        with pytest.raises(McovError, match="per-region iterator"):
            eng.region_stats_collect(tk)
        # ... and serves whole-contig regions
        eng.depth_sorted(b, wait=False)
        got = eng.region_stats_collect(eng.region_stats_submit(t[:3], a[:3], e[:3], slot=0))
        for k in keys:
            assert np.array_equal(got[k], whole[k][:3]), k
    # cap disabled: plain difference-array depth again
    with engine_for(lengths, max_depth=0) as eng:
        eng.depth_sorted(b)
        assert eng.pass_info()["cap_contigs"] == 0
        free, _, _ = cport.depth(b, lengths, mode="diff")
        assert np.array_equal(eng.copy_depth(0), free[off[0]:off[0] + lengths[0]])


def _capped_pile_batch():
    from metacov_b200 import ReadBatch
    rng = np.random.default_rng(19)
    lengths = np.array([2000, 1200], np.int32)
    ps0 = np.sort(np.r_[np.full(11000, 500), np.full(2500, 505), rng.integers(0, 1800, 3000)])
    ps1 = np.sort(rng.integers(0, 1100, 1500))
    tid = np.r_[np.zeros(len(ps0), np.int32), np.ones(len(ps1), np.int32)]
    pos = np.r_[ps0, ps1].astype(np.int32)
    n = len(tid)
    rl = rng.integers(60, 140, n).astype(np.uint32)
    b = ReadBatch(tid, pos, np.zeros(n, np.uint16), np.full(n, 30, np.uint8), np.arange(n + 1, dtype=np.uint32), rl << 4)
    return b, lengths


def test_cap_replay_precedes_every_consumer_of_an_async_pass():
    """depth_sorted(wait=False) defers the verdict, but the max_depth replay runs on the device in
    stream order: statistics, copies, run export and window means issued before the verdict has been
    looked at must already see the capped depth (oracle: the sequential htslib machine)."""
    b, lengths = _capped_pile_batch()
    want, off, info = cport.depth(b, lengths, mode="plp")
    assert info["dropped_by_cap"] > 0
    t, a, e = [0, 1, 0], [0, 0, 450], [2000, 1200, 700]
    keys = ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi")
    with engine_for(lengths) as eng:
        eng.depth_sorted(b, wait=False)
        got = eng.region_stats(t, a, e)                       # first synchronising call after the async pass
        ref = region_iterator_stats(b, lengths, t, a, e)
        for k in keys:
            assert np.array_equal(got[k], ref[k]), k
        t, a, e = t[:2], a[:2], e[:2]
        ref = cport.region_stats(want, off, lengths, t, a, e)
        assert eng.pass_info()["cap_contigs"] >= 1            # contig 0 (and contig 1, which shares its last tile)
        eng.depth_sorted(b, wait=False)
        assert np.array_equal(eng.copy_depth(0), want[off[0]:off[0] + lengths[0]])
        eng.depth_sorted(b, wait=False)
        runs = eng.depth_runs()
        d0 = np.repeat(runs["depth"][runs["tid"] == 0], (runs["end"] - runs["start"])[runs["tid"] == 0])
        assert np.array_equal(d0, want[off[0]:off[0] + lengths[0]])
        eng.depth_sorted(b, wait=False)
        wm = eng.window_means(500)
        assert np.allclose(wm[:4], want[off[0]:off[0] + 2000].reshape(4, 500).mean(axis=1))
        # pipelined statistics: the replay is part of the pass, so submit/collect deliver capped records too
        eng.depth_sorted(b, wait=False)
        tk = eng.region_stats_submit(t, a, e, slot=0)
        eng.depth_sorted(b, wait=False)                        # the next pass overwrites the depth
        tk2 = eng.region_stats_submit(t, a, e, slot=1)
        for tkt in (tk, tk2):
            got = eng.region_stats_collect(tkt)
            for k in keys:
                assert np.array_equal(got[k], ref[k]), k


@pytest.mark.parametrize("wl,scale", [("c2", 0.01), ("c5", 0.004)])
def test_wide_cigar_offsets_equal_narrow(wl, scale):
    """64-bit CIGAR offsets (mcov_depth_sorted_wide / mcov_push_reads_wide: batches of 2^32 or more ops,
    config C5 at full size) give the depth of the 32-bit entry points -- host and device-resident."""
    import torch
    from metacov_b200 import ReadBatch, synth
    w = synth.WORKLOADS[wl](scale)
    b, _ = synth.generate_host(w)
    bw, _ = synth.generate_host(w, wide=True)
    assert bw.cig_off.dtype == np.uint64
    want, _, _, _ = oracle_depth(b, w.contig_len)

    def same(eng):
        return all(np.array_equal(d, want[c]) for c, d in enumerate(full_depth(eng)))

    with engine_for(w.contig_len) as eng:
        eng.depth_sorted(bw)
        assert same(eng)
        eng.begin(); eng.push(bw); eng.finalize()
        assert same(eng)
        db, _ = synth.generate_device(w, 0, wide=True)
        assert db.cig_off.dtype == torch.int64
        eng.depth_sorted(db, wait=False)
        assert same(eng)
        eng.begin(); eng.push(db); eng.finalize()
        assert same(eng)


@pytest.mark.parametrize("wl,scale", [("c2", 0.01), ("c5", 0.002)])
def test_packed_host_transport_equals_soa_path(wl, scale):
    """mcov_depth_sorted_packed (contig prefix + u16 op counts, no mapq) rebuilds the SoA on the device."""
    from metacov_b200 import McovError, synth
    from metacov_b200.engine import pack_batch, packed_bytes
    w = synth.WORKLOADS[wl](scale)
    b, _ = synth.generate_host(w)
    packed = pack_batch(b, w.n_contigs)
    assert packed_bytes(packed) < sum(np.asarray(x).nbytes for x in b)
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted_packed(packed)
        want, dflat, off, info = oracle_depth(b, w.contig_len)
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c]), c
        pi = eng.pass_info()
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"] and pi["sorted"] == 1
        # op counts that do not add up to the op array are refused (the device would read cig[] by them)
        bad = dict(packed)
        bad["n_cigar"] = np.array(packed["n_cigar"], copy=True)
        bad["n_cigar"][len(bad["n_cigar"]) // 2] += 3
        with pytest.raises(McovError):
            eng.depth_sorted_packed(bad)
        # with mapq shipped and a mapq filter
        eng.set_filter(min_mapq=30)
        with pytest.raises(McovError):
            eng.depth_sorted_packed(packed)                     # mapq required when min_mapq > 0
        eng.depth_sorted_packed(pack_batch(b, w.n_contigs, with_mapq=True))
        want30, _, _, _ = oracle_depth(b, w.contig_len, min_mapq=30)
        assert np.array_equal(eng.copy_depth(0), want30[0])
    # unplaced reads at the end and pinned tensors
    z, fb = load_soa("fixture_soa.npz")
    with engine_for(z["lengths"]) as eng:
        eng.depth_sorted_packed(pack_batch(fb, 2, pinned=True))
        wantf, _, _, _ = oracle_depth(fb, z["lengths"])
        assert np.array_equal(eng.copy_depth(1), wantf[1]) and eng.pass_info()["n_pass"] == 3350


def test_full_size_c2_bit_exact_and_properties():
    """BASELINE config C2 at full size (10 M x 150 bp, 1 000 contigs): bit-exact against the C
    oracle, plus size-independent properties (mass conservation, idempotence, path equivalence)."""
    import torch
    from metacov_b200 import ReadBatch, synth
    w = synth.c2(1.0)
    db, _, drl = synth.generate_device(w, 0, want_reflen=True)
    hb = ReadBatch(*[np.ascontiguousarray(t.cpu().numpy()) for t in db])
    hb = ReadBatch(hb.tid, hb.pos, hb.flag.view(np.uint16), hb.mapq, hb.cig_off.view(np.uint32), hb.cig.view(np.uint32))
    want, off, info = cport.depth(hb, w.contig_len, mode="par", threads=os.cpu_count() or 4)
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted(db)
        pi = eng.pass_info()
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"]
        assert pi["max_depth_seen"] == int(want.max()) and pi["cap_contigs"] == 0
        # whole depth array, bit for bit (slot layout of the oracle = slot layout of the engine)
        assert eng.n_slots == len(want)
        buf = torch.empty(eng.n_slots, dtype=torch.int32, device="cuda")
        eng.bind_depth(buf)
        eng.depth_sorted(db)
        got = buf.cpu().numpy()
        assert np.array_equal(got, want)
        # mass conservation: sum(depth) == aligned bases (no read is clipped in this workload)
        assert int(got.astype(np.int64).sum()) == info["aligned_bases"]
        # idempotence and path equivalence (push path on the same buffer)
        eng.begin(); eng.push(db); eng.finalize()
        torch.cuda.synchronize()
        assert torch.equal(buf, torch.from_numpy(want).cuda())
        # statistics of every contig
        tid = np.arange(w.n_contigs, dtype=np.int32)
        st = eng.region_stats(tid, np.zeros_like(tid), w.contig_len)
        ref = cport.region_stats(want, off, w.contig_len, tid, np.zeros_like(tid), w.contig_len, threads=os.cpu_count() or 4)
        for k in ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi", "n_ge1"):
            assert np.array_equal(st[k], ref[k]), k
        assert int(st["sum"].sum()) == info["aligned_bases"]


def test_dense_tile_takes_unpacked_counters():
    """A tile touched by >= 32 768 reads leaves the packed (16+16 bit) counters of k_fused_tile_tma for two
    32-bit passes (starts, then ends); depth stays bit-exact either way (cap disabled: 70 000 reads start at
    one position)."""
    from metacov_b200 import ReadBatch
    rng = np.random.default_rng(21)
    lengths = np.array([9000, 4000], np.int32)
    ps0 = np.sort(np.r_[np.full(70000, 2500), np.full(30000, 2600), rng.integers(0, 8800, 20000)])
    ps1 = np.sort(rng.integers(0, 3900, 3000))
    tid = np.r_[np.zeros(len(ps0), np.int32), np.ones(len(ps1), np.int32)]
    pos = np.r_[ps0, ps1].astype(np.int32)
    n = len(tid)
    rl = rng.integers(50, 150, n)
    rl[:5] = 3000                                    # a few far reads across the dense tiles
    b = ReadBatch(tid, pos, np.zeros(n, np.uint16), np.full(n, 30, np.uint8), np.arange(n + 1, dtype=np.uint32),
                  (rl.astype(np.uint32) << 4))
    want, off, _ = cport.depth(b, lengths, mode="diff")
    with engine_for(lengths, max_depth=0) as eng:
        eng.depth_sorted(b)
        pi = eng.pass_info()
        assert pi["max_depth_seen"] == int(want.max()) and pi["max_depth_seen"] > 65536
        for c in range(2):
            assert np.array_equal(eng.copy_depth(c), want[off[c]:off[c] + lengths[c]]), c


def test_pipelined_statistics_equal_synchronous():
    """mcov_region_stats_submit / collect: two slots in flight across depth passes, records identical to
    mcov_region_stats_run; error reporting for what cannot be completed after the fact."""
    from metacov_b200 import McovError, _capi, synth
    w = synth.c2(0.01)
    b, _ = synth.generate_host(w)
    g = w.n_contigs
    tid = np.arange(g, dtype=np.int32)
    start = np.zeros(g, np.int32)
    end = w.contig_len.astype(np.int32).copy()
    end[3] = 0                                          # a zero-length region: zeroed record
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted(b)
        want = eng.region_stats(tid, start, end).copy()
        tickets = []
        for k in range(4):
            eng.depth_sorted(b, wait=False)
            tickets.append(eng.region_stats_submit(tid, start, end, slot=k & 1))
            if len(tickets) == 2:
                got = eng.region_stats_collect(tickets.pop(0))
                assert got.tobytes() == want.tobytes(), k
        assert eng.region_stats_collect(tickets.pop(0)).tobytes() == want.tobytes()
        # a slot cannot be submitted twice, nor collected twice
        eng.depth_sorted(b, wait=False)
        t = eng.region_stats_submit(tid, start, end, slot=0)
        with pytest.raises(McovError) as ei:
            eng.region_stats_submit(tid, start, end, slot=0)
        assert ei.value.code == _capi.MCOV_ERR_STATE
        eng.region_stats_collect(t)
        with pytest.raises(McovError):
            eng.region_stats_collect(t)
        # unsorted input: the verdict travels with the slot
        perm = np.random.default_rng(1).permutation(len(b.tid))
        from metacov_b200 import ReadBatch
        off = b.cig_off.astype(np.int64)
        nc = (off[1:] - off[:-1])[perm]
        cig = np.concatenate([b.cig[off[i]:off[i + 1]] for i in perm]) if len(perm) else b.cig
        ub = ReadBatch(b.tid[perm], b.pos[perm], b.flag[perm], b.mapq[perm],
                       np.concatenate(([0], np.cumsum(nc))).astype(np.uint32), cig)
        eng.depth_sorted(ub, wait=False)
        t = eng.region_stats_submit(tid, start, end, slot=1)
        with pytest.raises(McovError) as ei:
            eng.region_stats_collect(t)
        assert ei.value.code == _capi.MCOV_ERR_UNSORTED


def test_delta_host_transport_equals_soa_path():
    """mcov_depth_sorted_delta (u16 position differences + exceptions, u8 op counts, u16 ops): the SoA rebuilt
    on the device gives the same depth as the plain columns -- short reads, sparse contigs whose gaps exceed
    16 bits (exceptions), unplaced reads at the end, unsorted input (negative differences travel faithfully
    and the pass reports MCOV_ERR_UNSORTED), batches that do not qualify."""
    from metacov_b200 import McovError, ReadBatch, _capi, synth
    from metacov_b200.engine import pack_batch_delta, packed_bytes, pack_batch
    w = synth.c2(0.01)
    b, _ = synth.generate_host(w)
    pd = pack_batch_delta(b, w.n_contigs)
    assert packed_bytes(pd) < 0.65 * packed_bytes(pack_batch(b, w.n_contigs)) and len(pd["exc_index"]) == 0
    with engine_for(w.contig_len) as eng:
        eng.depth_sorted_delta(pd)
        want, dflat, off, info = oracle_depth(b, w.contig_len)
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c]), c
        pi = eng.pass_info()
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"] and pi["sorted"] == 1
        eng.set_filter(min_mapq=30)
        with pytest.raises(McovError):
            eng.depth_sorted_delta(pd)                           # mapq required when min_mapq > 0
        eng.depth_sorted_delta(pack_batch_delta(b, w.n_contigs, with_mapq=True, pinned=True))
        want30, _, _, _ = oracle_depth(b, w.contig_len, min_mapq=30)
        assert np.array_equal(eng.copy_depth(0), want30[0])
    # sparse reads on long contigs: gaps above 65535 become exceptions; first reads of contigs far from 0
    rng = np.random.default_rng(8)
    lengths = np.array([3_000_000, 500_000, 2_000_000], np.int32)
    tid = np.repeat(np.arange(3, dtype=np.int32), [40, 5, 30])
    pos = np.concatenate([np.sort(rng.integers(100_000, l - 200, k)) for l, k in zip(lengths, (40, 5, 30))]).astype(np.int32)
    n = len(tid)
    sb = ReadBatch(tid, pos, np.zeros(n, np.uint16), np.full(n, 60, np.uint8), np.arange(n + 1, dtype=np.uint32),
                   np.full(n, 150 << 4, np.uint32))
    ps = pack_batch_delta(sb, 3)
    assert len(ps["exc_index"]) > 10
    with engine_for(lengths) as eng:
        eng.depth_sorted_delta(ps)
        wants, _, _, _ = oracle_depth(sb, lengths)
        for c in range(3):
            assert np.array_equal(eng.copy_depth(c), wants[c]), c
        # unsorted inside a contig: the negative difference is an exception, the verdict is UNSORTED
        ub = ReadBatch(tid, pos[::-1].copy(), sb.flag, sb.mapq, sb.cig_off, sb.cig)
        with pytest.raises(McovError) as ei:
            eng.depth_sorted_delta(pack_batch_delta(ub, 3))
        assert ei.value.code == _capi.MCOV_ERR_UNSORTED
    # unplaced reads at the end (fixture) and empty input
    z, fb = load_soa("fixture_soa.npz")
    with engine_for(z["lengths"]) as eng:
        eng.depth_sorted_delta(pack_batch_delta(fb, 2, pinned=True))
        wantf, _, _, _ = oracle_depth(fb, z["lengths"])
        assert np.array_equal(eng.copy_depth(1), wantf[1]) and eng.pass_info()["n_pass"] == 3350
        empty = ReadBatch(*(np.zeros(0, a.dtype) for a in (fb.tid, fb.pos, fb.flag, fb.mapq)), np.zeros(1, np.uint32), np.zeros(0, np.uint32))
        eng.depth_sorted_delta(pack_batch_delta(empty, 2))
        assert eng.pass_info()["n_pass"] == 0 and not eng.copy_depth(0).any()
    # long reads do not qualify (thousands of ops per CIGAR): the caller falls back to pack_batch
    w5 = synth.c5(0.0005)
    b5, _ = synth.generate_host(w5)
    with pytest.raises(ValueError):
        pack_batch_delta(b5, w5.n_contigs)


def test_block_transport_equals_soa_path():
    """mcov_depth_sorted_block: the transport block of the native packer (one host-to-device copy: u8 position
    differences + exceptions, flag dictionary, CIGAR dictionary + explicit ops) rebuilt on the device gives the
    depth of the plain columns -- short reads, sparse contigs (exceptions), the fixture's unplaced tail, unsorted
    input, a filter that needs mapq, pinned and pageable buffers, a corrupted header."""
    from metacov_b200 import McovError, ReadBatch, _capi, synth
    from metacov_b200.engine import pack_block
    w = synth.c2(0.01)
    b, _ = synth.generate_host(w)
    with engine_for(w.contig_len) as eng:
        blk = pack_block(b, w.n_contigs, pinned=True)
        assert blk[1] < 3.0 * len(b.tid)
        eng.depth_sorted_block(blk)
        want, dflat, off, info = oracle_depth(b, w.contig_len)
        for c, d in enumerate(full_depth(eng)):
            assert np.array_equal(d, want[c]), c
        pi = eng.pass_info()
        assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"] and pi["sorted"] == 1
        eng.depth_sorted_block(blk, wait=False)                  # deferred verdict, statistics straight after
        tid = np.arange(w.n_contigs, dtype=np.int32)
        st = eng.region_stats(tid, np.zeros_like(tid), w.contig_len)
        ref = cport.region_stats(dflat, off, w.contig_len, tid, np.zeros_like(tid), w.contig_len)
        for k in ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi"):
            assert np.array_equal(st[k], ref[k]), k
        eng.set_filter(min_mapq=30)
        with pytest.raises(McovError):
            eng.depth_sorted_block(blk)                          # packed without mapq
        eng.depth_sorted_block(pack_block(b, w.n_contigs, with_mapq=True))
        want30, _, _, _ = oracle_depth(b, w.contig_len, min_mapq=30)
        assert np.array_equal(eng.copy_depth(0), want30[0])
        bad = np.array(blk[0].numpy()[:blk[1]], copy=True)
        bad[0] ^= 0xFF                                           # magic
        with pytest.raises(McovError):
            eng.depth_sorted_block((bad, len(bad)))
        with pytest.raises(McovError):
            eng.depth_sorted_block((blk[0], blk[1] - 64))        # shorter than the header says
    # another contig table: refused
    with engine_for(w.contig_len[:-1]) as eng:
        with pytest.raises(McovError):
            eng.depth_sorted_block(blk)
    rng = np.random.default_rng(8)
    lengths = np.array([3_000_000, 500_000, 2_000_000], np.int32)
    tid = np.repeat(np.arange(3, dtype=np.int32), [40, 5, 30])
    pos = np.concatenate([np.sort(rng.integers(100_000, l - 200, k)) for l, k in zip(lengths, (40, 5, 30))]).astype(np.int32)
    n = len(tid)
    sb = ReadBatch(tid, pos, np.zeros(n, np.uint16), np.full(n, 60, np.uint8), np.arange(n + 1, dtype=np.uint32),
                   np.full(n, 150 << 4, np.uint32))
    with engine_for(lengths) as eng:
        eng.depth_sorted_block(pack_block(sb, 3))
        wants, _, _, _ = oracle_depth(sb, lengths)
        for c in range(3):
            assert np.array_equal(eng.copy_depth(c), wants[c]), c
        ub = ReadBatch(tid, pos[::-1].copy(), sb.flag, sb.mapq, sb.cig_off, sb.cig)
        with pytest.raises(McovError) as ei:
            eng.depth_sorted_block(pack_block(ub, 3))
        assert ei.value.code == _capi.MCOV_ERR_UNSORTED
    z, fb = load_soa("fixture_soa.npz")
    with engine_for(z["lengths"]) as eng:
        eng.depth_sorted_block(pack_block(fb, 2, pinned=True))
        wantf, _, _, _ = oracle_depth(fb, z["lengths"])
        assert np.array_equal(eng.copy_depth(1), wantf[1]) and eng.pass_info()["n_pass"] == 3350
        empty = ReadBatch(*(np.zeros(0, a.dtype) for a in (fb.tid, fb.pos, fb.flag, fb.mapq)), np.zeros(1, np.uint32), np.zeros(0, np.uint32))
        eng.depth_sorted_block(pack_block(empty, 2))
        assert eng.pass_info()["n_pass"] == 0 and not eng.copy_depth(0).any()


@pytest.mark.parametrize("wl,scale", [("c2", 0.01), ("c5", 0.002)])
def test_filter_switches_count_del_and_reflen0(wl, scale):
    """The two switches SURVEY.md Appendix A-4 / 8(b) ask to keep: count_del = 0 (only M = X positions count, one
    interval per run of such ops) and reflen0_as_one (a read that consumes no reference occupies `pos`, as in older
    htslib) -- every entry point against the C oracle with the same switches; the defaults are the reference's."""
    from metacov_b200 import ReadBatch, synth
    from metacov_b200.engine import pack_block
    w = synth.WORKLOADS[wl](scale)
    b, _, reflen = synth.generate_host(w, want_reflen=True)
    # a few reads whose CIGAR consumes no reference (soft clip / insertion only), kept in sorted order
    cig = b.cig.copy()
    o = b.cig_off.astype(np.int64)
    single = np.nonzero(np.diff(o) == 1)[0][::97]
    cig[o[single]] = (cig[o[single]] & ~np.uint32(15)) | np.uint32(4)
    b = ReadBatch(b.tid, b.pos, b.flag, b.mapq, b.cig_off, cig)
    n = len(b.tid)
    for sw in (dict(count_del=0), dict(reflen0_as_one=1), dict(count_del=0, reflen0_as_one=1)):
        want, dflat, off, info = oracle_depth(b, w.contig_len, **sw)
        base, _, _, _ = oracle_depth(b, w.contig_len)
        if "count_del" in sw or len(single):
            assert any(not np.array_equal(x, y) for x, y in zip(want, base)), sw   # the switch changes something here
        with engine_for(w.contig_len, **sw) as eng:
            def same(tag):
                for c, d in enumerate(full_depth(eng)):
                    assert np.array_equal(d, want[c]), (sw, tag, c)
                pi = eng.pass_info()
                assert pi["n_pass"] == info["n_pass"] and pi["aligned_bases"] == info["aligned_bases"], (sw, tag)
            eng.depth_sorted(b); same("sorted")
            eng.begin(); eng.push(b); eng.finalize(); same("push")
            if wl == "c2":
                eng.depth_sorted_block(pack_block(b, w.n_contigs)); same("block")
            # streamed in three batches (the carry rule is the same; carried reads must not count twice)
            from test_gpu_stream import push_in_batches
            rl = np.asarray(reflen).copy()
            push_in_batches(eng, b, rl, np.r_[0, n // 3, 2 * n // 3, n])
            eng.region_stats([0], [0], [10])
            same("stream")


def test_warp_statistics_window_guess_refit_and_retry():
    """k_region_stats_warp reads a small region once, with its histogram window anchored from the first 512 slots.  Regions
    whose depth later leaves that window are counted again with the right anchor (range <= 1024 values) or go to the
    CTA-per-region kernel (wider range): all three outcomes, falling and rising depth, against the oracle."""
    from metacov_b200 import ReadBatch
    lengths = np.array([6400, 6400, 6400, 300], np.int32)
    tid, pos = [], []
    for c, (d0, d1) in enumerate(((6, 1), (8, 1), (1, 7))):          # reads per position in the first / second half
        p = np.r_[np.repeat(np.arange(0, 3000), d0), np.repeat(np.arange(3000, 6200), d1)]
        tid += [c] * len(p); pos += p.tolist()
    tid += [3] * 40; pos += sorted(np.random.default_rng(3).integers(0, 200, 40).tolist())
    n = len(tid)
    b = ReadBatch(np.array(tid, np.int32), np.array(pos, np.int32), np.zeros(n, np.uint16), np.full(n, 30, np.uint8),
                  np.arange(n + 1, dtype=np.uint32), np.full(n, 150 << 4, np.uint32))
    want, off, _ = cport.depth(b, lengths, mode="diff")
    t = [0, 1, 2, 0, 1, 2, 3, 0, 2]
    a = [1000, 1000, 1000, 0, 0, 0, 0, 2990, 3500]
    e = [5000, 5000, 5000, 6400, 6400, 6400, 300, 3003, 6700]
    with engine_for(lengths) as eng:
        eng.depth_sorted(b)
        assert np.array_equal(eng.copy_depth(0), want[off[0]:off[0] + 6400])
        got = eng.region_stats(t, a, e)
        ref = cport.region_stats(want, off, lengths, t, a, e)
        for k in ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi", "n_ge1"):
            assert np.array_equal(got[k], ref[k]), (k, got[k], ref[k])
        # the depth really does what the cases need: a fall of ~750 (refit), of ~1050 (retry), a rise of ~900 (refit)
        d0 = want[off[0] + 1000:off[0] + 5000]; d1 = want[off[1] + 1000:off[1] + 5000]; d2 = want[off[2] + 1000:off[2] + 5000]
        assert d0[:512].min() - d0.min() > 256 and d0.max() - d0.min() < 1024
        assert d1.max() - d1.min() >= 1024
        assert d2.max() - d2[:512].min() > 768 and d2.max() - d2.min() < 1024


def test_block_unpack_column_by_column():
    """mcov_block_unpack: the columns k_block_index / reduce / prefix / expand rebuild from a transport block are the
    columns it was packed from -- contig starts on, just before and just after the 2 048-read chunk borders, runs of
    empty contigs, an unplaced tail, batches of 0 / 1 / 2 047 / 2 048 / 2 049 reads, position exceptions and escapes in
    every chunk, explicit ops in the u16 and (an op of 4 096 or more) the u32 form, many small contigs (C3-like)."""
    from metacov_b200 import ReadBatch, synth
    from metacov_b200.engine import pack_block
    rng = np.random.default_rng(11)

    def check(b, n_contigs, with_mapq=False, pinned=False):
        blk = pack_block(b, n_contigs, with_mapq=with_mapq, pinned=pinned)
        with engine_for(np.full(n_contigs, 6_000_000, np.int32)) as eng:
            u = eng.block_unpack(blk)
        tid = np.asarray(b.tid)
        valid = (tid >= 0) & (tid < n_contigs)
        assert np.array_equal(u["tid"][valid], tid[valid]) and np.all(u["tid"][~valid] == -1)
        assert np.array_equal(u["pos"], np.asarray(b.pos)) and np.array_equal(u["flag"], np.asarray(b.flag))
        assert np.array_equal(u["cig_off"], np.asarray(b.cig_off)) and np.array_equal(u["cig"], np.asarray(b.cig))
        assert np.array_equal(u["mapq"], np.asarray(b.mapq)) if with_mapq else np.all(u["mapq"] == 0xff)
        return blk

    def batch(tid, wide=False, many_flags=False, big_gaps=False):
        n = len(tid)
        pos = np.zeros(n, np.int64)
        for c in np.unique(tid):
            m = tid == c
            gaps = rng.integers(0, 12, int(m.sum()))
            if big_gaps:
                gaps[rng.random(len(gaps)) < 0.02] = rng.integers(256, 40_000)
            pos[m] = np.cumsum(gaps) + rng.integers(0, 1000)
        flag = (rng.integers(0, 4096, n) if many_flags else rng.choice(np.array([99, 147, 83, 163, 1024 + 99]), n)).astype(np.uint16)
        n_op = rng.choice(np.array([1, 1, 1, 1, 2, 3, 5, 0]), n)
        off = np.concatenate(([0], np.cumsum(n_op))).astype(np.uint32)
        ln = rng.integers(1, 150, int(off[-1])).astype(np.uint32)
        ln[off[:-1][n_op == 1]] = 150                           # the common single-op CIGAR: a dictionary entry
        if wide and len(ln):
            ln[rng.integers(0, len(ln))] = 5000
        cig = (ln << 4) | rng.choice(np.array([0, 1, 2, 4, 7, 8], np.uint32), len(ln)).astype(np.uint32)
        return ReadBatch(tid.astype(np.int32), pos.astype(np.int32), flag, rng.integers(0, 61, n).astype(np.uint8), off, cig)

    # contig starts around the chunk borders; empty contigs in runs; an unplaced tail
    sizes = [2048, 0, 0, 2047, 1, 0, 2049, 4095, 1, 1, 0, 0, 0, 4096, 5, 0]
    tid = np.repeat(np.arange(len(sizes)), sizes)
    tid = np.r_[tid, np.full(3000, -1)]
    for kw in ({}, {"big_gaps": True}, {"many_flags": True, "big_gaps": True}, {"wide": True}):
        b = batch(tid, **kw)
        blk = check(b, len(sizes), with_mapq=bool(kw.get("wide")), pinned=bool(kw.get("big_gaps")))
    for n in (0, 1, 2047, 2048, 2049, 4096, 4097):
        check(batch(np.zeros(n, np.int64)), 1)
        check(batch(np.sort(rng.integers(0, 7, n))), 9, with_mapq=True)
        check(batch(np.full(n, -1)), 3)                            # nothing but unplaced reads
    # many small contigs (some empty), like C3
    check(batch(np.sort(rng.integers(0, 30_000, 60_000)), big_gaps=True), 30_000)
    w = synth.c3(0.002)
    b3, _ = synth.generate_host(w)
    check(b3, w.n_contigs)
    w = synth.c2(0.01)
    b2, _ = synth.generate_host(w)
    check(b2, w.n_contigs, pinned=True)


@pytest.mark.parametrize("seed", range(int(os.environ.get("MCOV_BLOCK_FUZZ", "6"))))
def test_block_unpack_random_batches(seed):
    """Random batches of tens of thousands of reads (dozens of 2 048-read chunks) through mcov_pack_block ->
    mcov_block_unpack: random contig structure (runs of empty contigs, contigs of one read, an unplaced tail), gap
    distributions that favour the nibble or the wide form, position exceptions, escapes, CIGARs of 0..9 ops with the
    occasional op of 4 096 and more.  MCOV_BLOCK_FUZZ=N runs N seeds (the builder ran 300: profiles/r02_fuzz.txt)."""
    from metacov_b200 import ReadBatch
    from metacov_b200.engine import pack_block
    rng = np.random.default_rng(50_000 + seed)
    n = int(rng.integers(3000, 120_000))
    n_contigs = int(rng.choice([1, 3, 40, 2000, 30_000]))
    # reads per contig: skewed, many empty
    w = rng.random(n_contigs) ** int(rng.integers(1, 6))
    if n_contigs > 10:
        w[rng.random(n_contigs) < 0.3] = 0
    if w.sum() == 0:
        w[0] = 1
    tid = np.sort(rng.choice(n_contigs, n, p=w / w.sum())).astype(np.int64)
    n_un = int(rng.integers(0, 3000)) if seed % 3 else 0
    tid = np.r_[tid, np.full(n_un, -1)]
    n = len(tid)
    mean_gap = float(rng.choice([1.5, 5, 12, 60, 400]))
    gaps = rng.geometric(1.0 / (1.0 + mean_gap), n) - 1
    gaps[rng.random(n) < float(rng.choice([0, 0.001, 0.02]))] = rng.integers(256, 3_000_000)
    pos = np.zeros(n, np.int64)
    first = np.r_[True, tid[1:] != tid[:-1]]
    seg = np.cumsum(first) - 1
    start_of = np.flatnonzero(first)
    csum = np.cumsum(gaps)
    pos = csum - csum[start_of][seg] + rng.integers(0, 5000, len(start_of))[seg]
    if seed % 5 == 4:                                      # a few reads out of order inside their contig: negative differences
        k = rng.integers(1, n, 20)
        pos[k] = np.maximum(pos[k] - rng.integers(1, 400, 20), 0)
    nf = int(rng.choice([3, 12, 400, 5000]))
    flag = rng.choice(rng.integers(0, 65536, nf), n).astype(np.uint16)
    n_op = rng.choice(np.array([1, 1, 1, 1, 1, 2, 3, 3, 5, 9, 0]), n)
    off = np.concatenate(([0], np.cumsum(n_op))).astype(np.uint32)
    ln = rng.integers(1, 151, int(off[-1])).astype(np.uint32)
    single = off[:-1][n_op == 1]
    ln[single] = rng.choice(np.array([150, 150, 150, 100, 75], np.uint32), len(single))
    if seed % 4 == 1 and len(ln):
        ln[rng.integers(0, len(ln), 3)] = rng.integers(4096, 100_000, 3)
    cig = (ln << 4) | rng.choice(np.array([0, 0, 0, 1, 2, 4, 7, 8], np.uint32), len(ln)).astype(np.uint32)
    b = ReadBatch(tid.astype(np.int32), pos.astype(np.int32), flag, rng.integers(0, 61, n).astype(np.uint8), off, cig)
    with_mapq = bool(seed % 2)
    blk = pack_block(b, n_contigs, with_mapq=with_mapq, pinned=bool(seed % 3 == 0))
    with engine_for(np.full(n_contigs, 2_000_000_000 // max(n_contigs, 1) + 1000, np.int32)) as eng:
        u = eng.block_unpack(blk)
    ok = b.tid >= 0
    assert np.array_equal(u["tid"][ok], b.tid[ok]) and np.all(u["tid"][~ok] == -1)
    assert np.array_equal(u["pos"], b.pos) and np.array_equal(u["flag"], b.flag)
    assert np.array_equal(u["cig_off"], b.cig_off) and np.array_equal(u["cig"], b.cig)
    assert np.array_equal(u["mapq"], b.mapq) if with_mapq else np.all(u["mapq"] == 0xff)
