"""Statistics of large regions from the tile kernel's per-tile depth histograms.

A one-shot fused pass that follows a statistics call with large regions leaves a depth histogram of every tile, and
the next statistics call counts the tiles that lie wholly inside a region from them instead of from the depth.  The
reference for every case here is the same reads' records with no histogram to trust: the first statistics call (which
builds the region plan after a pass that wrote none) and the push path (begin / push / finalize).  Records must agree
byte for byte, and with the C oracle."""
import numpy as np
import pytest

from oracle import cport

pytestmark = pytest.mark.gpu

TILE = 2048


def make_reads(lengths, n, seed, piles=()):
    """Sorted 150 bp reads spread over the contigs, plus `piles` = [(tid, pos, count, span)] of stacked reads."""
    from metacov_b200 import ReadBatch
    rng = np.random.default_rng(seed)
    tid = rng.integers(0, len(lengths), n)
    span = np.full(n, 150)
    pos = (rng.random(n) * (lengths[tid] - 150)).astype(np.int64)
    for t, p, k, s in piles:
        tid = np.r_[tid, np.full(k, t)]
        pos = np.r_[pos, np.full(k, p)]
        span = np.r_[span, np.full(k, s)]
    o = np.lexsort((pos, tid))
    tid, pos, span = tid[o].astype(np.int32), pos[o].astype(np.int32), span[o]
    m = len(tid)
    return ReadBatch(tid, pos, np.zeros(m, np.uint16), np.full(m, 30, np.uint8), np.arange(m + 1, dtype=np.uint32),
                     span.astype(np.uint32) << 4)


def border(eng, c, k):
    """Contig position of the k-th tile border inside contig c."""
    return (-eng.contig_offset(c)) % TILE + k * TILE


def regions(eng, lengths):
    """Whole contigs; regions starting / ending on a tile border, one slot inside, one slot outside and mid-tile; a
    region reaching past its contig's end; overlapping regions; and small regions among them."""
    rows = []
    for c, L in enumerate(lengths):
        L = int(L)
        rows.append((c, 0, L))
        b2, b9 = border(eng, c, 2), border(eng, c, 9)
        if b9 + 700 < L:
            for ds in (0, 1, -1, 1000):
                for de in (0, 1, -1, 700):
                    rows.append((c, b2 + ds, b9 + de))
            rows.append((c, b9, b9 + 8000))                            # small, starts on a border
        rows.append((c, L - 3 * TILE - 5, L + 500))                   # padding past the end
        rows.append((c, min(b2 + 10, L), L))                           # overlaps the ones above
        rows.append((c, 100, 4100))                                    # small
    t, s, e = (np.array(x, np.int32) for x in zip(*rows))
    return t, s, e


def stats(eng, reg):
    return eng.region_stats(*reg).copy()


def same(a, b):
    return a.tobytes() == b.tobytes()


def oracle(b, lengths, reg, **filt):
    d, off, _ = cport.depth(b, lengths, filt=cport.default_filter(**filt) if filt else None, mode="diff")
    return cport.region_stats(d, off, lengths, *reg)


def check_oracle(got, ref):
    for k in ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi", "n_ge1", "n_geN"):
        assert np.array_equal(got[k], ref[k]), k


def first_cached_push(eng, b, reg):
    """Records of the first statistics call, of the cached-plan call after a second pass, and of the push path."""
    eng.depth_sorted(b)
    first = stats(eng, reg)
    eng.depth_sorted(b)
    cached = stats(eng, reg)
    eng.begin(); eng.push(b); eng.finalize()
    push = stats(eng, reg)
    return first, cached, push


@pytest.mark.parametrize("piles", [(), ((0, 30000, 400, 150), (1, 5000, 150, 1800))], ids=["plain", "deep_piles"])
def test_tile_histograms_match_depth(piles):
    """Region borders on, next to and between tile borders, padding, overlaps, small regions; the deep piles push
    tiles out of the histogram window."""
    from metacov_b200 import CoverageEngine
    lengths = np.array([50000, 61234, 40001, 9000], np.int32)
    b = make_reads(lengths, 60000, 5, piles)
    with CoverageEngine(lengths) as eng:
        reg = regions(eng, lengths)
        first, cached, push = first_cached_push(eng, b, reg)
        assert same(first, cached) and same(first, push)
        check_oracle(cached, oracle(b, lengths, reg))


def test_tile_histograms_overflow_to_radix():
    """max_depth raised and a pile of 9 000: the region's record is flagged by the counting histogram and redone by
    the radix path, with and without tile histograms."""
    from metacov_b200 import CoverageEngine
    lengths = np.array([50000, 30000], np.int32)
    b = make_reads(lengths, 20000, 7, [(0, 20000, 9000, 150)])
    with CoverageEngine(lengths, filt={"max_depth": 100000}) as eng:
        reg = regions(eng, lengths)
        first, cached, push = first_cached_push(eng, b, reg)
        assert first["max"].max() >= 8191
        assert same(first, cached) and same(first, push)
        check_oracle(cached, oracle(b, lengths, reg, max_depth=100000))


def test_tile_histograms_with_cap_replay():
    """htslib's cap fires on contig 0 (a pile of 400 with max_depth = 100): the replayed contig's tiles lose their
    histograms; whole-contig regions and sub-regions (per-region replay) match the first call."""
    from metacov_b200 import CoverageEngine
    lengths = np.array([50000, 30000, 20000], np.int32)
    b = make_reads(lengths, 20000, 9, [(0, 20000, 400, 150)])
    with CoverageEngine(lengths, filt={"max_depth": 100}) as eng:
        reg = regions(eng, lengths)
        eng.depth_sorted(b)
        first = stats(eng, reg)
        assert eng.pass_info()["cap_contigs"] == 1
        eng.depth_sorted(b)
        cached = stats(eng, reg)
        assert same(first, cached)
        # the contigs where the cap does not fire also agree with the push path
        eng.begin(); eng.push(b); eng.finalize()
        push = stats(eng, reg)
        keep = reg[0] != 0
        assert same(cached[keep], push[keep])


def test_tile_histograms_async_block_and_region_change():
    """Asynchronous pass + submit / collect, the transport-block entry point, and a region set that changes between
    two passes."""
    from metacov_b200 import CoverageEngine
    from metacov_b200.engine import pack_block
    lengths = np.array([50000, 61234, 40001], np.int32)
    b = make_reads(lengths, 40000, 11, [(2, 9000, 300, 150)])
    with CoverageEngine(lengths) as eng:
        reg = regions(eng, lengths)
        eng.begin(); eng.push(b); eng.finalize()
        ref = stats(eng, reg)
        eng.depth_sorted(b, wait=False)
        assert same(eng.region_stats_collect(eng.region_stats_submit(*reg, slot=0)), ref)
        for _ in range(2):
            eng.depth_sorted(b, wait=False)
            assert same(eng.region_stats_collect(eng.region_stats_submit(*reg, slot=1)), ref)
        blk = pack_block(b, len(lengths))
        for _ in range(2):
            eng.depth_sorted_block(blk)
            assert same(stats(eng, reg), ref)
        # a new region set after a pass that wrote histograms for the old one
        reg2 = (np.array([0, 1, 2], np.int32), np.array([777, 2048, 0], np.int32), np.array([45000, 61234, 33333], np.int32))
        eng.begin(); eng.push(b); eng.finalize()
        ref2 = stats(eng, reg2)
        eng.depth_sorted(b)
        stats(eng, reg)
        eng.depth_sorted(b)
        assert same(stats(eng, reg2), ref2)
        check_oracle(ref2, oracle(b, lengths, reg2))


def test_tile_histograms_not_trusted_after_stream():
    """A streamed pass after a one-shot pass that wrote histograms: the statistics read the streamed depth."""
    from metacov_b200 import CoverageEngine
    lengths = np.array([50000, 61234], np.int32)
    b1 = make_reads(lengths, 30000, 13)
    b2 = make_reads(lengths, 30000, 14, [(1, 40000, 200, 150)])
    with CoverageEngine(lengths) as eng:
        reg = regions(eng, lengths)
        eng.depth_sorted(b1)
        stats(eng, reg)
        eng.depth_sorted(b1)
        stats(eng, reg)
        eng.stream_begin()
        eng.stream_push(b2, last=True)
        streamed = stats(eng, reg)
        check_oracle(streamed, oracle(b2, lengths, reg))
        eng.depth_sorted(b1)
        eng.begin(); eng.push(b2); eng.finalize()
        assert same(stats(eng, reg), streamed)


def test_tile_histograms_cap_inside_window():
    """The cap fires where the uncapped depth stays inside the histogram window (mean depth 30, a pile of 50 with
    max_depth = 45): only the marking of the replayed contig's tiles keeps their histograms out of the statistics."""
    from metacov_b200 import CoverageEngine
    lengths = np.array([50000, 50000], np.int32)
    b = make_reads(lengths, 20000, 17, [(0, 20000, 50, 150)])
    with CoverageEngine(lengths, filt={"max_depth": 45}) as eng:
        reg = (np.array([0, 1], np.int32), np.zeros(2, np.int32), lengths.copy())
        eng.depth_sorted(b)
        first = stats(eng, reg)
        assert eng.pass_info()["cap_contigs"] >= 1
        eng.depth_sorted(b)
        assert same(stats(eng, reg), first)
        # the capped depth differs from the uncapped one the tile kernel counted
        eng.set_filter(max_depth=0)
        eng.depth_sorted(b)
        assert not same(stats(eng, reg)[:1], first[:1])


def test_tile_histograms_route_and_resets():
    """The histogram route is taken: a write into the bound depth store after a pass that counted histograms (which
    the caller must not do) does not reach a whole-contig record, but does reach it once the store has been handed
    out by mcov_depth_ptr.  A count_del = 0 pass after one that counted histograms is read from its depth."""
    import torch
    from metacov_b200 import CoverageEngine, ReadBatch
    lengths = np.array([50000, 50000], np.int32)
    b = make_reads(lengths, 20000, 19)
    with CoverageEngine(lengths) as eng:
        buf = torch.zeros(eng.n_slots, dtype=torch.int32, device="cuda")
        eng.bind_depth(buf)
        reg = (np.array([0, 1], np.int32), np.zeros(2, np.int32), lengths.copy())
        eng.depth_sorted(b)
        ref = stats(eng, reg)
        eng.depth_sorted(b)
        slot = eng.contig_offset(0) + border(eng, 0, 5) + 100          # inside a tile wholly inside contig 0
        buf[slot] += 1000
        torch.cuda.synchronize()
        assert same(stats(eng, reg), ref)                              # counted from the tile's histogram
        assert eng.depth_ptr()
        got = stats(eng, reg)
        assert got["max"][0] >= 1000 and same(got[1:], ref[1:])
    # deletions: count_del = 1 counts them, count_del = 0 does not
    n = len(b.tid)
    ops = np.stack([np.full(n, 60 << 4), np.full(n, (20 << 4) | 2), np.full(n, 70 << 4)], axis=1).astype(np.uint32).ravel()
    bd = ReadBatch(b.tid, b.pos, b.flag, b.mapq, (np.arange(n + 1) * 3).astype(np.uint32), ops)
    with CoverageEngine(lengths) as eng:
        reg = (np.array([0, 1], np.int32), np.zeros(2, np.int32), lengths.copy())
        eng.depth_sorted(bd)
        with_del = stats(eng, reg)
        eng.depth_sorted(bd)
        eng.set_filter(count_del=False)
        eng.depth_sorted(bd)
        no_del = stats(eng, reg)
        eng.begin(); eng.push(bd); eng.finalize()
        assert same(stats(eng, reg), no_del) and not same(no_del, with_del)
        check_oracle(no_del, oracle(bd, lengths, reg, count_del=0))
