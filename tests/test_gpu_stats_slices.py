"""Large-region statistics under the cost-balanced slicing of k_stats_stream.

The plan cuts the large regions into one slice per CTA by cost and keeps whole regions together where it can; a tile
shared by two pieces that follow each other in slot order is staged once and its slots are counted into the piece
each belongs to.  Every record here is compared with the statistics of the depth copied back to the host, on the
first call of a plan (no tile histograms), on a call that uses the histograms counted for the plan, and on a call
whose plan differs from the one the histograms were counted for."""
import numpy as np
import pytest

from oracle import cport
from test_gpu_tile_hist import border, make_reads, same

pytestmark = pytest.mark.gpu

LENGTHS = np.array([200_000, 600_000, 90_017], np.int32)


def host_stats(eng, lengths, reg):
    """Records of the regions from the depth as copied back to the host (the C oracle's statistics)."""
    d = np.concatenate([eng.copy_depth(c) for c in range(len(lengths))])
    off = np.r_[0, np.cumsum(lengths.astype(np.int64))[:-1]]
    return cport.region_stats(d, off, lengths, *reg)


def check(got, ref):
    for k in ("sum", "sumsq", "iq_sum", "min", "max", "med_lo", "med_hi", "n_ge1", "n_geN"):
        assert np.array_equal(got[k], ref[k]), k


def three_calls(eng, b, reg):
    """First call of the plan (its pass counted no histograms), then two calls after passes that counted them."""
    eng.depth_sorted(b)
    first = eng.region_stats(*reg).copy()
    out = [first]
    for _ in range(2):
        eng.depth_sorted(b)
        out.append(eng.region_stats(*reg).copy())
    return out


def adjacent(eng, c, L, n, size):
    """n regions of `size` slots one after the other from contig c's start, their borders off the tile borders."""
    s = np.arange(n, dtype=np.int64) * size + 7
    keep = s + size <= L
    return [(c, int(a), int(a + size)) for a in s[keep]]


@pytest.mark.parametrize("size", [9_001, 10_007, 24_580, 50_000])
def test_adjacent_regions_share_border_tiles(size):
    """Consecutive large regions in slot order: several land in one slice, and the tile holding one region's tail and
    the next one's head is staged once.  A deep pile in a border tile and in the tiles around it takes their
    histograms out of the window (anchor 0xFFFF)."""
    from metacov_b200 import CoverageEngine
    with CoverageEngine(LENGTHS) as eng:
        p = int(7 + 3 * size - 40)                              # the border between the third and fourth region
        b = make_reads(LENGTHS, 60_000, 21, [(0, p, 400, 150), (0, border(eng, 0, 40) + 100, 300, 150)])
        rows = [r for c in range(len(LENGTHS)) for r in adjacent(eng, c, int(LENGTHS[c]), 100, size)]
        reg = tuple(np.array(x, np.int32) for x in zip(*rows))
        recs = three_calls(eng, b, reg)
        ref = host_stats(eng, LENGTHS, reg)
        for r in recs:
            check(r, ref)
        assert same(recs[0], recs[1]) and same(recs[1], recs[2])


def test_split_overlap_pad_and_order():
    """Overlapping large regions, a region reaching past its contig's end, a whole contig of 600 k slots, small regions
    among them, all given out of slot order."""
    from metacov_b200 import CoverageEngine
    with CoverageEngine(LENGTHS) as eng:
        b = make_reads(LENGTHS, 80_000, 23, [(1, 300_000, 500, 150)])
        L2 = int(LENGTHS[2])
        rows = [(1, 0, int(LENGTHS[1])),
                (0, 0, 30_000), (0, 15_000, 45_000), (0, 20_000, 180_000),   # overlapping
                (2, L2 - 20_000, L2 + 500),                       # padding past the end
                (2, 0, 9_000), (2, 100, 4_100), (0, 190_000, 200_000)]
        rows += adjacent(eng, 2, L2 - 20_000, 6, 11_111)
        rows = rows[::-1]                                         # out of slot order
        reg = tuple(np.array(x, np.int32) for x in zip(*rows))
        recs = three_calls(eng, b, reg)
        ref = host_stats(eng, LENGTHS, reg)
        for r in recs:
            check(r, ref)
        assert same(recs[0], recs[1]) and same(recs[1], recs[2])


def test_plan_differs_from_histograms():
    """Histograms counted for one plan, statistics of another: the tiles of the new plan are read from the depth."""
    from metacov_b200 import CoverageEngine
    with CoverageEngine(LENGTHS) as eng:
        b = make_reads(LENGTHS, 60_000, 25, [(1, 100_000, 300, 150)])
        reg_a = tuple(np.array(x, np.int32) for x in zip(*adjacent(eng, 1, int(LENGTHS[1]), 60, 10_007)))
        rows_b = [(c, int(s), int(s + 30_011)) for c in (0, 1) for s in range(3_001, int(LENGTHS[c]) - 30_011, 30_011)]
        reg_b = tuple(np.array(x, np.int32) for x in zip(*rows_b))
        three_calls(eng, b, reg_a)                                # the last pass counted histograms for plan a
        got = eng.region_stats(*reg_b).copy()
        check(got, host_stats(eng, LENGTHS, reg_b))
        eng.depth_sorted(b)
        got_b = eng.region_stats(*reg_b).copy()                   # now with the histograms counted for plan b
        assert same(got, got_b)


@pytest.mark.parametrize("rows", [
    [(0, 0, 2_300_000), (1, 7, 60_001)],                    # histograms counted: a region of 2 M slots, 300 k of padding
    [(0, 100_000, 1_000_000), (1, 7, 60_001)],              # under half of the tiles covered: plain slot costs
], ids=["histograms", "slots"])
def test_region_split_between_slices(rows):
    """A region costing several slices is cut between CTAs, merged in global memory and walked by the CTA whose piece
    arrives last; the plan itself reports the split."""
    from metacov_b200 import CoverageEngine
    lengths = np.array([2_000_000, 60_001], np.int32)
    with CoverageEngine(lengths) as eng:
        b = make_reads(lengths, 150_000, 27, [(0, 1_234_567, 400, 150)])
        reg = tuple(np.array(x, np.int32) for x in zip(*rows))
        recs = three_calls(eng, b, reg)
        ctas, splits = eng.region_plan_info()
        assert splits >= 1 and ctas > 2
        d = np.concatenate([eng.copy_depth(c) for c in range(len(lengths))])
        ref = cport.region_stats(d, np.r_[0, np.cumsum(lengths.astype(np.int64))[:-1]], lengths, *reg)
        for r in recs:
            check(r, ref)
        assert same(recs[0], recs[1]) and same(recs[1], recs[2])
