"""Region statistics, histogram merges, window means and run export on depth written straight into a bound store.

Every other test reaches the statistics kernels through depth made from reads: smooth, at most 8000, and 0 in every
slot outside a contig.  Here the test owns the depth store (``bind_depth`` + ``depth_ptr``) and writes exactly the
depth it wants: ties everywhere, value ranges of exactly 1024 and 1025 bins, steps that defeat the warp kernel's
window anchor, bands at and past the overflow bin, pieces of one region with disjoint ranges.  Every slot outside
``[off[c], off[c] + len[c])`` holds a poison value that no region may see: either >= 10^9, 7777, or one more than the
depth next to it, so that a slot read too many lands in the exact bins and changes the record.

The reference is ``ref_region_stats``: exact value counts of the region's slots plus its padding zeros in bin 0, so
it costs O(slots) whatever the padding (a region [L - 10, 2^31 - 1) of a short contig is answered at once).  The CPU
test checks it against the C oracle and against a plain sort of the materialised region."""
import numpy as np
import pytest

from oracle import cport

STATS_DTYPE = cport.ORC_STATS_DTYPE            # the layout of mcov_region_stats
FIELDS = ("sum", "sumsq", "iq_sum", "n_ge1", "n_geN", "min", "max", "med_lo", "med_hi", "reserved", "flags")
OVERFLOW = 8191                                # first depth of the counting histogram's overflow bin
HUGE = 2 ** 31 - 1
BREADTHS = (0, 1, 2, 1024, 8191)

# ---------------------------------------------------------------------------------------------------------------------
# reference


def _value_counts(x):
    """Distinct values of x (ascending) and their counts, both int64."""
    if len(x) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    lo, hi = int(x.min()), int(x.max())
    if hi - lo <= 4 * len(x) + 4096:
        bc = np.bincount((x - lo).astype(np.int64))
        nz = np.nonzero(bc)[0]
        return nz.astype(np.int64) + lo, bc[nz].astype(np.int64)
    v, c = np.unique(x, return_counts=True)
    return v.astype(np.int64), c.astype(np.int64)


def ref_region_stats(d, off, lengths, tid, start, end, breadths=(1,), plain_max=0):
    """{breadth_n: records} of the regions (tid, start, end) over the store d, from exact value counts.  Positions
    past the contig's end are depth 0.  Regions of at most `plain_max` positions are also checked against a sort of
    the materialised region."""
    g = len(tid)
    out = {bn: np.zeros(g, STATS_DTYPE) for bn in breadths}
    for i in range(g):
        c, a, b = int(tid[i]), int(start[i]), int(end[i])
        n = b - a
        if n <= 0:
            continue                                         # an all-zero record
        L = int(lengths[c])
        x = d[int(off[c]) + min(a, L): int(off[c]) + min(b, L)]
        vals, cnt = _value_counts(x)
        pad = n - len(x)
        if pad:
            if len(vals) and vals[0] == 0:
                cnt[0] += pad
            else:
                vals, cnt = np.r_[np.int64(0), vals], np.r_[np.int64(pad), cnt]
        cum = np.cumsum(cnt)
        k1, k2 = n // 4, n - n // 4
        inside = np.clip(np.minimum(cum, k2) - np.maximum(cum - cnt, k1), 0, None)
        rec = dict(sum=int((vals * cnt).sum()),
                   sumsq=int((vals.astype(np.uint64) ** 2 * cnt.astype(np.uint64)).sum()),
                   iq_sum=int((inside * vals).sum()),
                   n_ge1=n - (int(cnt[0]) if vals[0] == 0 else 0),
                   min=int(vals[0]), max=int(vals[-1]),
                   med_lo=int(vals[np.searchsorted(cum, (n - 1) // 2, side="right")]),
                   med_hi=int(vals[np.searchsorted(cum, n // 2, side="right")]),
                   reserved=0, flags=1 | (2 if vals[-1] >= OVERFLOW else 0))
        if n <= plain_max:
            _check_plain(x, n, rec, breadths, cnt, vals)
        for bn in breadths:
            r = out[bn][i]
            for k, v in rec.items():
                r[k] = v
            r["n_geN"] = int(cnt[vals >= bn].sum())
    return out


def _check_plain(x, n, rec, breadths, cnt, vals):
    z = np.zeros(n, np.int64)
    z[:len(x)] = x
    s = np.sort(z)
    plain = dict(sum=int(s.sum()), sumsq=int((s.astype(np.uint64) ** 2).sum()), iq_sum=int(s[n // 4: n - n // 4].sum()),
                 n_ge1=int((s >= 1).sum()), min=int(s[0]), max=int(s[-1]), med_lo=int(s[(n - 1) // 2]),
                 med_hi=int(s[n // 2]))
    for k, v in plain.items():
        assert rec[k] == v, (k, rec[k], v)
    for bn in breadths:
        assert int(cnt[vals >= bn].sum()) == int((s >= bn).sum())


# ---------------------------------------------------------------------------------------------------------------------
# depth generators (per contig, seeded)

EXACT_GENS = ("const", "u1", "u3", "u1023", "u1024", "u1025", "u8190", "walk", "spikes", "band_exact", "slices",
              "anchor_up", "anchor_down", "distinct1024", "distinct1025")
OVERFLOW_GENS = ("band_8191", "band_big", "spikes_big")


def gen_depth(kind, L, rng):
    """int32[L] depth of one contig.  Every value stays in [0, 2^20]."""
    if L == 0:
        return np.zeros(0, np.int32)
    if kind == "const":
        x = np.full(L, rng.integers(0, 3001))
    elif kind[0] == "u":                                      # i.i.d. uniform over [0, K]
        x = rng.integers(0, int(kind[1:]) + 1, L)
    elif kind == "walk":
        x = np.clip(1500 + np.cumsum(rng.integers(-4, 5, L)), 0, 3000)
    elif kind in ("spikes", "spikes_big"):                    # mostly 0, rare spikes
        x = np.zeros(L, np.int64)
        k = max(1, L // 1000)
        x[rng.integers(0, L, k)] = rng.integers(1, OVERFLOW if kind == "spikes" else 2 ** 20 + 1, k)
    elif kind == "anchor_up":           # the first 512 slots anchor the warp's window low; the rest lies above it
        x = rng.integers(900, 1101, L)
        x[:512] = rng.integers(100, 111, min(L, 512))
    elif kind == "anchor_down":         # ... anchored above 256, the rest lies below the window
        x = rng.integers(300, 401, L)
        x[:512] = rng.integers(900, 1001, min(L, 512))
    elif kind in ("distinct1024", "distinct1025"):            # exactly 1024 / 1025 distinct values, one range
        k = int(kind[-4:])
        v0 = int(rng.integers(1, 5000))
        x = rng.integers(v0, v0 + k, L)
        x[rng.permutation(L)[:min(L, k)]] = rng.permutation(np.arange(v0, v0 + k))[:min(L, k)]
        x[rng.integers(0, L)], x[rng.integers(0, L)] = v0, v0 + k - 1
    elif kind == "band_exact":
        x = rng.integers(7000, OVERFLOW, L)
    elif kind == "band_8191":
        x = rng.integers(7000, OVERFLOW + 1, L)
    elif kind == "band_big":
        x = rng.integers(0, 2 ** 20 + 1, L)
    elif kind == "slices":              # long stretches of 0..3 and of 6000..8190: pieces with disjoint ranges
        x = np.empty(L, np.int64)
        p, hi = 0, bool(rng.integers(0, 2))
        while p < L:
            q = min(L, p + int(rng.integers(1000, 60000)))
            x[p:q] = rng.integers(6000, OVERFLOW, q - p) if hi else rng.integers(0, 4, q - p)
            p, hi = q, not hi
    elif kind == "borders":             # runs that end on and next to multiples of 8192 slots, and runs across them
        cuts = sorted({k * 8192 + e for k in (1, 2, 3, 5, 8) for e in (-1, 0, 1)} | {0, L})
        cuts = [q for q in cuts if 0 <= q <= L]
        x = np.empty(L, np.int64)
        prev = -1
        for p, q in zip(cuts[:-1], cuts[1:]):
            v = int(rng.integers(0, 40))
            v = v + 1 if v == prev else v
            x[p:q], prev = v, v
    elif kind == "every":               # changes at every slot
        x = np.arange(L) % 977 + rng.integers(0, 2)
    else:
        raise ValueError(kind)
    return x.astype(np.int32)


# the store: (length, generator); "rot" contigs take a different generator of the fill's pool on every fill
CONTIGS = (
    (5_000_000, "rot"), (0, "rot"), (1, "rot"), (2, "rot"), (3, "rot"), (5, "rot"), (1_500_000, "rot"), (0, "rot"),
    (4000, "anchor_up"), (4000, "anchor_down"), (3000, "distinct1024"), (3000, "distinct1025"), (9000, "rot"),
    (1_500_000, "slices"), (20000, "rot"), (33333, "rot"), (80000, "borders"), (50000, "every"), (40000, "const"),
    (600_000, "rot"), (0, "rot"), (7, "rot"), (12000, "rot"), (2999, "rot"))
LENGTHS = np.array([c[0] for c in CONTIGS], np.int32)


def make_store(lengths, kinds, off, seed, pool, poison):
    """Depth of every contig, and poison in every other slot: 'big' (>= 10^9), 'mid' (7777) or 'near' (one more than
    the depth next to the gap, at most 8190)."""
    rng = np.random.default_rng(seed)
    d = np.empty(int(off[-1]), np.int32)
    for c, L in enumerate(lengths):
        kind = kinds[c] if kinds[c] != "rot" else pool[(5 * c + seed) % len(pool)]
        d[off[c]:off[c] + L] = gen_depth(kind, int(L), rng)
    for c, L in enumerate(lengths):
        g0, g1 = int(off[c]) + int(L), int(off[c + 1])
        if poison == "big":
            d[g0:g1] = rng.integers(10 ** 9, 2 ** 31 - 1, g1 - g0)
        elif poison == "mid":
            d[g0:g1] = 7777
        else:
            near = max(int(d[g0 - 1]) if L else 0, int(d[g1]) if g1 < len(d) and lengths[c + 1] else 0)
            d[g0:g1] = min(near + 1, OVERFLOW - 1)
    return d


# ---------------------------------------------------------------------------------------------------------------------
# region sets


def as_cols(rows):
    t, s, e = (np.array(x, np.int64) for x in zip(*rows))
    return t.astype(np.int32), s.astype(np.int32), e.astype(np.int32)


def mixed_set(lengths, rng, n_random=400):
    """Whole contigs (also of length 0), empty regions, regions reaching past the end or lying wholly past it,
    [L - 10, 2^31 - 1), lengths 1..9 at every start mod 4 at the start, middle and end of every contig, lengths
    8191 / 8192 / 8193, and hundreds of random overlapping regions, some listed twice."""
    rows = []
    for c, L in enumerate(int(x) for x in lengths):
        rows += [(c, 0, L), (c, 0, 0), (c, L, L), (c, L, L + 1), (c, L + 2, L + 9), (c, max(L - 10, 0), HUGE)]
        if L >= 1:
            rows.append((c, L - 1, L + 5))
        if L >= 3:
            rows.append((c, 1, L - 1))
        for base in sorted({0, (L // 2) & ~3, max(L - 12, 0) & ~3}):
            rows += [(c, s, s + k) for s in range(base, base + 4) for k in range(1, 10)]
        if L >= 8193 + 8:
            for k in (8191, 8192, 8193):
                rows += [(c, s, s + k) for s in (0, 1, 2, 3, L - k, L - k + 2, L // 3)]
    small = [c for c, L in enumerate(lengths) if 0 < L <= 100_000]
    extra = []
    for _ in range(n_random):
        c = int(rng.choice(small))
        L = int(lengths[c])
        a = int(rng.integers(0, L + 4))
        n = int(rng.choice([rng.integers(1, 10), rng.integers(1, 3000), rng.integers(1, 20000)]))
        extra.append((c, a, a + n))
    extra += [extra[i] for i in rng.integers(0, len(extra), n_random // 4)]
    rows += extra
    return as_cols([rows[i] for i in rng.permutation(len(rows))])


def clip(lengths, tid, start, end):
    L = lengths[tid].astype(np.int64)
    cs = np.minimum(start, L)
    n = np.minimum(end, L) - cs
    return n, (end.astype(np.int64) - start) - n


def stream_plan(lengths, tid, start, end, n_sm):
    """The balanced stream's plan as stats_launch (mcov_api.cu) builds it: regions with more than 8192 slots inside
    their contig are concatenated in list order and cut into slices of W slots, one per CTA, with
    grid = min(2 n_SM, max(1, total / 16384)) and W = max(4, ceil(total / grid) rounded up to 4).
    Returns (n_ctas, W, pieces of every region (0: not in the stream), concatenation end of every region)."""
    n, _ = clip(lengths, tid, start, end)
    big = n > 8192
    total = int(n[big].sum())
    if total == 0:
        return 0, 0, np.zeros(len(tid), np.int64), np.zeros(len(tid), np.int64)
    grid = min(2 * n_sm, max(1, total // 16384))
    W = max(4, (-(-total // grid) + 3) & ~3)
    ends = np.cumsum(np.where(big, n, 0))
    begins = ends - np.where(big, n, 0)
    pieces = np.where(big, (ends - 1) // W - begins // W + 1, 0)
    return -(-total // W), W, pieces, ends


def stream_set(lengths, rng, n_sm, extra_rows):
    """Large regions whose concatenation fills the whole grid (2 n_SM slices of W slots): a region ending exactly on a
    slice border, split regions with padding (one reaching 2^31 - 1), the same region twice, and about a hundred more
    split regions of random length; the small regions `extra_rows` are interleaved."""
    grid = 2 * n_sm
    W = 4 * -(-8_000_000 // (4 * grid))
    total = grid * W
    big = [c for c, L in enumerate(lengths) if L >= 600_000]
    L = {c: int(lengths[c]) for c in big}
    b0, b1, b2, b3 = big
    rows = [(b1, 0, 3 * W),                                  # three pieces, ends on the third slice border
            (b3, L[b3] - 2 * W - 5, L[b3] + 999),            # split, padded
            (b1, L[b1] - 3 * W, HUGE),                       # split, 2^31 - 1 - L positions of padding
            (b2, 12345, 12345 + 2 * W + 7), (b2, 12345, 12345 + 2 * W + 7)]    # listed twice
    rem = total - sum(min(e, L[c]) - s for c, s, e in rows)
    while rem > 400_000:
        n = int(rng.integers(8193, 200_001))
        c = int(rng.choice(big))
        s = int(rng.integers(0, L[c] - n + 1))
        rows.append((c, s, s + n))
        rem -= n
    for n in (rem // 2, rem - rem // 2):
        rows.append((b0, 777, 777 + n))
    rows = [(int(c), int(s), int(e)) for c, s, e in rows]
    for r in extra_rows:
        rows.insert(int(rng.integers(0, len(rows) + 1)), r)
    return as_cols(rows)


# ---------------------------------------------------------------------------------------------------------------------
# comparisons


def assert_records(got, want, reg, what, rows=None):
    rows = np.arange(len(want)) if rows is None else rows
    for k in FIELDS:
        bad = rows[got[k][rows] != want[k][rows]]
        if len(bad):
            i = int(bad[0])
            raise AssertionError("%s: %s differs on %d regions; first: region %d (tid %d, [%d, %d)): got %s, want %s"
                                 % (what, k, len(bad), i, reg[0][i], reg[1][i], reg[2][i], got[i], want[i]))


def assert_device_records(got, want, reg, what):
    """Records of the device-side routes: zero-length regions are not written; records whose depth reaches the
    overflow bin carry bit1 and are otherwise not exact."""
    nonempty = reg[2] > reg[1]
    ovf = (want["flags"] & 2) != 0
    assert_records(got, want, reg, what, np.nonzero(nonempty & ~ovf)[0])
    bad = np.nonzero(nonempty & ovf & ((got["flags"] & 2) == 0))[0]
    assert not len(bad), "%s: overflow not flagged on %d regions, first %d" % (what, len(bad), bad[0])


def test_reference_equals_c_oracle():
    """The reference against the C oracle (which sorts the materialised region) and against a numpy sort, on stores
    of every generator with poison between contigs and regions of small padding."""
    lengths = np.array([0, 1, 2, 3, 5, 4000, 4000, 3000, 3000, 9000, 20000, 700, 0, 33, 30000], np.int32)
    kinds = ["rot"] * 5 + ["anchor_up", "anchor_down", "distinct1024", "distinct1025"] + ["rot"] * 6
    _, off = cport.layout(lengths)
    for seed, (pool, poison) in enumerate([(EXACT_GENS, "big"), (OVERFLOW_GENS, "near"), (EXACT_GENS + OVERFLOW_GENS, "mid"),
                                           (("borders", "every", "slices"), "big")]):
        d = make_store(lengths, kinds, off, seed, pool, poison)
        rng = np.random.default_rng(seed)
        tid, st, en = mixed_set(lengths, rng, n_random=200)
        keep = en < HUGE                                      # the C oracle materialises the padding
        tid, st, en = tid[keep], st[keep], en[keep]
        refs = ref_region_stats(d, off, lengths, tid, st, en, BREADTHS, plain_max=100_000)
        for bn in BREADTHS:
            orc = cport.region_stats(d, off, lengths, tid, st, en, breadth_n=bn)
            got = refs[bn]
            for k in FIELDS[:-2]:
                assert np.array_equal(got[k], orc[k]), (seed, bn, k)
            assert np.array_equal(got["flags"] & 1, orc["flags"])
            assert np.array_equal((got["flags"] & 2) != 0, got["max"] >= OVERFLOW)
        assert (refs[1]["max"] >= OVERFLOW).any() == (seed in (1, 2))


# ---------------------------------------------------------------------------------------------------------------------
# the store on the GPU


class Store:
    def __init__(self):
        import torch
        from metacov_b200 import CoverageEngine, ReadBatch
        self.torch = torch
        self.lengths = LENGTHS
        self.kinds = [c[1] for c in CONTIGS]
        _, self.off = cport.layout(self.lengths)
        self.eng = CoverageEngine(self.lengths)
        assert self.eng.n_slots == self.off[-1]
        assert all(self.eng.contig_offset(c) == self.off[c] for c in range(len(self.lengths)))
        self.buf = torch.zeros(int(self.eng.n_slots), dtype=torch.int32, device="cuda")
        self.eng.bind_depth(self.buf)
        z = np.zeros(0, np.int32)
        self.eng.depth_sorted(ReadBatch(z, z, z.astype(np.uint16), z.astype(np.uint8), np.zeros(1, np.uint32),
                                        z.astype(np.uint32)))
        assert self.eng.depth_ptr() == self.buf.data_ptr()  # (also: the tile histograms are no longer trusted)
        self.n_sm = torch.cuda.get_device_properties(0).multi_processor_count
        self.d = None

    def fill(self, seed, pool=EXACT_GENS + OVERFLOW_GENS, poison="big"):
        self.d = make_store(self.lengths, self.kinds, self.off, seed, pool, poison)
        self.buf.copy_(self.torch.from_numpy(self.d))
        self.torch.cuda.synchronize()

    def ref(self, reg, breadths=(1,), plain_max=0):
        return ref_region_stats(self.d, self.off, self.lengths, *reg, breadths=breadths, plain_max=plain_max)

    def stats(self, reg, breadth_n=1):
        return self.eng.region_stats(*reg, breadth_n=breadth_n).copy()

    def dev_out(self, g):
        return self.torch.full((g * 64,), 0xA5, dtype=self.torch.uint8, device="cuda")

    def host(self, t):
        self.eng.sync()
        return t.cpu().numpy().view(STATS_DTYPE).copy()

    def sets(self, seed):
        """(mixed set, stream-targeted set, set with one region over every slice), plans checked."""
        rng = np.random.default_rng(1000 + seed)
        mixed = mixed_set(self.lengths, rng)
        small = np.nonzero(clip(self.lengths, *mixed)[0] <= 8192)[0]
        some = [tuple(int(x[i]) for x in mixed) for i in rng.choice(small, 300)]
        s1 = stream_set(self.lengths, rng, self.n_sm, some)
        n_ctas, W, pieces, ends = stream_plan(self.lengths, *s1, self.n_sm)
        _, pad = clip(self.lengths, *s1)
        split = pieces > 1
        assert n_ctas == 2 * self.n_sm, "the stream set no longer fills the whole grid"
        assert split.sum() >= 50, "fewer than 50 split regions"
        assert (split & (pad > 0)).any() and (split & (pad > 2 ** 30)).any(), "no split region with padding"
        assert (split & (ends % W == 0) & (ends < n_ctas * W)).any(), "no region ends on a slice border"
        assert (pieces >= 3).any()
        b0 = int(np.nonzero(self.lengths == self.lengths.max())[0][0])
        rows = [(b0, 7, int(self.lengths[b0]) + 1000)] + some[:60]
        s2 = as_cols(rows)
        n_ctas2, _, pieces2, _ = stream_plan(self.lengths, *s2, self.n_sm)
        assert n_ctas2 >= self.n_sm and pieces2[0] == n_ctas2, "no region spans every slice"
        return mixed, s1, s2


@pytest.fixture(scope="module")
def store():
    s = Store()
    yield s
    s.eng.close()


@pytest.mark.gpu
def test_region_stats_every_breadth(store):
    """region_stats == the reference, field by field, for five breadth thresholds, on three fills (three kinds of
    poison), for the mixed set and the stream-targeted set."""
    for f, poison in enumerate(("big", "mid", "near")):
        store.fill(f, poison=poison)
        for name, reg in zip(("mixed", "stream"), store.sets(f)[:2]):
            refs = store.ref(reg, BREADTHS, plain_max=100_000 if f == 0 else 0)
            for bn in BREADTHS:
                assert_records(store.stats(reg, bn), refs[bn], reg, "fill %d %s breadth %d" % (f, name, bn))


@pytest.mark.gpu
def test_cached_plan_across_fills_and_sets(store):
    """One plan run on three different fills in a row (the split regions' global scratch must come back zeroed),
    then a second set with one region over every slice, then the first set again."""
    mixed, s1, s2 = store.sets(3)
    for f, poison in ((3, "near"), (4, "big"), (5, "mid")):
        store.fill(f, poison=poison)
        assert_records(store.stats(s1), store.ref(s1)[1], s1, "stream set, fill %d" % f)
    assert_records(store.stats(s2), store.ref(s2)[1], s2, "one region over every slice")
    assert_records(store.stats(s1), store.ref(s1)[1], s1, "stream set again")
    assert_records(store.stats(mixed), store.ref(mixed)[1], mixed, "mixed set")
    assert_records(store.stats(s1), store.ref(s1)[1], s1, "stream set after the mixed set")


@pytest.mark.gpu
def test_three_routes(store):
    """The same records through region_stats, submit / collect on both slots (copied and viewed) and enqueue into
    device memory; then enqueue on depth that reaches the overflow bin."""
    torch = store.torch
    mixed, s1, _ = store.sets(6)
    store.fill(6, pool=EXACT_GENS, poison="near")
    for name, reg in (("mixed", mixed), ("stream", s1)):
        for bn in (1, 1024):
            want = store.ref(reg, (bn,))[bn]
            assert_records(store.stats(reg, bn), want, reg, "%s run" % name)
            for slot in (0, 1):
                for copy in (True, False):
                    got = store.eng.region_stats_collect(store.eng.region_stats_submit(*reg, breadth_n=bn, slot=slot),
                                                         copy=copy).copy()
                    assert_records(got, want, reg, "%s collect slot %d copy %s" % (name, slot, copy))
            out = store.dev_out(len(reg[0]))
            torch.cuda.synchronize()
            store.eng.region_stats_enqueue(*reg, out, breadth_n=bn)
            assert_device_records(store.host(out), want, reg, "%s enqueue" % name)
    store.fill(7, pool=OVERFLOW_GENS + ("slices",), poison="mid")
    for name, reg in (("mixed", mixed), ("stream", s1)):
        want = store.ref(reg)[1]
        assert (want["flags"] & 2).any() and not (want["flags"] & 2).all()
        out = store.dev_out(len(reg[0]))
        torch.cuda.synchronize()
        store.eng.region_stats_enqueue(*reg, out)
        assert_device_records(store.host(out), want, reg, "%s enqueue, overflow fill" % name)


def cut_parts(rng, lengths, c, a, b):
    """[a, b) cut into 1..5 consecutive parts: 1-slot parts at either end and, when the region reaches past its
    contig, a part wholly in the padding are among the candidates."""
    if b - a <= 1:
        return [(a, b)]
    L = int(lengths[c])
    cand = {a + 1, b - 1}
    if a < L < b:
        cand.add(L)
    if max(a, L) + 2 < b:
        cand.add(max(a, L) + (b - max(a, L)) // 2)
    cand |= set(int(x) for x in rng.integers(a + 1, b, 4))
    k = int(rng.integers(1, 6))
    cuts = sorted(int(x) for x in rng.choice(sorted(cand), min(k - 1, len(cand)), replace=False))
    p = [a] + cuts + [b]
    return list(zip(p[:-1], p[1:]))


@pytest.mark.gpu
def test_histogram_merge(store):
    """Every region cut into parts, each part's histogram added by its own region_hist_enqueue call (parts in shuffled
    order), then hist_stats_enqueue: the reference's records; where the overflow bin is populated, bit1."""
    torch = store.torch
    mixed, s1, _ = store.sets(8)
    big = np.nonzero(clip(store.lengths, *s1)[0] > 8192)[0]
    reg = tuple(np.r_[m, s[big]].astype(np.int32) for m, s in zip(mixed, s1))
    g = len(reg[0])
    rng = np.random.default_rng(8)
    parts = [cut_parts(rng, store.lengths, int(reg[0][i]), int(reg[1][i]), int(reg[2][i])) for i in range(g)]
    assert any(len(p) == 5 for p in parts) and any(b - a == 1 for p in parts for a, b in p if len(p) > 1)
    assert any(a >= store.lengths[reg[0][i]] and b > a for i, p in enumerate(parts) if len(p) > 1 for a, b in p)
    order = [rng.permutation(len(p)) for p in parts]
    for f, pool, poison in ((8, EXACT_GENS, "big"), (9, EXACT_GENS + OVERFLOW_GENS, "near")):
        store.fill(f, pool=pool, poison=poison)
        hist = torch.zeros((g, 8192), dtype=torch.int32, device="cuda")
        out = store.dev_out(g)
        torch.cuda.synchronize()
        for r in range(5):
            cols = [[], [], []]
            for i in range(g):
                a, b = parts[i][order[i][r]] if r < len(parts[i]) else (int(reg[1][i]), int(reg[1][i]))
                cols[0].append(int(reg[0][i])); cols[1].append(a); cols[2].append(b)
            store.eng.region_hist_enqueue(*as_cols(list(zip(*cols))), hist)
        for bn in (1, 1024):
            store.eng.hist_stats_enqueue(hist, g, out, breadth_n=bn)
            got = store.host(out)
            want = store.ref(reg, (bn,))[bn]
            ovf = (want["flags"] & 2) != 0
            assert_records(got, want, reg, "merged histograms, fill %d breadth %d" % (f, bn), np.nonzero(~ovf)[0])
            assert ((got["flags"][ovf] & 2) != 0).all()
        assert ovf.any() == (f == 9)


@pytest.mark.gpu
def test_window_means(store):
    """window_means == the exact int64 sum of each window over its length in float64, bit for bit; windows of 1, 3,
    4, 1000, 2048, 8193 slots and one longer than every contig (length-0 contigs give no window)."""
    for f, poison in ((10, "big"), (11, "near")):
        store.fill(f, poison=poison)
        for w in (1, 3, 4, 1000, 2048, 8193, int(store.lengths.max()) + 1):
            want = []
            for c, L in enumerate(int(x) for x in store.lengths):
                x = store.d[store.off[c]:store.off[c] + L].astype(np.int64)
                cs = np.r_[np.int64(0), np.cumsum(x)]
                s = np.arange(0, L, w)
                e = np.minimum(s + w, L)
                want.append((cs[e] - cs[s]) / (e - s))
            want = np.concatenate(want)
            got = store.eng.window_means(w)
            assert got.shape == want.shape and got.tobytes() == want.tobytes(), (f, w)


def ref_runs(d, off, lengths, tid0, tid1):
    cols = [[], [], [], []]
    for c in range(tid0, tid1):
        L = int(lengths[c])
        if L == 0:
            continue
        x = d[off[c]:off[c] + L]
        s = np.r_[0, np.nonzero(x[1:] != x[:-1])[0] + 1]
        e = np.r_[s[1:], L]
        for k, v in enumerate((np.full(len(s), c), s, e, x[s])):
            cols[k].append(v)
    out = np.zeros(sum(len(v) for v in cols[0]), dtype=[("tid", "<i4"), ("start", "<i4"), ("end", "<i4"), ("depth", "<i4")])
    for name, v in zip(out.dtype.names, cols):
        out[name] = np.concatenate(v) if v else []
    return out


@pytest.mark.gpu
def test_depth_runs(store):
    """depth_runs == a numpy run-length encoding per contig: all contigs, a sub-range, skip_zero; with a contig that
    changes at every slot, a constant one, run borders on and next to multiples of 8192 slots, runs across them."""
    for f, poison in ((12, "big"), (13, "near")):
        store.fill(f, poison=poison)
        n = len(store.lengths)
        for tid0, tid1 in ((0, n), (8, 19), (16, 17), (1, 2)):
            want = ref_runs(store.d, store.off, store.lengths, tid0, tid1)
            got = store.eng.depth_runs(tid0, tid1)
            assert got.tobytes() == want.tobytes(), (f, tid0, tid1)
            got = store.eng.depth_runs(tid0, tid1, skip_zero=True)
            assert got.tobytes() == want[want["depth"] != 0].tobytes(), (f, tid0, tid1)
        runs = ref_runs(store.d, store.off, store.lengths, 16, 17)
        assert {8191, 8192, 8193, 16384} <= set(runs["start"].tolist())


@pytest.mark.gpu
def test_every_statistics_kernel_ran(store):
    """The sets above reach every statistics kernel: the warp kernel and its retry kernel, the stream, the radix
    path, and the cross-device pair."""
    torch = store.torch
    store.eng.profile(True)
    try:
        mixed, s1, _ = store.sets(14)
        store.fill(14, pool=OVERFLOW_GENS, poison="near")
        for reg in (mixed, s1):
            assert_records(store.stats(reg), store.ref(reg)[1], reg, "profiled run")
        reg = tuple(x[:50] for x in mixed)
        hist = torch.zeros((50, 8192), dtype=torch.int32, device="cuda")
        out = store.dev_out(50)
        torch.cuda.synchronize()
        store.eng.region_hist_enqueue(*reg, hist)
        store.eng.hist_stats_enqueue(hist, 50, out)
        store.eng.sync()
        ran = store.eng.profile_read()
    finally:
        store.eng.profile(False)
    for k in ("k_region_stats_warp", "k_region_stats_small", "k_stats_stream", "k_sorted_stats", "k_region_hist",
              "k_hist_finish"):
        assert ran.get(k, (0, 0))[0] > 0, (k, sorted(ran))
