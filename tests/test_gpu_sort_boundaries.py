"""The shared union and term-sort engines at their size boundaries.

Lookup, boolean query, pattern search and prefix search build their posting unions with
`k2_large_run` (k12_union.cu), and merge sends its heavy terms (> 4096 values) through it; the
unions are placed by `place_unions` (k5_prefix.cu).  Ingest and pattern terms sort terms with K7's
segmented bitonic sort (k7_ingest.cu).  Each engine switches paths on constants:

    LG_TILE = 4096           values per shared-memory sort tile of k2_large_run
    gx <= 2048               CTAs per group: longer unions take the grid-stride loops
    BM_MIN_VALUES = 65536    shortest union considered for the bitmap path ...
    words <= 4 * len         ... when its map of (max >> 5) + 1 words is dense enough
    BM_CHUNK_WORDS = 32      words (1024 bits) one warp counts and expands
    4096 output values       k2_large_finish: enc_emit_cta at >= 4096, enc_emit_warp below
    32768                    groups / documents per grid row (the `y0` loops)
    kMaxSegs = 1024          sources of one group (k2_large_gather's s_moff table)
    K7_TILE = 2048           records per shared-memory tile of K7's sort

Every case here is a differential check against a plain numpy / Python reference that uses no
library code: np.unique(np.concatenate(sources)) for a union, sorted(set(terms)) for term order
(Python's bytes order is bytes.Compare).  Where the output has a `_val` stream, the stream is
decoded with the oracle's decoder and compared with the reference, and the bytes are compared
with the oracle's merge.  test_references_match_oracle checks the references themselves against
the oracle without a GPU."""
import bisect
import ctypes as C

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A
from inverted_index_2_b200.flat import FlatSegment, views_array
from test_gpu_parity import assert_merge_equal

gpu = pytest.mark.gpu

BM_MIN_VALUES = 1 << 16
U32 = np.uint32


@pytest.fixture(params=["general", "fused"])
def merge_path(request, monkeypatch):
    """Both bucket pipelines in front of k2_large_run: the general kernels (K1b -> K2b -> K6) and
    the fused bucket kernel (k12_fused.cu, II2_FUSED=1), which defers long terms to them."""
    monkeypatch.setenv("II2_FUSED", "1" if request.param == "fused" else "0")
    return request.param


# ---------------------------------------------------------------- references (numpy / Python)
def ref_union(sources):
    """np.unique(np.concatenate(sources)), as a sort and an adjacent-difference mask (numpy 2.3's
    hash-based np.unique takes seconds at millions of values; test_references_match_oracle checks
    that the two agree)."""
    if not sources:
        return np.zeros(0, dtype=U32)
    v = np.sort(np.concatenate([np.asarray(s, dtype=U32) for s in sources]))
    return v[np.concatenate(([True], v[1:] != v[:-1]))] if len(v) else v


def ref_prefix_search(seg_items, prefixes):
    """Per prefix (aligned with `prefixes`): the sorted-unique union of the lists of every term
    with that prefix over all segments, or None when no term has it.  seg_items: per segment a
    list of (term, values)."""
    by_term = {}
    for items in seg_items:
        for t, v in items:
            by_term.setdefault(t, []).append(np.asarray(v, dtype=U32))
    vocab = sorted(by_term)
    term_union = {}
    cache = {}
    out = []
    for p in prefixes:
        if p not in cache:
            lo = bisect.bisect_left(vocab, p)
            hi = lo
            while hi < len(vocab) and vocab[hi].startswith(p):
                hi += 1
            if hi == lo:
                cache[p] = None
            else:
                for t in vocab[lo:hi]:
                    if t not in term_union:
                        term_union[t] = ref_union(by_term[t])
                cache[p] = ref_union([term_union[t] for t in vocab[lo:hi]])
        out.append(cache[p])
    return out


def ref_merge(seg_items, removed=None):
    """Shard.Merge of decoded segments: [(term, values)] in bytes order.  A term held by one
    segment passes through (order and duplicates kept), a shared term is the sorted-unique union;
    removed values are dropped and a term left without values is dropped."""
    rem = np.zeros(0, dtype=U32) if removed is None else np.asarray(removed, dtype=U32)
    by_term = {}
    for items in seg_items:
        for t, v in items:
            by_term.setdefault(t, []).append(np.asarray(v, dtype=U32))
    out = []
    for t in sorted(by_term):
        srcs = by_term[t]
        v = srcs[0] if len(srcs) == 1 else ref_union(srcs)
        v = v[~np.isin(v, rem)]
        if len(v):
            out.append((t, v))
    return out


def ref_ingest(docs, removed=None):
    """Put of every document, then one Merge: [(term, values)] in bytes order, every term's
    values the sorted-unique values of the documents that hold it, removed values dropped."""
    rem = set() if removed is None else {int(x) for x in removed}
    vals = {}
    for terms, val in docs:
        for t in set(terms):
            vals.setdefault(t, set()).add(int(val))
    out = []
    for t in sorted(vals):
        v = sorted(vals[t] - rem)
        if v:
            out.append((t, np.array(v, dtype=U32)))
    return out


class RefPatternTerms:
    """(term, segments, postings, 0) of every term a glob made of literal bytes and an optional
    trailing `*` matches, in bytes order: instances and stored list lengths over the segments."""

    def __init__(self, seg_items):
        self.stats = {}
        for items in seg_items:
            for t, v in items:
                st = self.stats.setdefault(t, [0, 0])
                st[0] += 1
                st[1] += len(v)
        self.vocab = sorted(self.stats)

    def __call__(self, pattern):
        if pattern.endswith(b"*"):
            p = pattern[:-1]
            lo = hi = bisect.bisect_left(self.vocab, p)
            while hi < len(self.vocab) and self.vocab[hi].startswith(p):
                hi += 1
            hit = self.vocab[lo:hi]
        else:
            hit = [pattern] if pattern in self.stats else []
        return [(t, self.stats[t][0], self.stats[t][1], 0) for t in hit]


def decode_stream(orc, res):
    """The merge result's `_val` stream decoded by the oracle's decoder, one array per term."""
    n = res.terms_count
    if n == 0:
        return []
    words = np.frombuffer(res.val_bytes.tobytes(), dtype=U32)
    woff = np.append(res.val_off, np.uint64(res.val_size)).astype(np.uint64) // 4
    vals, off = orc.intcomp_decode_batch(words, woff)
    return [vals[int(off[i]):int(off[i + 1])] for i in range(n)]


def check_merge_result(orc, got, exp_items, oracle_res):
    """Terms, decoded `_val` stream and decoded lists against the reference; bytes against the
    oracle's merge."""
    assert got.terms() == [t for t, _ in exp_items]
    dec = decode_stream(orc, got)
    for (t, v), d in zip(exp_items, dec):
        assert np.array_equal(d, v), t
    for i, (t, v) in enumerate(exp_items):
        assert np.array_equal(got.post[int(got.post_off[i]):int(got.post_off[i + 1])], v), t
    assert_merge_equal(got, oracle_res)


# ---------------------------------------------------------------- builders
def flat_segment(items):
    """A decoded segment from (term, values) pairs in ascending term order, built from arrays."""
    tb, toff = FlatSegment._pack_terms([t for t, _ in items])
    lens = np.fromiter((len(v) for _, v in items), dtype=np.uint64, count=len(items))
    poff = np.zeros(len(items) + 1, dtype=np.uint64)
    np.cumsum(lens, out=poff[1:])
    post = (np.concatenate([np.asarray(v, dtype=U32) for _, v in items]) if items
            else np.zeros(0, dtype=U32))
    return FlatSegment(tb, toff, A.II2_SEG_DECODED, post=post, post_off=poff)


def group_layout(groups, nseg):
    """Group g's source j becomes term b"g%05d/%05d" in segment (g + j) % nseg; group g is
    prefix b"g%05d/".  Returns (per-segment items, segments, prefixes)."""
    per_seg = [[] for _ in range(nseg)]
    for g, sources in enumerate(groups):
        for j, src in enumerate(sources):
            per_seg[(g + j) % nseg].append((b"g%05d/%05d" % (g, j), src))
    for items in per_seg:
        items.sort(key=lambda x: x[0])
    segs = [flat_segment(items) for items in per_seg]
    return per_seg, segs, [b"g%05d/" % g for g in range(len(groups))]


def prefix_lists(engine, segs, prefixes, dev=False):
    """ii2_prefix_search(_dev) aligned with `prefixes` (None: not matched), every index read,
    repeated prefixes included."""
    blob, off = engine._prefix_args(prefixes)
    out = A.PrefixOut()
    if dev:
        rc = engine.lib.ii2_prefix_search_dev(engine._handles(segs), len(segs), A.np_ptr(blob, A.u8p),
                                              A.np_ptr(off, A.u32p), len(prefixes), C.byref(out))
    else:
        arr = views_array(segs)
        rc = engine.lib.ii2_prefix_search(arr, len(segs), A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p),
                                          len(prefixes), C.byref(out))
    engine._check(rc, "prefix_search")
    return engine._pattern_result(out)


def assert_lists_equal(got, exp, names):
    assert len(got) == len(exp)
    for g, e, name in zip(got, exp, names):
        if e is None:
            assert g is None, name
        else:
            assert g is not None, name
            assert np.array_equal(g, e), (name, len(g), len(e))


def split(values, parts):
    return [np.ascontiguousarray(x) for x in np.array_split(values, max(1, min(parts, len(values))))]


def launches(engine, fn):
    before = engine.kernel_launches()
    fn()
    return engine.kernel_launches() - before


def assert_sort_path_only(groups):
    """No group reaches the bitmap path: shorter than BM_MIN_VALUES or (max >> 5) + 1 > 4 * len."""
    for sources in groups:
        n = sum(len(s) for s in sources)
        if n >= BM_MIN_VALUES:
            m = max(int(s.max()) for s in sources if len(s))
            assert (m >> 5) + 1 > 4 * n


# ---------------------------------------------------------------- the references, without a GPU
def test_references_match_oracle(orc):
    """The numpy references above against the CPU oracle on small inputs: prefix unions, merge
    (pass-through of a single source, shared terms, removed values, a term emptied by them), ingest
    (repeats inside a document, empty documents, 16-byte ties) and the `_val` decoder."""
    rng = np.random.default_rng(3)
    for sources in ([], [[]], [[5, 5, 1]], [[0xFFFFFFFF, 0, 7], [7, 3, 0]],
                    [rng.integers(0, 1 << 32, 5000, dtype=np.uint64).astype(U32), rng.integers(0, 300, 5000)]):
        exp = np.unique(np.concatenate([np.asarray(s, dtype=U32) for s in sources] or [np.zeros(0, U32)]))
        assert ref_union(sources).dtype == U32 and np.array_equal(ref_union(sources), exp)
    per_seg = [[(b"a", [9, 3, 3, 7]), (b"ab", [5, 1, 5]), (b"b", [0xFFFFFFFF, 0, 5]), (b"gone", [8, 8])],
               [(b"ab", [1, 9, 9]), (b"abc", []), (b"ba", [5, 5, 1]), (b"gone", [8])],
               [(b"", [4]), (b"zz", rng.integers(0, 1 << 32, 50, dtype=np.uint64).astype(U32).tolist())]]
    segs = [FlatSegment.from_items(items) for items in per_seg]
    prefixes = [b"a", b"ab", b"abc", b"b", b"", b"c", b"zz", b"a"]
    exp = orc.prefix_search(segs, prefixes)
    got = ref_prefix_search(per_seg, prefixes)
    for p, g in zip(prefixes, got):
        assert (g is None) == (p not in exp), p
        if g is not None:
            assert g.tolist() == exp[p], p
    for removed in (None, np.array([3, 8], dtype=U32), np.array([0, 1, 5, 9], dtype=U32)):
        ores = orc.merge(segs, removed, decoded=True)
        ref = ref_merge(per_seg, removed)
        assert [(t, v.tolist()) for t, v in ref] == list(ores.as_dict().items())
        assert [d.tolist() for d in decode_stream(orc, ores)] == [v.tolist() for _, v in ref]
    ties = [b"x" * 15, b"x" * 15 + b"\0", b"x" * 15 + b"\0\0", b"", b"\xff" * 17, b"\xff" * 16,
            b"0123456789abcdef" + b"\xff", b"0123456789abcdef" + b"\0"]
    docs = [([], 1), (ties + ties[::-1], 7), ([b"q", b"q"], 7), ([], 2), ([b"x" * 15, b"q"], 9), ([], 3)]
    for removed in (None, np.array([7], dtype=U32)):
        ores = orc.ingest(docs, removed, decoded=True)
        ref = ref_ingest(docs, removed)
        assert [(t, v.tolist()) for t, v in ref] == list(ores.as_dict().items())
    assert ref_ingest([([], 1), ([], 2)]) == [] and orc.ingest([([], 1), ([], 2)]).terms_count == 0
    rr = orc.read_range(segs, b"a", b"a\xff")
    ref_terms = RefPatternTerms(per_seg)
    assert [t for t, _, _, _ in ref_terms(b"a*")] == rr.terms()
    assert [t for t, _, _, _ in ref_terms(b"*")] == orc.read_range(segs).terms()
    assert ref_terms(b"ab") == [(b"ab", 2, 6, 0)]
    assert ref_terms(b"x*") == [] and ref_terms(b"abcd") == []


# ---------------------------------------------------------------- 1. k2_large_run's sort path
# Union lengths on and around LG_TILE = 4096 (one tile, one value over, two tiles +- 1, three
# tiles + 1), 65535 (one below BM_MIN_VALUES), 2^17 + 3 and 2^20 + 1 (global bitonic stages up
# to kk = 2^18 / 2^21 over a ragged last tile).
SORT_LENGTHS = [1, 4095, 4096, 4097, 8191, 8192, 8193, 3 * 4096 + 1, 65535, (1 << 17) + 3, (1 << 20) + 1]
# 9,000,001 values: gx = min(ceil(9000001 / 4096), 2048) = 2048 CTAs for 2198 tiles, so
# k2_large_tile_sort and k2_large_tile_merge run their grid-stride loops (t0 += 2048 * 4096).
GRID_STRIDE_LEN = 9_000_001


def _sort_path_groups(rng, nseg):
    """Every length in every value shape.  Values are drawn over 2^32, so no union of 65536 or
    more values is dense enough for the bitmap path ((max >> 5) + 1 > 4 * len)."""
    groups = []
    for L in SORT_LENGTHS:
        vals = rng.integers(0, 1 << 32, size=L, dtype=np.uint64).astype(U32)
        groups.append([np.sort(x) for x in split(vals, nseg)])                 # sorted sources
        groups.append([np.sort(x)[::-1].copy() for x in split(vals, 3)])       # sorted descending
        groups.append(split(np.full(L, 0xC0FFEE42, dtype=U32), 3))              # all values equal
        pool = rng.integers(0, 1 << 32, size=max(1, L // 64), dtype=np.uint64).astype(U32)
        groups.append(split(pool[rng.integers(0, len(pool), size=L)], 4))      # heavy duplication
        one = rng.integers(0, 1 << 32, size=L, dtype=np.uint64).astype(U32)    # one unsorted source:
        one[1::5] = one[0::5][:len(one[1::5])]                                # a prefix still sorts
        groups.append([one])                                                   # and de-duplicates
    big = rng.integers(0, 1 << 32, size=GRID_STRIDE_LEN, dtype=np.uint64).astype(U32)
    groups.append([np.sort(x) for x in split(big, nseg)])
    return groups


@gpu
def test_prefix_sort_path_lengths(engine):
    """One prefix-search call (always_sort = 1) with a union of every length in SORT_LENGTHS and
    every value shape, plus one union past the 2048-CTA cap; then the same call over 1024
    segments (kMaxSegs: every group has 1024 sources, k2_large_gather's s_moff table is full)."""
    exp = None
    for nseg in (4, 1024):
        groups = _sort_path_groups(np.random.default_rng(11), nseg)
        assert_sort_path_only(groups)
        if exp is None:
            exp = [ref_union(g) for g in groups]
        per_seg, segs, prefixes = group_layout(groups, nseg)
        prefixes = prefixes + [b"h", prefixes[3]]     # unmatched; repeated
        got = prefix_lists(engine, segs, prefixes)
        assert_lists_equal(got, exp + [None, exp[3]], prefixes)
        del got


# ---------------------------------------------------------------- 2. k2_large_run's bitmap path
def _dense(rng, L, hi, parts):
    """L values in [0, hi] with hi itself present, in `parts` sorted sources."""
    v = rng.integers(0, hi + 1, size=L, dtype=np.uint64).astype(U32)
    v[rng.integers(0, L)] = hi
    return [np.sort(x) for x in split(v, parts)]


@gpu
def test_prefix_bitmap_thresholds(engine):
    """Unions on both sides of every bitmap-path condition of k2_large_run, through prefix search
    (always_sort = 1, so one source is enough); the path taken is shown by the launches: the
    bitmap path skips the global bitonic stages."""
    rng = np.random.default_rng(12)
    L4 = BM_MIN_VALUES + 5
    cases = {
        # len = 65535 < BM_MIN_VALUES: sort path; 65536 = BM_MIN_VALUES: bitmap path
        "len_65535": _dense(rng, 65535, (1 << 16) - 1, 3),
        "len_65536": _dense(rng, 65536, (1 << 16) - 1, 3),
        # max = 128 len - 1: (max >> 5) + 1 = 4 len words, bitmap; max = 128 len: 4 len + 1, sort
        "words_4len": _dense(rng, L4, 128 * L4 - 1, 2),
        "words_4len_plus_1": _dense(rng, L4, 128 * L4, 2),
        "one_source_4len": _dense(rng, L4, 128 * L4 - 1, 1),
        # every value 0: a one-word map
        "all_zero": split(np.zeros(70000, dtype=U32), 4),
        # largest value on the edges of the BM_CHUNK_WORDS = 32 word (1024-bit) expand chunk:
        # 1023 -> 32 words, one chunk; 1024 -> 33 words, a second chunk of one word; 5119 / 5120 ->
        # 160 / 161 words; 32 * 4097 - 1 -> 4097 words, the last word of a partial chunk
        "max_1023": _dense(rng, 70000, 1023, 3),
        "max_1024": _dense(rng, 70000, 1024, 3),
        "max_5119": _dense(rng, 70000, 5119, 3),
        "max_5120": _dense(rng, 70000, 5120, 3),
        "max_32x4097m1": _dense(rng, 70000, 32 * 4097 - 1, 3),
    }
    names = list(cases)
    groups = [cases[n] for n in names]
    exp = [ref_union(g) for g in groups]
    assert exp[names.index("all_zero")].tolist() == [0]
    for nseg in (1, 5):
        per_seg, segs, prefixes = group_layout(groups, nseg)
        assert_lists_equal(prefix_lists(engine, segs, prefixes), exp, names)
    # one group per call: the bitmap path launches fewer kernels than the sort path at the same length
    one = {}
    for n in ("len_65535", "len_65536", "words_4len", "words_4len_plus_1"):
        per_seg, segs, prefixes = group_layout([cases[n]], 2)
        res = []
        one[n] = launches(engine, lambda: res.append(prefix_lists(engine, segs, prefixes)))
        assert np.array_equal(res[0][0], exp[names.index(n)])
    assert one["len_65536"] < one["len_65535"]
    assert one["words_4len"] < one["words_4len_plus_1"]


@gpu
def test_prefix_bitmap_buffer_reuse(engine):
    """One call: a large bitmap group, then a smaller one, then sort-path groups, then another
    small bitmap group.  Every bitmap group of a call reuses the one map (sized for the largest);
    each clears and reads only its own (max >> 5) + 1 words."""
    rng = np.random.default_rng(13)
    groups = [
        _dense(rng, 1 << 20, (1 << 22) - 1, 4),            # bitmap, 131072 words
        _dense(rng, 70000, (1 << 17) - 1, 3),              # bitmap, 4096 words: stale bits above
        [np.sort(x) for x in split(rng.integers(0, 1 << 32, 70000, dtype=np.uint64).astype(U32), 3)],  # sort
        [np.sort(x) for x in split(rng.integers(0, 1 << 32, 5000, dtype=np.uint64).astype(U32), 2)],   # sort
        _dense(rng, 65536, 40000, 2),                      # bitmap, a map ending mid-chunk
        split(np.zeros(66000, dtype=U32), 2),              # bitmap, one word
    ]
    exp = [ref_union(g) for g in groups]
    for nseg in (3, 7):
        per_seg, segs, prefixes = group_layout(groups, nseg)
        assert_lists_equal(prefix_lists(engine, segs, prefixes), exp, prefixes)
        dsegs = [engine.upload(s) for s in segs]
        assert_lists_equal(prefix_lists(engine, dsegs, prefixes[::-1], dev=True), exp[::-1], prefixes[::-1])
        for d in dsegs:
            d.release()


@gpu
def test_merge_bitmap_path_removed_sets(engine, orc, merge_path):
    """A heavy merged term on the bitmap path (4 sources, 80000 values below 2^18: words = 8192
    <= 4 * len) under three removed sets: a dense one with its own bitmap (filtered word by word in
    k2_bm_count), a sparse one without a bitmap (under 64 values, one near 4e9: filtered in
    k2_large_finish), and one whose bitmap ends below the union's largest value (bitmap_bits =
    70016, mid-chunk: words above it are not masked).  A single-source dense term (70000 unsorted
    values with duplicates) passes through: one source never takes the bitmap path in a merge."""
    rng = np.random.default_rng(14)
    per_seg = [[] for _ in range(5)]
    for s in range(4):
        per_seg[s].append((b"heavy", np.sort(rng.integers(0, 1 << 18, 20000)).astype(U32)))
        per_seg[s].append((b"mid%d" % s, np.sort(rng.integers(0, 1 << 20, 50)).astype(U32)))
    per_seg[1].append((b"solo", rng.integers(0, 1 << 16, 70000).astype(U32)))
    per_seg[2].append((b"sparse", np.sort(rng.integers(0, 1 << 32, 40000, dtype=np.uint64)).astype(U32)))
    per_seg[4].append((b"sparse", np.sort(rng.integers(0, 1 << 32, 40000, dtype=np.uint64)).astype(U32)))
    for items in per_seg:
        items.sort(key=lambda x: x[0])
    segs = [flat_segment(items) for items in per_seg]
    heavy = ref_union([v for items in per_seg for t, v in items if t == b"heavy"])
    removed_sets = {
        "none": None,
        "dense_bitmap": np.unique(rng.integers(0, 1 << 18, 30000)).astype(U32),
        "sparse_no_bitmap": np.unique(np.append(rng.choice(heavy, 40), 4_000_000_000)).astype(U32),
        "bitmap_ends_below": np.unique(np.append(rng.integers(0, 70000, 5000), 70000)).astype(U32),
    }
    assert len(removed_sets["sparse_no_bitmap"]) < 64
    assert ((int(removed_sets["bitmap_ends_below"][-1]) + 32) & ~31) < int(heavy[-1])
    for name, rem in removed_sets.items():
        got = engine.merge(segs, rem, decoded=True)
        check_merge_result(orc, got, ref_merge(per_seg, rem), orc.merge(segs, rem, decoded=True))


@gpu
def test_merge_bitmap_term_removed_completely(engine, orc, merge_path):
    """A heavy term on the bitmap path (3 sources, 75000 values in [2^19, 2^19 + 2^16)) whose
    every value is removed, with the removed set's bitmap (k2_bm_count clears the map) and without
    one (a value near 4e9: k2_large_finish filters); the oracle decides whether the term is kept."""
    rng = np.random.default_rng(15)
    base = 1 << 19
    gone = [np.sort(rng.integers(base, base + (1 << 16), 25000)).astype(U32) for _ in range(3)]
    per_seg = [[(b"a_keep", np.array([1, 2, 3], dtype=U32)), (b"gone", gone[0])],
               [(b"gone", gone[1]), (b"z_keep", np.array([base - 1, base + (1 << 17)], dtype=U32))],
               [(b"gone", gone[2])]]
    segs = [flat_segment(items) for items in per_seg]
    all_gone = ref_union(gone)
    for rem in (all_gone, np.append(all_gone, U32(4_000_000_000))):
        got = engine.merge(segs, rem, decoded=True)
        ores = orc.merge(segs, rem, decoded=True)
        check_merge_result(orc, got, ref_merge(per_seg, rem), ores)
        assert b"gone" not in ores.terms()


@gpu
def test_merge_encoder_switch(engine, orc, merge_path):
    """k2_large_finish encodes with enc_emit_cta at >= 4096 output values and enc_emit_warp
    below.  Heavy merged terms (> 4096 input values) whose unions come to exactly 4095 and 4096
    values after de-duplication and the removed filter, on the sort path (sparse values) and on
    the bitmap path (73710+ values below 2^17; k2_bm_expand rewrites len[g], which moves the block
    table inside the encode slot).  val_bytes / val_off bit-exact with the oracle."""
    rng = np.random.default_rng(16)
    pool = rng.permutation(np.unique(rng.integers(1 << 28, 1 << 29, 40000)).astype(U32))
    take = iter(np.split(pool, np.cumsum([4095, 4096, 4200, 4201])[:4])[:4])
    rm = []
    items = [[] for _ in range(3)]

    def sort_term(name, vals):
        vals = np.sort(vals)
        n = len(vals)   # three overlapping sources: 3000 + (n - 2000) + n / 3 > 4096 input values
        for s, part in enumerate((vals[:3000], vals[2000:], vals[::3])):
            items[s].append((name, part))

    sort_term(b"s4095", next(take))
    sort_term(b"s4096", next(take))
    v = next(take)
    rm.append(v[:105])                  # 4200 - 105 = 4095 after the filter
    sort_term(b"s4095_rm", v)
    v = next(take)
    rm.append(v[:105])                  # 4201 - 105 = 4096
    sort_term(b"s4096_rm", v)

    def bitmap_term(name, vals):        # two sources of every value 9 times: >= 65536, words <= 4 len
        for s in range(2):
            items[s].append((name, np.sort(np.repeat(vals, 9))))

    dense = rng.permutation(1 << 17).astype(U32)
    bitmap_term(b"b4095", dense[:4095])
    bitmap_term(b"b4096", dense[4095:8191])
    v = dense[8191:13191]
    rm.append(v[:905])                  # 5000 - 905 = 4095
    bitmap_term(b"b4095_rm", v)
    v = dense[13191:18191]
    rm.append(v[:904])                  # 5000 - 904 = 4096
    bitmap_term(b"b4096_rm", v)
    items[2].append((b"small", np.array([7, 3, 3], dtype=U32)))
    for x in items:
        x.sort(key=lambda t: t[0])
    segs = [flat_segment(x) for x in items]
    rem_bitmap = np.unique(np.concatenate(rm)).astype(U32)               # < 2^29, >= 64 values: bitmap
    rem_search = np.append(rem_bitmap, U32(4_000_000_000))               # no bitmap: binary search
    for rem in (None, rem_bitmap, rem_search):
        got = engine.merge(segs, rem, decoded=True)
        ref = ref_merge(items, rem)
        if rem is not None:
            sizes = {t: len(v) for t, v in ref}
            assert {sizes[b"s4095_rm"], sizes[b"b4095_rm"]} == {4095}
            assert {sizes[b"s4096_rm"], sizes[b"b4096_rm"]} == {4096}
        check_merge_result(orc, got, ref, orc.merge(segs, rem, decoded=True))
        enc = engine.merge(segs, rem, decoded=False)
        ores = orc.merge(segs, rem, decoded=False)
        assert np.array_equal(enc.val_bytes, ores.val_bytes) and np.array_equal(enc.val_off, ores.val_off)


# ---------------------------------------------------------------- 4. past one grid row (32768)
def _row_workload(rng):
    """4 segments: 20000 small terms, dense terms D1/.. (below 2^16) and D2/.. (below 2^17) with
    80000 values each (bitmap path), sparse terms S/.. with 80000 values over 2^32 (sort path)."""
    per_seg = [[] for _ in range(4)]
    ids = [b"t%05d" % i for i in range(20000)]
    for s in range(4):
        keep = rng.random(20000) < 0.45
        lens = rng.integers(1, 9, size=20000)
        vals = rng.integers(0, 1 << 32, size=int(lens.sum()), dtype=np.uint64).astype(U32)
        off = np.concatenate([[0], np.cumsum(lens)])
        per_seg[s] += [(ids[i], vals[off[i]:off[i + 1]]) for i in np.nonzero(keep)[0]]
        per_seg[s].append((b"D1/%02d" % s, np.sort(rng.integers(0, 1 << 16, 20000)).astype(U32)))
        per_seg[s].append((b"D2/%02d" % s, np.sort(rng.integers(0, 1 << 17, 20000)).astype(U32)))
        per_seg[s].append((b"S/%02d" % s, np.sort(rng.integers(0, 1 << 32, 20000, dtype=np.uint64)).astype(U32)))
        per_seg[s].sort(key=lambda x: x[0])
    return per_seg, [flat_segment(x) for x in per_seg]


def _row_prefixes(rng, n):
    """Matched, unmatched and repeated prefixes and the empty one; the bitmap-path prefixes D1/ and
    D2/ at indices 32767 and 32768, one on each side of the 32768-group row split, and the
    sort-path prefix S/ (80000 values) at 32770, in the second row."""
    out = []
    for i in range(n):
        r = int(rng.integers(0, 6))
        k = int(rng.integers(0, 20000))
        if r == 0:
            out.append(b"t%05d" % k)              # one term
        elif r == 1:
            out.append(b"t%04d" % (k // 10))      # ten terms
        elif r == 2:
            out.append(b"t%03d" % (k // 100))     # a hundred terms
        elif r == 3:
            out.append(b"u%05d" % k)              # unmatched
        elif r == 4:
            out.append(b"t%05dx" % k)             # unmatched, past a term
        else:
            out.append(out[int(rng.integers(0, len(out)))] if out else b"")   # repeated
    out[0] = b""
    out[32767], out[32768], out[32769], out[32770] = b"D1/", b"D2/", b"D", b"S/"
    out[-1] = b""
    return out


@gpu
def test_prefix_search_past_one_grid_row(engine):
    """40000 prefixes in one call: k2_large_run and place_unions cut it into grid rows of 32768
    groups (the y0 loops).  Both the host-buffer and the resident call; a 32769-prefix call
    launches more kernels than a 32768-prefix call of the same prefixes."""
    rng = np.random.default_rng(17)
    per_seg, segs = _row_workload(rng)
    prefixes = _row_prefixes(rng, 40000)
    exp = ref_prefix_search(per_seg, prefixes)
    assert_lists_equal(prefix_lists(engine, segs, prefixes), exp, prefixes)
    dsegs = [engine.upload(s) for s in segs]
    assert_lists_equal(prefix_lists(engine, dsegs, prefixes, dev=True), exp, prefixes)
    res = {}
    n_one = launches(engine, lambda: res.setdefault(1, prefix_lists(engine, dsegs, prefixes[:32768], dev=True)))
    n_two = launches(engine, lambda: res.setdefault(2, prefix_lists(engine, dsegs, prefixes[:32769], dev=True)))
    assert_lists_equal(res[1], exp[:32768], prefixes[:32768])
    assert_lists_equal(res[2], exp[:32769], prefixes[:32769])
    assert n_two > n_one
    for d in dsegs:
        d.release()


def _glob_workload(rng):
    """16 segments over 12000 ids, every id as the terms t<id>, t<id>a and t<id>ab; a segment
    holds each term with probability 0.3 and 1..4 values."""
    vocab = [b"t%05d%s" % (i, suf) for i in range(12000) for suf in (b"", b"a", b"ab")]
    per_seg = []
    for s in range(16):
        keep = np.nonzero(rng.random(len(vocab)) < 0.3)[0]
        lens = rng.integers(1, 5, size=len(keep))
        vals = rng.integers(0, 1 << 20, size=int(lens.sum())).astype(U32)
        off = np.concatenate([[0], np.cumsum(lens)])
        per_seg.append([(vocab[i], vals[off[j]:off[j + 1]]) for j, i in enumerate(keep)])
    return per_seg, [flat_segment(x) for x in per_seg]


@gpu
def test_pattern_terms_past_one_grid_row(engine):
    """ii2_pattern_terms with 37003 distinct globs: pattern_prepare (api.cu) compiles every
    distinct (kind, edits, prefix length, bytes) once, so nu = 37003 internal patterns, and K7
    sorts nu documents (k7_sort_distinct(..., (int)nu, ...) in k10_pattern.cu): more than one grid
    row of 32768.  `*`, t0* and t1* match far more than K7_TILE = 2048 term instances (about
    173000, 144000 and 29000 over 16 segments): their documents take the global stages and
    k7_tile_merge.  Repeated globs map to the same internal pattern."""
    rng = np.random.default_rng(18)
    per_seg, segs = _glob_workload(rng)
    globs = [b"t%05d" % i for i in range(12000)]                # literal: one term or none
    globs += [b"t%05d*" % i for i in range(12000)]              # three terms
    globs += [b"t%05da*" % i for i in range(12000)]             # two terms
    globs += [b"u%05d*" % i for i in range(1000)]               # none
    globs += [b"*", b"t0*", b"t1*"]
    nu = len(set(globs))
    assert nu == 37003 and nu > 32768
    globs += globs[:50] + [b"*"]                                # repeats
    ref_terms = RefPatternTerms(per_seg)
    exp = [ref_terms(g) for g in globs]
    assert sum(n for _, n, _, _ in exp[globs.index(b"t1*")]) > 2048
    got = engine.pattern_terms(segs, globs)
    assert len(got) == len(globs)
    for g, e, e_got in zip(globs, exp, got):
        assert e_got == e, g
    # the grid-row split of K7, witnessed: one distinct glob more launches more kernels
    dsegs = [engine.upload(s) for s in segs]
    first = globs[:32768]
    res = {}
    n_one = launches(engine, lambda: res.setdefault(1, engine.pattern_terms_dev(dsegs, first)))
    n_two = launches(engine, lambda: res.setdefault(2, engine.pattern_terms_dev(dsegs, globs[:32769])))
    assert len(set(globs[:32769])) == 32769
    assert res[1] == exp[:32768] and res[2] == exp[:32769]
    assert n_two > n_one
    for d in dsegs:
        d.release()


# ---------------------------------------------------------------- 5. K7 through ii2_ingest
# Terms that tie on K7's 16-byte key window: k7_cmp then compares the bytes past it when both
# terms are longer than 16, else the lengths.
TIE16 = b"0123456789abcdef"
TIE_TERMS = ([TIE16 + t for t in (b"", b"\0", b"\0\0", b"\x01", b"\xff", b"\xff\xff", b"a", b"a\0", b"ab")]
             + [b"x" * 15, b"x" * 15 + b"\0", b"x" * 15 + b"\0\0", b"x" * 16, b"x" * 17, b"x" * 14 + b"\xff"]
             + [b"\xff" * 15, b"\xff" * 16, b"\xff" * 17, b"\xff" * 16 + b"\0"]
             + [b"", b"\0", b"\0" * 15, b"\0" * 16, b"\0" * 17])
DOC_SIZES = [1, 2047, 2048, 2049, 4095, 4096, 4097, 6145, 16387]   # around K7_TILE = 2048 and 2 * 2048


def _ingest_vocab(rng):
    """Random terms over a few byte values (0x00, 0x01, 0x7f, 0x80, 0xfe, 0xff, 'a', 'b'), so
    that many tie on long prefixes, plus the 16-byte ties."""
    alphabet = np.array([0, 1, 0x7F, 0x80, 0xFE, 0xFF, 97, 98], dtype=np.uint8)
    lens = rng.integers(0, 36, size=3000)
    flat = alphabet[rng.integers(0, len(alphabet), size=int(lens.sum()))].tobytes()
    off = np.concatenate([[0], np.cumsum(lens)])
    rand = [flat[off[i]:off[i + 1]] for i in range(3000)]
    rand += [TIE16 + r for r in rand[:500]]                     # ties on the window, tails differ
    return rand + TIE_TERMS


def _ingest_docs(rng):
    vocab = _ingest_vocab(rng)
    docs = []
    vals = rng.integers(0, 1 << 20, size=len(DOC_SIZES)).astype(np.int64)
    vals[3] = vals[1]                                           # two documents share a value
    for n, val in zip(DOC_SIZES, vals):
        if n == 4097:
            # a term repeated 100 times at sorted positions 2000..2099: across the tile boundary
            terms = [b"A%05d" % i for i in range(2000)] + [b"M"] * 100 + [b"Z%05d" % i for i in range(1997)]
        elif n == 16387:
            # 200 repeats at sorted positions 4000..4199: across the 4096 boundary of the stages
            terms = [b"A%05d" % i for i in range(4000)] + [b"M"] * 200 + [b"Z%05d" % i for i in range(12187)]
        elif n == 6145:
            # every 16-byte tie, each three times, among random terms
            terms = TIE_TERMS * 3
            terms = terms + [vocab[int(i)] for i in rng.integers(0, len(vocab), n - len(terms))]
        else:
            terms = [vocab[int(i)] for i in rng.integers(0, len(vocab), n)]
        order = rng.permutation(len(terms))
        terms = [terms[int(i)] for i in order]
        assert len(terms) == n
        docs.append((terms, int(val)))
    e = lambda v: ([], v)
    # empty documents at the start, in a run in the middle, alone and at the end
    return ([e(1), e(2)] + docs[:3] + [e(3), e(4), e(5)] + docs[3:6] + [e(6)] + docs[6:]
            + [e(7), e(8)])


@gpu
def test_ingest_tile_sizes_and_ties(engine, orc, merge_path):
    """One ingest call with documents of 1, 2047, 2048, 2049, 4095, 4096, 4097, 6145 and 16387
    terms (K7_TILE = 2048: one tile, one record over, two and three tiles, a ragged eighth tile),
    every 16-byte tie of k7_cmp, repeated terms whose sorted run crosses a tile boundary, and empty
    documents at the start, in a run and at the end (k7_emit's o_first back-fill); with and
    without a removed set.  Then a call in which every document is empty."""
    rng = np.random.default_rng(19)
    docs = _ingest_docs(rng)
    values = np.array(sorted({v for t, v in docs if t}), dtype=U32)
    sparse = np.unique(np.append(values[::2], U32(17))).astype(U32)            # < 64 values: no bitmap
    dense = np.unique(np.concatenate([values[1::2], np.arange(0, 1 << 20, 7, dtype=U32)]))  # bitmap
    for rem in (None, sparse, dense):
        got = engine.ingest(docs, rem, decoded=True)
        check_merge_result(orc, got, ref_ingest(docs, rem), orc.ingest(docs, rem, decoded=True))
    empty = [([], v) for v in (5, 6, 7, 8)]
    for rem in (None, sparse):
        got = engine.ingest(empty, rem, decoded=True)
        assert got.terms_count == 0
        assert_merge_equal(got, orc.ingest(empty, rem, decoded=True))


@gpu
def test_ingest_limits(engine, orc):
    """1024 documents (kMaxSegs) are one call, 1025 are II2_ERR_UNSUPPORTED; a term of 65535
    bytes is accepted, one of 65536 is II2_ERR_UNSUPPORTED."""
    from inverted_index_2_b200.engine import EngineError
    docs = [([b"d%04d" % (i % 37), b"all"], i) for i in range(1024)]
    got = engine.ingest(docs, None, decoded=True)
    check_merge_result(orc, got, ref_ingest(docs), orc.ingest(docs, None, decoded=True))
    with pytest.raises(EngineError) as e:
        engine.ingest(docs + [([b"one_more"], 5)], None)
    assert e.value.code == A.II2_ERR_UNSUPPORTED
    longest = [([b"L" * 65535, b"a"], 3), ([b"L" * 65535, b"b"], 4)]
    got = engine.ingest(longest, None, decoded=True)
    check_merge_result(orc, got, ref_ingest(longest), orc.ingest(longest, None, decoded=True))
    with pytest.raises(EngineError) as e:
        engine.ingest([([b"a"], 1), ([b"L" * 65536], 2)], None)
    assert e.value.code == A.II2_ERR_UNSUPPORTED
