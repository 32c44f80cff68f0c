"""GPU parity tests: the CUDA path behind the C-ABI (libii2.so) against the CPU oracle on the
same seeded inputs, bit-exact (integer / byte work — no tolerance anywhere), plus the
reference's own known-answer vectors run through the host mirror on the CUDA engine."""
import threading

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A
from inverted_index_2_b200 import synth
from inverted_index_2_b200.flat import FlatSegment
from scenario import (check_roaring_case, load_roaring_vectors, load_vectors, roaring_case_values,
                      run_index_scenario, run_shard_scenario)

pytestmark = pytest.mark.gpu
V = load_vectors()


def assert_merge_equal(got, exp, decoded=True):
    assert got.terms_count == exp.terms_count
    assert np.array_equal(got.term_off, exp.term_off)
    assert np.array_equal(got.term_bytes, exp.term_bytes)
    assert got.val_size == exp.val_size
    assert np.array_equal(got.val_off, exp.val_off)
    assert np.array_equal(got.val_bytes, exp.val_bytes)
    assert got.min_term == exp.min_term and got.max_term == exp.max_term
    assert got.terms_merged == exp.terms_merged
    assert got.postings_in == exp.postings_in
    assert got.postings_out == exp.postings_out
    if decoded:
        assert np.array_equal(got.post_off, exp.post_off)
        assert np.array_equal(got.post, exp.post)


def assert_read_equal(got, exp):
    assert got.n_terms == exp.n_terms
    assert np.array_equal(got.term_off, exp.term_off)
    assert np.array_equal(got.term_bytes, exp.term_bytes)
    assert np.array_equal(got.post_off, exp.post_off)
    assert np.array_equal(got.post, exp.post)


# ---------------------------------------------------------------- reference known answers
@pytest.mark.parametrize("sc", V["shard_scenarios"], ids=lambda s: s["name"])
def test_shard_scenarios(engine, sc):
    run_shard_scenario(engine, sc)


@pytest.mark.parametrize("sc", V["index_scenarios"], ids=lambda s: s["name"])
def test_index_scenarios(engine, sc):
    run_index_scenario(engine, sc)


@pytest.mark.parametrize("w", V["writer"], ids=lambda s: s["name"])
def test_writer_reader_roundtrip(engine, w):
    items = [(t.encode(), v) for t, v in w["items"]]
    if w["mode"] == "direct":
        seg = FlatSegment(*FlatSegment._pack_terms([t for t, _ in items]), A.II2_SEG_DIRECT,
                          val_off=np.array([v[0] for _, v in items], dtype=np.uint64))
    else:
        seg = FlatSegment.from_items(items).to_val(engine.intcomp_encode_batch)
        assert seg.val_off[1] == seg.val_off[2]  # empty list -> zero bytes (writer_test.go:15)
    assert engine.read_range([seg]).items() == items


@pytest.mark.parametrize("b", V["bitmask"], ids=lambda s: s["name"])
def test_bitmask_known_answers(engine, b):
    bm = engine.bitmask(b["init"])
    enc = [bm.put(p) for p in b["puts"]]
    assert bm.get(enc[0] + enc[1]).tolist() == b["get_concat_first"]
    assert bm.get(enc[1]).tolist() == b["get_second_index_order"]
    assert sorted(bm.get(enc[1]).tolist()) == b["get_second_sorted"]
    assert bm.all_values().tolist() == b["all_values"]


# ---------------------------------------------------------------- merge vs oracle
MERGE_CASES = [
    # terms, segs, postings, universe, removed_frac, presence
    (50, 2, 200, 1 << 8, 0.0, 0.7),
    (50, 3, 400, 1 << 8, 0.3, 0.7),
    (3000, 4, 20000, 1 << 12, 0.05, 0.5),
    (3000, 64, 150000, 1 << 16, 0.05, 0.5),
    (20000, 8, 400000, 1 << 16, 0.05, 0.5),
    (1000, 256, 300000, 1 << 14, 0.05, 0.3),
    (200, 16, 400000, 1 << 20, 0.05, 0.9),   # long lists: warp + CTA union paths
    (100000, 5, 600000, 1 << 24, 0.0, 0.5),
    (100000, 5, 600000, 1 << 24, 0.05, 0.5),  # removed set answered from the bitmap
]


@pytest.fixture(params=["general", "fused"])
def merge_path(request, monkeypatch):
    """Both bucket pipelines: the general kernels (K1b -> K2b -> K6, default) and the fused
    bucket kernel (k12_fused.cu, II2_FUSED=1) with its dense placement."""
    # (unset, the library picks the fused path for small calls only: force both ways)
    monkeypatch.setenv("II2_FUSED", "1" if request.param == "fused" else "0")
    return request.param


@pytest.mark.parametrize("case", MERGE_CASES, ids=lambda c: "t%d_s%d_p%d_u%d_r%g" % c[:5])
def test_merge_matches_oracle(engine, orc, case, merge_path):
    nt, ns, npost, uni, rf, pres = case
    w = synth.make_workload(nt, ns, npost, universe=uni, removed_frac=rf, presence=pres,
                            seed=nt + ns, max_len=4096 if nt <= 200 else 64)
    exp = orc.merge(w.segments, w.removed, decoded=True)
    got = engine.merge(w.segments, w.removed, decoded=True)
    assert_merge_equal(got, exp)
    # independent numpy answer (no oracle code involved)
    terms, vals, poff = w.expected_union(w.removed)
    assert np.array_equal(got.post, vals) and np.array_equal(got.post_off, poff)


def test_merge_all_segment_modes(engine, orc, merge_path):
    """DECODED, raw `_val` (file/reader.go:79-100) and direct mode (:73-77) inputs mixed."""
    w = synth.make_workload(5000, 6, 60000, universe=1 << 14, seed=7)
    segs = list(w.segments)
    segs[1] = segs[1].to_val(orc.intcomp_encode_batch)
    segs[4] = segs[4].to_val(orc.intcomp_encode_batch)
    tb, off = synth.gather_terms(w.term_bytes, w.term_off, np.arange(0, 5000, 3))
    segs.append(FlatSegment(tb, off, A.II2_SEG_DIRECT,
                            val_off=np.full(len(off) - 1, (7 << 32) | 123, dtype=np.uint64)))
    exp = orc.merge(segs, w.removed, decoded=True)
    got = engine.merge(segs, w.removed, decoded=True)
    assert_merge_equal(got, exp)


def test_merged_segment_reads_back(engine, orc):
    """The `_val` stream the GPU writes decodes (GPU and oracle decoder) to the merged lists."""
    w = synth.make_workload(4000, 5, 200000, universe=1 << 18, seed=11, max_len=1000)
    got = engine.merge(w.segments, w.removed, decoded=True)
    seg = got.to_segment()
    for backend in (engine, orc):
        rr = backend.read_range([seg])
        assert np.array_equal(rr.post, got.post) and np.array_equal(rr.post_off, got.post_off)
        assert np.array_equal(rr.term_bytes, got.term_bytes)


def test_single_source_passthrough_quirk(engine, orc, merge_path):
    """Survey Q4: a term seen in ONE segment is neither sorted nor deduped
    (file/types.go:14-22 only runs on equal terms); shared terms are."""
    a = FlatSegment.from_items([(b"only_a", [9, 3, 3, 7]), (b"shared", [5, 1, 5])])
    b = FlatSegment.from_items([(b"only_b", [2, 2, 1]), (b"shared", [1, 9, 9])])
    exp = orc.merge([a, b], None, decoded=True)
    got = engine.merge([a, b], None, decoded=True)
    assert_merge_equal(got, exp)
    assert got.as_dict() == {b"only_a": [9, 3, 3, 7], b"only_b": [2, 2, 1], b"shared": [1, 5, 9]}
    # one segment alone: everything passes through, removed values filtered in place
    exp1 = orc.merge([a], np.array([3], dtype=np.uint32), decoded=True)
    got1 = engine.merge([a], np.array([3], dtype=np.uint32), decoded=True)
    assert_merge_equal(got1, exp1)
    assert got1.as_dict() == {b"only_a": [9, 7], b"shared": [5, 1, 5]}


def test_merge_edge_cases(engine, orc, merge_path):
    empty = FlatSegment.from_items([])
    one = FlatSegment.from_items([(b"", [4]), (b"a", []), (b"b", [1, 2])])
    two = FlatSegment.from_items([(b"", [4, 5]), (b"a", []), (b"c" * 300, [8])])
    for segs, removed in [
        ([], None),
        ([empty], None),
        ([empty, empty], None),
        ([one], None),
        ([one, two], None),
        ([one, two, empty], np.array([4, 5, 8, 1, 2], dtype=np.uint32)),  # everything removed
        ([one, two], np.array([4, 4, 4, 8], dtype=np.uint32)),            # duplicates in removed (Q6)
    ]:
        if removed is not None:
            removed = np.sort(removed)
        exp = orc.merge(segs, removed, decoded=True)
        got = engine.merge(segs, removed, decoded=True)
        assert_merge_equal(got, exp)
    # all removed -> no segment is written (lazy writer, shard.go:197-205) but min/max are set (Q3)
    got = engine.merge([one, two], np.array([1, 2, 4, 5, 8], dtype=np.uint32), decoded=True)
    assert got.terms_count == 0 and got.val_size == 0
    assert got.min_term == b"" and got.max_term == b"c" * 300


def test_merge_long_and_similar_terms(engine, orc, merge_path):
    """Terms that only differ past the 16-byte key window, 1-byte terms (shard 0000, Q7),
    prefixes of one another, and > 2048 instances sharing one long prefix."""
    rng = np.random.default_rng(5)
    base = b"commonprefix/" * 3
    pool = sorted({base + bytes(rng.integers(97, 101, size=int(rng.integers(0, 12))).tolist())
                   for _ in range(3000)} | {b"a", b"b", b"ab", b"abc", b"\x00", b"\x00\x00", b"\xff"})
    segs = []
    for s in range(5):
        pick = [t for t in pool if rng.random() < 0.6]
        segs.append(FlatSegment.from_items(
            [(t, sorted(set(rng.integers(0, 500, size=int(rng.integers(1, 6))).tolist())))
             for t in pick]))
    removed = np.arange(0, 500, 7, dtype=np.uint32)
    assert_merge_equal(engine.merge(segs, removed, decoded=True),
                       orc.merge(segs, removed, decoded=True))
    lo, hi = pool[len(pool) // 3], pool[2 * len(pool) // 3]
    assert_read_equal(engine.read_range(segs, lo, hi), orc.read_range(segs, lo, hi))


def test_heavy_terms_multi_cta_union(engine, orc, merge_path):
    """Lists far larger than one CTA's shared memory (survey §7 hard part 2): the global
    bitonic path, the bitmap path of long dense unions ("heavy": 350k values below 2^20), heavy
    single-source lists (pass-through, survey Q4) and a long sparse union."""
    rng = np.random.default_rng(9)
    segs = []
    for s in range(6):
        items = [(b"heavy", np.unique(rng.integers(0, 1 << 20, size=60000)).tolist()),
                 (b"medium", np.unique(rng.integers(0, 1 << 16, size=3000)).tolist()),
                 (b"small%d" % s, [s, s + 1])]
        if s == 0:
            items.append((b"solo_heavy", rng.integers(0, 1 << 20, size=50000).tolist()))
        if s == 1:  # long, dense, ONE source: passes through unsorted, never the bitmap path
            items.append((b"solo_dense", rng.integers(0, 1 << 18, size=70000).tolist()))
        if s >= 4:  # long but sparse over the whole u32 range: stays on the sort path
            items.append((b"sparse", rng.integers(0, 1 << 32, size=40000, dtype=np.uint64).tolist()))
        segs.append(FlatSegment.from_items(sorted(items)))
    removed = np.unique(rng.integers(0, 1 << 20, size=50000)).astype(np.uint32)
    assert_merge_equal(engine.merge(segs, removed, decoded=True),
                       orc.merge(segs, removed, decoded=True))


def test_mid_and_medium_terms(engine, orc, merge_path):
    """Terms of 257 ... 4097+ values: one warp per term with 32 values per lane up to 1024
    (k2_mwarp_kernel), one CTA per term up to 4096 (k2_medium_kernel), the multi-CTA path beyond;
    every boundary, many and few sources, a source longer than 32 values, single-source
    pass-through with duplicates (survey Q4), values that all fall to the removed filter, with and
    without a removed bitmap (ids >= 2^29 force the binary-search filter)."""
    rng = np.random.default_rng(21)
    for hi_bits, rem_n in ((20, 30000), (31, 500)):
        sizes = [257, 300, 511, 512, 513, 1000, 1023, 1024, 1025, 1500, 2048, 4095, 4096, 4097, 6000]
        nseg = 12
        per_seg = [[] for _ in range(nseg)]
        for ti, total in enumerate(sizes):
            name = b"t%05d" % ti
            k = [2, 12, 5][ti % 3]                       # sources of the term
            cuts = np.sort(rng.integers(0, total + 1, size=k - 1))
            lens = np.diff(np.concatenate([[0], cuts, [total]]))
            for s_i, n in zip(rng.permutation(nseg)[:k], lens):
                vals = np.unique(rng.integers(0, 1 << hi_bits, size=int(n), dtype=np.int64)).tolist()
                per_seg[int(s_i)].append((name, vals))   # overlap between sources: the union dedups
        per_seg[0].append((b"u_solo", rng.integers(0, 1 << hi_bits, size=900, dtype=np.int64).tolist()))   # unsorted, kept
        per_seg[1].append((b"v_solo", [7, 7, 3] * 700))                                                   # CTA path, kept
        gone = np.arange(1000, 1700, dtype=np.int64)
        per_seg[2].append((b"w_gone", gone[:400].tolist()))
        per_seg[3].append((b"w_gone", gone[300:].tolist()))
        segs = [FlatSegment.from_items(sorted(x)) for x in per_seg]
        removed = np.unique(np.concatenate([rng.integers(0, 1 << hi_bits, size=rem_n, dtype=np.int64), gone])
                            ).astype(np.uint32)
        assert_merge_equal(engine.merge(segs, removed, decoded=True), orc.merge(segs, removed, decoded=True))
        assert_read_equal(engine.read_range(segs, b"t00003", b"v"), orc.read_range(segs, b"t00003", b"v"))


def test_medium_terms_of_many_short_sources(engine, orc, merge_path):
    """CTA-per-term union, the other gather: a term held by hundreds of segments with a few
    values each (sources located by search instead of a warp per source), terms that end exactly
    on a run / merge boundary of the shared-memory sort (512, 1024, 2048, 4096 values), empty
    leading and trailing sources, heavy overlap between sources."""
    rng = np.random.default_rng(77)
    nseg = 420
    per_seg = [[] for _ in range(nseg)]
    plans = [(b"a_1100", 1100, 300), (b"b_1536", 1536, 420), (b"c_2048", 2048, 400), (b"d_2049", 2049, 257),
             (b"e_3000", 3000, 420), (b"f_4096", 4096, 420), (b"g_1025", 1025, 129), (b"h_overlap", 2600, 420)]
    for name, total, k in plans:
        cuts = np.sort(rng.integers(0, total + 1, size=k - 1))
        lens = np.diff(np.concatenate([[0], cuts, [total]]))
        lens[0] = 0 if name != b"g_1025" else lens[0]   # an empty list in a segment that has the term
        uni = 1 << 12 if name == b"h_overlap" else 1 << 22
        for s_i, n in zip(rng.permutation(nseg)[:k], lens):
            vals = np.unique(rng.integers(0, uni, size=int(n), dtype=np.int64)).tolist()
            per_seg[int(s_i)].append((name, vals))
    for s_i in range(nseg):   # every segment needs at least one term
        per_seg[s_i].append((b"z_pad%03d" % (s_i % 7), [s_i, s_i + 1]))
    segs = [FlatSegment.from_items(sorted(x)) for x in per_seg]
    removed = np.unique(rng.integers(0, 1 << 22, size=40000, dtype=np.int64)).astype(np.uint32)
    assert_merge_equal(engine.merge(segs, removed, decoded=True), orc.merge(segs, removed, decoded=True))
    assert_merge_equal(engine.merge(segs, removed, decoded=False), orc.merge(segs, removed, decoded=False),
                       decoded=False)
    # the same terms as point reads over 420 segments (one kernel: lookups + the CTA union, with
    # the gather by search; 4096 values is its capacity, d_2049 has more sources than a bucket row)
    for name, _, _ in plans:
        assert_read_equal(engine.read_range(segs, name, name, removed=removed),
                          orc.read_range(segs, name, name, removed=removed))
        assert_read_equal(engine.read_range(segs, name, name), orc.read_range(segs, name, name))


def test_merge_pipelined_by_term_range(engine, orc, monkeypatch):
    """ii2_merge over host buffers cuts the term space into ranges and overlaps staging with
    the kernels; the concatenated result is the single-shot result, also when the output
    estimate taken from the first range is too small (exact re-copy) and for slices of
    segments that start past offset 0."""
    w = synth.make_workload(30000, 7, 400000, universe=1 << 16, removed_frac=0.1, seed=31,
                            max_len=300)
    segs = list(w.segments)
    segs.append(FlatSegment.from_items([(b"zzzz_only_here", [5, 3, 3])]))  # single-source tail
    exp = orc.merge(segs, w.removed, decoded=True)
    for parts, slack in (("1", None), ("2", None), ("5", None), ("8", "0.05"), ("3", "0.0")):
        monkeypatch.setenv("II2_MERGE_PARTS", parts)
        if slack is None:
            monkeypatch.delenv("II2_MERGE_SLACK", raising=False)
        else:
            monkeypatch.setenv("II2_MERGE_SLACK", slack)
        assert_merge_equal(engine.merge(segs, w.removed, decoded=True), exp)
        assert_merge_equal(engine.merge(segs, None, decoded=False),
                           orc.merge(segs, None, decoded=False), decoded=False)
    # pinned host arrays are gathered by a kernel instead of the copy engines
    import torch
    keep = []

    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()
    psegs = [FlatSegment(pinned(x.term_bytes), pinned(x.term_off), x.mode, post=pinned(x.post),
                         post_off=pinned(x.post_off)) for x in segs]
    for parts in ("2", "7"):
        monkeypatch.setenv("II2_MERGE_PARTS", parts)
        monkeypatch.delenv("II2_MERGE_SLACK", raising=False)
        assert_merge_equal(engine.merge(psegs, w.removed, decoded=True), exp)
    # both staging paths at three ranges: the gather kernel (pinned) and the copy engine (pageable)
    monkeypatch.setenv("II2_MERGE_PARTS", "3")
    assert_merge_equal(engine.merge(psegs, w.removed, decoded=True), exp)
    assert_merge_equal(engine.merge(segs, w.removed, decoded=True), exp)
    # as many ranges as the largest segment has terms: every cut is a different term
    tiny = [FlatSegment.from_items([(b"a", [1]), (b"b", [2]), (b"c", [3])]),
            FlatSegment.from_items([(b"b", [5]), (b"d", [1])])]
    for parts in ("2", "3"):
        monkeypatch.setenv("II2_MERGE_PARTS", parts)
        assert_merge_equal(engine.merge(tiny, None, decoded=True), orc.merge(tiny, None, decoded=True))
    # everything removed in the first ranges: min/max still come from the first / last range
    monkeypatch.setenv("II2_MERGE_PARTS", "4")
    monkeypatch.delenv("II2_MERGE_SLACK", raising=False)
    allrem = np.arange(0, 1 << 16, dtype=np.uint32)
    assert_merge_equal(engine.merge(segs, allrem, decoded=True), orc.merge(segs, allrem, decoded=True))
    monkeypatch.delenv("II2_MERGE_PARTS", raising=False)


@pytest.mark.parametrize("bucket", ["64", "200", "32", "1024"])
def test_merge_with_small_buckets(engine, orc, monkeypatch, bucket, merge_path):
    """A small call cut into many buckets (II2_BUCKET sets the instances per bucket): unequal
    segment sizes, a tiny segment and a range read are covered."""
    monkeypatch.setenv("II2_BUCKET", bucket)
    w = synth.make_workload(40000, 9, 500000, universe=1 << 18, removed_frac=0.07, seed=91,
                            max_len=200)
    segs = list(w.segments)
    segs.append(FlatSegment.from_items([(b"a", [9, 1]), (b"zzzzzzzz", [7])]))      # a tiny segment
    assert_merge_equal(engine.merge(segs, w.removed, decoded=True), orc.merge(segs, w.removed, decoded=True))
    lo = synth.term_at(w.term_bytes, w.term_off, 3000)
    hi = synth.term_at(w.term_bytes, w.term_off, 31000)
    assert_read_equal(engine.read_range(segs, lo, hi), orc.read_range(segs, lo, hi))
    monkeypatch.delenv("II2_BUCKET", raising=False)


def test_merge_pipelined_val_views(engine, orc, monkeypatch):
    """ii2_merge over `_val` views — what a Go caller holds: the mmap of <key>_val and the FST
    outputs (file/reader.go:50-52,79-100) — staged per term range and decoded on the device, one
    batched K3a call per range: equal to the oracle for 1, 2 and 5 ranges, with 64-bit byte
    offsets, with 32-bit word offsets (val_woff32), mixed with decoded views, and from pinned
    memory (gather kernel) as well as pageable memory (copy engines)."""
    w = synth.make_workload(30000, 7, 400000, universe=1 << 16, removed_frac=0.1, seed=33, max_len=300)
    segs = list(w.segments)
    segs.append(FlatSegment.from_items([(b"zzzz_only_here", [5, 3, 3])]))
    exp = orc.merge(segs, w.removed, decoded=True)
    vsegs = [x.to_val(orc.intcomp_encode_batch) for x in segs]
    v32 = [x.with_woff32() for x in vsegs]
    mixed = [a if i % 2 else b for i, (a, b) in enumerate(zip(vsegs, segs))]
    import torch
    keep = []

    def pinned(a):
        if a is None:
            return None
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()
    pv32 = [FlatSegment(pinned(x.term_bytes), pinned(x.term_off), x.mode, val_bytes=pinned(x.val_bytes),
                        val_size=x.val_size, val_woff32=pinned(x.val_woff32)) for x in v32]
    for parts in ("1", "2", "5"):
        monkeypatch.setenv("II2_MERGE_PARTS", parts)
        for views in (vsegs, v32, mixed, pv32):
            assert_merge_equal(engine.merge(views, w.removed, decoded=True), exp)
    # a corrupt FST output (not 4-byte aligned / past the file) is refused, not decoded
    from inverted_index_2_b200.engine import EngineError
    bad = list(vsegs)
    off = bad[2].val_off.copy()
    off[len(off) // 2] += 2
    bad[2] = FlatSegment(bad[2].term_bytes, bad[2].term_off, bad[2].mode, val_bytes=bad[2].val_bytes,
                         val_off=off, val_size=bad[2].val_size)
    monkeypatch.setenv("II2_MERGE_PARTS", "3")
    with pytest.raises(EngineError):
        engine.merge(bad, w.removed, decoded=True)
    monkeypatch.delenv("II2_MERGE_PARTS", raising=False)
    assert_merge_equal(engine.merge(v32, w.removed, decoded=True), exp)   # single shot


def test_merge_pipelined_unaligned_term_bytes(engine, orc, monkeypatch):
    """A caller's term_bytes may start at any address (a Go sub-slice, an mmap offset): on the
    copy-engine path every slice lands at the phase of its first offset, so the moved term base
    stays 4-byte aligned for the key loads (api.cu place())."""
    w = synth.make_workload(20000, 5, 200000, universe=1 << 16, removed_frac=0.1, seed=77)
    exp = orc.merge(w.segments, w.removed, decoded=True)
    odd = []
    for shift, x in enumerate(w.segments):
        buf = np.empty(len(x.term_bytes) + 8, dtype=np.uint8)
        view = buf[1 + (shift % 3):1 + (shift % 3) + len(x.term_bytes)]
        view[:] = x.term_bytes
        assert view.ctypes.data % 4 != 0
        odd.append(FlatSegment(view, x.term_off, x.mode, post=x.post, post_off=x.post_off))
    for parts in ("1", "3", "6"):
        monkeypatch.setenv("II2_MERGE_PARTS", parts)
        assert_merge_equal(engine.merge(odd, w.removed, decoded=True), exp)
    monkeypatch.delenv("II2_MERGE_PARTS", raising=False)


def test_merge_rejects_corrupt_offsets_and_unsorted_removed(engine, monkeypatch):
    """Raw C-ABI input is checked, not trusted: non-monotone offsets are II2_ERR_INVALID on the
    pipelined path too (before any size is computed from them), empty segments with NULL arrays
    are accepted, an unsorted removed list is refused."""
    from inverted_index_2_b200.engine import EngineError
    good = FlatSegment.from_items([(b"a%04d" % i, [i, i + 1]) for i in range(200)])
    bad_toff = good.term_off.copy()
    bad_toff[50] = bad_toff[120]          # not monotone
    bad = FlatSegment(good.term_bytes, bad_toff, good.mode, post=good.post, post_off=good.post_off)
    empty = FlatSegment.from_items([])
    for parts in ("1", "4"):
        monkeypatch.setenv("II2_MERGE_PARTS", parts)
        with pytest.raises(EngineError) as e:
            engine.merge([good, bad], None, decoded=True)
        assert e.value.code == A.II2_ERR_INVALID
        r = engine.merge([good, empty, good], None, decoded=True)
        assert r.terms_count == 200
    monkeypatch.delenv("II2_MERGE_PARTS", raising=False)
    with pytest.raises(EngineError) as e:
        engine.merge([good], np.array([5, 3, 900000, 7] * 40, dtype=np.uint32), decoded=True)
    assert e.value.code == A.II2_ERR_INVALID


def test_union_width_boundaries(engine, orc, merge_path):
    """Union kernel paths: two terms per warp (< 128 values), one term per warp (128..256),
    multi-CTA (> 256); single-source terms (unsorted, duplicates kept: Q4) paired with
    multi-source ones in the same warp; values needing 5 var-byte bytes and negative deltas."""
    rng = np.random.default_rng(21)
    lens = [0, 1, 2, 7, 8, 9, 15, 16, 17, 63, 64, 65, 120, 126, 127, 128, 129, 130, 200, 255, 256,
            257, 300, 511, 512, 513]
    items = [[], [], []]
    for i, L in enumerate(lens):
        for mode in range(4):
            term = b"t%03d_%d" % (i, mode)
            if mode == 0:    # three sources that share values: union shrinks
                pool = rng.integers(0, max(4, 2 * L), size=L).astype(np.uint32)
                cut = sorted(rng.integers(0, L + 1, size=2).tolist())
                parts = [pool[:cut[0]], pool[cut[0]:cut[1]], pool[cut[1]:]]
                for s in range(3):
                    items[s].append((term, np.unique(parts[s]).tolist()))
            elif mode == 1:  # single source, unsorted with duplicates, huge values
                vals = rng.integers(0, 1 << 32, size=L, dtype=np.uint64).astype(np.uint32)
                if L > 2:
                    vals[1] = vals[0]
                items[i % 3].append((term, vals.tolist()))
            elif mode == 2:  # two sources, exactly L distinct values in total (nothing merges)
                vals = rng.choice(1 << 30, size=L, replace=False).astype(np.uint32) * np.uint32(4)
                items[0].append((term, np.sort(vals[: L // 2]).tolist()))
                items[1].append((term, np.sort(vals[L // 2:]).tolist()))
            else:            # same list in every segment
                vals = np.unique(rng.integers(0, 1 << 20, size=L)).tolist()
                for s in range(3):
                    items[s].append((term, vals))
    segs = [FlatSegment.from_items(sorted(it)) for it in items]
    for removed in (None, np.unique(rng.integers(0, 1 << 12, size=600)).astype(np.uint32),
                    np.array([1, 5, 4000000000], dtype=np.uint32)):   # last: no bitmap (sparse)
        exp = orc.merge(segs, removed, decoded=True)
        got = engine.merge(segs, removed, decoded=True)
        assert_merge_equal(got, exp)
        assert_read_equal(engine.read_range(segs), orc.read_range(segs))


# ---------------------------------------------------------------- range reads vs oracle
def test_read_range_matches_oracle(engine, orc, merge_path):
    w = synth.make_workload(20000, 12, 300000, universe=1 << 16, seed=21)
    n = 20000
    t = lambda i: synth.term_at(w.term_bytes, w.term_off, i)
    bounds = [(None, None), (t(0), t(n - 1)), (t(100), t(100)), (t(5000), t(5200)),
              (None, t(3000)), (t(15000), None), (t(9000) + b"~", t(9100) + b"~"),
              (b"zzzzzzzzzzzzzzzzzzzzzzzz", None), (None, b"A"), (t(300), t(200)), (b"", None)]
    for lo, hi in bounds:
        assert_read_equal(engine.read_range(w.segments, lo, hi), orc.read_range(w.segments, lo, hi))
    # benchmark composition of config 3: read + Merge-style filter (survey Q2)
    for lo, hi in bounds[:6]:
        assert_read_equal(engine.read_range(w.segments, lo, hi, removed=w.removed),
                          orc.read_range(w.segments, lo, hi, removed=w.removed))


def test_point_reads(engine, orc, merge_path):
    """min == max: one kernel does the whole read (k4_point_kernel: <= 4096 values, terms <= 8192
    bytes); when it declines, or the term is longer, the call continues as an ordinary read.  A
    term that is everywhere, in one segment, nowhere (between terms, before the first, after the
    last), the empty term; with and without the removed filter; terms of > 4096 values; a term of
    > 256 values (the bucket is deferred to the general kernels); a term of > 8192 bytes in two
    segments and one that is absent; one-term windows with min < max (the ordinary kernels)."""
    rng = np.random.default_rng(5)
    nseg = 9
    per_seg = [[] for _ in range(nseg)]
    for s_i in range(nseg):
        per_seg[s_i].append((b"everywhere", sorted(set(rng.integers(0, 5000, size=20).tolist()))))
        per_seg[s_i].append((b"filler%02d" % s_i, [s_i, s_i + 100]))
        per_seg[s_i].append((b"big", sorted(set(rng.integers(0, 1 << 20, size=700).tolist()))))    # 6300 > 4096 in
        per_seg[s_i].append((b"mid", sorted(set(rng.integers(0, 1 << 20, size=60).tolist()))))     # ~540 values: deferred
    per_seg[3].append((b"only3", [9, 8, 8, 1]))       # single source: order and duplicates kept
    per_seg[5].append((b"hollow", []))                # present, no values
    per_seg[6].append((b"hollow", []))
    per_seg[7].append((b"solo_big", rng.integers(0, 1 << 20, size=5000).tolist()))   # one source, > 4096
    per_seg[4].append((b"", [4, 2]))                  # the empty term
    long_term = b"L" * 9000                           # longer than the point kernel stages
    per_seg[1].append((long_term, [1, 3]))
    per_seg[2].append((long_term, [2, 3, 70]))
    segs = [FlatSegment.from_items(sorted(x)) for x in per_seg]
    removed = np.unique(rng.integers(0, 5000, size=800)).astype(np.uint32)
    terms = [b"everywhere", b"only3", b"", b"big", b"mid", b"filler04", b"absent", b"everywhera", b"zzz",
             b"\x00", b"filler", b"hollow", b"solo_big", long_term, b"L" * 8999 + b"M"]
    windows = [(t, t) for t in terms] + [(t, t + b"\x00") for t in (b"everywhere", b"big")]
    for lo, hi in windows:
        assert_read_equal(engine.read_range(segs, lo, hi), orc.read_range(segs, lo, hi))
        assert_read_equal(engine.read_range(segs, lo, hi, removed=removed),
                          orc.read_range(segs, lo, hi, removed=removed))
    # resident segments: the same through the device API, results released between calls
    dsegs = [engine.upload(x) for x in segs]
    for t in terms:
        r = engine.read_range_dev(dsegs, t, t, None)
        assert_read_equal(r.download_read(), orc.read_range(segs, t, t))
        r.release()
    for d in dsegs:
        d.release()


def test_window_search_boundaries(engine, orc):
    """The 32-way warp search of the range windows (K4) and of the prefix windows (K5): segment
    sizes around the lane count and its powers (0, 1, 31..34, 1088..1090 = 33^2 +- 1, 36000 >
    33^3), bounds on every kind of position — a member, between members, before the first,
    after the last, equal min and max, min > max."""
    rng = np.random.default_rng(1234)
    tb, off = synth.make_terms(40000, 0x1EE7)
    sizes = [0, 1, 2, 31, 32, 33, 34, 65, 1088, 1089, 1090, 36000]
    segs = []
    for n in sizes:
        ids = np.sort(rng.choice(40000, size=n, replace=False))
        stb, stoff = synth.gather_terms(tb, off, ids)
        post = rng.integers(0, 1 << 20, size=n, dtype=np.int64).astype(np.uint32)
        segs.append(FlatSegment(stb, stoff, A.II2_SEG_DECODED, post=post,
                                post_off=np.arange(n + 1, dtype=np.uint64)))
    t = lambda i: synth.term_at(tb, off, i)
    picks = [0, 1, 2, 30, 31, 32, 33, 34, 1000, 1088, 1089, 20000, 39998, 39999]
    bounds = [(None, None), (b"", None), (None, b""), (b"\x00", b"\x01"), (b"zzzz", None), (None, b"zzzz")]
    for i in picks:
        bounds += [(t(i), t(i)), (t(i), None), (None, t(i)), (t(i) + b"\x00", None), (None, t(i)[:-1]),
                   (t(i), t(min(39999, i + 40))), (t(i)[:-1], t(min(39999, i + 33)) + b"~")]
    bounds.append((t(500), t(400)))
    for lo, hi in bounds:
        assert_read_equal(engine.read_range(segs, lo, hi), orc.read_range(segs, lo, hi))
    prefixes = [b"", t(0), t(39999), t(1089)[:4], t(20000)[:3], t(33)[:2], t(32)[:1], b"zzzz", b"\x00",
                t(31) + b"x"]
    _assert_prefix_equal(engine.prefix_search(segs, prefixes), orc.prefix_search(segs, prefixes))


def test_read_keeps_empty_lists(engine, orc, merge_path):
    seg = FlatSegment.from_items([(b"t1", [10, 500, 300]), (b"t2", []), (b"t3", [66, 5513])])
    got = engine.read_range([seg])
    assert got.items() == [(b"t1", [10, 500, 300]), (b"t2", []), (b"t3", [66, 5513])]
    assert_read_equal(got, orc.read_range([seg]))


# ---------------------------------------------------------------- PrefixSearch vs oracle
def _assert_prefix_equal(got, exp):
    assert sorted(got) == sorted(exp)
    for k in exp:
        assert [int(x) for x in got[k]] == list(exp[k]), k


def test_prefix_search_matches_oracle(engine, orc):
    """ii2_prefix_search against the literal scan of inverted_index.go:239-292: prefixes of
    every length (empty = everything, one byte, a whole term, longer than any term), absent
    prefixes (omitted from the map), duplicates, unsorted input order."""
    w = synth.make_workload(6000, 7, 90000, universe=1 << 16, seed=77)
    t = lambda i: synth.term_at(w.term_bytes, w.term_off, i)
    prefixes = [b"", b"a", b"Z", b"ab", t(10), t(10)[:5], t(4000)[:3], t(5999), t(0) + b"x",
                b"zzzzzz", b"\x00", t(123)[:2], t(123)[:2], b"q", t(77) + b"~" * 40]
    got = engine.prefix_search(w.segments, prefixes)
    exp = orc.prefix_search(w.segments, prefixes)
    assert b"" in exp and b"zzzzzz" not in exp
    _assert_prefix_equal(got, exp)
    # resident segments, one prefix per call
    dsegs = [engine.upload(s) for s in w.segments]
    for p in (b"", b"b", t(2000)[:4]):
        _assert_prefix_equal(engine.prefix_search_dev(dsegs, [p]), orc.prefix_search(w.segments, [p]))


def test_prefix_search_edge_cases(engine, orc):
    """One segment with unsorted and duplicated values (the final sort + compact applies even
    to a single source, unlike the merge's pass-through); a matching term with an empty list
    still creates the key; no segments / no prefixes; values at the u32 limits."""
    seg = FlatSegment.from_items([(b"aa", [9, 3, 3, 7]), (b"ab", []), (b"b", [0xFFFFFFFF, 0, 5]),
                                  (b"ba", [5, 5, 1])])
    for prefixes in ([b"a"], [b"ab"], [b"b", b"a", b"c"], [b"", b"ba"], []):
        got = engine.prefix_search([seg], prefixes)
        exp = orc.prefix_search([seg], prefixes)
        _assert_prefix_equal(got, exp)
    assert engine.prefix_search([seg], [b"ab"]) .keys() == {b"ab"}
    assert engine.prefix_search([], [b"a"]) == {}
    # a union far beyond one 4096-value sort tile (global bitonic stages)
    w = synth.make_workload(3000, 5, 400000, universe=1 << 20, seed=5)
    _assert_prefix_equal(engine.prefix_search(w.segments, [b""]),
                         orc.prefix_search(w.segments, [b""]))


# ---------------------------------------------------------------- segment directories
def test_merge_through_segment_files(engine, orc, tmp_path):
    """Real segment directories end to end (SURVEY 8f row 1): `<key>_fst` + `<key>_val` files ->
    open (vellum v1 FST reader) -> ii2_merge -> write (FST writer + the device `_val` stream) ->
    reopen -> identical to the oracle's merge of the same inputs."""
    from inverted_index_2_b200 import files
    w = synth.make_workload(4000, 6, 60000, universe=1 << 16, seed=91)
    d = str(tmp_path)
    for i, seg in enumerate(w.segments):
        files.write_segment(d, str(1000 + i), seg.to_val(engine.intcomp_encode_batch))
    opened = [files.open_segment(d, k) for k in files.list_segments(d)]
    assert [s.n_terms for s in opened] == [s.n_terms for s in w.segments]
    got = engine.merge(opened, w.removed, decoded=True)
    exp = orc.merge(w.segments, w.removed, decoded=True)
    assert_merge_equal(got, exp)
    files.write_segment(d, "2000", got)
    back = files.open_segment(d, "2000")
    assert np.array_equal(back.val_bytes, exp.val_bytes) and np.array_equal(back.val_off, exp.val_off)
    assert_read_equal(engine.read_range([back]), orc.read_range([exp.to_segment()]))
    lo, hi = synth.term_at(w.term_bytes, w.term_off, 500), synth.term_at(w.term_bytes, w.term_off, 900)
    ranged = [s for s in (files.open_segment(d, k, lo, hi) for k in files.list_segments(d)[:6]) if s]
    assert_read_equal(engine.read_range(ranged), orc.read_range(w.segments, lo, hi))


def test_index_on_disk_with_engine(engine, tmp_path):
    from host_mirror import InvertedIndex
    d = str(tmp_path)
    idx = InvertedIndex(engine, basedir=d)
    idx.put([b"aaaa", b"bbbb"], 1)
    idx.put([b"aaaa", b"bbbb"], 1)
    idx.put([b"aaaa"], 2)
    idx.put_removed([1])
    assert idx.merge(2, 3, 2) > 0
    again = InvertedIndex(engine, basedir=d)
    assert list(again.read(None, None)) == [(b"aaaa", [2])]  # inverted_index_test.go:59-82


# ---------------------------------------------------------------- ingest batching
def _random_docs(rng, n_docs, vocab, lo, hi):
    docs = []
    for d in range(n_docs):
        n = int(rng.integers(lo, hi + 1))
        pick = rng.integers(0, len(vocab), size=n)
        docs.append(([vocab[int(i)] for i in pick], int(rng.integers(0, 1 << 20))))
    return docs


def test_ingest_matches_put_then_merge(engine, orc, merge_path):
    """ii2_ingest = Put x D + one Merge (oracle chain): unsorted terms, terms repeated inside a
    document, documents sharing terms and values, an empty document, terms that agree on their
    first 16 / 32 bytes, a document far larger than one 2048-record sort tile, removed filter."""
    rng = np.random.default_rng(17)
    tb, off = synth.make_terms(3000, seed=5)
    base = [synth.term_at(tb, off, i) for i in range(3000)]
    long_ = [b"shared-prefix-of-sixteen+" + b"x" * int(k % 23) + bytes([65 + k % 7]) for k in range(200)]
    vocab = base + long_ + [b"", b"a", b"ab", b"abc"]
    docs = _random_docs(rng, 40, vocab, 0, 300)
    docs.append(([], 7))
    docs.append((list(vocab) + list(reversed(vocab)), 99))       # every term twice, 6400+ records
    docs.append(([b"zz", b"zz", b"zz"], 5))
    removed = np.unique(rng.integers(0, 1 << 20, size=2000)).astype(np.uint32)
    for rem in (None, removed):
        got = engine.ingest(docs, rem, decoded=True)
        exp = orc.ingest(docs, rem, decoded=True)
        assert_merge_equal(got, exp)
    # a value removed everywhere: nothing left
    only = [([b"t1", b"t0"], 3), ([b"t1"], 3)]
    assert engine.ingest(only, np.array([3], dtype=np.uint32)).terms_count == 0
    assert engine.ingest([], None).terms_count == 0
    assert engine.ingest(only, None, decoded=True).as_dict() == {b"t0": [3], b"t1": [3]}


def test_put_batch_on_host_mirror(engine, orc):
    from host_mirror import InvertedIndex
    from scenario import OracleBackend
    rng = np.random.default_rng(23)
    tb, off = synth.make_terms(500, seed=9)
    vocab = [synth.term_at(tb, off, i) for i in range(500)]
    docs = [(t, v) for t, v in _random_docs(rng, 30, vocab, 1, 60)]
    a, b, c = InvertedIndex(engine), InvertedIndex(OracleBackend(orc)), InvertedIndex(engine)
    a.put_batch(docs)
    b.put_batch(docs)
    for terms, val in docs:
        c.put(terms, val)
    assert list(a.read(None, None)) == list(b.read(None, None)) == list(c.read(None, None))


# ---------------------------------------------------------------- device-resident API
def test_resident_pipeline_and_multipass(engine, orc, merge_path):
    """Resident segments; a result adopted as a segment and merged again equals the one-pass
    merge (inputs are sorted-unique, so pass structure is invisible)."""
    w = synth.make_workload(8000, 9, 150000, universe=1 << 15, seed=33)
    dsegs = [engine.upload(s) for s in w.segments]
    drem = engine.upload_removed(w.removed)
    one = engine.merge_dev(dsegs, drem, encode=True, decoded=True).download_merge(decoded=True)
    assert_merge_equal(one, orc.merge(w.segments, w.removed, decoded=True))
    r1 = engine.merge_dev(dsegs[:4], drem, encode=False).to_segment()
    r2 = engine.merge_dev(dsegs[4:], drem, encode=False).to_segment()
    two = engine.merge_dev([r1, r2], drem, encode=True, decoded=True).download_merge(decoded=True)
    assert np.array_equal(two.val_bytes, one.val_bytes) and np.array_equal(two.post, one.post)
    assert np.array_equal(two.term_bytes, one.term_bytes)
    rd = engine.read_range_dev(dsegs, None, None).download_read()
    assert_read_equal(rd, orc.read_range(w.segments))
    info = engine.read_range_dev(dsegs, None, None, drem).info()
    assert info.postings_out == one.postings_out and info.terms_count == one.terms_count


def test_concurrent_callers(engine, orc):
    """The reference calls this path from many goroutines (inverted_index.go:83-103,
    shard_test.go:236-247): concurrent C-ABI calls from host threads."""
    ws = [synth.make_workload(2000, 4, 30000, universe=1 << 12, seed=100 + i) for i in range(8)]
    exp = [orc.merge(w.segments, w.removed, decoded=True) for w in ws]
    t = lambda w, i: synth.term_at(w.term_bytes, w.term_off, i)
    # reads too: a range, a point read (one kernel, "last CTA" tickets and pinned result words per
    # host thread) and a small range (single-bucket plan, early placement)
    bounds = [[(t(w, 100), t(w, 900)), (t(w, 555), t(w, 555)), (t(w, 40), t(w, 44))] for w in ws]
    exp_r = [[orc.read_range(w.segments, lo, hi, removed=w.removed) for lo, hi in b] for w, b in zip(ws, bounds)]
    got = [None] * len(ws)
    got_r = [None] * len(ws)
    errs = []

    def run(i):
        try:
            for _ in range(3):
                got[i] = engine.merge(ws[i].segments, ws[i].removed, decoded=True)
                got_r[i] = [engine.read_range(ws[i].segments, lo, hi, removed=ws[i].removed)
                            for lo, hi in bounds[i]]
        except Exception as e:  # pragma: no cover
            errs.append(e)
    th = [threading.Thread(target=run, args=(i,)) for i in range(len(ws))]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errs
    for g, e in zip(got, exp):
        assert_merge_equal(g, e)
    for gr, er in zip(got_r, exp_r):
        for g, e in zip(gr, er):
            assert_read_equal(g, e)


# ---------------------------------------------------------------- codec vs oracle
def _lists_to_flat(lists):
    off = np.zeros(len(lists) + 1, dtype=np.uint64)
    np.cumsum([len(x) for x in lists], out=off[1:])
    post = np.concatenate([np.asarray(x, dtype=np.uint32) for x in lists]) if lists else \
        np.zeros(0, dtype=np.uint32)
    return post.astype(np.uint32), off


def test_intcomp_matches_oracle(engine, orc):
    rng = np.random.default_rng(3)
    lists = [[], [0], [0xFFFFFFFF], [10, 500, 300], [5] * 200, list(range(128)), list(range(129)),
             list(range(127)), [0xFFFFFFFF, 0, 0xFFFFFFFF, 1] * 64]
    for n in (1, 2, 31, 32, 33, 127, 128, 129, 255, 256, 257, 1000, 4096, 70000):
        for gap in (1, 16, 4096):
            lists.append(np.cumsum(rng.integers(1, 2 * gap + 1, size=n)).astype(np.uint32).tolist())
        lists.append(rng.integers(0, 1 << 32, size=n, dtype=np.uint64).astype(np.uint32).tolist())
    post, off = _lists_to_flat(lists)
    ew, eo = orc.intcomp_encode_batch(post, off)
    gw, go = engine.intcomp_encode_batch(post, off)
    assert np.array_equal(go, eo) and np.array_equal(gw, ew)
    dv, do = engine.intcomp_decode_batch(ew, eo)
    assert np.array_equal(do, off) and np.array_equal(dv, post)
    ov, oo = orc.intcomp_decode_batch(gw, go)
    assert np.array_equal(oo, off) and np.array_equal(ov, post)


def test_intcomp_long_lists_block_parallel(engine, orc):
    """Lists of >= 8192 values are decoded block-parallel (header walk in shared memory, delta
    sums, scan, one warp per block): sizes around the threshold, with and without a var-byte
    tail, unsorted values (negative deltas, sums wrap modulo 2^32), streams longer than one
    16384-word walk window, several long lists next to short ones in one batch."""
    rng = np.random.default_rng(77)
    lists = [[7], [], list(range(300))]
    for n in (8191, 8192, 8193, 8192 + 127, 8192 + 128, 16384, 20000, 65536 + 5):
        lists.append(np.cumsum(rng.integers(1, 33, size=n)).astype(np.uint32).tolist())
    lists.append(rng.integers(0, 1 << 32, size=40000, dtype=np.uint64).astype(np.uint32).tolist())
    lists.append([5] * 30000)                                   # all widths 0: one-word blocks
    lists.append(np.cumsum(rng.integers(1, 1 << 20, size=150000) % (1 << 32)).astype(np.uint32).tolist())
    lists.append([0xFFFFFFFF, 0, 0xFFFFFFFF, 1] * 4096)         # 32-bit zig-zag groups
    lists.append([3, 2, 1])
    post, off = _lists_to_flat(lists)
    ew, eo = orc.intcomp_encode_batch(post, off)
    dv, do = engine.intcomp_decode_batch(ew, eo)
    assert np.array_equal(do, off) and np.array_equal(dv, post)
    gw, go = engine.intcomp_encode_batch(post, off)
    assert np.array_equal(go, eo) and np.array_equal(gw, ew)
    # a long list whose section ends before its blocks do, and one with a width above 32
    from inverted_index_2_b200.engine import EngineError
    one = np.arange(0, 3 * 16384, 3, dtype=np.uint32)
    w, o = orc.intcomp_encode_batch(one, np.array([0, len(one)], dtype=np.uint64))
    short = w.copy()
    short[0] += 128                     # one block more than the section holds
    bad_width = w.copy()
    bad_width[3] = (bad_width[3] & 0x00FFFFFF) | (40 << 24)
    for words in (short, bad_width):
        with pytest.raises(EngineError) as e:
            engine.intcomp_decode_batch(words, o)
        assert e.value.code == A.II2_ERR_CORRUPT
    hollow = np.array([16384, 3, 0, 5, 0x85], dtype=np.uint32)  # 128 blocks announced, none there
    with pytest.raises(EngineError) as e:
        engine.intcomp_decode_batch(hollow, np.array([0, 5], dtype=np.uint64))
    assert e.value.code == A.II2_ERR_CORRUPT


def test_intcomp_rejects_corrupt(engine):
    from inverted_index_2_b200.engine import EngineError
    words = np.array([256, 2, 0, 0], dtype=np.uint32)  # section length below its own header
    with pytest.raises(EngineError) as e:
        engine.intcomp_decode_batch(words, np.array([0, 4], dtype=np.uint64))
    assert e.value.code == A.II2_ERR_CORRUPT


# ---------------------------------------------------------------- bitmask vs oracle
@pytest.mark.parametrize("L", [16, 64, 1024, 4096, 5000, 70000, 300000])
def test_bitmask_matches_oracle(engine, orc, L):
    """file/bitmask_test.go:15-21 shape: dictionary = universe of 2L ids, values = random half."""
    rng = np.random.default_rng(L)
    universe = np.sort(rng.choice(1 << 26, size=2 * L, replace=False)).astype(np.uint32)
    vals = rng.permutation(universe)[:L]
    g, o = engine.bitmask(universe), orc.Bitmask(universe)
    eg, eo = g.put(vals), o.put(vals, fast=True)
    assert eg == eo
    assert np.array_equal(g.get(eo), o.get(eo))
    assert np.array_equal(np.sort(g.get(eg)), np.sort(vals))
    # grow-on-miss from an empty dictionary, duplicates inside and across puts
    g2, o2 = engine.bitmask(), orc.Bitmask()
    for k in range(3):
        batch = np.concatenate([vals[k::3], vals[: L // 4], rng.integers(0, 50, size=20).astype(np.uint32)])
        assert g2.put(batch) == o2.put(batch, fast=True)
        assert np.array_equal(g2.all_values(), o2.all_values())
    assert np.array_equal(g2.get(eg[:0] + g2.put(vals)), o2.get(o2.put(vals, fast=True)))


def test_bitmask_slow_oracle_shape(engine, orc):
    """Against the literal O(L*D) slices.Index restatement, incl. duplicate dictionary entries."""
    init = [7, 3, 7, 9, 3]
    g, o = engine.bitmask(init), orc.Bitmask(init)
    for batch in ([3, 7, 11, 11, 9], [], [100, 3, 100, 200], [7]):
        assert g.put(batch) == o.put(batch, fast=False)
    assert g.all_values().tolist() == o.all_values().tolist() == [7, 3, 7, 9, 3, 11, 100, 200]
    enc = o.put([9, 200, 7], fast=False)
    assert g.get(enc).tolist() == o.get(enc).tolist()


def test_bitmask_full_chunk_run_container(engine, orc):
    """A full 65536-index chunk becomes the run container [0,65535] (run cookie, odd-sized
    header); with >= 4 containers the offset header returns."""
    for n in (65536, 65536 + 10, 5 * 65536 + 4097):
        vals = np.arange(n, dtype=np.uint32) * 3
        g, o = engine.bitmask(), orc.Bitmask()
        eg, eo = g.put(vals), o.put(vals, fast=True)
        assert eg == eo
        assert np.array_equal(g.get(eg), vals) and np.array_equal(o.get(eg), vals)


@pytest.mark.parametrize("case", load_roaring_vectors(), ids=lambda c: c["name"])
def test_bitmask_bytes_match_roaring_format_spec(engine, case):
    """K3b's Bitmask.Put bytes against the vectors packed from the public RoaringFormatSpec
    (tests/golden/make_roaring_vectors.py) — no oracle involved."""
    bm = engine.bitmask(np.arange(case["dict_n"], dtype=np.uint32))
    vals = roaring_case_values(case)
    data = bm.put(vals)
    check_roaring_case(case, data)
    assert sorted(set(bm.get(data).tolist())) == sorted(set(vals.tolist()))


def test_bitmask_out_of_bound_and_trailing_bytes(engine, orc):
    from inverted_index_2_b200.engine import EngineError
    big = engine.bitmask([5, 6, 7])
    enc = big.put([7])
    assert big.get(enc + b"\x01\x02\x03garbage").tolist() == [7]  # bitmask_test.go:44-46
    small = engine.bitmask([5])
    with pytest.raises(EngineError) as e:
        small.get(enc)
    assert e.value.code == A.II2_ERR_BITMASK_OOB
    with pytest.raises(EngineError) as e:
        small.get(b"\x00\x01\x02\x03\x04")
    assert e.value.code == A.II2_ERR_CORRUPT


# ---------------------------------------------------------------- cross-shard exchange (C-ABI)
def test_comm_world1_read_and_prefix_gather(engine, orc):
    """ii2_comm_init / ii2_read_gather / ii2_prefix_gather with a world of one rank: the gathered
    read is the local read (offsets rebased by 0) and the prefix union is the local one."""
    w = synth.make_workload(5000, 6, 60000, universe=1 << 16, seed=12)
    dsegs = [engine.upload(s) for s in w.segments]
    lo = synth.term_at(w.term_bytes, w.term_off, 100)
    hi = synth.term_at(w.term_bytes, w.term_off, 4000)
    engine.comm_init(engine.comm_unique_id(), 0, 1)
    try:
        assert engine.comm_info() == (0, 1)
        r = engine.read_range_dev(dsegs, lo, hi, None)
        g = engine.read_gather(r, 0)
        assert_read_equal(g.download_read(), orc.read_range(w.segments, lo, hi))
        g2 = engine.read_gather(r, -1)      # every rank receives
        assert_read_equal(g2.download_read(), r.download_read())
        empty = engine.read_range_dev(dsegs, b"~~~~", None, None)   # nothing in range
        ge = engine.read_gather(empty, 0).download_read()
        assert ge.n_terms == 0 and ge.term_off.tolist() == [0] and ge.post_off.tolist() == [0]
        pref = [b"", lo[:2], hi[:3], b"zzzz", lo[:1]]
        got = engine.prefix_search_gather(dsegs, pref, 0)
        exp = orc.prefix_search(w.segments, pref)
        assert sorted(got) == sorted(exp)
        assert all([int(x) for x in got[k]] == exp[k] for k in exp)
    finally:
        engine.comm_shutdown()
    assert engine.comm_info() == (0, 0)
