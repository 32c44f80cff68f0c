"""Batched exact-term reads (ii2_lookup, ii2_lookup_dev): every key of a batch must get exactly
the term and list that ii2_read_range_dev(key, key, rem) returns on the same handles, and that
the CPU oracle's read_range returns — absent keys, single-source pass-through (survey Q4),
sorted-unique unions, empty lists, the removed filter by bitmap and by sorted list, the one-CTA
union and the heavy path beyond 4096 values, large batches, concurrent callers and devices."""
import ctypes as C
import json
import os
import threading
import traceback

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A
from inverted_index_2_b200.flat import FlatSegment

LOOKUP_SYMBOLS = ("ii2_lookup_dev", "ii2_lookup", "ii2_lookup_out_free")


# ---------------------------------------------------------------- CPU, no device
def test_lookup_symbols_exported_and_bound():
    from inverted_index_2_b200.engine import load_library
    lib = load_library()
    for name in LOOKUP_SYMBOLS:
        assert name in A.PROTOTYPES
        fn = getattr(lib, name)
        assert fn.restype == A.PROTOTYPES[name][0] and fn.argtypes == A.PROTOTYPES[name][1]


def test_lookup_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    from inverted_index_2_b200.engine import load_library
    lib = load_library()
    out = A.LookupOut()
    off = (C.c_uint32 * 1)(0)
    assert lib.ii2_lookup_dev(None, 0, None, off, 0, None, C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert lib.ii2_lookup(None, 0, None, off, 0, None, 0, C.byref(out)) == A.II2_ERR_NO_DEVICE


# ---------------------------------------------------------------- helpers
def _check(engine, orc, segs, keys, removed=None, dsegs=None, bitmap=None):
    """lookup_dev over resident copies of `segs` against read_range_dev and the oracle, key by
    key.  bitmap: None = whatever ii2_removed_upload picks, False = force a sorted-list-only set."""
    own = dsegs is None
    if own:
        dsegs = [engine.upload(s) for s in segs]
    drem = None
    if removed is not None:
        r = np.asarray(removed, dtype=np.uint32)
        if bitmap is False and len(r) >= 64:  # ids >= 2^29 keep the set a sorted list only
            assert int(r.max()) >= (1 << 29)
        drem = engine.upload_removed(r)
    try:
        got = engine.lookup_dev(dsegs, keys, drem)
        assert len(got) == len(keys)
        for k, g in zip(keys, got):
            exp = orc.read_range(segs, k, k, removed=removed)
            dev = engine.read_range_dev(dsegs, k, k, drem)
            r = dev.download_read()
            dev.release()
            assert r.n_terms == exp.n_terms, k
            if exp.n_terms == 0:
                assert g is None, k
            else:
                assert g is not None, k
                assert np.array_equal(g, exp.post), k
                assert np.array_equal(g, r.post), k
        return got
    finally:
        if drem is not None:
            drem.release()
        if own:
            for s in dsegs:
                s.release()


def _absent_keys(vocab):
    """Keys that are not terms of `vocab`: before the first, after the last, between two terms,
    proper prefixes and extensions of terms, 0x00 / 0xFF bytes, long keys."""
    vs = set(vocab)
    cand = [b"\x00", b"\xff" * 3, (max(vocab) if vocab else b"") + b"\xff", b"\x00" + (min(vocab) if vocab else b""),
            b"q" * 300, bytes(range(256)) + b"\x01" * 60]
    for t in vocab[:: max(1, len(vocab) // 20)]:
        cand += [t[:-1], t + b"\x00", t + b"\xff", t + b"m"]
    for a, b in zip(vocab[:-1:7], vocab[1::7]):
        cand.append(a + b"\x00")
    return [k for k in cand if k not in vs]


def _keys_for(rng, vocab):
    """Every vocabulary term, absent keys, the empty key, duplicates; shuffled."""
    keys = list(vocab) + _absent_keys(vocab) + [b""]
    keys += [vocab[int(i)] for i in rng.integers(0, len(vocab), size=min(20, len(vocab)))] if vocab else []
    rng.shuffle(keys)
    return keys


def _fuzz_segments(rng, vocab, nseg, hi_bits):
    segs = []
    for _ in range(nseg):
        frac = rng.choice([0.0, 0.05, 0.5, 1.0])
        items = []
        for t in vocab:
            if rng.random() >= frac:
                continue
            n = int(rng.choice([0, 1, 2, 3, 7, 40, 130, 300], p=[.05, .3, .2, .2, .1, .1, .03, .02]))
            vals = rng.integers(0, 1 << hi_bits, size=n, dtype=np.int64)
            if rng.random() < 0.7:
                vals = np.unique(vals)
            items.append((t, vals.tolist()))  # else unsorted, with duplicates
        segs.append(FlatSegment.from_items(items))
    return segs


def _terms(rng, n):
    out = {bytes(rng.integers(0, 256, size=int(rng.integers(0, 6))).tolist()) for _ in range(n // 2)}
    out |= {bytes(rng.choice(list(b"abcXYZ"), size=int(rng.integers(1, 12))).tolist()) for _ in range(n // 2)}
    return sorted(out)


# ---------------------------------------------------------------- GPU, exactness
@pytest.mark.gpu
def test_lookup_golden_segments(engine, orc):
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.json")
    with open(path) as f:
        cases = json.load(f)["writer"]
    segs = [FlatSegment.from_items([(t.encode(), v) for t, v in c["items"]]) for c in cases]
    vocab = sorted({t.encode() for c in cases for t, _ in c["items"]})
    keys = _keys_for(np.random.default_rng(5), vocab)
    for removed in (None, [10, 66]):
        _check(engine, orc, segs, keys, removed)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(24))
def test_lookup_random_shard_contents(engine, orc, seed):
    rng = np.random.default_rng(7000 + seed)
    hi_bits = [8, 16, 32][seed % 3]
    vocab = _terms(rng, int(rng.integers(2, 300)))
    segs = _fuzz_segments(rng, vocab, int(rng.integers(1, 20)), hi_bits)
    keys = _keys_for(rng, vocab)
    mode = seed % 3  # no removed set, a bitmap-backed one, a sorted-list-only one
    removed, bitmap = None, None
    if mode == 1:
        removed = np.unique(rng.integers(0, 1 << min(hi_bits, 20), size=500)).astype(np.uint32)
    elif mode == 2:
        removed = np.unique(np.concatenate([rng.integers(0, 1 << hi_bits, size=300),
                                            [(1 << 30) + 5]])).astype(np.uint32)
        bitmap = False
    _check(engine, orc, segs, keys, removed, bitmap=bitmap)


@pytest.mark.gpu
@pytest.mark.parametrize("nseg", [1, 2, 47, 1024])
@pytest.mark.parametrize("rem_mode", ["none", "bitmap", "sorted"])
def test_lookup_segment_counts(engine, orc, nseg, rem_mode):
    rng = np.random.default_rng(nseg)
    vocab = sorted({b"t%05d" % i for i in rng.integers(0, 3000, size=200)})
    segs = []
    for _ in range(nseg):
        pick = [t for t in vocab if rng.random() < (0.5 if nseg < 47 else 0.02)]
        segs.append(FlatSegment.from_items(
            [(t, np.unique(rng.integers(0, 5000, size=int(rng.integers(0, 9)))).tolist()) for t in pick]))
    keys = _keys_for(rng, vocab)
    removed = {"none": None,
               "bitmap": np.arange(0, 5000, 7, dtype=np.uint32),
               "sorted": np.concatenate([np.arange(0, 5000, 7), [1 << 30]]).astype(np.uint32)}[rem_mode]
    _check(engine, orc, segs, keys, removed)


# ---------------------------------------------------------------- GPU, quirks
@pytest.mark.gpu
def test_lookup_quirks(engine, orc):
    a = FlatSegment.from_items([(b"empty_only", []), (b"only_a", [9, 3, 3, 7]), (b"shared", [5, 1, 5]),
                                (b"to_remove", [4, 8])])
    b = FlatSegment.from_items([(b"empty_only", []), (b"shared", [1, 9, 9]), (b"shared_empty", [])])
    c = FlatSegment.from_items([(b"shared_empty", [6, 2])])
    segs = [a, b, c]
    keys = [b"only_a", b"shared", b"empty_only", b"to_remove", b"shared_empty", b"missing"]
    got = dict(zip(keys, _check(engine, orc, segs, keys)))
    assert got[b"only_a"].tolist() == [9, 3, 3, 7]           # one source: as stored (Q4)
    assert got[b"shared"].tolist() == [1, 5, 9]              # two sources: sorted-unique
    assert got[b"shared_empty"].tolist() == [2, 6]           # an empty source still sorts
    assert got[b"empty_only"] is not None and len(got[b"empty_only"]) == 0  # kept without rem
    assert got[b"missing"] is None
    got = dict(zip(keys, _check(engine, orc, segs, keys, removed=[4, 8])))
    assert got[b"to_remove"] is None                         # emptied by rem: not found
    assert got[b"empty_only"] is None
    assert got[b"only_a"].tolist() == [9, 3, 3, 7]


# ---------------------------------------------------------------- GPU, sizes
@pytest.mark.gpu
@pytest.mark.parametrize("nsrc", [1, 40])
def test_lookup_union_sizes(engine, orc, nsrc):
    """Unions of 4095, 4096, 4097 and ~100 000 values: the one-CTA union and the heavy path."""
    rng = np.random.default_rng(nsrc)
    sizes = {b"k4095": 4095, b"k4096": 4096, b"k4097": 4097, b"k100k": 100_000}
    per_seg = [[] for _ in range(nsrc)]
    for t, n in sizes.items():
        vals = rng.permutation(np.arange(n, dtype=np.int64) * 3 + 1)  # n distinct values
        for s, part in enumerate(np.array_split(vals, nsrc)):
            per_seg[s].append((t, part.tolist() if nsrc == 1 else np.sort(part).tolist()))
    for s in range(nsrc):
        per_seg[s].append((b"small", [s, s + 1]))
    segs = [FlatSegment.from_items(sorted(x)) for x in per_seg]
    keys = list(sizes) + [b"small", b"k4096", b"nope", b"k100k"]
    got = _check(engine, orc, segs, keys)
    for k, g in zip(keys, got):
        if k in sizes:
            assert len(g) == sizes[k]
    _check(engine, orc, segs, keys, removed=np.arange(1, 12000, 3, dtype=np.uint32))


@pytest.mark.gpu
def test_lookup_empty_batches(engine):
    seg = engine.upload(FlatSegment.from_items([(b"a", [1])]))
    assert engine.lookup_dev([seg], []) == []
    assert engine.lookup_dev([], [b"a", b""]) == [None, None]
    assert engine.lookup([], []) == []
    seg.release()


@pytest.mark.gpu
def test_lookup_c3_workload_65536_keys(engine):
    """65 536 random keys (about 10 % absent) over the C3 shape: 256 segments of a 1 M-term
    vocabulary, 5 % removed, checked against the workload's own numpy union.  30 M postings keep
    the reference computation short."""
    from inverted_index_2_b200 import synth
    w = synth.make_workload(1_000_000, 256, 30_000_000, seed=0xC3, presence=0.125)
    terms, vals, poff = w.expected_union(w.removed)
    n = len(w.term_off) - 1
    rng = np.random.default_rng(11)
    ids = rng.integers(0, n, size=65536)
    absent = rng.random(65536) < 0.1
    keys = [synth.term_at(w.term_bytes, w.term_off, int(i)) + (b"\x00" if a else b"")
            for i, a in zip(ids, absent)]
    dsegs = [engine.upload(s) for s in w.segments]
    drem = engine.upload_removed(w.removed)
    got = engine.lookup_dev(dsegs, keys, drem)
    pos = np.searchsorted(terms, ids)
    for j, (i, a) in enumerate(zip(ids, absent)):
        hit = not a and pos[j] < len(terms) and terms[pos[j]] == i
        if not hit:
            assert got[j] is None, j
        else:
            assert np.array_equal(got[j], vals[int(poff[pos[j]]):int(poff[pos[j] + 1])]), j
    drem.release()
    for s in dsegs:
        s.release()


# ---------------------------------------------------------------- GPU, concurrency and devices
@pytest.mark.gpu
def test_lookup_concurrent_threads(engine):
    from inverted_index_2_b200 import synth
    w = synth.make_workload(20000, 16, 400000, universe=1 << 16, seed=21)
    dsegs = [engine.upload(s) for s in w.segments]
    drem = engine.upload_removed(w.removed)
    n = len(w.term_off) - 1
    batches = []
    for t in range(8):
        rng = np.random.default_rng(100 + t)
        batches.append([synth.term_at(w.term_bytes, w.term_off, int(i)) + (b"!" if i % 9 == 0 else b"")
                        for i in rng.integers(0, n, size=3000)])
    serial = [engine.lookup_dev(dsegs, b, drem if t % 2 else None) for t, b in enumerate(batches)]
    results, errs = [None] * 8, []

    def run(t):
        try:
            for _ in range(3):
                results[t] = engine.lookup_dev(dsegs, batches[t], drem if t % 2 else None)
        except BaseException:
            errs.append(traceback.format_exc())
    ts = [threading.Thread(target=run, args=(t,)) for t in range(8)]
    [x.start() for x in ts]
    [x.join() for x in ts]
    assert not errs, "\n".join(errs)
    for s_, r in zip(serial, results):
        assert len(s_) == len(r)
        for a, b in zip(s_, r):
            assert (a is None and b is None) or np.array_equal(a, b)


def _two_device_worker(q):
    try:
        from inverted_index_2_b200.engine import Engine, EngineError
        from oracle import orc
        orc.lib()
        eng = Engine(devices=[0, 1])
        segs = [FlatSegment.from_items([(b"a", [3, 1]), (b"b", [2])]),
                FlatSegment.from_items([(b"b", [7, 2]), (b"c", [])])]
        eng.set_device(1)
        d1 = [eng.upload(s) for s in segs]
        assert all(d.device == 1 for d in d1)
        keys = [b"a", b"b", b"c", b"d"]
        got = eng.lookup_dev(d1, keys)
        for k, g in zip(keys, got):
            e = orc.read_range(segs, k, k)
            assert (g is None) == (e.n_terms == 0)
            if g is not None:
                assert np.array_equal(g, e.post)
        eng.set_device(0)
        d0 = eng.upload(segs[0])
        try:
            eng.lookup_dev([d0, d1[1]], keys)
            raise AssertionError("mixed devices accepted")
        except EngineError as e:
            assert e.code == A.II2_ERR_INVALID
        q.put(None)
    except BaseException:
        q.put(traceback.format_exc())


@pytest.mark.gpu
def test_lookup_on_second_device():
    import multiprocessing as mp

    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    p = ctx.Process(target=_two_device_worker, args=(q,))
    p.start()
    err = q.get(timeout=900)
    p.join(timeout=120)
    assert err is None, err
    assert p.exitcode == 0


# ---------------------------------------------------------------- GPU, errors
@pytest.mark.gpu
def test_lookup_errors(engine):
    seg = engine.upload(FlatSegment.from_items([(b"a", [1])]))
    lib = engine.lib
    h = engine._handles([seg])
    kb = (C.c_uint8 * 4)(*b"abcd")
    out = A.LookupOut()
    good = (C.c_uint32 * 3)(0, 1, 2)
    assert lib.ii2_lookup_dev(h, 1, C.cast(kb, A.u8p), good, 2, None, None) == A.II2_ERR_INVALID
    bad = (C.c_uint32 * 3)(0, 3, 2)
    assert lib.ii2_lookup_dev(h, 1, C.cast(kb, A.u8p), bad, 2, None, C.byref(out)) == A.II2_ERR_INVALID
    assert lib.ii2_lookup_dev(h, 1, None, good, 2, None, C.byref(out)) == A.II2_ERR_INVALID
    many = (C.c_void_p * 1025)(*([seg.h] * 1025))
    assert lib.ii2_lookup_dev(many, 1025, C.cast(kb, A.u8p), good, 2, None, C.byref(out)) == \
        A.II2_ERR_UNSUPPORTED
    long_key = (C.c_uint8 * 65536)()
    off = (C.c_uint32 * 2)(0, 65536)
    assert lib.ii2_lookup_dev(h, 1, C.cast(long_key, A.u8p), off, 1, None, C.byref(out)) == \
        A.II2_ERR_UNSUPPORTED
    assert engine.lookup_dev([seg], [bytes(long_key)[:65535]]) == [None]  # the longest key allowed
    seg.release()
