"""Boolean term queries (ii2_query, ii2_query_dev): every query's result must equal the answer
composed here with Python sets from the CPU oracle — values(TERM t) = the set of
orc.read_range(t, t)'s list, values(PREFIX p) = orc.prefix_search's found[p] — intersected over
the required clauses, minus the excluded ones and the removed set.  No GPU code produces an
expected answer, except on the full-size workload, where the device's own lookup and prefix
search lists (already checked against the oracle elsewhere) are intersected with numpy."""
import ctypes as C
import threading
import traceback

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A
from inverted_index_2_b200 import synth
from inverted_index_2_b200.flat import FlatSegment

QUERY_SYMBOLS = ("ii2_query_dev", "ii2_query", "ii2_query_out_free")
TILE, STAGE = 2048, 8192  # k9_query.cu: driver values per tile, window values staged in smem


# ---------------------------------------------------------------- CPU, no device
def test_query_symbols_exported_and_bound():
    from inverted_index_2_b200.engine import load_library
    lib = load_library()
    for name in QUERY_SYMBOLS:
        assert name in A.PROTOTYPES
        fn = getattr(lib, name)
        assert fn.restype == A.PROTOTYPES[name][0] and fn.argtypes == A.PROTOTYPES[name][1]


def test_query_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    from inverted_index_2_b200.engine import Engine, load_library
    lib = load_library()
    batch, keep = Engine._query_args([[(True, [(b"a", False)])]])
    out = A.QueryOut()
    assert lib.ii2_query_dev(None, 0, C.byref(batch), None, C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert lib.ii2_query(None, 0, C.byref(batch), None, 0, C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert out.n_queries == 0 and not out.values and not out.value_off


def _unpack(b: A.QueryBatch):
    """The inverse of Engine._query_args, read back through the struct's pointers."""
    na, nc, nq = int(b.natoms), int(b.nclauses), int(b.nqueries)
    aoff = A.from_ptr(b.atom_off, na + 1, np.uint32)
    blob = A.from_ptr(b.atom_bytes, int(aoff[-1]), np.uint8).tobytes()
    kind = A.from_ptr(b.atom_kind, na, np.uint8)
    cao = A.from_ptr(b.clause_atom_off, nc + 1, np.uint32)
    excl = A.from_ptr(b.clause_excluded, nc, np.uint8)
    qco = A.from_ptr(b.query_clause_off, nq + 1, np.uint32)
    atoms = [(blob[aoff[i]:aoff[i + 1]], bool(kind[i] == A.II2_ATOM_PREFIX)) for i in range(na)]
    clauses = [(not excl[c], atoms[cao[c]:cao[c + 1]]) for c in range(nc)]
    return [clauses[qco[q]:qco[q + 1]] for q in range(nq)]


def test_query_packing_round_trips():
    from inverted_index_2_b200.engine import Engine
    queries = [
        [(True, [(b"error", False), (b"time", True)]), (True, [(b"db", True)]), (False, [(b"debug", False)])],
        [(True, [])],
        [(False, [(b"", True)]), (True, [(b"", False), (b"\x00\xff", True)])],
        [(True, [(b"x" * 300, False)] * 3)],
    ]
    for qs in (queries, [], [[]]):
        b, keep = Engine._query_args(qs)
        assert _unpack(b) == qs
    b, keep = Engine._query_args(queries)
    assert (int(b.natoms), int(b.nclauses), int(b.nqueries)) == (10, 7, 4)


# ---------------------------------------------------------------- expected answers
class Expect:
    """Composes answers from the oracle with Python sets (memoised per atom)."""

    def __init__(self, orc, segs, removed=None):
        self.orc, self.segs = orc, segs
        self.removed = set(int(v) for v in removed) if removed is not None else set()
        self.memo = {}

    def atom(self, term, is_prefix):
        k = (term, is_prefix)
        if k not in self.memo:
            if is_prefix:
                v = self.orc.prefix_search(self.segs, [term]).get(term, [])
            else:
                r = self.orc.read_range(self.segs, term, term)
                v = r.post if r.n_terms else []
            self.memo[k] = set(int(x) for x in v)
        return self.memo[k]

    def clause(self, atoms):
        out = set()
        for t, p in atoms:
            out |= self.atom(t, p)
        return out

    def query(self, clauses):
        req = [self.clause(a) for r, a in clauses if r]
        exc = [self.clause(a) for r, a in clauses if not r]
        res = set.intersection(*req)
        for e in exc:
            res -= e
        return np.array(sorted(res - self.removed), dtype=np.uint32)


def _run(engine, orc, segs, queries, removed=None, dsegs=None, exp=None):
    own = dsegs is None
    if own:
        dsegs = [engine.upload(s) for s in segs]
    drem = engine.upload_removed(np.asarray(removed, dtype=np.uint32)) if removed is not None else None
    try:
        got = engine.query_dev(dsegs, queries, drem)
    finally:
        if drem is not None:
            drem.release()
        if own:
            for s in dsegs:
                s.release()
    exp = exp or Expect(orc, segs, removed)
    assert len(got) == len(queries)
    for i, (q, g) in enumerate(zip(queries, got)):
        assert g.dtype == np.uint32
        assert np.array_equal(g, exp.query(q)), (i, q)
    return got


# ---------------------------------------------------------------- GPU, against the reference's own vectors
@pytest.mark.gpu
def test_query_golden_prefix_vectors(engine, orc):
    """TestSearchByPrefix (inverted_index_test.go:196-220): one Put per segment; the prefixes as
    one-clause queries equal prefix_search_dev."""
    puts = [(b"a12", 1), (b"a13", 1), (b"a13", 2), (b"a20", 3), (b"a30", 4),
            (b"termA", 5), (b"termB", 6), (b"termC", 7)]
    segs = [FlatSegment.direct([t], v) for t, v in puts]
    dsegs = [engine.upload(s) for s in segs]
    prefixes = [b"a1", b"term", b"unknown", b"", b"a"]
    got = _run(engine, orc, segs, [[(True, [(p, True)])] for p in prefixes], dsegs=dsegs)
    ref = engine.prefix_search_dev(dsegs, prefixes)
    for p, g in zip(prefixes, got):
        assert np.array_equal(g, ref.get(p, np.zeros(0, np.uint32))), p
    assert got[0].tolist() == [1, 2] and got[1].tolist() == [5, 6, 7] and len(got[2]) == 0


@pytest.mark.gpu
def test_query_term_is_a_set(engine, orc):
    """A one-term query is the sorted-unique lookup_dev list, also for a single-source list that
    is stored unsorted with duplicates (quirk Q4: lookup returns it as stored)."""
    a = FlatSegment.from_items([(b"only_a", [9, 3, 3, 7]), (b"shared", [5, 1, 5]), (b"u32", [0xFFFFFFFF, 0])])
    b = FlatSegment.from_items([(b"empty", []), (b"shared", [1, 9, 9])])
    segs = [a, b]
    dsegs = [engine.upload(s) for s in segs]
    terms = [b"only_a", b"shared", b"u32", b"empty", b"missing"]
    got = _run(engine, orc, segs, [[(True, [(t, False)])] for t in terms], dsegs=dsegs)
    look = engine.lookup_dev(dsegs, terms)
    for t, g, lk in zip(terms, got, look):
        assert np.array_equal(g, np.unique(lk) if lk is not None else np.zeros(0, np.uint32)), t
    assert got[0].tolist() == [3, 7, 9] and got[2].tolist() == [0, 0xFFFFFFFF]


# ---------------------------------------------------------------- GPU, randomised batches
def _vocab(rng, n):
    out = {bytes(rng.choice(list(b"abcxyz"), size=int(rng.integers(1, 8))).tolist()) for _ in range(n)}
    out |= {bytes(rng.integers(0, 256, size=int(rng.integers(1, 4))).tolist()) for _ in range(n // 8)}
    return sorted(out)


def _segments(rng, vocab, nseg, hi_bits):
    segs = []
    for _ in range(nseg):
        frac = rng.choice([0.05, 0.3, 0.8]) if nseg < 64 else 0.03
        items = []
        for t in vocab:
            if rng.random() >= frac:
                continue
            n = int(rng.choice([0, 1, 3, 10, 60, 400], p=[.05, .25, .25, .25, .15, .05]))
            vals = rng.integers(0, 1 << hi_bits, size=n, dtype=np.int64)
            if rng.random() < 0.8:
                vals = np.unique(vals)
            items.append((t, vals.tolist()))  # else unsorted, with duplicates
        segs.append(FlatSegment.from_items(items))
    return segs


def _atom(rng, vocab):
    r = rng.random()
    t = vocab[int(rng.integers(0, len(vocab)))]
    if r < 0.35:
        return (t, False)
    if r < 0.7:
        return (t[:int(rng.integers(0, len(t) + 1))], True)
    if r < 0.8:
        return (t + b"\x00", bool(rng.random() < 0.5))  # absent term / unmatched prefix
    if r < 0.85:
        return (b"", False)  # the empty term
    if r < 0.9:
        return (b"", True)  # the whole index
    return (b"\xff\xff\xff", bool(rng.random() < 0.5))


def _queries(rng, vocab, n):
    qs = []
    for _ in range(n):
        ncl = int(rng.integers(1, 7))
        clauses = []
        for _ in range(ncl):
            na = int(rng.integers(0, 6)) if rng.random() < 0.1 else int(rng.integers(1, 6))
            clauses.append((bool(rng.random() < 0.6), [_atom(rng, vocab) for _ in range(na)]))
        if not any(r for r, _ in clauses):
            if rng.random() < 0.5:  # only excluded clauses but one
                clauses[int(rng.integers(0, ncl))] = (True, clauses[0][1] or [_atom(rng, vocab)])
            else:
                clauses.append((True, [_atom(rng, vocab)]))
        if rng.random() < 0.1:
            clauses.append(clauses[0])  # a duplicate clause
        qs.append(clauses)
    qs += [qs[int(i)] for i in rng.integers(0, len(qs), size=3)]  # duplicate queries
    return qs


@pytest.mark.gpu
@pytest.mark.parametrize("nseg", [1, 3, 64, 300])
@pytest.mark.parametrize("rem_mode", ["none", "bitmap", "sorted"])
def test_query_random_batches(engine, orc, nseg, rem_mode):
    seed = nseg * 7 + len(rem_mode)
    rng = np.random.default_rng(seed)
    hi_bits = 12 if nseg < 64 else 16
    vocab = _vocab(rng, 60)
    segs = _segments(rng, vocab, nseg, hi_bits)
    removed = {"none": None,
               "bitmap": np.unique(rng.integers(0, 1 << hi_bits, size=300)).astype(np.uint32),
               "sorted": np.unique(np.concatenate([rng.integers(0, 1 << hi_bits, size=300),
                                                   [(1 << 30) + 3]])).astype(np.uint32)}[rem_mode]
    queries = _queries(rng, vocab, 40)
    exp = Expect(orc, segs, removed)
    dsegs = [engine.upload(s) for s in segs]
    got = _run(engine, orc, segs, queries, removed, dsegs=dsegs, exp=exp)
    if nseg == 3:  # the host-view entry point gives the same answers
        again = engine.query(segs, queries, removed)
        assert all(np.array_equal(a, b) for a, b in zip(got, again))
    for s in dsegs:
        s.release()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(6))
def test_query_random_shapes(engine, orc, seed):
    """Seeded mixes of segment counts, value widths and clause shapes."""
    rng = np.random.default_rng(9100 + seed)
    hi_bits = [8, 20, 32][seed % 3]
    vocab = _vocab(rng, int(rng.integers(5, 120)))
    segs = _segments(rng, vocab, int(rng.integers(1, 12)), hi_bits)
    removed = np.unique(rng.integers(0, 1 << min(hi_bits, 20), size=200)).astype(np.uint32) \
        if seed % 2 else None
    _run(engine, orc, segs, _queries(rng, vocab, 60), removed)


# ---------------------------------------------------------------- GPU, intersection shapes
def _shape_segments(named):
    """Every term's values split over two segments (sorted parts), so atoms are true unions."""
    a, b = [], []
    for t in sorted(named):
        v = np.asarray(named[t], dtype=np.uint32)
        a.append((t, np.sort(v[0::2]).tolist()))
        b.append((t, np.sort(v[1::2]).tolist()))
    return [FlatSegment.from_items(a), FlatSegment.from_items(b)]


def _pairs_queries(pairs):
    qs = []
    for x, y in pairs:
        qs += [[(True, [(x, False)]), (True, [(y, False)])],
               [(True, [(x, False)]), (False, [(y, False)])],
               [(True, [(y, False)]), (False, [(x, False)])],
               [(True, [(x, False), (y, False)]), (True, [(x, False)])]]
    return qs


@pytest.mark.gpu
def test_query_driver_tile_edges(engine, orc):
    """Drivers of 1, TILE-1, TILE, TILE+1 and many tiles against a superset, a subset and an
    interleaved list; the driver is the smaller clause whichever side of the query it is on."""
    rng = np.random.default_rng(3)
    big = np.unique(rng.integers(0, 1 << 22, size=300_000)).astype(np.uint32)
    named = {b"big": big, b"odd": big[1::2], b"evenv": big[big % 2 == 0]}
    for n in (1, TILE - 1, TILE, TILE + 1, 5 * TILE + 7, 40_000):
        named[b"d%06d" % n] = np.sort(rng.choice(big, size=n, replace=False))
    segs = _shape_segments(named)
    pairs = [(t, o) for t in named if t.startswith(b"d") for o in (b"big", b"odd", b"evenv")]
    _run(engine, orc, segs, _pairs_queries(pairs))


@pytest.mark.gpu
def test_query_windows_and_sizes(engine, orc):
    """Windows below and above the shared-memory stage (the global gallop path), skewed (1 vs
    10^6) and balanced (10^6 vs 10^6) sizes, disjoint / identical / interleaved lists, values 0
    and 2^32-1."""
    rng = np.random.default_rng(4)
    m1 = np.unique(rng.integers(0, 1 << 32, size=1_050_000, dtype=np.uint64)).astype(np.uint32)[:1_000_000]
    m2 = np.unique(rng.integers(0, 1 << 32, size=1_050_000, dtype=np.uint64)).astype(np.uint32)[:1_000_000]
    m1 = np.union1d(m1, [0, 0xFFFFFFFF]).astype(np.uint32)
    ev = np.arange(0, 2_000_000, 2, dtype=np.uint32)
    named = {
        b"m1": m1, b"m2": m2, b"m1copy": m1.copy(),
        b"one": m1[500_000:500_001],
        b"sparse": np.sort(rng.choice(m1, size=3000, replace=False)),   # windows of ~10^6/3000*2048 > STAGE
        b"dense": m1[100_000:100_000 + 3 * TILE],                       # windows of one tile
        b"evens": ev, b"odds": ev + 1, b"thirds": np.arange(0, 3_000_000, 3, dtype=np.uint32),
        b"edges": np.array([0, 1, 0xFFFFFFFE, 0xFFFFFFFF], dtype=np.uint32),
        b"edges2": np.array([0, 0xFFFFFFFF], dtype=np.uint32),
        b"disj_lo": np.arange(0, 50_000, dtype=np.uint32), b"disj_hi": np.arange(50_000, 90_000, dtype=np.uint32),
    }
    segs = _shape_segments(named)
    pairs = [(b"m1", b"m2"), (b"m1", b"m1copy"), (b"one", b"m1"), (b"one", b"m2"), (b"sparse", b"m1"),
             (b"sparse", b"m2"), (b"dense", b"m1"), (b"evens", b"odds"), (b"evens", b"thirds"),
             (b"edges", b"edges2"), (b"edges", b"m1"), (b"disj_lo", b"disj_hi"), (b"disj_lo", b"evens")]
    queries = _pairs_queries(pairs)
    queries += [[(True, [(b"sparse", False)]), (True, [(b"m1", False)]), (False, [(b"m2", False)]),
                 (True, [(b"m1copy", False), (b"one", False)])],
                [(True, [(b"evens", False), (b"odds", False)]), (True, [(b"thirds", False)]),
                 (False, [(b"disj_lo", False)])]]
    removed = np.concatenate([m1[::97], [0xFFFFFFFF]]).astype(np.uint32)
    exp = Expect(orc, segs)
    dsegs = [engine.upload(s) for s in segs]
    _run(engine, orc, segs, queries, dsegs=dsegs, exp=exp)
    exp_r = Expect(orc, segs, removed)
    exp_r.memo = exp.memo
    _run(engine, orc, segs, queries, removed, dsegs=dsegs, exp=exp_r)
    for s in dsegs:
        s.release()


# ---------------------------------------------------------------- GPU, batches and threads
def _small_workload():
    w = synth.make_workload(20000, 16, 400000, universe=1 << 18, seed=31)
    n = len(w.term_off) - 1
    t = lambda i: synth.term_at(w.term_bytes, w.term_off, int(i))
    return w, n, t


def _workload_queries(rng, n, t, count):
    qs = []
    for _ in range(count):
        a, b, c = (t(i) for i in rng.integers(0, n, size=3))
        shape = int(rng.integers(0, 4))
        if shape == 0:
            qs.append([(True, [(a, False)]), (True, [(b[:1], True)])])
        elif shape == 1:
            qs.append([(True, [(a[:2], True)]), (True, [(b[:1], True), (c, False)]), (False, [(c[:2], True)])])
        elif shape == 2:
            qs.append([(True, [(a[:1], True)]), (True, [(b[:1], True)])])
        else:
            qs.append([(True, [(a, False), (b, False), (c + b"!", False)])])
    return qs


@pytest.mark.gpu
def test_query_batch_equals_single_calls(engine):
    """10 000 queries in one call equal the same queries called one at a time; query over views
    equals query_dev."""
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    drem = engine.upload_removed(w.removed)
    qs = _workload_queries(np.random.default_rng(12), n, t, 10_000)
    batch = engine.query_dev(dsegs, qs, drem)
    for i, q in enumerate(qs):
        assert np.array_equal(batch[i], engine.query_dev(dsegs, [q], drem)[0]), i
    views = engine.query(w.segments, qs[:500], w.removed)
    assert all(np.array_equal(a, b) for a, b in zip(batch[:500], views))
    drem.release()
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_query_concurrent_threads(engine):
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    drem = engine.upload_removed(w.removed)
    batches = [_workload_queries(np.random.default_rng(200 + k), n, t, 400) for k in range(4)]
    serial = [engine.query_dev(dsegs, b, drem if k % 2 else None) for k, b in enumerate(batches)]
    results, errs = [None] * 4, []

    def run(k):
        try:
            for _ in range(3):
                results[k] = engine.query_dev(dsegs, batches[k], drem if k % 2 else None)
        except BaseException:
            errs.append(traceback.format_exc())
    ts = [threading.Thread(target=run, args=(k,)) for k in range(4)]
    [x.start() for x in ts]
    [x.join() for x in ts]
    assert not errs, "\n".join(errs)
    for s_, r in zip(serial, results):
        assert len(s_) == len(r) and all(np.array_equal(a, b) for a, b in zip(s_, r))
    drem.release()
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_query_empty_batches(engine):
    seg = engine.upload(FlatSegment.from_items([(b"a", [1])]))
    assert engine.query_dev([seg], []) == []
    got = engine.query_dev([], [[(True, [(b"a", False)])], [(True, [])]])
    assert [len(g) for g in got] == [0, 0]
    got = engine.query_dev([seg], [[(True, [])], [(True, []), (False, [(b"a", False)])]])
    assert [len(g) for g in got] == [0, 0]
    assert engine.query([], []) == []
    seg.release()


# ---------------------------------------------------------------- GPU, errors
def _raw(engine, dsegs, batch, removed=None):
    out = A.QueryOut()
    out.n_queries = 77  # must come back zeroed
    h = engine._handles(dsegs)
    rc = engine.lib.ii2_query_dev(h, len(dsegs), C.byref(batch) if batch is not None else None,
                                  removed, C.byref(out))
    if rc == A.II2_OK:
        engine.lib.ii2_query_out_free(C.byref(out))
    else:
        assert (out.n_queries, out.clause_values) == (0, 0) and not out.values and not out.value_off \
            and not out._owner
    return rc


@pytest.mark.gpu
def test_query_errors(engine):
    from inverted_index_2_b200.engine import Engine
    seg = engine.upload(FlatSegment.from_items([(b"a", [1]), (b"b", [1, 2])]))
    good_q = [[(True, [(b"a", False), (b"b", True)]), (False, [(b"b", False)])]]

    def batch(qs=good_q):
        return Engine._query_args(qs)

    b, keep = batch()
    assert _raw(engine, [seg], b) == A.II2_OK
    assert engine.lib.ii2_query_dev(engine._handles([seg]), 1, C.byref(b), None, None) == A.II2_ERR_INVALID
    assert _raw(engine, [seg], None) == A.II2_ERR_INVALID

    def mutate(field_array_index, idx, value):
        b, keep = batch()
        keep[field_array_index][idx] = value
        return _raw(engine, [seg], b), keep
    # keep = [blob, atom_off, kind, clause_atom_off, excluded, query_clause_off]
    assert mutate(1, 1, 5)[0] == A.II2_ERR_INVALID       # atom_off not monotone (5 > 2)
    assert mutate(1, 0, 1)[0] == A.II2_ERR_INVALID       # first atom offset != 0
    assert mutate(3, 0, 1)[0] == A.II2_ERR_INVALID       # first clause offset != 0
    assert mutate(3, 1, 4)[0] == A.II2_ERR_INVALID       # clause offsets not monotone
    assert mutate(3, 2, 2)[0] == A.II2_ERR_INVALID       # last clause offset != natoms
    assert mutate(5, 1, 1)[0] == A.II2_ERR_INVALID       # last query offset != nclauses
    assert mutate(5, 0, 1)[0] == A.II2_ERR_INVALID       # first query offset != 0
    assert mutate(2, 0, 2)[0] == A.II2_ERR_INVALID       # unknown atom kind
    assert mutate(4, 1, 2)[0] == A.II2_ERR_INVALID       # unknown clause flag
    assert mutate(4, 0, 1)[0] == A.II2_ERR_INVALID       # no required clause left
    b, keep = batch([[(False, [(b"a", False)])]])
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID
    b, keep = batch([[]])
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID   # a query without clauses
    b, keep = batch()
    b.atom_off = C.cast(None, A.u32p)
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID
    b, keep = batch()
    b.atom_bytes = C.cast(None, A.u8p)
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID
    # implementation limits
    b, keep = batch()
    assert _raw(engine, [seg] * 1025, b) == A.II2_ERR_UNSUPPORTED
    b, keep = batch([[(True, [(b"q" * 65536, False)])]])
    assert _raw(engine, [seg], b) == A.II2_ERR_UNSUPPORTED
    assert len(engine.query_dev([seg], [[(True, [(b"q" * 65535, True)])]])[0]) == 0  # longest allowed
    b, keep = batch([[(True, [(b"a", False)] * 1025)]])
    assert _raw(engine, [seg], b) == A.II2_ERR_UNSUPPORTED
    assert engine.query_dev([seg], [[(True, [(b"a", False)] * 1024)]])[0].tolist() == [1]
    # natoms x nseg >= 2^32: 2^22 one-atom clauses (empty terms) of one query over 1024 segments
    n = 1 << 22
    aoff, kind = np.zeros(n + 1, dtype=np.uint32), np.zeros(n, dtype=np.uint8)
    cao, excl = np.arange(n + 1, dtype=np.uint32), np.zeros(n, dtype=np.uint8)
    qco = np.array([0, n], dtype=np.uint32)
    b = A.QueryBatch()
    b.atom_bytes, b.atom_off, b.atom_kind, b.natoms = A.np_ptr(kind, A.u8p), A.np_ptr(aoff, A.u32p), \
        A.np_ptr(kind, A.u8p), n
    b.clause_atom_off, b.clause_excluded, b.nclauses = A.np_ptr(cao, A.u32p), A.np_ptr(excl, A.u8p), n
    b.query_clause_off, b.nqueries = A.np_ptr(qco, A.u32p), 1
    assert _raw(engine, [seg] * 1024, b) == A.II2_ERR_UNSUPPORTED
    seg.release()


@pytest.mark.gpu
def test_query_union_limit(engine):
    """A union of 2^32 values or more is II2_ERR_UNSUPPORTED: a term of 2^22 values held by 1024
    segments (the same 16 MiB segment 1024 times)."""
    seg = engine.upload(FlatSegment(np.frombuffer(b"big", dtype=np.uint8).copy(),
                                    np.array([0, 3], dtype=np.uint32), A.II2_SEG_DECODED,
                                    post=np.arange(1 << 22, dtype=np.uint32),
                                    post_off=np.array([0, 1 << 22], dtype=np.uint64)))
    from inverted_index_2_b200.engine import Engine
    b, keep = Engine._query_args([[(True, [(b"big", False)])]])
    assert _raw(engine, [seg] * 1024, b) == A.II2_ERR_UNSUPPORTED
    got = engine.query_dev([seg] * 4, [[(True, [(b"big", False), (b"bi", True)])]])
    assert np.array_equal(got[0], np.arange(1 << 22, dtype=np.uint32))
    seg.release()


# ---------------------------------------------------------------- GPU, full size
@pytest.mark.gpu
def test_query_c2_full_size(engine):
    """The C2 workload (64 segments, 100 M postings): queries of 1- and 2-byte prefixes and terms
    equal np.intersect1d / np.setdiff1d over the device's prefix_search_dev / lookup_dev lists."""
    w = synth.make_workload(1_000_000, 64, 100_000_000, seed=0xC2)
    dsegs = [engine.upload(s) for s in w.segments]
    n = len(w.term_off) - 1
    rng = np.random.default_rng(0xC2)
    t = lambda i: synth.term_at(w.term_bytes, w.term_off, int(i))
    qs = []
    for _ in range(24):
        a, b, c = (t(i) for i in rng.integers(0, n, size=3))
        qs += [[(True, [(a, False)]), (True, [(b[:2], True)])],
               [(True, [(a[:2], True)]), (True, [(b[:2], True)]), (False, [(c[:2], True)])],
               [(True, [(a[:1], True)]), (True, [(b[:1], True)])],
               [(True, [(a[:1], True)]), (False, [(b[:1], True), (c, False)])]]
    got = engine.query_dev(dsegs, qs)
    prefixes = sorted({p for q in qs for _, atoms in q for p, isp in atoms if isp})
    terms = sorted({p for q in qs for _, atoms in q for p, isp in atoms if not isp})
    pre = engine.prefix_search_dev(dsegs, prefixes)
    look = dict(zip(terms, engine.lookup_dev(dsegs, terms)))
    empty = np.zeros(0, dtype=np.uint32)

    def atom(p, isp):
        v = pre.get(p, empty) if isp else look[p]
        return empty if v is None else np.unique(v)

    for i, q in enumerate(qs):
        req, exc = [], []
        for r, atoms in q:
            u = empty
            for p, isp in atoms:
                u = np.union1d(u, atom(p, isp))
            (req if r else exc).append(u.astype(np.uint32))
        e = req[0]
        for x in req[1:]:
            e = np.intersect1d(e, x, assume_unique=True)
        for x in exc:
            e = np.setdiff1d(e, x, assume_unique=True)
        assert np.array_equal(got[i], e), (i, q)
    for s in dsegs:
        s.release()
