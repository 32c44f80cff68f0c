"""The terms each wildcard or fuzzy pattern matches (ii2_pattern_terms, ii2_pattern_terms_dev).

The expected answers never come from GPU code.  A glob is decided by a Python `re` bytes pattern
and a fuzzy pattern by a numpy dynamic-programming Levenshtein distance (the helpers of
test_gpu_pattern.py); the matching terms are grouped by bytes over the segments' own dictionaries
(or, at full size, over the generator's term ids), counting instances and stored list lengths."""
import ctypes as C
import threading
import traceback

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A
from inverted_index_2_b200 import synth
from inverted_index_2_b200.flat import FlatSegment
from test_gpu_pattern import (_patterns, _raw, _segments, _small_workload, _vocab, _workload_patterns,
                              esc, levenshtein, matches, same)

TERMS_SYMBOLS = ("ii2_pattern_terms_dev", "ii2_pattern_terms", "ii2_terms_out_free")


# ---------------------------------------------------------------- CPU, no device
def test_pattern_terms_symbols_exported_and_bound():
    from inverted_index_2_b200.engine import load_library
    lib = load_library()
    for name in TERMS_SYMBOLS:
        assert name in A.PROTOTYPES
        fn = getattr(lib, name)
        assert fn.restype == A.PROTOTYPES[name][0] and fn.argtypes == A.PROTOTYPES[name][1]


def test_pattern_terms_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    from inverted_index_2_b200.engine import Engine, load_library
    lib = load_library()
    batch, keep = Engine._pattern_args([b"a*", (b"abc", 1, 0)])
    out = A.TermsOut()
    assert lib.ii2_pattern_terms_dev(None, 0, C.byref(batch), C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert lib.ii2_pattern_terms(None, 0, C.byref(batch), C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert out.n_patterns == 0 and out.n_terms == 0 and not out.term_bytes and not out._owner


# ---------------------------------------------------------------- the oracle
class TermOracle:
    """(term, segments, postings, distance) of every pattern over the segments' dictionaries."""

    def __init__(self, segs):
        self.segs = [(s.terms(), np.diff(s.post_off).astype(np.int64).tolist()) for s in segs]
        self.vocab = sorted({t for terms, _ in self.segs for t in terms})

    def answer(self, pat):
        hit = {self.vocab[i] for i in np.nonzero(matches(self.vocab, pat))[0]}
        stats = {}
        for terms, lens in self.segs:
            for t, n in zip(terms, lens):
                if t in hit:
                    st = stats.setdefault(t, [0, 0])
                    st[0] += 1
                    st[1] += n
        out = sorted(stats)
        if isinstance(pat, bytes) or not out:
            dist = [0] * len(out)
        else:
            q, k, P = pat
            dist = levenshtein([t[P:] for t in out], q[P:]).tolist()
        return [(t, stats[t][0], stats[t][1], int(d)) for t, d in zip(out, dist)]


def check_terms(got, exp, pats):
    assert len(got) == len(exp) == len(pats)
    for i, (g, e, p) in enumerate(zip(got, exp, pats)):
        assert g == e, (i, p, g[:4], e[:4])


# ---------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("nseg", [1, 3, 64, 300])
def test_pattern_terms_random(engine, nseg):
    rng = np.random.default_rng(5000 + nseg)
    vocab = _vocab(rng, 80)
    segs = _segments(rng, vocab, nseg)
    pats = _patterns(rng, vocab, 120)
    dsegs = [engine.upload(s) for s in segs]
    got = engine.pattern_terms_dev(dsegs, pats)
    oracle = TermOracle(segs)
    check_terms(got, [oracle.answer(p) for p in pats], pats)
    # a pattern has terms exactly when pattern search says it matched
    search = engine.pattern_search_dev(dsegs, pats)
    assert [len(g) > 0 for g in got] == [v is not None for v in search]
    if nseg == 3:
        assert engine.pattern_terms(segs, pats) == got  # the host-view entry point
        # a handle passed twice counts twice
        twice = engine.pattern_terms_dev(dsegs + dsegs[:1], pats)
        check_terms(twice, [TermOracle(segs + segs[:1]).answer(p) for p in pats], pats)
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_terms_agree_with_lookup_and_reads(engine):
    """The sorted-unique union of lookup_dev over a pattern's terms is pattern_search_dev's
    answer; glob esc(p)* returns the distinct terms of read_range_dev that start with p."""
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    pats = _workload_patterns(np.random.default_rng(11), n, t, 40) + [b"*", b"zzz*"]
    terms = engine.pattern_terms_dev(dsegs, pats)
    search = engine.pattern_search_dev(dsegs, pats)
    for p, ts, v in zip(pats, terms, search):
        if not ts:
            assert v is None, p
            continue
        lists = engine.lookup_dev(dsegs, [x[0] for x in ts])
        assert all(lst is not None for lst in lists), p
        assert same(np.unique(np.concatenate(lists)).astype(np.uint32), v), p
        assert sum(x[2] for x in ts) >= len(v)
    r = engine.read_range_dev(dsegs)
    try:
        rr = r.download_read()
    finally:
        r.release()
    tb = rr.term_bytes.tobytes()
    every = [tb[rr.term_off[i]:rr.term_off[i + 1]] for i in range(len(rr.term_off) - 1)]
    rng = np.random.default_rng(12)
    prefixes = sorted({every[int(i)][:int(rng.integers(0, 6))] for i in rng.integers(0, len(every), 30)})
    prefixes += [b"", b"\xff"]
    got = engine.pattern_terms_dev(dsegs, [esc(p) + b"*" for p in prefixes])
    for p, g in zip(prefixes, got):
        assert [x[0] for x in g] == [x for x in every if x.startswith(p)], p
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_terms_batch_and_empty_calls(engine):
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    pats = _workload_patterns(np.random.default_rng(5), n, t, 50)
    pats += pats[:7] + [b"*", b"*"]  # repeats
    batch = engine.pattern_terms_dev(dsegs, pats)
    for i, p in enumerate(pats):
        assert batch[i] == engine.pattern_terms_dev(dsegs, [p])[0], (i, p)
    check_terms(batch, [TermOracle(w.segments).answer(p) for p in pats], pats)
    assert len(batch[-1]) == len({x for s in w.segments for x in s.terms()})
    assert engine.pattern_terms_dev(dsegs, []) == []
    assert engine.pattern_terms_dev([], [b"*", (b"a", 1, 0)]) == [[], []]
    assert engine.pattern_terms([], []) == []
    for s in dsegs:
        s.release()
    seg = engine.upload(FlatSegment.from_items([(b"", []), (b"a", [1]), (b"ab", [2, 2]), (b"b", [])]))
    got = engine.pattern_terms_dev([seg, seg], [b"", b"b", b"?", b"c*", (b"", 0, 0), (b"x", 1, 0),
                                                (b"ac", 2, 0), b"a*"])
    assert got == [[(b"", 2, 0, 0)], [(b"b", 2, 0, 0)], [(b"a", 2, 2, 0), (b"b", 2, 0, 0)], [],
                   [(b"", 2, 0, 0)], [(b"", 2, 0, 1), (b"a", 2, 2, 1), (b"b", 2, 0, 1)],
                   [(b"", 2, 0, 2), (b"a", 2, 2, 1), (b"ab", 2, 4, 1), (b"b", 2, 0, 2)],
                   [(b"a", 2, 2, 0), (b"ab", 2, 4, 0)]]
    seg.release()


@pytest.mark.gpu
def test_pattern_terms_concurrent_threads(engine):
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    batches = [_workload_patterns(np.random.default_rng(400 + k), n, t, 30) for k in range(8)]
    serial = [engine.pattern_terms_dev(dsegs, b) for b in batches]
    results, errs = [None] * 8, []

    def run(k):
        try:
            for _ in range(3):
                results[k] = engine.pattern_terms_dev(dsegs, batches[k])
        except BaseException:
            errs.append(traceback.format_exc())
    ts = [threading.Thread(target=run, args=(k,)) for k in range(8)]
    [x.start() for x in ts]
    [x.join() for x in ts]
    assert not errs, "\n".join(errs)
    assert serial == results
    for s in dsegs:
        s.release()


def _raw_terms(engine, dsegs, batch):
    out = A.TermsOut()
    out.n_terms = 77  # must come back zeroed
    rc = engine.lib.ii2_pattern_terms_dev(engine._handles(dsegs), len(dsegs),
                                          C.byref(batch) if batch is not None else None, C.byref(out))
    if rc == A.II2_OK:
        engine.lib.ii2_terms_out_free(C.byref(out))
    else:
        assert out.n_terms == 0 and out.n_patterns == 0 and not out.term_bytes and not out._owner
    return rc


@pytest.mark.gpu
def test_pattern_terms_errors_and_limits(engine):
    """Every grammar error and limit gives pattern search's error code."""
    from inverted_index_2_b200.engine import Engine
    seg = engine.upload(FlatSegment.from_items([(b"a" * 70, [3]), (b"ab", [1]), (b"b", [1, 2])]))
    assert engine.lib.ii2_pattern_terms_dev(engine._handles([seg]), 1, None, None) == A.II2_ERR_INVALID
    assert _raw_terms(engine, [seg], None) == A.II2_ERR_INVALID

    def both(b, segs):
        return _raw_terms(engine, segs, b), _raw(engine, segs, b)
    cases = [[b"a*", bad] for bad in (b"[abc", b"ab\\", b"\\", b"[", b"[]", b"[!]", b"[a\\", b"[a-\\",
                                      b"ok*", b"x[]][")]
    cases += [[(b"ab", 1, 3)], [(b"ab", 1, 2)], [b"a" * 64, b"[x"], [b"a" * 63], [b"a" * 64],
              [b"*".join([b"?"] * 63) + b"*"], [b"[ab]" * 64], [(b"a" * 64, 2, 0)], [(b"a" * 65, 2, 0)],
              [(b"a" * 66, 1, 2)], [(b"a" * 67, 1, 2)], [(b"ab", 3, 0)], [b"*" * 65535], [b"*" * 65536]]
    codes = set()
    for pats in cases:
        b, keep = Engine._pattern_args(pats)
        t, p = both(b, [seg])
        assert t == p, pats
        codes.add(t)
    assert codes == {A.II2_OK, A.II2_ERR_INVALID, A.II2_ERR_UNSUPPORTED}
    b, keep = Engine._pattern_args([b"a*"])
    assert both(b, [seg] * 1024) == (A.II2_OK,) * 2
    assert both(b, [seg] * 1025) == (A.II2_ERR_UNSUPPORTED,) * 2
    # malformed batches
    b, keep = Engine._pattern_args([b"a", (b"b", 1, 0)])
    keep[2][0] = 2
    assert both(b, [seg]) == (A.II2_ERR_INVALID,) * 2                     # unknown kind
    b, keep = Engine._pattern_args([b"a", b"b"])
    keep[1][1] = 5
    assert both(b, [seg]) == (A.II2_ERR_INVALID,) * 2                     # offsets not monotone
    b, keep = Engine._pattern_args([b"a", b"b"])
    keep[1][0] = 1
    assert both(b, [seg]) == (A.II2_ERR_INVALID,) * 2                     # first offset != 0
    b, keep = Engine._pattern_args([(b"a", 1, 0)])
    b.max_edits = C.cast(None, A.u8p)
    assert both(b, [seg]) == (A.II2_ERR_INVALID,) * 2                     # fuzzy without max_edits
    b, keep = Engine._pattern_args([b"a*"])
    b.max_edits, b.prefix_len = C.cast(None, A.u8p), C.cast(None, A.u32p)
    assert both(b, [seg]) == (A.II2_OK,) * 2                              # NULLs without fuzzy
    # npat x nseg >= 2^32: 2^22 copies of one pattern over 1024 segments
    n = 1 << 22
    off = np.arange(n + 1, dtype=np.uint32)
    blob = np.full(n + 1, ord("b"), dtype=np.uint8)
    kind = np.zeros(n, dtype=np.uint8)
    b = A.PatternBatch()
    b.pat_bytes, b.pat_off, b.pat_kind, b.npat = A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p), \
        A.np_ptr(kind, A.u8p), n
    assert _raw_terms(engine, [seg] * 1024, b) == A.II2_ERR_UNSUPPORTED
    # the union limit of pattern search does not apply: 1024 instances of a 2^22-value list
    big = engine.upload(FlatSegment(np.frombuffer(b"big", dtype=np.uint8).copy(),
                                    np.array([0, 3], dtype=np.uint32), A.II2_SEG_DECODED,
                                    post=np.arange(1 << 22, dtype=np.uint32),
                                    post_off=np.array([0, 1 << 22], dtype=np.uint64)))
    assert engine.pattern_terms_dev([big] * 1024, [b"b*", (b"bug", 1, 0)]) == \
        [[(b"big", 1024, 1 << 32, 0)], [(b"big", 1024, 1 << 32, 1)]]
    big.release()
    got = engine.pattern_terms_dev([seg], [b"a" * 62 + b"*", (b"a" * 68, 2, 4), (b"ab", 2, 0)])
    assert got == [[(b"a" * 70, 1, 1, 0)], [(b"a" * 70, 1, 1, 2)], [(b"ab", 1, 1, 0), (b"b", 1, 2, 1)]]
    seg.release()


# ---------------------------------------------------------------- GPU, full size
@pytest.mark.gpu
def test_pattern_terms_c3_full_size(engine):
    """The C3 workload (1 M terms, 256 segments, 100 M postings): `*` returns every distinct term
    with its instance and posting counts from the generator; the mixed patterns of the pattern
    search test against numpy over the generator's dictionary."""
    w = synth.make_workload(1_000_000, 256, 100_000_000, seed=0xC3, presence=0.125)
    dsegs = [engine.upload(s) for s in w.segments]
    n = len(w.term_off) - 1
    terms = [synth.term_at(w.term_bytes, w.term_off, i) for i in range(n)]
    inst = np.zeros(n, dtype=np.int64)
    post = np.zeros(n, dtype=np.int64)
    for seg, ids in zip(w.segments, w.seg_term_ids):
        np.add.at(inst, ids, 1)
        np.add.at(post, ids, np.diff(seg.post_off).astype(np.int64))
    rng = np.random.default_rng(0xC3)
    a, b, c = (terms[int(i)] for i in rng.integers(0, n, size=3))
    pats = [b"*", a[:3] + b"*", b"*" + b[3:6] + b"*", b"*" + c[-2:], a[:2] + b"?" + a[3:5] + b"*",
            b"*[xyz]Q*", (a[:-1] + b"z", 1, 0), (b[1:], 2, 0), (c + b"k", 1, 2), (a[:6] + a[7:], 2, 2)]
    got = engine.pattern_terms_dev(dsegs, pats)
    for p, g in zip(pats, got):
        hit = np.arange(n) if p == b"*" else np.nonzero(matches(terms, p))[0]
        hit = [int(i) for i in hit if inst[i]]
        hit.sort(key=lambda i: terms[i])
        if isinstance(p, bytes):
            dist = [0] * len(hit)
        else:
            dist = levenshtein([terms[i][p[2]:] for i in hit], p[0][p[2]:]).tolist() if hit else []
        exp = [(terms[i], int(inst[i]), int(post[i]), int(d)) for i, d in zip(hit, dist)]
        assert g == exp, (p, g[:3], exp[:3])
    assert len(got[0]) == int((inst > 0).sum()) and sum(x[1] for x in got[0]) == int(inst.sum())
    assert sum(x[2] for x in got[0]) == sum(int(s.post_off[-1]) for s in w.segments)
    for s in dsegs:
        s.release()
