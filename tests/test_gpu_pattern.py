"""Wildcard (glob) and fuzzy term patterns (ii2_pattern_search, ii2_pattern_search_dev).

The expected answers never come from GPU code.  The terms and lists are those of the CPU oracle's
orc.read_range(segs) (or, on the full-size workload, the generator's own dictionary and lists); a
glob is translated to a Python `re` bytes pattern (fullmatch, DOTALL), a fuzzy pattern is decided
by a plain dynamic-programming Levenshtein distance, vectorised with numpy over the distinct terms;
the values of the matching terms are unioned with numpy."""
import ctypes as C
import re
import threading
import traceback

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A
from inverted_index_2_b200 import synth
from inverted_index_2_b200.flat import FlatSegment

PATTERN_SYMBOLS = ("ii2_pattern_search_dev", "ii2_pattern_search")
META = b"*?[]\\"


# ---------------------------------------------------------------- CPU, no device
def test_pattern_symbols_exported_and_bound():
    from inverted_index_2_b200.engine import load_library
    lib = load_library()
    for name in PATTERN_SYMBOLS:
        assert name in A.PROTOTYPES
        fn = getattr(lib, name)
        assert fn.restype == A.PROTOTYPES[name][0] and fn.argtypes == A.PROTOTYPES[name][1]


def test_pattern_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    from inverted_index_2_b200.engine import Engine, load_library
    lib = load_library()
    batch, keep = Engine._pattern_args([b"a*", (b"abc", 1, 0)])
    out = A.PrefixOut()
    assert lib.ii2_pattern_search_dev(None, 0, C.byref(batch), C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert lib.ii2_pattern_search(None, 0, C.byref(batch), C.byref(out)) == A.II2_ERR_NO_DEVICE
    assert out.n_prefixes == 0 and not out.values and not out.value_off and not out.matched


def test_pattern_packing():
    from inverted_index_2_b200.engine import Engine
    pats = [b"a*b", (b"hello", 2, 1), b"", (b"", 0, 0), b"[!x]?\\*"]
    b, keep = Engine._pattern_args(pats)
    n = int(b.npat)
    assert n == 5
    off = A.from_ptr(b.pat_off, n + 1, np.uint32)
    blob = A.from_ptr(b.pat_bytes, int(off[-1]), np.uint8).tobytes()
    kind = A.from_ptr(b.pat_kind, n, np.uint8).tolist()
    med = A.from_ptr(b.max_edits, n, np.uint8).tolist()
    pl = A.from_ptr(b.prefix_len, n, np.uint32).tolist()
    assert [blob[off[i]:off[i + 1]] for i in range(n)] == [b"a*b", b"hello", b"", b"", b"[!x]?\\*"]
    assert kind == [0, 1, 0, 1, 0] and med[1] == 2 and pl[1] == 1


def esc(t: bytes) -> bytes:
    """t as a glob of literals"""
    return b"".join(b"\\" + bytes([c]) if c in META else bytes([c]) for c in t)


def glob_regex(p: bytes):
    """The glob grammar of include/ii2.h as a compiled Python regex and its element count; None
    for a grammar error."""
    out, n, i, elems = [], len(p), 0, 0

    def lit(c):
        return re.escape(bytes([c]))
    while i < n:
        c = p[i]
        if c == ord("*"):
            out.append(b".*")
            i += 1
        elif c == ord("?"):
            out.append(b".")
            elems += 1
            i += 1
        elif c == ord("["):
            j, neg = i + 1, False
            if j < n and p[j] in b"!^":
                neg, j = True, j + 1
            members, first, closed = set(), True, False
            while j < n:
                if p[j] == ord("]") and not first:
                    closed = True
                    break
                first = False
                lo = p[j]
                if lo == ord("\\"):
                    j += 1
                    if j >= n:
                        break
                    lo = p[j]
                j += 1
                hi = lo
                if j + 1 < n and p[j] == ord("-") and p[j + 1] != ord("]"):
                    j += 1
                    hi = p[j]
                    if hi == ord("\\"):
                        j += 1
                        if j >= n:
                            break
                        hi = p[j]
                    j += 1
                members |= set(range(lo, hi + 1))
            if not closed:
                return None, 0
            if neg:
                members = set(range(256)) - members
            out.append(b"[" + b"".join(lit(x) for x in sorted(members)) + b"]" if members else b"(?!)")
            elems += 1
            i = j + 1
        elif c == ord("\\"):
            if i + 1 >= n:
                return None, 0
            out.append(lit(p[i + 1]))
            elems += 1
            i += 2
        else:
            out.append(lit(c))
            elems += 1
            i += 1
    return re.compile(b"".join(out), re.DOTALL), elems


def levenshtein(terms: list[bytes], q: bytes) -> np.ndarray:
    """Edit distance (insert / delete / substitute one byte) of q to every term: the plain
    dynamic program, one row per byte of q, vectorised over the terms."""
    n = len(terms)
    lens = np.array([len(t) for t in terms], dtype=np.int64)
    L = int(lens.max()) if n else 0
    T = np.full((n, max(L, 1)), -1, dtype=np.int16)
    for i, t in enumerate(terms):
        T[i, :len(t)] = np.frombuffer(t, dtype=np.uint8)
    prev = np.tile(np.arange(L + 1, dtype=np.int32), (n, 1))
    for i, c in enumerate(q, 1):
        best = np.minimum(prev[:, :-1] + (T[:, :L] != c), prev[:, 1:] + 1)
        cur = np.empty_like(prev)
        cur[:, 0] = i
        for j in range(1, L + 1):
            cur[:, j] = np.minimum(best[:, j - 1], cur[:, j - 1] + 1)
        prev = cur
    return prev[np.arange(n), lens] if n else np.zeros(0, dtype=np.int32)


def matches(terms: list[bytes], pat) -> np.ndarray:
    """Boolean mask over terms."""
    if isinstance(pat, bytes):
        rx, _ = glob_regex(pat)
        return np.array([rx.fullmatch(t) is not None for t in terms], dtype=bool)
    q, k, P = pat
    cand = np.array([t[:P] == q[:P] for t in terms], dtype=bool)
    out = np.zeros(len(terms), dtype=bool)
    idx = np.nonzero(cand)[0]
    if len(idx):
        out[idx] = levenshtein([terms[i][P:] for i in idx], q[P:]) <= k
    return out


class Expect:
    """Answers over the terms and lists of orc.read_range(segs)."""

    def __init__(self, orc, segs):
        r = orc.read_range(segs)
        self.terms = [bytes(r.term_bytes[r.term_off[i]:r.term_off[i + 1]]) for i in range(r.n_terms)]
        self.lists = [np.asarray(r.post[r.post_off[i]:r.post_off[i + 1]], dtype=np.uint32)
                      for i in range(r.n_terms)]

    def answer(self, pat):
        m = np.nonzero(matches(self.terms, pat))[0]
        if len(m) == 0:
            return None
        return np.unique(np.concatenate([self.lists[i] for i in m] + [np.zeros(0, np.uint32)])).astype(np.uint32)


def same(got, exp):
    if exp is None:
        return got is None
    return got is not None and got.dtype == np.uint32 and np.array_equal(got, exp)


def check(got, exp, pats):
    assert len(got) == len(pats)
    for i, (g, e, p) in enumerate(zip(got, exp, pats)):
        assert same(g, e), (i, p, None if g is None else g[:8], None if e is None else e[:8])


# ---------------------------------------------------------------- random vocabularies
def _vocab(rng, n):
    """Terms over every byte value, with metacharacters, empty and > 64-byte terms."""
    out = {bytes(rng.choice(list(b"abcxyz*?[]\\-!^"), size=int(rng.integers(1, 9))).tolist())
           for _ in range(n)}
    out |= {bytes(rng.integers(0, 256, size=int(rng.integers(1, 6))).tolist()) for _ in range(n // 4)}
    out |= {b"", b"a" * 70, b"ab" * 40 + b"x", b"\x00", b"\xff" * 3}
    return sorted(out)


def _segments(rng, vocab, nseg):
    segs = []
    for s in range(nseg):
        if s % 17 == 5:
            segs.append(FlatSegment.from_items([]))  # an empty segment
            continue
        frac = rng.choice([0.1, 0.4, 0.9]) if nseg < 64 else 0.05
        items = []
        for t in vocab:
            if rng.random() >= frac:
                continue
            n = int(rng.choice([0, 1, 3, 20, 200], p=[.1, .3, .3, .2, .1]))
            vals = rng.integers(0, 1 << 14, size=n, dtype=np.int64)
            if rng.random() < 0.7:
                vals = np.unique(vals)
            items.append((t, vals.tolist()))  # else unsorted, with duplicates
        segs.append(FlatSegment.from_items(items))
    return segs


def _glob_from(rng, t):
    """A glob made from term t: metacharacters escaped, then ?, *, sets, negated sets and ranges
    spliced in."""
    parts = [esc(bytes([c])) for c in t[:40]] + ([b"*"] if len(t) > 40 else [])  # <= 63 elements
    for _ in range(int(rng.integers(0, 4))):
        pos = int(rng.integers(0, len(parts) + 1))
        r = rng.random()
        if r < 0.25:
            parts.insert(pos, b"*")
        elif r < 0.45 and parts:
            parts[min(pos, len(parts) - 1)] = b"?"
        elif r < 0.6 and parts:
            i = min(pos, len(parts) - 1)
            c = t[i] if i < len(t) else ord("a")
            parts[i] = b"[" + esc(bytes([c])) + b"xz]"
        elif r < 0.75 and parts:
            i = min(pos, len(parts) - 1)
            parts[i] = b"[!" + esc(bytes([int(rng.integers(0, 256))])) + b"]"
        elif r < 0.9 and parts:
            i = min(pos, len(parts) - 1)
            parts[i] = b"[a-y\\]]"
        else:
            parts.insert(pos, b"*")
            parts.insert(pos, b"*")
    return b"".join(parts)


def _fuzzy_from(rng, t):
    """t with 0 .. 3 random single-byte edits, max_edits 0 .. 2, P 0 .. 3 (clipped)."""
    q = bytearray(t)
    for _ in range(int(rng.integers(0, 4))):
        r = rng.random()
        i = int(rng.integers(0, len(q) + 1))
        if r < 0.34:
            q.insert(i, int(rng.integers(0, 256)))
        elif r < 0.67 and q:
            del q[min(i, len(q) - 1)]
        elif q:
            q[min(i, len(q) - 1)] = int(rng.integers(0, 256))
    q = bytes(q[:64])
    return (q, int(rng.integers(0, 3)), min(int(rng.integers(0, 4)), len(q)))


def _patterns(rng, vocab, n):
    pats = []
    for _ in range(n):
        t = vocab[int(rng.integers(0, len(vocab)))]
        pats.append(_glob_from(rng, t) if rng.random() < 0.55 else _fuzzy_from(rng, t))
    pats += [b"*", b"", b"*a*", b"?", b"??*", (b"", 2, 0), b"[]]*", b"*\\*", b"[^a-z]*"]
    pats += [pats[int(i)] for i in rng.integers(0, len(pats), size=4)]  # duplicates
    return pats


@pytest.mark.gpu
@pytest.mark.parametrize("nseg", [1, 3, 64, 300])
def test_pattern_random(engine, orc, nseg):
    rng = np.random.default_rng(4000 + nseg)
    vocab = _vocab(rng, 80)
    segs = _segments(rng, vocab, nseg)
    pats = _patterns(rng, vocab, 120)
    exp = Expect(orc, segs)
    dsegs = [engine.upload(s) for s in segs]
    got = engine.pattern_search_dev(dsegs, pats)
    check(got, [exp.answer(p) for p in pats], pats)
    if nseg == 3:  # the host-view entry point gives the same answers
        again = engine.pattern_search(segs, pats)
        assert all(same(a, b) for a, b in zip(again, got))
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_equivalences(engine, orc):
    """glob esc(p)* == prefix_search_dev(p); glob esc(t) and fuzzy (t, 0, 0) == the TERM atom of
    query_dev (the sorted-unique values of t), over a vocabulary with every byte value."""
    rng = np.random.default_rng(77)
    vocab = _vocab(rng, 120) + [bytes([c]) + b"q" for c in range(256)]
    vocab = sorted(set(vocab))
    segs = _segments(rng, vocab, 5)
    dsegs = [engine.upload(s) for s in segs]
    picks = [vocab[int(i)] for i in rng.integers(0, len(vocab), size=60)] + [b"", b"zz-absent"]
    prefixes = sorted({t[:int(rng.integers(0, len(t) + 1))] for t in picks}) + [b"\xfe"]
    got = engine.pattern_search_dev(dsegs, [esc(p) + b"*" for p in prefixes])
    ref = engine.prefix_search_dev(dsegs, prefixes)
    for p, g in zip(prefixes, got):
        assert same(g, ref.get(p)), p
    terms = [t for t in picks if len(t) <= 63]  # a literal glob / fuzzy word within the limits
    lit = engine.pattern_search_dev(dsegs, [esc(t) for t in terms])
    fz = engine.pattern_search_dev(dsegs, [(t, 0, 0) for t in terms])
    fzp = engine.pattern_search_dev(dsegs, [(t, 0, len(t)) for t in terms])
    q = engine.query_dev(dsegs, [[(True, [(t, False)])] for t in terms])
    look = engine.lookup_dev(dsegs, terms)
    for t, a, b, c, d, lk in zip(terms, lit, fz, fzp, q, look):
        assert (a is None) == (lk is None), t
        e = d if lk is not None else None
        assert same(a, e) and same(b, e) and same(c, e), t
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_dense_star(engine):
    """`*` over a workload whose union is dense enough for the bitmap path, and `?*` / `*?*`
    (every non-empty term) against numpy."""
    w = synth.make_workload(20000, 16, 400000, universe=1 << 18, seed=31)
    dsegs = [engine.upload(s) for s in w.segments]
    got = engine.pattern_search_dev(dsegs, [b"*", b"?*", b"*?*", b"**"])
    exp = np.unique(np.concatenate([s.post for s in w.segments])).astype(np.uint32)
    assert len(exp) >= 1 << 16
    for g in got:
        assert same(g, exp)
    for s in dsegs:
        s.release()


def _small_workload():
    w = synth.make_workload(20000, 16, 400000, universe=1 << 18, seed=32)
    t = lambda i: synth.term_at(w.term_bytes, w.term_off, int(i))
    return w, len(w.term_off) - 1, t


def _workload_patterns(rng, n, t, count):
    pats = []
    for _ in range(count):
        a = t(rng.integers(0, n))
        r = int(rng.integers(0, 5))
        if r == 0:
            pats.append(a[:3] + b"*")
        elif r == 1:
            pats.append(b"*" + a[2:5] + b"*")
        elif r == 2:
            pats.append(a[:2] + b"?" + a[3:])
        else:
            pats.append((a[:-1] + b"Q", int(rng.integers(1, 3)), int(rng.integers(0, 3))))
    return pats


@pytest.mark.gpu
def test_pattern_batch_equals_single_calls(engine, orc):
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    pats = _workload_patterns(np.random.default_rng(5), n, t, 60)
    pats += pats[:7]  # duplicates
    batch = engine.pattern_search_dev(dsegs, pats)
    for i, p in enumerate(pats):
        assert same(batch[i], engine.pattern_search_dev(dsegs, [p])[0]), (i, p)
    exp = Expect(orc, w.segments)
    check(batch, [exp.answer(p) for p in pats], pats)
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_concurrent_threads(engine):
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    batches = [_workload_patterns(np.random.default_rng(300 + k), n, t, 40) for k in range(8)]
    serial = [engine.pattern_search_dev(dsegs, b) for b in batches]
    results, errs = [None] * 8, []

    def run(k):
        try:
            for _ in range(3):
                results[k] = engine.pattern_search_dev(dsegs, batches[k])
        except BaseException:
            errs.append(traceback.format_exc())
    ts = [threading.Thread(target=run, args=(k,)) for k in range(8)]
    [x.start() for x in ts]
    [x.join() for x in ts]
    assert not errs, "\n".join(errs)
    for s_, r in zip(serial, results):
        assert len(s_) == len(r) and all(same(a, b) for a, b in zip(s_, r))
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_gather_devices_halves(engine):
    """ii2_prefix_gather_devices of two calls over the two halves of the segments equals one call
    over all of them."""
    w, n, t = _small_workload()
    dsegs = [engine.upload(s) for s in w.segments]
    pats = _workload_patterns(np.random.default_rng(9), n, t, 30) + [b"*", b"zzz*"]
    whole = engine.pattern_search_dev(dsegs, pats)
    parts = [engine.pattern_search_dev_out(dsegs[:7], pats), engine.pattern_search_dev_out(dsegs[7:], pats)]
    try:
        keys = list(range(len(pats)))
        merged = engine.prefix_gather_devices(parts, keys, 0)
    finally:
        for o in parts:
            engine.prefix_out_free(o)
    for i, g in enumerate(whole):
        assert same(merged.get(i), g), (i, pats[i])
    for s in dsegs:
        s.release()


@pytest.mark.gpu
def test_pattern_empty_calls(engine):
    seg = engine.upload(FlatSegment.from_items([(b"", []), (b"a", [1]), (b"b", [])]))
    assert engine.pattern_search_dev([seg], []) == []
    assert engine.pattern_search_dev([], [b"*", (b"a", 1, 0)]) == [None, None]
    assert engine.pattern_search([], []) == []
    got = engine.pattern_search_dev([seg], [b"", b"b", b"?", b"c*", (b"", 0, 0), (b"x", 1, 0)])
    assert [None if g is None else g.tolist() for g in got] == [[], [], [1], None, [], [1]]
    seg.release()


def _raw(engine, dsegs, batch):
    out = A.PrefixOut()
    out.n_prefixes = 77  # must come back zeroed
    rc = engine.lib.ii2_pattern_search_dev(engine._handles(dsegs), len(dsegs),
                                           C.byref(batch) if batch is not None else None, C.byref(out))
    if rc == A.II2_OK:
        engine.lib.ii2_prefix_out_free(C.byref(out))
    else:
        assert out.n_prefixes == 0 and not out.values and not out.value_off and not out.matched \
            and not out._owner
    return rc


@pytest.mark.gpu
def test_pattern_errors_and_limits(engine):
    from inverted_index_2_b200.engine import Engine
    seg = engine.upload(FlatSegment.from_items([(b"a" * 70, [3]), (b"ab", [1]), (b"b", [1, 2])]))

    def rc(pats, segs=None):
        b, keep = Engine._pattern_args(pats)
        return _raw(engine, [seg] if segs is None else segs, b)
    assert rc([b"a*"]) == A.II2_OK
    assert engine.lib.ii2_pattern_search_dev(engine._handles([seg]), 1, None, None) == A.II2_ERR_INVALID
    assert _raw(engine, [seg], None) == A.II2_ERR_INVALID
    # grammar
    for bad in (b"[abc", b"ab\\", b"\\", b"[", b"[]", b"[!]", b"[a\\", b"[a-\\", b"ok*", b"x[]]["):
        assert rc([b"a*", bad]) == (A.II2_OK if bad == b"ok*" else A.II2_ERR_INVALID), bad
        assert glob_regex(bad)[0] is None or bad == b"ok*"
    assert rc([(b"ab", 1, 3)]) == A.II2_ERR_INVALID                      # P > len(q)
    assert rc([(b"ab", 1, 2)]) == A.II2_OK
    b, keep = Engine._pattern_args([b"a", (b"b", 1, 0)])
    keep[2][0] = 2
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID                   # unknown kind
    b, keep = Engine._pattern_args([b"a", b"b"])
    keep[1][1] = 5
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID                   # offsets not monotone
    b, keep = Engine._pattern_args([b"a", b"b"])
    keep[1][0] = 1
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID                   # first offset != 0
    b, keep = Engine._pattern_args([(b"a", 1, 0)])
    b.max_edits = C.cast(None, A.u8p)
    assert _raw(engine, [seg], b) == A.II2_ERR_INVALID                   # fuzzy without max_edits
    b, keep = Engine._pattern_args([b"a*"])
    b.max_edits, b.prefix_len = C.cast(None, A.u8p), C.cast(None, A.u32p)
    assert _raw(engine, [seg], b) == A.II2_OK                            # NULLs without fuzzy
    # an INVALID pattern wins over an UNSUPPORTED one
    assert rc([b"a" * 64, b"[x"]) == A.II2_ERR_INVALID
    # limits at their boundaries
    assert rc([b"a" * 63]) == A.II2_OK and rc([b"a" * 64]) == A.II2_ERR_UNSUPPORTED
    assert rc([b"*".join([b"?"] * 63) + b"*"]) == A.II2_OK
    assert rc([b"[ab]" * 64]) == A.II2_ERR_UNSUPPORTED
    assert rc([(b"a" * 64, 2, 0)]) == A.II2_OK and rc([(b"a" * 65, 2, 0)]) == A.II2_ERR_UNSUPPORTED
    assert rc([(b"a" * 66, 1, 2)]) == A.II2_OK and rc([(b"a" * 67, 1, 2)]) == A.II2_ERR_UNSUPPORTED
    assert rc([(b"ab", 3, 0)]) == A.II2_ERR_UNSUPPORTED
    assert rc([b"*" * 65535]) == A.II2_OK and rc([b"*" * 65536]) == A.II2_ERR_UNSUPPORTED
    assert rc([b"a*"], [seg] * 1025) == A.II2_ERR_UNSUPPORTED
    assert rc([b"a*"], [seg] * 1024) == A.II2_OK
    got = engine.pattern_search_dev([seg], [b"a" * 63, b"a" * 62 + b"*", (b"a" * 64, 2, 0), (b"a" * 68, 2, 4),
                                            b"?" * 63 + b"*", (b"ab", 2, 0)])
    assert [None if g is None else g.tolist() for g in got] == [None, [3], None, [3], [3], [1, 2]]
    # npat x nseg >= 2^32: 2^22 copies of one pattern over 1024 segments
    n = 1 << 22
    off = np.arange(n + 1, dtype=np.uint32)
    blob = np.full(n + 1, ord("b"), dtype=np.uint8)
    kind = np.zeros(n, dtype=np.uint8)
    b = A.PatternBatch()
    b.pat_bytes, b.pat_off, b.pat_kind, b.npat = A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p), \
        A.np_ptr(kind, A.u8p), n
    assert _raw(engine, [seg] * 1024, b) == A.II2_ERR_UNSUPPORTED
    seg.release()


@pytest.mark.gpu
def test_pattern_union_limit(engine):
    """A pattern whose matched postings reach 2^32 is II2_ERR_UNSUPPORTED: a term of 2^22 values
    held by 1024 segments (the same segment 1024 times)."""
    seg = engine.upload(FlatSegment(np.frombuffer(b"big", dtype=np.uint8).copy(),
                                    np.array([0, 3], dtype=np.uint32), A.II2_SEG_DECODED,
                                    post=np.arange(1 << 22, dtype=np.uint32),
                                    post_off=np.array([0, 1 << 22], dtype=np.uint64)))
    from inverted_index_2_b200.engine import Engine
    b, keep = Engine._pattern_args([b"b*"])
    assert _raw(engine, [seg] * 1024, b) == A.II2_ERR_UNSUPPORTED
    b, keep = Engine._pattern_args([b"*g", (b"bug", 1, 0)])
    assert _raw(engine, [seg] * 1024, b) == A.II2_ERR_UNSUPPORTED
    got = engine.pattern_search_dev([seg] * 4, [b"b?g", (b"bg", 1, 1), b"*x"])
    assert same(got[0], np.arange(1 << 22, dtype=np.uint32)) and same(got[1], got[0]) and got[2] is None
    seg.release()


# ---------------------------------------------------------------- GPU, full size
@pytest.mark.gpu
def test_pattern_c3_full_size(engine):
    """The C3 workload (1 M terms, 256 segments, 100 M postings): a few anchored and unanchored
    globs and fuzzy patterns against numpy over the generator's dictionary and lists."""
    w = synth.make_workload(1_000_000, 256, 100_000_000, seed=0xC3, presence=0.125)
    dsegs = [engine.upload(s) for s in w.segments]
    n = len(w.term_off) - 1
    terms = [synth.term_at(w.term_bytes, w.term_off, i) for i in range(n)]
    rng = np.random.default_rng(0xC3)
    a, b, c = (terms[int(i)] for i in rng.integers(0, n, size=3))
    pats = [a[:3] + b"*", b"*" + b[3:6] + b"*", b"*" + c[-2:], a[:2] + b"?" + a[3:5] + b"*", b"*[xyz]Q*",
            (a[:-1] + b"z", 1, 0), (b[1:], 2, 0), (c + b"k", 1, 2), (a[:6] + a[7:], 2, 2)]
    got = engine.pattern_search_dev(dsegs, pats)
    for p, g in zip(pats, got):
        hit = np.nonzero(matches(terms, p))[0]
        parts = []
        for seg, ids in zip(w.segments, w.seg_term_ids):
            sel = np.nonzero(np.isin(ids, hit))[0]
            for i in sel:
                parts.append(seg.post[seg.post_off[i]:seg.post_off[i + 1]])
        exp = np.unique(np.concatenate(parts)).astype(np.uint32) if parts else None
        assert same(g, exp), p
    for s in dsegs:
        s.release()
