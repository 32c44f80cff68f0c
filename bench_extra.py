#!/usr/bin/env python3
"""bench_extra.py — the other BASELINE.json configurations, one JSON line each:
  C1  4 x Put(all terms) + Merge as one ii2_ingest call (device sort of every document)
  C3  term-range read union across 256 segments with 5 % removed_list filtering (µs per call)
  C4  file/bitmask + intcomp encode/decode sweep, posting-list lengths 16 .. 16M
  prefix  PrefixSearch batches over 64 resident segments (µs per call)
  lookup  batched exact-term reads (ii2_lookup_dev) on the C3 and C2 workloads, Q = 1 .. 65 536
        keys per call, against a loop of point reads for Q <= 256
  query  boolean queries (ii2_query_dev) on the C2 and C3 workloads, Q = 1 .. 4096 per call, three
        shapes, against lookup_dev + prefix_search_dev + host numpy set operations
  multidev  one process over every visible GPU (Engine(devices=...)): weak-scaling compaction from
        one host thread per device, a 1 % read partitioned over the devices + ii2_read_gather_devices,
        and ii2_prefix_gather_devices of the prefix batch; each checked against one device
bench.py stays the headline (C2 compaction); these lines are evidence for SURVEY §8 rows."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from inverted_index_2_b200 import synth  # noqa: E402


def _peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"])
    except Exception:
        return 6650.0


PEAK = _peak()  # GB/s, measured copy bandwidth (fallback: B200_PROFILING.md)


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), float(np.percentile(ts, 99))


def c3(eng, a):
    w = synth.make_workload(a.terms, 256, a.postings, seed=0xC3, presence=0.125)
    dsegs = [eng.upload(s) for s in w.segments]
    drem = eng.upload_removed(w.removed)
    n = len(w.term_off) - 1
    rng = np.random.default_rng(3)
    out = []
    for frac in (0.001, 0.01, 0.1, 1.0):
        span = max(1, int(n * frac))
        lat, info = [], None
        for _ in range(16 if frac < 1 else 4):
            lo = int(rng.integers(0, n - span + 1))
            tlo = synth.term_at(w.term_bytes, w.term_off, lo)
            thi = synth.term_at(w.term_bytes, w.term_off, lo + span - 1)

            def call():
                nonlocal info
                r = eng.read_range_dev(dsegs, tlo, thi, drem)
                info = r.info()
                r.release()
            med, _ = timed(call, 3)
            lat.append(med)
        eng.prof_enable(True)
        call()
        phases = {p["name"]: round(1e3 * p["ms"] / max(1, p["count"]), 1) for p in eng.prof_read()}
        host = {p["name"]: round(1e3 * p["host_ms"] / max(1, p["count"]), 1) for p in eng.prof_read()}
        eng.prof_enable(False)
        out.append({"range_frac": frac, "terms": int(info.terms_count), "phase_us": phases,
                    "host_us": host,
                    "postings_in": int(info.postings_in), "postings_out": int(info.postings_out),
                    "median_us": 1e6 * float(np.median(lat)), "p99_us": 1e6 * float(np.max(lat)),
                    "postings_in_per_s": int(info.postings_in) / float(np.median(lat))})
    print(json.dumps({"config": "C3 range read, 256 segments, 5% removed (read + merge-style filter)",
                      "terms": a.terms, "postings": w.postings_in, "results": out}))


def prefix(eng, a):
    """PrefixSearch (inverted_index.go:192-295) as one ii2_prefix_search_dev call over resident
    segments: batches of 16 prefixes of 3, 2 and 1 bytes, and the empty prefix (everything)."""
    w = synth.make_workload(a.terms, 64, a.postings, seed=0xC2)
    dsegs = [eng.upload(s) for s in w.segments]
    n = len(w.term_off) - 1
    rng = np.random.default_rng(6)
    out = []
    for plen, count in ((3, 16), (2, 16), (1, 16), (0, 1)):
        picks = sorted({synth.term_at(w.term_bytes, w.term_off, int(i))[:plen]
                        for i in rng.integers(0, n, size=count)})
        res = None

        def call():
            nonlocal res
            res = eng.prefix_search_dev(dsegs, picks)
        med, worst = timed(call, 3)
        eng.prof_enable(True)
        call()
        phases = {p["name"]: round(1e3 * p["ms"] / max(1, p["count"]), 1) for p in eng.prof_read()}
        eng.prof_enable(False)
        out.append({"prefix_len": plen, "prefixes": len(picks),
                    "values_out": int(sum(len(v) for v in res.values())),
                    "median_us": 1e6 * med, "max_us": 1e6 * worst, "phase_us": phases})
    print(json.dumps({"config": "PrefixSearch over 64 resident segments (one C-ABI call per batch, "
                                "results downloaded)", "terms": a.terms, "postings": w.postings_in,
                      "results": out}))


def lookup(eng, a):
    """Read(t, t) for Q keys as ONE ii2_lookup_dev call (results downloaded) on the C3 workload
    (256 segments, 5 % removed: read + merge-style filter) and the 64-segment C2 workload, random
    keys of which ~10 % are absent (a term with a byte appended).  For Q <= 256 the same keys are
    also read one by one (read_range_dev(t, t) + download), and every batch must equal that loop."""
    card = _card()
    rows = []
    for name, nseg, pres, seed, with_rem in (("C3", 256, 0.125, 0xC3, True), ("C2", 64, 0.5, 0xC2, False)):
        w = synth.make_workload(a.terms, nseg, a.postings, seed=seed, presence=pres)
        dsegs = [eng.upload(s) for s in w.segments]
        drem = eng.upload_removed(w.removed) if with_rem else None
        n = len(w.term_off) - 1
        rng = np.random.default_rng(8)
        for q in (1, 16, 256, 4096, 65536):
            ids = rng.integers(0, n, size=q)
            absent = rng.random(q) < 0.1
            keys = [synth.term_at(w.term_bytes, w.term_off, int(i)) + (b"\x01" if x else b"")
                    for i, x in zip(ids, absent)]
            res = None

            def call():
                nonlocal res
                res = eng.lookup_dev(dsegs, keys, drem)
            med, p99 = timed(call, 50 if q <= 4096 else 10)
            out = int(sum(len(v) for v in res if v is not None))
            row = {"workload": name, "segments": nseg, "removed": with_rem, "keys": q,
                   "found": int(sum(v is not None for v in res)), "postings_out": out,
                   "median_us": 1e6 * med, "p99_us": 1e6 * p99, "us_per_key": 1e6 * med / q,
                   "postings_out_per_s": out / med}
            if q <= 256:
                loop = None

                def point_loop():
                    nonlocal loop
                    loop = []
                    for k in keys:
                        r = eng.read_range_dev(dsegs, k, k, drem)
                        d = r.download_read()
                        r.release()
                        loop.append(d.post if d.n_terms else None)
                lmed, lp99 = timed(point_loop, 10 if q <= 16 else 3)
                same = all((x is None and y is None) or (x is not None and y is not None and np.array_equal(x, y))
                           for x, y in zip(res, loop))
                row.update({"point_loop_median_us": 1e6 * lmed, "point_loop_us_per_key": 1e6 * lmed / q,
                            "speedup_vs_point_loop": lmed / med, "same_as_point_loop": bool(same)})
                if not same:
                    raise SystemExit(f"lookup: batch of {q} keys on {name} differs from the point reads")
            rows.append(row)
        for s in dsegs:
            s.release()
        if drem is not None:
            drem.release()
    print(json.dumps({"config": "batched term lookup (ii2_lookup_dev, results downloaded)", "cards": card,
                      "terms": a.terms, "postings": a.postings, "results": rows}))


def _compose(eng, dsegs, drem, removed, queries):
    """The same answers as a caller composes them without ii2_query_dev: one lookup_dev call for
    the batch's distinct terms, one prefix_search_dev call for its distinct prefixes, then numpy
    set operations per query on the host (prefix search does not filter: the removed set is
    subtracted here).  Returns (answers, values downloaded)."""
    terms = sorted({t for q in queries for _, atoms in q for t, p in atoms if not p})
    prefixes = sorted({t for q in queries for _, atoms in q for t, p in atoms if p})
    look = dict(zip(terms, eng.lookup_dev(dsegs, terms, drem))) if terms else {}
    pre = eng.prefix_search_dev(dsegs, prefixes) if prefixes else {}
    empty = np.zeros(0, dtype=np.uint32)
    lists = {(t, False): (np.unique(v) if v is not None else empty) for t, v in look.items()}
    for t in prefixes:
        v = pre.get(t, empty)
        lists[(t, True)] = np.setdiff1d(v, removed, assume_unique=True) if removed is not None else v
    out = []
    for q in queries:
        req, exc = [], []
        for r, atoms in q:
            u = lists[atoms[0]]
            for at in atoms[1:]:
                u = np.union1d(u, lists[at])
            (req if r else exc).append(u)
        req.sort(key=len)
        e = req[0]
        for x in req[1:]:
            e = np.intersect1d(e, x, assume_unique=True)
        for x in exc:
            e = np.setdiff1d(e, x, assume_unique=True)
        out.append(e)
    downloaded = sum(len(v) for v in look.values() if v is not None) + sum(len(v) for v in pre.values())
    return out, downloaded


def query(eng, a):
    """Boolean queries (ii2_query_dev, results downloaded) on the C2 workload (64 segments) and
    the C3 workload (256 segments, 5 % removed), Q = 1 .. 4096 queries per call, in three shapes:
    a term AND a 2-byte prefix; two 2-byte prefixes AND NOT a third; two 1-byte prefixes (clauses
    of about 1.8 M values).  Each row also times the composition a caller writes without it
    (_compose) and exits non-zero if the answers differ.  The host composition of two 1-byte
    prefixes costs ~30 ms per query, so it runs up to Q = 256 there, and the first 256 answers of
    the Q = 4096 batch are checked against it."""
    card = _card()
    rows = []
    shapes = {
        "term_and_prefix2": lambda a_, b_, c_: [(True, [(a_, False)]), (True, [(b_[:2], True)])],
        "prefix2_and_prefix2_not_prefix2": lambda a_, b_, c_: [(True, [(a_[:2], True)]), (True, [(b_[:2], True)]),
                                                               (False, [(c_[:2], True)])],
        "prefix1_and_prefix1": lambda a_, b_, c_: [(True, [(a_[:1], True)]), (True, [(b_[:1], True)])],
    }
    for name, nseg, pres, seed, with_rem in (("C2", 64, 0.5, 0xC2, False), ("C3", 256, 0.125, 0xC3, True)):
        w = synth.make_workload(a.terms, nseg, a.postings, seed=seed, presence=pres)
        dsegs = [eng.upload(s) for s in w.segments]
        drem = eng.upload_removed(w.removed) if with_rem else None
        removed = w.removed if with_rem else None
        n = len(w.term_off) - 1
        rng = np.random.default_rng(9)
        for shape, make in shapes.items():
            picks = rng.integers(0, n, size=(4096, 3))
            allq = [make(*(synth.term_at(w.term_bytes, w.term_off, int(i)) for i in row)) for row in picks]
            ref256 = None
            for q in (1, 16, 256, 4096):
                queries = allq[:q]
                res = None

                def call():
                    nonlocal res
                    res = eng.query_dev(dsegs, queries, drem)
                med, p99 = timed(call, 20 if q <= 256 else 5)
                eng.prof_enable(True)
                call()
                phases = {p["name"]: round(1e3 * p["ms"] / max(1, p["count"]), 1) for p in eng.prof_read()}
                eng.prof_enable(False)
                row = {"workload": name, "segments": nseg, "removed": with_rem, "shape": shape, "queries": q,
                       "median_us": 1e6 * med, "p99_us": 1e6 * p99, "values_downloaded": int(sum(len(v) for v in res)),
                       "phase_us": phases}
                if shape == "prefix1_and_prefix1" and q > 256:
                    same = all(np.array_equal(x, y) for x, y in zip(res[:256], ref256))
                    row.update({"compose": "not run (host intersections of ~1.8 M values per query); the "
                                           "first 256 answers equal the Q = 256 composition",
                                "same_as_compose": bool(same)})
                else:
                    comp = None

                    def composed():
                        nonlocal comp
                        comp = _compose(eng, dsegs, drem, removed, queries)
                    heavy = shape == "prefix1_and_prefix1" and q >= 16
                    cmed, cp99 = timed(composed, 1 if heavy or q == 4096 else 5)
                    same = all(np.array_equal(x, y) for x, y in zip(res, comp[0]))
                    if q == 256:
                        ref256 = comp[0]
                    row.update({"compose_median_us": 1e6 * cmed, "compose_p99_us": 1e6 * cp99,
                                "compose_values_downloaded": int(comp[1]), "speedup_vs_compose": cmed / med,
                                "same_as_compose": bool(same)})
                rows.append(row)
                print(json.dumps(row), file=sys.stderr, flush=True)
                if not row["same_as_compose"]:
                    raise SystemExit(f"query: {shape} x {q} on {name} differs from the composed answers")
        for s in dsegs:
            s.release()
        if drem is not None:
            drem.release()
    print(json.dumps({"config": "boolean queries (ii2_query_dev, results downloaded) vs lookup_dev + "
                                "prefix_search_dev + host numpy set operations", "cards": card,
                      "terms": a.terms, "postings": a.postings, "results": rows}))


def c1(eng, a):
    """BASELINE configs[0] shape through ii2_ingest: 4 x Put(all terms, val = 1..4) + Merge as
    ONE call — every document's terms are handed over SHUFFLED (Put sorts them, shard.go:34)."""
    tb, off = synth.make_terms(a.terms)
    raw = tb.tobytes()
    terms = [raw[int(off[i]):int(off[i + 1])] for i in range(a.terms)]
    rng = np.random.default_rng(1)
    docs = []
    for val in (1, 2, 3, 4):
        perm = rng.permutation(a.terms)
        docs.append(([terms[int(i)] for i in perm], val))
    res = None

    def call():
        nonlocal res
        res = eng.ingest(docs, None, decoded=True)
    t0 = time.perf_counter()
    call()
    first = time.perf_counter() - t0
    eng.prof_enable(True)
    t0 = time.perf_counter()
    call()
    second = time.perf_counter() - t0
    phases = {p["name"]: round(p["ms"] / max(1, p["count"]), 2) for p in eng.prof_read()}
    eng.prof_enable(False)
    ok = (res.terms_count == a.terms and np.array_equal(res.term_bytes, tb)
          and np.array_equal(res.post, np.tile(np.array([1, 2, 3, 4], dtype=np.uint32), a.terms)))
    print(json.dumps({"config": "C1 ingest: 4 documents x all terms (shuffled), one ii2_ingest call "
                                "(ctypes marshalling of 4 x %d Python terms included)" % a.terms,
                      "terms": a.terms, "postings": 4 * a.terms, "first_call_ms": 1e3 * first,
                      "call_ms": 1e3 * second, "device_phase_ms": phases,
                      "result_is_every_term_to_1234": bool(ok)}))


def c4(eng, a):
    from oracle import orc  # checker only
    rows = []
    rng = np.random.default_rng(4)
    for lg in range(4, 25, 4):
        L = 1 << lg
        nlists = max(1, a.c4_values // L)  # >= 64M values per timing (SURVEY 8d)
        for gap in (1, 16, 4096):
            gaps = rng.integers(1, 2 * gap + 1, size=L * nlists, dtype=np.int64)
            starts = np.arange(nlists, dtype=np.int64) * L
            c = np.cumsum(gaps)
            vals = (c - np.repeat(c[starts] - gaps[starts], L)).astype(np.uint32)
            off = (np.arange(nlists + 1, dtype=np.uint64) * np.uint64(L))
            words = woff = None

            words, woff = eng.intcomp_encode_batch(vals, off)
            # the C-ABI calls themselves, on pinned host buffers (no numpy copies of the results)
            import ctypes as C
            import torch
            from inverted_index_2_b200 import _abi as A
            keep = [torch.from_numpy(x).pin_memory() for x in (vals, off, words, woff)]
            pv, po, pw, pwo = (t.numpy() for t in keep)

            def enc():
                wp, op = A.u32p(), A.u64p()
                eng._check(eng.lib.ii2_intcomp_encode_u32(A.np_ptr(pv, A.u32p), A.np_ptr(po, A.u64p),
                                                          nlists, C.byref(wp), C.byref(op)), "enc")
                eng.lib.ii2_free(wp)
                eng.lib.ii2_free(op)

            def dec():
                vp, op = A.u32p(), A.u64p()
                eng._check(eng.lib.ii2_intcomp_decode_u32(A.np_ptr(pw, A.u32p), A.np_ptr(pwo, A.u64p),
                                                          nlists, C.byref(vp), C.byref(op)), "dec")
                eng.lib.ii2_free(vp)
                eng.lib.ii2_free(op)
            te, _ = timed(enc, 3)
            td, _ = timed(dec, 3)
            eng.prof_enable(True)
            for _ in range(3):
                enc()
                dec()
            ph = {k["name"]: k["ms"] / k["count"] for k in eng.prof_read()}
            eng.prof_enable(False)
            alg = 4.0 * len(vals) + 4.0 * len(words)  # decoded values + stream words, each once
            if lg <= 12:  # parity spot check on the small cases
                ew, eo = orc.intcomp_encode_batch(vals[:L * min(nlists, 64)], off[:min(nlists, 64) + 1])
                assert np.array_equal(ew, words[:len(ew)]) and np.array_equal(eo, woff[:len(eo)])
            rows.append({"codec": "intcomp", "L": L, "lists": nlists, "gap": gap,
                         "ratio": 4.0 * len(vals) / (4.0 * len(words)),
                         "encode_values_per_s": len(vals) / te, "decode_values_per_s": len(vals) / td,
                         "api": "ii2_intcomp_*_u32 on pinned host buffers (H2D + kernels + D2H)",
                         "device_encode_ms": ph.get("k3a_encode"), "device_decode_ms": ph.get("k3a_decode"),
                         "device_encode_gbs": alg / ph["k3a_encode"] / 1e6 if ph.get("k3a_encode") else None,
                         "device_decode_gbs": alg / ph["k3a_decode"] / 1e6 if ph.get("k3a_decode") else None,
                         "encode_frac_of_hbm_peak": alg / ph["k3a_encode"] / 1e6 / PEAK if ph.get("k3a_encode") else None,
                         "decode_frac_of_hbm_peak": alg / ph["k3a_decode"] / 1e6 / PEAK if ph.get("k3a_decode") else None})
    for lg in range(4, 25, 4):
        L = 1 << lg
        universe = np.sort(rng.choice(max(4 * L, 1 << 10), size=2 * L, replace=False)).astype(np.uint32)
        vals = rng.permutation(universe)[:L]
        bm = eng.bitmask(universe)
        enc = None

        enc = bm.put(vals)
        import ctypes as C
        import torch
        from inverted_index_2_b200 import _abi as A
        tv = torch.from_numpy(np.ascontiguousarray(vals)).pin_memory()
        te_ = torch.from_numpy(np.frombuffer(enc, dtype=np.uint8).copy()).pin_memory()
        pv, pe = tv.numpy(), te_.numpy()

        def put():  # the C-ABI call itself on pinned buffers (no Python copies of the result)
            bp, nb = A.u8p(), C.c_uint64()
            eng._check(eng.lib.ii2_bitmask_put(bm.h, A.np_ptr(pv, A.u32p), L, C.byref(bp), C.byref(nb)), "put")
            eng.lib.ii2_free(bp)

        def get():
            vp, vn = A.u32p(), C.c_uint64()
            eng._check(eng.lib.ii2_bitmask_get(bm.h, A.np_ptr(pe, A.u8p), len(pe), C.byref(vp), C.byref(vn)), "get")
            eng.lib.ii2_free(vp)
        tp, _ = timed(put, 3)
        tg, _ = timed(get, 3)
        eng.prof_enable(True)
        for _ in range(3):
            put()
            get()
        ph = {k["name"]: k["ms"] / k["count"] for k in eng.prof_read()}
        eng.prof_enable(False)
        alg = 4.0 * L + len(enc)  # values + serialised bitmap, each once (SURVEY 8d)
        rows.append({"codec": "bitmask", "L": L, "dictionary": 2 * L, "bytes": len(enc),
                     "put_values_per_s": L / tp, "get_values_per_s": L / tg,
                     "api": "ii2_bitmask_put/get on pinned host buffers (H2D + kernels + D2H)",
                     "device_put_ms": ph.get("k3b_put"), "device_get_ms": ph.get("k3b_get"),
                     "note": "device_*_ms = the call's stream time INCLUDING its H2D / D2H copies "
                             "(64 MB of values at L = 16 M); kernels_*_ms = kernels only",
                     "kernels_put_ms": ph.get("k3b_put_kernels"), "kernels_get_ms": ph.get("k3b_get_kernels"),
                     "kernels_put_values_per_s": L / (ph["k3b_put_kernels"] * 1e-3) if ph.get("k3b_put_kernels") else None,
                     "kernels_get_values_per_s": L / (ph["k3b_get_kernels"] * 1e-3) if ph.get("k3b_get_kernels") else None,
                     "kernels_put_gbs": alg / ph["k3b_put_kernels"] / 1e6 if ph.get("k3b_put_kernels") else None,
                     "device_put_values_per_s": L / (ph["k3b_put"] * 1e-3) if ph.get("k3b_put") else None,
                     "device_put_gbs": alg / ph["k3b_put"] / 1e6 if ph.get("k3b_put") else None,
                     "device_get_gbs": alg / ph["k3b_get"] / 1e6 if ph.get("k3b_get") else None})
    print(json.dumps({"config": "C4 codec sweep, list lengths 16..16M", "results": rows}))


def _card():
    """Card name and power limit, read in the same run as the numbers (read-only query)."""
    import subprocess
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except Exception as e:  # noqa: BLE001
        q = [f"nvidia-smi unavailable: {e}"]
    return q


_POOL = None  # one long-lived host thread per device (no thread start inside a timed call)


def _in_threads(fns):
    """Runs fns[i] on worker thread i of the pool, all at once; their results in order."""
    global _POOL
    import queue
    import threading
    if _POOL is None or len(_POOL) < len(fns):
        _POOL = []
        for _ in range(max(len(fns), 16)):
            q_in, q_out = queue.Queue(), queue.Queue()

            def loop(q_in=q_in, q_out=q_out):
                while True:
                    f = q_in.get()
                    try:
                        q_out.put((True, f()))
                    except BaseException as e:  # noqa: BLE001
                        q_out.put((False, repr(e)))
            threading.Thread(target=loop, daemon=True).start()
            _POOL.append((q_in, q_out))
    for (q_in, _), f in zip(_POOL, fns):
        q_in.put(f)
    got = [q_out.get() for (_, q_out), _f in zip(_POOL, fns)]
    errs = [v for ok, v in got if not ok]
    if errs:
        raise RuntimeError("; ".join(errs))
    return [v for _, v in got]


def _partition(w, k):
    from inverted_index_2_b200 import sharded
    from inverted_index_2_b200.flat import FlatSegment
    keys = sharded.shard_keys_of_sorted(w.term_bytes, w.term_off)
    bounds = sharded.partition_shard_keys(np.bincount(keys, minlength=1024).astype(float), k)
    parts = []
    for r in range(k):
        lo, hi = np.searchsorted(keys, [bounds[r], bounds[r + 1]])
        out = []
        for seg, ids in zip(w.segments, w.seg_term_ids):
            a, b = np.searchsorted(ids, [lo, hi])
            toff, poff = seg.term_off[a:b + 1], seg.post_off[a:b + 1]
            out.append(FlatSegment(seg.term_bytes[int(toff[0]):int(toff[-1])].copy(),
                                   (toff - toff[0]).astype(np.uint32), seg.mode,
                                   post=seg.post[int(poff[0]):int(poff[-1])].copy(),
                                   post_off=(poff - poff[0]).astype(np.uint64)))
        parts.append(out)
    return parts


def multidev(a):
    import torch
    from inverted_index_2_b200.engine import Engine
    n = torch.cuda.device_count()
    devs = list(range(min(n, 16)))
    eng = Engine(devices=devs)
    N = len(devs)
    card = _card()
    # ---- weak scaling: every device compacts its own copy of the C2 workload (bench.py's shape)
    w = synth.make_workload(a.terms, 64, a.postings, seed=0xC2, removed_frac=0.05)
    res = {}

    def setup(d):
        eng.set_device(d)
        return [eng.upload(s) for s in w.segments], eng.upload_removed(w.removed)
    held = _in_threads([lambda d=d: setup(d) for d in devs])

    def compact(i):
        segs, rem = held[i]
        r = eng.merge_dev(segs, rem, encode=True, decoded=False)
        r.release()

    def rate(idx, reps=5):
        _in_threads([lambda i=i: compact(i) for i in idx])  # warm-up
        t0 = time.perf_counter()
        for _ in range(reps):
            _in_threads([lambda i=i: compact(i) for i in idx])
        return len(idx) * reps * w.postings_in / (time.perf_counter() - t0) / 1e9
    single = rate([0])
    agg = rate(list(range(N)))
    # (an efficiency is a scaling figure: it means nothing with one device)
    res["weak_scaling"] = {"devices": N, "single_device_gpostings_s": single, "aggregate_gpostings_s": agg,
                           "efficiency": agg / (N * single) if N > 1 else None}
    for segs, rem in held:
        [s.release() for s in segs]
        rem.release()
    # ---- 1 % read of one index partitioned over the devices, gathered to device 0
    parts = _partition(w, N)
    eng.set_device(devs[0])
    whole = [eng.upload(s) for s in w.segments]
    dparts = _in_threads([lambda r=r: (eng.set_device(devs[r]), [eng.upload(s) for s in parts[r]])[1]
                          for r in range(N)])
    eng.set_device(devs[0])
    nt = len(w.term_off) - 1
    rng = np.random.default_rng(5)
    lat, checked = [], 0
    for _ in range(8):
        span = max(1, nt // 100)
        lo = int(rng.integers(0, nt - span + 1))
        tlo = synth.term_at(w.term_bytes, w.term_off, lo)
        thi = synth.term_at(w.term_bytes, w.term_off, lo + span - 1)
        ts = []
        for rep in range(4):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            reads = _in_threads([lambda r=r: eng.read_range_dev(dparts[r], tlo, thi) for r in range(N)])
            g = eng.read_gather_devices(reads, devs[0])
            ts.append(time.perf_counter() - t0)
            if rep == 3:
                got = g.download_read()
                ref = eng.read_range_dev(whole, tlo, thi).download_read()
                for f in ("term_bytes", "term_off", "post", "post_off"):
                    assert np.array_equal(getattr(got, f), getattr(ref, f)), f
                checked += 1
            [x.release() for x in reads]
            g.release()
        lat.append(float(np.median(ts[1:])))
    res["read_1pct_gather_us"] = {"median_us": 1e6 * float(np.median(lat)), "max_us": 1e6 * float(np.max(lat)),
                                  "positions_verified": checked,
                                  "what": "per-device ii2_read_range_dev from one long-lived host thread per "
                                          "device + ii2_read_gather_devices to device 0, wall clock"}
    # ---- prefix search over the devices, gathered on device 0
    prow = []
    for plen, count in ((3, 16), (2, 16), (1, 16), (0, 1)):
        picks = sorted({synth.term_at(w.term_bytes, w.term_off, int(i))[:plen]
                        for i in rng.integers(0, nt, size=count)})
        ref = eng.prefix_search_dev(whole, picks)

        def call():
            return eng.prefix_gather_devices(dparts, picks, devs[0])
        got = call()
        assert sorted(got) == sorted(ref) and all(np.array_equal(got[k], ref[k]) for k in ref)
        med, worst = timed(call, 3)
        prow.append({"prefix_len": plen, "prefixes": len(picks), "median_us": 1e6 * med, "max_us": 1e6 * worst})
    res["prefix_gather"] = prow
    print(json.dumps({"config": f"multidev: one process over {N} device(s)", "cards": card,
                      "terms": a.terms, "postings": w.postings_in, "results": res}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--which", default="c3,c4")
    ap.add_argument("--c4-values", type=int, default=1 << 26)
    ap.add_argument("--terms", type=int, default=1_000_000)
    ap.add_argument("--postings", type=int, default=100_000_000)
    a = ap.parse_args()
    if "multidev" in a.which:  # binds every visible device: a process of its own
        multidev(a)
        return
    from inverted_index_2_b200.engine import Engine
    eng = Engine(0)
    if "c1" in a.which:
        c1(eng, a)
    if "c3" in a.which:
        c3(eng, a)
    if "c4" in a.which:
        c4(eng, a)
    if "prefix" in a.which:
        prefix(eng, a)
    if "lookup" in a.which:
        lookup(eng, a)
    if "query" in a.which:
        query(eng, a)


if __name__ == "__main__":
    main()
