"""One process, several GPUs: device-bound handles, per-device runtime state and the in-process
gathers (ii2_set_device, ii2_result_device, ii2_read_gather_devices, ii2_prefix_gather_devices)
against the CPU oracle.

The pytest process has bound device 0 (session fixture), so cases that bind another device set
run in a spawned process; they skip below two GPUs.  The single-GPU cases gather partitions that
all live on device 0: the same kernel, without peers."""
import ctypes as C
import threading
import time
import traceback

import numpy as np
import pytest

from inverted_index_2_b200 import _abi as A

PREFIXES_OF = lambda lo, hi: [b"", lo[:1], lo[:2], hi[:2], b"zzzz", b"Q"]  # noqa: E731


def _workload():
    from inverted_index_2_b200 import synth
    return synth.make_workload(30000, 8, 400000, universe=1 << 18, seed=77)


def _partitions(w, k):
    """k contiguous shard-key ranges of the index (sharded.partition_shard_keys), each as the
    slices of every segment that fall into it."""
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


def _same_read(got, exp):
    assert got.n_terms == exp.n_terms
    for f in ("term_bytes", "term_off", "post", "post_off"):
        assert np.array_equal(getattr(got, f), getattr(exp, f)), f


def _same_prefix(got, exp):
    assert {k: [int(x) for x in v] for k, v in got.items()} == {k: list(v) for k, v in exp.items()}


def _bounds(w):
    from inverted_index_2_b200 import synth
    nt = len(w.term_off) - 1
    t = lambda i: synth.term_at(w.term_bytes, w.term_off, i)  # noqa: E731
    lo, hi = t(nt // 10), t(nt - nt // 10)
    return {
        "closed": (lo, hi),
        "open_min": (None, hi),
        "open_max": (lo, None),
        "open": (None, None),
        "absent": (lo + b"\x00", hi + b"\x00"),  # bounds that are not terms of the index
        "point": (t(nt // 3), t(nt // 3)),
        "narrow": (t(nt // 2), t(nt // 2 + 40)),  # most partitions are empty in range
    }


# ---------------------------------------------------------------- CPU, no device
def test_new_entry_points_need_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    from inverted_index_2_b200.engine import load_library
    lib = load_library()
    assert lib.ii2_set_device(0) == A.II2_ERR_NO_DEVICE
    d = C.c_int()
    assert lib.ii2_result_device(None, C.byref(d)) == A.II2_ERR_NO_DEVICE
    h = C.c_void_p()
    assert lib.ii2_read_gather_devices(None, 0, 0, C.byref(h)) == A.II2_ERR_NO_DEVICE
    out = A.PrefixOut()
    assert lib.ii2_prefix_gather_devices(None, 0, 0, C.byref(out)) == A.II2_ERR_NO_DEVICE


# ---------------------------------------------------------------- one GPU, device 0
@pytest.fixture(scope="module")
def wl():
    return _workload()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 7])
def test_read_gather_devices_on_one_device(engine, orc, wl, k):
    parts = _partitions(wl, k)
    dparts = [[engine.upload(s) for s in p] for p in parts]
    try:
        for name, (lo, hi) in _bounds(wl).items():
            reads = [engine.read_range_dev(ds, lo, hi) for ds in dparts]
            g = engine.read_gather_devices(reads, 0)
            assert g.device == 0 and engine.result_device(g) == 0
            _same_read(g.download_read(), orc.read_range(wl.segments, lo, hi))
            if name == "closed":  # the gathered result as a segment, read again
                from inverted_index_2_b200 import synth
                nt = len(wl.term_off) - 1
                lo2 = synth.term_at(wl.term_bytes, wl.term_off, nt // 4)
                hi2 = synth.term_at(wl.term_bytes, wl.term_off, nt // 2)
                seg = g.to_segment()
                assert seg.device == 0
                again = engine.read_range_dev([seg], lo2, hi2).download_read()
                _same_read(again, orc.read_range(wl.segments, lo2, hi2))
                seg.release()
            for r in reads:
                r.release()
            g.release()
    finally:
        for ds in dparts:
            for s in ds:
                s.release()


@pytest.mark.gpu
def test_prefix_gather_devices_on_one_device(engine, orc, wl):
    from inverted_index_2_b200 import synth
    nt = len(wl.term_off) - 1
    lo = synth.term_at(wl.term_bytes, wl.term_off, nt // 10)
    hi = synth.term_at(wl.term_bytes, wl.term_off, nt - nt // 10)
    pref = PREFIXES_OF(lo, hi)
    dparts = [[engine.upload(s) for s in p] for p in _partitions(wl, 3)]
    got = engine.prefix_gather_devices(dparts, pref, 0)
    _same_prefix(got, orc.prefix_search(wl.segments, pref))


@pytest.mark.gpu
def test_multidevice_errors_on_one_device(engine, wl):
    from inverted_index_2_b200.engine import EngineError
    lib = engine.lib
    bound = engine.device
    ints = lambda *v: (C.c_int * len(v))(*v)  # noqa: E731
    assert lib.ii2_init(ints(bound, bound), 2) == A.II2_ERR_INVALID        # duplicate
    assert lib.ii2_init(ints(bound, 4096), 2) == A.II2_ERR_INVALID         # out of range
    assert b"out of range" in lib.ii2_last_error()
    assert lib.ii2_init(ints(4096), 1) == A.II2_ERR_INVALID                # another set
    assert lib.ii2_init(ints(bound), 1) == A.II2_OK                        # the bound set
    assert lib.ii2_set_device(4096) == A.II2_ERR_INVALID
    assert lib.ii2_set_device(-1) == A.II2_ERR_INVALID
    assert lib.ii2_set_device(bound) == A.II2_OK
    ds = [engine.upload(s) for s in wl.segments]
    enc = engine.merge_dev(ds, None, encode=True, decoded=False)  # encoded only
    with pytest.raises(EngineError) as e:
        engine.read_gather_devices([enc], bound)
    assert e.value.code == A.II2_ERR_INVALID
    with pytest.raises(EngineError) as e:
        engine.read_gather_devices([], 4096)
    assert e.value.code == A.II2_ERR_INVALID
    empty = engine.read_gather_devices([], bound).download_read()
    assert empty.n_terms == 0 and empty.term_off.tolist() == [0] and empty.post_off.tolist() == [0]
    a = engine.prefix_search_dev_out(ds, [b"a", b"b"])
    b = engine.prefix_search_dev_out(ds, [b"a"])
    try:
        with pytest.raises(EngineError) as e:
            engine.prefix_gather_devices([a, b], [b"a", b"b"], bound)
        assert e.value.code == A.II2_ERR_INVALID
    finally:
        engine.prefix_out_free(a)
        engine.prefix_out_free(b)
    enc.release()
    for s in ds:
        s.release()


# ---------------------------------------------------------------- several GPUs, spawned
def _threads(fns):
    errs = []

    def run(f):
        try:
            f()
        except BaseException:
            errs.append(traceback.format_exc())
    ts = [threading.Thread(target=run, args=(f,)) for f in fns]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, "\n".join(errs)


def _multi_worker(devs, q):
    try:
        _multi_checks(devs)
        q.put(None)
    except BaseException:
        q.put(traceback.format_exc())


def _multi_checks(devs):
    import torch
    from inverted_index_2_b200 import synth
    from inverted_index_2_b200.engine import Engine, EngineError
    from oracle import orc
    orc.lib()
    N = len(devs)
    from inverted_index_2_b200.engine import load_library
    lib = load_library(build_if_needed=False)
    ints = lambda *v: (C.c_int * len(v))(*v)  # noqa: E731
    # refused before anything is bound: out of range, duplicate
    assert lib.ii2_init(ints(devs[0], 4096), 2) == A.II2_ERR_INVALID
    assert lib.ii2_init(ints(devs[0], devs[0]), 2) == A.II2_ERR_INVALID
    with pytest.raises(ValueError):
        Engine(devices=[])
    eng = Engine(devices=devs)
    assert eng.lib.ii2_init(ints(*reversed(devs)), N) == A.II2_OK  # the same set
    assert eng.lib.ii2_init(ints(devs[0]), 1) == A.II2_ERR_INVALID  # another set
    uid = (C.c_uint8 * 128)()
    assert eng.lib.ii2_comm_init(C.cast(uid, A.u8p), 0, 1) == A.II2_ERR_INVALID  # NCCL: one GPU each
    w = _workload()
    parts = _partitions(w, N)
    nt = len(w.term_off) - 1
    lo = synth.term_at(w.term_bytes, w.term_off, nt // 10)
    hi = synth.term_at(w.term_bytes, w.term_off, nt - nt // 10)
    place = [devs[(r + 1) % N] for r in range(N)]  # partition r lives on place[r]: not device order

    # ---- per-device uploads and merges, one thread per device
    dparts, drems, merged = [None] * N, [None] * N, [None] * N

    def upload_and_merge(r):
        eng.set_device(place[r])
        dparts[r] = [eng.upload(s) for s in parts[r]]
        drems[r] = eng.upload_removed(w.removed)
        assert all(s.device == place[r] for s in dparts[r]) and drems[r].device == place[r]
        both = eng.merge_dev(dparts[r], drems[r], encode=True, decoded=True)
        dec = eng.merge_dev(dparts[r], drems[r], encode=False, decoded=True)
        assert both.device == place[r] and eng.result_device(dec) == place[r]
        merged[r] = (both.download_merge(decoded=True), dec.download_read())
        both.release()
        dec.release()
    _threads([lambda r=r: upload_and_merge(r) for r in range(N)])
    eng.set_device(devs[0])
    for r in range(N):
        exp = orc.merge(parts[r], w.removed, decoded=True)
        m, d = merged[r]
        for f in ("term_bytes", "term_off", "val_off", "val_bytes", "post", "post_off"):
            assert np.array_equal(getattr(m, f), getattr(exp, f)), (r, f)
        for f in ("term_bytes", "term_off", "post", "post_off"):
            assert np.array_equal(getattr(d, f), getattr(exp, f)), (r, f)
        # the same merge on device 0, byte for byte
        s0 = [eng.upload(s) for s in parts[r]]
        r0 = eng.upload_removed(w.removed)
        m0 = eng.merge_dev(s0, r0, encode=True, decoded=True).download_merge(decoded=True)
        for f in ("term_bytes", "term_off", "val_off", "val_bytes", "post", "post_off"):
            assert np.array_equal(getattr(m0, f), getattr(m, f)), (r, f)

    # ---- reads gathered to the first and the last device, prefix search gathered
    exp_read = orc.read_range(w.segments, lo, hi)
    for root in (devs[0], devs[-1]):
        reads = [eng.read_range_dev(dparts[r], lo, hi) for r in range(N)]
        assert [x.device for x in reads] == place
        g = eng.read_gather_devices(reads, root)
        assert g.device == root and eng.result_device(g) == root
        _same_read(g.download_read(), exp_read)
        seg = g.to_segment()
        assert seg.device == root
        _same_read(eng.read_range_dev([seg], lo, hi).download_read(), exp_read)
        pref = PREFIXES_OF(lo, hi)
        _same_prefix(eng.prefix_gather_devices(dparts, pref, root), orc.prefix_search(w.segments, pref))

    # ---- concurrency: host-buffer merges (set_device) and resident reads on every device at once,
    # plus one thread that switches devices between calls
    exp_m = [orc.merge(parts[r], w.removed, decoded=True) for r in range(N)]
    exp_r = [orc.read_range(parts[r], lo, hi) for r in range(N)]

    def busy(r):
        eng.set_device(place[r])
        for _ in range(3):
            got = eng.merge(parts[r], w.removed, decoded=True)
            assert np.array_equal(got.val_bytes, exp_m[r].val_bytes) and np.array_equal(got.post, exp_m[r].post)
            _same_read(eng.read_range_dev(dparts[r], lo, hi).download_read(), exp_r[r])

    def switcher():
        for i in range(2 * N):
            r = i % N
            eng.set_device(place[r])
            _same_read(eng.read_range(parts[r], lo, hi), exp_r[r])
    _threads([lambda r=r: busy(r) for r in range(N)] + [switcher])

    # ---- pinned memory on another device: the pool was filled on device 0; point read and a
    # 0.1 % range read (windows exchange through pinned memory) on device 1
    eng.set_device(devs[0])
    full0 = [eng.upload(s) for s in w.segments]
    t = synth.term_at(w.term_bytes, w.term_off, nt // 3)
    _same_read(eng.read_range_dev(full0, t, t).download_read(), orc.read_range(w.segments, t, t))
    eng.set_device(devs[1])
    full1 = [eng.upload(s) for s in w.segments]
    assert all(s.device == devs[1] for s in full1)
    a, b = synth.term_at(w.term_bytes, w.term_off, nt // 2), synth.term_at(w.term_bytes, w.term_off, nt // 2 + nt // 1000)
    for x, y in ((t, t), (a, b)):
        _same_read(eng.read_range_dev(full1, x, y).download_read(), orc.read_range(w.segments, x, y))

    # ---- mixed devices: refused, and both devices keep working
    for segs, rem in (([full0[0], full1[1]], None), (full1[:2], drems[place.index(devs[0])])):
        with pytest.raises(EngineError) as e:
            eng.merge_dev(segs, rem, encode=True, decoded=False)
        assert e.value.code == A.II2_ERR_INVALID and b"different devices" in eng.lib.ii2_last_error()
    for segs in (full0, full1):
        _same_read(eng.read_range_dev(segs, a, b).download_read(), orc.read_range(w.segments, a, b))

    # ---- a result of device 1 released from a thread that selected device 0
    res1 = eng.read_range_dev(full1, lo, hi)
    assert res1.device == devs[1]

    def release_elsewhere():
        eng.set_device(devs[0])
        res1.release()
        eng.sync()
    _threads([release_elsewhere])
    _same_read(eng.read_range_dev(full1, lo, hi).download_read(), exp_read)

    # ---- a caller-owned stream of device 1 serves device 1's calls only
    user = torch.cuda.Stream(device=devs[1])

    def with_stream():
        eng.set_device(devs[1])
        eng.set_stream(user.cuda_stream)
        with torch.cuda.device(devs[1]), torch.cuda.stream(user):
            torch.cuda._sleep(int(4e8))  # ~0.2 s queued on the user stream
        t0 = time.perf_counter()
        _same_read(eng.read_range(w.segments, a, b), orc.read_range(w.segments, a, b))
        waited = time.perf_counter() - t0
        assert waited > 0.05, f"device-1 call did not run behind the user stream ({waited:.3f} s)"
        eng.set_device(devs[0])  # no binding there: the library's own stream of device 0
        _same_read(eng.read_range(w.segments, a, b), orc.read_range(w.segments, a, b))
        eng.set_device(devs[1])
        eng.set_stream(None)
    _threads([with_stream])
    for s in full0 + full1 + [x for p in dparts for x in p]:
        s.release()


def _spawn_multi(n):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < n:
        pytest.skip(f"needs {n} GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    p = ctx.Process(target=_multi_worker, args=(list(range(n)), q))
    p.start()
    err = q.get(timeout=900)
    p.join(timeout=120)
    assert err is None, err
    assert p.exitcode == 0


@pytest.mark.gpu
@pytest.mark.timeout(1200)
def test_two_devices_one_process():
    _spawn_multi(2)


@pytest.mark.gpu
@pytest.mark.timeout(1200)
def test_all_devices_one_process():
    import torch
    n = torch.cuda.device_count()
    if n <= 2:
        pytest.skip("needs more than two GPUs")
    _spawn_multi(min(n, 8))
