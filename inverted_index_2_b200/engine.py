"""ctypes binding of libii2.so (include/ii2.h) — the CUDA engine behind the host mirror.

This is the Python stand-in for the cgo stub of INTEGRATION.md: every method is one
C-ABI call.  There is no CPU path: if the library cannot be loaded or no sm_100 device
can be bound, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import _abi as A
from .flat import FlatSegment, MergeResult, ReadResult, views_array

_HERE = os.path.dirname(os.path.abspath(__file__))


class EngineError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str = ""):
        super().__init__(f"ii2: {what} (code {code}){': ' + detail if detail else ''}")
        self.code = code


def load_library(build_if_needed: bool = True) -> C.CDLL:
    """Loads libii2.so built in-tree; never falls back to anything else."""
    so = os.path.join(_HERE, "libii2.so")
    alt = os.environ.get("II2_LIB")  # tuning sweeps: another build of the same library
    if alt:
        lib = C.CDLL(alt)
        # (an older build may lack the newest entry points: bind what it exports)
        A.bind(lib, {k: v for k, v in A.PROTOTYPES.items() if hasattr(lib, k)})
        return lib
    if build_if_needed and os.path.isdir(os.path.join(_HERE, "csrc")):
        from .build import build
        try:
            so = build()
        except Exception:
            if not os.path.exists(so):
                raise
    if not os.path.exists(so):
        raise RuntimeError("libii2.so is missing: run `python -m inverted_index_2_b200.build`")
    lib = C.CDLL(so)
    A.bind(lib, A.PROTOTYPES)
    return lib


def _bytes_arg(b: bytes | None):
    if b is None:
        return C.cast(None, A.u8p), 0, None
    buf = (C.c_uint8 * max(1, len(b))).from_buffer_copy(b.ljust(1, b"\0"))
    return C.cast(buf, A.u8p), len(b), buf


class DeviceSegment:
    """A segment resident in HBM (ii2_seg) of CUDA device `device`."""

    def __init__(self, eng: "Engine", handle: int, n_terms: int, device: int):
        self.eng, self.h, self.n_terms, self.device = eng, handle, n_terms, device

    def release(self):
        if self.h:
            self.eng.lib.ii2_seg_release(self.h)
            self.h = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class DeviceRemoved:
    def __init__(self, eng: "Engine", handle: int, device: int):
        self.eng, self.h, self.device = eng, handle, device

    def release(self):
        if self.h:
            self.eng.lib.ii2_removed_release(self.h)
            self.h = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class DeviceResult:
    """Merge / read result resident in HBM (ii2_result) of CUDA device `device`."""

    def __init__(self, eng: "Engine", handle: int, device: int):
        self.eng, self.h, self.device = eng, handle, device

    def info(self) -> A.ResultInfo:
        info = A.ResultInfo()
        self.eng._check(self.eng.lib.ii2_result_info_get(self.h, C.byref(info)), "result_info")
        return info

    def download_merge(self, decoded: bool = True) -> MergeResult:
        out = A.MergeOut()
        self.eng._check(self.eng.lib.ii2_result_download_merge(
            self.h, A.II2_MERGE_WANT_DECODED if decoded else 0, C.byref(out)), "download_merge")
        try:
            return MergeResult.from_c(out, decoded)
        finally:
            self.eng.lib.ii2_merge_out_free(C.byref(out))

    def download_read(self) -> ReadResult:
        out = A.ReadOut()
        self.eng._check(self.eng.lib.ii2_result_download_read(self.h, C.byref(out)), "download_read")
        try:
            return ReadResult.from_c(out)
        finally:
            self.eng.lib.ii2_read_out_free(C.byref(out))

    def as_tensors(self, device_index: int = 0) -> dict:
        """Zero-copy torch views of the result's device arrays (valid until release()); the
        NCCL gather of cross-shard reads works on these.  Unsigned data is viewed as the signed
        type of the same width (NCCL has no unsigned 32/64-bit types)."""
        import torch
        info = self.info()

        class _Arr:
            def __init__(self, ptr, n, typestr):
                self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr,
                                                 "data": (int(ptr), False), "version": 2}

        def view(ptr, n, typestr, dt):
            if not ptr or int(n) == 0:
                return torch.zeros(0, dtype=dt, device=f"cuda:{device_index}")
            return torch.as_tensor(_Arr(ptr, n, typestr), device=f"cuda:{device_index}")
        t = int(info.terms_count)
        return {
            "term_bytes": view(info.d_term_bytes, info.term_bytes, "|u1", torch.uint8),
            "term_off": view(info.d_term_off, t + 1, "<i4", torch.int32),
            "post": view(info.d_post, info.postings_out, "<i4", torch.int32),
            "post_off": view(info.d_post_off, t + 1 if info.d_post_off else 0, "<i8", torch.int64),
        }

    def to_segment(self) -> DeviceSegment:
        h = C.c_void_p()
        n = int(self.info().terms_count)
        self.eng._check(self.eng.lib.ii2_result_to_seg(self.h, C.byref(h)), "result_to_seg")
        return DeviceSegment(self.eng, h.value, n, self.device)

    def release(self):
        if self.h:
            self.eng.lib.ii2_result_release(self.h)
            self.h = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class Bitmask:
    """file/bitmask.go Bitmask[uint32] on the device (not thread-safe, like :10)."""

    def __init__(self, eng: "Engine", init=None):
        self.eng = eng
        v = np.ascontiguousarray(init if init is not None else [], dtype=np.uint32)
        h = C.c_void_p()
        eng._check(eng.lib.ii2_bitmask_new(A.np_ptr(v, A.u32p) if len(v) else C.cast(None, A.u32p),
                                           len(v), C.byref(h)), "bitmask_new")
        self.h = h.value

    def __del__(self):
        try:
            if self.h:
                self.eng.lib.ii2_bitmask_free(self.h)
                self.h = None
        except Exception:
            pass

    def all_values(self) -> np.ndarray:
        vp, n = A.u32p(), C.c_uint64()
        self.eng._check(self.eng.lib.ii2_bitmask_all_values(self.h, C.byref(vp), C.byref(n)),
                        "bitmask_all_values")
        out = A.from_ptr(vp, n.value, np.uint32)
        self.eng.lib.ii2_free(vp)
        return out

    def put(self, values) -> bytes:
        v = np.ascontiguousarray(values, dtype=np.uint32)
        bp, nb = A.u8p(), C.c_uint64()
        self.eng._check(self.eng.lib.ii2_bitmask_put(
            self.h, A.np_ptr(v, A.u32p) if len(v) else C.cast(None, A.u32p), len(v), C.byref(bp),
            C.byref(nb)), "bitmask_put")
        data = C.string_at(bp, nb.value)
        self.eng.lib.ii2_free(bp)
        return data

    def get(self, enc: bytes) -> np.ndarray:
        p, n, keep = _bytes_arg(enc)
        vp, vn = A.u32p(), C.c_uint64()
        self.eng._check(self.eng.lib.ii2_bitmask_get(self.h, p, n, C.byref(vp), C.byref(vn)),
                        "bitmask_get")
        out = A.from_ptr(vp, vn.value, np.uint32)
        self.eng.lib.ii2_free(vp)
        return out


class Engine:
    """The process's GPUs (ii2_init binds them): one device, or with `devices` a set of them.

    With a set, host-buffer calls and uploads of a thread run on the device it selected with
    set_device (devices[0] by default); calls on resident handles run on the handles' device."""

    _default = None
    _lock = threading.Lock()

    def __init__(self, device: int = 0, devices: list[int] | None = None):
        self.lib = load_library()
        devs = [int(d) for d in devices] if devices is not None else [device]
        if not devs:
            raise ValueError("Engine(devices=...) needs at least one device")
        arr = (C.c_int * max(1, len(devs)))(*devs)
        rc = self.lib.ii2_init(arr, len(devs))
        if rc != A.II2_OK:
            raise EngineError(rc, "ii2_init failed — no CPU fallback exists",
                              self.lib.ii2_last_error().decode())
        self.device = devs[0]
        self.devices = devs
        self._tls = threading.local()

    def set_device(self, device: int) -> None:
        """Device of this thread's host-buffer calls and uploads (one of `devices`)."""
        self._check(self.lib.ii2_set_device(int(device)), "set_device")
        self._tls.device = int(device)

    def selected_device(self) -> int:
        return getattr(self._tls, "device", self.device)

    @classmethod
    def default(cls) -> "Engine":
        with cls._lock:
            if cls._default is None:
                cls._default = cls(int(os.environ.get("LOCAL_RANK", "0")))
            return cls._default

    def _check(self, rc: int, what: str):
        if rc != A.II2_OK:
            raise EngineError(rc, f"{what}: {self.lib.ii2_strerror(rc).decode()}",
                              self.lib.ii2_last_error().decode())

    # ---- host-buffer calls (what cgo would call from Shard.Merge / Shard.Read) ------
    def merge(self, segs: list[FlatSegment], removed=None, decoded: bool = False) -> MergeResult:
        arr = views_array(segs)
        r = np.ascontiguousarray(removed if removed is not None else [], dtype=np.uint32)
        out = A.MergeOut()
        self._check(self.lib.ii2_merge(arr, len(segs),
                                       A.np_ptr(r, A.u32p) if len(r) else C.cast(None, A.u32p),
                                       len(r), A.II2_MERGE_WANT_DECODED if decoded else 0,
                                       C.byref(out)), "merge")
        try:
            return MergeResult.from_c(out, decoded)
        finally:
            self.lib.ii2_merge_out_free(C.byref(out))

    def read_range(self, segs: list[FlatSegment], min_term: bytes | None = None,
                   max_term: bytes | None = None, removed=None) -> ReadResult:
        arr = views_array(segs)
        pmin, nmin, k1 = _bytes_arg(min_term)
        pmax, nmax, k2 = _bytes_arg(max_term)
        if removed is None:
            rp, nr, keep = C.cast(None, A.u32p), 0, None
        else:
            keep = np.ascontiguousarray(removed, dtype=np.uint32)
            if len(keep) == 0:
                keep = np.zeros(1, dtype=np.uint32)
                rp, nr = A.np_ptr(keep, A.u32p), 0
            else:
                rp, nr = A.np_ptr(keep, A.u32p), len(keep)
        out = A.ReadOut()
        self._check(self.lib.ii2_read_range(arr, len(segs), pmin, nmin, pmax, nmax, rp, nr,
                                            C.byref(out)), "read_range")
        try:
            return ReadResult.from_c(out)
        finally:
            self.lib.ii2_read_out_free(C.byref(out))

    # ---- device-resident calls -----------------------------------------------------
    def upload(self, seg: FlatSegment) -> DeviceSegment:
        v = seg.view()
        h = C.c_void_p()
        self._check(self.lib.ii2_seg_upload(C.byref(v), C.byref(h)), "seg_upload")
        return DeviceSegment(self, h.value, seg.n_terms, self.selected_device())

    def upload_removed(self, removed) -> DeviceRemoved:
        r = np.ascontiguousarray(removed, dtype=np.uint32)
        h = C.c_void_p()
        self._check(self.lib.ii2_removed_upload(
            A.np_ptr(r, A.u32p) if len(r) else C.cast(None, A.u32p), len(r), C.byref(h)),
            "removed_upload")
        return DeviceRemoved(self, h.value, self.selected_device())

    def _call_device(self, segs, removed) -> int:
        """Where a call on these handles runs (and its result lives)."""
        if segs:
            return segs[0].device
        return removed.device if removed is not None else self.selected_device()

    def result_device(self, res: DeviceResult) -> int:
        d = C.c_int(-1)
        self._check(self.lib.ii2_result_device(res.h, C.byref(d)), "result_device")
        return d.value

    @staticmethod
    def _handles(segs: list[DeviceSegment]):
        arr = (C.c_void_p * max(1, len(segs)))()
        for i, s in enumerate(segs):
            arr[i] = s.h
        return arr

    def merge_dev(self, segs: list[DeviceSegment], removed: DeviceRemoved | None = None,
                  encode: bool = True, decoded: bool = False) -> DeviceResult:
        flags = (A.II2_RESULT_ENCODED if encode else 0) | (A.II2_RESULT_DECODED if decoded else 0)
        h = C.c_void_p()
        self._check(self.lib.ii2_merge_dev(self._handles(segs), len(segs),
                                           removed.h if removed else None, flags, C.byref(h)),
                    "merge_dev")
        return DeviceResult(self, h.value, self._call_device(segs, removed))

    def read_range_dev(self, segs: list[DeviceSegment], min_term: bytes | None = None,
                       max_term: bytes | None = None, removed: DeviceRemoved | None = None
                       ) -> DeviceResult:
        pmin, nmin, k1 = _bytes_arg(min_term)
        pmax, nmax, k2 = _bytes_arg(max_term)
        h = C.c_void_p()
        self._check(self.lib.ii2_read_range_dev(self._handles(segs), len(segs), pmin, nmin, pmax,
                                                nmax, removed.h if removed else None, C.byref(h)),
                    "read_range_dev")
        return DeviceResult(self, h.value, self._call_device(segs, removed))

    # ---- ingest batching (Shard.Put x D + Shard.Merge as one call) ----------------------------
    def ingest(self, docs: list[tuple[list[bytes], int]], removed=None, decoded: bool = False
               ) -> MergeResult:
        """docs: (terms in any order, value) per document; returns the merged segment."""
        arr = (A.DocView * max(1, len(docs)))()
        keep = []
        for i, (terms, val) in enumerate(docs):
            off = np.zeros(len(terms) + 1, dtype=np.uint32)
            if terms:
                off[1:] = np.cumsum([len(t) for t in terms])
            blob = np.frombuffer(b"".join(terms) + b"\0", dtype=np.uint8).copy()
            keep.append((off, blob))
            arr[i].n_terms = len(terms)
            arr[i].term_bytes = A.np_ptr(blob, A.u8p)
            arr[i].term_off = A.np_ptr(off, A.u32p)
            arr[i].value = int(val)
        r = np.ascontiguousarray(removed if removed is not None else [], dtype=np.uint32)
        out = A.MergeOut()
        self._check(self.lib.ii2_ingest(arr, len(docs),
                                        A.np_ptr(r, A.u32p) if len(r) else C.cast(None, A.u32p),
                                        len(r), A.II2_MERGE_WANT_DECODED if decoded else 0,
                                        C.byref(out)), "ingest")
        try:
            return MergeResult.from_c(out, decoded)
        finally:
            self.lib.ii2_merge_out_free(C.byref(out))

    # ---- PrefixSearch (inverted_index.go:192-295) ----------------------------------------
    @staticmethod
    def _prefix_args(prefixes: list[bytes]):
        off = np.zeros(len(prefixes) + 1, dtype=np.uint32)
        if prefixes:
            off[1:] = np.cumsum([len(p) for p in prefixes], dtype=np.uint64)
        blob = np.frombuffer(b"".join(prefixes) + b"\0", dtype=np.uint8).copy()
        return blob, off

    @staticmethod
    def _query_args(queries: list) -> tuple[A.QueryBatch, list]:
        """Packs queries into ii2_query_batch's three CSR levels.  A query is a list of clauses,
        a clause is (required: bool, [(bytes, is_prefix: bool), ...]).  Returns the struct and
        the arrays it points into (keep them alive for the call)."""
        atoms, kinds, clause_atom_off, excluded, query_clause_off = [], [], [0], [], [0]
        for clauses in queries:
            for required, alist in clauses:
                for term, is_prefix in alist:
                    atoms.append(bytes(term))
                    kinds.append(A.II2_ATOM_PREFIX if is_prefix else A.II2_ATOM_TERM)
                clause_atom_off.append(len(atoms))
                excluded.append(0 if required else 1)
            query_clause_off.append(len(excluded))
        blob, aoff = Engine._prefix_args(atoms)
        # one spare element each: no array is ever empty
        kind = np.array(kinds + [0], dtype=np.uint8)
        cao = np.array(clause_atom_off, dtype=np.uint32)
        excl = np.array(excluded + [0], dtype=np.uint8)
        qco = np.array(query_clause_off, dtype=np.uint32)
        b = A.QueryBatch()
        b.atom_bytes = A.np_ptr(blob, A.u8p)
        b.atom_off = A.np_ptr(aoff, A.u32p)
        b.atom_kind = A.np_ptr(kind, A.u8p)
        b.natoms = len(atoms)
        b.clause_atom_off = A.np_ptr(cao, A.u32p)
        b.clause_excluded = A.np_ptr(excl, A.u8p)
        b.nclauses = len(excluded)
        b.query_clause_off = A.np_ptr(qco, A.u32p)
        b.nqueries = len(queries)
        return b, [blob, aoff, kind, cao, excl, qco]

    def _prefix_result(self, prefixes: list[bytes], out: A.PrefixOut) -> dict[bytes, np.ndarray]:
        """Zero-copy: the returned arrays are views of the library's pinned result buffer, which
        is released (ii2_prefix_out_free) when the last view is garbage collected."""
        import weakref
        n = int(out.n_prefixes)
        off = A.from_ptr(out.value_off, n + 1, np.uint64)
        matched = A.from_ptr(out.matched, n, np.uint8)
        total = int(off[-1]) if n else 0
        lib = self.lib
        if total == 0:
            lib.ii2_prefix_out_free(C.byref(out))
            empty = np.zeros(0, dtype=np.uint32)
            return {p: empty for i, p in enumerate(prefixes) if matched[i]}
        vals = np.ctypeslib.as_array(out.values, shape=(total,))
        weakref.finalize(vals, lambda o=out: lib.ii2_prefix_out_free(C.byref(o)))
        return {p: vals[int(off[i]):int(off[i + 1])] for i, p in enumerate(prefixes) if matched[i]}

    def prefix_search(self, segs: list[FlatSegment], prefixes: list[bytes]
                      ) -> dict[bytes, np.ndarray]:
        """found[prefix] for every prefix with at least one matching term, over host views."""
        arr = views_array(segs)
        blob, off = self._prefix_args(prefixes)
        out = A.PrefixOut()
        self._check(self.lib.ii2_prefix_search(arr, len(segs), A.np_ptr(blob, A.u8p),
                                               A.np_ptr(off, A.u32p), len(prefixes),
                                               C.byref(out)), "prefix_search")
        return self._prefix_result(prefixes, out)

    def prefix_search_dev(self, segs: list[DeviceSegment], prefixes: list[bytes]
                          ) -> dict[bytes, np.ndarray]:
        blob, off = self._prefix_args(prefixes)
        out = A.PrefixOut()
        self._check(self.lib.ii2_prefix_search_dev(self._handles(segs), len(segs),
                                                   A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p),
                                                   len(prefixes), C.byref(out)),
                    "prefix_search_dev")
        return self._prefix_result(prefixes, out)

    # ---- batched term lookup: Read(t, t) for many keys at once --------------------------
    def _lookup_result(self, out: A.LookupOut) -> list[np.ndarray | None]:
        try:
            n = int(out.n_keys)
            found = A.from_ptr(out.found, n, np.uint8)
            off = A.from_ptr(out.post_off, n + 1, np.uint64)
            post = A.from_ptr(out.post, int(off[-1]) if n else 0, np.uint32)
        finally:
            self.lib.ii2_lookup_out_free(C.byref(out))
        return [post[int(off[i]):int(off[i + 1])] if found[i] else None for i in range(n)]

    def lookup(self, segs: list[FlatSegment], keys: list[bytes], removed=None
               ) -> list[np.ndarray | None]:
        """Read(key, key) for every key over host views: the key's list, or None if no term is
        found (aligned with `keys`)."""
        arr = views_array(segs)
        blob, off = self._prefix_args(keys)
        if removed is None:
            rp, nr, keep = C.cast(None, A.u32p), 0, None
        else:
            keep = np.ascontiguousarray(removed, dtype=np.uint32)
            nr = len(keep)
            if nr == 0:
                keep = np.zeros(1, dtype=np.uint32)
            rp = A.np_ptr(keep, A.u32p)
        out = A.LookupOut()
        self._check(self.lib.ii2_lookup(arr, len(segs), A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p),
                                        len(keys), rp, nr, C.byref(out)), "lookup")
        return self._lookup_result(out)

    def lookup_dev(self, segs: list[DeviceSegment], keys: list[bytes],
                   removed: DeviceRemoved | None = None) -> list[np.ndarray | None]:
        """Read(key, key) for every key over resident segments, in one call on their device."""
        blob, off = self._prefix_args(keys)
        out = A.LookupOut()
        self._check(self.lib.ii2_lookup_dev(self._handles(segs), len(segs), A.np_ptr(blob, A.u8p),
                                            A.np_ptr(off, A.u32p), len(keys),
                                            removed.h if removed else None, C.byref(out)),
                    "lookup_dev")
        return self._lookup_result(out)

    # ---- boolean term queries: AND / OR / NOT over exact terms and prefixes ------------------
    def _query_result(self, out: A.QueryOut) -> list[np.ndarray]:
        try:
            n = int(out.n_queries)
            off = A.from_ptr(out.value_off, n + 1, np.uint64)
            vals = A.from_ptr(out.values, int(off[-1]) if n else 0, np.uint32)
        finally:
            self.lib.ii2_query_out_free(C.byref(out))
        return [vals[int(off[i]):int(off[i + 1])] for i in range(n)]

    def query(self, segs: list[FlatSegment], queries: list, removed=None) -> list[np.ndarray]:
        """The values of every query over host views (see query_dev), aligned with `queries`."""
        arr = views_array(segs)
        batch, keep = self._query_args(queries)
        if removed is None:
            rp, nr, rkeep = C.cast(None, A.u32p), 0, None
        else:
            rkeep = np.ascontiguousarray(removed, dtype=np.uint32)
            nr = len(rkeep)
            if nr == 0:
                rkeep = np.zeros(1, dtype=np.uint32)
            rp = A.np_ptr(rkeep, A.u32p)
        out = A.QueryOut()
        self._check(self.lib.ii2_query(arr, len(segs), C.byref(batch), rp, nr, C.byref(out)), "query")
        return self._query_result(out)

    def query_dev(self, segs: list[DeviceSegment], queries: list,
                  removed: DeviceRemoved | None = None) -> list[np.ndarray]:
        """Boolean queries over resident segments in one call on their device.  A query is a list
        of clauses (required: bool, [(bytes, is_prefix: bool), ...]); its result is the ascending
        values in every required clause and in no excluded one (nor in `removed`), a clause
        holding the values of any of its exact terms or prefixes."""
        batch, keep = self._query_args(queries)
        out = A.QueryOut()
        self._check(self.lib.ii2_query_dev(self._handles(segs), len(segs), C.byref(batch),
                                           removed.h if removed else None, C.byref(out)), "query_dev")
        return self._query_result(out)

    # ---- term patterns: wildcard (glob) and fuzzy matching --------------------------------
    @staticmethod
    def _pattern_args(patterns: list) -> tuple[A.PatternBatch, list]:
        """Packs patterns into ii2_pattern_batch: `bytes` is a glob, (bytes, max_edits,
        prefix_len) a fuzzy pattern.  Returns the struct and the arrays it points into (keep
        them alive for the call)."""
        pats, kinds, edits, plens = [], [], [], []
        for p in patterns:
            if isinstance(p, (bytes, bytearray)):
                pats.append(bytes(p))
                kinds.append(A.II2_PATTERN_GLOB)
                edits.append(0)
                plens.append(0)
            else:
                q, k, plen = p
                pats.append(bytes(q))
                kinds.append(A.II2_PATTERN_FUZZY)
                edits.append(int(k))
                plens.append(int(plen))
        blob, off = Engine._prefix_args(pats)
        # one spare element each: no array is ever empty
        kind = np.array(kinds + [0], dtype=np.uint8)
        med = np.array(edits + [0], dtype=np.uint8)
        pl = np.array(plens + [0], dtype=np.uint32)
        b = A.PatternBatch()
        b.pat_bytes = A.np_ptr(blob, A.u8p)
        b.pat_off = A.np_ptr(off, A.u32p)
        b.pat_kind = A.np_ptr(kind, A.u8p)
        b.max_edits = A.np_ptr(med, A.u8p)
        b.prefix_len = A.np_ptr(pl, A.u32p)
        b.npat = len(pats)
        return b, [blob, off, kind, med, pl]

    def _pattern_result(self, out: A.PrefixOut) -> list[np.ndarray | None]:
        try:
            n = int(out.n_prefixes)
            matched = A.from_ptr(out.matched, n, np.uint8)
            off = A.from_ptr(out.value_off, n + 1, np.uint64)
            vals = A.from_ptr(out.values, int(off[-1]) if n else 0, np.uint32)
        finally:
            self.lib.ii2_prefix_out_free(C.byref(out))
        return [vals[int(off[i]):int(off[i + 1])] if matched[i] else None for i in range(n)]

    def pattern_search(self, segs: list[FlatSegment], patterns: list) -> list[np.ndarray | None]:
        """pattern_search_dev over host views (uploaded for the call)."""
        arr = views_array(segs)
        batch, keep = self._pattern_args(patterns)
        out = A.PrefixOut()
        self._check(self.lib.ii2_pattern_search(arr, len(segs), C.byref(batch), C.byref(out)),
                    "pattern_search")
        return self._pattern_result(out)

    def pattern_search_dev_out(self, segs: list[DeviceSegment], patterns: list) -> A.PrefixOut:
        """ii2_pattern_search_dev's raw output (a prefix output: input of prefix_gather_devices,
        with the pattern list in place of the prefixes); free it with prefix_out_free."""
        batch, keep = self._pattern_args(patterns)
        out = A.PrefixOut()
        self._check(self.lib.ii2_pattern_search_dev(self._handles(segs), len(segs), C.byref(batch),
                                                    C.byref(out)), "pattern_search_dev")
        return out

    def pattern_search_dev(self, segs: list[DeviceSegment], patterns: list) -> list[np.ndarray | None]:
        """Wildcard and fuzzy term matching over resident segments in one call on their device.
        A pattern is `bytes` (a glob: `*`, `?`, `[...]`, `\\x`) or (bytes, max_edits, prefix_len)
        (terms within max_edits byte edits of it whose first prefix_len bytes are equal).  Aligned
        with `patterns`: the sorted-unique values of every matching term, or None when no term
        matches."""
        return self._pattern_result(self.pattern_search_dev_out(segs, patterns))

    def _terms_result(self, out: A.TermsOut) -> list[list[tuple[bytes, int, int, int]]]:
        try:
            n, nt = int(out.n_patterns), int(out.n_terms)
            poff = A.from_ptr(out.pattern_term_off, n + 1, np.uint64)
            toff = A.from_ptr(out.term_off, nt + 1, np.uint64)
            tb = A.from_ptr(out.term_bytes, int(toff[-1]) if nt else 0, np.uint8).tobytes()
            seg = A.from_ptr(out.segments, nt, np.uint32).tolist()
            post = A.from_ptr(out.postings, nt, np.uint64).tolist()
            dist = A.from_ptr(out.distance, nt, np.uint8).tolist()
            toff = toff.tolist()
            poff = poff.tolist()
        finally:
            self.lib.ii2_terms_out_free(C.byref(out))
        terms = [(tb[toff[j]:toff[j + 1]], seg[j], post[j], dist[j]) for j in range(nt)]
        return [terms[poff[i]:poff[i + 1]] for i in range(n)]

    def pattern_terms(self, segs: list[FlatSegment], patterns: list
                      ) -> list[list[tuple[bytes, int, int, int]]]:
        """pattern_terms_dev over host views (uploaded for the call)."""
        arr = views_array(segs)
        batch, keep = self._pattern_args(patterns)
        out = A.TermsOut()
        self._check(self.lib.ii2_pattern_terms(arr, len(segs), C.byref(batch), C.byref(out)),
                    "pattern_terms")
        return self._terms_result(out)

    def pattern_terms_dev(self, segs: list[DeviceSegment], patterns: list
                          ) -> list[list[tuple[bytes, int, int, int]]]:
        """The terms each pattern matches over resident segments, in one call on their device.
        Patterns as in pattern_search_dev.  Aligned with `patterns`: the distinct matching terms
        in bytes order, each as (term, segments, postings, distance): the term's instances over
        `segs`, the sum of their stored list lengths, and for a fuzzy pattern its edit distance
        (0 for a glob)."""
        batch, keep = self._pattern_args(patterns)
        out = A.TermsOut()
        self._check(self.lib.ii2_pattern_terms_dev(self._handles(segs), len(segs), C.byref(batch),
                                                   C.byref(out)), "pattern_terms_dev")
        return self._terms_result(out)

    # ---- codec -----------------------------------------------------------------------
    def intcomp_encode_batch(self, post: np.ndarray, post_off: np.ndarray):
        post = np.ascontiguousarray(post, dtype=np.uint32)
        off = np.ascontiguousarray(post_off, dtype=np.uint64)
        n = len(off) - 1
        wp, op = A.u32p(), A.u64p()
        self._check(self.lib.ii2_intcomp_encode_u32(
            A.np_ptr(post, A.u32p) if len(post) else C.cast(None, A.u32p), A.np_ptr(off, A.u64p), n,
            C.byref(wp), C.byref(op)), "intcomp_encode")
        woff = A.from_ptr(op, n + 1, np.uint64)
        words = A.from_ptr(wp, int(woff[-1]) if n else 0, np.uint32)
        self.lib.ii2_free(wp)
        self.lib.ii2_free(op)
        return words, woff

    def intcomp_decode_batch(self, words: np.ndarray, word_off: np.ndarray):
        words = np.ascontiguousarray(words, dtype=np.uint32)
        woff = np.ascontiguousarray(word_off, dtype=np.uint64)
        n = len(woff) - 1
        vp, op = A.u32p(), A.u64p()
        self._check(self.lib.ii2_intcomp_decode_u32(
            A.np_ptr(words, A.u32p) if len(words) else C.cast(None, A.u32p), A.np_ptr(woff, A.u64p),
            n, C.byref(vp), C.byref(op)), "intcomp_decode")
        off = A.from_ptr(op, n + 1, np.uint64)
        vals = A.from_ptr(vp, int(off[-1]) if n else 0, np.uint32)
        self.lib.ii2_free(vp)
        self.lib.ii2_free(op)
        return vals, off

    def bitmask(self, init=None) -> Bitmask:
        return Bitmask(self, init)

    # ---- cross-shard exchange (NCCL behind the C-ABI; one process per GPU) -----------------
    def comm_unique_id(self) -> bytes:
        buf = (C.c_uint8 * 128)()
        self._check(self.lib.ii2_comm_unique_id(C.cast(buf, A.u8p)), "comm_unique_id")
        return bytes(buf)

    def comm_init(self, uid: bytes, rank: int, world: int) -> None:
        buf = (C.c_uint8 * 128).from_buffer_copy(uid.ljust(128, b"\0")[:128])
        self._check(self.lib.ii2_comm_init(C.cast(buf, A.u8p), rank, world), "comm_init")

    def comm_info(self) -> tuple[int, int]:
        r, w = C.c_int(), C.c_int()
        self.lib.ii2_comm_info(C.byref(r), C.byref(w))
        return r.value, w.value

    def comm_shutdown(self) -> None:
        self.lib.ii2_comm_shutdown()

    def read_gather(self, local: DeviceResult, root: int = 0) -> DeviceResult:
        """Collective (every rank): the rank-ordered concatenation of the ranks' decoded read
        results on `root` (every rank if root < 0) — InvertedIndex.Read over all shards."""
        h = C.c_void_p()
        self._check(self.lib.ii2_read_gather(local.h, root, C.byref(h)), "read_gather")
        return DeviceResult(self, h.value, local.device)

    def prefix_search_gather(self, segs: list[DeviceSegment], prefixes: list[bytes], root: int = 0
                             ) -> dict[bytes, np.ndarray]:
        """Collective: this rank's prefix search over its resident shards, then the per-prefix
        sorted-unique union of every rank's values on `root` (other ranks get {})."""
        blob, off = self._prefix_args(prefixes)
        local, merged = A.PrefixOut(), A.PrefixOut()
        self._check(self.lib.ii2_prefix_search_dev(self._handles(segs), len(segs),
                                                   A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p),
                                                   len(prefixes), C.byref(local)), "prefix_search_dev")
        try:
            self._check(self.lib.ii2_prefix_gather(C.byref(local), root, C.byref(merged)), "prefix_gather")
        finally:
            self.lib.ii2_prefix_out_free(C.byref(local))
        return self._prefix_result(prefixes, merged)

    # ---- in-process gathers over the devices of this process -----------------------------
    def read_gather_devices(self, parts: list[DeviceResult], root_device: int) -> DeviceResult:
        """The part-ordered concatenation of decoded read results that live on any of this
        process's devices, on `root_device` (one peer-reading kernel there)."""
        arr = (C.c_void_p * max(1, len(parts)))()
        for i, p in enumerate(parts):
            arr[i] = p.h
        h = C.c_void_p()
        self._check(self.lib.ii2_read_gather_devices(arr, len(parts), int(root_device), C.byref(h)),
                    "read_gather_devices")
        return DeviceResult(self, h.value, int(root_device))

    def prefix_search_dev_out(self, segs: list[DeviceSegment], prefixes: list[bytes]) -> A.PrefixOut:
        """ii2_prefix_search_dev's raw output (input of prefix_gather_devices); free it with
        prefix_out_free."""
        blob, off = self._prefix_args(prefixes)
        out = A.PrefixOut()
        self._check(self.lib.ii2_prefix_search_dev(self._handles(segs), len(segs),
                                                   A.np_ptr(blob, A.u8p), A.np_ptr(off, A.u32p),
                                                   len(prefixes), C.byref(out)), "prefix_search_dev")
        return out

    def prefix_out_free(self, out: A.PrefixOut) -> None:
        self.lib.ii2_prefix_out_free(C.byref(out))

    def prefix_gather_devices(self, parts: list, prefixes: list[bytes], root_device: int
                              ) -> dict[bytes, np.ndarray]:
        """found[prefix] over several devices: `parts` are raw prefix outputs of `prefixes`
        (prefix_search_dev_out; the caller keeps and frees them) or groups of resident segments
        (searched here, each group on its own device); the union runs on `root_device`."""
        outs, owned = [], []
        try:
            for p in parts:
                if isinstance(p, A.PrefixOut):
                    outs.append(p)
                else:
                    o = self.prefix_search_dev_out(list(p), prefixes)
                    owned.append(o)
                    outs.append(o)
            arr = (A.PrefixOut * max(1, len(outs)))(*outs)
            merged = A.PrefixOut()
            self._check(self.lib.ii2_prefix_gather_devices(arr, len(outs), int(root_device),
                                                           C.byref(merged)), "prefix_gather_devices")
        finally:
            for o in owned:
                self.prefix_out_free(o)
        return self._prefix_result(prefixes, merged)

    # ---- misc --------------------------------------------------------------------------
    def set_stream(self, cuda_stream: int | None):
        self._check(self.lib.ii2_set_stream(cuda_stream), "set_stream")

    def sync(self):
        self._check(self.lib.ii2_sync(), "sync")

    def prof_enable(self, on: bool):
        self._check(self.lib.ii2_prof_enable(int(on)), "prof_enable")

    def prof_read(self) -> list[dict]:
        arr = (A.ProfEntry * 32)()
        n = self.lib.ii2_prof_read(arr, 32)
        if n < 0:
            self._check(n, "prof_read")
        return [{"name": arr[i].name.decode(), "ms": float(arr[i].ms),
                 "host_ms": float(arr[i].host_ms), "count": int(arr[i].count)}
                for i in range(n)]

    def kernel_launches(self) -> int:
        return int(self.lib.ii2_kernel_launches())

    def shard_key(self, term: bytes) -> int:
        p, n, keep = _bytes_arg(term)
        return int(self.lib.ii2_shard_key(p, n))
