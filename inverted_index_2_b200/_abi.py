"""ctypes mirror of include/ii2.h (structs, error codes, prototypes).

The same struct layouts are used to call the product library (libii2.so, CUDA)
and — from tests/bench only — the CPU oracle (oracle/libii2_oracle.so), which
shares the view/out structs so identical inputs can be handed to both.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

II2_OK = 0
II2_ERR_INVALID = -1
II2_ERR_NOMEM = -2
II2_ERR_CUDA = -3
II2_ERR_NO_DEVICE = -4
II2_ERR_BITMASK_OOB = -5
II2_ERR_CORRUPT = -6
II2_ERR_UNSUPPORTED = -7

II2_SEG_DECODED = 0
II2_SEG_VAL = 1
II2_SEG_DIRECT = 2

II2_MERGE_WANT_DECODED = 1
II2_RESULT_ENCODED = 1
II2_RESULT_DECODED = 2

II2_ATOM_TERM = 0
II2_ATOM_PREFIX = 1

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)


class SegView(C.Structure):
    _fields_ = [
        ("n_terms", C.c_uint64),
        ("term_bytes", u8p),
        ("term_off", u32p),
        ("mode", C.c_int32),
        ("post", u32p),
        ("post_off", u64p),
        ("val_bytes", u8p),
        ("val_off", u64p),
        ("val_size", C.c_uint64),
        ("val_woff32", u32p),
    ]


class MergeOut(C.Structure):
    _fields_ = [
        ("terms_count", C.c_uint64),
        ("term_bytes", u8p),
        ("term_off", u32p),
        ("val_off", u64p),
        ("val_bytes", u8p),
        ("val_size", C.c_uint64),
        ("has_minmax", C.c_int32),
        ("min_term", u8p),
        ("min_term_len", C.c_uint32),
        ("max_term", u8p),
        ("max_term_len", C.c_uint32),
        ("post", u32p),
        ("post_off", u64p),
        ("terms_merged", C.c_uint64),
        ("postings_in", C.c_uint64),
        ("postings_out", C.c_uint64),
        ("_owner", C.c_void_p),
    ]


class ReadOut(C.Structure):
    _fields_ = [
        ("n_terms", C.c_uint64),
        ("term_bytes", u8p),
        ("term_off", u32p),
        ("post", u32p),
        ("post_off", u64p),
        ("_owner", C.c_void_p),
    ]


class DocView(C.Structure):
    _fields_ = [
        ("n_terms", C.c_uint64),
        ("term_bytes", u8p),
        ("term_off", u32p),
        ("value", C.c_uint32),
    ]


class PrefixOut(C.Structure):
    _fields_ = [
        ("n_prefixes", C.c_uint64),
        ("matched", u8p),
        ("values", u32p),
        ("value_off", u64p),
        ("_owner", C.c_void_p),
    ]


class LookupOut(C.Structure):
    _fields_ = [
        ("n_keys", C.c_uint64),
        ("found", u8p),
        ("post", u32p),
        ("post_off", u64p),
        ("postings_in", C.c_uint64),
        ("_owner", C.c_void_p),
    ]


class QueryBatch(C.Structure):
    _fields_ = [
        ("atom_bytes", u8p),
        ("atom_off", u32p),
        ("atom_kind", u8p),
        ("natoms", C.c_uint32),
        ("clause_atom_off", u32p),
        ("clause_excluded", u8p),
        ("nclauses", C.c_uint32),
        ("query_clause_off", u32p),
        ("nqueries", C.c_uint32),
    ]


class QueryOut(C.Structure):
    _fields_ = [
        ("n_queries", C.c_uint64),
        ("values", u32p),
        ("value_off", u64p),
        ("clause_values", C.c_uint64),
        ("_owner", C.c_void_p),
    ]


class FstTerms(C.Structure):
    _fields_ = [
        ("n_terms", C.c_uint64),
        ("term_bytes", u8p),
        ("term_off", u32p),
        ("values", u64p),
        ("fst_len", C.c_uint64),
        ("_owner", C.c_void_p),
    ]


class RemovedLists(C.Structure):
    _fields_ = [
        ("n_lists", C.c_uint64),
        ("timestamps", C.POINTER(C.c_int64)),
        ("off", u64p),
        ("values", u32p),
        ("_owner", C.c_void_p),
    ]


class ResultInfo(C.Structure):
    _fields_ = [
        ("terms_count", C.c_uint64),
        ("term_bytes", C.c_uint64),
        ("postings_out", C.c_uint64),
        ("postings_in", C.c_uint64),
        ("terms_merged", C.c_uint64),
        ("val_size", C.c_uint64),
        ("d_term_bytes", C.c_void_p),
        ("d_term_off", C.c_void_p),
        ("d_post", C.c_void_p),
        ("d_post_off", C.c_void_p),
        ("d_val_bytes", C.c_void_p),
        ("d_val_off", C.c_void_p),
    ]


class ProfEntry(C.Structure):
    _fields_ = [("name", C.c_char_p), ("ms", C.c_double), ("host_ms", C.c_double),
                ("count", C.c_uint64)]


# name -> (restype, argtypes); every symbol include/ii2.h declares.
PROTOTYPES = {
    "ii2_init": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "ii2_shutdown": (C.c_int, []),
    "ii2_abi_version": (C.c_int, []),
    "ii2_strerror": (C.c_char_p, [C.c_int]),
    "ii2_last_error": (C.c_char_p, []),
    "ii2_set_stream": (C.c_int, [C.c_void_p]),
    "ii2_set_device": (C.c_int, [C.c_int]),
    "ii2_kernel_launches": (C.c_uint64, []),
    "ii2_prof_enable": (C.c_int, [C.c_int]),
    "ii2_prof_read": (C.c_int, [C.POINTER(ProfEntry), C.c_int]),
    "ii2_free": (None, [C.c_void_p]),
    "ii2_merge": (C.c_int, [C.POINTER(SegView), C.c_int, u32p, C.c_uint64, C.c_uint32,
                            C.POINTER(MergeOut)]),
    "ii2_merge_out_free": (None, [C.POINTER(MergeOut)]),
    "ii2_ingest": (C.c_int, [C.POINTER(DocView), C.c_int, u32p, C.c_uint64, C.c_uint32,
                             C.POINTER(MergeOut)]),
    "ii2_read_range": (C.c_int, [C.POINTER(SegView), C.c_int, u8p, C.c_size_t, u8p, C.c_size_t,
                                 u32p, C.c_uint64, C.POINTER(ReadOut)]),
    "ii2_read_out_free": (None, [C.POINTER(ReadOut)]),
    "ii2_seg_upload": (C.c_int, [C.POINTER(SegView), C.POINTER(C.c_void_p)]),
    "ii2_seg_release": (None, [C.c_void_p]),
    "ii2_removed_upload": (C.c_int, [u32p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "ii2_removed_release": (None, [C.c_void_p]),
    "ii2_merge_dev": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_uint32,
                                C.POINTER(C.c_void_p)]),
    "ii2_read_range_dev": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, u8p, C.c_size_t, u8p,
                                     C.c_size_t, C.c_void_p, C.POINTER(C.c_void_p)]),
    "ii2_result_info_get": (C.c_int, [C.c_void_p, C.POINTER(ResultInfo)]),
    "ii2_result_download_merge": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(MergeOut)]),
    "ii2_result_download_read": (C.c_int, [C.c_void_p, C.POINTER(ReadOut)]),
    "ii2_result_to_seg": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "ii2_result_release": (None, [C.c_void_p]),
    "ii2_sync": (C.c_int, []),
    "ii2_result_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "ii2_prefix_search_dev": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, u8p, u32p, C.c_uint32,
                                        C.POINTER(PrefixOut)]),
    "ii2_prefix_search": (C.c_int, [C.POINTER(SegView), C.c_int, u8p, u32p, C.c_uint32,
                                    C.POINTER(PrefixOut)]),
    "ii2_prefix_out_free": (None, [C.POINTER(PrefixOut)]),
    "ii2_lookup_dev": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, u8p, u32p, C.c_uint32, C.c_void_p,
                                 C.POINTER(LookupOut)]),
    "ii2_lookup": (C.c_int, [C.POINTER(SegView), C.c_int, u8p, u32p, C.c_uint32, u32p, C.c_uint64,
                             C.POINTER(LookupOut)]),
    "ii2_lookup_out_free": (None, [C.POINTER(LookupOut)]),
    "ii2_query_dev": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(QueryBatch), C.c_void_p,
                                C.POINTER(QueryOut)]),
    "ii2_query": (C.c_int, [C.POINTER(SegView), C.c_int, C.POINTER(QueryBatch), u32p, C.c_uint64,
                            C.POINTER(QueryOut)]),
    "ii2_query_out_free": (None, [C.POINTER(QueryOut)]),
    "ii2_comm_unique_id": (C.c_int, [u8p]),
    "ii2_comm_init": (C.c_int, [u8p, C.c_int, C.c_int]),
    "ii2_comm_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ii2_comm_shutdown": (None, []),
    "ii2_read_gather": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "ii2_prefix_gather": (C.c_int, [C.POINTER(PrefixOut), C.c_int, C.POINTER(PrefixOut)]),
    "ii2_read_gather_devices": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int,
                                          C.POINTER(C.c_void_p)]),
    "ii2_prefix_gather_devices": (C.c_int, [C.POINTER(PrefixOut), C.c_int, C.c_int,
                                            C.POINTER(PrefixOut)]),
    "ii2_intcomp_encode_u32": (C.c_int, [u32p, u64p, C.c_uint64, C.POINTER(u32p),
                                         C.POINTER(u64p)]),
    "ii2_intcomp_decode_u32": (C.c_int, [u32p, u64p, C.c_uint64, C.POINTER(u32p),
                                         C.POINTER(u64p)]),
    "ii2_bitmask_new": (C.c_int, [u32p, C.c_uint64, C.POINTER(C.c_void_p)]),
    "ii2_bitmask_free": (None, [C.c_void_p]),
    "ii2_bitmask_all_values": (C.c_int, [C.c_void_p, C.POINTER(u32p), C.POINTER(C.c_uint64)]),
    "ii2_bitmask_put": (C.c_int, [C.c_void_p, u32p, C.c_uint64, C.POINTER(u8p),
                                  C.POINTER(C.c_uint64)]),
    "ii2_bitmask_get": (C.c_int, [C.c_void_p, u8p, C.c_uint64, C.POINTER(u32p),
                                  C.POINTER(C.c_uint64)]),
    "ii2_fst_read": (C.c_int, [u8p, C.c_uint64, u8p, C.c_size_t, u8p, C.c_size_t,
                               C.POINTER(FstTerms)]),
    "ii2_fst_terms_free": (None, [C.POINTER(FstTerms)]),
    "ii2_fst_get": (C.c_int, [u8p, C.c_uint64, u8p, C.c_size_t, C.POINTER(C.c_uint64),
                              C.POINTER(C.c_int)]),
    "ii2_fst_len": (C.c_int, [u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "ii2_fst_build": (C.c_int, [u8p, u32p, u64p, C.c_uint64, C.POINTER(u8p),
                                C.POINTER(C.c_uint64)]),
    "ii2_fst_free": (None, [C.c_void_p]),
    "ii2_removed_list_encode": (C.c_int, [C.POINTER(C.c_int64), u64p, u32p, C.c_uint64,
                                          C.POINTER(u8p), C.POINTER(C.c_uint64)]),
    "ii2_removed_list_decode": (C.c_int, [u8p, C.c_uint64, C.POINTER(RemovedLists)]),
    "ii2_removed_lists_free": (None, [C.POINTER(RemovedLists)]),
    "ii2_shard_key": (C.c_uint32, [u8p, C.c_size_t]),
}


def bind(lib: C.CDLL, prototypes: dict) -> None:
    """Attach restype/argtypes; raises AttributeError if a symbol is missing."""
    for name, (res, args) in prototypes.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args


def np_ptr(a: np.ndarray | None, typ):
    if a is None:
        return C.cast(None, typ)
    return a.ctypes.data_as(typ)


def from_ptr(ptr, n: int, dtype) -> np.ndarray:
    """Copy n elements out of a C pointer into a fresh numpy array."""
    n = int(n)
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    addr = C.cast(ptr, C.c_void_p).value
    buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(addr)
    return np.frombuffer(buf, dtype=dtype, count=n).copy()
