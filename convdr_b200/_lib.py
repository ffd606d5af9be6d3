"""ctypes binding of the C ABI in include/b2f.h.  Fails loudly when the library is missing."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libb2f.so")

# every symbol include/b2f.h declares (checked by tests/test_abi.py against the header)
SYMBOLS = {
    "b2f_device_count": (C.c_int, []),
    "b2f_create": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "b2f_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "b2f_add_with_ids": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "b2f_add_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "b2f_reserve": (C.c_int, [C.c_void_p, C.c_int64]),
    "b2f_add_flat_file": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_double),
                                    C.POINTER(C.c_double)]),
    "b2f_write_flat_file": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p]),
    "b2f_rank_dedup_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int,
                                        C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2f_add_synthetic": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_uint64, C.c_uint64,
                                    C.c_float, C.c_int64]),
    "b2f_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_search_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_search_device_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_search_finish": (C.c_int, [C.c_void_p]),
    "b2f_selector_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                      C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "b2f_selector_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "b2f_selector_destroy": (None, [C.c_void_p]),
    "b2f_search_sel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_search_device_async_sel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                              C.c_void_p]),
    "b2f_search_xchg_async_sel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_int]),
    "b2f_merge_packed_device_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64,
                                                C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_xchg_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p]),
    "b2f_xchg_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b2f_search_xchg_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "b2f_xchg_flush": (C.c_int, [C.c_void_p]),
    "b2f_search_xchg_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "b2f_merge_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int,
                                   C.c_void_p, C.c_void_p]),
    "b2f_reconstruct_n": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_void_p]),
    "b2f_reconstruct_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "b2f_search_and_reconstruct_sel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                                 C.c_void_p, C.c_void_p]),
    "b2f_search_and_reconstruct_device_sel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "b2f_reset": (C.c_int, [C.c_void_p]),
    "b2f_ntotal": (C.c_int64, [C.c_void_p]),
    "b2f_shard_rows": (C.c_int64, [C.c_void_p, C.c_int]),
    "b2f_num_shards": (C.c_int, [C.c_void_p]),
    "b2f_stream": (C.c_void_p, [C.c_void_p, C.c_int]),
    "b2f_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "b2f_get_stat": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double)]),
    "b2f_destroy": (None, [C.c_void_p]),
    "b2f_last_error": (C.c_char_p, []),
    "b2f_version": (C.c_char_p, []),
}

_lib = None


def load() -> C.CDLL:
    """Load libb2f.so (built in-tree by `python -m convdr_b200.build`).  No fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m convdr_b200.build` "
            "(nvcc, sm_100a).  convdr_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().b2f_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """FAISS surfaces C++ exceptions as RuntimeError (SURVEY §8b); so do we."""
    if rc != 0:
        raise RuntimeError(f"b2f error {rc}: {last_error()}")
