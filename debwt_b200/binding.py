"""ctypes binding of the C ABI declared in include/debwt_b200.h (libdebwt_b200.so).

The shared library is the product; this module only marshals numpy buffers into plain pointers.
It fails loudly when the library is missing or no CUDA device is present -- there is no CPU
fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdebwt_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "debwt_b200.h")

c_u64 = ctypes.c_uint64
c_p = ctypes.c_void_p


class DebwtError(RuntimeError):
    pass


class ShardStats(ctypes.Structure):
    _fields_ = [(n, c_u64) for n in ("n_symbols", "n_records", "n_keys", "n_keys_local", "n_branch", "n_blue", "n_codes", "arena_bytes")] + \
               [(n, ctypes.c_float) for n in ("ms_total", "ms_sort", "ms_sort_sweeps")] + [("sort_sweeps", ctypes.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Stats(ctypes.Structure):
    _fields_ = [(n, c_u64) for n in ("n_symbols", "n_records", "n_keys", "n_branch", "n_blue", "n_codes", "n_special")] + \
               [(n, ctypes.c_float) for n in ("ms_h2d", "ms_pack", "ms_extract", "ms_sort", "ms_sort_sweeps", "ms_classify", "ms_special",
                                              "ms_codes", "ms_bluesort", "ms_emit", "ms_d2h", "ms_total")] + \
               [("sort_launches", ctypes.c_uint32), ("sort_sweeps", ctypes.c_uint32), ("total_launches", ctypes.c_uint32),
                ("reserved_", ctypes.c_uint32), ("arena_bytes", c_u64), ("arena_used_bytes", c_u64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_SIGS = {
    "debwt_last_error": (ctypes.c_char_p, []),
    "debwt_device_count": (ctypes.c_int, []),
    "debwt_launch_count": (ctypes.c_uint64, []),
    "debwt_create": (ctypes.c_int, [ctypes.POINTER(c_p), ctypes.c_int]),
    "debwt_destroy": (None, [c_p]),
    "debwt_set_sort_config": (ctypes.c_int, [c_p, ctypes.c_int]),
    "debwt_set_blue_grouping": (ctypes.c_int, [c_p, ctypes.c_int]),
    "debwt_set_ambiguity_policy": (ctypes.c_int, [c_p, ctypes.c_int, c_u64]),
    "debwt_set_records": (ctypes.c_int, [c_p, ctypes.POINTER(c_p), ctypes.POINTER(c_u64), c_u64]),
    "debwt_set_text": (ctypes.c_int, [c_p, c_p, c_u64, c_p, c_u64]),
    "debwt_set_text_device": (ctypes.c_int, [c_p, c_p, c_u64, c_p, c_u64]),
    "debwt_ingest_begin": (ctypes.c_int, [c_p, c_u64]),
    "debwt_ingest_reserve": (ctypes.c_int, [c_p, ctypes.POINTER(c_p), ctypes.POINTER(c_u64)]),
    "debwt_ingest_commit": (ctypes.c_int, [c_p, c_u64]),
    "debwt_ingest_append": (ctypes.c_int, [c_p, c_p, c_u64]),
    "debwt_ingest_end": (ctypes.c_int, [c_p, c_p, c_u64]),
    "debwt_host_alloc": (c_p, [c_u64]),
    "debwt_host_free": (None, [c_p]),
    "debwt_build": (ctypes.c_int, [c_p, ctypes.c_int]),
    "debwt_result_sizes": (ctypes.c_int, [c_p, ctypes.POINTER(c_u64), ctypes.POINTER(c_u64), ctypes.POINTER(c_u64)]),
    "debwt_result_copy": (ctypes.c_int, [c_p, c_p, c_p, c_p]),
    "debwt_get_stats": (ctypes.c_int, [c_p, ctypes.POINTER(Stats)]),
    "debwt_shard_create": (ctypes.c_int, [ctypes.POINTER(c_p), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]),
    "debwt_shard_destroy": (None, [c_p]),
    "debwt_shard_set_sort_config": (ctypes.c_int, [c_p, ctypes.c_int]),
    "debwt_shard_slice": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_u64, ctypes.POINTER(c_u64), ctypes.POINTER(c_u64)]),
    "debwt_shard_build": (ctypes.c_int, [c_p, c_p, ctypes.c_int, c_u64, c_p, c_u64]),
    "debwt_shard_result_device": (ctypes.c_int, [c_p, ctypes.POINTER(c_p), ctypes.POINTER(c_u64)]),
    "debwt_shard_result_copy": (ctypes.c_int, [c_p, c_p, c_p, c_p]),
    "debwt_shard_get_stats": (ctypes.c_int, [c_p, ctypes.POINTER(ShardStats)]),
    "debwt_build_multi": (ctypes.c_int, [c_p, ctypes.c_int, c_p, c_u64, c_p, c_u64, c_p, c_p, c_p, ctypes.POINTER(ShardStats)]),
    "debwt_index_build": (ctypes.c_int, [c_p]),
    "debwt_index_sizes": (ctypes.c_int, [c_p, ctypes.POINTER(c_u64)]),
    "debwt_index_copy": (ctypes.c_int, [c_p, c_p, c_p]),
    "debwt_index_count": (ctypes.c_int, [c_p, c_p, c_p, c_u64, c_p]),
    "debwt_set_result": (ctypes.c_int, [c_p, c_p, c_u64, c_p, c_u64, c_u64]),
    "debwt_index_sample_sa": (ctypes.c_int, [c_p, ctypes.c_uint32, ctypes.POINTER(ctypes.c_float)]),
    "debwt_index_sa": (ctypes.c_int, [c_p, c_p, c_u64, c_p]),
    "debwt_index_locate": (ctypes.c_int, [c_p, c_p, c_p, c_u64, c_p, c_p, c_u64]),
    "debwt_verify_text": (ctypes.c_int, [c_p, c_p, c_u64, ctypes.POINTER(c_u64), ctypes.POINTER(ctypes.c_float)]),
    "debwt_verify_text_device": (ctypes.c_int, [c_p, c_p, c_u64, ctypes.POINTER(c_u64), ctypes.POINTER(ctypes.c_float)]),
    "debwt_verify_bwt_device": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_u64, c_p, ctypes.POINTER(c_u64),
                                                ctypes.POINTER(ctypes.c_float)]),
    "debwt_verify_walk_device": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_u64, c_p, c_u64, ctypes.POINTER(c_u64), c_p]),
    "debwt_synth_random_bases": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_u64]),
    "debwt_synth_insert_family": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_u64, c_u64, c_u64, c_u64, c_p]),
    "debwt_synth_mutate": (ctypes.c_int, [ctypes.c_int, c_p, c_p, c_u64, c_u64, c_u64]),
    "debwt_k_pack": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p]),
    "debwt_k_extract": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_p]),
    "debwt_k_radix_sort_u64": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]),
    "debwt_k_rle": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_p, ctypes.POINTER(c_u64)]),
    "debwt_k_group_masks": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_p]),
    "debwt_k_branch_kmers": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_p, c_p, c_u64, ctypes.POINTER(c_u64)]),
    "debwt_k_codes": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_p, c_u64, ctypes.POINTER(c_u64), c_p, c_p, c_p, c_u64,
                                      ctypes.POINTER(c_u64)]),
    "debwt_k_sort_blue": (ctypes.c_int, [ctypes.c_int, c_p, c_u64, c_p, c_u64, c_p, c_p]),
    "debwt_bench_sort": (ctypes.c_int, [ctypes.c_int, c_u64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]),
    "debwt_bench_sort_passes": (ctypes.c_int, [ctypes.c_int, c_u64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float),
                                                ctypes.POINTER(ctypes.c_float)]),
}

_lib = None


DEV_HEADER = os.path.join(os.path.dirname(HERE), "include", "debwt_b200_dev.h")


def declared_symbols(header: str = HEADER):
    """Every function name the given header declares."""
    with open(header) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(debwt_[a-z0-9_]+)\s*\(", src)))


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise DebwtError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(there is no CPU fallback)")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise DebwtError(lib().debwt_last_error().decode(errors="replace"))
