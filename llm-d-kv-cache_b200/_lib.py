"""ctypes binding of libkvb.so (include/kvb.h).  No CPU fallback: if the library is missing or a
compute entry point fails, callers get an exception."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkvb.so")

KVB_OK = 0
ABI_VERSION = 5
COPY_DEFAULT, COPY_LDG, COPY_BULK = 0, 1, 2
TIER_FILE, TIER_HOST_ARENA = 0, 1
MAX_PODS_PER_KEY = 13
KEY_ENGINE, KEY_REQUEST = 0, 1
SCORE_TOUCH_LRU, SCORE_NO_TOUCH, SCORE_TIME_KERNELS, SCORE_COPY_TOKENS, SCORE_TWO_KERNELS, SCORE_PINNED_IO = 1, 2, 4, 8, 16, 32


class KvbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libkvb error {code}: {msg}")
        self.code = code
        self.msg = msg


class EngineOpts(C.Structure):
    _fields_ = [
        ("io_threads", C.c_int32), ("gpu_blocks_per_file", C.c_int32), ("read_preferring_workers", C.c_int32),
        ("max_write_queued_seconds", C.c_float), ("tier", C.c_int32), ("copy_flags", C.c_int32),
        ("host_arena_bytes", C.c_int64), ("chunk_bytes", C.c_int64), ("direct_host_io", C.c_int32),
        ("strict_load_errors", C.c_int32), ("gds_mode", C.c_int32), ("arena_alloc_mode", C.c_int32),
    ]


class EngineStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "bytes_stored", "bytes_loaded", "files_stored", "files_loaded", "files_skipped_existing",
        "writes_dropped", "load_failures", "kernels_launched", "h2d_bytes", "d2h_bytes")]


class IndexStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in (
        "live_keys", "tombstones", "table_slots", "engine_keys", "ops_applied", "flushes_parallel",
        "flushes_sequential", "flushes_planned", "plan_fallbacks", "replay_resumes", "rehashes", "lru_evictions", "order_builds", "order_stale_skipped", "order_scans")] + [
        ("last_hash_us", C.c_float), ("last_score_us", C.c_float)]


class PodEntryC(C.Structure):
    _fields_ = [("pod", C.c_uint16), ("tier", C.c_uint8), ("speculative", C.c_uint8)]


class KvEvent(C.Structure):  # kvb_kv_event_t
    _fields_ = [("type", C.c_int32), ("stream", C.c_int32), ("token_off", C.c_int64), ("n_tokens", C.c_int64),
                ("engine_key_off", C.c_int64), ("n_engine_keys", C.c_int64), ("parent_engine_key", C.c_uint64),
                ("root_hash", C.c_uint64), ("entry", PodEntryC), ("pad", C.c_int32)]


EVENT_BLOCK_STORED, EVENT_BLOCK_REMOVED, EVENT_OTHER, EVENT_POD_CLEARED = 0, 1, 2, 3


class IpcMem(C.Structure):
    _fields_ = [("handle", C.c_uint8 * 64), ("offset", C.c_int64)]


_vp, _i32, _i64, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
_P = C.POINTER

# name -> (restype, argtypes); every function declared in include/kvb.h
SIGNATURES = {
    "kvb_abi_version": (C.c_int, []),
    "kvb_last_error": (C.c_char_p, []),
    "kvb_device_count": (C.c_int, []),
    "kvb_host_alloc": (C.c_int, [C.c_size_t, _P(_vp)]),
    "kvb_host_free": (C.c_int, [_vp]),
    "kvb_host_alloc_mode": (C.c_int, [C.c_size_t, C.c_int, _P(_vp)]),
    "kvb_pool_create": (C.c_int, [C.c_int, _P(_vp), _i32, _i64, _i64, _i64, _P(_vp)]),
    "kvb_pool_destroy": (None, [_vp]),
    "kvb_pool_block_bytes": (_i64, [_vp]),
    "kvb_pool_mark_peer": (C.c_int, [_vp, C.c_int]),
    "kvb_gather_blocks": (C.c_int, [_vp, _P(_i64), _i64, _vp, _vp, C.c_int]),
    "kvb_scatter_blocks": (C.c_int, [_vp, _P(_i64), _i64, _vp, _vp, C.c_int]),
    "kvb_gather_blocks_dev": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.c_int]),
    "kvb_scatter_blocks_dev": (C.c_int, [_vp, _vp, _i64, _vp, _vp, C.c_int]),
    "kvb_launch_count": (_i64, []),
    "kvb_engine_default_opts": (None, [_P(EngineOpts)]),
    "kvb_engine_create": (C.c_int, [_vp, _P(EngineOpts), _P(_vp)]),
    "kvb_engine_destroy": (None, [_vp]),
    "kvb_engine_store": (C.c_int, [_vp, _i64, _i32, _P(C.c_char_p), _P(_i64), _P(_i64), _vp]),
    "kvb_engine_load": (C.c_int, [_vp, _i64, _i32, _P(C.c_char_p), _P(_i64), _P(_i64), _vp]),
    "kvb_engine_poll": (C.c_int, [_vp, _P(_i64), _P(_i32), _i32]),
    "kvb_engine_wait": (C.c_int, [_vp, _i64]),
    "kvb_engine_exists": (C.c_int, [_vp, C.c_char_p]),
    "kvb_engine_lookup_prefix": (C.c_int, [_vp, _i32, _P(C.c_char_p), _P(_i32)]),
    "kvb_engine_lookup_prefix_hashes": (C.c_int, [_vp, C.c_char_p, _vp, _i32, _P(_i32)]),
    "kvb_engine_arena_clear": (C.c_int, [_vp]),
    "kvb_engine_get_stats": (C.c_int, [_vp, _P(EngineStats)]),
    "kvb_fnv64a": (_u64, [_vp, C.c_size_t]),
    "kvb_init_hash": (C.c_int, [C.c_int, _u64, C.c_char_p, C.c_size_t, _P(_u64)]),
    "kvb_hash_token_blocks": (C.c_int, [C.c_int, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "kvb_hash_token_blocks_dev": (C.c_int, [C.c_int, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, C.c_int64, _vp]),
    "kvb_index_create": (C.c_int, [C.c_int, _i64, _i32, _i64, _P(_vp)]),
    "kvb_index_destroy": (None, [_vp]),
    "kvb_index_set_tier_weight": (C.c_int, [_vp, C.c_uint8, C.c_double, C.c_int]),
    "kvb_index_add": (C.c_int, [_vp, _vp, _i64, C.c_int, _vp, _i64, _P(PodEntryC), _i32]),
    "kvb_index_evict": (C.c_int, [_vp, _u64, C.c_int, _P(PodEntryC), _i32]),
    "kvb_index_get_request_key": (C.c_int, [_vp, _u64, _P(_u64)]),
    "kvb_index_num_keys": (_i64, [_vp]),
    "kvb_index_ingest_events": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _i32, _P(_i32)]),
    "kvb_index_remove_pods": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _P(_i64), _P(_i64)]),
    "kvb_index_flush": (C.c_int, [_vp, _vp]),
    "kvb_index_get_stats": (C.c_int, [_vp, _P(IndexStats)]),
    "kvb_index_lookup": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _vp, _P(_i64)]),
    "kvb_index_score_batch": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _i32, _vp, _vp, _vp]),
    "kvb_index_score_tokens_batch": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _i32,
                                               _vp, _vp, _vp]),
    "kvb_index_host_peek": (C.c_int, [_vp, _u64, _P(PodEntryC), _i32]),
    "kvb_ipc_export": (C.c_int, [C.c_int, _vp, _P(IpcMem)]),
    "kvb_ipc_import": (C.c_int, [C.c_int, _P(IpcMem), _P(_vp)]),
    "kvb_ipc_close": (C.c_int, [C.c_int, _vp, _i64]),
    "kvb_enable_peer_access": (C.c_int, [C.c_int, C.c_int]),
    "kvb_migrate_blocks": (C.c_int, [_vp, _vp, _P(_i64), _P(_i64), _i64, _vp, C.c_int]),
}

_lib = None


def load() -> C.CDLL:
    """Load libkvb.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python llm-d-kv-cache_b200/build.py` "
            "(nvcc, sm_100a).  There is no CPU fallback for this path.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    bind(lib)  # AttributeError => ABI mismatch, fail loudly
    if lib.kvb_abi_version() != ABI_VERSION:
        raise ImportError(f"libkvb ABI version {lib.kvb_abi_version()} != {ABI_VERSION}")
    _lib = lib
    return lib


def bind(lib, names=None) -> None:
    """Attach restype / argtypes of the declared entry points to a loaded library."""
    for name, (res, args) in SIGNATURES.items():
        if names is not None and name not in names:
            continue
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args


def check(rc: int) -> int:
    if rc < 0:
        raise KvbError(rc, load().kvb_last_error().decode("utf-8", "replace"))
    return rc
