"""ctypes binding of libcpbus.so (the C-ABI in include/cpbus.h).

This is plumbing only: every data-path call goes straight to the CUDA library.
There is no Python or CPU fallback — if the library is missing `load()` raises,
and on a box without a GPU `cpbus_create` returns CPBUS_ENODEV.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CPBUS_LIB") or os.path.join(HERE, "libcpbus.so")   # CPBUS_LIB: A/B builds of the same library

N_CODES = 17
MASK_ALL = 0x0001FFFF
TARGET_ALL = 0xFFFFFFFF
F_TICK, F_UNICAST = 0x1, 0x2
CFG_LOSSLESS, CFG_DIGEST = 0x1, 0x2
STORE_AUTO, STORE_V4, STORE_V8, STORE_BULK = 0, 1, 2, 3

OK, EINVAL, ENOMEM, ECUDA, EAGAIN, ENOSPC, ENOENT, ECLOSED, ENODEV, EORDER, ETIMEDOUT = 0, -1, -2, -3, -4, -5, -6, -7, -8, -9, -10
PUT_STAMP, PUT_RAW, PUT_NOWAIT = 0, 1, 2
EPHEMERAL_BIT, EPHEMERAL_SLOTS = 0x80000000, 65536


class Event(C.Structure):
    """cpbus_event: the frozen 32-byte record."""
    _fields_ = [("seq", C.c_uint64), ("ts_ns", C.c_uint64), ("code", C.c_uint32),
                ("source_id", C.c_uint32), ("target", C.c_uint32), ("flags", C.c_uint32)]

    def astuple(self):
        return (self.seq, self.ts_ns, self.code, self.source_id, self.target, self.flags)


class Config(C.Structure):
    _fields_ = [("n_max_subs", C.c_uint32), ("ring_cap", C.c_uint32), ("batch_cap", C.c_uint32),
                ("timers_per_sub", C.c_uint32), ("flags", C.c_uint32), ("device", C.c_int32),
                ("sub_id_base", C.c_uint32), ("store_path", C.c_uint32), ("stream", C.c_void_p),
                ("grid_ctas", C.c_uint32), ("reserved", C.c_uint32 * 5)]


class Digest(C.Structure):
    _fields_ = [("count", C.c_uint64), ("digest", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("publishes", C.c_uint64), ("deliveries", C.c_uint64), ("ticks", C.c_uint64),
                ("batches", C.c_uint64), ("kernel_launches", C.c_uint64), ("overwritten", C.c_uint64),
                ("published_by_code", C.c_uint64 * N_CODES), ("n_subs", C.c_uint32), ("n_timers", C.c_uint32),
                ("now_ns", C.c_uint64), ("intern_entries", C.c_uint64), ("intern_bytes", C.c_uint64),
                ("ephemeral_live", C.c_uint64), ("ephemeral_recycled", C.c_uint64),
                ("admit_passes", C.c_uint64), ("admit_skipped", C.c_uint64), ("admit_partial", C.c_uint64), ("device_splits", C.c_uint64)]


class PairCount(C.Structure):
    _fields_ = [("code", C.c_uint32), ("source_id", C.c_uint32), ("count", C.c_uint64)]


assert C.sizeof(Event) == 32

# every symbol include/cpbus.h declares: (restype, argtypes)
_P = C.POINTER
SYMBOLS = {
    "cpbus_create": (C.c_int, [_P(Config), _P(C.c_void_p)]),
    "cpbus_destroy": (C.c_int, [C.c_void_p]),
    "cpbus_create_sharded": (C.c_int, [_P(Config), _P(C.c_int32), C.c_uint32, _P(C.c_void_p)]),
    "cpbus_shard_range": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, _P(C.c_uint32), _P(C.c_uint32)]),
    "cpbus_intern": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, _P(C.c_uint32)]),
    "cpbus_source": (C.c_int, [C.c_void_p, C.c_uint32, C.c_char_p, C.c_size_t, _P(C.c_size_t)]),
    "cpbus_intern_ephemeral": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t, _P(C.c_uint32)]),
    "cpbus_subscribe": (C.c_int, [C.c_void_p, C.c_uint32, _P(C.c_uint32)]),
    "cpbus_subscribe_many": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, _P(C.c_uint32)]),
    "cpbus_subscribe_pairs": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, _P(C.c_uint32)]),
    "cpbus_subscribe_pairs_many": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, _P(C.c_uint32)]),
    "cpbus_unsubscribe": (C.c_int, [C.c_void_p, C.c_uint32]),
    "cpbus_set_mask": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "cpbus_timer_add": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32, C.c_int, _P(C.c_uint32)]),
    "cpbus_timer_add_many": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_uint32, C.c_int]),
    "cpbus_timer_cancel": (C.c_int, [C.c_void_p, C.c_uint32]),
    "cpbus_publish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "cpbus_send": (C.c_int, [C.c_void_p, C.c_uint32, _P(Event)]),
    "cpbus_advance": (C.c_int, [C.c_void_p, C.c_uint64]),
    "cpbus_flush": (C.c_int, [C.c_void_p]),
    "cpbus_sync": (C.c_int, [C.c_void_p]),
    "cpbus_publish_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64]),
    "cpbus_publish_device_staged": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p, C.c_size_t]),
    "cpbus_stream_create": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _P(C.c_void_p), C.c_char_p]),
    "cpbus_stream_open": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint32, _P(C.c_void_p)]),
    "cpbus_stream_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, _P(C.c_void_p)]),
    "cpbus_stream_put": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint32]),
    "cpbus_stream_fanout": (C.c_int, [C.c_void_p, C.c_size_t, C.c_uint64]),
    "cpbus_stream_poll": (C.c_int, [C.c_void_p, _P(C.c_int), _P(C.c_size_t), _P(C.c_uint64)]),
    "cpbus_stream_status": (C.c_int, [C.c_void_p]),
    "cpbus_stream_set_timeout": (C.c_int, [C.c_void_p, C.c_uint32]),
    "cpbus_stream_close": (C.c_int, [C.c_void_p]),
    "cpbus_shared_alloc": (C.c_int, [C.c_void_p, C.c_size_t, _P(C.c_void_p), C.c_char_p]),
    "cpbus_shared_open": (C.c_int, [C.c_void_p, C.c_char_p, _P(C.c_void_p)]),
    "cpbus_shared_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cpbus_drain": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, _P(C.c_size_t), _P(C.c_uint64)]),
    "cpbus_drain_many": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, _P(C.c_size_t)]),
    "cpbus_consume_all": (C.c_int, [C.c_void_p]),
    "cpbus_peek_window": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "cpbus_digest": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "cpbus_digest_fold": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _P(C.c_uint64 * 4)]),
    "cpbus_digest_fold_begin": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _P(C.c_uint32)]),
    "cpbus_digest_fold_end": (C.c_int, [C.c_void_p, C.c_uint32, _P(C.c_uint64 * 4)]),
    "cpbus_step_result_begin": (C.c_int, [C.c_void_p, _P(C.c_uint32)]),
    "cpbus_step_result_end": (C.c_int, [C.c_void_p, C.c_uint32, _P(C.c_uint64 * 4)]),
    "cpbus_debug_events": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "cpbus_stats": (C.c_int, [C.c_void_p, _P(Stats)]),
    "cpbus_publish_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "cpbus_device_ptrs": (C.c_int, [C.c_void_p, _P(C.c_void_p), _P(C.c_void_p)]),
    "cpbus_code_name": (C.c_char_p, [C.c_int]),
    "cpbus_code_from_string": (C.c_int, [C.c_char_p]),
    "cpbus_strerror": (C.c_char_p, [C.c_int]),
    "cpbus_last_cuda_error": (C.c_char_p, []),
    "cpbus_abi_version": (C.c_uint32, []),
    "cpbus_split_plan": (C.c_int, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_size_t, _P(C.c_size_t)]),
    "cpbus_mask_order": (C.c_size_t, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]),
    "cpbus_record_hash": (C.c_uint64, [_P(Event)]),
    "cpbus_digest_multiplier": (C.c_uint64, []),
}

_lib = None


class CpbusError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        lib = load()
        msg = lib.cpbus_strerror(status).decode()
        if status == ECUDA:
            msg += ": " + lib.cpbus_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} ({status})")


def load() -> C.CDLL:
    """Load libcpbus.so; fail loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)   # AttributeError if the .so does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(status: int, where: str) -> int:
    if status != OK:
        raise CpbusError(status, where)
    return status
