"""ctypes binding of include/sgr.h (lib/libsgr.so).

The product path has no CPU fallback: if the CUDA library cannot be built or loaded this
module raises, and if no sm_100 device is present sgr_create fails with SGR_ERR_NO_DEVICE.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import build as _build

SGR_OK = 0
ERR_NAMES = {
    -1: "SGR_ERR_INVALID", -2: "SGR_ERR_NO_DEVICE", -3: "SGR_ERR_CUDA", -4: "SGR_ERR_NO_PROGRAM",
    -5: "SGR_ERR_NOT_LOADED", -6: "SGR_ERR_UNSUPPORTED", -7: "SGR_ERR_OOM", -8: "SGR_ERR_STATE",
    -9: "SGR_ERR_DIST", -10: "SGR_ERR_CAPACITY", -11: "SGR_ERR_AGAIN",
}
SGR_ERR_INVALID, SGR_ERR_NO_DEVICE, SGR_ERR_CUDA, SGR_ERR_NO_PROGRAM, SGR_ERR_NOT_LOADED = -1, -2, -3, -4, -5
SGR_ERR_UNSUPPORTED, SGR_ERR_OOM, SGR_ERR_STATE, SGR_ERR_DIST, SGR_ERR_CAPACITY = -6, -7, -8, -9, -10
SGR_ERR_AGAIN = -11

REC_FIXED64, REC_VAR16 = 0, 1
ST_EXISTS, ST_CHANGED, ST_ERROR = 1, 2, 4
MAX_STATE_BYTES, MAX_TYPES, MAX_OPS = 128, 16, 8
IF_EXISTS, MATERIALISE, CREATE, TOMBSTONE, THROW = 0, 1, 2, 3, 4
OP_SET, OP_ADD_I32, OP_SUB_I32, OP_ADD_I64, OP_SUB_I64 = 0, 1, 2, 3, 4


class SgrError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {message}")
        self.code = code


class InvalidStateStoreException(SgrError):
    """SGR_ERR_STATE: the store is not readable now (org.apache.kafka.streams.errors.InvalidStateStoreException
    in the reference, passed through as a failed Future by SurgeAggregateStore.scala:31-46)."""


class sgr_op(C.Structure):
    _fields_ = [("opcode", C.c_uint8), ("reserved", C.c_uint8), ("dst_off", C.c_uint16),
                ("src_off", C.c_uint16), ("len", C.c_uint16)]


class sgr_rule(C.Structure):
    _fields_ = [("exists_rule", C.c_uint8), ("n_ops", C.c_uint8), ("reserved", C.c_uint8 * 6),
                ("ops", sgr_op * MAX_OPS)]


class sgr_fold_program(C.Structure):
    _fields_ = [("state_bytes", C.c_uint32), ("record_kind", C.c_uint32), ("n_types", C.c_uint32),
                ("n_f64_fields", C.c_uint32), ("f64_field_off", C.c_uint16 * 8), ("rules", sgr_rule * MAX_TYPES)]


class sgr_config(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_uint32), ("reserved", C.c_uint64 * 6)]


class sgr_dist_stats(C.Structure):
    _fields_ = [("n_sent", C.c_uint64), ("n_sent_remote", C.c_uint64), ("n_recv", C.c_uint64), ("n_local_aggregates", C.c_uint64),
                ("ms_count", C.c_float), ("ms_counts_exchange", C.c_float), ("ms_scatter", C.c_float), ("ms_exchange", C.c_float),
                ("ms_group", C.c_float), ("ms_fold", C.c_float), ("ms_pipeline", C.c_float), ("exchange_record_bytes", C.c_uint32),
                ("reserved", C.c_uint32 * 4)]


class sgr_stats(C.Structure):
    _fields_ = [("n_aggregates", C.c_uint64), ("n_events", C.c_uint64), ("event_bytes", C.c_uint64),
                ("algorithmic_bytes", C.c_uint64), ("n_errors", C.c_uint64), ("n_long_segments", C.c_uint64),
                ("ms_h2d", C.c_float), ("ms_group", C.c_float), ("ms_fold", C.c_float), ("ms_d2h", C.c_float),
                ("fold_launches", C.c_uint32), ("reserved", C.c_uint32 * 7)]


class sgr_ingest_stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_bytes", "n_trailing_bytes", "n_batches", "n_records", "n_markers", "n_null_values",
                                          "n_control_batches", "n_aborted_batches", "n_aborted_records", "n_duplicates", "n_new_keys",
                                          "n_compressed_bytes", "n_decompressed_bytes")] + [("reserved", C.c_uint64 * 3)]


class sgr_json_field(C.Structure):
    _fields_ = [("name", C.c_char_p), ("kind", C.c_uint8), ("reserved", C.c_uint8), ("dst_off", C.c_uint16), ("len", C.c_uint32)]


class sgr_json_event(C.Structure):
    _fields_ = [("type_name", C.c_char_p), ("event_type", C.c_uint32), ("n_fields", C.c_uint32), ("fields", sgr_json_field * 8)]


JSON_I32, JSON_I64, JSON_F64, JSON_UUID, JSON_PSTR = 0, 1, 2, 3, 4
VALUE_PACKED, VALUE_PROTOBUF_EVENT, VALUE_JSON = 0, 1, 2

# every symbol include/sgr.h declares: (name, restype, argtypes)
_P = C.c_void_p
ABI = [
    ("sgr_abi_version", C.c_int32, []),
    ("sgr_create", C.c_int32, [C.POINTER(sgr_config), C.POINTER(_P)]),
    ("sgr_destroy", C.c_int32, [_P]),
    ("sgr_last_error", C.c_char_p, [_P]),
    ("sgr_register_program", C.c_int32, [_P, C.POINTER(sgr_fold_program)]),
    ("sgr_load_events", C.c_int32, [_P, _P, C.c_uint64, _P, C.c_uint64]),
    ("sgr_load_events_device", C.c_int32, [_P, _P, C.c_uint64, _P, C.c_uint64]),
    ("sgr_load_events_indexed", C.c_int32, [_P, _P, C.c_uint64, _P, C.c_uint64, _P, C.c_uint64]),
    ("sgr_load_events_indexed_device", C.c_int32, [_P, _P, C.c_uint64, _P, C.c_uint64, _P, C.c_uint64]),
    ("sgr_load_unsorted", C.c_int32, [_P, _P, C.c_uint64, C.c_uint64]),
    ("sgr_load_unsorted_device", C.c_int32, [_P, _P, C.c_uint64, C.c_uint64]),
    ("sgr_fold_unsorted", C.c_int32, [_P, _P, C.c_uint64, C.c_uint64]),
    ("sgr_fold_unsorted_device", C.c_int32, [_P, _P, C.c_uint64, C.c_uint64]),
    ("sgr_set_initial_states", C.c_int32, [_P, _P, C.c_uint64]),
    ("sgr_fold", C.c_int32, [_P]),
    ("sgr_fold_async", C.c_int32, [_P]),
    ("sgr_wait", C.c_int32, [_P]),
    ("sgr_fold_incremental", C.c_int32, [_P, _P, C.c_uint64]),
    ("sgr_fold_incremental_device", C.c_int32, [_P, _P, C.c_uint64]),
    ("sgr_load_keys", C.c_int32, [_P, _P, _P, C.c_uint64]),
    ("sgr_get", C.c_int32, [_P, _P, C.c_uint32, _P, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]),
    ("sgr_get_index", C.c_int32, [_P, C.c_uint64, _P, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_int32),
                                  C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("sgr_key_index", C.c_int32, [_P, _P, C.c_uint32, C.POINTER(C.c_uint64)]),
    ("sgr_export_states", C.c_int32, [_P, _P, C.c_uint64, _P, _P, _P]),
    ("sgr_states_device", C.c_int32, [_P, C.POINTER(_P), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    ("sgr_events_device", C.c_int32, [_P, C.POINTER(_P), C.POINTER(C.c_uint64), C.POINTER(_P)]),
    ("sgr_get_stats", C.c_int32, [_P, C.POINTER(sgr_stats)]),
    ("sgr_set_option", C.c_int32, [_P, C.c_char_p, C.c_int64]),
    ("sgr_stream", C.c_int32, [_P, C.POINTER(_P)]),
    ("sgr_dist_unique_id", C.c_int32, [_P]),
    ("sgr_dist_init", C.c_int32, [_P, C.c_int32, C.c_int32, _P, C.c_uint64]),
    ("sgr_dist_set_partitions", C.c_int32, [_P, _P, C.c_uint64]),
    ("sgr_dist_ipc_export", C.c_int32, [_P, _P]),
    ("sgr_dist_ipc_import", C.c_int32, [_P, _P]),
    ("sgr_dist_route_and_fold", C.c_int32, [_P, _P, C.c_uint64, C.c_int32]),
    ("sgr_dist_recv_base", C.c_int32, [_P, C.POINTER(C.c_void_p)]),
    ("sgr_dist_set_peers", C.c_int32, [_P, _P]),
    ("sgr_dist_reserve", C.c_int32, [_P, C.c_uint64]),
    ("sgr_states_hash", C.c_int32, [_P, C.POINTER(C.c_uint64)]),
    ("sgr_dist_get_stats", C.c_int32, [_P, C.POINTER(sgr_dist_stats)]),
    ("sgr_dist_local_aggregates", C.c_int32, [_P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("sgr_partitions_for_keys", C.c_int32, [_P, _P, C.c_uint64, C.c_uint32, C.c_int32, _P]),
    ("sgr_string_hash_utf16", C.c_int32, [_P, C.c_uint32]),
    ("sgr_partition_for_key_utf8", C.c_int32, [_P, C.c_uint32, C.c_uint32, C.c_int32, C.POINTER(C.c_int32)]),
    ("sgr_ingest_create", C.c_int32, [C.POINTER(_P)]),
    ("sgr_ingest_destroy", C.c_int32, [_P]),
    ("sgr_ingest_last_error", C.c_char_p, [_P]),
    ("sgr_ingest_set_value_framing", C.c_int32, [_P, C.c_int32]),
    ("sgr_ingest_set_json_packer", C.c_int32, [_P, C.c_char_p, C.POINTER(sgr_json_event), C.c_uint32, C.c_int32]),
    ("sgr_ingest_set_null_value_type", C.c_int32, [_P, C.c_int32]),
    ("sgr_ingest_set_dictionary_limits", C.c_int32, [_P, C.c_uint64, C.c_uint64]),
    ("sgr_ingest_set_aborted", C.c_int32, [_P, C.c_int32, _P, _P, C.c_uint64]),
    ("sgr_ingest_record_batches", C.c_int32, [_P, C.c_int32, _P, C.c_uint64, C.POINTER(sgr_ingest_stats)]),
    ("sgr_ingest_record_batches_mt", C.c_int32, [_P, C.c_uint32, _P, _P, _P, C.c_uint32, _P]),
    ("sgr_ingest_set_allocator", C.c_int32, [_P, _P, _P]),
    ("sgr_ingest_pending", C.c_int32, [_P, C.POINTER(_P), C.POINTER(C.c_uint64)]),
    ("sgr_ingest_keys", C.c_int32, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_uint64)]),
    ("sgr_ingest_mark_folded", C.c_int32, [_P]),
    ("sgr_ingest_offsets", C.c_int32, [_P, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("sgr_ingest_get_stats", C.c_int32, [_P, C.POINTER(sgr_ingest_stats)]),
    ("sgr_append_keys", C.c_int32, [_P, _P, _P, _P, C.c_uint64]),
    ("sgr_dingest_create", C.c_int32, [_P, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]),
    ("sgr_dingest_destroy", C.c_int32, [_P]),
    ("sgr_dingest_last_error", C.c_char_p, [_P]),
    ("sgr_dingest_set_null_value_type", C.c_int32, [_P, C.c_int32]),
    ("sgr_dingest_set_aborted", C.c_int32, [_P, C.c_int32, _P, _P, C.c_uint64]),
    ("sgr_dingest_submit", C.c_int32, [_P, C.c_int32, _P, C.c_uint64, _P]),
    ("sgr_dingest_fold", C.c_int32, [_P, _P]),
    ("sgr_dingest_offsets", C.c_int32, [_P, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("sgr_dingest_reset", C.c_int32, [_P]),
    ("sgr_dingest_last_timing", C.c_int32, [_P, _P]),
    ("sgr_dingest_get_stats", C.c_int32, [_P, _P]),
    ("sgr_grow_states", C.c_int32, [_P, C.c_uint64]),
    ("sgr_fold_ingested", C.c_int32, [_P, _P]),
    ("sgr_crc32c", C.c_uint32, [_P, C.c_uint64]),
    ("sgr_crc32c_portable", C.c_uint32, [_P, C.c_uint64]),
    ("sgr_xxh32", C.c_uint32, [_P, C.c_uint64, C.c_uint32]),
    ("sgr_lz4_frame_decode", C.c_int32, [_P, C.c_uint64, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
]

_lib: Optional[C.CDLL] = None


def library_path() -> str:
    return _build.LIB


def load_library(rebuild: bool = False) -> C.CDLL:
    """Load lib/libsgr.so, building it with nvcc if it is missing or stale. Raises if it cannot."""
    global _lib
    if _lib is not None and not rebuild:
        return _lib
    path = _build.LIB
    if rebuild or not os.path.exists(path):
        path = _build.build(force=rebuild)
    lib = C.CDLL(path)
    for name, restype, argtypes in ABI:
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.sgr_abi_version() != 1:
        raise RuntimeError("libsgr.so ABI version mismatch")
    _lib = lib
    return lib


def check(lib: C.CDLL, handle, rc: int) -> None:
    if rc == SGR_OK:
        return
    msg = lib.sgr_last_error(handle)
    text = msg.decode("utf-8", "replace") if msg else ""
    if rc == SGR_ERR_STATE:
        raise InvalidStateStoreException(rc, text)
    raise SgrError(rc, text)
