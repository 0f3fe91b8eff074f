"""ctypes binding of include/etl_decode.h (libetl_decode.so).

This is the same binding a Rust / cgo / JNI shim would write (see INTEGRATION.md): plain pointers
and sizes, no torch types.  The library is built in-tree by etl_b200.build (nvcc, sm_100a) and the
import fails loudly if it is missing — there is no CPU fallback for the decode path.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

u8p, u32p, u64p, i32p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)


class ColumnSchema(C.Structure):
    _fields_ = [("name", C.c_char_p), ("type_oid", C.c_uint32), ("modifier", C.c_int32),
                ("ordinal_position", C.c_int32), ("primary_key_ordinal_position", C.c_int32),
                ("nullable", C.c_uint8), ("_pad", C.c_uint8 * 7)]


class StreamState(C.Structure):
    _fields_ = [("final_lsn", C.c_uint64), ("next_tx_ordinal", C.c_uint64), ("in_tx", C.c_uint8), ("_pad", C.c_uint8 * 7)]


class FirstError(C.Structure):
    _fields_ = [("record_index", C.c_uint64), ("seq", C.c_uint32), ("code", C.c_uint32), ("kind", C.c_uint32), ("_pad", C.c_uint32)]


class DecInput(C.Structure):
    _fields_ = [("host_buf", C.c_void_p), ("dev_buf", C.c_void_p), ("len", C.c_uint64), ("anchors", C.c_void_p),
                ("dev_anchors", C.c_void_p), ("n_anchors", C.c_uint64), ("anchor_stride", C.c_uint32), ("max_frame_len", C.c_uint32),
                ("relation_offsets", C.c_void_p), ("n_relations", C.c_uint64), ("carry_in", StreamState)]


class Seam(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_cells", C.c_uint64), ("heap_bytes", C.c_uint64), ("lsn", C.c_uint64),
                ("ord", C.c_uint64), ("has_begin", C.c_uint8), ("closed", C.c_uint8), ("_pad", C.c_uint8 * 6)]


class CopyInput(C.Structure):
    _fields_ = [("host_buf", C.c_void_p), ("dev_buf", C.c_void_p), ("len", C.c_uint64), ("row_offsets", C.c_void_p),
                ("dev_row_offsets", C.c_void_p), ("n_rows", C.c_uint64)]


HOST_ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64)


class ArrowColumn(C.Structure):
    _fields_ = [("arrow_type", C.c_uint32), ("_pad", C.c_uint32), ("validity", C.c_void_p), ("values", C.c_void_p),
                ("offsets", C.c_void_p), ("data", C.c_void_p), ("data_bytes", C.c_uint64)]


class Planes(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_cells", C.c_uint64), ("heap_bytes", C.c_uint64),
                ("rec_off", C.c_void_p), ("rec_kind", C.c_void_p), ("rec_flags", C.c_void_p), ("rec_rel", C.c_void_p),
                ("rec_schema", C.c_void_p), ("rec_start_lsn", C.c_void_p), ("rec_commit_lsn", C.c_void_p),
                ("rec_tx_ordinal", C.c_void_p), ("rec_cell_base", C.c_void_p), ("rec_tuple_bytes", C.c_void_p),
                ("rec_heap_hint", C.c_void_p), ("cell_tag", C.c_void_p),
                ("cell_val", C.c_void_p), ("cell_aux", C.c_void_p), ("heap", C.c_void_p)]


class Summary(C.Structure):
    _fields_ = [("first_error", FirstError), ("carry_out", StreamState), ("insert_bytes", C.c_uint64),
                ("update_bytes", C.c_uint64), ("delete_bytes", C.c_uint64), ("n_events", C.c_uint64),
                ("n_schemas", C.c_uint32), ("gpu_launches", C.c_uint32), ("kernel_ms", C.c_float),
                ("h2d_ms", C.c_float), ("d2h_ms", C.c_float), ("index_ms", C.c_float),
                ("emit_ms", C.c_float), ("frames_ms", C.c_float), ("walk_ms", C.c_float), ("spans_ms", C.c_float), ("cells_ms", C.c_float), ("long_ms", C.c_float), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("span_bytes", C.c_uint64),
                ("record_index_base", C.c_uint64), ("abi_version", C.c_uint32), ("_pad2", C.c_uint32)]


class SchemaInfo(C.Structure):
    _fields_ = [("table_id", C.c_uint32), ("n_cols", C.c_uint32), ("n_identity", C.c_uint32), ("_pad", C.c_uint32),
                ("snapshot_id", C.c_uint64), ("effective_off", C.c_uint64), ("col_kind", u8p), ("col_flags", u8p),
                ("col_index", i32p)]


# every symbol include/etl_decode.h declares (tests check the library exports all of them)
EXPORTS = [
    "etl_dec_abi_version", "etl_stage_create", "etl_stage_destroy", "etl_stage_reset", "etl_stage_append",
    "etl_stage_append_framed", "etl_stage_view", "etl_dec_create", "etl_dec_set_stream", "etl_dec_destroy",
    "etl_dec_last_error", "etl_dec_put_table_schema", "etl_dec_reset_relations", "etl_dec_decode",
    "etl_dec_decode_begin", "etl_dec_decode_finish", "etl_dec_batch_free", "etl_dec_batch_planes",
    "etl_dec_batch_summary", "etl_dec_batch_schema", "etl_dec_decode_sharded", "etl_dec_comm_unique_id", "etl_dec_comm_init", "etl_dec_comm_init_host",
    "etl_dec_kind_for_type_oid", "etl_dec_mem_info",
    "etl_dec_copy_decode", "etl_dec_arrow_emit", "etl_dec_arrow_emit_ex", "etl_dec_arrow_rows", "etl_dec_arrow_cols",
    "etl_dec_arrow_row_records", "etl_dec_arrow_column", "etl_dec_arrow_list_values", "etl_dec_arrow_free", "etl_dec_batch_device_stream", "etl_shim_materialise", "etl_shim_event_count", "etl_shim_size_hint", "etl_shim_total_size_hint", "etl_shim_owned_bytes",
    "etl_shim_json_text", "etl_shim_event_list_free",
]

_lib = None


def lib_path() -> str:
    return _build.DECODE_LIB


def load(build: bool = True):
    """Load libetl_decode.so (building it first if the sources are newer). Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    # an existing in-tree library is loaded as is (the GPU box receives the prebuilt .so; file times are
    # not preserved by the snapshot, so no staleness check here — `python -m etl_b200.build` rebuilds)
    path = _build.DECODE_LIB
    if build and not os.path.exists(path):
        path = _build.build_decode()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: the CUDA decode library must be built (python -m etl_b200.build)")
    L = C.CDLL(path)
    vp = C.c_void_p
    L.etl_dec_abi_version.restype = C.c_uint32
    L.etl_stage_create.argtypes = [C.c_uint64, C.c_uint32, C.POINTER(vp)]
    L.etl_stage_destroy.argtypes = [vp]
    L.etl_stage_destroy.restype = None
    L.etl_stage_reset.argtypes = [vp]
    L.etl_stage_reset.restype = None
    L.etl_stage_append.argtypes = [vp, vp, C.c_uint32]
    L.etl_stage_append_framed.argtypes = [vp, vp, C.c_uint64]
    L.etl_stage_view.argtypes = [vp, C.POINTER(DecInput)]
    L.etl_dec_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.etl_dec_set_stream.argtypes = [vp, vp]
    L.etl_dec_destroy.argtypes = [vp]
    L.etl_dec_destroy.restype = None
    L.etl_dec_last_error.argtypes = [vp]
    L.etl_dec_last_error.restype = C.c_char_p
    L.etl_dec_put_table_schema.argtypes = [vp, C.c_uint32, C.c_uint64, C.POINTER(ColumnSchema), C.c_uint32]
    L.etl_dec_reset_relations.argtypes = [vp]
    L.etl_dec_decode.argtypes = [vp, C.POINTER(DecInput), C.c_uint32, C.POINTER(vp)]
    L.etl_dec_decode_begin.argtypes = [vp, C.POINTER(DecInput), C.c_uint32, C.POINTER(Seam)]
    L.etl_dec_decode_finish.argtypes = [vp, C.POINTER(StreamState), C.c_uint64, C.POINTER(vp)]
    L.etl_dec_batch_free.argtypes = [vp]
    L.etl_dec_batch_free.restype = None
    L.etl_dec_batch_planes.argtypes = [vp, C.c_int, C.POINTER(Planes)]
    L.etl_dec_batch_summary.argtypes = [vp, C.POINTER(Summary)]
    L.etl_dec_batch_schema.argtypes = [vp, C.c_uint32, C.POINTER(SchemaInfo)]
    L.etl_dec_decode_sharded.argtypes = [vp, C.POINTER(DecInput), C.c_uint32, C.POINTER(vp)]
    L.etl_dec_comm_unique_id.argtypes = [vp, C.c_uint32]
    L.etl_dec_comm_init.argtypes = [vp, vp, C.c_uint32, C.c_int, C.c_int]
    L.etl_dec_comm_init_host.argtypes = [vp, C.c_int, C.c_int, HOST_ALLGATHER_FN, vp]
    L.etl_dec_kind_for_type_oid.argtypes = [C.c_uint32]
    L.etl_dec_kind_for_type_oid.restype = C.c_uint32
    L.etl_dec_mem_info.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.etl_dec_copy_decode.argtypes = [vp, C.c_uint32, C.POINTER(CopyInput), C.c_uint32, C.POINTER(vp)]
    L.etl_dec_arrow_emit.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(vp)]
    L.etl_dec_arrow_emit_ex.argtypes = [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(vp)]
    L.etl_dec_arrow_rows.argtypes = [vp]
    L.etl_dec_arrow_rows.restype = C.c_uint64
    L.etl_dec_arrow_cols.argtypes = [vp]
    L.etl_dec_arrow_cols.restype = C.c_uint32
    L.etl_dec_arrow_row_records.argtypes = [vp, C.c_int]
    L.etl_dec_arrow_row_records.restype = C.c_void_p
    L.etl_dec_arrow_column.argtypes = [vp, C.c_uint32, C.c_int, C.POINTER(ArrowColumn)]
    L.etl_dec_arrow_list_values.argtypes = [vp, C.c_uint32, C.c_int, C.POINTER(ArrowColumn), C.POINTER(C.c_uint64)]
    L.etl_dec_arrow_free.argtypes = [vp]
    L.etl_dec_arrow_free.restype = None
    L.etl_dec_batch_device_stream.argtypes = [vp]
    L.etl_dec_batch_device_stream.restype = C.c_void_p
    L.etl_shim_materialise.argtypes = [vp, vp, vp, C.POINTER(vp)]
    for f in ("etl_shim_event_count", "etl_shim_total_size_hint", "etl_shim_owned_bytes"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = C.c_uint64
    L.etl_shim_size_hint.argtypes = [vp, C.c_uint64]
    L.etl_shim_size_hint.restype = C.c_uint64
    L.etl_shim_json_text.argtypes = [vp, C.c_uint64, C.c_uint32, C.c_char_p, C.c_uint64]
    L.etl_shim_json_text.restype = C.c_int64
    L.etl_shim_event_list_free.argtypes = [vp]
    L.etl_shim_event_list_free.restype = None
    _lib = L
    return L


RESULTS_TO_HOST = 0x1
NO_TIMING = 0x4

# etl_dec_arrow_emit_ex flags and the Arrow types of etl_arrow_column.arrow_type
ARROW_FORMATTED = 0x1
(ARROW_UNSUPPORTED, ARROW_BOOLEAN, ARROW_INT32, ARROW_INT64, ARROW_FLOAT32, ARROW_FLOAT64, ARROW_UTF8, ARROW_LARGE_BINARY,
 ARROW_DATE32, ARROW_TIME64_US, ARROW_TIMESTAMP_US, ARROW_TIMESTAMPTZ_US, ARROW_UUID, ARROW_LIST) = range(14)
