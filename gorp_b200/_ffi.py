"""ctypes binding of include/gorp_cuda.h. The CUDA library is mandatory: importing this module fails loudly
when libgorpcuda.so is missing (build it with `python -m gorp_b200.build`)."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GORP_LIB") or os.path.join(HERE, "libgorpcuda.so")  # GORP_LIB: A/B runs against another build

if not os.path.exists(LIB_PATH):
    raise ImportError("gorp_b200: %s not found — run `python -m gorp_b200.build` (there is no CPU fallback)" % LIB_PATH)

lib = C.CDLL(LIB_PATH)

GORP_OK, GORP_E_ARG, GORP_E_DEFINITION, GORP_E_UNSUPPORTED, GORP_E_BLOB, GORP_E_CUDA, GORP_E_OOM, GORP_E_INTERNAL = \
    0, -1, -2, -3, -4, -5, -6, -7


class Result(C.Structure):
    _fields_ = [("n_lines", C.c_int64), ("n_extractions", C.c_int32), ("span_stride", C.c_int32),
                ("ext_id", C.POINTER(C.c_int32)), ("line_off", C.POINTER(C.c_int64)),
                ("spans", C.POINTER(C.c_int32)),
                ("histogram", C.POINTER(C.c_int64)), ("owner", C.c_void_p)]


class MatchResult(C.Structure):
    _fields_ = [("n_lines", C.c_int64), ("accept_off", C.POINTER(C.c_int64)), ("accept", C.POINTER(C.c_int32)), ("owner", C.c_void_p)]


class BlobInfo(C.Structure):
    _fields_ = [("n_states", C.c_uint32), ("n_classes", C.c_uint32), ("n_extractions", C.c_uint32),
                ("reserved", C.c_uint32)]


class ExtractionInfo(C.Structure):
    _fields_ = [("n_groups", C.c_uint32), ("n_extractor_names", C.c_uint32),
                ("name", C.POINTER(C.c_uint16)), ("name_len", C.c_uint32),
                ("automaton_regex", C.POINTER(C.c_uint16)), ("automaton_regex_len", C.c_uint32),
                ("jdk_regex", C.POINTER(C.c_uint16)), ("jdk_regex_len", C.c_uint32),
                ("append_json", C.POINTER(C.c_char)), ("append_json_len", C.c_uint32)]


class DeviceResult(C.Structure):
    _fields_ = [("n_lines", C.c_int64), ("span_stride", C.c_int32), ("reserved", C.c_int32),
                ("d_ext_id", C.c_void_p), ("d_line_off", C.c_void_p),
                ("d_spans", C.c_void_p), ("d_histogram", C.c_void_p),
                ("d_n_lines", C.c_void_p)]


class ValueTable(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_columns", C.c_int32), ("reserved", C.c_int32),
                ("d_row", C.c_void_p), ("d_offsets", C.POINTER(C.c_void_p)), ("d_data", C.POINTER(C.c_void_p)),
                ("d_valid", C.POINTER(C.c_void_p)), ("null_count", C.POINTER(C.c_int64))]


class DeviceTables(C.Structure):
    _fields_ = [("n_tables", C.c_int32), ("unit_bytes", C.c_int32), ("tables", C.POINTER(ValueTable))]


# every symbol include/gorp_cuda.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = [
    "gorp_abi_version", "gorp_last_error", "gorp_device_count", "gorp_compile_definition", "gorp_compile_patterns",
    "gorp_blob_free", "gorp_blob_get_info", "gorp_blob_get_extraction", "gorp_blob_get_extractor_name",
    "gorp_blob_get_tables", "gorp_engine_create", "gorp_engine_destroy", "gorp_extract_lines", "gorp_extract_text", "gorp_extract_text_latin1", "gorp_extract_text_utf8", "gorp_extract_text_utf8_bytes", "gorp_extract_lines_utf8", "gorp_match_all_lines", "gorp_match_result_release",
    "gorp_result_release", "gorp_extract_text_device", "gorp_extract_lines_device", "gorp_extract_text_utf8_device",
    "gorp_extract_lines_utf8_device", "gorp_extract_tables_device", "gorp_extract_text_utf8_tables", "gorp_extract_lines_utf8_tables",
    "gorp_kernel_times",
]

lib.gorp_abi_version.restype = C.c_int
lib.gorp_last_error.restype = C.c_char_p
lib.gorp_device_count.restype = C.c_int
lib.gorp_compile_definition.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
lib.gorp_compile_patterns.argtypes = [C.POINTER(C.POINTER(C.c_uint16)), C.POINTER(C.c_uint32), C.c_uint32,
                                      C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
lib.gorp_blob_free.argtypes = [C.c_void_p]
lib.gorp_blob_free.restype = None
lib.gorp_blob_get_info.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(BlobInfo)]
lib.gorp_blob_get_extraction.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.POINTER(ExtractionInfo)]
lib.gorp_blob_get_extractor_name.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint32,
                                             C.POINTER(C.POINTER(C.c_uint16)), C.POINTER(C.c_uint32)]
lib.gorp_blob_get_tables.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.POINTER(C.c_uint16)),
                                     C.POINTER(C.POINTER(C.c_int32)), C.POINTER(C.POINTER(C.c_int32)),
                                     C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.POINTER(C.c_int32))]
lib.gorp_engine_create.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
lib.gorp_engine_destroy.argtypes = [C.c_void_p]
lib.gorp_engine_destroy.restype = None
lib.gorp_extract_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result)]
lib.gorp_extract_text.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result)]
lib.gorp_extract_text_latin1.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result)]
lib.gorp_extract_text_utf8.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result)]
lib.gorp_extract_text_utf8_bytes.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result)]
lib.gorp_extract_lines_utf8.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result)]
lib.gorp_match_all_lines.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(MatchResult)]
lib.gorp_match_result_release.argtypes = [C.c_void_p, C.POINTER(MatchResult)]
lib.gorp_match_result_release.restype = None
lib.gorp_result_release.argtypes = [C.c_void_p, C.POINTER(Result)]
lib.gorp_result_release.restype = None
lib.gorp_extract_text_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                         C.POINTER(DeviceResult)]
lib.gorp_extract_lines_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                          C.POINTER(DeviceResult)]
lib.gorp_extract_text_utf8_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                              C.POINTER(DeviceResult)]
lib.gorp_extract_lines_utf8_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                               C.POINTER(DeviceResult)]
lib.gorp_extract_tables_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(DeviceTables)]
lib.gorp_extract_text_utf8_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result), C.POINTER(DeviceTables)]
lib.gorp_extract_lines_utf8_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(Result), C.POINTER(DeviceTables)]
lib.gorp_kernel_times.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.c_int,
                                  C.POINTER(C.c_int), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int]
FLAG_SYNC, FLAG_TIME_KERNELS = 1, 2


def last_error() -> str:
    return (lib.gorp_last_error() or b"").decode("utf-8", "replace")
