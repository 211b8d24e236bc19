"""Builds and loads tests/host/hosttest.cpp (test-only CPU interpreter of the product's compiled tables)."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    out = os.path.join(HERE, "_build", "libgorp_hosttest.so")
    srcs = [os.path.join(HERE, "host", "hosttest.cpp")] + sorted(glob.glob(os.path.join(ROOT, "gorp_b200/csrc/host/*.cpp")))
    deps = srcs + glob.glob(os.path.join(ROOT, "gorp_b200/csrc/host/*.hpp"))
    if not os.path.exists(out) or any(os.path.getmtime(s) > os.path.getmtime(out) for s in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-o", out] + srcs)
    _lib = C.CDLL(out)
    return _lib


def run(blob_bytes: bytes, text: np.ndarray, starts: np.ndarray, ends: np.ndarray, stride: int, fused: bool = False):
    """fused=True interprets the one-pass automaton (host/fused.hpp); returns None for ext when it is not available."""
    lib = load()
    text = np.ascontiguousarray(text, dtype=np.uint16)
    starts = np.ascontiguousarray(starts, dtype=np.int64)
    ends = np.ascontiguousarray(ends, dtype=np.int64)
    n = len(starts)
    ext = np.empty(n, dtype=np.int32)
    spans = np.full((n, max(stride, 1)), -1, dtype=np.int32)
    stats = np.zeros(8, dtype=np.uint32)
    err = C.create_string_buffer(1024)
    P = C.c_void_p
    fn = lib.ht_run_fused if fused else lib.ht_run
    rc = fn(blob_bytes, C.c_size_t(len(blob_bytes)), P(text.ctypes.data), P(starts.ctypes.data), P(ends.ctypes.data),
                    C.c_int64(n), P(ext.ctypes.data), P(spans.ctypes.data), C.c_int(max(stride, 1)), P(stats.ctypes.data), err,
                    C.c_int(1024))
    if rc == 1 and fused:
        return None, err.value.decode(), stats
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return ext, spans[:, :stride], stats


def run_fused_tail(blob_bytes: bytes, text: np.ndarray, starts: np.ndarray, ends: np.ndarray, stride: int):
    """Interprets the fused walk's table (the one-pass automaton as one tail image) the way kernels/tailwalk.cu walks it in
    "all" mode. Returns (ext, spans) or None when the definition gets no one-pass automaton / it exceeds the image limits."""
    lib = load()
    text = np.ascontiguousarray(text, dtype=np.uint16)
    starts = np.ascontiguousarray(starts, dtype=np.int64)
    ends = np.ascontiguousarray(ends, dtype=np.int64)
    n = len(starts)
    ext = np.empty(n, dtype=np.int32)
    spans = np.full((n, max(stride, 1)), -1, dtype=np.int32)
    err = C.create_string_buffer(1024)
    P = C.c_void_p
    rc = lib.ht_run_fused_tail(blob_bytes, C.c_size_t(len(blob_bytes)), P(text.ctypes.data), P(starts.ctypes.data), P(ends.ctypes.data),
                               C.c_int64(n), P(ext.ctypes.data), P(spans.ctypes.data), C.c_int(max(stride, 1)), err, C.c_int(1024))
    if rc == 1:
        return None
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return ext, spans[:, :stride]


def run_walk(blob_bytes: bytes, text: np.ndarray, stride: int, smem_variant: bool):
    """Interprets the tables of the big-definition text path (host/walktables.hpp) the way kernels/dfawalk.cu and
    kernels/capwalk.cu walk them. Returns (ext, spans) or None when the tables are not available."""
    lib = load()
    text = np.ascontiguousarray(text, dtype=np.uint16)
    cap = int((text == 10).sum()) + 2
    ext = np.empty(cap, dtype=np.int32)
    spans = np.full((cap, max(stride, 1)), -1, dtype=np.int32)
    err = C.create_string_buffer(1024)
    P = C.c_void_p
    lib.ht_run_walk.restype = C.c_int64
    n = lib.ht_run_walk(blob_bytes, C.c_size_t(len(blob_bytes)), P(text.ctypes.data), C.c_int64(len(text)), C.c_int(1 if smem_variant else 0),
                        C.c_int64(cap), P(ext.ctypes.data), P(spans.ctypes.data), C.c_int(max(stride, 1)), err, C.c_int(1024))
    if n == -2:
        return None
    if n < 0:
        raise RuntimeError(err.value.decode())
    return ext[:n], spans[:n, :stride]


def run_tails(blob_bytes: bytes, text: np.ndarray, stride: int):
    """Interprets the early-exit DFA table + tail automata (host/tails.hpp) the way kernels/dfawalk.cu (K2b) and
    kernels/tailwalk.cu walk them. Returns (ext, spans, stats) or None when the definition gets no tails."""
    lib = load()
    text = np.ascontiguousarray(text, dtype=np.uint16)
    cap = int((text == 10).sum()) + 2
    ext = np.empty(cap, dtype=np.int32)
    spans = np.full((cap, max(stride, 1)), -1, dtype=np.int32)
    stats = np.zeros(4, dtype=np.uint64)
    err = C.create_string_buffer(1024)
    P = C.c_void_p
    lib.ht_run_tails.restype = C.c_int64
    n = lib.ht_run_tails(blob_bytes, C.c_size_t(len(blob_bytes)), P(text.ctypes.data), C.c_int64(len(text)), C.c_int64(cap),
                         P(ext.ctypes.data), P(spans.ctypes.data), C.c_int(max(stride, 1)), P(stats.ctypes.data), err, C.c_int(1024))
    if n == -2:
        return None
    if n < 0:
        raise RuntimeError(err.value.decode())
    return ext[:n], spans[:n, :stride], stats


LAYOUT_FIELDS = ("max_regs", "stride", "fused", "fused_slots", "fused_outcomes", "fused_multi", "fused_image", "fused_table_bytes",
                 "capimg", "cap_fast", "tails", "pike")


def layout(blob_bytes: bytes):
    """Which side of each table limit a definition lands on (tests/host/hosttest.cpp: ht_layout): a dict of LAYOUT_FIELDS
    and "tail", the per-extraction availability of the tail image."""
    lib = load()
    out = np.zeros(len(LAYOUT_FIELDS), dtype=np.uint32)
    tail = np.zeros(4096, dtype=np.uint8)
    err = C.create_string_buffer(1024)
    P = C.c_void_p
    n = lib.ht_layout(blob_bytes, C.c_size_t(len(blob_bytes)), P(out.ctypes.data), P(tail.ctypes.data), C.c_int(len(tail)), err, C.c_int(1024))
    if n < 0:
        raise RuntimeError(err.value.decode())
    d = dict(zip(LAYOUT_FIELDS, (int(v) for v in out)))
    d["tail"] = [bool(v) for v in tail[:n]]
    return d
