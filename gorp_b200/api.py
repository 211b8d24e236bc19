"""Host-side mirror of the reference's public API for the hot path, over the C ABI (include/gorp_cuda.h).

Same names, argument meaning and error behaviour as salesforce/gorp (gorp-core/src/main/java/com/salesforce/gorp/):
  DefinitionReader.reader(..).read() -> Gorp           DefinitionReader.java:51-84
  Gorp.extract / extractSafe / extractAll              Gorp.java:145-186 (+ the new batch entry point)
  Gorp.getExtractions() / CookedExtraction             Gorp.java:131, model/CookedExtraction.java:18-66
  ExtractionResult.getId/getInput/asMap                ExtractionResult.java:39-88
  DefinitionParseException / ExtractionException       DefinitionParseException.java:17, ExtractionException.java:15

Every extract goes through libgorpcuda on the GPU; there is no CPU path. A host without a CUDA device can still
compile definitions (DefinitionReader.read) and inspect the exported tables, but any extract raises GorpCudaError.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np

from . import _ffi
from ._ffi import lib

MISS = -1


class DefinitionParseException(IOError):
    pass


class UnsupportedDefinition(DefinitionParseException):
    """Definition is valid for reference gorp but uses a construct the GPU path refuses (see DESIGN.md)."""


class ExtractionException(IOError):
    def __init__(self, input_, msg):
        super().__init__(msg)
        self.input = input_

    def getInput(self):
        return self.input


class GorpCudaError(RuntimeError):
    pass


def _check(rc):
    if rc == 0:
        return
    msg = _ffi.last_error()
    if rc == _ffi.GORP_E_DEFINITION:
        raise DefinitionParseException(msg)
    if rc == _ffi.GORP_E_UNSUPPORTED:
        raise UnsupportedDefinition(msg)
    if rc == _ffi.GORP_E_ARG:
        raise ValueError(msg)
    raise GorpCudaError("libgorpcuda error %d: %s" % (rc, msg))


def _u16(ptr, n):
    return bytes(C.cast(ptr, C.POINTER(C.c_uint8 * (2 * n))).contents).decode("utf-16-le", "surrogatepass") if n else ""


def to_units(s) -> np.ndarray:
    """Java String -> UTF-16 code units."""
    if isinstance(s, np.ndarray):
        return s.astype(np.uint16, copy=False)
    return np.frombuffer(s.encode("utf-16-le", "surrogatepass"), dtype="<u2")


class Blob:
    """A DfaExport blob (owned copy of the native allocation)."""

    def __init__(self, ptr, length):
        self._ptr, self.length = ptr, length

    @classmethod
    def from_definition(cls, text: str):
        data = text.encode("utf-8", "surrogatepass")
        p, n = C.c_void_p(), C.c_size_t()
        _check(lib.gorp_compile_definition(data, len(data), C.byref(p), C.byref(n)))
        return cls(p, n.value)

    @classmethod
    def from_patterns(cls, patterns):
        arrs = [to_units(p).copy() for p in patterns]
        ptrs = (C.POINTER(C.c_uint16) * len(arrs))(*[a.ctypes.data_as(C.POINTER(C.c_uint16)) for a in arrs])
        lens = (C.c_uint32 * len(arrs))(*[len(a) for a in arrs])
        p, n = C.c_void_p(), C.c_size_t()
        _check(lib.gorp_compile_patterns(ptrs, lens, len(arrs), C.byref(p), C.byref(n)))
        return cls(p, n.value)

    def bytes(self) -> bytes:
        return C.string_at(self._ptr, self.length)

    def info(self):
        bi = _ffi.BlobInfo()
        _check(lib.gorp_blob_get_info(self._ptr, self.length, C.byref(bi)))
        return bi.n_states, bi.n_classes, bi.n_extractions

    def extraction(self, i):
        xi = _ffi.ExtractionInfo()
        _check(lib.gorp_blob_get_extraction(self._ptr, self.length, i, C.byref(xi)))
        names = []
        for k in range(xi.n_extractor_names):
            p, n = C.POINTER(C.c_uint16)(), C.c_uint32()
            _check(lib.gorp_blob_get_extractor_name(self._ptr, self.length, i, k, C.byref(p), C.byref(n)))
            names.append(_u16(p, n.value))
        raw = C.string_at(xi.append_json, xi.append_json_len).decode("utf-8") if xi.append_json_len else ""
        extra = None
        for part in raw.split("\n") if raw else []:
            try:
                obj = json.loads(part)
            except ValueError as e:
                raise DefinitionParseException("Invalid JSON content to 'append': %s" % e)
            if not isinstance(obj, dict):
                raise DefinitionParseException("Invalid 'append' value: must be JSON Object, or sequence of key/value pairs")
            extra = obj if extra is None else {**extra, **obj}
        return {"n_groups": xi.n_groups, "name": _u16(xi.name, xi.name_len),
                "automaton_regex": _u16(xi.automaton_regex, xi.automaton_regex_len),
                "jdk_regex": _u16(xi.jdk_regex, xi.jdk_regex_len), "extractor_names": names, "extra": extra}

    def tables(self):
        """(classmap u16[65536], transitions i32[S,C], accept_first i32[S], accept lists) — Automata's arrays."""
        S, Cn, _ = self.info()
        cm, tr, af = C.POINTER(C.c_uint16)(), C.POINTER(C.c_int32)(), C.POINTER(C.c_int32)()
        ao, al = C.POINTER(C.c_uint32)(), C.POINTER(C.c_int32)()
        _check(lib.gorp_blob_get_tables(self._ptr, self.length, C.byref(cm), C.byref(tr), C.byref(af), C.byref(ao), C.byref(al)))
        classmap = np.ctypeslib.as_array(cm, (65536,)).copy()
        trans = np.ctypeslib.as_array(tr, (S * Cn,)).copy().reshape(S, Cn)
        first = np.ctypeslib.as_array(af, (S,)).copy()
        off = np.ctypeslib.as_array(ao, (S + 1,)).copy()
        lst = np.ctypeslib.as_array(al, (max(int(off[-1]), 1),)).copy()[:int(off[-1])]
        return classmap, trans, first, [lst[off[s]:off[s + 1]].tolist() for s in range(S)]

    def __del__(self):
        if getattr(self, "_ptr", None):
            lib.gorp_blob_free(self._ptr)
            self._ptr = None


class CookedExtraction:
    def __init__(self, index, d):
        self._index, self._name = index, d["name"]
        self._regexp_source, self._automaton_source = d["jdk_regex"], d["automaton_regex"]
        self._extractor_names, self._append = d["extractor_names"], d["extra"]

    def getName(self):
        return self._name

    def getExtra(self):
        return self._append

    def getRegexpSource(self):
        return self._regexp_source

    def getRegexpDesc(self):
        return self._regexp_source

    def getExtractorNames(self):
        return list(self._extractor_names)

    def constructMatch(self, input_, values):
        return ExtractionResult(self._name, input_, self, self._extractor_names, values)


class ExtractionResult:
    def __init__(self, id_, input_, extr, names, values):
        self._id, self._input, self._matched, self._names, self._values = id_, input_, extr, names, values

    def getId(self):
        return self._id

    def getInput(self):
        return self._input

    def getMatchedExtraction(self):
        return self._matched

    def getExtra(self):
        return self._matched.getExtra()

    def asMap(self, idAs=None):
        out = {}
        if idAs is not None:
            out[idAs] = self._id
        for n, v in zip(self._names, self._values):
            out[n] = v
        extra = self.getExtra()
        if extra is not None:
            out.update(extra)
        return out


def _host_array(ptr, n, dtype):
    """numpy copy of n elements at host address ptr."""
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(np.ctypeslib.as_ctypes_type(dtype))), (n,)).copy()


class ValueColumn:
    """One extractor name of a ValueTable in Arrow large_string layout: value r is data[offsets[r]:offsets[r + 1]] (UTF-8),
    null where bit r of `valid` (LSB first) is 0."""

    def __init__(self, offsets, data, valid, null_count):
        self.offsets, self.data, self.valid, self.null_count = offsets, data, valid, null_count


class ValueTable:
    """What ExtractionResult.asMap() gives for the lines of one extraction, as columns: `rows` (int64) are the indexes of
    those lines in the batch, ascending; `columns` maps each extractor name to a ValueColumn."""

    def __init__(self, name, rows, columns):
        self.name, self.rows, self.columns = name, rows, columns

    @property
    def n_rows(self):
        return len(self.rows)

    def to_arrow(self):
        """A pyarrow.Table of large_string columns over this table's buffers (no copy). An extraction without groups gives
        a table without columns."""
        import pyarrow as pa
        n = len(self.rows)
        arrays = [pa.LargeStringArray.from_buffers(n, pa.py_buffer(c.offsets), pa.py_buffer(c.data), pa.py_buffer(c.valid), c.null_count)
                  for c in self.columns.values()]
        return pa.Table.from_arrays(arrays, names=list(self.columns))


def _value_tables(gorp, dt: _ffi.DeviceTables):
    """numpy copies of the host tables of a gorp_extract_*_utf8_tables call."""
    out = []
    for e in range(dt.n_tables):
        t = dt.tables[e]
        n = int(t.n_rows)
        x = gorp._extractions[e]
        cols = {}
        for k, name in enumerate(x.getExtractorNames()[:t.n_columns]):
            off = _host_array(t.d_offsets[k], n + 1, np.int64)
            cols[name] = ValueColumn(off, _host_array(t.d_data[k], int(off[-1]), np.uint8), _host_array(t.d_valid[k], (n + 7) // 8, np.uint8),
                                     int(t.null_count[k]))
        out.append(ValueTable(x.getName(), _host_array(t.d_row, n, np.int64), cols))
    return out


class ExtractionBatch:
    """Columnar result of one batch call: numpy copies of the gorp_result arrays + lazy ExtractionResult views.
    `units` is the text the offsets index, in `encoding`: UTF-16 units, or the caller's UTF-8 bytes (byte coordinates);
    a line or a value is decoded from its own slice only. `tables` (the UTF-8 calls with tables=True, else None): one
    ValueTable per extraction."""

    def __init__(self, gorp, units, res: _ffi.Result, sep, encoding="utf-16-le", tables=None):
        n = res.n_lines
        self.gorp, self.units, self.sep, self.n_lines, self.encoding = gorp, units, sep, n, encoding
        self.tables = None if tables is None else _value_tables(gorp, tables)
        self.ext_id = np.ctypeslib.as_array(res.ext_id, (max(n, 1),))[:n].copy()
        self.line_off = np.ctypeslib.as_array(res.line_off, (n + 1,)).copy()
        self.span_stride = w = int(res.span_stride)
        # one fixed-size row of (start, end) pairs per line; entries beyond 2 * groups(ext_id) are -1
        self.spans = np.ctypeslib.as_array(res.spans, (max(n * w, 1),))[:n * w].copy().reshape(n, w)
        self.histogram = np.ctypeslib.as_array(res.histogram, (res.n_extractions + 2,)).copy()

    def __len__(self):
        return self.n_lines

    def line(self, i) -> str:
        a, b = int(self.line_off[i]), int(self.line_off[i + 1]) - self.sep
        return self.units[a:b].tobytes().decode(self.encoding, "surrogatepass")

    def spans_of(self, i):
        e = int(self.ext_id[i])
        if e < 0:
            return []
        s = self.spans[i, :2 * len(self.gorp._extractions[e].getExtractorNames())]
        return list(zip(s[0::2].tolist(), s[1::2].tolist()))

    def result(self, i, safe=False):
        """What Gorp.extract(line i) returns / throws."""
        e = int(self.ext_id[i])
        if e == MISS:
            return None
        if e < 0:
            if safe:
                return None  # extractSafe: the fallback loop retries the same extraction (Gorp.java:178-185)
            x = self.gorp._extractions[-2 - e]
            raise ExtractionException(self.line(i),
                                      "Internal error: high-level match for extraction #%d (%s) failed to match generated regexp: %s"
                                      % (-2 - e, x.getName(), x.getRegexpDesc()))
        x = self.gorp._extractions[e]
        a = int(self.line_off[i])
        vals = []
        for (s, t) in self.spans_of(i):
            vals.append(None if s < 0 else self.units[a + s:a + t].tobytes().decode(self.encoding, "surrogatepass"))
        return x.constructMatch(self.line(i), vals)

    def results(self, safe=False):
        return [self.result(i, safe) for i in range(self.n_lines)]


class Gorp:
    def __init__(self, blob: Blob, devices=None):
        self._blob = blob
        _, _, n = blob.info()
        self._extractions = [CookedExtraction(i, blob.extraction(i)) for i in range(n)]
        self._devices = devices
        self._engine = None

    # -- reference accessors
    def getExtractions(self):
        return list(self._extractions)

    def blob(self):
        return self._blob

    def _eng(self):
        if self._engine is None:
            h = C.c_void_p()
            if self._devices:
                arr = (C.c_int * len(self._devices))(*self._devices)
                _check(lib.gorp_engine_create(self._blob._ptr, self._blob.length, arr, len(self._devices), C.byref(h)))
            else:
                _check(lib.gorp_engine_create(self._blob._ptr, self._blob.length, None, 0, C.byref(h)))
            self._engine = h
        return self._engine

    # -- batch entry points (the new API)
    def extractAll(self, lines, safe=False):
        """Gorp.extractAll(List<String>) -> list of ExtractionResult | None; raises ExtractionException at the
        first capture failure unless safe (mirrors extract / extractSafe per line)."""
        return self.extract_batch_lines(lines).results(safe)

    def extract_batch_lines(self, lines) -> ExtractionBatch:
        arrs = [to_units(s) for s in lines]
        off = np.zeros(len(arrs) + 1, dtype=np.int64)
        if arrs:
            np.cumsum([len(a) for a in arrs], out=off[1:])
        units = np.concatenate(arrs) if arrs else np.zeros(0, dtype=np.uint16)
        units = np.ascontiguousarray(units, dtype=np.uint16)
        res = _ffi.Result()
        _check(lib.gorp_extract_lines(self._eng(), units.ctypes.data, off.ctypes.data, len(arrs), C.byref(res)))
        try:
            return ExtractionBatch(self, units, res, 0)
        finally:
            lib.gorp_result_release(self._eng(), C.byref(res))

    def extract_batch_lines_utf8(self, lines, offsets=None, tables=False) -> ExtractionBatch:
        """extract_batch_lines for strings held as UTF-8 bytes (gorp_extract_lines_utf8, all of the engine's devices): a '\\n'
        inside a string is data. `lines` is a sequence of bytes / str (str is UTF-8-encoded), or with `offsets` a bytes-like
        buffer in which string i is bytes [offsets[i], offsets[i+1]) (int64; offsets[0] may be > 0, as in an Arrow slice).
        line_off and spans are byte offsets into that buffer; the batch decodes only what a line(), spans_of() or result()
        asks for. A string that is not well-formed UTF-8 on its own raises ValueError. tables=True: the batch also holds the
        values as one ValueTable per extraction (`.tables`, gorp_extract_lines_utf8_tables)."""
        if offsets is None:
            parts = [s.encode("utf-8") if isinstance(s, str) else bytes(s) for s in lines]
            off = np.zeros(len(parts) + 1, dtype=np.int64)
            if parts:
                np.cumsum([len(p) for p in parts], out=off[1:])
            b = np.frombuffer(b"".join(parts), dtype=np.uint8)
        else:
            b = np.ascontiguousarray(np.frombuffer(lines, dtype=np.uint8) if isinstance(lines, (bytes, bytearray, memoryview)) else lines,
                                     dtype=np.uint8)
            off = np.ascontiguousarray(offsets, dtype=np.int64)
            if off.ndim != 1 or len(off) < 1:
                raise ValueError("offsets must hold n_lines + 1 entries")
            if int(off[-1]) > len(b):
                raise ValueError("offsets reach past the end of the buffer")
        res, dt = _ffi.Result(), _ffi.DeviceTables() if tables else None
        if tables:
            _check(lib.gorp_extract_lines_utf8_tables(self._eng(), b.ctypes.data, off.ctypes.data, len(off) - 1, C.byref(res), C.byref(dt)))
        else:
            _check(lib.gorp_extract_lines_utf8(self._eng(), b.ctypes.data, off.ctypes.data, len(off) - 1, C.byref(res)))
        try:
            return ExtractionBatch(self, b, res, 0, encoding="utf-8", tables=dt)
        finally:
            lib.gorp_result_release(self._eng(), C.byref(res))

    def extract_batch_text(self, text) -> ExtractionBatch:
        """Gorp.extractAll(CharBuffer): '\\n'-separated UTF-16 text (str or uint16 array)."""
        units = np.ascontiguousarray(to_units(text), dtype=np.uint16)
        res = _ffi.Result()
        _check(lib.gorp_extract_text(self._eng(), units.ctypes.data, len(units), C.byref(res)))
        try:
            return ExtractionBatch(self, units, res, 1)
        finally:
            lib.gorp_result_release(self._eng(), C.byref(res))

    def extract_batch_text_latin1(self, data) -> ExtractionBatch:
        """'\n'-separated text held as ISO-8859-1 bytes (bytes or uint8 array), what a JDK 9+ String with the LATIN1 coder
        holds: widened to UTF-16 on the device, results identical to extract_batch_text on the zero-extended text."""
        b = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data, dtype=np.uint8)
        res = _ffi.Result()
        _check(lib.gorp_extract_text_latin1(self._eng(), b.ctypes.data, len(b), C.byref(res)))
        try:
            return ExtractionBatch(self, b.astype(np.uint16), res, 1)
        finally:
            lib.gorp_result_release(self._eng(), C.byref(res))

    def extract_batch_text_utf8(self, data, byte_offsets=False, tables=False) -> ExtractionBatch:
        """'\n'-separated text held as UTF-8 bytes (a log file as it is on disk): decoded to UTF-16 on the device, results are
        those of extract_batch_text on the decoded text (offsets in UTF-16 units). Malformed UTF-8 raises ValueError.
        byte_offsets=True: line_off and spans are byte offsets into `data` (gorp_extract_text_utf8_bytes, all of the engine's
        devices); the batch slices `data` and decodes only what a line(), spans_of() or result() asks for. tables=True (with
        byte_offsets only): the batch also holds the values as one ValueTable per extraction (`.tables`,
        gorp_extract_text_utf8_tables)."""
        if tables and not byte_offsets:
            raise ValueError("tables=True needs byte_offsets=True: the tables hold bytes of `data`")
        b = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data, dtype=np.uint8)
        res = _ffi.Result()
        if byte_offsets:
            dt = _ffi.DeviceTables() if tables else None
            if tables:
                _check(lib.gorp_extract_text_utf8_tables(self._eng(), b.ctypes.data, len(b), C.byref(res), C.byref(dt)))
            else:
                _check(lib.gorp_extract_text_utf8_bytes(self._eng(), b.ctypes.data, len(b), C.byref(res)))
            try:
                return ExtractionBatch(self, b, res, 1, encoding="utf-8", tables=dt)
            finally:
                lib.gorp_result_release(self._eng(), C.byref(res))
        _check(lib.gorp_extract_text_utf8(self._eng(), b.ctypes.data, len(b), C.byref(res)))
        try:
            units = np.frombuffer(b.tobytes().decode("utf-8").encode("utf-16-le"), dtype=np.uint16)
            return ExtractionBatch(self, units, res, 1)
        finally:
            lib.gorp_result_release(self._eng(), C.byref(res))

    def match_all(self, lines):
        """PolyMatcher.match for a batch (Gorp.getMatcher().match(s) per string): list of ascending index lists."""
        arrs = [to_units(s) for s in lines]
        off = np.zeros(len(arrs) + 1, dtype=np.int64)
        if arrs:
            np.cumsum([len(a) for a in arrs], out=off[1:])
        units = np.ascontiguousarray(np.concatenate(arrs) if arrs else np.zeros(0, dtype=np.uint16), dtype=np.uint16)
        res = _ffi.MatchResult()
        _check(lib.gorp_match_all_lines(self._eng(), units.ctypes.data, off.ctypes.data, len(arrs), C.byref(res)))
        try:
            n = res.n_lines
            aoff = np.ctypeslib.as_array(res.accept_off, (n + 1,)).copy()
            acc = np.ctypeslib.as_array(res.accept, (max(int(aoff[-1]), 1),))[:int(aoff[-1])].copy()
            return [acc[aoff[i]:aoff[i + 1]].tolist() for i in range(n)]
        finally:
            lib.gorp_match_result_release(self._eng(), C.byref(res))

    # -- per-line API of the reference, served by a batch of one
    def extract(self, input_: str):
        return self.extract_batch_lines([input_]).result(0, safe=False)

    def extractSafe(self, input_: str):
        return self.extract_batch_lines([input_]).result(0, safe=True)

    def close(self):
        if self._engine is not None:
            lib.gorp_engine_destroy(self._engine)
            self._engine = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class DefinitionReader:
    def __init__(self, contents: str):
        self._contents = contents

    @staticmethod
    def reader(src):
        """reader(File) / reader(String) of the reference: a path to an existing file or the definition text."""
        if isinstance(src, (bytes, os.PathLike)) or (isinstance(src, str) and "\n" not in src and os.path.isfile(src)):
            with open(src, "rb") as f:
                return DefinitionReader(f.read().decode("utf-8", "replace"))
        return DefinitionReader(src)

    def read(self, devices=None) -> Gorp:
        return Gorp(Blob.from_definition(self._contents), devices)
