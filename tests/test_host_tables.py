"""gorp_extract_text_utf8_tables / gorp_extract_lines_utf8_tables: the UTF-8 host calls that also return the values as one
Arrow-layout table per extraction in pinned host memory.

Every call is held to four things: its rows equal those of the plain call (gorp_extract_text_utf8_bytes /
gorp_extract_lines_utf8) on the same engine and bytes; every table equals a torch reference built on the GPU from those rows
and the caller's bytes (row indexes, offsets, values, bitmaps with their padding, null counts, n_rows == histogram[e],
64-byte alignment); on one device every buffer is byte-identical to gorp_extract_tables_device after the device-resident
UTF-8 call on the same bytes; on a prefix of the lines the values equal the oracle's asMap(). The Python layer's tables,
and their pyarrow form where pyarrow imports, are checked against the same buffers."""
import ctypes as C
import os
import subprocess
import sys
import threading

import numpy as np
import pytest
import torch

from gorp_b200 import Blob, DefinitionReader, Gorp, _ffi, corpus
from oracle import gorp_oracle
from tests import reference_vectors as V
from tests.test_device_forms import make_gorp
from tests.test_table_limits import groups_def, outcomes_def
from tests.test_utf8_byte_offsets import long_lines, mix_lines
from tests.test_utf8_device import placed
from tests.test_utf8_lines import odd_strings, offsets_of
from tests.test_value_tables import _dev, corpus_lines

DEV = torch.device("cuda", 0)
NESTED_DEF = "extract n {\n template $o($i(%{[a-z]+})$j(%{[0-9]*}))=$c(%{\\S+})\n}\n"


# ---------------------------------------------------------------- calls and snapshots
def _host(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(np.ctypeslib.as_ctypes_type(dtype))), (n,)).copy()


def _pad64(n):
    return (n + 63) // 64 * 64


def rows_of(res):
    n, w = int(res.n_lines), int(res.span_stride)
    return {"n": n, "stride": w, "ext": _host(res.ext_id, n, np.int32), "off": _host(res.line_off, n + 1, np.int64),
            "spans": _host(res.spans, n * w, np.int32).reshape(n, w), "hist": _host(res.histogram, res.n_extractions + 2, np.int64)}


def tables_of(dt, fetch=_host):
    """Every buffer of `dt` (bitmaps with their padding to 64 bytes) and its address; `fetch(ptr, n, dtype)` reads memory."""
    out = []
    for e in range(dt.n_tables):
        t = dt.tables[e]
        n = int(t.n_rows)
        cols = []
        for k in range(t.n_columns):
            off = fetch(t.d_offsets[k], n + 1, np.int64)
            cols.append({"off": off, "data": fetch(t.d_data[k], int(off[-1]), np.uint8), "valid": fetch(t.d_valid[k], _pad64((n + 7) // 8), np.uint8),
                         "nulls": int(t.null_count[k]), "ptrs": (int(t.d_offsets[k]), int(t.d_data[k] or 0), int(t.d_valid[k]))})
        out.append({"n": n, "row": fetch(t.d_row, n, np.int64), "row_ptr": int(t.d_row or 0), "cols": cols})
    return out


def _dev_fetch(ptr, n, dtype):
    ts = {np.int64: "<i8", np.uint8: "|u1"}[dtype]
    return _dev(ptr, (n,), ts).cpu().numpy().view(dtype)


def _args(buf, off):
    b = np.frombuffer(bytes(buf), dtype=np.uint8)
    o = None if off is None else np.ascontiguousarray(off, dtype=np.int64)
    return b, o


def plain_call(g, buf, off=None):
    b, o = _args(buf, off)
    res = _ffi.Result()
    if o is None:
        rc = _ffi.lib.gorp_extract_text_utf8_bytes(g._eng(), b.ctypes.data, len(b), C.byref(res))
    else:
        rc = _ffi.lib.gorp_extract_lines_utf8(g._eng(), b.ctypes.data, o.ctypes.data, len(o) - 1, C.byref(res))
    if rc:
        return rc, _ffi.last_error(), None
    try:
        return rc, "", rows_of(res)
    finally:
        _ffi.lib.gorp_result_release(g._eng(), C.byref(res))


def tables_call(g, buf, off=None, keep=False, null_tables=False):
    """(rc, message, rows, tables) of the tables call; the result is released unless `keep` (then also returned)."""
    b, o = _args(buf, off)
    res, dt = _ffi.Result(), _ffi.DeviceTables()
    tp = None if null_tables else C.byref(dt)
    if o is None:
        rc = _ffi.lib.gorp_extract_text_utf8_tables(g._eng(), b.ctypes.data, len(b), C.byref(res), tp)
    else:
        rc = _ffi.lib.gorp_extract_lines_utf8_tables(g._eng(), b.ctypes.data, o.ctypes.data, len(o) - 1, C.byref(res), tp)
    if rc:
        return rc, _ffi.last_error(), None, None
    assert dt.unit_bytes == 1
    snap = (rc, "", rows_of(res), tables_of(dt))
    if keep:
        return snap + (res, dt)
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
    return snap


def device_tables(g, buf, off=None):
    """gorp_extract_tables_device after the device-resident UTF-8 call on the same bytes (one device)."""
    t, ptr = placed(bytes(buf))
    dres = _ffi.DeviceResult()
    st = torch.cuda.current_stream(DEV).cuda_stream
    if off is None:
        rc = _ffi.lib.gorp_extract_text_utf8_device(g._eng(), 0, ptr, len(buf), st, _ffi.FLAG_SYNC, C.byref(dres))
    else:
        d_off = torch.from_numpy(np.ascontiguousarray(off, dtype=np.int64)).to(DEV)
        rc = _ffi.lib.gorp_extract_lines_utf8_device(g._eng(), 0, ptr, d_off.data_ptr(), len(off) - 1, st, _ffi.FLAG_SYNC, C.byref(dres))
    assert rc == 0, _ffi.last_error()
    dt = _ffi.DeviceTables()
    assert _ffi.lib.gorp_extract_tables_device(g._eng(), 0, st, _ffi.FLAG_SYNC, C.byref(dt)) == 0, _ffi.last_error()
    return tables_of(dt, _dev_fetch)


# ---------------------------------------------------------------- checks
def _bits(v):
    n = v.numel()
    pad = torch.zeros((n + 7) // 8 * 8, dtype=torch.int32, device=v.device)
    pad[:n] = v.to(torch.int32)
    return (pad.view(-1, 8) << torch.arange(8, device=v.device, dtype=torch.int32)).sum(dim=1).to(torch.uint8)


def same_rows(a, b):
    assert a["n"] == b["n"] and a["stride"] == b["stride"]
    for k in ("ext", "off", "spans", "hist"):
        assert np.array_equal(a[k], b[k]), k


def same_tables(a, b):
    """Buffer for buffer (contents; not the addresses)."""
    assert len(a) == len(b)
    for e, (x, y) in enumerate(zip(a, b)):
        assert x["n"] == y["n"] and np.array_equal(x["row"], y["row"]) and len(x["cols"]) == len(y["cols"]), e
        for k, (p, q) in enumerate(zip(x["cols"], y["cols"])):
            for f in ("off", "data", "valid"):
                assert np.array_equal(p[f], q[f]), (e, k, f)
            assert p["nulls"] == q["nulls"], (e, k)


def check_reference(g, rows, tabs, buf):
    """Every table against the torch reference over `rows` and the caller's bytes."""
    E = len(g.getExtractions())
    assert len(tabs) == E
    ext = torch.from_numpy(rows["ext"]).to(DEV)
    off = torch.from_numpy(rows["off"]).to(DEV)
    sp = torch.from_numpy(rows["spans"]).to(DEV)
    text = torch.from_numpy(np.frombuffer(bytes(buf), dtype=np.uint8).copy()).to(DEV)
    blob = g.blob()
    for e in range(E):
        t = tabs[e]
        n = t["n"]
        assert n == rows["hist"][e], (e, n)
        assert t["row_ptr"] % 64 == 0 and t["row_ptr"]
        want_rows = torch.nonzero(ext == e).flatten()
        assert np.array_equal(t["row"], want_rows.cpu().numpy()), e
        groups = blob.extraction(e)["n_groups"] if rows["stride"] else 0
        assert len(t["cols"]) == groups
        starts = off[want_rows]
        for k, col in enumerate(t["cols"]):
            assert all(p % 64 == 0 and p for p in col["ptrs"]), (e, k, col["ptrs"])
            s, u = sp[want_rows, 2 * k].to(torch.int64), sp[want_rows, 2 * k + 1].to(torch.int64)
            valid = s >= 0
            ln = torch.where(valid, u - s, 0)
            want_off = torch.zeros(n + 1, dtype=torch.int64, device=DEV)
            torch.cumsum(ln, 0, out=want_off[1:])
            assert np.array_equal(col["off"], want_off.cpu().numpy()), (e, k)
            assert col["nulls"] == int((~valid).sum()), (e, k)
            nbytes = (n + 7) // 8
            assert np.array_equal(col["valid"][:nbytes], _bits(valid).cpu().numpy()), (e, k)
            assert not col["valid"][nbytes:].any(), (e, k)
            total = int(want_off[-1])
            if total:
                src0 = starts + torch.where(valid, s, 0)
                idx = torch.repeat_interleave(src0, ln) + torch.arange(total, device=DEV) - torch.repeat_interleave(want_off[:-1], ln)
                assert np.array_equal(col["data"], text[idx].cpu().numpy()), (e, k)


def check_oracle(definition, rows, tabs, lines):
    """Table e, row r, column k == asMap()[name_k] of line i (None exactly at the nulls) for the given prefix of lines."""
    o = gorp_oracle.Gorp(definition)
    row_of = {}
    for e, t in enumerate(tabs):
        for r, i in enumerate(t["row"].tolist()):
            if i < len(lines):
                row_of[i] = (e, r)
    for i, line in enumerate(lines):
        try:
            want = o.extract_map(line)
        except gorp_oracle.ExtractionError:
            want = None
        if want is None:
            assert i not in row_of and rows["ext"][i] < 0, i
            continue
        e, r = row_of[i]
        got = {}
        for k, nm in enumerate(o.extractions[e].extractor_names):
            col = tabs[e]["cols"][k]
            ok = (col["valid"][r // 8] >> (r % 8)) & 1
            got[nm] = col["data"][col["off"][r]:col["off"][r + 1]].tobytes().decode("utf-8") if ok else None
        assert got == {nm: want[nm] for nm in o.extractions[e].extractor_names}, (i, line[:80])


def check_api(g, buf, off, tabs):
    """The Python layer: ExtractionBatch.tables holds the same buffers; to_arrow() (when pyarrow imports) validates and
    holds the same values."""
    if off is None:
        batch = g.extract_batch_text_utf8(bytes(buf), byte_offsets=True, tables=True)
    else:
        batch = g.extract_batch_lines_utf8(bytes(buf), off, tables=True)
    assert len(batch.tables) == len(tabs)
    try:
        import pyarrow  # noqa: F401
    except ImportError:
        pyarrow = None
    for x, vt in zip(tabs, batch.tables):
        assert np.array_equal(vt.rows, x["row"]) and len(vt.columns) == len(x["cols"])
        n = x["n"]
        for col, vc in zip(x["cols"], vt.columns.values()):
            assert np.array_equal(vc.offsets, col["off"]) and np.array_equal(vc.data, col["data"])
            assert np.array_equal(vc.valid, col["valid"][:(n + 7) // 8]) and vc.null_count == col["nulls"]
        if pyarrow is not None:
            at = vt.to_arrow()
            at.validate(full=True)
            assert at.column_names == list(vt.columns)
            for col, name in zip(x["cols"], vt.columns):
                want = [col["data"][col["off"][r]:col["off"][r + 1]].tobytes().decode("utf-8") if (col["valid"][r // 8] >> (r % 8)) & 1 else None
                        for r in range(n)]
                assert at.column(name).to_pylist() == want, (vt.name, name)
                assert str(at.schema.field(name).type) == "large_string"
    return batch


def check_all(g, buf, off=None, definition=None, oracle_lines=(), device=True, api=True):
    """Every check of the module on one batch (text form when `off` is None). Returns (rows, tables)."""
    rc, msg, plain = plain_call(g, buf, off)
    assert rc == 0, msg
    rc, msg, rows, tabs = tables_call(g, buf, off)
    assert rc == 0, msg
    same_rows(plain, rows)
    check_reference(g, rows, tabs, buf)
    if device:
        same_tables(tabs, device_tables(g, buf, off))
    if oracle_lines:
        check_oracle(definition, rows, tabs, oracle_lines)
    if api:
        check_api(g, buf, off, tabs)
    return rows, tabs


def both_forms(g, definition, lines, oracle_prefix=600, before=b"\xe9abc", **kw):
    """The text form on the lines joined with '\\n', and the lines form on the strings placed `before`-many bytes into the
    buffer (off[0] > 0)."""
    text = "".join(s + "\n" for s in lines).encode("utf-8")
    check_all(g, text, definition=definition, oracle_lines=[s for s in lines[:oracle_prefix]], **kw)
    parts = [s.encode("utf-8") for s in lines]
    check_all(g, before + b"".join(parts), offsets_of(parts) + len(before), definition=definition, oracle_lines=lines[:oracle_prefix], **kw)


# ---------------------------------------------------------------- inputs
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["readme", "weblog", "syslog200", "utf16mix", "simple"])
def test_config_corpora(name, monkeypatch):
    d = corpus.CONFIGS[name][0]
    g = make_gorp(d, monkeypatch)
    n = {"syslog200": 60_000, "utf16mix": 100_000}.get(name, 200_000)
    lines = [s for s in corpus_lines(name, n) if not any(0xD800 <= ord(ch) <= 0xDFFF for ch in s)]
    both_forms(g, d, lines, oracle_prefix=1500)


@pytest.mark.gpu
@pytest.mark.parametrize("definition", [corpus.WEBLOG_DEF, V.README_DEF, NESTED_DEF], ids=["weblog", "readme", "nested"])
def test_line_mix(definition, monkeypatch):
    """Multi-byte values, values of 70 000 bytes and more, '\\r', empty lines; '\\n' inside strings of the lines form."""
    g = make_gorp(definition, monkeypatch)
    lines = mix_lines()[-3000:] + long_lines() + ["", "abc=x\r", "abc12=y\U0001F600", "q=\x0b", "abc=a\x0bb", "=", "1=2"] * 3
    both_forms(g, definition, lines, oracle_prefix=400)
    with_nl = lines[:500] + [s + "\n" + s for s in odd_strings()] + ["abc=x\nz", "[1]: GET 2ms /a\nb"]
    parts = [s.encode("utf-8") for s in with_nl]
    check_all(g, b"".join(parts), offsets_of(parts), definition=definition, oracle_lines=with_nl[:600])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["groups31", "outcomes400", "no_groups", "never_matched", "pike", "match_only"])
def test_definitions(case, monkeypatch):
    """A 31-group extraction; 400 extractions with MISS and CAPTURE_FAIL lines; extractions without groups; extractions
    without rows; the Pike fallback under a forced state limit; a match-only engine (rows, no columns)."""
    rng = np.random.default_rng(9)
    env = {}
    if case == "groups31":
        d = groups_def(31)
        lines = [":".join("".join(rng.choice(list("abcxyz"), size=int(rng.integers(1, 6)))) for _ in range(31)) for _ in range(700)]
        lines += ["a:b", "", "é:" * 30 + "é"]
    elif case == "outcomes400":
        d = outcomes_def(400)
        lines = ["abc=%d" % i for i in rng.permutation(400)] * 3 + ["x=1", "", "abc=400", "zz=399", "abc=a\x0bb"] * 50
    elif case == "no_groups":
        d = "extract e {\n template abc\n}\nextract f {\n template x%{[0-9]+}\n}\nextract g {\n template %{\\S+}\n}\n"
        lines = ["abc", "x12", "y", "", "abc", "a\x0bb"] * 200
    elif case == "never_matched":
        d = ("extract a {\n template never$x(%{[0-9]+})\n}\nextract b {\n template $y(%{[a-z]+})=$z(%{[0-9]+})\n}\n"
             "extract c {\n template zzz$w(%{[a-z]+})\n}\n")
        lines = ["ab=12", "x=1", "", "q"] * 300
    elif case == "pike":
        d = "extract e {\n template " + ":".join("$%s(%%{[ab:]*})" % n for n in "abcdefghi") + "\n}\n"
        env = {"GORP_TDFA_MAX_STATES": "2"}
        lines = ["".join(rng.choice(list("ab:::é"), size=int(rng.integers(0, 40)))) for _ in range(3000)]
    else:
        d = None
        lines = ["[1]: GET 2ms /a", "abc", "", "x12", "é"] * 300
    if d is None:
        g = Gorp(Blob.from_patterns(["\\[[0-9]+\\]: .*", "abc", "x[0-9]+"]), devices=[0])
    else:
        g = make_gorp(d, monkeypatch, env=env)
    # (the Python oracle is too slow for 400 extractions; test_table_limits pins those rows by construction)
    both_forms(g, d, lines, oracle_prefix=0 if case in ("outcomes400", "match_only") else 600)
    if case == "match_only":
        _, _, rows, tabs = tables_call(g, "".join(s + "\n" for s in lines).encode("utf-8"))
        assert rows["stride"] == 0 and all(not t["cols"] for t in tabs) and sum(t["n"] for t in tabs) == rows["hist"][:3].sum() > 0
    if case == "never_matched":
        _, _, _, tabs = tables_call(g, "".join(s + "\n" for s in lines).encode("utf-8"))
        for e in (0, 2):
            assert tabs[e]["n"] == 0 and tabs[e]["cols"][0]["off"].tolist() == [0]


@pytest.mark.gpu
def test_empty_and_unmatched_batches(monkeypatch):
    g = make_gorp(corpus.WEBLOG_DEF, monkeypatch)
    for buf in (b"", b"\n", b"nothing here\nnor here", b"\n\n\n"):
        rows, tabs = check_all(g, buf)
        assert all(t["n"] == 0 for t in tabs)
    for parts in ([], [b""], [b"nothing", b"", b"x\ny"]):
        for before in (b"", b"\xe4\xb8\xadzz"):
            rows, tabs = check_all(g, before + b"".join(parts), offsets_of(parts) + len(before))
            assert all(t["n"] == 0 for t in tabs) and all(c["off"].tolist() == [0] for t in tabs for c in t["cols"])


# ---------------------------------------------------------------- several devices
def _pieces(buf, off, piece):
    """Start line and end line of every piece the engine cuts the batch into (engine.cu, plan_pieces)."""
    out = []
    if off is None:
        n, u, line = len(buf), 0, 0
        while u < n:
            cut = min(u + piece, n)
            if cut < n:
                i = buf.find(b"\n", cut - 1)
                cut = n if i < 0 else i + 1
            nl = buf.count(b"\n", u, cut)
            out.append((line, line + nl + (1 if cut == n and buf[-1:] != b"\n" else 0)))
            line += nl
            u = cut
    else:
        n, l = len(off) - 1, 0
        while l < n:
            l1 = int(np.searchsorted(off[l + 1:], off[l] + piece, side="right")) + l
            l1 = min(max(l1, l + 1), n)
            out.append((l, l1))
            l = l1
    return out


def _row_bases(rows, buf, off, piece, n_devices):
    """(table, row base) of every device after the first that holds rows of a table with columns."""
    pcs = _pieces(buf, off, piece)
    G = min(n_devices, len(pcs))
    out = set()
    for d in range(1, G):
        first = pcs[len(pcs) * d // G][0]
        last = pcs[len(pcs) * (d + 1) // G - 1][1]
        for e in range(len(rows["hist"]) - 2):
            base = int((rows["ext"][:first] == e).sum())
            if (rows["ext"][first:last] == e).any():
                out.add((e, base))
    return out


def several_engines():
    n = _ffi.lib.gorp_device_count()
    out = [[0, 0], [0, 0, 0]]
    if n >= 2:
        out.append(list(range(n)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("devices", several_engines(), ids=lambda d: "devices=" + ",".join(map(str, d)))
def test_several_devices(devices, monkeypatch):
    """Contiguous line ranges per device context, several pieces each: the tables equal those of a one-device engine buffer
    for buffer. The batches are chosen so that the row bases of the devices fall at every residue mod 8 for tables with
    columns (bitmap shifts, and bitmap bytes shared by two devices)."""
    piece = 6000
    monkeypatch.setenv("GORP_PIECE_UNITS", str(piece))
    one = DefinitionReader.reader(corpus.WEBLOG_DEF).read(devices=[0])
    many = DefinitionReader.reader(corpus.WEBLOG_DEF).read(devices=devices)
    base_lines = mix_lines()[-1500:] + corpus.weblog_lines(1500, seed=4)
    residues = set()
    for j in range(12):
        lines = base_lines[j * 7:] + ["[%d]: GET %dms /é" % (j, j)] * j + ["x" * 80] * (j % 3)
        text = "".join(s + "\n" for s in lines).encode("utf-8")
        parts = [s.encode("utf-8") for s in lines]
        for buf, off in ((text, None), (b"ab" + b"".join(parts), offsets_of(parts) + 2), (text[:-1], None)):
            _, _, rows1, tabs1 = tables_call(one, buf, off)
            rc, msg, rows, tabs = tables_call(many, buf, off)
            assert rc == 0, msg
            same_rows(rows1, rows)
            same_tables(tabs1, tabs)
            residues |= {b % 8 for e, b in _row_bases(rows, buf, off, piece, len(devices)) if tabs[e]["cols"]}
        if j == 0:
            check_reference(many, rows, tabs, buf)
            check_api(many, buf, off, tabs)
    assert residues == set(range(8)), residues


# ---------------------------------------------------------------- errors, lifetime, concurrency
@pytest.mark.gpu
def test_errors_match_plain_calls(monkeypatch):
    monkeypatch.setenv("GORP_PIECE_UNITS", "3000")
    for devices in ([0], [0, 0]):
        g = DefinitionReader.reader(V.README_DEF).read(devices=devices)
        good = ("[1]: GET 2ms /abé\n" * 400).encode("utf-8")
        for buf in (good + b"[2]: GET 2ms /x\xffy\n" + good, good + b"\xe4", b"\x80" + good, good * 3 + b"x\xc3(\n"):
            rc, msg, _ = plain_call(g, buf)
            assert rc == _ffi.GORP_E_ARG and "malformed UTF-8" in msg
            assert tables_call(g, buf)[:2] == (rc, msg)
        parts = [b"[1]: GET 2ms /ab\xc3\xa9"] * 300
        for bad, off in ((parts + [b"x\xc3", b"\xa9y"], None), (parts, np.array([-1, 4], dtype=np.int64)),
                         (parts, np.array([0, 10, 9, 20], dtype=np.int64))):
            o = offsets_of(bad) if off is None else off
            rc, msg, _ = plain_call(g, b"".join(bad), o)
            assert rc == _ffi.GORP_E_ARG and msg
            assert tables_call(g, b"".join(bad), o)[:2] == (rc, msg)
        for off in (None, offsets_of(parts)):
            assert tables_call(g, b"".join(parts), off, null_tables=True)[0] == _ffi.GORP_E_ARG
        check_all(g, good, device=False, api=False)  # the engine still gives correct tables


@pytest.mark.gpu
def test_lifetime(monkeypatch):
    """A result's tables stay as they are while other calls (host, tables, device-resident) run on the engine, and go back
    to the engine with the result. A tables call makes gorp_extract_tables_device fail."""
    g = make_gorp(corpus.WEBLOG_DEF, monkeypatch)
    lines = corpus.weblog_lines(20000, seed=11)
    text = "".join(s + "\n" for s in lines).encode("utf-8")
    rc, msg, rows, tabs, res, dt = tables_call(g, text, keep=True)
    assert rc == 0, msg
    check_all(g, text[: len(text) // 2].rsplit(b"\n", 1)[0] + b"\n")
    parts = [s.encode("utf-8") for s in lines[::-1]]
    tables_call(g, b"".join(parts), offsets_of(parts))
    plain_call(g, text)
    device_tables(g, text[:5000])
    same_rows(rows, rows_of(res))
    same_tables(tabs, tables_of(dt))
    # a tables call leaves no device-resident result to make tables of
    device_tables(g, text[:5000])
    tables_call(g, text[:3000])
    out = _ffi.DeviceTables()
    assert _ffi.lib.gorp_extract_tables_device(g._eng(), 0, torch.cuda.current_stream(DEV).cuda_stream, _ffi.FLAG_SYNC, C.byref(out)) == _ffi.GORP_E_ARG
    # release: the pinned buffers return to the engine, and the next call of no larger size reuses them
    row_buffer = tabs[0]["row_ptr"]
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
    assert not res.owner
    rc, msg, _, again, res2, _ = tables_call(g, text[:4000], keep=True)
    assert rc == 0 and again[0]["row_ptr"] == row_buffer
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res2))


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0], [0, 0]], ids=["one-device", "devices=0,0"])
def test_two_threads(devices, monkeypatch):
    monkeypatch.setenv("GORP_PIECE_UNITS", "50000")
    g = DefinitionReader.reader(corpus.WEBLOG_DEF).read(devices=devices)
    lines = mix_lines()
    halves = [lines[k::2] for k in range(2)]
    texts = ["".join(s + "\n" for s in h).encode("utf-8") for h in halves]
    parts = [[s.encode("utf-8") for s in h] for h in halves]
    calls = [lambda k: tables_call(g, texts[k]), lambda k: tables_call(g, b"".join(parts[k]), offsets_of(parts[k]))]
    want = {(k, c): calls[c](k) for k in range(2) for c in range(2)}
    errors = []

    def worker(k):
        try:
            for i in range(6):
                c = (i + k) % 2
                rc, msg, rows, tabs = calls[c](k)
                assert rc == 0, msg
                same_rows(want[k, c][2], rows)
                same_tables(want[k, c][3], tabs)
        except Exception as ex:  # noqa: BLE001
            errors.append(ex)

    th = [threading.Thread(target=worker, args=(k,)) for k in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors


# ---------------------------------------------------------------- without a GPU
def test_tables_need_byte_offsets():
    g = DefinitionReader.reader(V.README_DEF).read()
    with pytest.raises(ValueError, match="byte_offsets"):
        g.extract_batch_text_utf8(b"[1]: GET 2ms /a\n", tables=True)


def test_pyarrow_not_imported_at_load():
    code = "import sys, gorp_b200, gorp_b200.api; assert 'pyarrow' not in sys.modules, 'pyarrow imported'"
    subprocess.run([sys.executable, "-s", "-c", code], check=True, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
