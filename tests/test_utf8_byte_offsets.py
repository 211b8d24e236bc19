"""gorp_extract_text_utf8_bytes: the UTF-8 text form with its results in byte coordinates of the caller's buffer.

Every result must be exactly the unit-coordinate result of gorp_extract_text_utf8 moved to bytes: ext_id and histogram
equal, line offsets and span boundaries mapped through the bytes each UTF-16 unit of the decoded text comes from, -1 where
the unit form has -1, and every boundary on the first byte of a UTF-8 sequence."""
import ctypes as C
import threading

import numpy as np
import pytest

from gorp_b200 import DefinitionReader, _ffi, corpus
from tests import reference_vectors as V

pytestmark = pytest.mark.gpu

PIECES = (None, "3000", "70000")
BAD_SEQUENCES = (b"\xc0\xaf", b"\xed\xa0\x80", b"\xf4\x90\x80\x80", b"\x80", b"\xe4\xb8", b"\xf0\x9f\x98", b"\xff")


def unit_to_byte_map(units):
    """map[u] = byte offset of UTF-16 unit u of the decoded text (u <= n_units + 1, the end of an unterminated last line)."""
    u = np.asarray(units, dtype=np.uint32)
    nbytes = np.where(u < 0x80, 1, np.where(u < 0x800, 2, 3)).astype(np.int64)
    nbytes[(u >= 0xD800) & (u < 0xDC00)] = 4  # a high surrogate stands for the whole 4-byte sequence
    nbytes[(u >= 0xDC00) & (u < 0xE000)] = 0
    m = np.zeros(len(u) + 2, dtype=np.int64)
    np.cumsum(nbytes, out=m[1:len(u) + 1])
    m[-1] = m[-2] + 1
    return m


def check_bytes_form(g, data, piece=None, monkeypatch=None):
    """The new call against the unit form on the same bytes and the numpy conversion; returns both batches."""
    if monkeypatch is not None:
        if piece:
            monkeypatch.setenv("GORP_PIECE_UNITS", piece)
        else:
            monkeypatch.delenv("GORP_PIECE_UNITS", raising=False)
    bu = g.extract_batch_text_utf8(data)
    bb = g.extract_batch_text_utf8(data, byte_offsets=True)
    assert bb.n_lines == bu.n_lines and bb.span_stride == bu.span_stride
    assert (bb.ext_id == bu.ext_id).all() and (bb.histogram == bu.histogram).all()
    m = unit_to_byte_map(bu.units)
    assert (bb.line_off == m[bu.line_off]).all(), np.flatnonzero(bb.line_off != m[bu.line_off])[:10]
    starts_u = bu.line_off[:-1, None]
    want = np.where(bu.spans >= 0, m[starts_u + np.maximum(bu.spans, 0)] - m[starts_u], -1)
    assert ((bb.spans >= 0) == (bu.spans >= 0)).all()
    assert (bb.spans == want).all(), np.flatnonzero((bb.spans != want).any(axis=1))[:10]
    raw = np.frombuffer(bytes(data), dtype=np.uint8)
    at = (bb.line_off[:-1, None] + bb.spans)[bb.spans >= 0]
    at = at[at < len(raw)]
    assert ((raw[at] & 0xC0) != 0x80).all()
    return bu, bb


def mix_lines():
    lines = corpus.utf16_mix_lines(6000, seed=12)
    lines = [s for s in lines if not any(0xD800 <= ord(ch) <= 0xDFFF for ch in s)]  # lone surrogates have no UTF-8 form
    lines += ["", "é" * 40, "éü" * 30 + "x", "中文" * 30, "\U0001F600" * 25, "", "[1]: GET 2ms /\U00010400Жx",
              "[2]: PUT 31ms /a\U0001F600béc", "[7]: HEAD 12ms /中\U0001F600文/é", "x" * 5000 + "é",
              "[3]: GET 9ms /" + "é中\U0001F600a" * 1250]
    return lines


def long_lines():
    rng = np.random.default_rng(17)
    lines = corpus.weblog_lines(300, seed=8)
    body = "".join(rng.choice(list("abcdefghij0123456789/"), size=70000))
    lines += ["[1]: GET 2ms /" + body, "[2]: PUT 31ms /" + body * 3 + "é" + body, "[3]: GET 2ms /" + body + " tail",
              "[4]: HEAD 7ms /" + body[:64990], "[5]: GET 2ms /" + body + "\x0bq", "[6]: GET 2ms /" + "\U0001F600" * 40000,
              "[8]: PUT 5ms /" + "é" * 70000 + " x"]
    return lines


def utf8_of(lines, terminated=True):
    return ("\n".join(lines) + ("\n" if terminated else "")).encode("utf-8")


def corpus_text(units):
    return np.asarray(units, dtype=np.uint16).tobytes().decode("utf-16-le").encode("utf-8")


@pytest.mark.parametrize("case", ["mix-weblog", "mix-readme", "readme", "readme-twopass", "weblog", "syslog200"])
def test_equivalence_with_unit_form(monkeypatch, case):
    """Line mix of 1- to 4-byte sequences, the config corpora (fused walk, K2b + K4c, K4b), pieces of every size."""
    if case.endswith("twopass"):
        monkeypatch.setenv("GORP_FORCE_TWOPASS", "1")
    if case.startswith("mix"):
        d = corpus.WEBLOG_DEF if case == "mix-weblog" else V.README_DEF
        lines = mix_lines()
        datas = [utf8_of(lines), utf8_of(lines, terminated=False)]
    elif case.startswith("readme"):
        d, gen = corpus.CONFIGS["readme"]
        t = corpus_text(gen(30000, seed=5))
        datas = [t, t[:-1]]
    elif case == "weblog":
        d, lines = corpus.WEBLOG_DEF, corpus.weblog_lines(8000, seed=3)
        datas = [utf8_of(lines), utf8_of(lines, terminated=False)]
    else:
        d, lines = corpus.SYSLOG200_DEF, corpus.syslog200_lines(3000, seed=6)
        datas = [utf8_of(lines), utf8_of(lines, terminated=False)]
    g = DefinitionReader.reader(d).read()
    for piece in PIECES:
        for data in datas:
            check_bytes_form(g, data, piece, monkeypatch)


def test_very_long_lines(monkeypatch):
    """Lines of 70 000 units and more (the tail walk's 32-bit kernel), ASCII and non-ASCII: one warp walks each."""
    monkeypatch.setenv("GORP_FORCE_TWOPASS", "1")
    lines = long_lines()
    for d in (V.README_DEF, corpus.WEBLOG_DEF):
        g = DefinitionReader.reader(d).read()
        for piece in PIECES:
            for data in (utf8_of(lines), utf8_of(lines, terminated=False)):
                _, bb = check_bytes_form(g, data, piece, monkeypatch)
        if d == V.README_DEF:  # (its path group takes the whole long line)
            assert int(bb.spans.max()) > 65535


def test_values_decode_from_byte_slices(monkeypatch):
    """result(i).asMap() on the byte-coordinate batch equals the unit-form batch and extract_batch_text of the decoded text."""
    for d, lines in ((corpus.WEBLOG_DEF, mix_lines()[:3000] + mix_lines()[-11:]), (V.README_DEF, mix_lines()[-11:] + long_lines()[-4:])):
        g = DefinitionReader.reader(d).read()
        data = utf8_of(lines, terminated=False)
        bb = g.extract_batch_text_utf8(data, byte_offsets=True)
        bu = g.extract_batch_text_utf8(data)
        b16 = g.extract_batch_text(data.decode("utf-8"))
        assert bb.units.dtype == np.uint8 and len(bb.units) == len(data)
        for i in range(bb.n_lines):
            assert bb.line(i) == bu.line(i) == b16.line(i) == lines[i]
            got = [bb.result(i, safe=True), bu.result(i, safe=True), b16.result(i, safe=True)]
            if got[0] is None:
                assert got[1] is None and got[2] is None
            else:
                assert got[0].asMap("id") == got[1].asMap("id") == got[2].asMap("id")
                assert got[0].getInput() == lines[i]


def call_bytes(g, buf):
    res = _ffi.Result()
    rc = _ffi.lib.gorp_extract_text_utf8_bytes(g._eng(), buf.ctypes.data, len(buf), C.byref(res))
    if rc != 0:
        return rc, _ffi.last_error()
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
    return rc, ""


def test_malformed_and_edge_inputs():
    g = DefinitionReader.reader(V.README_DEF).read()
    good = "[1]: GET 2ms /abc\n".encode("utf-8") * 300
    for bad in BAD_SEQUENCES:
        rc, msg = call_bytes(g, np.frombuffer(good + b"/x" + bad + b"y\n" + good, dtype=np.uint8))
        assert rc == _ffi.GORP_E_ARG and "malformed UTF-8 at byte %d" % (len(good) + 2) in msg, (bad, msg)
    with pytest.raises(ValueError, match="malformed UTF-8 at byte 1"):
        g.extract_batch_text_utf8(b"a\xff\n", byte_offsets=True)
    b = g.extract_batch_text_utf8(b"", byte_offsets=True)
    assert b.n_lines == 0 and b.line_off.tolist() == [0]
    one = "[1]: GET 2ms /é".encode("utf-8")
    b = g.extract_batch_text_utf8(one, byte_offsets=True)
    assert b.ext_id.tolist() == [1] and b.line_off.tolist() == [0, len(one) + 1]
    assert b.result(0).asMap()["path"] == "/é" and b.spans_of(0)[-1] == (13, len(one))


def multi_engines():
    n = _ffi.lib.gorp_device_count()
    out = [[0, 0]]
    if n >= 2:
        out.append(list(range(n)))
    return out


@pytest.mark.parametrize("devices", multi_engines(), ids=lambda d: "devices=" + ",".join(map(str, d)))
def test_several_devices(monkeypatch, devices):
    """Contiguous line-aligned byte ranges per device context (two contexts on one GPU with devices=[0, 0]): results
    identical to a one-device engine; the lowest malformed byte wins; the unit form on the same engine is unchanged."""
    monkeypatch.setenv("GORP_PIECE_UNITS", "40000")
    lines = mix_lines()
    for d in (corpus.WEBLOG_DEF, V.README_DEF):
        one = DefinitionReader.reader(d).read()
        many = DefinitionReader.reader(d).read(devices=devices)
        for data in (utf8_of(lines), utf8_of(lines, terminated=False)):
            b1 = one.extract_batch_text_utf8(data, byte_offsets=True)
            bm = check_bytes_form(many, data)[1]
            assert bm.n_lines == b1.n_lines and (bm.ext_id == b1.ext_id).all() and (bm.line_off == b1.line_off).all()
            assert (bm.spans == b1.spans).all() and (bm.histogram == b1.histogram).all()
            u1, um = one.extract_batch_text_utf8(data), many.extract_batch_text_utf8(data)
            assert (um.line_off == u1.line_off).all() and (um.spans == u1.spans).all() and (um.ext_id == u1.ext_id).all()
    data = bytearray(utf8_of(lines))
    cut = data.rfind(b"\n", 0, len(data) - 2000) + 1  # a line in the last device's range
    first = data.find(b"\n", len(data) // 2) + 1       # ... and one that may be in an earlier range
    for where in ([cut], [first, cut]):
        bad = bytearray(data)
        for p in where:
            bad[p:p + 1] = b"\xff"
        buf = np.frombuffer(bytes(bad), dtype=np.uint8)
        rc1, m1 = call_bytes(one, buf)
        rcm, mm = call_bytes(many, buf)
        assert rc1 == rcm == _ffi.GORP_E_ARG and m1 == mm and "malformed UTF-8 at byte %d " % min(where) in mm, (m1, mm)
    b1 = one.extract_batch_text_utf8(bytes(data), byte_offsets=True)  # the engines are still usable
    bm = many.extract_batch_text_utf8(bytes(data), byte_offsets=True)
    assert (bm.spans == b1.spans).all() and (bm.line_off == b1.line_off).all()


@pytest.mark.parametrize("devices", [None, [0, 0]], ids=["one-device", "devices=0,0"])
def test_concurrent_byte_and_unit_calls(monkeypatch, devices):
    """Two threads mixing the byte-coordinate call and gorp_extract_text_utf8 on one engine get their sequential results."""
    monkeypatch.setenv("GORP_PIECE_UNITS", "60000")
    g = DefinitionReader.reader(corpus.WEBLOG_DEF).read(devices=devices)
    lines = mix_lines()
    datas = [utf8_of(lines[k::2]) for k in range(2)]
    want = {(k, bo): g.extract_batch_text_utf8(datas[k], byte_offsets=bo) for k in range(2) for bo in (False, True)}
    errors = []

    def worker(t):
        try:
            for rep in range(6):
                k, bo = (t + rep) % 2, rep % 2 == t
                b, w = g.extract_batch_text_utf8(datas[k], byte_offsets=bo), want[(k, bo)]
                assert b.n_lines == w.n_lines and (b.ext_id == w.ext_id).all() and (b.spans == w.spans).all()
                assert (b.line_off == w.line_off).all() and (b.histogram == w.histogram).all()
        except Exception as ex:  # noqa: BLE001
            errors.append(repr(ex))

    ts = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors[:3]
