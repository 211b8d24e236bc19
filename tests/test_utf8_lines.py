"""gorp_extract_lines_utf8: Gorp.extractAll(List<String>) for strings held as UTF-8 bytes, results in byte coordinates.

Every result must be exactly the result of gorp_extract_lines on the decoded strings moved to bytes: ext_id and histogram
equal, line_off a copy of the caller's offsets, span boundaries mapped through the bytes each UTF-16 unit comes from, -1
where the unit form has -1, and every boundary on the first byte of a UTF-8 sequence. A string that is not well-formed
UTF-8 on its own fails the call at the lowest byte where Python's strict decoder fails on some string."""
import ctypes as C
import threading

import numpy as np
import pytest

from gorp_b200 import DefinitionReader, _ffi, corpus
from tests import reference_vectors as V
from tests.test_utf8_byte_offsets import BAD_SEQUENCES, long_lines, mix_lines, unit_to_byte_map

pytestmark = pytest.mark.gpu

PIECES = (None, "3000", "70000")
TIERS = {"default": {}, "twopass": {"GORP_FORCE_TWOPASS": "1"}, "notails": {"GORP_FORCE_TWOPASS": "1", "GORP_NO_TAILS": "1"},
         "k1k2_k4": {"GORP_FORCE_TWOPASS": "1", "GORP_FORCE_K1K2": "1", "GORP_FORCE_K4": "1"}, "general": {"GORP_FORCE_GENERAL": "1"}}


def set_piece(monkeypatch, piece):
    if piece:
        monkeypatch.setenv("GORP_PIECE_UNITS", piece)
    else:
        monkeypatch.delenv("GORP_PIECE_UNITS", raising=False)


def offsets_of(parts):
    off = np.zeros(len(parts) + 1, dtype=np.int64)
    if parts:
        np.cumsum([len(p) for p in parts], out=off[1:])
    return off


def check_lines_form(g, strings, buf=None, off=None):
    """The new call (on `strings`, or on `buf` / `off` when given) against gorp_extract_lines on the decoded strings."""
    bu = g.extract_batch_lines(strings)
    if buf is None:
        bb = g.extract_batch_lines_utf8(strings)
        buf, off = bytes(bb.units), offsets_of([s.encode("utf-8") for s in strings])
    else:
        bb = g.extract_batch_lines_utf8(buf, off)
    assert bb.n_lines == bu.n_lines == len(strings) and bb.span_stride == bu.span_stride
    assert (bb.ext_id == bu.ext_id).all() and (bb.histogram == bu.histogram).all()
    assert bb.line_off.tolist() == np.asarray(off).tolist()
    # the decoded strings joined: unit u of string i maps to byte m[u] - m[start_i] of string i (no pair crosses a string)
    m = unit_to_byte_map(bu.units)
    assert (m[bu.line_off] - m[bu.line_off[0]] == bb.line_off - bb.line_off[0]).all()
    starts_u = bu.line_off[:-1, None]
    want = np.where(bu.spans >= 0, m[starts_u + np.maximum(bu.spans, 0)] - m[starts_u], -1)
    assert ((bb.spans >= 0) == (bu.spans >= 0)).all()
    assert (bb.spans == want).all(), np.flatnonzero((bb.spans != want).any(axis=1))[:10]
    raw = np.frombuffer(bytes(buf), dtype=np.uint8)
    ends = bb.line_off[1:, None] + np.zeros_like(bb.spans)
    at = bb.line_off[:-1, None] + bb.spans
    inside = (bb.spans >= 0) & (at < ends)
    assert ((raw[at[inside]] & 0xC0) != 0x80).all()
    return bu, bb


def corpus_lines(case):
    if case.startswith("mix"):
        return (corpus.WEBLOG_DEF if case == "mix-weblog" else V.README_DEF), mix_lines()
    if case == "readme":
        d, gen = corpus.CONFIGS["readme"]
        return d, np.asarray(gen(30000, seed=5), dtype=np.uint16).tobytes().decode("utf-16-le").split("\n")[:-1]
    if case == "weblog":
        return corpus.WEBLOG_DEF, corpus.weblog_lines(8000, seed=3)
    return corpus.SYSLOG200_DEF, corpus.syslog200_lines(3000, seed=6)


@pytest.mark.parametrize("tier", list(TIERS))
@pytest.mark.parametrize("case", ["mix-weblog", "mix-readme", "readme", "weblog", "syslog200"])
def test_equivalence_with_lines_form(monkeypatch, case, tier):
    """Line mix of 1- to 4-byte sequences and the config corpora, every tier the lines form takes, pieces of every size."""
    for k, v in TIERS[tier].items():
        monkeypatch.setenv(k, v)
    d, lines = corpus_lines(case)
    g = DefinitionReader.reader(d).read()
    for piece in PIECES:
        set_piece(monkeypatch, piece)
        check_lines_form(g, lines)


def odd_strings():
    return ["[1]: GET 2ms /a\nb", "[2]: PUT 3ms /x\r", "", "\n", "\r\n", "[3]: GET 4ms /é\n中", "[4]: HEAD 5ms /\U0001F600\n\n",
            "", "[5]: GET 6ms /ok", "line one\nline two\n[6]: GET 7ms /no"]


@pytest.mark.parametrize("tier", ["default", "twopass"])
def test_odd_strings(monkeypatch, tier):
    """Embedded '\\n' and '\\r' are data (one row per string), empty strings, an empty batch, strings of 70 000 units and
    more, ASCII and non-ASCII."""
    for k, v in TIERS[tier].items():
        monkeypatch.setenv(k, v)
    for d in (V.README_DEF, corpus.WEBLOG_DEF):
        g = DefinitionReader.reader(d).read()
        for piece in PIECES:
            set_piece(monkeypatch, piece)
            _, bb = check_lines_form(g, odd_strings() * 50 + mix_lines()[-11:])
            assert [bb.line(i) for i in range(10)] == odd_strings()
            _, bb = check_lines_form(g, long_lines() + odd_strings())
            if d == V.README_DEF:
                assert int(bb.spans.max()) > 65535
            check_lines_form(g, [""] * 7)
            b = g.extract_batch_lines_utf8([])
            assert b.n_lines == 0 and b.line_off.tolist() == [0] and b.histogram.sum() == 0
            b = g.extract_batch_lines_utf8(b"\xff\xfe", np.array([1], dtype=np.int64))
            assert b.n_lines == 0 and b.line_off.tolist() == [1]


@pytest.mark.parametrize("piece", PIECES)
def test_callers_offsets(monkeypatch, piece):
    """off[0] > 0 and malformed garbage outside [off[0], off[n]): the results are those of the compacted buffer, shifted."""
    set_piece(monkeypatch, piece)
    g = DefinitionReader.reader(corpus.WEBLOG_DEF).read()
    lines = mix_lines()
    parts = [s.encode("utf-8") for s in lines]
    compact = g.extract_batch_lines_utf8(parts)
    for head in (1, 7, 16, 4099):
        garbage = (b"\xff\x80\xc3" * 2000)[:head]
        buf = garbage + b"".join(parts) + b"\x80\xf4\x90"
        off = offsets_of(parts) + head
        _, bb = check_lines_form(g, lines, buf, off)
        assert (bb.line_off == compact.line_off + head).all() and (bb.spans == compact.spans).all()
        assert (bb.ext_id == compact.ext_id).all()
        # an Arrow slice: strings [a, b) of the column, the offsets as they are
        a, b = 1000, 4000
        _, bs = check_lines_form(g, lines[a:b], buf, off[a:b + 1])
        assert (bs.spans == compact.spans[a:b]).all() and (bs.ext_id == compact.ext_id[a:b]).all()


def test_pike_vm_fallback(monkeypatch):
    """Capture automata beyond the state limit go through the simulated Pike VM, which reads the decoded piece and its unit
    offsets."""
    names = "abcdefghi"
    ambiguous = "extract e {\n template " + ":".join("$%s(%%{[ab:]*})" % n for n in names) + "\n}\n"
    rng = np.random.default_rng(23)
    amb_lines = ["".join(rng.choice(list("ab:::é"), size=rng.integers(0, 40))) for _ in range(3000)]
    for limit in ("2", "500"):
        monkeypatch.setenv("GORP_TDFA_MAX_STATES", limit)
        for d, lines in ((ambiguous, amb_lines), (V.README_DEF, mix_lines()[-11:] + ["[1]: GET 2ms /" + "é" * 3000]),
                         (corpus.WEBLOG_DEF, mix_lines()[:1500])):
            g = DefinitionReader.reader(d).read()
            for piece in (None, "3000"):
                set_piece(monkeypatch, piece)
                check_lines_form(g, lines)


def test_values():
    """result(i).asMap("id") and line(i) decode from the caller's bytes and equal extract_batch_lines."""
    for d, lines in ((corpus.WEBLOG_DEF, mix_lines()[:3000] + mix_lines()[-11:] + odd_strings()),
                     (V.README_DEF, mix_lines()[-11:] + long_lines()[-4:] + odd_strings())):
        g = DefinitionReader.reader(d).read()
        bb = g.extract_batch_lines_utf8(lines)
        bu = g.extract_batch_lines(lines)
        assert bb.units.dtype == np.uint8
        for i in range(bb.n_lines):
            assert bb.line(i) == bu.line(i) == lines[i]
            got = [bb.result(i, safe=True), bu.result(i, safe=True)]
            if got[0] is None:
                assert got[1] is None
            else:
                assert got[0].asMap("id") == got[1].asMap("id") and got[0].getInput() == lines[i]


def first_bad_byte(buf, off):
    """The lowest byte at which Python's strict decoder fails on some string on its own, or None."""
    bad = None
    for i in range(len(off) - 1):
        try:
            bytes(buf[off[i]:off[i + 1]]).decode("utf-8")
        except UnicodeDecodeError as ex:
            p = int(off[i]) + ex.start
            bad = p if bad is None else min(bad, p)
    return bad


def call_lines(g, buf, off):
    b = np.frombuffer(bytes(buf), dtype=np.uint8)
    o = np.ascontiguousarray(off, dtype=np.int64)
    res = _ffi.Result()
    rc = _ffi.lib.gorp_extract_lines_utf8(g._eng(), b.ctypes.data, o.ctypes.data, len(o) - 1, C.byref(res))
    if rc != 0:
        return rc, _ffi.last_error()
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
    return rc, ""


def expect_malformed(g, buf, off):
    want = first_bad_byte(buf, off)
    assert want is not None
    rc, msg = call_lines(g, buf, off)
    assert rc == _ffi.GORP_E_ARG and "malformed UTF-8 at byte %d " % want in msg, (want, msg)


@pytest.mark.parametrize("piece", [None, "3000"])
def test_malformed_input(monkeypatch, piece):
    set_piece(monkeypatch, piece)
    g = DefinitionReader.reader(V.README_DEF).read()
    good = ["[1]: GET 2ms /abé", "中文\U0001F600", "x"] * 300
    gp = [s.encode("utf-8") for s in good]
    check = lambda: check_lines_form(g, good)  # noqa: E731  (the engine still gives correct results)
    for bad in BAD_SEQUENCES:
        parts = gp + [b"[2]: GET 2ms /x" + bad + b"y"] + gp
        expect_malformed(g, b"".join(parts), offsets_of(parts))
        parts = gp + [b"/x" + bad] + gp  # at the end of a string, the next string well-formed
        expect_malformed(g, b"".join(parts), offsets_of(parts))
        check()
    # the concatenation is well-formed ("xéy"), both strings are not: the byte of \xc3
    parts = gp + [b"x\xc3", b"\xa9y"] + gp
    expect_malformed(g, b"".join(parts), offsets_of(parts))
    assert first_bad_byte(b"".join(parts), offsets_of(parts)) == sum(map(len, gp)) + 1
    # a string that starts with a continuation byte after a complete sequence; after a 4-byte sequence cut after 1, 2, 3 bytes
    for parts in ([b"x\xc3\xa9", b"\xa9y"], [b"\xf0", b"\x9f\x98\x80"], [b"a\xf0\x9f", b"\x98\x80"], [b"ab\xf0\x9f\x98", b"\x80"],
                  [b"\xe4", b"", b"\xb8\xad"], [b"\x80abc"]):
        parts = gp + parts + gp
        expect_malformed(g, b"".join(parts), offsets_of(parts))
    # two faults: the lowest wins
    parts = gp + [b"\xff"] + gp + [b"x\xe4", b"\xb8\xad"] + gp
    expect_malformed(g, b"".join(parts), offsets_of(parts))
    parts = gp + [b"x\xe4", b"\xb8\xad"] + gp + [b"\xff"] + gp
    expect_malformed(g, b"".join(parts), offsets_of(parts))
    check()
    # strings cut at random byte positions of well-formed text, and random corruption: the Python oracle decides
    rng = np.random.default_rng(41)
    text = "".join(mix_lines()[-11:]).encode("utf-8")
    for trial in range(60):
        cuts = np.sort(rng.choice(np.arange(1, len(text)), size=int(rng.integers(1, 40)), replace=False))
        off = np.concatenate(([0], cuts, [len(text)])).astype(np.int64)
        buf = bytearray(text)
        if trial % 3 == 0:
            buf[int(rng.integers(0, len(buf)))] = int(rng.choice([0x80, 0xbf, 0xc3, 0xe4, 0xf0, 0xff, 0x41]))
        if first_bad_byte(buf, off) is None:
            assert call_lines(g, buf, off)[0] == 0
        else:
            expect_malformed(g, buf, off)
    check()
    # offsets
    buf = b"[1]: GET 2ms /abc" * 4
    for off, msg in (([-1, 4], "offsets must start at >= 0"), ([0, 10, 9, 20], "offsets must be non-decreasing \\(line 1\\)")):
        with pytest.raises(ValueError, match=msg):
            g.extract_batch_lines_utf8(buf, np.array(off, dtype=np.int64))
    with pytest.raises(ValueError, match="malformed UTF-8 at byte 3"):
        g.extract_batch_lines_utf8([b"ab", b"c\xff"])
    check()


def multi_engines():
    n = _ffi.lib.gorp_device_count()
    out = [[0, 0]]
    if n >= 2:
        out.append(list(range(n)))
    return out


@pytest.mark.parametrize("devices", multi_engines(), ids=lambda d: "devices=" + ",".join(map(str, d)))
def test_several_devices(monkeypatch, devices):
    """Contiguous ranges of strings per device context: results identical to a one-device engine; the lowest malformed byte
    wins across devices."""
    monkeypatch.setenv("GORP_PIECE_UNITS", "40000")
    lines = mix_lines() + odd_strings()
    parts = [s.encode("utf-8") for s in lines]
    for d in (corpus.WEBLOG_DEF, V.README_DEF):
        one = DefinitionReader.reader(d).read()
        many = DefinitionReader.reader(d).read(devices=devices)
        b1 = one.extract_batch_lines_utf8(parts)
        bm = check_lines_form(many, lines)[1]
        assert bm.n_lines == b1.n_lines and (bm.ext_id == b1.ext_id).all() and (bm.line_off == b1.line_off).all()
        assert (bm.spans == b1.spans).all() and (bm.histogram == b1.histogram).all()
    n = len(parts)
    for where in ([n - 20], [n // 2, n - 20], [n // 4, n // 2]):
        bad = list(parts)
        for i in where:
            bad[i] = bad[i] + b"\xe4"  # a truncated sequence at the string's end
        buf, off = b"".join(bad), offsets_of(bad)
        want = first_bad_byte(buf, off)
        rc1, m1 = call_lines(one, buf, off)
        rcm, mm = call_lines(many, buf, off)
        assert rc1 == rcm == _ffi.GORP_E_ARG and m1 == mm and "malformed UTF-8 at byte %d " % want in mm, (m1, mm)
    bm = check_lines_form(many, lines)[1]  # still usable
    assert (bm.spans == one.extract_batch_lines_utf8(parts).spans).all()


@pytest.mark.parametrize("devices", [None, [0, 0]], ids=["one-device", "devices=0,0"])
def test_concurrent_calls(monkeypatch, devices):
    """Two threads mixing this call, gorp_extract_lines and gorp_extract_text_utf8_bytes on one engine get their
    sequential results."""
    monkeypatch.setenv("GORP_PIECE_UNITS", "60000")
    g = DefinitionReader.reader(corpus.WEBLOG_DEF).read(devices=devices)
    lines = mix_lines()
    halves = [lines[k::2] for k in range(2)]
    calls = {"utf8": lambda k: g.extract_batch_lines_utf8(halves[k]), "utf16": lambda k: g.extract_batch_lines(halves[k]),
             "text": lambda k: g.extract_batch_text_utf8(("\n".join(halves[k]) + "\n").encode("utf-8"), byte_offsets=True)}
    want = {(k, c): calls[c](k) for k in range(2) for c in calls}
    errors = []

    def worker(t):
        try:
            for rep in range(9):
                k, c = (t + rep) % 2, list(calls)[(rep + t) % 3]
                b, w = calls[c](k), want[(k, c)]
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
