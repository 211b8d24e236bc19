"""The UTF-8 device-resident calls (gorp_extract_text_utf8_device, gorp_extract_lines_utf8_device) against the host forms.

A caller that holds UTF-8 in HBM (a cuDF / Arrow string column, a file read into device memory, a torch uint8 tensor) gets
the results of gorp_extract_text_utf8_bytes / gorp_extract_lines_utf8 on the same bytes, in byte coordinates, from one
launch per stage over the whole batch. Every comparison here is with the host call on the same engine: ext_id, line_off,
spans and histogram identical, and on failure the same status and message. At scale (one launch past 2^32 bytes) the ASCII
text of config #2 is compared with the UTF-16 device calls on the same lines, where bytes and units coincide, and a 1 M-line
prefix with the oracle."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from gorp_b200 import _ffi, corpus, corpusgen, parityhash
from tests import reference_vectors as V
from tests.test_device_forms import Rows, device_views, fetch, make_gorp, n_bins, window_histogram, window_rows
from tests.test_gpu_parity import TIERS, assert_matches_oracle
from tests.test_utf8_byte_offsets import BAD_SEQUENCES, long_lines, mix_lines, utf8_of
from tests.test_utf8_lines import TIERS as LINES_TIERS
from tests.test_utf8_lines import odd_strings, offsets_of

pytestmark = pytest.mark.gpu
FLAGS = _ffi.FLAG_SYNC
DEV = torch.device("cuda", 0)


# ---------------------------------------------------------------- calls
def stream_handle(stream):
    return (torch.cuda.current_stream(DEV) if stream is None else stream).cuda_stream


def text8_call(g, ptr, n_bytes, stream=None, flags=FLAGS, dev_index=0):
    """(status, message, gorp_device_result) of gorp_extract_text_utf8_device."""
    dres = _ffi.DeviceResult()
    rc = _ffi.lib.gorp_extract_text_utf8_device(g._eng(), dev_index, ptr, n_bytes, stream_handle(stream), flags, C.byref(dres))
    return rc, (_ffi.last_error() if rc else ""), dres


def lines8_call(g, ptr, d_off, n_lines, stream=None, flags=FLAGS, dev_index=0):
    dres = _ffi.DeviceResult()
    rc = _ffi.lib.gorp_extract_lines_utf8_device(g._eng(), dev_index, ptr, d_off.data_ptr(), n_lines, stream_handle(stream), flags,
                                                 C.byref(dres))
    return rc, (_ffi.last_error() if rc else ""), dres


def host_text(g, data):
    """(status, message, Rows) of gorp_extract_text_utf8_bytes on `data`."""
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    res = _ffi.Result()
    rc = _ffi.lib.gorp_extract_text_utf8_bytes(g._eng(), buf.ctypes.data, len(buf), C.byref(res))
    return _host_rows(g, rc, res)


def host_lines(g, data, off):
    buf = np.frombuffer(bytes(data), dtype=np.uint8)
    o = np.ascontiguousarray(off, dtype=np.int64)
    res = _ffi.Result()
    rc = _ffi.lib.gorp_extract_lines_utf8(g._eng(), buf.ctypes.data, o.ctypes.data, len(o) - 1, C.byref(res))
    return _host_rows(g, rc, res)


def _host_rows(g, rc, res):
    if rc:
        return rc, _ffi.last_error(), None
    n, w = int(res.n_lines), int(res.span_stride)
    rows = Rows(n, w, np.ctypeslib.as_array(res.ext_id, (max(n, 1),))[:n].copy(),
                np.ctypeslib.as_array(res.line_off, (n + 1,)).copy(),
                np.ctypeslib.as_array(res.spans, (max(n * w, 1),))[:n * w].reshape(n, w).copy(),
                np.ctypeslib.as_array(res.histogram, (res.n_extractions + 2,)).copy())
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
    return rc, "", rows


def returned_offsets(dres):
    """The n_lines + 1 entries behind a result's d_line_off (fetch() shows an empty result's offsets as [0])."""
    return torch.as_tensor(parityhash.DeviceArray(dres.d_line_off, (int(dres.n_lines) + 1,), "<i8"), device=DEV).cpu().numpy()


def placed(data, shift=0, before=b"", after=b""):
    """A uint8 CUDA tensor holding before + data + after at `shift` bytes past a 512-byte boundary; returns (tensor, address
    of data)."""
    raw = np.frombuffer(bytes(before) + bytes(data) + bytes(after), dtype=np.uint8)
    t = torch.zeros(shift + len(raw) + 64, dtype=torch.uint8, device=DEV)
    assert t.data_ptr() % 512 == 0
    t[shift:shift + len(raw)] = torch.from_numpy(raw.copy()).to(DEV)
    return t, t.data_ptr() + shift + len(before)


def expect_text(g, data, shift=0, after=b"", **kw):
    """The device text form on `data` (at `shift`, followed by `after`) equals the host byte form on `data`: same rows, or the
    same failure."""
    t, ptr = placed(data, shift, after=after)
    rc, msg, dres = text8_call(g, ptr, len(data), **kw)
    got = fetch(dres, n_bins(g), DEV, stream=kw.get("stream")) if rc == 0 else None  # (valid until the next call)
    hrc, hmsg, want = host_text(g, data)
    assert (rc, msg) == (hrc, hmsg)
    if rc == 0:
        got.same_as(want)
    return rc


def expect_lines(g, data, off, before=b"", after=b"", **kw):
    """The device lines form on strings [off[i], off[i+1]) of `data`, placed after `before` (offsets shifted with it), equals
    gorp_extract_lines_utf8 on `data` and `off`."""
    t, ptr = placed(data, 0, before, after)
    base = ptr - len(before)
    shifted = np.asarray(off, dtype=np.int64) + len(before)
    d_off = torch.from_numpy(shifted).to(DEV)
    rc, msg, dres = lines8_call(g, base, d_off, len(off) - 1, **kw)
    got = None
    if rc == 0:  # (valid until the next call) d_line_off is the caller's d_off; its n_lines + 1 entries are read through it
        assert int(dres.d_line_off) == d_off.data_ptr()
        got = fetch(dres, n_bins(g), DEV, stream=kw.get("stream"))
        got.line_off = returned_offsets(dres)
    hrc, hmsg, want = host_lines(g, data, off)
    if hrc == 0:
        hmsg = ""
    else:  # (a byte named in the message moves with the offsets)
        hmsg = re.sub(r"at byte (\d+)", lambda m: "at byte %d" % (int(m.group(1)) + len(before)), hmsg)
    assert (rc, msg) == (hrc, hmsg)
    if rc == 0:
        got.same_as(want, off_shift=len(before))
    return rc


# ---------------------------------------------------------------- 1. text form = host byte form
def corpus_utf8(name):
    if name == "utf16mix":  # config #5 without its lone-surrogate lines (they have no UTF-8 form)
        from tools_utf8_byte_offsets import mix_corpus
        return corpus.CONFIGS["utf16mix"][0], mix_corpus(6000)[0].tobytes()
    if name == "mix":
        return corpus.WEBLOG_DEF, utf8_of(mix_lines())
    d = corpus.CONFIGS[name][0]
    n = {"readme": 30000, "weblog": 8000, "syslog200": 3000}[name]
    return d, corpusgen.host_text(name, 0, n).tobytes().decode("utf-16-le").encode("utf-8")


@pytest.mark.parametrize("tier", list(TIERS))
def test_text_form_equals_host_byte_form(tier, monkeypatch):
    """readme (fused walk), weblog (K2b + K4c), syslog200 (K4b), utf16mix and the UTF-8 line mix; with and without the final
    '\\n'; d_text 32-byte aligned and only 16-byte aligned."""
    for name in ("readme", "weblog", "syslog200", "utf16mix", "mix"):
        d, data = corpus_utf8(name)
        assert data.endswith(b"\n")
        g = make_gorp(d, monkeypatch, TIERS[tier])
        for text in (data, data[:-1]):
            for shift in (0, 16):
                assert expect_text(g, text, shift) == 0


# ---------------------------------------------------------------- 2. lines form = gorp_extract_lines_utf8
@pytest.mark.parametrize("tier", list(LINES_TIERS))
def test_lines_form_equals_host_lines_form(tier, monkeypatch):
    """Embedded '\\n' and '\\r', empty strings, an empty batch, strings of 70 000 bytes and more, d_off[0] at every residue
    mod 16 with malformed garbage before d_off[0] and after d_off[n]."""
    garbage = b"\xff\x80\xc3\n[1]: GET 2ms /a\n\xe4"
    for d in (V.README_DEF, corpus.WEBLOG_DEF):
        g = make_gorp(d, monkeypatch, LINES_TIERS[tier])
        for strings in (odd_strings() * 50 + mix_lines()[-11:], long_lines() + odd_strings(), [""] * 7, mix_lines()[:2000]):
            parts = [s.encode("utf-8") for s in strings]
            data, off = b"".join(parts), offsets_of(parts)
            assert expect_lines(g, data, off) == 0
            assert expect_lines(g, data, off, before=garbage * 3, after=garbage) == 0
        parts = [s.encode("utf-8") for s in mix_lines()[-40:] + odd_strings()]
        data, off = b"".join(parts), offsets_of(parts)
        for head in range(16):  # head bytes of garbage, the last one a lead byte
            before = ((garbage * 2)[:head - 1] + b"\xc3")[:head]
            assert len(before) == head
            assert expect_lines(g, data, off, before=before, after=b"\xf0\x9f") == 0
        assert expect_lines(g, b"", np.zeros(1, dtype=np.int64)) == 0  # an empty batch
        assert expect_lines(g, b"", np.zeros(1, dtype=np.int64), before=garbage, after=garbage) == 0
        # an Arrow slice: strings [a, b) of a column, its offsets as they are
        assert expect_lines(g, data[off[5]:off[30]], off[5:31] - off[5], before=data[:off[5]], after=data[off[30]:]) == 0


def test_pike_vm_fallback(monkeypatch):
    """Capture automata beyond the state limit: the simulated Pike VM reads the decoded text and its unit offsets."""
    names = "abcdefghi"
    ambiguous = "extract e {\n template " + ":".join("$%s(%%{[ab:]*})" % n for n in names) + "\n}\n"
    rng = np.random.default_rng(23)
    lines = ["".join(rng.choice(list("ab:::é"), size=rng.integers(0, 40))) for _ in range(3000)]
    monkeypatch.setenv("GORP_TDFA_MAX_STATES", "2")
    g = make_gorp(ambiguous, monkeypatch)
    parts = [s.encode("utf-8") for s in lines]
    assert expect_lines(g, b"".join(parts), offsets_of(parts), before=b"\xe9abc") == 0
    assert expect_text(g, utf8_of(lines)) == 0
    assert expect_text(g, utf8_of(lines, terminated=False), shift=16) == 0


# ---------------------------------------------------------------- 3. failures match the host forms
def test_failures_match_host_forms(monkeypatch):
    """Every malformed case of the host tests gives the host call's status and message; so do offsets below 0 and decreasing
    offsets; a d_text that is not 16-byte aligned is refused; after every failure the next call is correct."""
    g = make_gorp(V.README_DEF, monkeypatch)
    good_text = "[1]: GET 2ms /abc\n".encode("utf-8") * 300
    good = ["[1]: GET 2ms /abé", "中文\U0001F600", "x"] * 300
    gp = [s.encode("utf-8") for s in good]

    def still_right():
        assert expect_text(g, utf8_of(mix_lines()[-11:])) == 0
        assert expect_lines(g, b"".join(gp), offsets_of(gp), before=b"\x80") == 0

    for bad in BAD_SEQUENCES:
        assert expect_text(g, good_text + b"/x" + bad + b"y\n" + good_text) == _ffi.GORP_E_ARG
        assert expect_text(g, good_text + b"/x" + bad, shift=16) == _ffi.GORP_E_ARG
        for parts in (gp + [b"[2]: GET 2ms /x" + bad + b"y"] + gp, gp + [b"/x" + bad] + gp):
            assert expect_lines(g, b"".join(parts), offsets_of(parts), before=b"abc") == _ffi.GORP_E_ARG
        still_right()
    assert expect_text(g, b"a\xff\n") == _ffi.GORP_E_ARG
    split = ([b"x\xc3", b"\xa9y"], [b"x\xc3\xa9", b"\xa9y"], [b"\xf0", b"\x9f\x98\x80"], [b"a\xf0\x9f", b"\x98\x80"], [b"ab\xf0\x9f\x98", b"\x80"],
             [b"\xe4", b"", b"\xb8\xad"], [b"\x80abc"], [b"ab", b"c\xff"])
    for parts in split:
        parts = gp + parts + gp
        assert expect_lines(g, b"".join(parts), offsets_of(parts)) == _ffi.GORP_E_ARG
    for parts in (gp + [b"\xff"] + gp + [b"x\xe4", b"\xb8\xad"] + gp, gp + [b"x\xe4", b"\xb8\xad"] + gp + [b"\xff"] + gp):
        assert expect_lines(g, b"".join(parts), offsets_of(parts)) == _ffi.GORP_E_ARG
    still_right()
    # strings cut at random byte positions of well-formed text, and random corruption
    rng = np.random.default_rng(41)
    text = "".join(mix_lines()[-11:]).encode("utf-8")
    outcomes = set()
    for trial in range(60):
        cuts = np.sort(rng.choice(np.arange(1, len(text)), size=int(rng.integers(1, 40)), replace=False))
        off = np.concatenate(([0], cuts, [len(text)])).astype(np.int64)
        buf = bytearray(text)
        if trial % 3 == 0:
            buf[int(rng.integers(0, len(buf)))] = int(rng.choice([0x80, 0xbf, 0xc3, 0xe4, 0xf0, 0xff, 0x41]))
        outcomes.add(expect_lines(g, bytes(buf), off, before=b"\xc3" * (trial % 16)))
        outcomes.add(expect_text(g, bytes(buf[:int(cuts[0])]), shift=16 * (trial % 2)))
    assert outcomes == {0, _ffi.GORP_E_ARG}
    still_right()
    # offsets: the host check's messages, found on the device
    buf = b"[1]: GET 2ms /abc" * 40
    for off in ([-1, 4], [0, 10, 9, 20], [3, 2], [0, 5, 5, 700, 8, 9], [0, 20, 30, 10], [0, -5, 10], [5, 6, 7, 8, 1 << 40, 9, 10]):
        off = np.array(off, dtype=np.int64)
        hrc, hmsg, _ = host_lines(g, buf, off)
        assert hrc == _ffi.GORP_E_ARG and "offsets must" in hmsg
        t, ptr = placed(buf)
        rc, msg, _ = lines8_call(g, ptr, torch.from_numpy(off).to(DEV), len(off) - 1)
        assert (rc, msg) == (hrc, hmsg)
        still_right()
    # bases that are not 16-byte aligned
    t, ptr = placed(good_text)
    d_off = torch.from_numpy(offsets_of(gp)).to(DEV)
    for shift in (1, 2, 8):
        rc, msg, _ = text8_call(g, ptr + shift, 100)
        assert rc == _ffi.GORP_E_ARG and "16-byte aligned" in msg
        rc, msg, _ = lines8_call(g, ptr + shift, d_off, len(gp))
        assert rc == _ffi.GORP_E_ARG and "16-byte aligned" in msg
    still_right()


# ---------------------------------------------------------------- 4. the caller's bounds
def _cut_points(data):
    """Byte counts that cut the text: 16 consecutive ones (every residue mod 16) near the end, and m*4096 - 1, m*4096,
    m*4096 + 1 (the UTF-8 count tile) and the same around m*8192 (K1's tile) for the first and last two m."""
    k = data.rfind(b"\n", 0, len(data) - 200) + 1
    cuts = [k + 5 + j for j in range(16)]
    leads = [i for i, b in enumerate(data) if b >= 0xC2]
    for lead in (leads[len(leads) // 4], leads[len(leads) // 2], leads[-1]):  # inside a multi-byte sequence
        cuts += [lead + 1, lead + 2]
    for tile in (4096, 8192):
        ms = list(range(1, len(data) // tile))
        for m in ms[:2] + ms[-2:]:
            cuts += [tile * m - 1, tile * m, tile * m + 1]
    return sorted(set(cuts))


@pytest.mark.parametrize("d", [V.README_DEF, corpus.WEBLOG_DEF], ids=["readme", "weblog"])
def test_nothing_read_past_the_callers_bounds(d, monkeypatch):
    """The bytes inside a larger tensor, with poison that would change a result or fail validation if it were read: the rest
    of the cut line, '\\n' and whole matching lines, malformed bytes, the head of a multi-byte sequence. Text form: poison
    after n_bytes. Lines form: poison before d_off[0] and after d_off[n]. Results equal the host byte form on the exact
    bytes; a cut inside a multi-byte sequence fails exactly as the host call on the same bytes."""
    g = make_gorp(d, monkeypatch)
    data = utf8_of(mix_lines()[:400] + mix_lines()[-11:] + corpus.weblog_lines(300, seed=8))
    assert len(data) > 4 * 8192
    whole = "\n[1]: GET 2ms /x\n[2]: PUT 31ms /a\U0001F600b\n".encode("utf-8")
    outcomes = []
    for cut in _cut_points(data):
        exact = data[:cut]
        for poison in (data[cut:cut + 3000], whole * 20, b"\xff\x80\xbf", b"\xe4", b"\xf0\x9f\x98"):
            outcomes.append(expect_text(g, exact, shift=16 * (cut % 2), after=poison))
        # lines form: the lines before the cut and the cut line, without separators, between poison
        lines = exact.split(b"\n")
        lines = lines[-300:]
        off = offsets_of(lines)
        flat = b"".join(lines)
        for before in (data[:37] + lines[-1][:5], b"\xff" * 3, b"[1]: GET 2ms /x\xe4"):
            outcomes.append(expect_lines(g, flat, off, before=before, after=data[cut:cut + 3000]))
            outcomes.append(expect_lines(g, flat, off, before=before, after=b"\x80\xf4\x90"))
    assert 0 in outcomes and _ffi.GORP_E_ARG in outcomes  # (some cuts fall inside a sequence)


# ---------------------------------------------------------------- 5. streams, contexts, timing
def _kernel_times(g, dev_index, reset):
    names, tot = (C.c_char_p * 32)(), (C.c_double * 32)()
    cnt, calls, launches = C.c_int(), C.c_int64(), C.c_int64()
    assert _ffi.lib.gorp_kernel_times(g._eng(), dev_index, names, tot, 32, C.byref(cnt), C.byref(calls), C.byref(launches), reset) == 0
    return {names[i].decode() for i in range(cnt.value)}, calls.value


def test_streams_and_contexts(monkeypatch):
    """Calls on caller streams, alternating with gorp_extract_text_device on the same context (shared scratch); two contexts
    of one engine on one GPU; GORP_FLAG_TIME_KERNELS names the UTF-8 stages."""
    d = corpus.WEBLOG_DEF
    g = make_gorp(d, monkeypatch, devices=(0, 0))
    nb = n_bins(g)
    data = utf8_of(mix_lines())
    parts = [s.encode("utf-8") for s in mix_lines()]
    flat, off = b"".join(parts), offsets_of(parts)
    want_t = host_text(g, data)[2]
    want_l = host_lines(g, flat, off)[2]
    t8, p8 = placed(data)
    tl, pl = placed(flat, before=b"\xc3x")
    d_off = torch.from_numpy(off + 2).to(DEV)
    units = corpusgen.device_text("weblog", 0, 20000, DEV)
    want_u = fetch(_utf16_text(g, units, None, 0), nb, DEV)
    s1, s2 = torch.cuda.Stream(DEV), torch.cuda.Stream(DEV)
    for rep in range(3):
        for dev_index in (0, 1):
            st = (s1, s2)[(rep + dev_index) % 2]
            rc, msg, dres = text8_call(g, p8, len(data), stream=st, flags=0, dev_index=dev_index)
            assert rc == 0, msg
            fetch(dres, nb, DEV, stream=st).same_as(want_t)
            fetch(_utf16_text(g, units, (s2, s1)[(rep + dev_index) % 2], dev_index), nb, DEV, stream=(s2, s1)[(rep + dev_index) % 2]).same_as(want_u)
            rc, msg, dres = lines8_call(g, pl - 2, d_off, len(parts), stream=st, flags=0, dev_index=dev_index)
            assert rc == 0, msg
            fetch(dres, nb, DEV, stream=st).same_as(want_l, off_shift=2)
    torch.cuda.synchronize(DEV)
    for idx in (2, -1):
        assert text8_call(g, p8, len(data), dev_index=idx)[0] == _ffi.GORP_E_ARG
        assert lines8_call(g, pl, d_off, len(parts), dev_index=idx)[0] == _ffi.GORP_E_ARG
    # timed calls: the same rows, and the stage names
    _kernel_times(g, 0, reset=1)
    for _ in range(2):
        rc, msg, dres = text8_call(g, p8, len(data), flags=_ffi.FLAG_TIME_KERNELS | _ffi.FLAG_SYNC)
        fetch(dres, nb, DEV).same_as(want_t)
    names, calls = _kernel_times(g, 0, reset=1)
    assert calls == 2 and {"utf8_count", "utf8_decode", "utf8_nl_index", "utf8_rows", "k1_count_newlines"} <= names, names
    for _ in range(2):
        rc, msg, dres = lines8_call(g, pl - 2, d_off, len(parts), flags=_ffi.FLAG_TIME_KERNELS | _ffi.FLAG_SYNC)
        fetch(dres, nb, DEV).same_as(want_l, off_shift=2)
    names, calls = _kernel_times(g, 0, reset=1)
    assert calls == 2 and {"utf8_count", "utf8_line_units", "utf8_decode", "utf8_rows"} <= names, names
    # an empty text
    rc, msg, dres = text8_call(g, p8, 0)
    assert rc == 0 and dres.n_lines == 0 and (fetch(dres, nb, DEV).histogram == 0).all()


def test_host_call_after_an_unsynced_device_call(monkeypatch):
    """A UTF-8 device call left running on a side stream (no GORP_FLAG_SYNC, nothing fetched), then at once a host call on
    the same context: the host call's staging copies wait for the device call, which decodes into and stages through the
    same engine buffers. Each host call's rows equal those of the same call on a context that nothing else uses."""
    d = corpus.WEBLOG_DEF
    g = make_gorp(d, monkeypatch)
    ref = make_gorp(d, monkeypatch)
    lines = mix_lines()
    big_text = utf8_of(lines * 48)  # ~50 MB: the device call is still running when the host call starts
    parts = [s.encode("utf-8") for s in lines * 48]
    big_flat, big_off = b"".join(parts), offsets_of(parts)
    assert len(big_text) > 32 << 20
    t8, p8 = placed(big_text)
    tl, pl = placed(big_flat)
    d_off = torch.from_numpy(big_off).to(DEV)
    other = corpus.weblog_lines(3000, seed=5)  # the host calls' input: different lines, prepared before the device calls
    other_text, other_parts = utf8_of(other), [s.encode("utf-8") for s in other]
    other_flat, other_off = b"".join(other_parts), offsets_of(other_parts)
    other_units = np.frombuffer(("\n".join(other) + "\n").encode("utf-16-le"), dtype=np.uint16)
    host_calls = {
        "text_utf8_bytes": lambda e: host_text(e, other_text),
        "lines_utf8": lambda e: host_lines(e, other_flat, other_off),
        "text_utf16": lambda e: _host_rows(e, *_utf16_host_text(e, other_units)),
    }
    want = {k: f(ref)[2] for k, f in host_calls.items()}
    side = torch.cuda.Stream(DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))  # (the inputs were placed on the current stream)
    for rep in range(3):
        for k, f in host_calls.items():
            for form in ("text", "lines"):
                if form == "text":
                    rc, msg, _ = text8_call(g, p8, len(big_text), stream=side, flags=0)
                else:
                    rc, msg, _ = lines8_call(g, pl, d_off, len(parts), stream=side, flags=0)
                assert rc == 0, msg
                rc, msg, rows = f(g)
                assert rc == 0, msg
                rows.same_as(want[k])
    side.synchronize()
    # and the device calls still give their results after the host calls
    rc, msg, dres = text8_call(g, p8, len(big_text), stream=side, flags=0)
    assert rc == 0, msg
    fetch(dres, n_bins(g), DEV, stream=side).same_as(host_text(ref, big_text)[2])


def _utf16_host_text(g, units):
    res = _ffi.Result()
    rc = _ffi.lib.gorp_extract_text(g._eng(), units.ctypes.data, len(units), C.byref(res))
    return rc, res


def _utf16_text(g, units, stream, dev_index):
    dres = _ffi.DeviceResult()
    rc = _ffi.lib.gorp_extract_text_device(g._eng(), dev_index, units.data_ptr(), units.numel(), stream_handle(stream), 0, C.byref(dres))
    assert rc == 0, _ffi.last_error()
    return dres


# ---------------------------------------------------------------- 6. one launch past 2^32 bytes
def _clone(dres, nb):
    ext, off, sp, hist = device_views(dres, nb, DEV)
    return int(dres.n_lines), int(dres.span_stride), ext.clone(), off.clone(), sp.clone(), hist.clone()


def _same(a, b):
    assert a[0] == b[0] and a[1] == b[1]
    for x, y, what in zip(a[2:], b[2:], ("ext_id", "line_off", "spans", "histogram")):
        assert torch.equal(x, y), what


def test_one_launch_past_2_32_bytes(monkeypatch):
    """Config #2 (ASCII) at 72 M lines, 4.5 GB, generated on the device and narrowed to bytes there: the UTF-8 text form
    equals gorp_extract_text_device on the UTF-16 text bit for bit, and the UTF-8 lines form (the same lines without
    separators, int64 offsets) equals gorp_extract_lines_device; the first 1 M lines of both against the oracle."""
    name, n = "readme", 72_000_000
    d = corpus.CONFIGS[name][0]
    g = make_gorp(d, monkeypatch)
    nb = n_bins(g)
    u16 = corpusgen.device_text(name, 0, n, DEV)
    u8 = u16.to(torch.uint8)
    assert u8.numel() > (1 << 32) + (1 << 27) and int(u16.max()) < 0x80
    rc, msg, dres = text8_call(g, u8.data_ptr(), u8.numel())
    assert rc == 0, msg
    got = _clone(dres, nb)
    want = _clone(_utf16_text(g, u16, None, 0), nb)
    _same(got, want)
    assert got[0] == n and int(got[3][-1]) == u8.numel()
    # the oracle on a 1 M-line prefix
    w1 = 1_000_000
    text = corpusgen.host_text(name, 0, w1)
    prefix = window_histogram(window_rows(got[2], got[3], got[4], 0, w1), nb - 2)
    assert_matches_oracle(d, prefix, text=text)
    # the lines form: strings = lines without their '\n'
    line_off = want[3]
    del got, want
    del u8
    f16 = torch.cat([c[c != 10] for c in u16.split(1 << 28)])  # (in pieces: the index of one mask over GBs would be 8x its size)
    del u16
    f8 = f16.to(torch.uint8)
    off = line_off - torch.arange(n + 1, device=DEV, dtype=torch.int64)
    off[-1] = f8.numel()
    del line_off
    assert f8.numel() > (1 << 32)
    rc, msg, dres = lines8_call(g, f8.data_ptr(), off, n)
    assert rc == 0, msg
    got = _clone(dres, nb)
    d16 = _ffi.DeviceResult()
    st = torch.cuda.current_stream(DEV).cuda_stream
    assert _ffi.lib.gorp_extract_lines_device(g._eng(), 0, f16.data_ptr(), off.data_ptr(), n, st, FLAGS, C.byref(d16)) == 0, _ffi.last_error()
    _same(got, _clone(d16, nb))
    assert int(d16.d_line_off) == off.data_ptr() == int(dres.d_line_off)
    # ... and its prefix holds the text form's rows (checked against the oracle above)
    rows = window_histogram(window_rows(got[2], _text_offsets(got[3], w1), got[4], 0, w1), nb - 2)
    rows.same_as(prefix)


def _text_offsets(lines_off, w1):
    """Line offsets of the '\\n'-separated text from the offsets of the same lines without separators."""
    return lines_off[:w1 + 1] + torch.arange(w1 + 1, device=lines_off.device, dtype=torch.int64)
