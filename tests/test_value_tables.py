"""gorp_extract_tables_device: the values of the last device-resident extract call as one Arrow-layout table per extraction.

Every table is compared exactly with a torch reference built from the rows of the same call (nonzero(ext_id == e), the
span columns, lengths, cumsum, a gather from the caller's text in chunks of rows): row indexes, offsets, values, validity
bitmap with its padding, null counts, n_rows == histogram[e] and 64-byte alignment of every buffer. On a prefix of each
input the values are also held to the oracle's asMap(). The inputs run through all four device-resident calls."""
import ctypes as C

import numpy as np
import pytest
import torch

from gorp_b200 import _ffi, corpus, corpusgen, parityhash
from oracle import gorp_oracle, jdkre
from tests import reference_vectors as V
from tests.test_device_forms import device_views, make_gorp, n_bins
from tests.test_table_limits import groups_def, outcomes_def
from tests.test_utf8_byte_offsets import long_lines, mix_lines
from tests.test_utf8_device import placed
from tests.test_utf8_lines import odd_strings

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
FORMS = ("text16", "lines16", "text8", "lines8")


# ---------------------------------------------------------------- calls
def _st(stream):
    return (torch.cuda.current_stream(DEV) if stream is None else stream).cuda_stream


def tables_call(g, stream=None, flags=_ffi.FLAG_SYNC, dev_index=0):
    dt = _ffi.DeviceTables()
    rc = _ffi.lib.gorp_extract_tables_device(g._eng(), dev_index, _st(stream), flags, C.byref(dt))
    return rc, (_ffi.last_error() if rc else ""), dt


def _u16(s):
    return np.asarray(jdkre.to_units(s), dtype=np.uint16)


def _offsets(parts):
    off = np.zeros(len(parts) + 1, dtype=np.int64)
    np.cumsum([len(p) for p in parts], out=off[1:])
    return off


class Call:
    """One device-resident extract call on `lines`: `base` is the caller's buffer from the call's d_text on (int16 or uint8),
    `dres` its result, `keep` whatever must stay alive."""

    def __init__(self, g, form, lines=None, stream=None, flags=_ffi.FLAG_SYNC, text16=None, text8=None, before=b""):
        self.g, self.form = g, form
        dres = _ffi.DeviceResult()
        eng, st = g._eng(), _st(stream)
        if form == "text16":
            if text16 is None:
                text16 = torch.from_numpy(_u16("".join(s + "\n" for s in lines)).view(np.int16)).to(DEV)
            self.base, self.keep = text16, ()
            rc = _ffi.lib.gorp_extract_text_device(eng, 0, text16.data_ptr(), text16.numel(), st, flags, C.byref(dres))
        elif form == "lines16":
            parts = [_u16(s) for s in lines]
            flat = np.concatenate(parts + [np.zeros(8, np.uint16)])
            self.base = torch.from_numpy(flat.view(np.int16)).to(DEV)
            d_off = torch.from_numpy(_offsets(parts)).to(DEV)
            self.keep = (d_off,)
            rc = _ffi.lib.gorp_extract_lines_device(eng, 0, self.base.data_ptr(), d_off.data_ptr(), len(parts), st, flags, C.byref(dres))
        elif form == "text8":
            if text8 is None:
                text8 = "".join(s + "\n" for s in lines).encode("utf-8")
            if isinstance(text8, torch.Tensor):
                t, ptr = text8, text8.data_ptr()
                n = text8.numel()
            else:
                t, ptr = placed(text8)
                n = len(text8)
            self.base, self.keep = t[ptr - t.data_ptr():], (t,)
            rc = _ffi.lib.gorp_extract_text_utf8_device(eng, 0, ptr, n, st, flags, C.byref(dres))
        else:
            parts = [s.encode("utf-8") for s in lines]
            t, ptr = placed(b"".join(parts), 0, before, b"\xf0\x9f")
            base = ptr - len(before)
            d_off = torch.from_numpy(_offsets(parts) + len(before)).to(DEV)
            self.base, self.keep = t[base - t.data_ptr():], (t, d_off)
            rc = _ffi.lib.gorp_extract_lines_utf8_device(eng, 0, base, d_off.data_ptr(), len(parts), st, flags, C.byref(dres))
        assert rc == 0, _ffi.last_error()
        self.dres = dres
        self.unit_bytes = 2 if form.endswith("16") else 1


# ---------------------------------------------------------------- the reference
def _dev(ptr, shape, typestr):
    if int(np.prod(shape)) == 0:
        return torch.empty(shape, dtype={"<i8": torch.int64, "<i2": torch.int16, "|u1": torch.uint8}[typestr], device=DEV)
    return torch.as_tensor(parityhash.DeviceArray(ptr, shape, typestr), device=DEV)


def _aligned(ptr):
    assert ptr and int(ptr) % 64 == 0, hex(int(ptr or 0))


def _bits(v):
    """Arrow validity bytes (LSB first) of bool tensor v (length a multiple of 8 except at the end)."""
    n = v.numel()
    pad = torch.zeros((n + 7) // 8 * 8, dtype=torch.int32, device=v.device)
    pad[:n] = v.to(torch.int32)
    return (pad.view(-1, 8) << torch.arange(8, device=v.device, dtype=torch.int32)).sum(dim=1).to(torch.uint8)


def check_tables(call, dt, chunk=1 << 20):
    """Every table of `dt` against the torch reference over the rows of `call`. Returns the largest column (units)."""
    g = call.g
    E = n_bins(g) - 2
    ext, off, sp, hist = device_views(call.dres, E + 2, DEV)
    hist = hist.cpu().tolist()
    assert dt.n_tables == E and dt.unit_bytes == call.unit_bytes
    ts = "<i2" if call.unit_bytes == 2 else "|u1"
    blob = g.blob()
    largest = 0
    for e in range(E):
        t = dt.tables[e]
        n = int(t.n_rows)
        assert n == hist[e], (e, n, hist[e])
        _aligned(t.d_row)
        want_rows = torch.nonzero(ext == e).flatten()
        assert torch.equal(_dev(t.d_row, (n,), "<i8"), want_rows), e
        groups = blob.extraction(e)["n_groups"] if sp.shape[1] else 0
        assert t.n_columns == groups
        starts = off[want_rows]
        for k in range(groups):
            s, u = sp[want_rows, 2 * k].to(torch.int64), sp[want_rows, 2 * k + 1].to(torch.int64)
            valid = s >= 0
            ln = torch.where(valid, u - s, 0)
            want_off = torch.zeros(n + 1, dtype=torch.int64, device=DEV)
            torch.cumsum(ln, 0, out=want_off[1:])
            for p in (t.d_offsets[k], t.d_data[k], t.d_valid[k]):
                _aligned(p)
            assert torch.equal(_dev(t.d_offsets[k], (n + 1,), "<i8"), want_off), (e, k)
            assert int(t.null_count[k]) == int((~valid).sum()), (e, k)
            nbytes = (n + 7) // 8
            bitmap = _dev(t.d_valid[k], ((nbytes + 63) // 64 * 64,), "|u1")
            assert torch.equal(bitmap[:nbytes], _bits(valid)), (e, k)
            assert int(bitmap[nbytes:].count_nonzero()) == 0, (e, k)
            total = int(want_off[-1])
            largest = max(largest, total)
            data = _dev(t.d_data[k], (total,), ts)
            src0 = starts + torch.where(valid, s, 0)
            for a in range(0, n, chunk):
                b = min(a + chunk, n)
                o0, o1 = int(want_off[a]), int(want_off[b])
                if o1 == o0:
                    continue
                lc = ln[a:b]
                idx = torch.repeat_interleave(src0[a:b], lc) + torch.arange(o0, o1, device=DEV) - torch.repeat_interleave(want_off[a:b], lc)
                assert torch.equal(data[o0:o1], call.base[idx]), (e, k, a)
    return largest


def check_oracle(call, dt, definition, lines):
    """Table e, row r, column k == asMap()[name_k] of the line (None exactly at the nulls) on the given prefix of lines."""
    o = gorp_oracle.Gorp(definition)
    E = len(o.extractions)
    ext = device_views(call.dres, E + 2, DEV)[0][:len(lines)].cpu().numpy()
    row_of = {}
    for e in range(E):
        t = dt.tables[e]
        rows = _dev(t.d_row, (int(t.n_rows),), "<i8").cpu().numpy()
        for r, line in enumerate(rows):
            if line < len(lines):
                row_of[int(line)] = (e, r)
    cols = {}
    for i, line in enumerate(lines):
        want = None
        try:
            want = o.extract_map(line)
        except gorp_oracle.ExtractionError:
            pass
        if want is None:
            assert i not in row_of and ext[i] < 0
            continue
        e, r = row_of[i]
        names = o.extractions[e].extractor_names
        got = {}
        t = dt.tables[e]
        for k, nm in enumerate(names):
            if (e, k) not in cols:
                nrow = int(t.n_rows)
                cols[e, k] = (_dev(t.d_offsets[k], (nrow + 1,), "<i8").cpu().numpy(),
                              _dev(t.d_valid[k], ((nrow + 7) // 8,), "|u1").cpu().numpy())
            o_k, v_k = cols[e, k]
            if not (v_k[r // 8] >> (r % 8)) & 1:
                got[nm] = None
                continue
            a, b = int(o_k[r]), int(o_k[r + 1])
            raw = _dev(int(t.d_data[k]) + a * call.unit_bytes, (b - a,), "<i2" if call.unit_bytes == 2 else "|u1").cpu().numpy()
            got[nm] = raw.view(np.uint16).tobytes().decode("utf-16-le", "surrogatepass") if call.unit_bytes == 2 else raw.tobytes().decode("utf-8")
        assert got == {nm: want[nm] for nm in names}, (i, line[:80])


def run_all_forms(g, definition, lines, oracle_prefix=2000, before=b"\xe9abc"):
    for form in FORMS:
        call = Call(g, form, lines, before=before)
        rc, msg, dt = tables_call(g)
        assert rc == 0, msg
        check_tables(call, dt)
        if oracle_prefix:
            check_oracle(call, dt, definition, lines[:oracle_prefix])


# ---------------------------------------------------------------- inputs
def corpus_lines(name, n):
    text = corpusgen.host_text(name, 0, n)
    return text.tobytes().decode("utf-16-le", "surrogatepass").split("\n")[:n]


@pytest.mark.parametrize("name", ["readme", "weblog", "syslog200", "utf16mix", "simple"])
def test_config_corpora(name, monkeypatch):
    """About 200 k lines of each config through the four device-resident calls (utf16mix without its lone surrogates in the
    UTF-8 forms, which have no UTF-8 form)."""
    d = corpus.CONFIGS[name][0]
    g = make_gorp(d, monkeypatch)
    n = {"syslog200": 60_000, "utf16mix": 100_000}.get(name, 200_000)
    lines = corpus_lines(name, n)
    # the UTF-16 forms on the text as it is
    for form in ("text16", "lines16"):
        call = Call(g, form, lines)
        rc, msg, dt = tables_call(g)
        assert rc == 0, msg
        check_tables(call, dt)
        check_oracle(call, dt, d, lines[:1500])
    ok8 = [s for s in lines if not any(0xD800 <= ord(ch) <= 0xDFFF for ch in s)]
    for form in ("text8", "lines8"):
        call = Call(g, form, ok8)
        rc, msg, dt = tables_call(g)
        assert rc == 0, msg
        check_tables(call, dt)
        check_oracle(call, dt, d, ok8[:1500])


def test_line_mix(monkeypatch):
    """Empty lines, CAPTURE_FAIL lines, nested and empty groups, surrogate pairs, 70 000-unit lines; '\\n' inside strings of
    the lines forms (the text forms take the strings without it). (A group of the supported subset always participates
    (SURVEY.md, Appendix C.5), so no definition yields a (-1, -1) span: every bitmap here is all ones, and the test checks
    that null_count is 0.)"""
    nested = "extract n {\n template $o($i(%{[a-z]+})$j(%{[0-9]*}))=$c(%{\\S+})\n}\n"
    for d in (corpus.WEBLOG_DEF, V.README_DEF, nested):
        g = make_gorp(d, monkeypatch)
        lines = mix_lines()[-3000:] + long_lines() + ["", "abc=x", "abc12=y\U0001F600", "q=\x0b", "abc=a\x0bb", "=", "1=2"] * 3
        run_all_forms(g, d, lines, oracle_prefix=400)
        with_nl = lines[:500] + [s + "\n" + s for s in odd_strings()] + ["abc=x\nz", "[1]: GET 2ms /a\nb"]
        for form in ("lines16", "lines8"):
            call = Call(g, form, with_nl)
            rc, msg, dt = tables_call(g)
            assert rc == 0, msg
            check_tables(call, dt)


def test_unaligned_utf8_offsets(monkeypatch):
    """A UTF-8 lines call whose d_off[0] sits at every residue mod 16."""
    g = make_gorp(V.README_DEF, monkeypatch)
    lines = mix_lines()[-500:]
    for head in range(1, 16):
        call = Call(g, "lines8", lines, before=b"\xe4" * head)
        rc, msg, dt = tables_call(g)
        assert rc == 0, msg
        check_tables(call, dt)


@pytest.mark.parametrize("case", ["no_groups", "groups31", "outcomes400", "never_matched", "pike"])
def test_definitions(case, monkeypatch):
    """0 columns; a 31-group extraction; 400 extractions; extractions without rows; the Pike fallback under a forced state
    limit."""
    rng = np.random.default_rng(5)
    if case == "no_groups":
        d = "extract e {\n template abc\n}\nextract f {\n template x%{[0-9]+}\n}\n"
        lines = ["abc", "x12", "y", "", "abc"] * 200
    elif case == "groups31":
        d = groups_def(31)
        lines = [":".join("".join(rng.choice(list("abcxyz"), size=int(rng.integers(1, 6)))) for _ in range(31)) for _ in range(700)]
        lines += ["a:b", "", "é:" * 30 + "é"]
    elif case == "outcomes400":
        d = outcomes_def(400)
        lines = ["abc=%d" % i for i in rng.permutation(400)] * 3 + ["x=1", "", "abc=400", "zz=399"] * 50
    elif case == "never_matched":
        d = ("extract a {\n template never$x(%{[0-9]+})\n}\nextract b {\n template $y(%{[a-z]+})=$z(%{[0-9]+})\n}\n"
             "extract c {\n template zzz$w(%{[a-z]+})\n}\n")
        lines = ["ab=12", "x=1", "", "q"] * 300
    else:
        names = "abcdefghi"
        d = "extract e {\n template " + ":".join("$%s(%%{[ab:]*})" % n for n in names) + "\n}\n"
        monkeypatch.setenv("GORP_TDFA_MAX_STATES", "2")
        lines = ["".join(rng.choice(list("ab:::é"), size=int(rng.integers(0, 40)))) for _ in range(3000)]
    g = make_gorp(d, monkeypatch)
    # (the Python oracle is too slow for 400 extractions; test_table_limits pins those rows by construction)
    run_all_forms(g, d, lines, oracle_prefix=0 if case == "outcomes400" else 600)
    if case == "never_matched":
        rc, msg, dt = tables_call(g)
        for e in (0, 2):
            assert dt.tables[e].n_rows == 0
            assert _dev(dt.tables[e].d_offsets[0], (1,), "<i8").tolist() == [0]


# ---------------------------------------------------------------- errors and conventions
def test_source_rules(monkeypatch):
    """No prior call, a host call, gorp_match_all_lines, a failed device call in between: GORP_E_ARG. A second device call:
    the tables follow it. Two contexts on one GPU are independent. dev_index out of range is refused."""
    lines = mix_lines()[-300:]
    g = make_gorp(V.README_DEF, monkeypatch)
    rc, msg, _ = tables_call(g)
    assert rc == _ffi.GORP_E_ARG and "device-resident result" in msg
    Call(g, "text16", lines)
    assert tables_call(g)[0] == 0
    assert tables_call(g)[0] == 0  # a second tables call replaces the first
    # a host-form call
    units = _u16("".join(s + "\n" for s in lines))
    res = _ffi.Result()
    assert _ffi.lib.gorp_extract_text(g._eng(), units.ctypes.data, len(units), C.byref(res)) == 0
    _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
    assert tables_call(g)[0] == _ffi.GORP_E_ARG
    # gorp_match_all_lines
    Call(g, "text8", lines)
    parts = [_u16(s) for s in lines]
    flat, off = np.concatenate(parts), _offsets(parts)
    mres = _ffi.MatchResult()
    assert _ffi.lib.gorp_match_all_lines(g._eng(), flat.ctypes.data, off.ctypes.data, len(parts), C.byref(mres)) == 0
    _ffi.lib.gorp_match_result_release(g._eng(), C.byref(mres))
    assert tables_call(g)[0] == _ffi.GORP_E_ARG
    # a device call that fails (malformed UTF-8)
    Call(g, "text16", lines)
    t, ptr = placed(b"[1]: GET 2ms /a\xff\n")
    dres = _ffi.DeviceResult()
    assert _ffi.lib.gorp_extract_text_utf8_device(g._eng(), 0, ptr, 17, _st(None), _ffi.FLAG_SYNC, C.byref(dres)) == _ffi.GORP_E_ARG
    assert tables_call(g)[0] == _ffi.GORP_E_ARG
    # a second device call: the tables follow it
    Call(g, "text16", lines)
    second = Call(g, "lines8", lines[:100])
    rc, msg, dt = tables_call(g)
    assert rc == 0 and dt.unit_bytes == 1
    check_tables(second, dt)
    # two contexts on one GPU
    g2 = make_gorp(V.README_DEF, monkeypatch, devices=(0, 0))
    a = Call(g2, "text16", lines)
    dres = _ffi.DeviceResult()
    b8 = torch.from_numpy(np.frombuffer("".join(s + "\n" for s in lines[:50]).encode("utf-8"), dtype=np.uint8).copy()).to(DEV)
    assert _ffi.lib.gorp_extract_text_utf8_device(g2._eng(), 1, b8.data_ptr(), b8.numel(), _st(None), _ffi.FLAG_SYNC, C.byref(dres)) == 0
    rc, msg, dt = tables_call(g2, dev_index=0)
    assert rc == 0, msg
    check_tables(a, dt)
    rc, msg, dt1 = tables_call(g2, dev_index=1)
    assert rc == 0 and dt1.unit_bytes == 1 and dt1.tables[0].n_rows + dt1.tables[1].n_rows + dt1.tables[2].n_rows <= 50
    for bad in (-1, 2):
        assert tables_call(g2, dev_index=bad)[0] == _ffi.GORP_E_ARG


def test_stream_and_stage_times(monkeypatch):
    """A non-default stream (no GORP_FLAG_SYNC: the caller orders on the stream), and the stages in gorp_kernel_times."""
    g = make_gorp(corpus.WEBLOG_DEF, monkeypatch)
    lines = corpus_lines("weblog", 50_000)
    names = (C.c_char_p * 16)()
    ms = (C.c_double * 16)()
    n, calls, launches = C.c_int(), C.c_int64(), C.c_int64()

    def stages():
        assert _ffi.lib.gorp_kernel_times(g._eng(), 0, names, ms, 16, C.byref(n), C.byref(calls), C.byref(launches), 1) == 0
        return [names[i].decode() for i in range(n.value)]

    s = torch.cuda.Stream(DEV)
    with torch.cuda.stream(s):
        call = Call(g, "text8", lines, stream=s, flags=_ffi.FLAG_TIME_KERNELS)
        stages()  # (gorp_kernel_times leaves the result readable)
        rc, msg, dt = tables_call(g, stream=s, flags=_ffi.FLAG_TIME_KERNELS)
        assert rc == 0, msg
        check_tables(call, dt)
    s.synchronize()
    assert stages() == ["tables_rank", "tables_len", "tables_scan", "tables_gather"]


# ---------------------------------------------------------------- bench scale
@pytest.mark.parametrize("name,n,forms", [("readme", 130_000_000, ("text16", "text8")), ("syslog200", 40_000_000, ("text16",))])
def test_bench_scale(name, n, forms, monkeypatch):
    """Config #2 through the UTF-16 and the UTF-8 text calls, config #4 at 40 M lines. Config #2 runs at 130 M lines rather
    than its bench size: the `path` column of its largest table holds about 0.83 x 2^31 units per 100 M lines, and it must
    hold more than 2^31."""
    g = make_gorp(corpus.CONFIGS[name][0], monkeypatch)
    u16 = corpusgen.device_text(name, 0, n, DEV)
    largest = 0
    for form in forms:
        if form == "text16":
            call = Call(g, form, text16=u16)
        else:
            assert int(u16.max()) < 0x80
            call = Call(g, form, text8=u16.to(torch.uint8))
        rc, msg, dt = tables_call(g)
        assert rc == 0, msg
        largest = max(largest, check_tables(call, dt, chunk=1 << 22))
        del call, dt
        torch.cuda.empty_cache()
    if name == "readme":
        assert largest > 1 << 31, largest
