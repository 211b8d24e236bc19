"""Parity tests proper: the CUDA path, called through the C ABI (gorp_b200.api -> libgorpcuda.so), against the
oracle on the same inputs. Bit-exact: same extraction index / MISS / capture failure per line, identical spans."""
import itertools

import numpy as np
import pytest

from gorp_b200 import DefinitionReader, ExtractionException, corpus
from oracle import gorp_oracle, jdkre
from tests import reference_vectors as V
from tests.test_host_compile import ALL_DEFS, FUZZ_PATTERNS, TRICKY_LINES

pytestmark = pytest.mark.gpu


def check_against_oracle(definition, text=None, lines=None, gorp=None):
    g = gorp or DefinitionReader.reader(definition).read()
    o = gorp_oracle.Gorp(definition)
    G = max(len(x.extractor_names) for x in o.extractions)
    if lines is not None:
        b = g.extract_batch_lines(lines)
        units = [np.asarray(jdkre.to_units(s), dtype=np.uint16) for s in lines]
        off = np.zeros(len(lines) + 1, dtype=np.int64)
        np.cumsum([len(u) for u in units], out=off[1:])
        flat = np.concatenate(units) if units else np.zeros(0, np.uint16)
        oe, osp = o.extract_batch(flat, off, threads=0)
        assert (b.line_off == off).all()
    else:
        b = g.extract_batch_text(text)
        starts, ends = gorp_oracle.split_lines(text)
        oe, osp = o.extract_batch(text, (starts, ends), threads=0)
        assert b.n_lines == len(starts)
        assert (b.line_off[:-1] == starts).all() and (b.line_off[1:] - 1 == ends).all()
    assert (b.ext_id == oe).all(), np.flatnonzero(b.ext_id != oe)[:10]
    # one fixed row of 2 * (widest extraction's groups) entries per line: 2*groups valid entries for a matched line,
    # -1 everywhere else (padding, MISS rows, capture-failed rows) -- exactly the oracle's layout
    assert b.span_stride == 2 * G and b.spans.shape == (b.n_lines, 2 * G)
    assert (b.spans == osp[:, :2 * G]).all(), np.flatnonzero((b.spans != osp[:, :2 * G]).any(axis=1))[:10]
    E = len(o.extractions)
    hist = np.zeros(E + 2, dtype=np.int64)
    np.add.at(hist, np.where(oe >= 0, oe, np.where(oe == -1, E, E + 1)), 1)
    assert (b.histogram == hist).all()
    return g, b, oe


# ---------------------------------------------------------------- the reference's own vectors through the GPU
@pytest.mark.parametrize("case", V.FULL_EXACT)
def test_reference_extract_vectors_exact(case):
    g = DefinitionReader.reader(case[0]).read()
    for s, want in case[1]:
        r = g.extract(s)
        assert r is not None and r.asMap("id") == want and r.getInput() == s


@pytest.mark.parametrize("case", V.FULL_SUBSET)
def test_reference_extract_vectors_subset(case):
    g = DefinitionReader.reader(case[0]).read()
    for s, want in case[1]:
        m = g.extract(s).asMap("id")
        for k, v in want.items():
            assert m[k] == v


@pytest.mark.parametrize("case", V.POLY_DSL)
def test_reference_polymatch_vectors(case):
    g = DefinitionReader.reader(case[0]).read()
    b = g.extract_batch_lines([s for s, _ in case[1]])
    for i, (_, want) in enumerate(case[1]):
        e = int(b.ext_id[i])
        assert (e if e >= -1 else -2 - e) == want[0]


def test_multipattern_first_accept():
    from gorp_b200 import Blob, Gorp
    g = Gorp(Blob.from_patterns(V.MULTI_PATTERNS))
    b = g.extract_batch_lines([s for s, _ in V.MULTI_CASES])
    assert b.ext_id.tolist() == [w[0] if w else -1 for _, w in V.MULTI_CASES]


def test_match_all_accept_lists():
    """gorp_match_all_lines: the full accept lists of PolyMatcher.match (reference MultiPatternTest.java:12-27 incl. the
    multi-accept cases {1,2} and {3,4}), and for a definition with overlapping extractions the oracle's lists."""
    from gorp_b200 import Blob, Gorp
    from oracle import brics
    g = Gorp(Blob.from_patterns(V.MULTI_PATTERNS))
    got = g.match_all([s for s, _ in V.MULTI_CASES])
    assert got == [list(w) for _, w in V.MULTI_CASES]
    assert any(len(w) > 1 for w in got)
    d = corpus.WEBLOG_DEF
    g3 = DefinitionReader.reader(d).read()
    o = gorp_oracle.Gorp(d)
    pm = brics.PolyMatcher([x.autom_source for x in o.extractions])
    lines = corpus.weblog_lines(1500, seed=6) + ["", "x"]
    got = g3.match_all(lines)
    want = [pm.match(jdkre.to_units(s)) for s in lines]
    assert got == want
    assert sum(len(w) > 1 for w in want) > 100  # CombinedGet and CombinedOther both accept a GET line
    assert g3.match_all([]) == []


def test_readme_sample_line_is_a_miss_and_exception_text():
    g = DefinitionReader.reader(V.README_DEF).read()
    assert g.extract("102456879: GET 123ms 200 /rest-service/v1/endpoint?foo=bar") is None
    # U+000B inside \S+ : DFA accepts, java.util.regex rejects -> ExtractionException (SURVEY D1)
    with pytest.raises(ExtractionException) as ei:
        g.extract("[1]: GET 2ms /a\x0bb")
    assert "Internal error: high-level match for extraction #1 (GetRequest) failed to match generated regexp: " in str(ei.value)
    assert g.extractSafe("[1]: GET 2ms /a\x0bb") is None
    rs = g.extractAll(["[1]: PUT 2ms /a", "nope", "[1]: HEAD 2ms /b"])
    assert [r.getId() if r else None for r in rs] == ["PutRequest", None, "OtherRequest"]


# ---------------------------------------------------------------- oracle parity on seeded inputs
@pytest.mark.parametrize("case", ALL_DEFS)
def test_tricky_lines_text_and_lines_form(case):
    lines = [c[0] for c in case[1]] + TRICKY_LINES
    g, _, _ = check_against_oracle(case[0], lines=lines)
    units = [np.asarray(jdkre.to_units(s), dtype=np.uint16) for s in lines]
    text = np.concatenate([np.concatenate((u, [10])) for u in units]).astype(np.uint16)
    check_against_oracle(case[0], text=text, gorp=g)


@pytest.mark.parametrize("definition", FUZZ_PATTERNS)
def test_fuzz_small_alphabet(definition):
    rng = np.random.default_rng(11)
    lines = ["".join(t) for n in range(0, 6) for t in itertools.product("abc:", repeat=n)]
    lines += ["".join(rng.choice(list("abcd: "), size=rng.integers(6, 40))) for _ in range(5000)]
    check_against_oracle(definition, lines=lines)


@pytest.mark.parametrize("name,n", [("simple", 300000), ("readme", 300000), ("weblog", 60000), ("syslog200", 60000),
                                    ("utf16mix", 60000)])
def test_config_corpora(name, n, monkeypatch):
    """The five BASELINE.json configs (prefixes the oracle finishes in seconds): #1 simple.grp, #2 README, #3 nginx /
    Apache definition with parametric templates, #4 200 extractions (combined DFA > shared memory, L2-resident
    table), #5 non-ASCII UTF-16 + divergence characters + 10 KB outliers."""
    d, gen = corpus.CONFIGS[name]
    text = gen(n)
    if name in ("weblog", "syslog200", "utf16mix"):  # the big-definition path with and without the early exit / tail automata
        for no_tails in ("0", "1"):
            if no_tails == "1":
                monkeypatch.setenv("GORP_NO_TAILS", "1")
            check_against_oracle(d, text=text)
            check_against_oracle(d, text=text[:-1])  # last line not terminated
        monkeypatch.delenv("GORP_NO_TAILS")
    _, b, oe = check_against_oracle(d, text=text)
    assert b.n_lines == n and (oe >= 0).sum() > n // 3
    if name == "utf16mix":
        assert (oe <= -2).sum() > 0, "config #5 must exercise the DFA-accepts / java.util.regex-rejects outcome"
        assert int(np.diff(b.line_off).max()) > 5000
    if name == "syslog200":
        assert len(set(oe[oe >= 0].tolist())) == 200


def test_edge_cases():
    g = DefinitionReader.reader(V.README_DEF).read()
    z = np.zeros(0, dtype=np.uint16)
    assert g.extract_batch_text(z).n_lines == 0
    assert g.extract_batch_lines([]).n_lines == 0
    for s in ["\n", "\n\n", "[1]: GET 2ms /a", "[1]: GET 2ms /a\n", "\n[1]: GET 2ms /a", "a\n\nb", "[1]: GET 2ms /a\r\n[1]: GET 2ms /a"]:
        check_against_oracle(V.README_DEF, text=np.asarray(jdkre.to_units(s), dtype=np.uint16), gorp=g)
    # List<String> form: strings may be empty or contain '\n' themselves (it is data there)
    check_against_oracle(V.README_DEF, lines=["", "[1]: GET 2ms /a\nb", "", "[1]: GET 2ms /a", ""], gorp=g)
    # a definition that accepts the empty line
    d = "extract e {\n template $x(%{a*})\n}\n"
    check_against_oracle(d, text=np.asarray(jdkre.to_units("\n\naa\n"), dtype=np.uint16))


def test_lines_form_rejects_decreasing_offsets():
    """gorp_extract_lines validates the caller's offsets on the host (GORP_E_ARG, never a CUDA fault): one-thread scan for
    small batches, split over threads from 2^20 lines on."""
    import ctypes as C
    from gorp_b200 import _ffi
    g = DefinitionReader.reader(V.README_DEF).read()
    for n, bad_at in ((10, 4), (1 << 21, 1_500_000)):
        text = np.full(n, ord("x"), dtype=np.uint16)
        off = np.arange(n + 1, dtype=np.int64)
        res = _ffi.Result()
        assert _ffi.lib.gorp_extract_lines(g._eng(), text.ctypes.data, off.ctypes.data, n, C.byref(res)) == 0
        assert res.n_lines == n
        _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
        off[bad_at + 1] = off[bad_at] - 1
        rc = _ffi.lib.gorp_extract_lines(g._eng(), text.ctypes.data, off.ctypes.data, n, C.byref(res))
        assert rc != 0 and ("line %d" % bad_at).encode() in _ffi.lib.gorp_last_error()
    off = np.asarray([-1, 0, 1], dtype=np.int64)
    assert _ffi.lib.gorp_extract_lines(g._eng(), text.ctypes.data, off.ctypes.data, 2, C.byref(res)) != 0


def test_long_and_ragged_lines():
    rng = np.random.default_rng(5)
    lines = []
    for k in range(400):
        n = int(rng.choice([0, 1, 7, 8, 9, 63, 64, 65, 1000, 5000, 10000]))
        path = "/" + "".join(rng.choice(list("abcdefghij0123456789/"), size=n))
        lines.append("[%d]: %s %dms %s" % (rng.integers(1, 10**9), rng.choice(["GET", "PUT", "POST", "x y"]), rng.integers(1, 999), path))
    lines.append("[1]: GET 2ms /" + "\U0001F600" * 3000)
    lines.append("[1]: GET 2ms /" + "a" * 9000 + " tail")
    check_against_oracle(V.README_DEF, lines=lines)
    check_against_oracle(V.README_DEF, text=np.concatenate(
        [np.concatenate((np.asarray(jdkre.to_units(s), dtype=np.uint16), [10])) for s in lines]).astype(np.uint16))


def test_non_ascii_divergence_corpus():
    """Config-5 style inputs: non-ASCII fields, surrogate pairs, lone surrogates, the DFA-vs-JDK divergence characters."""
    rng = np.random.default_rng(9)
    specials = ["\x0b", "\x08", "\u0085", "\u2028", "\u2029", "\r", "\ud83d", "\ude00", "\U0001F600", "\u00e9", "\u0416",
                "\u4e2d", "\U00010400", "\t", "\x0c"]
    lines = []
    for k in range(20000):
        path = list("/" + "".join(rng.choice(list("abcxyz012/"), size=rng.integers(3, 30))))
        for _ in range(rng.integers(0, 3)):
            path.insert(rng.integers(0, len(path) + 1), specials[rng.integers(0, len(specials))])
        lines.append("[%d]: %s %dms %s" % (rng.integers(1, 10**9), rng.choice(["GET", "PUT", "HEAD", "\u0416"]), rng.integers(1, 999), "".join(path)))
    _, b, oe = check_against_oracle(V.README_DEF, lines=lines)
    assert (oe <= -2).sum() > 100 and (oe == -1).sum() > 100 and (oe >= 0).sum() > 1000


def test_full_size_properties():
    """Config #2 at scale (tiling a seeded block): the results of a tiled corpus are the tiled results of the block."""
    d, gen = corpus.CONFIGS["readme"]
    block = gen(250000, seed=123)
    reps = 16
    g, b1, _ = check_against_oracle(d, text=block)
    big = np.tile(block, reps)
    b = g.extract_batch_text(big)
    assert b.n_lines == reps * b1.n_lines
    assert (b.histogram == reps * b1.histogram).all()
    assert (b.ext_id.reshape(reps, -1) == b1.ext_id[None, :]).all()
    assert (b.spans.reshape(reps, b1.n_lines, -1) == b1.spans[None, :, :]).all()
    assert (np.diff(b.line_off) > 0).all()


@pytest.mark.parametrize("name,n,reps", [("weblog", 40000, 40), ("syslog200", 40000, 40), ("utf16mix", 30000, 30)])
def test_full_size_properties_big_definitions(name, n, reps):
    """Configs #3-#5 at scale (1.2-1.6 M lines: many work items per extraction, many items per CTA): the results of a
    tiled corpus are the tiled results of the block, which is checked line by line against the oracle."""
    d, gen = corpus.CONFIGS[name]
    block = gen(n, seed=321)
    g, b1, _ = check_against_oracle(d, text=block)
    b = g.extract_batch_text(np.tile(block, reps))
    assert b.n_lines == reps * b1.n_lines
    assert (b.histogram == reps * b1.histogram).all()
    assert (b.ext_id.reshape(reps, -1) == b1.ext_id[None, :]).all()
    assert (b.spans.reshape(reps, b1.n_lines, -1) == b1.spans[None, :, :]).all()
    assert (np.diff(b.line_off).reshape(reps, -1) == np.diff(b1.line_off)[None, :]).all()


TIERS = {"k1_fusedwalk": {},
         "linewalk_capwalk_notails": {"GORP_FORCE_TWOPASS": "1", "GORP_NO_TAILS": "1"},
         "linewalk_tailwalk_flush1": {"GORP_FORCE_TWOPASS": "1", "GORP_TAIL_FLUSH": "1"},
         "linewalk_tailwalk512": {"GORP_FORCE_TWOPASS": "1", "GORP_TAIL_THREADS": "512"},
         "linewalk_cut_tailwalk384": {"GORP_FORCE_TWOPASS": "1", "GORP_TAIL_THREADS": "384"},
         "linewalk_capwalk": {"GORP_FORCE_TWOPASS": "1"},
         "linewalk_k4": {"GORP_FORCE_TWOPASS": "1", "GORP_FORCE_K4": "1"},
         "k1k2_capwalk": {"GORP_FORCE_TWOPASS": "1", "GORP_FORCE_K1K2": "1"},
         "twopass_fast": {"GORP_FORCE_TWOPASS": "1", "GORP_FORCE_K1K2": "1", "GORP_FORCE_K4": "1"},
         "general": {"GORP_FORCE_GENERAL": "1"}}
_TIER_ENV = ("GORP_FORCE_TWOPASS", "GORP_FORCE_GENERAL", "GORP_FORCE_K1K2", "GORP_FORCE_K4", "GORP_NO_TAILS", "GORP_TAIL_FLUSH",
             "GORP_TAIL_THREADS")


@pytest.mark.parametrize("tier", list(TIERS))
def test_every_kernel_tier_text_form(tier, monkeypatch):
    """The text form takes the fastest tier the definition allows; force each tier in turn (the engine reads the
    GORP_FORCE_* switches when it is created) and hold all of them to the same oracle."""
    for k in _TIER_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in TIERS[tier].items():
        monkeypatch.setenv(k, v)
    rng = np.random.default_rng(21)
    for name, n in (("simple", 60000), ("readme", 120000)):
        d, gen = corpus.CONFIGS[name]
        check_against_oracle(d, text=gen(n, seed=77))
    # dense, ragged and non-ASCII text: many short/empty lines (tiles with more line starts than threads), long lines
    specials = ["\\x0b", "\\x08", "", " ", "\\r", "\\ud83d", "\\ude00", "\\U0001F600", "\\u00e9", "\\u4e2d", "\\t"]
    specials = [s.encode("ascii").decode("unicode_escape") for s in specials]
    lines = []
    for k in range(30000):
        r = rng.random()
        if r < 0.3:
            lines.append("")
        elif r < 0.4:
            lines.append("x" * int(rng.integers(1, 4)))
        else:
            path = list("/" + "".join(rng.choice(list("abcxyz012/"), size=int(rng.choice([3, 10, 30, 200, 3000], p=[.3, .3, .3, .09, .01])))))
            for _ in range(rng.integers(0, 2)):
                path.insert(rng.integers(0, len(path) + 1), specials[rng.integers(0, len(specials))])
            lines.append("[%d]: %s %dms %s" % (rng.integers(1, 10**9), rng.choice(["GET", "PUT", "HEAD"]), rng.integers(1, 999), "".join(path)))
    text = np.concatenate([np.concatenate((np.asarray(jdkre.to_units(s), dtype=np.uint16), [10])) for s in lines]).astype(np.uint16)
    check_against_oracle(V.README_DEF, text=text)
    check_against_oracle(V.README_DEF, text=text[:-1])  # last line not terminated


def test_pike_vm_fallback(monkeypatch):
    """Capture automata that cannot be determinised within the limits are not refused: a simulated Pike VM decides their
    lines (kernels/pike.cu). The state limit is forced down so that (a) every extraction and (b) only the large ones of a
    definition take the fallback; text and List<String> form, every outcome, against the oracle."""
    names = "abcdefghi"
    ambiguous = "extract e {\n template " + ":".join("$%s(%%{[ab:]*})" % n for n in names) + "\n}\n"  # 9 groups, 2 812 states
    rng = np.random.default_rng(23)
    amb_lines = ["".join(rng.choice(list("ab:::"), size=rng.integers(0, 40))) for _ in range(3000)]
    for limit in ("2", "500"):
        monkeypatch.setenv("GORP_TDFA_MAX_STATES", limit)
        check_against_oracle(ambiguous, lines=amb_lines)
        check_against_oracle(ambiguous, text=corpus.lines_to_text(amb_lines))
        for d, lines in ((V.README_DEF, TRICKY_LINES + ["[1]: GET 2ms /" + "a" * 3000]), (corpus.WEBLOG_DEF, corpus.utf16_mix_lines(1500, seed=4))):
            check_against_oracle(d, lines=lines)
            check_against_oracle(d, text=corpus.lines_to_text(lines))
            monkeypatch.setenv("GORP_FORCE_TWOPASS", "1")
            check_against_oracle(d, text=corpus.lines_to_text(lines))
            monkeypatch.delenv("GORP_FORCE_TWOPASS")


def test_tail_walk_very_long_lines(monkeypatch):
    """Lines of 65 000 units and more leave the 16-bit tail walk for the one-thread-per-line kernel with 32-bit positions;
    results stay exact (spans far beyond 65 535, non-ASCII content, a candidate that ends as MISS / CAPTURE_FAIL)."""
    monkeypatch.setenv("GORP_FORCE_TWOPASS", "1")  # the README definition would otherwise take the fused walk
    rng = np.random.default_rng(17)
    lines = corpus.weblog_lines(300, seed=8)
    body = "".join(rng.choice(list("abcdefghij0123456789/"), size=70000))
    lines += ["[1]: GET 2ms /" + body, "[2]: PUT 31ms /" + body * 3 + "\u00e9" + body, "[3]: GET 2ms /" + body + " tail",
              "[4]: HEAD 7ms /" + body[:64990], "[5]: GET 2ms /" + body + "\x0bq", "[6]: GET 2ms /" + "\U0001F600" * 40000]
    _, b, oe = check_against_oracle(V.README_DEF, text=corpus.lines_to_text(lines))
    assert int(b.spans.max()) > 65535 and (oe[-6:] >= 0).sum() >= 3
    check_against_oracle(corpus.WEBLOG_DEF, text=corpus.lines_to_text(lines))


def test_host_calls_pipelined_in_pieces(monkeypatch):
    """gorp_extract_text / gorp_extract_lines cut a batch into line-aligned pieces (H2D of the next piece overlaps the
    kernels and the D2H of the previous ones); tiny pieces here, so every seam, the row-capacity growth and the
    lines-form staging get exercised."""
    d, gen = corpus.CONFIGS["readme"]
    text = gen(50000, seed=5)
    for piece in ("1024", "70000", "1000000"):
        monkeypatch.setenv("GORP_PIECE_UNITS", piece)
        g, b, _ = check_against_oracle(d, text=text)
        check_against_oracle(d, text=text[:-1], gorp=g)
    monkeypatch.setenv("GORP_PIECE_UNITS", "3000")
    lines = corpus.weblog_lines(4000, seed=3) + ["", "x" * 9000, ""]
    check_against_oracle(corpus.WEBLOG_DEF, lines=lines)
    check_against_oracle(corpus.WEBLOG_DEF, text=corpus.lines_to_text(lines))


def test_latin1_text_form(monkeypatch):
    """gorp_extract_text_latin1: ISO-8859-1 bytes in, widened on the device; identical to the UTF-16 call on the
    zero-extended text and to the oracle (including pieces whose seams fall anywhere in the byte buffer)."""
    rng = np.random.default_rng(31)
    for name, n in (("readme", 50000), ("weblog", 8000)):
        d, gen = corpus.CONFIGS[name]
        text = gen(n, seed=11)
        assert int(text.max()) < 256
        # sprinkle Latin-1 supplement characters (and the divergence characters that fit a byte: VT, BS, NEL, CR)
        text = text.copy()
        pos = rng.integers(0, len(text), size=n // 4)
        pos = pos[text[pos] != 10]
        text[pos] = rng.choice(np.array([0xE9, 0xFC, 0xA0, 0x85, 0x0B, 0x08, 0x0D, 0xFF], dtype=np.uint16), size=len(pos))
        for piece in (None, "5000"):
            if piece:
                monkeypatch.setenv("GORP_PIECE_UNITS", piece)
            g, b16, oe = check_against_oracle(d, text=text)
            for t in (text, text[:-1]):
                b16 = g.extract_batch_text(t)
                b8 = g.extract_batch_text_latin1(t.astype(np.uint8))
                assert b8.n_lines == b16.n_lines and b8.span_stride == b16.span_stride
                assert (b8.ext_id == b16.ext_id).all() and (b8.line_off == b16.line_off).all()
                assert (b8.spans == b16.spans).all() and (b8.histogram == b16.histogram).all()
        monkeypatch.delenv("GORP_PIECE_UNITS", raising=False)
    g = DefinitionReader.reader(V.README_DEF).read()
    assert g.extract_batch_text_latin1(b"").n_lines == 0
    assert g.extract_batch_text_latin1(b"[1]: GET 2ms /a").ext_id.tolist() == [1]


def test_fused_walk_launch_times_are_stable(monkeypatch):
    """Round 1 found the chunk-owner one-pass kernel of that time bistable (11.5 or 17.4 ms per launch, depending on unrelated
    allocation sizes). Every launch of a series of the default path of small definitions (K1 + fused walk) must run at the
    same speed whatever the sizes of the result allocations are: the row arrays are padded by 0 / 64 K / 1 M rows
    (GORP_PAD_ROWS shifts every allocation that follows), 25 launches each."""
    import ctypes as C
    import torch
    from gorp_b200 import _ffi, corpusgen
    from gorp_b200.api import Blob, _check
    dev = torch.device("cuda", 0)
    d_text = corpusgen.device_text("readme", 0, 12_000_000, dev)
    blob = Blob.from_definition(V.README_DEF)
    times = {}
    for pad in ("0", "65536", "1048576"):
        monkeypatch.setenv("GORP_PAD_ROWS", pad)
        eng = C.c_void_p()
        _check(_ffi.lib.gorp_engine_create(blob._ptr, blob.length, None, 0, C.byref(eng)))
        dres = _ffi.DeviceResult()
        stream = torch.cuda.current_stream().cuda_stream
        ms = []
        for k in range(28):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _check(_ffi.lib.gorp_extract_text_device(eng, 0, d_text.data_ptr(), d_text.numel(), stream, 0, C.byref(dres)))
            e1.record()
            torch.cuda.synchronize()
            if k >= 3:
                ms.append(e0.elapsed_time(e1))
        assert dres.n_lines == 12_000_000
        _ffi.lib.gorp_engine_destroy(eng)
        times[pad] = ms
    allms = [t for v in times.values() for t in v]
    assert max(allms) < 1.2 * min(allms), {k: (round(min(v), 3), round(max(v), 3)) for k, v in times.items()}


def test_concurrent_calls_on_one_engine(monkeypatch):
    """include/gorp_cuda.h promises that concurrent gorp_extract_* calls on one engine are allowed (the reference's Gorp is
    immutable and "fully thread-safe", Gorp.java:22): 4 threads x several calls each, text and lines form mixed, every
    result identical to the sequential one."""
    import threading
    monkeypatch.setenv("GORP_PIECE_UNITS", "60000")  # several pieces per call: the pipelined path with its shared buffers
    jobs = []
    for name, n in (("readme", 30000), ("weblog", 4000)):
        d, gen = corpus.CONFIGS[name]
        g = DefinitionReader.reader(d).read()
        texts = [gen(n, seed=50 + k) for k in range(4)]
        want = [g.extract_batch_text(t) for t in texts]
        jobs.append((g, texts, want))
    errors = []

    def worker(k):
        try:
            for rep in range(3):
                for g, texts, want in jobs:
                    t = texts[(k + rep) % 4]
                    w = want[(k + rep) % 4]
                    b = g.extract_batch_text(t) if (k + rep) % 2 == 0 else g.extract_batch_text_latin1(t.astype(np.uint8))
                    assert b.n_lines == w.n_lines and (b.ext_id == w.ext_id).all() and (b.spans == w.spans).all()
                    assert (b.line_off == w.line_off).all() and (b.histogram == w.histogram).all()
        except Exception as ex:  # noqa: BLE001
            errors.append(repr(ex))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:3]


def test_utf8_text_form(monkeypatch):
    """gorp_extract_text_utf8: UTF-8 bytes in, decoded to UTF-16 on the device; identical to the UTF-16 call on the decoded
    text (1- to 4-byte sequences, pieces whose seams fall anywhere, last line unterminated); malformed input is refused."""
    lines = corpus.utf16_mix_lines(6000, seed=12)
    lines = [s for s in lines if not any(0xD800 <= ord(ch) <= 0xDFFF for ch in s)]  # lone surrogates have no UTF-8 form
    lines += ["", "\u00e9" * 40, "\u4e2d\u6587" * 30, "\U0001F600" * 25, "[1]: GET 2ms /\U00010400\u0416x", "x" * 5000 + "\u00e9"]
    text = "\n".join(lines) + "\n"
    for d in (corpus.WEBLOG_DEF, V.README_DEF):
        g = DefinitionReader.reader(d).read()
        for piece in (None, "3000", "70000"):
            if piece:
                monkeypatch.setenv("GORP_PIECE_UNITS", piece)
            for t in (text, text[:-1]):
                b16 = g.extract_batch_text(t)
                b8 = g.extract_batch_text_utf8(t.encode("utf-8"))
                assert b8.n_lines == b16.n_lines and b8.span_stride == b16.span_stride
                assert (b8.ext_id == b16.ext_id).all() and (b8.line_off == b16.line_off).all()
                assert (b8.spans == b16.spans).all() and (b8.histogram == b16.histogram).all()
            monkeypatch.delenv("GORP_PIECE_UNITS", raising=False)
        check_against_oracle(d, text=np.frombuffer(text.encode("utf-16-le"), dtype=np.uint16), gorp=g)
    g = DefinitionReader.reader(V.README_DEF).read()
    assert g.extract_batch_text_utf8(b"").n_lines == 0
    assert g.extract_batch_text_utf8("[1]: GET 2ms /\u00e9".encode("utf-8")).ext_id.tolist() == [1]
    good = "[1]: GET 2ms /abc\n".encode("utf-8") * 300
    for bad in (b"\xc0\xaf", b"\xed\xa0\x80", b"\xf4\x90\x80\x80", b"\x80", b"\xe4\xb8", b"\xf0\x9f\x98", b"\xff"):
        with pytest.raises(ValueError) as ei:
            g._eng()  # (engine exists)
            from gorp_b200 import _ffi
            import ctypes as C
            buf = np.frombuffer(good + b"/x" + bad + b"y\n" + good, dtype=np.uint8)
            res = _ffi.Result()
            rc = _ffi.lib.gorp_extract_text_utf8(g._eng(), buf.ctypes.data, len(buf), C.byref(res))
            if rc != 0:
                raise ValueError(_ffi.last_error())
            _ffi.lib.gorp_result_release(g._eng(), C.byref(res))
        assert "malformed UTF-8 at byte %d" % (len(good) + 2) in str(ei.value), (bad, str(ei.value))


def test_multi_device_engine(monkeypatch):
    """One engine over several GPUs: contiguous line-aligned ranges per device, rows concatenated in device order."""
    from gorp_b200 import _ffi
    n = _ffi.lib.gorp_device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    monkeypatch.setenv("GORP_PIECE_UNITS", "200000")
    d, gen = corpus.CONFIGS["readme"]
    g = DefinitionReader.reader(d).read(devices=list(range(n)))
    text = gen(120000, seed=9)
    check_against_oracle(d, text=text, gorp=g)
    check_against_oracle(d, text=text[:-1], gorp=g)
    b16, b8 = g.extract_batch_text(text), g.extract_batch_text_latin1(text.astype(np.uint8))  # the corpus is ASCII
    assert (b8.ext_id == b16.ext_id).all() and (b8.line_off == b16.line_off).all() and (b8.spans == b16.spans).all()
    assert (b8.histogram == b16.histogram).all()
    lines = corpus.weblog_lines(5000, seed=4)
    g3 = DefinitionReader.reader(corpus.WEBLOG_DEF).read(devices=list(range(n)))
    check_against_oracle(corpus.WEBLOG_DEF, lines=lines, gorp=g3)
    check_against_oracle(corpus.WEBLOG_DEF, text=corpus.lines_to_text(lines), gorp=g3)
    # two host threads x all devices on the same engine: a call keeps every participating device until its rows are out
    import threading
    want = g.extract_batch_text(text)
    errors = []

    def worker():
        try:
            for _ in range(4):
                b = g.extract_batch_text(text)
                assert (b.ext_id == want.ext_id).all() and (b.spans == want.spans).all() and (b.line_off == want.line_off).all()
        except Exception as ex:  # noqa: BLE001
            errors.append(repr(ex))
    ts = [threading.Thread(target=worker) for _ in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors[:3]
