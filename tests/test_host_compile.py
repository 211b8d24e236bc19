"""Host-side compile logic of the product (definition front-end, brics DFA product, JDK -> Pike program -> TDFA)
checked on the CPU: the tables libgorpcuda derives are interpreted by the test-only library tests/host/hosttest.cpp
and compared with the oracle. No compute call of the product runs here (there is no GPU)."""
import numpy as np
import pytest

from gorp_b200 import DefinitionParseException, DefinitionReader, UnsupportedDefinition
from oracle import frontend, gorp_oracle, jdkre
from tests import hostlib
from tests import reference_vectors as V

TRICKY_LINES = [
    "", "x", "[1]: GET 2ms /a", "[1]: GET 2ms /a\x0b", "[1]: GET 2ms /a\x08b", "[1]:\x0bGET 2ms /a",
    "[12]: PUT 5ms /\U0001F600/x", "[12]: POST 5ms /\ud83d", "[12]: HEAD 77ms /p\u0085q", "[12]: HEAD 77ms /p\u2028",
    "[12]: GET 5ms /\ud83d\ude00\ud83d", "[12]: GET 5ms /\ude00\ud83d\ude00", "[3]: PUT 1ms /x\r",
    "<1>ts (Accepted) ", "<1>t\x0bs (Accepted) ", "<1>\U00010000 (Accepted) \t ", "value=foobar",
    "[1]:  \t GET   2ms \t /a", "[1]: GETX 2ms /a", "[1]: get_1 2ms /a b", "[1]: GET 2ms ",
]

ALL_DEFS = [V.FULL_SIMPLE, V.FULL_INTERMEDIATE, V.FULL_FULL, V.PARAM_EXTRACTOR, V.PARAM_TEMPLATE, V.POLY_SIMPLE,
            V.POLY_INTERMEDIATE, V.POLY_QUOTED, V.POLY_COMPLEX, (V.README_DEF, []), (V.SIMPLE_GRP, [])]


def pack(lines):
    units = [np.asarray(jdkre.to_units(s), dtype=np.uint16) for s in lines]
    text = np.concatenate([np.concatenate((u, [10])) for u in units]).astype(np.uint16)
    starts, ends = gorp_oracle.split_lines(text)
    assert len(starts) == len(lines)
    return text, starts, ends


def compare_host_tables(definition, lines, fused=False, need_fused=True):
    g = DefinitionReader.reader(definition).read()
    o = gorp_oracle.Gorp(definition)
    text, starts, ends = pack(lines)
    G = max(len(x.extractor_names) for x in o.extractions)
    ext, spans, stats = hostlib.run(g.blob().bytes(), text, starts, ends, 2 * G, fused=fused)
    if ext is None:  # the one-pass automaton was refused for this definition (the two-pass tables still serve it)
        assert not need_fused, spans
        return stats
    oe, osp = o.extract_batch(text, (starts, ends), threads=1)
    bad = [i for i in range(len(lines)) if ext[i] != oe[i] or (spans[i] != osp[i]).any()]
    assert not bad, [(lines[i], int(ext[i]), int(oe[i]), spans[i].tolist(), osp[i].tolist()) for i in bad[:5]]
    return stats


@pytest.mark.parametrize("case", ALL_DEFS)
def test_tables_reproduce_oracle(case):
    compare_host_tables(case[0], [c[0] for c in case[1]] + TRICKY_LINES)


@pytest.mark.parametrize("name", ["weblog", "syslog200", "utf16mix"])
def test_config_definitions_reproduce_oracle(name):
    """Configs #3-#5 (gorp_b200/corpus.py): host tables vs oracle on generated lines + the tricky lines."""
    from gorp_b200 import corpus
    d, _ = corpus.CONFIGS[name]
    gen = {"weblog": corpus.weblog_lines, "syslog200": corpus.syslog200_lines, "utf16mix": corpus.utf16_mix_lines}[name]
    stats = compare_host_tables(d, gen(1200) + TRICKY_LINES, need_fused=False)
    if name == "syslog200":
        assert stats[0] * (stats[1] + 1) * 2 > 227 * 1024, "config #4's combined DFA must outgrow shared memory"


@pytest.mark.parametrize("case", ALL_DEFS)
def test_one_pass_automaton_reproduces_oracle(case):
    """host/fused.hpp: DFA x capture automata folded into one automaton, interpreted one table lookup per unit."""
    stats = compare_host_tables(case[0], [c[0] for c in case[1]] + TRICKY_LINES, fused=True)
    assert stats[0] == 1


def compare_fused_walk(definition, lines):
    """The fused walk's table (host/tails.hpp: build_fused_tailset -> TailImage), interpreted as kernels/tailwalk.cu walks it in
    "all" mode, against the oracle — text form ('\n'-separated) and List<String> form (a '\n' inside a string is content)."""
    g = DefinitionReader.reader(definition).read()
    o = gorp_oracle.Gorp(definition)
    G = max(len(x.extractor_names) for x in o.extractions)
    text, starts, ends = pack(lines)
    got = hostlib.run_fused_tail(g.blob().bytes(), text, starts, ends, 2 * G)
    if got is None:
        return False
    oe, osp = o.extract_batch(text, (starts, ends), threads=1)
    bad = [i for i in range(len(lines)) if got[0][i] != oe[i] or (got[1][i] != osp[i]).any()]
    assert not bad, [(lines[i], int(got[0][i]), int(oe[i]), got[1][i].tolist(), osp[i].tolist()) for i in bad[:5]]
    # List<String> form: strings that hold a '\n'
    withnl = [s for s in lines if s] + ["a\nb", "[1]: GET 2ms /a\n", "\n"]
    units = [np.asarray(jdkre.to_units(s), dtype=np.uint16) for s in withnl]
    off = np.zeros(len(withnl) + 1, dtype=np.int64)
    np.cumsum([len(u) for u in units], out=off[1:])
    flat = np.concatenate(units).astype(np.uint16)
    got = hostlib.run_fused_tail(g.blob().bytes(), flat, off[:-1], off[1:], 2 * G)
    oe, osp = o.extract_batch(flat, off, threads=1)
    bad = [i for i in range(len(withnl)) if got[0][i] != oe[i] or (got[1][i] != osp[i]).any()]
    assert not bad, [(withnl[i], int(got[0][i]), int(oe[i]), got[1][i].tolist(), osp[i].tolist()) for i in bad[:5]]
    return True


@pytest.mark.parametrize("case", ALL_DEFS)
def test_fused_walk_table_reproduces_oracle(case):
    assert compare_fused_walk(case[0], [c[0] for c in case[1]] + TRICKY_LINES)


@pytest.mark.parametrize("case", ALL_DEFS)
def test_exported_tables_are_the_reference_tables(case):
    """The blob holds Automata._alphabet/_transitions/_accept exactly as the oracle's restatement builds them."""
    g = DefinitionReader.reader(case[0]).read()
    a = gorp_oracle.Gorp(case[0]).matcher.automata
    cm, tr, af, al = g.blob().tables()
    assert g.blob().info()[:2] == (a.n_states, a.stride)
    assert (cm == a.alphabet).all() and (tr.reshape(-1) == a.transitions).all() and (af == a.accept_first).all()
    assert al == a.accept


@pytest.mark.parametrize("case", V.DERIVED_STRINGS)
def test_generated_strings(case):
    g = DefinitionReader.reader(case[0]).read()
    xs = g.getExtractions()
    assert len(xs) == len(case[1])
    for x, (name, autom, jdk, names) in zip(xs, case[1]):
        assert (x.getName(), x._automaton_source, x.getRegexpSource(), x.getExtractorNames()) == (name, autom, jdk, names)


@pytest.mark.parametrize("case", V.ERROR_KATS)
def test_definition_errors(case):
    with pytest.raises(DefinitionParseException) as ei:
        DefinitionReader.reader(case[0]).read()
    msg = str(ei.value).lower()
    for sub in case[1]:
        assert sub.lower() in msg, (sub, msg)


def test_append_and_names():
    g = DefinitionReader.reader("pattern %a a\ntemplate @base (%a:foo)\nextract rule1 {  \n"
                                "  template @base value=$MyValue(%a:%{\\w+})\n  append { \"enabled\" : true, \"x\" : 3 }\n}").read()
    x = g.getExtractions()[0]
    assert x.getExtra() == {"enabled": True, "x": 3}
    assert x.getRegexpSource() == "\\(a:foo\\)[ \t]+value=(a:\\w+)"
    assert x.getExtractorNames() == ["MyValue"]


UNSUPPORTED = [
    "pattern %p a\\b\nextract x {\n template %p\n}\n",          # \b: backspace vs word boundary (SURVEY D4)
    "pattern %p ^a\nextract x {\n template %p\n}\n",            # anchors (D5)
    "pattern %p a*+\nextract x {\n template %p\n}\n",           # possessive (D8)
    "pattern %p [a[b]]\nextract x {\n template %p\n}\n",        # nested class (D9)
    "pattern %p (a*)*\nextract x {\n template %p\n}\n",         # nullable loop body
]


@pytest.mark.parametrize("definition", UNSUPPORTED)
def test_unsupported_definitions_are_refused(definition):
    with pytest.raises(UnsupportedDefinition):
        DefinitionReader.reader(definition).read()
    with pytest.raises(jdkre.Unsupported):
        gorp_oracle.Gorp(definition)


FUZZ_PATTERNS = [
    # (definition body pattern pieces exercising ambiguity / priorities / counted repeats / lazy / alternation)
    "extract a {\n template $x(%{.*}) $y(%{.*})\n}\n",
    "extract a {\n template $x(%{.*}):$y(%{.*}):$z(%{.*})\n}\n",
    "extract a {\n template $x(%{[a-c]*})$y(%{[b-d]*})$z(%{[a-d]*})\n}\n",
    "extract a {\n template $x(%{(a|ab)})$y(%{(c|bcd)})$z(%{d*})\n}\n",
    "extract a {\n template $x(%{a{2,4}})$y(%{a{0,3}})$z(%{a*})\n}\n",
    "extract a {\n template $x(%{a*?})$y(%{a+?})$z(%{a*})\n}\n",
    "extract a {\n template $x(%{(ab|a)(bc|c)?})$y(%{[abc]*})\n}\n",
    "extract a {\n template $x(%{\\S+}) $y(%{\\S+( \\S+)*})\n}\n",
    "extract a {\n template $x(%{[^:]*}):$y(%{.{1,3}})$z(%{.*})\n}\n",
    "extract first {\n template $x(%{a+})b\n}\nextract second {\n template $x(%{[ab]+})\n}\nextract third {\n template $y(%{.*})\n}\n",
    "extract a {\n template $x(%{(a|b)*})$y(%{(ab)*})$z(%{b?a?})\n}\n",
    "extract a {\n template $o($i(%{a*})$j(%{b*}))$k(%{[ab]*})\n}\n",
]


@pytest.mark.parametrize("definition", FUZZ_PATTERNS)
def test_fused_walk_table_fuzz(definition):
    rng = np.random.default_rng(5)
    lines = ["".join(rng.choice(list("abcd: "), size=int(rng.integers(0, 9)))) for _ in range(400)]
    compare_fused_walk(definition, lines)


@pytest.mark.parametrize("definition", FUZZ_PATTERNS)
def test_fuzz_small_alphabet(definition):
    """Every string over a tiny alphabet up to length 7 (plus random longer ones): TDFA == backtracking oracle."""
    import itertools
    rng = np.random.default_rng(7)
    alpha = "abcd: "
    lines = ["".join(t) for n in range(0, 6) for t in itertools.product("abc:", repeat=n)]
    lines += ["".join(rng.choice(list(alpha), size=rng.integers(6, 24))) for _ in range(3000)]
    stats = compare_host_tables(definition, lines)
    assert stats[3] < 5000
    compare_host_tables(definition, lines, fused=True, need_fused=False)


def test_product_dfa_language_vs_component_dfas():
    """build_product == running every component DFA on its own (PolyMatcher.match semantics, all accept lists)."""
    from oracle import brics
    pats = V.MULTI_PATTERNS
    from gorp_b200 import Blob
    b = Blob.from_patterns(pats)
    cm, tr, af, al = b.tables()
    m = brics.PolyMatcher(pats)
    for s, want in V.MULTI_CASES:
        p = 0
        for c in jdkre.to_units(s):
            p = tr[p, cm[c]]
            if p < 0:
                break
        got = [] if p < 0 else al[p]
        assert got == want == m.match(jdkre.to_units(s)), s


def compare_walk_tables(definition, lines, drop_last_newline=False):
    """Tables of the big-definition text path (host/walktables.hpp: class-indexed DFA rows with SKIP / DEADSCAN / FIN,
    per-extraction capture images with SKIP / DEAD / SLOW / FRZ) interpreted the way the kernels walk them — both the
    shared-memory variant (no FRZ rows, highest id survives) and the L1/L2 variant — against the oracle."""
    g = DefinitionReader.reader(definition).read()
    o = gorp_oracle.Gorp(definition)
    text, starts, ends = pack(lines)
    if drop_last_newline:
        text = text[:-1]
    G = max(len(x.extractor_names) for x in o.extractions)
    oe, osp = o.extract_batch(text, (starts, ends), threads=1)
    for smem_variant in (True, False):
        r = hostlib.run_walk(g.blob().bytes(), text, 2 * G, smem_variant)
        assert r is not None
        ext, spans = r
        assert len(ext) == len(lines)
        bad = [i for i in range(len(lines)) if ext[i] != oe[i] or (spans[i] != osp[i][:2 * G]).any()]
        assert not bad, [(lines[i], int(ext[i]), int(oe[i]), spans[i].tolist(), osp[i].tolist()) for i in bad[:5]]


@pytest.mark.parametrize("case", ALL_DEFS)
def test_walk_tables_reproduce_oracle(case):
    lines = [c[0] for c in case[1]] + TRICKY_LINES
    compare_walk_tables(case[0], lines)
    compare_walk_tables(case[0], [s for s in lines if s] + ["[1]: GET 2ms /tail"], drop_last_newline=True)


@pytest.mark.parametrize("name", ["weblog", "syslog200", "utf16mix"])
def test_walk_tables_on_config_definitions(name):
    from gorp_b200 import corpus
    d, _ = corpus.CONFIGS[name]
    gen = {"weblog": corpus.weblog_lines, "syslog200": corpus.syslog200_lines, "utf16mix": corpus.utf16_mix_lines}[name]
    compare_walk_tables(d, gen(800) + TRICKY_LINES)


def compare_tails(definition, lines, drop_last_newline=False, need_tails=False):
    """The early-exit DFA table and the per-extraction tail automata (host/tails.hpp) interpreted the way K2b and the tail
    walk run them, against the oracle: same outcome (MISS / MATCH / CAPTURE_FAIL) and spans on every line."""
    g = DefinitionReader.reader(definition).read()
    o = gorp_oracle.Gorp(definition)
    text, starts, ends = pack(lines)
    if drop_last_newline:
        text = text[:-1]
    G = max(len(x.extractor_names) for x in o.extractions)
    oe, osp = o.extract_batch(text, (starts, ends), threads=1)
    r = hostlib.run_tails(g.blob().bytes(), text, 2 * G)
    if r is None:
        assert not need_tails
        return None
    ext, spans, stats = r
    assert len(ext) == len(lines)
    bad = [i for i in range(len(lines)) if ext[i] != oe[i] or (spans[i] != osp[i][:2 * G]).any()]
    assert not bad, [(lines[i], int(ext[i]), int(oe[i]), spans[i].tolist(), osp[i].tolist()) for i in bad[:5]]
    return stats


@pytest.mark.parametrize("case", ALL_DEFS)
def test_tail_automata_reproduce_oracle(case):
    lines = [c[0] for c in case[1]] + TRICKY_LINES
    compare_tails(case[0], lines)
    compare_tails(case[0], [s for s in lines if s] + ["[1]: GET 2ms /tail"], drop_last_newline=True)


@pytest.mark.parametrize("name", ["readme", "simple", "weblog", "syslog200", "utf16mix"])
def test_tail_automata_on_config_definitions(name):
    from gorp_b200 import corpus
    d, _ = corpus.CONFIGS[name]
    if name in ("readme", "simple"):
        text = corpus.CONFIGS[name][1](1500)
        lines = "".join(map(chr, text.tolist())).split("\n")[:-1]
    else:
        lines = {"weblog": corpus.weblog_lines, "syslog200": corpus.syslog200_lines, "utf16mix": corpus.utf16_mix_lines}[name](1500)
    stats = compare_tails(d, lines + TRICKY_LINES, need_tails=True)
    if name == "syslog200":  # the walk over the combined DFA stops after the app name: most lines leave it early
        assert stats[0] > 0.9 * len(lines) and stats[2] < 64, stats.tolist()


def test_tail_automata_fuzz_small_alphabet():
    rng = np.random.default_rng(5)
    for definition in FUZZ_PATTERNS:
        lines = ["".join(rng.choice(list("abcd: "), size=rng.integers(0, 24))) for _ in range(1500)]
        compare_tails(definition, lines)


def test_pike_vm_fallback_reproduces_oracle(monkeypatch):
    """Extractions whose determinisation exceeds the limits are not refused: their lines are decided by a simulated Pike
    VM (host/capture.hpp: PikeTables, kernels/pike.cu). With the state limit forced down to 2 EVERY extraction of every
    definition takes that path: same outcomes and spans as the oracle."""
    monkeypatch.setenv("GORP_TDFA_MAX_STATES", "2")
    for case in ALL_DEFS:
        compare_host_tables(case[0], [c[0] for c in case[1]] + TRICKY_LINES)
    rng = np.random.default_rng(13)
    for definition in FUZZ_PATTERNS:
        lines = ["".join(rng.choice(list("abcd: "), size=rng.integers(0, 24))) for _ in range(1200)]
        compare_host_tables(definition, lines)
    from gorp_b200 import corpus
    compare_host_tables(corpus.WEBLOG_DEF, corpus.utf16_mix_lines(600) + TRICKY_LINES)


def test_minimised_capture_automata_reproduce_oracle():
    """minimise_tdfa (Moore minimisation of the tagged automata, used for the tables of the bucketed capture walk) on every
    definition and fuzz pattern, including the small ones the engine leaves unminimised: same outcomes and spans."""
    lib = hostlib.load()
    lib.ht_set_force_minimise(1)
    try:
        for case in ALL_DEFS:
            compare_host_tables(case[0], [c[0] for c in case[1]] + TRICKY_LINES)
        rng = np.random.default_rng(3)
        for definition in FUZZ_PATTERNS:
            lines = ["".join(rng.choice(list("abcd: "), size=rng.integers(0, 24))) for _ in range(1500)]
            compare_host_tables(definition, lines)
    finally:
        lib.ht_set_force_minimise(0)
