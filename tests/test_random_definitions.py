"""Randomly generated definitions, together with lines they match, on every kernel tier and input form against the oracle.

The other parity tests run hand-picked definitions. Which kernels a definition reaches depends on its shape (extraction
count, group count, overlap, ambiguity): the fused walk, the two passes with tail automata, the bucketed capture walk with
its interleaved items and 512-thread tail walk, the one-line-per-thread capture kernel with its skip list, the Pike fix-up.
A seeded generator builds definitions of every such shape, and for each one the lines that exercise the kernels' edges:

  * every piece of a template (literals, separators, extractors over `\\d+ \\w+ \\S+ \\s+ . .* .+? [^:]* ...`, random regexes,
    nested groups, group-less `%{...}` and `%p` pieces, named patterns and templates) carries a sampler of strings it
    matches, so that a sampled line matches its extraction;
  * each sampled line is mutated once: U+000B / U+0008 inside a `\\S` / `\\s` run and U+0085 / U+2028 / '\\r' or an emoji
    under `.` (the DFA accepts, java.util.regex rejects: CAPTURE_FAIL), a lone surrogate, one unit dropped or doubled;
  * empty lines, lengths of every residue mod 32, surrogate pairs across 16-unit block edges, lines of more than 65 000 units,
    and for the List<String> form strings that contain '\\n'.

The CPU part holds the generator to outcome quotas, pins the population to both sides of every table layout switch
(tests/host/hosttest.cpp: ht_layout), and runs every definition through the CPU interpreters of the tables against the
oracle, which separates a table bug from a kernel bug. The GPU part runs every definition through every tier, the Pike
fallback, the byte forms and the device-resident calls, counts which capture kernels ran, and runs the definitions with the
most extractions at 2 M lines.
"""
import functools
import re

import numpy as np
import pytest

from gorp_b200 import DefinitionReader, UnsupportedDefinition, _ffi
from oracle import gorp_oracle, jdkre
from tests import hostlib
from tests.test_fuzz_partners import random_regex
from tests.test_gpu_parity import TIERS, _TIER_ENV, assert_matches_oracle
from tests.test_host_compile import TRICKY_LINES, pack

SEED = 20261022
# (how many definitions, extraction count range) per regime: the fused walk; two passes with tails or fused tables near the
# shared-memory bound; interleaved items and the 512-thread tail walk (>= 64 extractions)
REGIMES = ((18, 1, 4), (10, 8, 40), (5, 64, 120))
LONG = 65_500

# ---------------------------------------------------------------- pieces: DSL text + a sampler of strings they match
ASCII_S = "abcdefxyzABC0123456789/._-"
NON_ASCII = "éЖ中ü"
DOT_SAFE = ASCII_S + " :=" + NON_ASCII


def _chars(rng, alphabet, lo, hi):
    return "".join(rng.choice(list(alphabet), size=int(rng.integers(lo, hi + 1))))


def _s_run(rng, lo, hi):
    s = _chars(rng, ASCII_S + NON_ASCII, lo, hi)
    if s and rng.random() < 0.15:
        i = int(rng.integers(0, len(s) + 1))
        s = s[:i] + "\U0001F600" + s[i:]  # a surrogate pair inside \S+ (one code point, not whitespace in either dialect)
    return s


# regex -> (tag, sampler, filler alphabet for extending the segment or None). Tags name what a mutation may do to a segment.
ATOMS = {
    "\\d+": ("d", lambda r: _chars(r, "0123456789", 1, 6), "0123456789"),
    "\\w+": ("w", lambda r: _chars(r, "abcxyzQ_09", 1, 8), "abcxyz_09"),
    "\\S+": ("S", lambda r: _s_run(r, 1, 8), ASCII_S + NON_ASCII),
    "\\s+": ("s", lambda r: _chars(r, " \t", 1, 3), None),
    ".": ("dot1", lambda r: _chars(r, DOT_SAFE, 1, 1), None),
    ".*": ("dot", lambda r: _chars(r, DOT_SAFE, 0, 8), DOT_SAFE),
    ".+?": ("dot", lambda r: _chars(r, DOT_SAFE, 1, 8), DOT_SAFE),
    ".{2}": ("dotn", lambda r: _chars(r, DOT_SAFE, 2, 2), None),
    "[^:]*": ("neg", lambda r: _chars(r, ASCII_S + " =" + NON_ASCII, 0, 8), ASCII_S + NON_ASCII),
    "[a-c]{1,3}": ("abc", lambda r: _chars(r, "abc", 1, 3), None),
    "(GET|PUT|POST)": ("verb", lambda r: str(r.choice(["GET", "PUT", "POST"])), None),
}
CLEAN = ["\\d+", "\\w+", "[a-c]{1,3}", "(GET|PUT|POST)"]
AMBIGUOUS = "[a-z:]+"  # between ':' separators: the capture automaton copies registers (no tail automaton)
LAZY = {"\\d+": "\\d+?", "\\w+": "\\w*?", "\\S+": "\\S+?", ".*": ".*?"}
LITERALS = ["id", "k", "ms", "x", "GET", "é", "Ж", "中", "ab"]
SEPARATORS = [":", "=", "/", " "]


class Piece:
    """One template piece: DSL text, named patterns / templates it needs, groups it adds, and a sampler that returns a list of
    (tag, text) segments whose concatenation the piece matches."""

    def __init__(self, dsl, groups, sampler, decls=()):
        self.dsl, self.groups, self.sampler, self.decls = dsl, groups, sampler, list(decls)


def _segment(tag, fn):
    return lambda r: [(tag, fn(r))]


def _rr_sampler(rng, regex):
    """A sampler for a random_regex output: strings over its alphabet that Python's re (a backtracker of the same family as
    java.util.regex, which agrees with brics on this subset) fullmatches. None when none is found."""
    rx = re.compile(regex)
    found = sorted({s for s in ("".join(rng.choice(list("abc:"), size=int(rng.integers(0, 7)))) for _ in range(300)) if rx.fullmatch(s)})
    if not found:
        return None
    return lambda r: [("rr", found[int(r.integers(0, len(found)))])]


def separated(pieces):
    """`pieces` with a '=' after each `%p` / `@t` reference that is followed by more than a separator (it would read as a
    longer name)."""
    out = []
    for p in pieces:
        if out and re.search(r"[%@]\w+$", out[-1].dsl) and p.dsl[0] not in ":=/ ":
            out.append(Piece("=", 0, lambda r: [("lit", "=")]))
        out.append(p)
    return out


class Gen:
    """Seeded generator of definitions (gorp DSL) with per-extraction line samplers."""

    def __init__(self, rng, clean=False):
        self.rng = rng
        self.clean = clean  # every extractor over a class without ':' and followed by ':' (one-pass automata stay small)
        self.n_names = 0
        self.n_patterns = 0
        self.n_templates = 0

    def name(self):
        self.n_names += 1
        return "g%d" % self.n_names

    def regex_piece(self):
        """(regex DSL text, sampler) of one extractor body."""
        r = self.rng.random()
        if self.clean:
            k = CLEAN[int(self.rng.integers(0, len(CLEAN)))]
            return k, _segment(ATOMS[k][0], ATOMS[k][1])
        if r < 0.12:
            for _ in range(20):
                p = random_regex(self.rng, depth=1, top=False)
                if "{" in p and "}" not in p:
                    continue
                s = _rr_sampler(self.rng, p)
                if s is not None:  # (a template pastes the pattern as it is: a top-level '|' needs a group)
                    return "(%s)" % p if "|" in p else p, s
        keys = list(ATOMS)
        k = keys[int(self.rng.integers(0, len(keys)))]
        tag, fn, _ = ATOMS[k]
        if k in LAZY and self.rng.random() < 0.25:
            k = LAZY[k]
        return k, _segment(tag, fn)

    def extractor(self, with_groups):
        """An extractor piece: `$g(%{re})`, `$g(%p)` with `pattern %p re`, nested `$o($i(..)$j(..))`, or group-less
        `%{re}` / `%p`."""
        rng = self.rng
        if with_groups and rng.random() < 0.1:
            (a, sa), (b, sb) = self.regex_piece(), self.regex_piece()
            o, i, j = self.name(), self.name(), self.name()
            return Piece("$%s($%s(%%{%s})$%s(%%{%s}))" % (o, i, a, j, b), 3, lambda r: sa(r) + sb(r))
        body, s = self.regex_piece()
        decls = []
        if rng.random() < 0.25:
            self.n_patterns += 1
            ref = "%%p%d" % self.n_patterns
            decls.append("pattern %s %s" % (ref, body))
        else:
            ref = "%%{%s}" % body
        if with_groups and rng.random() < 0.8:
            return Piece("$%s(%s)" % (self.name(), ref), 1, s, decls)
        return Piece(ref, 0, s, decls)

    def literal(self):
        rng = self.rng
        if rng.random() < 0.5:
            sep = SEPARATORS[int(rng.integers(0, len(SEPARATORS)))]
            if sep == " ":  # a template space is `[ \t]+`
                return Piece(" ", 0, lambda r: [("ws", str(r.choice([" ", " ", "\t", "  "])))])
            return Piece(sep, 0, lambda r, t=sep: [("lit", t)])
        lit = LITERALS[int(rng.integers(0, len(LITERALS)))]
        return Piece(lit, 0, lambda r, t=lit: [("lit", t)])

    def ambiguous(self):
        n = self.name()
        return Piece(":$%s(%%{%s}):" % (n, AMBIGUOUS), 1, lambda r: [("lit", ":"), ("amb", _chars(r, "abz:", 1, 6)), ("lit", ":")])

    def body(self, n_pieces, with_groups):
        """A sequence of pieces; now and then a run of them moves into a named template referenced as `@t`."""
        rng = self.rng
        pieces = []
        if self.clean:
            for k in range(n_pieces):
                pieces += [self.extractor(with_groups) if rng.random() < 0.8 else self.literal(), Piece(":", 0, lambda r: [("lit", ":")])]
            return separated(pieces)
        for k in range(n_pieces):
            pieces.append(self.extractor(with_groups) if (k % 2 == 0) == (rng.random() < 0.8) else self.literal())
        if with_groups and rng.random() < 0.08:
            pieces.insert(int(rng.integers(0, len(pieces) + 1)), self.ambiguous())
        pieces = separated(pieces)
        i = int(rng.integers(0, max(len(pieces) - 1, 1)))
        if len(pieces) >= 2 and rng.random() < 0.15 and " " not in (pieces[i].dsl, pieces[i + 1].dsl):
            a, b = pieces[i], pieces[i + 1]
            self.n_templates += 1
            t = "@t%d" % self.n_templates
            decls = a.decls + b.decls + ["template %s %s%s" % (t, a.dsl, b.dsl)]
            pieces[i:i + 2] = [Piece(t, a.groups + b.groups, lambda r: a.sampler(r) + b.sampler(r), decls)]
        return pieces

    def definition(self, n_ext, no_groups=False):
        """(definition text, per-extraction piece lists). Extractions come in families that share a prefix of pieces (several
        stay alive to the end of a line); in many-extraction definitions every family starts with its own keyword."""
        rng = self.rng
        exts = []
        while len(exts) < n_ext:
            fam = min(int(rng.integers(1, 5)), n_ext - len(exts))
            prefix = self.body(int(rng.integers(0, 3)), not no_groups)
            if n_ext > 4:
                kw = "f%d" % len(exts)
                prefix = [Piece(kw, 0, lambda r, t=kw: [("lit", t)])] + prefix
            for _ in range(fam):
                exts.append(prefix + self.body(int(rng.integers(1, 5)), not no_groups))
        exts = [separated(p) for p in exts]
        for p in exts:  # a template line is trimmed: no whitespace piece at either end
            while p and p[-1].dsl == " ":
                p.pop()
            while p and p[0].dsl == " ":
                p.pop(0)
            if not p:
                p.append(Piece("x", 0, lambda r: [("lit", "x")]))
        decls, seen = [], set()
        out = []
        for i, pieces in enumerate(exts):
            for p in pieces:
                for d in p.decls:
                    if d not in seen:
                        seen.add(d)
                        decls.append(d)
            out.append("extract e%d {\n template %s\n}\n" % (i, "".join(p.dsl for p in pieces)))
        return "\n".join(decls) + "\n" + "".join(out), exts


# ---------------------------------------------------------------- lines
def sample(pieces, rng):
    return [seg for p in pieces for seg in p.sampler(rng)]


def mutate(segs, rng):
    """One mutation of a sampled line (a list of segments); returns the line."""
    segs = [list(s) for s in segs]
    kind = int(rng.integers(0, 6))

    def pick(tags):
        idx = [i for i, (t, _) in enumerate(segs) if t in tags]
        return idx[int(rng.integers(0, len(idx)))] if idx else None

    def insert(i, ch):
        t = segs[i][1]
        k = int(rng.integers(0, len(t) + 1))
        segs[i][1] = t[:k] + ch + t[k:]

    if kind == 0 and (i := pick(("S", "s"))) is not None:
        insert(i, str(rng.choice(["\x0b", "\x08"])))
    elif kind == 1 and (i := pick(("dot", "dot1", "dotn"))) is not None:
        ch = str(rng.choice(["\u0085", "\u2028", "\r"]))
        if segs[i][0] == "dot":
            insert(i, ch)
        else:
            segs[i][1] = ch + segs[i][1][1:]
    elif kind == 2 and (i := pick(("dot", "dot1", "dotn"))) is not None:
        if segs[i][0] == "dot":
            insert(i, "\U0001F600")
        else:  # `.` / `.{n}`: one java.util.regex character, two UTF-16 units
            segs[i][1] = "\U0001F600" + segs[i][1][1:]
    elif kind == 3:
        i = pick(("S", "dot", "neg"))
        if i is None:
            i = int(rng.integers(0, len(segs))) if segs else None
        if i is None:
            return str(rng.choice(["\ud83d", "\ude00"]))
        insert(i, str(rng.choice(["\ud83d", "\ude00"])))
    else:
        s = "".join(t for _, t in segs)
        if not s:
            return "x"
        k = int(rng.integers(0, len(s)))
        return s[:k] + s[k + 1:] if kind == 4 else s[:k + 1] + s[k:]
    return "".join(t for _, t in segs)


def _units(s):
    return len(jdkre.to_units(s))


def extend(segs, rng, extra):
    """The line of `segs` with `extra` more units in its first extensible segment (None when it has none)."""
    for i, (t, txt) in enumerate(segs):
        fill = {"d": "0123456789", "w": "abcxyz_09", "S": ASCII_S, "dot": DOT_SAFE, "neg": ASCII_S}.get(t)
        if fill:
            out = [s for _, s in segs]
            out[i] = txt + "".join(rng.choice(list(fill), size=extra))
            return "".join(out)
    return None


class Case:
    """One generated definition and its inputs: `lines` for the text form ('\\n'-separated), `strings` for the List<String>
    form (the same lines and some that hold '\\n'); `n_sampled` leading lines are sampled before mutation."""

    def __init__(self, index, definition, n_ext, no_groups, lines, n_sampled, strings):
        self.index, self.definition, self.n_ext, self.no_groups = index, definition, n_ext, no_groups
        self.lines, self.n_sampled, self.strings = lines, n_sampled, strings

    def __repr__(self):
        return "def%d(E=%d%s)" % (self.index, self.n_ext, ", no groups" if self.no_groups else "")


def make_lines(exts, rng, with_long):
    per = max(2, 120 // len(exts))
    sampled = [sample(p, rng) for p in exts for _ in range(per)]
    lines = ["".join(t for _, t in s) for s in sampled]
    n_sampled = len(lines)
    lines += [mutate(s, rng) for s in sampled]
    lines += ["", "", ""]
    # every residue of the line length mod 32 (and so mod 16)
    ext_lines = [s for s in sampled if extend(s, rng, 0) is not None]
    if ext_lines:
        base = ext_lines[int(rng.integers(0, len(ext_lines)))]
        L0 = _units(extend(base, rng, 0))
        for r in range(32):
            lines.append(extend(base, rng, (r - L0) % 32 + 32 * int(rng.integers(0, 2))))
    # surrogate pairs across a 16-unit block edge of the text form: the high surrogate at a text offset of 15 mod 16
    pos = sum(_units(s) + 1 for s in lines)
    for s in sampled[:6]:
        head = "".join(t for _, t in s)
        for tag, txt in s:
            if tag in ("S", "dot", "neg") and txt:
                before = "".join(t for _, t in s[:s.index((tag, txt))])
                k = (15 - (pos + _units(before) + 1)) % 16
                pad = "".join(rng.choice(list(ASCII_S), size=k))
                head = before + txt[:1] + pad + "\U0001F600" + "".join(t for _, t in s[s.index((tag, txt)):])[1:]
                break
        lines.append(head)
        pos += _units(head) + 1
    if with_long:
        long_src = [s for s in sampled if sum(1 for t, _ in s if t in ("S", "dot", "neg", "w", "d")) == 1]
        if long_src:
            s = long_src[int(rng.integers(0, len(long_src)))]
            long_line = extend(s, rng, LONG)
            lines += [long_line, long_line + "\x0b", long_line[:len(long_line) // 2]]
    lines += TRICKY_LINES[:6]
    strings = lines + [lines[0] + "\n" + lines[1], "\n", lines[2] + "\n", "\n" + lines[3]]
    return lines, n_sampled, strings


@functools.lru_cache(maxsize=None)
def population():
    rng = np.random.default_rng(SEED)
    cases = []
    for count, lo, hi in REGIMES:
        made = 0
        while made < count:
            g = Gen(rng, clean=rng.random() < (0.5 if hi <= 4 else 0.3))
            n_ext = int(rng.integers(lo, hi + 1))
            no_groups = len(cases) % 6 == 1 and hi <= 40  # whole definitions without a group
            definition, exts = g.definition(n_ext, no_groups)
            try:
                gorp_oracle.Gorp(definition)
                DefinitionReader.reader(definition).read()
            except (UnsupportedDefinition, jdkre.Unsupported):
                continue
            lines, n_sampled, strings = make_lines(exts, rng, with_long=len(cases) % 5 == 0)
            cases.append(Case(len(cases), definition, n_ext, no_groups, lines, n_sampled, strings))
            made += 1
    return cases


CASES = list(range(sum(r[0] for r in REGIMES)))


@functools.lru_cache(maxsize=None)
def blob(i):
    return DefinitionReader.reader(population()[i].definition).read().blob().bytes()


@functools.lru_cache(maxsize=None)
def layout(i):
    return hostlib.layout(blob(i))


@functools.lru_cache(maxsize=None)
def oracle_text(i):
    """(text, ext, spans) of the text form."""
    c = population()[i]
    text, starts, ends = pack(c.lines)
    oe, osp = gorp_oracle.Gorp(c.definition).extract_batch(text, (starts, ends), threads=0)
    return text, oe, osp


@functools.lru_cache(maxsize=None)
def oracle_strings(i):
    """(flat units, offsets, ext, spans) of the List<String> form."""
    c = population()[i]
    units = [np.asarray(jdkre.to_units(s), dtype=np.uint16) for s in c.strings]
    off = np.zeros(len(units) + 1, dtype=np.int64)
    np.cumsum([len(u) for u in units], out=off[1:])
    flat = np.concatenate(units)
    oe, osp = gorp_oracle.Gorp(c.definition).extract_batch(flat, off, threads=0)
    return flat, off, oe, osp


# ---------------------------------------------------------------- CPU
def test_sampler_outcome_quotas():
    """The generator makes lines that match: every sampled line is MATCH or CAPTURE_FAIL for some extraction, and over the
    population MATCH, MISS and CAPTURE_FAIL each have their share."""
    n = match = miss = fail = 0
    for i in CASES:
        c = population()[i]
        _, oe, _ = oracle_text(i)
        assert (oe[:c.n_sampled] != -1).all(), [c.lines[k] for k in np.flatnonzero(oe[:c.n_sampled] == -1)[:5]]
        n += len(oe)
        match += int((oe >= 0).sum())
        miss += int((oe == -1).sum())
        fail += int((oe <= -2).sum())
    print("lines %d: MATCH %.1f %%, MISS %.1f %%, CAPTURE_FAIL %.1f %%" % (n, 100 * match / n, 100 * miss / n, 100 * fail / n))
    assert match >= 0.25 * n and miss >= 0.10 * n and fail >= 0.02 * n, (n, match, miss, fail)


# minimum number of definitions on each side (yes, no) of each layout switch; the bucketed capture image is refused only at
# 63 tag registers (tests/test_table_limits.py: ambiguous31), which random definitions do not reach
LAYOUT_SIDES = {"fused_image": (3, 3), "tails": (3, 3), "capimg": (10, 0), "cap_fast": (3, 3)}


def test_layout_coverage():
    """The population reaches both sides of every table layout switch the kernels branch on, so that a change of the
    generator or of the table builders cannot quietly drop a path."""
    lays = [layout(i) for i in CASES]
    counts = {}
    for k in LAYOUT_SIDES:
        counts[k] = (sum(1 for x in lays if x[k]), sum(1 for x in lays if not x[k]))
    counts["stride0"] = (sum(1 for x in lays if x["stride"] == 0), sum(1 for x in lays if x["stride"] > 0))
    counts["ext>=64"] = (sum(1 for i in CASES if population()[i].n_ext >= 64), sum(1 for i in CASES if population()[i].n_ext < 64))
    counts["some_without_tail"] = (sum(1 for x in lays if x["tails"] and not all(x["tail"])), sum(1 for x in lays if x["tails"] and all(x["tail"])))
    print("definitions on each side (yes, no):", counts)
    for k, (yes, no) in LAYOUT_SIDES.items():
        assert counts[k][0] >= yes and counts[k][1] >= no, (k, counts[k])
    assert min(counts["stride0"]) >= 3 and min(counts["ext>=64"]) >= 4 and min(counts["some_without_tail"]) >= 2, counts


@pytest.mark.parametrize("i", CASES)
def test_cpu_interpreters_reproduce_oracle(i):
    """Every table the definition gets, interpreted on the CPU the way the kernels walk it, against the oracle: text form
    (with and without the final '\\n') and, for the fused walk, the List<String> form."""
    c = population()[i]
    b = blob(i)
    lay = layout(i)
    stride = lay["stride"]
    text, oe, osp = oracle_text(i)
    starts, ends = gorp_oracle.split_lines(text)
    runs = {"general": hostlib.run(b, text, starts, ends, stride)[:2]}
    if lay["fused"]:
        runs["fused"] = hostlib.run(b, text, starts, ends, stride, fused=True)[:2]
    if lay["fused_image"]:
        runs["fused_walk"] = hostlib.run_fused_tail(b, text, starts, ends, stride)
    if lay["capimg"]:
        for smem in (True, False):
            runs["walk_smem%d" % smem] = hostlib.run_walk(b, text, stride, smem)
    if lay["tails"]:
        runs["tails"] = hostlib.run_tails(b, text, stride)[:2]
    for k, (ext, spans) in runs.items():
        bad = np.flatnonzero((ext != oe) | (spans != osp[:, :stride]).any(axis=1))
        assert not len(bad), (k, [(c.lines[j], int(ext[j]), int(oe[j])) for j in bad[:3]])
    # the last line unterminated (a non-empty line: an empty unterminated last line is no line)
    cut = text[:-1] if text[-2] != 10 else text
    for k, r in (("walk", hostlib.run_walk(b, cut, stride, False) if lay["capimg"] else None),
                 ("tails", hostlib.run_tails(b, cut, stride) if lay["tails"] else None)):
        if r is not None:
            assert (r[0] == oe).all() and (r[1] == osp[:, :stride]).all(), k
    if lay["fused_image"]:
        flat, off, se, ssp = oracle_strings(i)
        ext, spans = hostlib.run_fused_tail(b, flat, off[:-1], off[1:], stride)
        assert (ext == se).all() and (spans == ssp[:, :stride]).all()


# ---------------------------------------------------------------- a definition without groups (fixed cases)
# A rule set that only classifies: no extraction has a group, so the result rows are empty (stride 0). The reference still
# runs Pattern.matcher(line).matches() for the extraction the DFA picks, and reports CAPTURE_FAIL when it fails: brics `\S`
# takes U+000B and `.` takes U+2028, java.util.regex takes neither (SURVEY D1).
ZERO_GROUPS = "pattern %w \\S+\nextract a {\n template id=%w\n}\nextract b {\n template %{\\S+}\n}\nextract c {\n template %{.*}\n}\n"
ZERO_LINES = ["a\x0bb", "id=a\x0bb", "id=ab", "x\u2028", "x y", "", "a\x0b", "id=\U0001F600\x0b", "ab", "\x0b", "é \u2028中", "a b\r"] * 40


def _zero_expect(lines):
    text, starts, ends = pack(lines)
    return text, gorp_oracle.Gorp(ZERO_GROUPS).extract_batch(text, (starts, ends), threads=0)


def test_zero_group_definition_tables():
    """The oracle and the CPU interpreters agree that the lines the JDK regex rejects are CAPTURE_FAIL."""
    text, (oe, osp) = _zero_expect(ZERO_LINES)
    assert osp.shape == (len(ZERO_LINES), 0)
    assert oe[:12].tolist() == [-3, -2, 0, 1, 2, 2, -3, -2, 1, -3, -4, -4]
    b = DefinitionReader.reader(ZERO_GROUPS).read().blob().bytes()
    starts, ends = gorp_oracle.split_lines(text)
    assert (hostlib.run(b, text, starts, ends, 0)[0] == oe).all()
    assert hostlib.layout(b)["stride"] == 0


def _engine(definition, monkeypatch, env):
    """A Gorp whose engine is created under `env` (the engine reads the switches when it is created)."""
    for k in _TIER_ENV + ("GORP_TDFA_MAX_STATES",):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    g = DefinitionReader.reader(definition).read()
    g._eng()
    return g


def _utf8_ok(s):
    try:
        s.encode("utf-8")
        return True
    except UnicodeEncodeError:  # a lone surrogate has no UTF-8 form
        return False


@pytest.mark.gpu
@pytest.mark.parametrize("tier", list(TIERS))
def test_zero_group_definition_every_tier(tier, monkeypatch):
    """CAPTURE_FAIL, not MATCH, for the lines the JDK regex rejects: text and List<String> form, UTF-8 byte forms."""
    from tests.test_utf8_byte_offsets import check_bytes_form
    from tests.test_utf8_lines import check_lines_form
    text, (oe, osp) = _zero_expect(ZERO_LINES)
    g = _engine(ZERO_GROUPS, monkeypatch, TIERS[tier])
    assert_matches_oracle(ZERO_GROUPS, g.extract_batch_text(text), text=text, expect=(oe, osp))
    assert_matches_oracle(ZERO_GROUPS, g.extract_batch_text(text[:-1]), text=text[:-1], expect=(oe, osp))
    assert_matches_oracle(ZERO_GROUPS, g.extract_batch_lines(ZERO_LINES), lines=ZERO_LINES, expect=(oe, osp))
    bu, _ = check_bytes_form(g, ("\n".join(ZERO_LINES) + "\n").encode("utf-8"))
    assert_matches_oracle(ZERO_GROUPS, bu, text=text, expect=(oe, osp))
    bu, _ = check_lines_form(g, ZERO_LINES)
    assert_matches_oracle(ZERO_GROUPS, bu, lines=ZERO_LINES, expect=(oe, osp))


# ---------------------------------------------------------------- GPU: every generated definition
PIKE_LIMITS = ("2", "40")  # every extraction / only the larger capture automata take the Pike fix-up


@pytest.mark.gpu
@pytest.mark.parametrize("i", CASES)
def test_every_tier_and_form(i, monkeypatch):
    """Text form (with and without the final '\\n') and List<String> form under every tier and under the Pike fallback;
    Latin-1 and UTF-8 byte forms; the device-resident calls at a 32-byte aligned base and at one that is only 16-byte
    aligned: all against the oracle."""
    import torch
    from tests.test_device_forms import fetch, lines_call, n_bins, text_call, to_device
    from tests.test_utf8_byte_offsets import check_bytes_form
    from tests.test_utf8_lines import check_lines_form
    c = population()[i]
    d = c.definition
    text, oe, osp = oracle_text(i)
    flat, off, se, ssp = oracle_strings(i)
    envs = [TIERS[t] for t in TIERS] + [{"GORP_TDFA_MAX_STATES": m} for m in PIKE_LIMITS] + \
           [{"GORP_TDFA_MAX_STATES": m, "GORP_FORCE_TWOPASS": "1"} for m in PIKE_LIMITS]
    for env in envs:
        g = _engine(d, monkeypatch, env)
        assert_matches_oracle(d, g.extract_batch_text(text), text=text, expect=(oe, osp))
        assert_matches_oracle(d, g.extract_batch_text(text[:-1]), text=text[:-1], expect=(oe, osp))  # (the last line is not empty)
        assert_matches_oracle(d, g.extract_batch_lines(c.strings), lines=c.strings, expect=(se, ssp))
    g = _engine(d, monkeypatch, {})
    # byte forms: the lines that have a Latin-1 / a UTF-8 form
    keep = [k for k, s in enumerate(c.lines) if all(ord(ch) < 256 for ch in s)]
    t1 = pack([c.lines[k] for k in keep])[0]
    assert_matches_oracle(d, g.extract_batch_text_latin1(t1.astype(np.uint8)), text=t1, expect=(oe[keep], osp[keep]))
    keep = [k for k, s in enumerate(c.lines) if _utf8_ok(s)]
    sub = [c.lines[k] for k in keep]
    t8 = pack(sub)[0]
    data = ("\n".join(sub) + "\n").encode("utf-8")
    for dd, tt in ((data, t8), (data[:-1], t8[:-1])):
        bu, _ = check_bytes_form(g, dd)
        assert_matches_oracle(d, bu, text=tt, expect=(oe[keep], osp[keep]))
    keep = [k for k, s in enumerate(c.strings) if _utf8_ok(s)]
    bu, _ = check_lines_form(g, [c.strings[k] for k in keep])
    assert_matches_oracle(d, bu, lines=[c.strings[k] for k in keep], expect=(se[keep], ssp[keep]))
    # device-resident calls
    dev = torch.device("cuda", 0)
    nb = n_bins(g)
    d_text = torch.zeros(len(text) + 64, dtype=torch.int16, device=dev)
    assert d_text.data_ptr() % 512 == 0
    for shift in (0, 8):  # 0 and 16 bytes past a 32-byte boundary (the latter takes K2 / K4)
        d_text.zero_()
        d_text[shift:shift + len(text)] = to_device(text, dev)
        assert_matches_oracle(d, fetch(text_call(g, d_text, len(text), unit_shift=shift), nb, dev), text=text, expect=(oe, osp))
    rows = fetch(lines_call(g, to_device(flat, dev), torch.from_numpy(off).to(dev), len(c.strings)), nb, dev)
    assert_matches_oracle(d, rows, lines=c.strings, expect=(se, ssp))


CAPTURE_KERNELS = ("k4c_fusedwalk", "k4c_tailwalk", "k4b_capwalk", "k4_tdfa_capture")


@pytest.mark.gpu
def test_capture_kernels_reached(monkeypatch):
    """gorp_kernel_times of the default device-resident text and lines calls, and of the text call under the forced Pike
    limit: how many definitions reached each capture kernel. Each must be reached by several."""
    import torch
    from tests.test_device_forms import lines_call, text_call, to_device
    from tests.test_table_limits import _kernel_times
    dev = torch.device("cuda", 0)
    flags = _ffi.FLAG_TIME_KERNELS | _ffi.FLAG_SYNC
    counts = {}

    def timed(g, call, key):
        _kernel_times(g)
        call()
        for k in _kernel_times(g):
            counts[(key, k)] = counts.get((key, k), 0) + 1

    for i in CASES:
        c = population()[i]
        text = oracle_text(i)[0]
        flat, off = oracle_strings(i)[:2]
        d_text, d_flat, d_off = to_device(text, dev), to_device(flat, dev), torch.from_numpy(off).to(dev)
        g = _engine(c.definition, monkeypatch, {})
        timed(g, lambda: text_call(g, d_text, len(text), flags=flags), "text")
        timed(g, lambda: lines_call(g, d_flat, d_off, len(c.strings), flags=flags), "lines")
        g = _engine(c.definition, monkeypatch, {"GORP_TDFA_MAX_STATES": "2"})
        timed(g, lambda: text_call(g, d_text, len(text), flags=flags), "pike")
    reached = {(f, k): counts.get((f, k), 0) for f in ("text", "lines") for k in CAPTURE_KERNELS}
    reached[("pike", "pike_fixup")] = counts.get(("pike", "pike_fixup"), 0)
    print("definitions per capture kernel:", reached)
    for k in CAPTURE_KERNELS:
        assert reached[("text", k)] >= 3, reached
    assert reached[("lines", "k4_tdfa_capture")] >= 3 and reached[("lines", "k4c_tailwalk")] >= 3, reached
    assert reached[("pike", "pike_fixup")] == len(CASES), reached


@pytest.mark.gpu
def test_most_extractions_at_scale(monkeypatch):
    """The three definitions with the most extractions over 2 M lines drawn from their inputs (no line of 65 000 units):
    many work items per CTA, many buckets. Text form, default tier, every line against the oracle."""
    for i in sorted(CASES, key=lambda k: -population()[k].n_ext)[:3]:
        d = population()[i].definition
        text, oe, osp = oracle_text(i)
        starts, ends = gorp_oracle.split_lines(text)
        short = np.flatnonzero(ends - starts < 1000)
        pick = short[np.random.default_rng(i).integers(0, len(short), size=2_000_000)]
        lens = (ends - starts + 1)[pick]
        first = np.concatenate(([0], np.cumsum(lens)[:-1]))
        big = text[np.repeat(starts[pick] - first, lens) + np.arange(int(lens.sum()))]
        g = _engine(d, monkeypatch, {})
        assert_matches_oracle(d, g.extract_batch_text(big), text=big, expect=(oe[pick], osp[pick]))
