"""Definitions at the limits of the table encodings, on every kernel tier.

The kernels are built around fixed limits: result rows of up to 62 entries (31 groups), up to 32 tag registers in registers
and more in local memory (up to 62), tail / fused-walk tables of 10-bit row ids and 6-bit op slots, fused walks with hundreds
of outcomes. Each definition here sits just below or just above one of them:

  * one extraction with 1..31 ':'-separated groups (span strides 2..62), and one wide extraction mixed with narrow ones
    (rows padded with -1);
  * ambiguous groups ('[a-z:]+' between ':'), whose capture automata copy registers: no fused walk, no tails, 33-63 tag
    registers; at 63 the bucketed capture image is refused too and the one-line-per-thread capture kernel takes the lines;
  * 255 / 256 / 257 / 400 extractions of the shape `$x(%{[a-z]+})=I` (256 / 257 / 258 / 401 fused outcomes; the last
    one's table outgrows shared memory and takes two passes);
  * fused op slots at 61 / 62 (the 6-bit slot field with its dummy) and 63 (the fused image is refused).

The CPU part pins every definition to its side of each limit (tests/host/hosttest.cpp: ht_layout), so that a change of the
table builders cannot make the GPU part pass by moving a definition to another path, and runs the definitions through the
CPU interpreters of the tables against the oracle. The GPU part runs them under every tier of tests/test_gpu_parity.py in
text and List<String> form against the oracle, and checks from gorp_kernel_times which capture kernel the default path ran.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from gorp_b200 import DefinitionReader, _ffi
from oracle import gorp_oracle, jdkre
from tests import hostlib
from tests.test_gpu_parity import TIERS, _TIER_ENV, assert_matches_oracle
from tests.test_host_compile import pack


def groups_def(n, cls="[a-z]+"):
    return "extract e {\n template " + ":".join("$g%d(%%{%s})" % (i, cls) for i in range(n)) + "\n}\n"


def outcomes_def(n):
    return "".join("extract e%d {\n template $x(%%{[a-z]+})=%d\n}\n" % (i, i) for i in range(n))


# one 28-group extraction, then narrow ones (rows of the narrow ones are padded with -1 up to 56 entries); the last group of
# the wide one is \S+, whose DFA dialect accepts units java.util.regex rejects (CAPTURE_FAIL)
MIXED = (groups_def(27).replace("\n}\n", ":$g27(%{\\S+})\n}\n") +
         "extract n1 {\n template $a(%{[0-9]+})=$b(%{[a-z]+})\n}\nextract n2 {\n template #$a(%{[^#]*})\n}\n")
# 31 groups (61 op slots) and one more extraction that adds one op slot (62) or two (63)
SLOTS62 = groups_def(31) + "extract f {\n template =$y(%{x*})\n}\n"
SLOTS63 = groups_def(31) + "extract f {\n template $y(%{[0-9]+})=\n}\n"

# name -> (definition, expected layout fields, capture kernel of the default text-form path)
FUSED = "k4c_fusedwalk"
EDGE = {}
for _n in (1, 2, 7, 15, 16, 17, 28, 30, 31):
    EDGE["groups%d" % _n] = (groups_def(_n), dict(stride=2 * _n, max_regs=2 * _n - 1, fused=1, fused_slots=2 * _n - 1,
                                                  fused_image=1, capimg=1, cap_fast=int(2 * _n - 1 <= 30), tails=1), FUSED)
EDGE["mixed28"] = (MIXED, dict(stride=56, fused=1, fused_image=1, capimg=1, tails=1), FUSED)
for _n, _regs in ((16, 33), (20, 41), (31, 63)):
    EDGE["ambiguous%d" % _n] = (groups_def(_n, "[a-z:]+"), dict(stride=2 * _n, max_regs=_regs, fused=0, tails=0, cap_fast=0, pike=0,
                                                                capimg=int(_regs < 63)),
                                "k4b_capwalk" if _regs < 63 else "k4_tdfa_capture")
for _n in (255, 256, 257):
    EDGE["outcomes%d" % _n] = (outcomes_def(_n), dict(stride=2, fused=1, fused_outcomes=_n + 1, fused_image=1, tails=1), FUSED)
EDGE["outcomes400"] = (outcomes_def(400), dict(stride=2, fused=1, fused_outcomes=401, fused_image=1, tails=1), "k4c_tailwalk")
EDGE["slots62"] = (SLOTS62, dict(stride=62, fused=1, fused_slots=62, fused_image=1, tails=1), FUSED)
EDGE["slots63"] = (SLOTS63, dict(stride=62, fused=1, fused_slots=63, fused_image=0, tails=1), "k4c_tailwalk")

OUTCOME_DEFS = [k for k in EDGE if k.startswith("outcomes")]
SPLIT_DEFS = ["ambiguous31"]
ORACLE_DEFS = [k for k in EDGE if k not in OUTCOME_DEFS + SPLIT_DEFS]
FUSED_SMEM_LIMIT = 200 * 1024  # engine.cu: the fused walk's tables must leave room in shared memory


@functools.lru_cache(maxsize=None)
def blob(name):
    return DefinitionReader.reader(EDGE[name][0]).read().blob().bytes()


@functools.lru_cache(maxsize=None)
def layout(name):
    return hostlib.layout(blob(name))


# ---------------------------------------------------------------- inputs
def _n_groups(name):
    return layout(name)["stride"] // 2


def edge_lines(name, seed=0):
    """Lines for a definition of the ':'-separated group shape, or of the outcome-count shape."""
    rng = np.random.default_rng(seed)
    if name in OUTCOME_DEFS:
        n = int(name[len("outcomes"):])
        lines = ["abc=%d" % i for i in range(n)] + ["x=%d" % i for i in range(0, n, 7)]
        lines += ["abc=", "=1", "1=1", "abc=%d" % n, "ab=0x", "", "é=1", "a\U0001F600=2", "zz=%d" % (n - 1)] * 3
        order = rng.permutation(len(lines))
        return [lines[i] for i in order]
    G = _n_groups(name)
    alpha = "abcdefghijklmnopqrstuvwxyz"
    lines = []
    # identical lengths with len + 1 a multiple of 16: every lane of a warp ends in the same 16-unit iteration (the worst case
    # of K4b's row staging: 32 x stride entries); 8 warps' worth
    L = ((2 * G - 1) // 16 + 1) * 16 - 1
    for k in range(256):
        sizes = np.ones(G, dtype=np.int64)
        extra = L - (2 * G - 1)
        for _ in range(extra):
            sizes[rng.integers(0, G)] += 1
        lines.append(":".join("".join(rng.choice(list(alpha), size=int(s))) for s in sizes))
    assert all(len(s) == L for s in lines[:256])
    # ragged lines (every residue of the line start mod 16 and of line * stride mod 8 comes round), empty lines
    for k in range(600):
        r = rng.random()
        if r < 0.1:
            lines.append("")
            continue
        # ':' inside the groups of the ambiguous definitions (the oracle backtracks over where the groups split: not at 31 groups)
        amb = ":" if name.startswith("ambiguous") and G <= 20 else ""
        parts = ["".join(rng.choice(list(alpha + amb), size=int(rng.integers(1, 9)))) for _ in range(G)]
        if r < 0.2:  # a group too few or too many: MISS
            parts = parts[:-1] if rng.random() < 0.5 else parts + ["q"]
        elif r < 0.3:  # non-ASCII units and surrogate pairs inside a group
            i = int(rng.integers(0, G))
            parts[i] = parts[i] + rng.choice(["é", "中", "\U0001F600", "\ud83d", "\x0b", " "])
        elif r < 0.35:  # an upper-case letter: MISS
            parts[0] = "Q" + parts[0]
        lines.append(":".join(parts))
    if name == "mixed28":
        lines += ["12=abc", "7=x", "=abc", "#", "#anything é \U0001F600", "#\x0b", "1=" + "a" * 300]
        lines += [ln + "\x0bx" for ln in lines[:40]]  # \S+ (the last group) takes VT in the DFA dialect only: CAPTURE_FAIL
    if name.startswith("slots"):
        lines += ["=", "=xxx", "=12", "12=", "1=", "=1x", "x1="] * 5
    return lines


def expected_outcome_rows(name, lines):
    """Outcome-count definitions, by construction: `w=I` with w in [a-z]+ and I < n is extraction I with span (0, len(w)),
    anything else is MISS (the python oracle is too slow on hundreds of extractions)."""
    n = int(name[len("outcomes"):])
    ext = np.full(len(lines), -1, dtype=np.int32)
    spans = np.full((len(lines), 2), -1, dtype=np.int32)
    for i, s in enumerate(lines):
        w, eq, num = s.partition("=")
        if eq and w and all("a" <= ch <= "z" for ch in w) and num.isdigit() and str(int(num)) == num and int(num) < n:
            ext[i] = int(num)
            spans[i] = (0, len(w))
    return ext, spans


def expected_split_rows(G, lines):
    """An extraction of G ambiguous groups ('[a-z:]+' joined by ':') on lines without empty ':'-separated fields, by
    construction: a line of [a-z:] with n >= G fields matches; java.util.regex's greedy groups give the first n - G + 1
    fields to group 0 and one field to each later group. (The oracle backtracks over every split: too slow at 31 groups.)"""
    ext = np.full(len(lines), -1, dtype=np.int32)
    spans = np.full((len(lines), 2 * G), -1, dtype=np.int32)
    for i, s in enumerate(lines):
        fields = s.split(":")
        assert all(fields), s
        if len(fields) < G or any(not ("a" <= ch <= "z" or ch == ":") for ch in s):
            continue
        ends = np.cumsum([len(f) + 1 for f in fields]) - 1  # end of each field
        starts = ends - np.asarray([len(f) for f in fields])
        k0 = len(fields) - G
        ext[i] = 0
        spans[i, 0], spans[i, 1] = 0, ends[k0]
        for g in range(1, G):
            spans[i, 2 * g], spans[i, 2 * g + 1] = starts[k0 + g], ends[k0 + g]
    return ext, spans


@functools.lru_cache(maxsize=None)
def expected(name):
    """(lines, ext, spans) of a definition's input."""
    lines = edge_lines(name)
    if name in OUTCOME_DEFS:
        ext, spans = expected_outcome_rows(name, lines)
        return lines, ext, spans
    if name in SPLIT_DEFS:
        lines = [s for s in lines if s]  # (an empty line has an empty field)
        ext, spans = expected_split_rows(_n_groups(name), lines)
        return lines, ext, spans
    text, starts, ends = pack(lines)
    ext, spans = gorp_oracle.Gorp(EDGE[name][0]).extract_batch(text, (starts, ends), threads=0)
    return lines, ext, spans


# ---------------------------------------------------------------- CPU: layouts and table interpreters
@pytest.mark.parametrize("name", list(EDGE))
def test_layout_sides_of_the_limits(name):
    got = layout(name)
    want = EDGE[name][1]
    assert {k: got[k] for k in want} == want, got
    if name.startswith("outcomes"):  # every extraction keeps its tail; the 400-extraction table outgrows shared memory
        assert all(got["tail"]), got["tail"]
        assert (got["fused_table_bytes"] > FUSED_SMEM_LIMIT) == (name == "outcomes400"), got["fused_table_bytes"]
    elif got["fused_image"]:
        assert got["fused_table_bytes"] < FUSED_SMEM_LIMIT // 2


def test_limits_are_crossed():
    """The set as a whole reaches each limit from both sides."""
    regs = [layout(k)["max_regs"] for k in EDGE]
    strides = {layout(k)["stride"] for k in EDGE}
    assert {56, 60, 62} <= strides and any(32 < r < 63 for r in regs) and max(regs) >= 63 and 31 in regs
    assert {layout(k)["fused_outcomes"] for k in OUTCOME_DEFS} == {256, 257, 258, 401}
    assert {layout(k)["fused_slots"] for k in ("groups31", "slots62", "slots63")} == {61, 62, 63}


def test_outcome_lines_cover_every_extraction():
    for name in OUTCOME_DEFS:
        lines, ext, _ = expected(name)
        n = int(name[len("outcomes"):])
        assert set(ext.tolist()) == set(range(-1, n))


@pytest.mark.parametrize("name", ORACLE_DEFS)
def test_cpu_interpreters_reproduce_oracle(name):
    """The tables of every path the definition can take, interpreted on the CPU (tests/host/hosttest.cpp), against the oracle."""
    lines, oe, osp = expected(name)
    lay = layout(name)
    stride = lay["stride"]
    text, starts, ends = pack(lines)
    runs = {"general": hostlib.run(blob(name), text, starts, ends, stride)[:2]}
    if lay["fused"]:
        runs["fused"] = hostlib.run(blob(name), text, starts, ends, stride, fused=True)[:2]
    if lay["fused_image"]:
        runs["fused_walk"] = hostlib.run_fused_tail(blob(name), text, starts, ends, stride)
    if lay["capimg"]:
        for smem in (True, False):
            runs["walk_smem%d" % smem] = hostlib.run_walk(blob(name), text, stride, smem)
    if lay["tails"]:
        runs["tails"] = hostlib.run_tails(blob(name), text, stride)[:2]
    for k, (ext, spans) in runs.items():
        assert (ext == oe).all(), (k, np.flatnonzero(ext != oe)[:10])
        assert (spans == osp[:, :stride]).all(), (k, np.flatnonzero((spans != osp[:, :stride]).any(axis=1))[:10])
    assert (oe >= 0).sum() > len(lines) // 3 and (oe == -1).sum() > 10
    if name == "mixed28":
        assert (oe <= -2).sum() > 10


def test_split_rule_is_the_oracle():
    """The construction of expected_split_rows agrees with the oracle on 16 ambiguous groups (lines with ':' inside groups)."""
    lines = [s for s in edge_lines("ambiguous16") if s and "" not in s.split(":")]
    ext, spans = expected_split_rows(16, lines)
    text, starts, ends = pack(lines)
    oe, osp = gorp_oracle.Gorp(EDGE["ambiguous16"][0]).extract_batch(text, (starts, ends), threads=0)
    assert (ext == oe).all() and (spans == osp[:, :32]).all()
    assert sum(s.count(":") > 15 for s, e in zip(lines, ext) if e == 0) > 50


@pytest.mark.parametrize("name", SPLIT_DEFS)
def test_cpu_interpreters_split_rule(name):
    """ambiguous31 (63 registers): the general tables, the only ones it gets, against the rows known by construction."""
    lines, ext_w, spans_w = expected(name)
    assert layout(name)["capimg"] == 0 and (ext_w == 0).sum() > len(lines) // 2
    text, starts, ends = pack(lines)
    ext, spans = hostlib.run(blob(name), text, starts, ends, 62)[:2]
    assert (ext == ext_w).all(), np.flatnonzero(ext != ext_w)[:10]
    assert (spans == spans_w).all(), np.flatnonzero((spans != spans_w).any(axis=1))[:10]


@pytest.mark.parametrize("name", OUTCOME_DEFS)
def test_cpu_interpreters_outcome_counts(name):
    """The outcome-count definitions against their expected rows: every table that serves them on the GPU."""
    lines, ext_w, spans_w = expected(name)
    text, starts, ends = pack(lines)
    runs = {"general": hostlib.run(blob(name), text, starts, ends, 2)[:2],
            "fused_walk": hostlib.run_fused_tail(blob(name), text, starts, ends, 2),
            "walk": hostlib.run_walk(blob(name), text, 2, True),
            "tails": hostlib.run_tails(blob(name), text, 2)[:2]}
    for k, (ext, spans) in runs.items():
        assert (ext == ext_w).all(), (k, np.flatnonzero(ext != ext_w)[:10])
        assert (spans == spans_w).all(), (k, np.flatnonzero((spans != spans_w).any(axis=1))[:10])


# ---------------------------------------------------------------- GPU: every tier, both forms
def _hold(name, b, lines, text=None):
    """assert_matches_oracle with the expected rows of `expected` (the oracle's, or known by construction)."""
    _, ext, spans = expected(name)
    if text is not None:
        assert_matches_oracle(EDGE[name][0], b, text=text, expect=(ext, spans))
    else:
        assert_matches_oracle(EDGE[name][0], b, lines=lines, expect=(ext, spans))


@pytest.mark.gpu
@pytest.mark.parametrize("tier", list(TIERS))
@pytest.mark.parametrize("name", list(EDGE))
def test_edge_definitions_every_tier(name, tier, monkeypatch):
    for k in _TIER_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in TIERS[tier].items():
        monkeypatch.setenv(k, v)
    lines = expected(name)[0]
    g = DefinitionReader.reader(EDGE[name][0]).read()
    text, _, _ = pack(lines)
    _hold(name, g.extract_batch_text(text), lines, text=text)
    _hold(name, g.extract_batch_lines(lines), lines)


def _kernel_times(g):
    names, tot = (C.c_char_p * 32)(), (C.c_double * 32)()
    cnt, calls, launches = C.c_int(), C.c_int64(), C.c_int64()
    assert _ffi.lib.gorp_kernel_times(g._eng(), 0, names, tot, 32, C.byref(cnt), C.byref(calls), C.byref(launches), 1) == 0
    return {names[i].decode() for i in range(cnt.value)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EDGE))
def test_edge_definitions_take_the_intended_path(name, monkeypatch):
    """The default text-form path of each definition, named by gorp_kernel_times: the layout side it was built for."""
    import torch
    for k in _TIER_ENV:
        monkeypatch.delenv(k, raising=False)
    lines = expected(name)[0]
    text, _, _ = pack(lines)
    g = DefinitionReader.reader(EDGE[name][0]).read()
    dev = torch.device("cuda", 0)
    d_text = torch.from_numpy(text.view(np.int16)).to(dev)
    _kernel_times(g)
    dres = _ffi.DeviceResult()
    rc = _ffi.lib.gorp_extract_text_device(g._eng(), 0, d_text.data_ptr(), len(text), torch.cuda.current_stream().cuda_stream,
                                           _ffi.FLAG_TIME_KERNELS | _ffi.FLAG_SYNC, C.byref(dres))
    assert rc == 0, _ffi.last_error()
    assert dres.n_lines == len(lines)
    names = _kernel_times(g)
    want = EDGE[name][2]
    capture = {"k4c_fusedwalk", "k4c_tailwalk", "k4b_capwalk", "k4_tdfa_capture"}
    assert want in names, names
    if want == FUSED:
        assert names & capture == {FUSED}, names
    elif want == "k4_tdfa_capture":
        assert names & capture == {want}, names
