"""The device-resident calls (gorp_extract_text_device, gorp_extract_lines_device) against the oracle.

These are the calls bench.py times: one launch over the whole HBM-resident text, with no host pieces in between. So they
are the only way into launches of more than 32 M units (line offsets past 2^31 and 2^32, fused-walk items of up to 1024
lines, buckets of millions of lines), into caller buffers with arbitrary bounds and 16-byte (not 32-byte) aligned bases,
and into the caller's streams. Text comes from gorp_b200.corpusgen (line i is a pure function of the seed and i): the
device copy feeds the call, the host copy of the same lines feeds the oracle.

The checkers themselves run on the CPU (test_checkers_catch_corruption): each of them must fail on a result with one
span, ext_id, offset or histogram bin changed."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from gorp_b200 import DefinitionReader, _ffi, corpus, corpusgen, parityhash
from oracle import gorp_oracle, jdkre
from tests import reference_vectors as V
from tests.test_gpu_parity import _TIER_ENV, TIERS, assert_matches_oracle
from tests.test_host_compile import TRICKY_LINES

gpu = pytest.mark.gpu
FLAGS = _ffi.FLAG_SYNC


class Rows:
    """A result as numpy arrays: the fields assert_matches_oracle reads."""

    def __init__(self, n_lines, span_stride, ext_id, line_off, spans, histogram):
        self.n_lines, self.span_stride = n_lines, span_stride
        self.ext_id, self.line_off, self.spans, self.histogram = ext_id, line_off, spans, histogram

    def same_as(self, other, off_shift=0):
        assert self.n_lines == other.n_lines and self.span_stride == other.span_stride
        assert (self.ext_id == other.ext_id).all(), np.flatnonzero(self.ext_id != other.ext_id)[:10]
        assert (self.spans == other.spans).all(), np.flatnonzero((self.spans != other.spans).any(axis=1))[:10]
        assert (self.line_off == other.line_off + off_shift).all()
        assert (self.histogram == other.histogram).all()


def _dev_array(ptr, shape, typestr, dev):
    return torch.as_tensor(parityhash.DeviceArray(ptr, shape, typestr), device=dev)


def device_views(dres, n_bins, dev):
    """(ext_id, line_off, spans, histogram) of a gorp_device_result as torch tensors over the engine's buffers."""
    n, w = int(dres.n_lines), int(dres.span_stride)
    ext, sp = parityhash.device_results(dres, dev)
    off = _dev_array(dres.d_line_off, (n + 1,), "<i8", dev) if n else torch.zeros(1, dtype=torch.int64, device=dev)
    hist = _dev_array(dres.d_histogram, (n_bins,), "<i8", dev)
    return ext, off, sp, hist


def fetch(dres, n_bins, dev, stream=None):
    """Host copy of a gorp_device_result (read on `stream`, default: the current one)."""
    with torch.cuda.stream(stream) if stream is not None else torch.cuda.stream(torch.cuda.current_stream(dev)):
        ext, off, sp, hist = device_views(dres, n_bins, dev)
        return Rows(int(dres.n_lines), int(dres.span_stride), ext.cpu().numpy(), off.cpu().numpy(), sp.cpu().numpy(),
                    hist.cpu().numpy())


def make_gorp(definition, monkeypatch, env=None, devices=(0,)):
    """A Gorp whose engine is created under `env` (the engine reads the GORP_FORCE_* switches when it is created)."""
    for k in _TIER_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    g = DefinitionReader.reader(definition).read(devices=list(devices))
    g._eng()
    return g


def n_bins(g):
    return len(g.getExtractions()) + 2


def text_call(g, d_text, n_units, stream=None, flags=FLAGS, dev_index=0, unit_shift=0):
    dres = _ffi.DeviceResult()
    st = torch.cuda.current_stream().cuda_stream if stream is None else stream.cuda_stream
    rc = _ffi.lib.gorp_extract_text_device(g._eng(), dev_index, d_text.data_ptr() + 2 * unit_shift, n_units, st, flags, C.byref(dres))
    assert rc == 0, _ffi.last_error()
    return dres


def lines_call(g, d_text, d_off, n_lines, flags=FLAGS, unit_shift=0):
    dres = _ffi.DeviceResult()
    st = torch.cuda.current_stream().cuda_stream
    rc = _ffi.lib.gorp_extract_lines_device(g._eng(), 0, d_text.data_ptr() + 2 * unit_shift, d_off.data_ptr(), n_lines, st, flags,
                                            C.byref(dres))
    assert rc == 0, _ffi.last_error()
    return dres


def to_device(units, dev):
    return torch.from_numpy(np.ascontiguousarray(units, dtype=np.uint16).view(np.int16)).to(dev)


@functools.lru_cache(maxsize=None)
def oracle_text(name, n):
    """Host text of lines [0, n) of corpus `name` and the oracle's rows for it."""
    text = corpusgen.host_text(name, 0, n)
    oe, osp = gorp_oracle.Gorp(corpus.CONFIGS[name][0]).extract_batch(text, gorp_oracle.split_lines(text), threads=0)
    return text, oe, osp


def oracle_rows(definition, text, threads=0):
    return gorp_oracle.Gorp(definition).extract_batch(text, gorp_oracle.split_lines(text), threads=threads)


# ---------------------------------------------------------------- checkers of whole results on the device (torch)
def check_line_offsets(line_off, lens):
    """The text form's index of a corpus with line lengths `lens`: line_off == [0, cumsum(lens + 1)]."""
    want = torch.cumsum(lens.to(torch.int64) + 1, dim=0)
    assert int(line_off[0]) == 0
    bad = torch.nonzero(line_off[1:] != want).flatten()
    assert bad.numel() == 0, bad[:10].tolist()


def check_histogram(hist, ext_id, n_ext):
    bins = torch.where(ext_id >= 0, ext_id, torch.where(ext_id == -1, n_ext, n_ext + 1)).to(torch.int64)
    want = torch.bincount(bins, minlength=n_ext + 2)
    assert torch.equal(hist.to(torch.int64), want), (hist.tolist(), want.tolist())


def check_span_rows(ext_id, spans, lens, n_groups, chunk=1 << 22):
    """Every row: a matched line holds 2 * n_groups(ext) entries, each pair (-1, -1) or 0 <= s <= e <= len; every other
    entry, and every entry of a MISS or capture-failed row, is -1."""
    n, w = spans.shape
    groups = torch.as_tensor(n_groups, dtype=torch.int64, device=spans.device)
    col = torch.arange(w, device=spans.device)
    for lo in range(0, n, chunk):
        hi = min(lo + chunk, n)
        e = ext_id[lo:hi].to(torch.int64)
        sp = spans[lo:hi].to(torch.int64)
        used = col[None, :] < torch.where(e >= 0, 2 * groups[e.clamp(min=0)], 0)[:, None]
        bad = torch.nonzero((~used & (sp != -1)).any(dim=1)).flatten()
        assert bad.numel() == 0, ("entries past the row's groups", (bad[:10] + lo).tolist())
        s, t, u = sp[:, 0::2], sp[:, 1::2], used[:, 0::2]
        ok = ((s == -1) & (t == -1)) | ((s >= 0) & (s <= t) & (t <= lens[lo:hi].to(torch.int64)[:, None]))
        bad = torch.nonzero((u & ~ok).any(dim=1)).flatten()
        assert bad.numel() == 0, ("spans outside the line", (bad[:10] + lo).tolist())


def device_lengths(name, first_line, n, dev):
    """Lengths (without the '\\n') of lines [first_line, first_line + n) of corpus `name`, made on the device."""
    lib, h = corpusgen._load(), corpusgen._host_program(corpusgen.program(name))
    lens = torch.empty(n, dtype=torch.int32, device=dev)
    assert lib.cg_lengths_device(C.byref(h), corpusgen.SEEDS[name], first_line, n, lens.data_ptr(),
                                 torch.cuda.current_stream(dev).cuda_stream) == 0
    return lens


def window_rows(ext, off, sp, w0, w1):
    """Rows [w0, w1) of a device result on the host, offsets relative to line w0 (the host text of those lines)."""
    e = ext[w0:w1].cpu().numpy()
    o = (off[w0:w1 + 1] - off[w0]).cpu().numpy()
    return Rows(w1 - w0, sp.shape[1], e, o, sp[w0:w1].cpu().numpy(), None)


def window_histogram(rows, n_ext):
    e = rows.ext_id
    rows.histogram = np.bincount(np.where(e >= 0, e, np.where(e == -1, n_ext, n_ext + 1)), minlength=n_ext + 2)
    return rows


# ---------------------------------------------------------------- text form: every config, every tier, one big launch
TEXT_LINES = {"simple": 1_200_000, "readme": 1_200_000, "weblog": 300_000, "syslog200": 300_000, "utf16mix": 300_000}
TEXT_CASES = [(name, "k1_fusedwalk") for name in TEXT_LINES] + \
             [(name, tier) for name in ("readme", "weblog") for tier in TIERS if tier != "k1_fusedwalk"]


@gpu
@pytest.mark.parametrize("name,tier", TEXT_CASES)
def test_text_form_matches_oracle(name, tier, monkeypatch):
    """One launch over 40-75 M units (more than one 32 M-unit host piece), every line against the oracle; then the same
    pointer with n_units - 1 (the final '\\n' stays readable just past the end, and must not be read)."""
    dev = torch.device("cuda", 0)
    d = corpus.CONFIGS[name][0]
    text, oe, osp = oracle_text(name, TEXT_LINES[name])
    assert len(text) > 32 << 20
    g = make_gorp(d, monkeypatch, TIERS[tier])
    d_text = corpusgen.device_text(name, 0, TEXT_LINES[name], dev)
    for n_units in (len(text), len(text) - 1):
        rows = fetch(text_call(g, d_text, n_units), n_bins(g), dev)
        assert_matches_oracle(d, rows, text=text[:n_units], expect=(oe, osp))


# ---------------------------------------------------------------- lines form
def _mixed_lines():
    """Corpus lines, TRICKY_LINES, empty strings, strings that contain '\\n', strings of 70 000 units and more; as uint16
    arrays, in a seeded order."""
    rng = np.random.default_rng(41)
    out = []
    for name, n in (("readme", 20000), ("weblog", 5000)):
        t = corpusgen.host_text(name, 0, n)
        s, e = gorp_oracle.split_lines(t)
        out += [t[a:b] for a, b in zip(s, e)]
    body = "".join(rng.choice(list("abcdefghij0123456789/"), size=70000))
    extra = TRICKY_LINES + [""] * 40 + ["\n", "\n\n", "[1]: GET 2ms /a\nb", "[2]: PUT 3ms /x\n", "\n[3]: GET 2ms /a"]
    extra += ["[1]: GET 2ms /" + body, "[3]: GET 2ms /" + body + " tail", "[6]: GET 2ms /" + "\U0001F600" * 40000,
              "[2]: PUT 31ms /" + body * 2 + "é" + body]
    out += [np.asarray(jdkre.to_units(s), dtype=np.uint16) for s in extra]
    return [out[i] for i in rng.permutation(len(out))]


MIXED = functools.lru_cache(maxsize=None)(_mixed_lines)


@functools.lru_cache(maxsize=None)
def oracle_lines(definition):
    lines = MIXED()
    off = np.zeros(len(lines) + 1, dtype=np.int64)
    np.cumsum([len(u) for u in lines], out=off[1:])
    flat = np.concatenate(lines)
    oe, osp = gorp_oracle.Gorp(definition).extract_batch(flat, off, threads=0)
    return flat, off, oe, osp


LINES_TIERS = {"default": {}, "no_tails": {"GORP_NO_TAILS": "1"}, **{t: v for t, v in TIERS.items() if t != "k1_fusedwalk"}}


def _garbage(rng, n):
    """Units that would change a result if read as part of a line: '\\n', a matching line head, non-ASCII."""
    head = np.asarray(jdkre.to_units("\n[1]: GET 2ms /éx\n"), dtype=np.uint16)
    return np.resize(np.concatenate((head, rng.integers(1, 0xD7FF, size=7).astype(np.uint16))), n)


@gpu
@pytest.mark.parametrize("tier", list(LINES_TIERS))
def test_lines_form_matches_oracle(tier, monkeypatch):
    """gorp_extract_lines_device with d_off an int64 CUDA tensor whose first offset is past garbage, against the oracle and
    against the host-buffer call gorp_extract_lines on the same strings."""
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(43)
    for d in (V.README_DEF, corpus.WEBLOG_DEF):
        flat, off, oe, osp = oracle_lines(d)
        g = make_gorp(d, monkeypatch, LINES_TIERS[tier])
        pre = 1013
        buf = np.concatenate((_garbage(rng, pre), flat, _garbage(rng, 517)))
        d_buf, d_off = to_device(buf, dev), torch.from_numpy(off + pre).to(dev)
        n = len(off) - 1
        rows = fetch(lines_call(g, d_buf, d_off, n), n_bins(g), dev)
        assert_matches_oracle(d, rows, lines=MIXED(), expect=(oe, osp), line_off0=pre)
        host = g.extract_batch_lines(MIXED())
        rows.same_as(Rows(host.n_lines, host.span_stride, host.ext_id, host.line_off, host.spans, host.histogram), off_shift=pre)


# ---------------------------------------------------------------- the caller's buffer bounds
def _cuts(text, starts, ends):
    """n_units values that cut a line in the middle: 16 consecutive ones (every residue mod 16) inside a line near the end,
    and 8192 m - 1, 8192 m, 8192 m + 1 (K1's tile) for the first and last two m where all three are mid-line."""
    k = int(np.flatnonzero(ends - starts >= 24)[-3])
    cuts = [int(starts[k]) + 4 + j for j in range(16)]
    ms = [m for m in range(1, len(text) // 8192) if not (text[8192 * m - 3:8192 * m + 2] == 10).any()]
    for m in ms[:2] + ms[-2:]:
        cuts += [8192 * m - 1, 8192 * m, 8192 * m + 1]
    return cuts


def _cut_expect(d, text, starts, oe, osp, cut):
    """The oracle's rows for text[:cut]: the lines before the cut one as they were, the cut line on its own."""
    k = int(np.searchsorted(starts, cut, side="right")) - 1
    assert starts[k] < cut and text[cut - 1] != 10 and text[cut] != 10
    ce, csp = oracle_rows(d, text[starts[k]:cut], threads=1)
    return k, np.concatenate((oe[:k], ce)), np.concatenate((osp[:k], csp))


@gpu
@pytest.mark.parametrize("name,n", [("readme", 60000), ("weblog", 20000)])
def test_nothing_read_past_the_callers_bounds(name, n, monkeypatch):
    """The text in a larger tensor, followed by poison that would change a result if it were read (the rest of the cut line
    and the lines after it; or '\\n' and whole matching lines); in the lines form also poison before off[0] and after
    off[n]. Cuts at every residue of n_units mod 16 and around K1's 8192-unit tiles, always mid-line: results equal the
    oracle's on the exact text."""
    dev = torch.device("cuda", 0)
    d = corpus.CONFIGS[name][0]
    text, oe, osp = oracle_text(name, n)
    starts, ends = gorp_oracle.split_lines(text)
    g = make_gorp(d, monkeypatch)
    nb = n_bins(g)
    for cut in _cuts(text, starts, ends):
        k, ce, csp = _cut_expect(d, text, starts, oe, osp, cut)
        exact = text[:cut]
        for poison in (text[cut:cut + 4000], np.concatenate(([10], text[:4000]))):
            rows = fetch(text_call(g, to_device(np.concatenate((exact, poison)), dev), cut), nb, dev)
            assert_matches_oracle(d, rows, text=exact, expect=(ce, csp))
        # lines form: the last 2000 lines before the cut one and the cut line, without separators, between poison
        k0 = max(0, k - 2000)
        lines = [text[a:b] for a, b in zip(starts[k0:k], ends[k0:k])] + [text[starts[k]:cut]]
        flat = np.concatenate(lines)
        off = np.zeros(len(lines) + 1, dtype=np.int64)
        np.cumsum([len(u) for u in lines], out=off[1:])
        pre = np.concatenate((text[:37], text[starts[k]:starts[k] + 5]))  # a whole line, then the head of the cut one
        buf = np.concatenate((pre, flat, text[cut:cut + 3000]))
        rows = fetch(lines_call(g, to_device(buf, dev), torch.from_numpy(off + len(pre)).to(dev), len(lines)), nb, dev)
        assert_matches_oracle(d, rows, lines=lines, expect=(ce[k0:], csp[k0:]), line_off0=len(pre))


# ---------------------------------------------------------------- base alignment
@gpu
@pytest.mark.parametrize("name,n", [("readme", 200000), ("weblog", 60000)])
def test_base_alignment(name, n, monkeypatch):
    """Bases at 0, 16 and 32 bytes past a 512-byte boundary give identical results that match the oracle, in both forms
    (a base that is 16 but not 32-byte aligned takes the kernels with 16-byte loads); bases at 2, 4 and 8 bytes are
    refused with GORP_E_ARG."""
    dev = torch.device("cuda", 0)
    d = corpus.CONFIGS[name][0]
    text, oe, osp = oracle_text(name, n)
    starts, ends = gorp_oracle.split_lines(text)
    flat = text[text != 10]  # the lines form: the same lines without separators
    off = np.zeros(n + 1, dtype=np.int64)
    off[:-1] = starts - np.arange(n)
    off[-1] = len(flat)
    lines = [flat[a:b] for a, b in zip(off[:-1], off[1:])]
    g = make_gorp(d, monkeypatch)
    nb = n_bins(g)
    d_text, d_flat = torch.zeros(len(text) + 64, dtype=torch.int16, device=dev), torch.zeros(len(flat) + 64, dtype=torch.int16, device=dev)
    assert d_text.data_ptr() % 512 == 0 and d_flat.data_ptr() % 512 == 0
    first = {}
    for shift in (0, 8, 16):
        d_text.zero_()
        d_text[shift:shift + len(text)] = to_device(text, dev)
        d_flat.zero_()
        d_flat[shift:shift + len(flat)] = to_device(flat, dev)
        rt = fetch(text_call(g, d_text, len(text), unit_shift=shift), nb, dev)
        rl = fetch(lines_call(g, d_flat, torch.from_numpy(off).to(dev), n, unit_shift=shift), nb, dev)
        if not first:
            assert_matches_oracle(d, rt, text=text, expect=(oe, osp))
            assert_matches_oracle(d, rl, lines=lines, expect=(oe, osp))
            first = {"text": rt, "lines": rl}
        else:
            rt.same_as(first["text"])
            rl.same_as(first["lines"])
    d_off = torch.from_numpy(off).to(dev)
    st = torch.cuda.current_stream().cuda_stream
    for shift in (1, 2, 4):
        dres = _ffi.DeviceResult()
        rc = _ffi.lib.gorp_extract_text_device(g._eng(), 0, d_text.data_ptr() + 2 * shift, len(text), st, FLAGS, C.byref(dres))
        assert rc == _ffi.GORP_E_ARG and "16-byte aligned" in _ffi.last_error()
        rc = _ffi.lib.gorp_extract_lines_device(g._eng(), 0, d_flat.data_ptr() + 2 * shift, d_off.data_ptr(), n, st, FLAGS, C.byref(dres))
        assert rc == _ffi.GORP_E_ARG and "16-byte aligned" in _ffi.last_error()


# ---------------------------------------------------------------- flags, streams, contexts
def _kernel_times(g, reset):
    names, tot = (C.c_char_p * 16)(), (C.c_double * 16)()
    cnt, calls, launches = C.c_int(), C.c_int64(), C.c_int64()
    assert _ffi.lib.gorp_kernel_times(g._eng(), 0, names, tot, 16, C.byref(cnt), C.byref(calls), C.byref(launches), reset) == 0
    return {names[i].decode() for i in range(cnt.value)}, calls.value


@gpu
@pytest.mark.parametrize("name,kernel", [("readme", "k4c_fusedwalk"), ("weblog", "k4c_tailwalk")])
def test_flags_streams_and_contexts(name, kernel, monkeypatch):
    dev = torch.device("cuda", 0)
    d = corpus.CONFIGS[name][0]
    n = 100000
    text, oe, osp = oracle_text(name, n)
    g = make_gorp(d, monkeypatch, devices=(0, 0))
    nb = n_bins(g)
    d_text = corpusgen.device_text(name, 0, n, dev)
    base = fetch(text_call(g, d_text, len(text), flags=0), nb, dev)
    assert_matches_oracle(d, base, text=text, expect=(oe, osp))
    # timed calls give the same rows, and gorp_kernel_times counts them and names the kernels of the path that ran
    _kernel_times(g, reset=1)
    for _ in range(3):
        fetch(text_call(g, d_text, len(text), flags=_ffi.FLAG_TIME_KERNELS | _ffi.FLAG_SYNC), nb, dev).same_as(base)
    names, calls = _kernel_times(g, reset=1)
    assert calls == 3 and kernel in names and "k1_count_newlines" in names, (calls, names)
    # a stream of the caller's, and calls that alternate between two streams of one context
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    fetch(text_call(g, d_text, len(text), stream=s1, flags=0), nb, dev, stream=s1).same_as(base)
    half = n // 2
    cut = int(gorp_oracle.split_lines(text)[0][half])  # a second text: the first half of the lines
    other = Rows(half, base.span_stride, base.ext_id[:half], base.line_off[:half + 1], base.spans[:half], None)
    window_histogram(other, nb - 2)
    for rep in range(2):
        fetch(text_call(g, d_text, len(text), stream=s1, flags=0), nb, dev, stream=s1).same_as(base)
        fetch(text_call(g, d_text, cut, stream=s2, flags=0), nb, dev, stream=s2).same_as(other)
    torch.cuda.synchronize(dev)
    # the second context of the engine on the same GPU; indexes outside the engine's devices are refused
    fetch(text_call(g, d_text, len(text), dev_index=1), nb, dev).same_as(base)
    st = torch.cuda.current_stream().cuda_stream
    for idx in (2, -1):
        dres = _ffi.DeviceResult()
        assert _ffi.lib.gorp_extract_text_device(g._eng(), idx, d_text.data_ptr(), len(text), st, FLAGS, C.byref(dres)) == _ffi.GORP_E_ARG
    # an empty text
    dres = text_call(g, d_text, 0)
    assert dres.n_lines == 0
    assert (fetch(dres, nb, dev).histogram == 0).all()


# ---------------------------------------------------------------- one launch past 2^32 units
SCALE = [("readme", 72_000_000, "all"), ("syslog200", 40_000_000, "windows"), ("utf16mix", 35_200_000, "windows")]
CHUNK = 4 << 20
WINDOW = 4096


@gpu
@pytest.mark.parametrize("name,n,coverage", SCALE)
def test_one_launch_past_2_32_units(name, n, coverage, monkeypatch):
    """One text-form launch over more than 2^32 units (readme: 72 M lines, 4.5 G units; syslog200 at the bench's 40 M lines,
    11.3 GB; utf16mix at the 35.2 M lines of a one-GPU config #5 shard, 12.5 GB). On the device, over every line: the line
    index, the histogram and the span-row invariants. Against the oracle: every line of readme in 4 M-line chunks; for the
    others the windows around the lines that hold units 2^31 and 2^32, the last lines and 16 seeded random windows."""
    dev = torch.device("cuda", 0)
    d = corpus.CONFIGS[name][0]
    o = gorp_oracle.Gorp(d)
    g = make_gorp(d, monkeypatch)
    nb = n_bins(g)
    d_text = corpusgen.device_text(name, 0, n, dev)
    n_units = d_text.numel()
    assert n_units > (1 << 32) + (1 << 27), n_units
    dres = text_call(g, d_text, n_units)
    del d_text
    assert dres.n_lines == n
    ext, off, sp, hist = device_views(dres, nb, dev)
    lens = device_lengths(name, 0, n, dev)
    check_line_offsets(off, lens)
    assert int(off[-1]) == n_units
    check_histogram(hist, ext, nb - 2)
    check_span_rows(ext, sp, lens, [len(x.extractor_names) for x in o.extractions])
    del lens
    if coverage == "all":
        windows = [(lo, min(lo + CHUNK, n)) for lo in range(0, n, CHUNK)]
    else:
        at = torch.searchsorted(off, torch.tensor([1 << 31, 1 << 32], dtype=torch.int64, device=dev), right=True) - 1
        windows = [(max(0, int(k) - WINDOW // 2), min(n, int(k) + WINDOW // 2)) for k in at.tolist()]
        windows.append((n - WINDOW, n))
        rng = np.random.default_rng(47)
        windows += [(int(w), int(w) + WINDOW) for w in rng.integers(0, n - WINDOW, size=16)]
    for w0, w1 in windows:
        rows = window_histogram(window_rows(ext, off, sp, w0, w1), nb - 2)
        text = corpusgen.host_text(name, w0, w1 - w0)
        assert_matches_oracle(d, rows, text=text)


# ---------------------------------------------------------------- the checkers fail on a corrupted result (CPU only)
def test_checkers_catch_corruption():
    """A correct synthetic result passes every checker; one changed span, ext_id, offset or histogram bin fails them."""
    d = V.README_DEF
    o = gorp_oracle.Gorp(d)
    text = np.concatenate((corpus.readme_corpus(3000, seed=1), corpus.lines_to_text(TRICKY_LINES)))
    starts, ends = gorp_oracle.split_lines(text)
    oe, osp = oracle_rows(d, text)
    E, G = len(o.extractions), max(len(x.extractor_names) for x in o.extractions)
    assert (oe >= 0).sum() > 1000 and (oe == -1).sum() > 10
    groups = [len(x.extractor_names) for x in o.extractions]

    def good():
        hist = np.bincount(np.where(oe >= 0, oe, np.where(oe == -1, E, E + 1)), minlength=E + 2)
        return Rows(len(starts), 2 * G, oe.copy(), np.append(starts, len(text)), osp[:, :2 * G].copy(), hist)

    def device_checks(r):
        ext, off, sp, hist = (torch.from_numpy(np.ascontiguousarray(a)) for a in (r.ext_id, r.line_off, r.spans, r.histogram))
        lens = torch.from_numpy((ends - starts).astype(np.int32))
        check_line_offsets(off, lens)
        check_histogram(hist, ext, E)
        check_span_rows(ext, sp, lens, groups, chunk=1000)

    assert_matches_oracle(d, good(), text=text)
    device_checks(good())
    m = int(np.flatnonzero(oe >= 0)[7])
    miss = int(np.flatnonzero(oe == -1)[3])
    last = 2 * groups[oe[m]] - 1

    def corrupt_span(r):
        r.spans[m, last] += 1  # end of the last group past the line, or inside it but wrong

    def corrupt_span_padding(r):
        r.spans[miss, 0] = 0

    def corrupt_span_order(r):
        r.spans[m, 0], r.spans[m, 1] = r.spans[m, 1] + 1, r.spans[m, 0]

    def corrupt_ext(r):
        r.ext_id[miss] = 0

    def corrupt_offset(r):
        r.line_off[500] += 1

    def corrupt_hist(r):
        r.histogram[0] -= 1
        r.histogram[E] += 1

    for f in (corrupt_span, corrupt_span_padding, corrupt_span_order, corrupt_ext, corrupt_offset, corrupt_hist):
        r = good()
        f(r)
        with pytest.raises(AssertionError):
            assert_matches_oracle(d, r, text=text)
        if f is not corrupt_span:  # a span moved inside its line is only visible to the oracle comparison
            with pytest.raises(AssertionError):
                device_checks(r)
    r = good()
    r.spans[m, last] = ends[m] - starts[m] + 1  # one past the line's end
    with pytest.raises(AssertionError):
        device_checks(r)
