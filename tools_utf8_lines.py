"""List<String> form over UTF-8 strings on one GPU: gorp_extract_lines on the strings' UTF-16 against gorp_extract_lines_utf8
on their UTF-8 bytes with int64 offsets (and, since no string here contains '\\n', gorp_extract_text_utf8_bytes on the strings
joined by '\\n'), all called through ctypes on pinned host buffers, so no Python-side encode or decode is timed.

    python tools_utf8_lines.py [--ascii-lines 20000000] [--mix-lines 4000000] [--runs 3] [--calls 5] [--out DIR]

Corpora: config #2 (`readme`, ASCII), and config #5 (`utf16mix`) without its lone-surrogate lines (they have no UTF-8 form).
Each run times `--calls` calls of one entry point with a host clock (a call returns after its last D2H copy); the entry
points alternate, after one warm-up call each. Host-to-device bytes are counted from the inputs (text + int64 offsets).
A separate torch.profiler pass over one call of each gives the device time per kernel and of the H2D copies, among them
the kernels of the UTF-8 lines form: utf8_count_kernel, utf8_line_units_kernel (unit offsets of the strings + boundary
validation) and utf8_rows_kernel (rows back to byte offsets). Prints one JSON document (and writes it to
DIR/utf8_lines.json).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import sys
import time

import numpy as np

sys.dont_write_bytecode = True

from tools_utf8_byte_offsets import ascii_corpus, gpu_identity, mix_corpus  # noqa: E402


def split_lines(text8):
    """'\\n'-terminated UTF-8 bytes -> (strings' bytes without the '\\n', int64 byte offsets, UTF-16 units, int64 unit offsets)."""
    nl = np.flatnonzero(text8 == 10)
    n = len(nl)
    starts = np.concatenate(([0], nl[:-1] + 1)).astype(np.int64)
    lens = (nl - starts).astype(np.int64)
    compact = text8[text8 != 10]
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    if not (compact >= 0x80).any():
        units = compact.astype(np.uint16)
        uoff = off
    else:
        strs = compact.tobytes().decode("utf-8")
        units = np.frombuffer(strs.encode("utf-16-le"), dtype=np.uint16)
        # units per string: 1 per byte that is not a continuation byte, 2 for a 4-byte lead
        per_byte = np.where((compact & 0xC0) == 0x80, 0, np.where(compact >= 0xF0, 2, 1)).astype(np.int64)
        cum = np.zeros(len(compact) + 1, dtype=np.int64)
        np.cumsum(per_byte, out=cum[1:])
        uoff = cum[off]
        assert uoff[-1] == len(units)
    return compact, off, units, uoff


def pinned(arr):
    import torch
    t = torch.empty(arr.nbytes, dtype=torch.uint8).pin_memory()
    v = t.numpy().view(arr.dtype)
    v[:] = arr
    return t, v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ascii-lines", type=int, default=20_000_000)
    ap.add_argument("--mix-lines", type=int, default=4_000_000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from gorp_b200 import _ffi, corpus
    from gorp_b200.api import Blob, _check
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    lib = _ffi.lib
    report = {"gpu": gpu_identity(), "calls_per_run": args.calls, "runs": args.runs, "corpora": {}}
    kinds = ("utf16_lines", "utf8_lines", "utf8_text_bytes")
    for name, definition, make in (("readme_ascii", corpus.README_DEF, lambda: (ascii_corpus(args.ascii_lines), 0)),
                                   ("utf16mix", corpus.WEBLOG_DEF, lambda: mix_corpus(args.mix_lines))):
        text8, dropped = make()
        compact, off, units, uoff = split_lines(text8)
        n = len(off) - 1
        keep = [pinned(a) for a in (text8, compact, off, units, uoff)]
        h_text8, h_compact, h_off, h_units, h_uoff = (v for _, v in keep)
        del text8, compact, units
        h2d = {"utf16_lines": h_units.nbytes + h_uoff.nbytes, "utf8_lines": h_compact.nbytes + h_off.nbytes, "utf8_text_bytes": h_text8.nbytes}
        blob = Blob.from_definition(definition)
        eng = C.c_void_p()
        _check(lib.gorp_engine_create(blob._ptr, blob.length, None, 0, C.byref(eng)))
        res = _ffi.Result()

        def call(kind, digest=False):
            if kind == "utf16_lines":
                rc = lib.gorp_extract_lines(eng, h_units.ctypes.data, h_uoff.ctypes.data, n, C.byref(res))
            elif kind == "utf8_lines":
                rc = lib.gorp_extract_lines_utf8(eng, h_compact.ctypes.data, h_off.ctypes.data, n, C.byref(res))
            else:
                rc = lib.gorp_extract_text_utf8_bytes(eng, h_text8.ctypes.data, h_text8.size, C.byref(res))
            _check(rc)
            nl = res.n_lines
            out = nl
            if digest:  # (outside the timed calls)
                ext = np.ctypeslib.as_array(res.ext_id, (max(nl, 1),))[:nl]
                out = (int(nl), int(ext.astype(np.int64).sum()), int(res.span_stride))
            lib.gorp_result_release(eng, C.byref(res))
            return out

        digests = {k: call(k, True) for k in kinds}  # warm-up (and: same lines, same extraction ids)
        ms = {k: [] for k in kinds}
        for _ in range(args.runs):
            for kind in kinds:
                t0 = time.perf_counter()
                for _ in range(args.calls):
                    call(kind)
                ms[kind].append((time.perf_counter() - t0) / args.calls * 1e3)
        from torch.profiler import ProfilerActivity, profile
        prof_out = {}
        for kind in kinds:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(kind)
                torch.cuda.synchronize()
            per, h2d_ms = {}, 0.0
            for ev in prof.events():
                if ev.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                if ev.name.startswith("Memcpy HtoD"):
                    h2d_ms += ev.device_time_total / 1e3
                elif not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
                    per[ev.name] = per.get(ev.name, 0.0) + ev.device_time_total / 1e3
            total = sum(per.values())
            short = {}
            for k, v in per.items():
                m = re.search(r"(\w+_kernel)", k)
                key = m.group(1) if m else k[:60]
                short[key] = short.get(key, 0.0) + v
            prof_out[kind] = {"kernel_ms_total": total, "h2d_copy_ms": h2d_ms,
                              "top": dict(sorted(((k, round(v, 4)) for k, v in short.items()), key=lambda kv: -kv[1])[:12])}
            if kind == "utf8_lines":
                for k in ("utf8_count_kernel", "utf8_line_units_kernel", "utf8_write_kernel", "utf8_rows_kernel"):
                    prof_out[kind][k + "_ms"] = short.get(k, 0.0)
                    prof_out[kind][k + "_share"] = short.get(k, 0.0) / total if total else None
        lib.gorp_engine_destroy(eng)
        best = {k: min(v) for k, v in ms.items()}
        report["corpora"][name] = {
            "strings": int(n), "utf8_bytes": int(h_compact.nbytes), "utf16_units": int(h_units.size),
            "lone_surrogate_lines_dropped": int(dropped), "same_results": len(set(digests.values())) == 1, "digests": digests,
            "h2d_bytes": h2d, "ms_per_call": {k: [round(x, 3) for x in v] for k, v in ms.items()},
            "lines_per_s_best": {k: n / (v / 1e3) for k, v in best.items()},
            "utf8_over_utf16_lines_best": best["utf8_lines"] / best["utf16_lines"],
            "profiler": prof_out,
        }
        del keep, h_text8, h_compact, h_off, h_units, h_uoff
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "utf8_lines.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
