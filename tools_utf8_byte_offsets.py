"""UTF-8 text form on one GPU: gorp_extract_text_utf8 (UTF-16 unit offsets) against gorp_extract_text_utf8_bytes (byte
offsets of the caller's buffer), both called through ctypes on a pinned host buffer, so no Python-side decode is timed.

    python tools_utf8_byte_offsets.py [--ascii-lines 20000000] [--mix-lines 4000000] [--runs 3] [--calls 5] [--out DIR]

Corpora: config #2 (`readme`, ASCII) as UTF-8, and config #5 (`utf16mix`) without its lone-surrogate lines (they have no
UTF-8 form). Each run times `--calls` calls of one entry point with a host clock (a call returns after its last D2H copy);
the two entry points alternate, after one warm-up call each. A separate torch.profiler pass over one call of each gives
the device time per kernel, among them the two kernels of the byte form: utf8_nl_count_mask_kernel (byte '\\n' index) and
utf8_rows_kernel (rows converted to byte offsets). Prints one JSON document (and writes it to DIR/utf8_byte_offsets.json).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

sys.dont_write_bytecode = True


def gpu_identity():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        out["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError) as ex:
        out["nvidia_smi"] = "unavailable: %s" % ex
    return out


def ascii_corpus(n_lines):
    from gorp_b200 import corpusgen
    return corpusgen.host_text("readme", 0, n_lines).astype(np.uint8)  # config #2 is ASCII: the bytes are its UTF-8


def mix_corpus(n_lines):
    from gorp_b200 import corpusgen
    text = corpusgen.host_text("utf16mix", 0, n_lines).tobytes().decode("utf-16-le", "surrogatepass")
    lone = re.compile("[\ud800-\udfff]")  # a surrogate left after decoding is a lone one
    lines = text.split("\n")
    kept = [s for s in lines[:-1] if not lone.search(s)]
    return np.frombuffer(("\n".join(kept) + "\n").encode("utf-8"), dtype=np.uint8), len(lines) - 1 - len(kept)


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
    entry = {"units": lib.gorp_extract_text_utf8, "bytes": lib.gorp_extract_text_utf8_bytes}
    for name, definition, make in (("readme_ascii", corpus.README_DEF, lambda: (ascii_corpus(args.ascii_lines), 0)),
                                   ("utf16mix", corpus.WEBLOG_DEF, lambda: mix_corpus(args.mix_lines))):
        data, dropped = make()
        host = torch.empty(len(data), dtype=torch.uint8).pin_memory()
        host.numpy()[:] = data
        del data
        buf = host.numpy()
        blob = Blob.from_definition(definition)
        eng = C.c_void_p()
        _check(lib.gorp_engine_create(blob._ptr, blob.length, None, 0, C.byref(eng)))
        res = _ffi.Result()

        def call(kind, digest=False):
            _check(entry[kind](eng, buf.ctypes.data, buf.size, C.byref(res)))
            n = res.n_lines
            out = n
            if digest:  # (outside the timed calls)
                ext = np.ctypeslib.as_array(res.ext_id, (max(n, 1),))[:n]
                out = (int(n), int(ext.astype(np.int64).sum()), int(res.span_stride))
            lib.gorp_result_release(eng, C.byref(res))
            return out

        same = call("units", True) == call("bytes", True)  # warm-up (and: same lines, same extraction ids)
        ms = {"units": [], "bytes": []}
        for _ in range(args.runs):
            for kind in ("units", "bytes"):
                t0 = time.perf_counter()
                for _ in range(args.calls):
                    n_lines = call(kind)
                ms[kind].append((time.perf_counter() - t0) / args.calls * 1e3)
        # device time per kernel: one call of each entry point under torch.profiler (a pass of its own)
        from torch.profiler import ProfilerActivity, profile
        kernels = {}
        for kind in ("units", "bytes"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(kind)
                torch.cuda.synchronize()
            per = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA and not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
                    per[ev.name] = per.get(ev.name, 0.0) + ev.device_time_total / 1e3
            total = sum(per.values())
            short = {}
            for k, v in per.items():
                m = re.search(r"(\w+_kernel)", k)
                key = m.group(1) if m else k[:60]
                short[key] = short.get(key, 0.0) + v
            kernels[kind] = {"kernel_ms_total": total,
                             "top": dict(sorted(((k, round(v, 4)) for k, v in short.items()), key=lambda kv: -kv[1])[:12])}
            if kind == "bytes":
                for k in ("utf8_nl_count_mask_kernel", "utf8_rows_kernel"):
                    kernels[kind][k + "_ms"] = short.get(k, 0.0)
                    kernels[kind][k + "_share"] = short.get(k, 0.0) / total if total else None
        _ffi.lib.gorp_engine_destroy(eng)
        best = {k: min(v) for k, v in ms.items()}
        report["corpora"][name] = {
            "bytes": int(buf.size), "lines": int(n_lines), "lone_surrogate_lines_dropped": int(dropped), "same_results": same,
            "ms_per_call": {k: [round(x, 3) for x in v] for k, v in ms.items()},
            "lines_per_s_best": {k: n_lines / (v / 1e3) for k, v in best.items()},
            "bytes_over_units_best": best["bytes"] / best["units"],
            "profiler": kernels,
        }
        buf = None
        del host
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "utf8_byte_offsets.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
