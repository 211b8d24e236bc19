"""UTF-8 held in HBM on one GPU: gorp_extract_text_utf8_device and gorp_extract_lines_utf8_device against
gorp_extract_text_device on the same lines as UTF-16 (what bench.py's `value` times).

    python tools_utf8_device.py [--configs readme:100000000,syslog200:40000000] [--runs 5] [--calls 3] [--out DIR]

Corpora: config #2 (`readme`, 100 M lines) and config #4 (`syslog200`, 40 M lines), generated on the device by corpusgen
and narrowed to bytes there (both are ASCII, so the UTF-8 bytes are the UTF-16 units narrowed). The lines form takes the
same lines without their '\\n' and int64 offsets. Each run times `--calls` calls of each entry point with CUDA events on
the calling stream, the three entry points alternating inside the run, after three warm-up calls each; the texts are far
larger than the 126 MB L2. A separate torch.profiler pass over one call of each gives the device time per kernel. The
card's name and power limit are read in the same run. Prints one JSON document (and writes it to DIR/utf8_device.json).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import sys

sys.dont_write_bytecode = True

from tools_utf8_byte_offsets import gpu_identity  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="readme:100000000,syslog200:40000000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from gorp_b200 import DefinitionReader, _ffi, corpus, corpusgen
    from gorp_b200.api import _check
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    lib = _ffi.lib
    dev = torch.device("cuda", 0)
    report = {"gpu": gpu_identity(), "runs": args.runs, "calls_per_run": args.calls, "configs": {}}
    kinds = ("utf8_text_device", "utf16_text_device", "utf8_lines_device")
    for item in args.configs.split(","):
        name, n = item.split(":")
        n = int(n)
        g = DefinitionReader.reader(corpus.CONFIGS[name][0]).read(devices=[0])
        eng = g._eng()
        n_bins = len(g.getExtractions()) + 2
        u16 = corpusgen.device_text(name, 0, n, dev)
        assert int(u16.max()) < 0x80, "the corpus must be ASCII to be narrowed to UTF-8 bytes"
        u8 = u16.to(torch.uint8)
        stream = torch.cuda.current_stream(dev)
        st = stream.cuda_stream
        dres = _ffi.DeviceResult()
        _check(lib.gorp_extract_text_device(eng, 0, u16.data_ptr(), u16.numel(), st, _ffi.FLAG_SYNC, C.byref(dres)))
        assert dres.n_lines == n
        line_off = torch.as_tensor(_dev_array(dres.d_line_off, n + 1), device=dev).clone()
        f8 = torch.cat([c[c != 10] for c in u8.split(1 << 28)])  # (in pieces: the index of one mask over GBs would be 8x its size)
        off = line_off - torch.arange(n + 1, device=dev, dtype=torch.int64)
        off[-1] = f8.numel()
        del line_off

        def call(kind):
            if kind == "utf8_text_device":
                _check(lib.gorp_extract_text_utf8_device(eng, 0, u8.data_ptr(), u8.numel(), st, 0, C.byref(dres)))
            elif kind == "utf16_text_device":
                _check(lib.gorp_extract_text_device(eng, 0, u16.data_ptr(), u16.numel(), st, 0, C.byref(dres)))
            else:
                _check(lib.gorp_extract_lines_utf8_device(eng, 0, f8.data_ptr(), off.data_ptr(), n, st, 0, C.byref(dres)))

        digests = {}
        for kind in kinds:
            for _ in range(3):
                call(kind)
            torch.cuda.synchronize(dev)
            ext = torch.as_tensor(_dev_array(dres.d_ext_id, n, "<i4"), device=dev)
            digests[kind] = (int(dres.n_lines), int(ext.to(torch.int64).sum()), tuple(torch.as_tensor(_dev_array(dres.d_histogram, n_bins, "<i8"), device=dev).tolist()))
        ms = {k: [] for k in kinds}
        for _ in range(args.runs):
            for kind in kinds:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(args.calls):
                    call(kind)
                e1.record(stream)
                e1.synchronize()
                ms[kind].append(e0.elapsed_time(e1) / args.calls)
        from torch.profiler import ProfilerActivity, profile
        prof_out = {}
        for kind in kinds:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(kind)
                torch.cuda.synchronize(dev)
            per = {}
            for ev in prof.events():
                if ev.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                m = re.search(r"(\w+_kernel\w*)", ev.name)
                key = ("copy " if ev.name.startswith("Memcpy") else "") + (m.group(1) if m else ev.name[:60])
                per[key] = per.get(key, 0.0) + ev.device_time_total / 1e3
            prof_out[kind] = {"device_ms_total": round(sum(per.values()), 4),
                              "per_kernel_ms": dict(sorted(((k, round(v, 4)) for k, v in per.items()), key=lambda kv: -kv[1]))}
        best = {k: min(v) for k, v in ms.items()}
        report["configs"][name] = {
            "lines": n, "utf8_bytes": int(u8.numel()), "lines_form_bytes": int(f8.numel()), "same_ext_ids": len(set(digests.values())) == 1,
            "digests": digests, "ms_per_call": {k: [round(x, 3) for x in v] for k, v in ms.items()},
            "best_ms": {k: round(v, 3) for k, v in best.items()},
            "utf8_text_minus_utf16_text_ms": round(best["utf8_text_device"] - best["utf16_text_device"], 3),
            "profiler": prof_out,
        }
        del u16, u8, f8, off, g
        torch.cuda.empty_cache()
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "utf8_device.json"), "w") as f:
            f.write(text + "\n")


def _dev_array(ptr, n, typestr="<i8"):
    from gorp_b200 import parityhash
    return parityhash.DeviceArray(ptr, (n,), typestr)


if __name__ == "__main__":
    main()
