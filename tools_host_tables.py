"""UTF-8 text in pinned host memory to value tables in host memory: gorp_extract_text_utf8_tables against the plain
gorp_extract_text_utf8_bytes on the same bytes, end to end (both calls return once their results are in host memory).

    python tools_host_tables.py [--configs readme:30000000,syslog200:10000000] [--runs 5] [--out DIR]

Corpora: config #2 (`readme`) and config #4 (`syslog200`), generated on the device by corpusgen, narrowed to bytes (both
are ASCII) and copied once to pinned host memory. Each run times one plain call and one tables call with a host clock,
alternating, after one warm-up call of each; one GPU, and two when present. Reports lines/s, the bytes of the tables,
and the device-to-host bytes of each call (rows, line offsets, spans and histogram; the tables add their row indexes,
offsets, values and bitmaps). The card's name and power limit are read in the same run. Prints one JSON document (and
writes it to DIR/host_tables.json).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

sys.dont_write_bytecode = True

from tools_utf8_byte_offsets import gpu_identity  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="readme:30000000,syslog200:10000000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from gorp_b200 import DefinitionReader, _ffi, corpus, corpusgen
    from gorp_b200.api import _check
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    lib = _ffi.lib
    dev = torch.device("cuda", 0)
    n_gpus = torch.cuda.device_count()
    report = {"gpu": gpu_identity(), "runs": args.runs, "configs": {}}
    for item in args.configs.split(","):
        name, n = item.split(":")
        n = int(n)
        u16 = corpusgen.device_text(name, 0, n, dev)
        assert int(u16.max()) < 0x80, "the corpus must be ASCII to be narrowed to UTF-8 bytes"
        host = torch.empty(u16.numel(), dtype=torch.uint8, pin_memory=True)
        host.copy_(u16.to(torch.uint8))
        del u16
        torch.cuda.empty_cache()
        per_config = {"lines": n, "utf8_bytes": int(host.numel()), "gpus": {}}
        for G in sorted({1, min(2, n_gpus)}):
            g = DefinitionReader.reader(corpus.CONFIGS[name][0]).read(devices=list(range(G)))
            eng = g._eng()

            def call(tables):
                res, dt = _ffi.Result(), _ffi.DeviceTables()
                t0 = time.perf_counter()
                if tables:
                    _check(lib.gorp_extract_text_utf8_tables(eng, host.data_ptr(), host.numel(), C.byref(res), C.byref(dt)))
                else:
                    _check(lib.gorp_extract_text_utf8_bytes(eng, host.data_ptr(), host.numel(), C.byref(res)))
                ms = (time.perf_counter() - t0) * 1e3
                nl, w = int(res.n_lines), int(res.span_stride)
                rows_d2h = nl * 4 + (nl + 1) * 8 + nl * w * 4 + (res.n_extractions + 2) * 8
                table_bytes = 0
                if tables:
                    for e in range(dt.n_tables):
                        t = dt.tables[e]
                        r = int(t.n_rows)
                        table_bytes += r * 8
                        for k in range(t.n_columns):
                            values = C.cast(t.d_offsets[k], C.POINTER(C.c_int64))[r]
                            table_bytes += (r + 1) * 8 + values + (r + 7) // 8
                hist = tuple(res.histogram[i] for i in range(res.n_extractions + 2))
                lib.gorp_result_release(eng, C.byref(res))
                return ms, nl, hist, rows_d2h, table_bytes

            call(False)
            call(True)
            ms = {"plain": [], "tables": []}
            digest = {}
            for _ in range(args.runs):
                for kind in ("plain", "tables"):
                    t, nl, hist, rows_d2h, table_bytes = call(kind == "tables")
                    ms[kind].append(round(t, 2))
                    digest[kind] = (nl, hist)
            best = {k: min(v) for k, v in ms.items()}
            per_config["gpus"][str(G)] = {
                "ms_per_call": ms, "best_ms": best,
                "mlines_per_s": {k: round(n / (v / 1e3) / 1e6, 1) for k, v in best.items()},
                "table_bytes": table_bytes, "d2h_bytes": {"plain": rows_d2h, "tables": rows_d2h + table_bytes},
                "same_rows": digest["plain"] == digest["tables"], "tables_minus_plain_ms": round(best["tables"] - best["plain"], 2),
            }
            g.close()
        report["configs"][name] = per_config
        del host
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "host_tables.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
