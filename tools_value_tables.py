"""Value tables of a device-resident result (gorp_extract_tables_device) on one GPU, after the UTF-16 and the UTF-8 text calls.

    python tools_value_tables.py [--configs readme:100000000,syslog200:40000000] [--runs 5] [--out DIR]

Corpora: config #2 (`readme`, 100 M lines) and config #4 (`syslog200`, 40 M lines), generated on the device by corpusgen and
narrowed to bytes there for the UTF-8 call (both are ASCII). For each input form, after three warm-up pairs, each run times
with CUDA events on the calling stream the extract call alone, then the extract call followed by the tables call; the
tables call's time is the difference of the two (the tables call needs an extract call right before it). The inputs are
far larger than the 126 MB L2. A separate torch.profiler pass over one tables call gives the device time per kernel. The
bytes the call must move are counted from the tables themselves: ext_id read, the span entries of the matched rows read,
the values read and written, offsets, row indexes and bitmaps written. The caller's alternative today, the same tables
built from the rows with torch (nonzero, cumsum, repeat_interleave, a gather), is timed once per form. The card's name and
power limit are read in the same run. Prints one JSON document (and writes it to DIR/value_tables.json).
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

HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU


def torch_tables(torch, ext, off, sp, base, groups, chunk=1 << 24):
    """What a caller builds today from the rows: per extraction the row indexes, per group offsets, validity and values."""
    out = []
    for e, g in enumerate(groups):
        rows = torch.nonzero(ext == e).flatten()
        cols = []
        starts = off[rows]
        for k in range(g):
            s, t = sp[rows, 2 * k].to(torch.int64), sp[rows, 2 * k + 1].to(torch.int64)
            valid = s >= 0
            ln = torch.where(valid, t - s, 0)
            o = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=ext.device)
            torch.cumsum(ln, 0, out=o[1:])
            data = torch.empty(int(o[-1]), dtype=base.dtype, device=ext.device)
            src0 = starts + torch.where(valid, s, 0)
            for a in range(0, rows.numel(), chunk):
                b = min(a + chunk, rows.numel())
                o0, o1 = int(o[a]), int(o[b])
                lc = ln[a:b]
                idx = torch.repeat_interleave(src0[a:b], lc) + torch.arange(o0, o1, device=ext.device) - torch.repeat_interleave(o[a:b], lc)
                data[o0:o1] = base[idx]
            cols.append((o, valid, data))
        out.append((rows, cols))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="readme:100000000,syslog200:40000000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from gorp_b200 import DefinitionReader, _ffi, corpus, corpusgen, parityhash
    from gorp_b200.api import _check
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs a GPU")
    lib = _ffi.lib
    dev = torch.device("cuda", 0)
    report = {"gpu": gpu_identity(), "runs": args.runs, "hbm_tbps_datasheet": HBM_TBPS, "configs": {}}
    for item in args.configs.split(","):
        name, n = item.split(":")
        n = int(n)
        g = DefinitionReader.reader(corpus.CONFIGS[name][0]).read(devices=[0])
        eng = g._eng()
        n_ext = len(g.getExtractions())
        groups = [g.blob().extraction(e)["n_groups"] for e in range(n_ext)]
        u16 = corpusgen.device_text(name, 0, n, dev)
        assert int(u16.max()) < 0x80, "the corpus must be ASCII to be narrowed to UTF-8 bytes"
        u8 = u16.to(torch.uint8)
        stream = torch.cuda.current_stream(dev)
        st = stream.cuda_stream
        dres = _ffi.DeviceResult()
        dt = _ffi.DeviceTables()

        def extract(form):
            if form == "utf16_text_device":
                _check(lib.gorp_extract_text_device(eng, 0, u16.data_ptr(), u16.numel(), st, 0, C.byref(dres)))
            else:
                _check(lib.gorp_extract_text_utf8_device(eng, 0, u8.data_ptr(), u8.numel(), st, 0, C.byref(dres)))

        def tables():
            _check(lib.gorp_extract_tables_device(eng, 0, st, 0, C.byref(dt)))

        entry = {"lines": n, "utf16_units": int(u16.numel()), "forms": {}}
        for form in ("utf16_text_device", "utf8_text_device"):
            for _ in range(3):
                extract(form)
                tables()
            torch.cuda.synchronize(dev)
            # what the call moves, from the tables of this input
            rows = sum(int(dt.tables[e].n_rows) for e in range(n_ext))
            values = sum(int(dt.tables[e].n_rows) * int(dt.tables[e].n_columns) for e in range(n_ext))
            ub = int(dt.unit_bytes)
            units = 0
            for e in range(n_ext):
                t = dt.tables[e]
                for k in range(t.n_columns):
                    last = torch.as_tensor(parityhash.DeviceArray(int(t.d_offsets[k]) + 8 * int(t.n_rows), (1,), "<i8"), device=dev)
                    units += int(last.item())
            moved = 4 * n + 8 * values + 2 * ub * units + 8 * (values + n_ext) + 8 * rows + values // 8
            both, alone = [], []
            for _ in range(args.runs):
                for with_tables, acc in ((False, alone), (True, both)):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    extract(form)
                    if with_tables:
                        tables()
                    e1.record(stream)
                    e1.synchronize()
                    acc.append(e0.elapsed_time(e1))
            tables_ms = min(both) - min(alone)
            from torch.profiler import ProfilerActivity, profile
            extract(form)
            torch.cuda.synchronize(dev)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                tables()
                torch.cuda.synchronize(dev)
            per = {}
            for ev in prof.events():
                if ev.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                m = re.search(r"(tables_\w+_kernel|scan_\w+_kernel)", ev.name)
                key = ("copy " if ev.name.startswith("Memcpy") else "") + (m.group(1) if m else ev.name[:60])
                per[key] = per.get(key, 0.0) + ev.device_time_total / 1e3
            # the caller's alternative: the same tables from the rows, with torch
            extract(form)
            torch.cuda.synchronize(dev)
            ext = torch.as_tensor(parityhash.DeviceArray(dres.d_ext_id, (n,), "<i4"), device=dev).clone()
            off = torch.as_tensor(parityhash.DeviceArray(dres.d_line_off, (n + 1,), "<i8"), device=dev).clone()
            sp = torch.as_tensor(parityhash.DeviceArray(dres.d_spans, (n, int(dres.span_stride)), "<i4"), device=dev).clone()
            base = u16 if form == "utf16_text_device" else u8
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ref = torch_tables(torch, ext, off, sp, base, groups)
            e1.record(stream)
            e1.synchronize()
            torch_ms = e0.elapsed_time(e1)
            del ref, ext, off, sp
            torch.cuda.empty_cache()
            entry["forms"][form] = {
                "matched_lines": rows, "values": values, "value_units": units, "unit_bytes": ub, "bytes_moved": moved,
                "extract_ms": [round(x, 3) for x in alone], "extract_plus_tables_ms": [round(x, 3) for x in both],
                "tables_ms_best": round(tables_ms, 3),
                "tables_gbps": round(moved / (tables_ms * 1e-3) / 1e9, 1) if tables_ms > 0 else None,
                "share_of_hbm_peak": round(moved / (tables_ms * 1e-3) / (HBM_TBPS * 1e12), 3) if tables_ms > 0 else None,
                "profiler_ms": {"device_ms_total": round(sum(per.values()), 4),
                                "per_kernel_ms": dict(sorted(((k, round(v, 4)) for k, v in per.items()), key=lambda kv: -kv[1]))},
                "torch_reference_ms": round(torch_ms, 3),
            }
        report["configs"][name] = entry
        del u16, u8, g
        torch.cuda.empty_cache()
    text = json.dumps(report, indent=1)
    print(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "value_tables.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
