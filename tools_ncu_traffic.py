#!/usr/bin/env python
"""DRAM traffic per kernel and text byte from an ncu metrics pass, for bench.py's `roofline.traffic`.

    ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none --csv \
        --log-file gpurun_out/T_<workload>.csv python bench.py --workload <workload> --steps 1 --warmup 3 \
        --lines-per-gpu N --skip-e2e --skip-cpu --configs "" > gpurun_out/T_<workload>.json
    python tools_ncu_traffic.py profiles/ncu_traffic.json <workload> gpurun_out/T_<workload>.csv gpurun_out/T_<workload>.json

The LAST launch of every kernel in the log belongs to the timed step (warm-ups and the parity prefix come first). The
result is merged into the JSON file: {workload: {timer name: {"dram_bytes_per_text_byte": x, "dram_read": r, "dram_write": w,
"ncu_time_ms": t, "source": csv}}} — bench.py multiplies by the bytes of its own launch."""
import csv
import json
import os
import sys

TIMER_OF = [("nl_count", "k1_count_newlines"), ("scan_", "scan_tiles"), ("nl_scatter", "k1_scatter_newlines"), ("nl_finish", "k1_scatter_newlines"),
            ("k1_finish", "k1_scatter_newlines"), ("linewalk", "k2b_linewalk_scan"), ("histogram", "k3_histogram"), ("bucket_", "k4b_bucket"),
            ("tailwalk", "k4c_tailwalk"), ("tail_long", "k4c_tailwalk"), ("capwalk", "k4b_capwalk"), ("dfa_direct", "k2_dfa_scan"),
            ("dfa_scan", "k2_dfa_scan"), ("tdfa", "k4_tdfa_capture")]


def main():
    out_path, workload, csv_path, json_path = sys.argv[1:5]
    bench = json.loads([ln for ln in open(json_path) if ln.startswith("{")][-1])
    text_bytes = bench["config"].get("bytes_per_gpu") or bench["roofline"]["algorithmic_bytes_per_launch"]
    timers = set(bench["roofline"]["all_kernels_ms"])
    rows = list(csv.reader(ln for ln in open(csv_path) if ln.startswith('"')))
    hdr = rows[0]
    i_name, i_metric, i_val, i_id = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("ID")
    last = {}  # kernel name -> {metric: value} of its last launch
    for r in rows[1:]:
        name = r[i_name].split("(")[0].split("::")[-1]
        ent = last.setdefault(name, {"id": -1})
        if int(r[i_id]) > ent["id"]:
            last[name] = ent = {"id": int(r[i_id])}
        if int(r[i_id]) == ent["id"]:
            ent[r[i_metric]] = float(r[i_val].replace(",", ""))
    agg = {}
    for name, m in last.items():
        timer = next((t for k, t in TIMER_OF if k in name), None)
        if timer == "k4c_tailwalk" and "k4c_fusedwalk" in timers:  # the same kernel in "all" mode (small definitions)
            timer = "k4c_fusedwalk"
        if timer is None or timer not in timers:
            continue
        a = agg.setdefault(timer, {"dram_read": 0.0, "dram_write": 0.0, "ncu_time_ms": 0.0, "kernels": []})
        a["dram_read"] += m.get("dram__bytes_read.sum", 0.0)
        a["dram_write"] += m.get("dram__bytes_write.sum", 0.0)
        a["ncu_time_ms"] += m.get("gpu__time_duration.sum", 0.0) / 1e6
        a["kernels"].append(name)
    for a in agg.values():
        a["dram_bytes_per_text_byte"] = (a["dram_read"] + a["dram_write"]) / text_bytes
        a["source"] = os.path.basename(csv_path)
        a["text_bytes_of_the_capture"] = text_bytes
    data = json.load(open(out_path)) if os.path.exists(out_path) else {}
    data[workload] = agg
    json.dump(data, open(out_path, "w"), indent=1, sort_keys=True)
    tot = sum(a["dram_read"] + a["dram_write"] for a in agg.values())
    print("%s: %d kernels, step DRAM traffic %.2f GB for %.2f GB of text (%.2fx); read %.2fx" % (
        workload, len(agg), tot / 1e9, text_bytes / 1e9, tot / text_bytes, sum(a["dram_read"] for a in agg.values()) / text_bytes))
    for t, a in sorted(agg.items(), key=lambda kv: -kv[1]["ncu_time_ms"]):
        print("  %-22s %7.3f ms  read %.2fx  write %.2fx" % (t, a["ncu_time_ms"], a["dram_read"] / text_bytes, a["dram_write"] / text_bytes))


if __name__ == "__main__":
    main()
