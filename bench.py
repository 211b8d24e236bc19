#!/usr/bin/env python
"""bench.py — benchmark of the gorp batch extraction path (BASELINE.json metric) over all five BASELINE configs.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path (newline index -> combined DFA -> capture -> result rows -> histogram) over one
batch of synthetic log text resident in HBM. N > 1: one process per GPU (torchrun), lines sharded as independent
contiguous ranges, tables replicated, no data-path collective ("weak" scaling: the same lines per GPU for every N).

  value        config #2 (README definition, 100 M lines per GPU), whole-job lines/s, device-resident C-ABI entry point
  configs[]    the same measurement for config #4 (200 extractions — the config the 40 %-of-HBM target is stated on),
               #5, #3 and #1: {workload, lines, ms_per_step, value, roofline{kernel, frac, whole_step_frac, traffic},
               parity{...}} — config #4 first
  e2e          config #2 through gorp_extract_text with HOST buffers: pinned host text -> H2D -> kernels -> D2H of
               every result array, all inside the timed region
  roofline     dominant kernel of config #2: algorithmic input bytes per launch / its CUDA-event time vs measured HBM peak
  cpu_baseline the oracle's C restatement of the reference loop on the host cores (JVM unavailable here)

Parity inside the bench (the parity tests proper are tests/ -m gpu): per config, the order-independent 64-bit hash of
(line index, ext_id, spans) of the first 1 M lines of every rank's shard computed from the GPU result must equal the hash
computed from the CPU oracle's result for the same lines (regenerated on the CPU: line i of a corpus is a pure function
of (seed, i), gorp_b200/corpusgen.py), the device-generated text must equal the host-generated text there, and the
histogram must equal the per-line outcomes. `parity.corpus_hash` sums all shards: the same number for every GPU count.

--impl reference times the CPU restatement alone (the reference is pure Java; no JVM exists in this image), same
`config` as this arm, on a bounded sample of it per step.

--dump-outputs DIR writes what the last timed step of `value` returned (rank 0's shard) as DIR/<name>.npy, so that two
builds can be compared output for output: the whole histogram, and ext_id / line_off / spans of a fixed, seeded sample of
lines (line_index) sized to keep all files under 64 MB. Integers are stored exactly: float32 for ext_id, float64 for the rest.
The corpus is a pure function of (workload, line index), so the same arguments give the same inputs on every run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the bench writes nothing into the tree (it may be read-only)

import numpy as np  # noqa: E402

METRIC = "log lines/sec and input GB/s per B200 (match+capture)"
# --workload: BASELINE.json configs; the headline (default) is config #2, the one the metric is quoted on for 1 GPU
WORKLOADS = {
    "readme": ("config#2 README Put/Get/OtherRequest 3-extraction definition, synthetic access-log lines", 1_000_000),
    "simple": ("config#1 samples/simple.grp, synthetic matching/non-matching lines", 1_000_000),
    "weblog": ("config#3 ~20-extraction nginx/Apache access+error definition with parametric templates, mixed line lengths", 200_000),
    "syslog200": ("config#4 200-extraction definition, combined DFA outgrows shared memory", 200_000),
    "utf16mix": ("config#5 nginx/Apache definition, non-ASCII UTF-16 + divergence characters + 10 KB outlier lines", 200_000),
}
PREFIX_LINES = 1_000_000          # per rank: lines whose GPU rows are compared with the CPU oracle's (hash + histogram)
CONFIG5_TOTAL_LINES = 281_600_000  # config #5: 100 GB of UTF-16 (355 B per line on average), sharded over the ranks
EXTRA_CONFIGS = ["syslog200", "utf16mix", "weblog", "simple"]  # configs[] order: the 40 %-target config first
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # written by tools_ncu_traffic.py from an ncu --set full capture
DUMP_BYTES = 56 << 20  # --dump-outputs: all .npy files together stay below 64 MB
DUMP_SEED = 0x5EED00D0  # --dump-outputs: the sampled lines depend on this seed and the line count only


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """{workload: {kernel: {"dram_bytes_per_text_byte": x, "source": file}}} from the committed ncu capture, or {}."""
    try:
        return json.load(open(TRAFFIC_FILE))
    except Exception:  # noqa: BLE001
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.t0, self.t1 = index, None, [], None, None

    def launch(self):
        """Start nvidia-smi early (it needs ~0.1-0.3 s to come up); only the samples taken between start() and stop()
        are reported."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)

            def pump():
                for ln in self.proc.stdout:
                    self.lines.append((time.perf_counter(), ln))
            self.t = threading.Thread(target=pump, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def start(self):
        if self.proc is None:
            self.launch()
        self.t0 = time.perf_counter()

    def stop(self):
        self.t1 = time.perf_counter()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)  # let the sample that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [ln for (t, ln) in self.lines if self.t0 <= t <= self.t1 + 0.06]
        if not inside and self.lines:  # region shorter than the sampling period: the sample closest to it
            inside = [min(self.lines, key=lambda x: abs(x[0] - self.t1))[1]]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_lines(workload, first_line, n):
    """Lines [first_line, first_line + n) of the workload's corpus, generated on the CPU (gorp_b200/corpusgen.py: line i is
    a pure function of (seed, i); the GPU shards hold the same units, generated on the device)."""
    from gorp_b200 import corpusgen
    return corpusgen.host_text(workload, first_line, n)


def definition_of(workload):
    from gorp_b200 import corpus
    return corpus.CONFIGS[workload][0]


def config_dict(workload, lines_per_gpu, world, n_bins):
    """The `config` object of a bench line; the reference arm prints the same object."""
    desc, _ = WORKLOADS[workload]
    return {"workload": desc, "lines_per_gpu": lines_per_gpu, "lines": lines_per_gpu * world,
            "corpus": "counter-based generator: line i = f(seed, i), no tiling; rank r holds lines [r*L, (r+1)*L), generated on the device",
            "l2": "the input of a step (GBs per GPU) is far larger than L2, no flush needed",
            "parallelism": "lines sharded per GPU as contiguous ranges, tables replicated; no data-path collective"
                           + (", one NCCL all-reduce of the %d-bin histogram per step" % n_bins if world > 1 else "")}


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU algorithm (C restatement, all host threads). Same config as the GPU arm; every
    step processes a bounded sample of it (as many lines of the workload as keep the whole run within a few minutes)."""
    if rank != 0:
        return
    from oracle import gorp_oracle
    cores = os.cpu_count() or 1
    o = gorp_oracle.Gorp(definition_of(args.workload))
    probe = host_lines(args.workload, 0, 200_000)
    pst = gorp_oracle.split_lines(probe)
    o.extract_batch(probe, pst, threads=cores)  # build + page-in
    t0 = time.perf_counter()
    o.extract_batch(probe, pst, threads=cores)
    rate = len(pst[0]) / max(time.perf_counter() - t0, 1e-6)
    total_lines = args.lines_per_gpu * world
    budget = args.ref_budget_s / max(args.steps + args.warmup, 1)
    sample_lines = total_lines if args.ref_lines == 0 else args.ref_lines
    sample_lines = int(min(sample_lines, max(rate * budget * 0.8, 200_000)))
    text = host_lines(args.workload, 0, sample_lines)
    starts, ends = gorp_oracle.split_lines(text)
    for _ in range(args.warmup):
        o.extract_batch(text, (starts, ends), threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.extract_batch(text, (starts, ends), threads=cores)
    dt = (time.perf_counter() - t0) / args.steps
    n = len(starts)
    val = n / dt
    n_bins = len(o.extractions) + 2
    sample = "the first %d lines (%.2f GB UTF-16) of the config's %d lines per step, all %d host threads" % (n, text.nbytes / 1e9, total_lines, cores)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "lines/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16", "data": "synthetic", "input_gb_per_s": text.nbytes / dt / 1e9,
        "config": config_dict(args.workload, args.lines_per_gpu, world, n_bins),
        "reference_note": "the reference is pure Java and no JVM exists in this image: C restatement of Gorp.extract "
                          "(oracle/gorp_oracle.c), one extract per line, static partition over host threads; a rate metric, "
                          "measured on a bounded sample of the config per step",
        "cpu_baseline": {"value": val, "unit": "lines/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "lines/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def dump_outputs(out_dir, dres, n_bins, dev):
    """Writes the gorp_device_result of the last call as DIR/<name>.npy: n_lines and the histogram whole, the per-line
    arrays at a seeded sample of lines (line_index; every line when they fit): ext_id[i], (line_off[i], line_off[i + 1])
    and the span row of line i."""
    import torch
    from gorp_b200 import parityhash
    n, stride = int(dres.n_lines), int(dres.span_stride)
    ext_t, sp_t = parityhash.device_results(dres, dev)
    off_t = torch.as_tensor(parityhash.DeviceArray(dres.d_line_off, (n + 1,), "<i8"), device=dev)
    hist_t = torch.as_tensor(parityhash.DeviceArray(dres.d_histogram, (n_bins,), "<i8"), device=dev)
    per_line = 8 + 4 + 16 + 8 * stride
    n_sample = min(n, (DUMP_BYTES - 8 * (n_bins + 1)) // per_line)
    idx = np.arange(n) if n_sample == n else np.sort(np.random.default_rng(DUMP_SEED).choice(n, n_sample, replace=False))
    idx_t = torch.from_numpy(idx).to(dev)
    arrays = {"n_lines": np.array([n], dtype=np.float64),
              "histogram": hist_t.cpu().numpy().astype(np.float64),
              "line_index": idx.astype(np.float64),
              "ext_id": ext_t[idx_t].cpu().numpy().astype(np.float32),
              "line_off": torch.stack((off_t[idx_t], off_t[idx_t + 1]), dim=1).cpu().numpy().astype(np.float64),
              "spans": sp_t[idx_t].cpu().numpy().astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print("[bench] outputs of the last timed step: %d of %d lines -> %s" % (n_sample, n, out_dir), file=sys.stderr)


class Env:
    pass


def bind_numa(cudart, index):
    """Bind this rank (CPU affinity + preferred memory node) to the NUMA node of its GPU, so that the pinned host buffers of
    the end-to-end leg are local to the GPU's PCIe root: with 8 ranks on two sockets the H2D copies would otherwise cross the
    socket interconnect. Returns what was done (reported in the bench line)."""
    import ctypes
    import platform
    info = {"node": None, "cpus": None, "mempolicy": None}
    try:
        err, bdf = cudart.cudaDeviceGetPCIBusId(32, index)
        bdf = (bdf.decode() if isinstance(bdf, bytes) else str(bdf)).split(chr(0))[0].strip().lower()
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return info
        info["node"] = node
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus & os.sched_getaffinity(0) or cpus)
            info["cpus"] = len(os.sched_getaffinity(0))
        nr = {"x86_64": 238, "aarch64": 237}.get(platform.machine())
        if nr is not None:
            mask = (ctypes.c_ulong * 16)()
            mask[node // (8 * ctypes.sizeof(ctypes.c_ulong))] |= 1 << (node % (8 * ctypes.sizeof(ctypes.c_ulong)))
            rc = ctypes.CDLL(None, use_errno=True).syscall(nr, 1, mask, 16 * 8 * ctypes.sizeof(ctypes.c_ulong) + 1)  # MPOL_PREFERRED
            info["mempolicy"] = "preferred" if rc == 0 else "errno %d" % ctypes.get_errno()
    except Exception as ex:  # noqa: BLE001
        info["error"] = str(ex)[:120]
    return info


def device_config_run(env, workload, lines_per_gpu, steps, warmup, sampler=None, keep=False, first_line=None, corpus_note=None,
                      dump_dir=None):
    """One config, device-resident: returns the result dict (and, with keep=True, the engine / text for the e2e leg)."""
    torch, dist, lib, _ffi, Blob, _check, cudart = env.torch, env.dist, env.lib, env.ffi, env.Blob, env.check, env.cudart
    from gorp_b200 import corpusgen, parityhash, sharding
    from oracle import gorp_oracle
    rank, world, dev = env.rank, env.world, env.dev
    desc, _ = WORKLOADS[workload]
    n_lines = lines_per_gpu
    first_line = rank * n_lines if first_line is None else first_line
    t0 = time.perf_counter()
    d_text = corpusgen.device_text(workload, first_line, n_lines, dev)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    n_units = d_text.numel()
    in_bytes = n_units * 2
    blob = Blob.from_definition(definition_of(workload))
    n_bins = blob.info()[2] + 2
    eng = C.c_void_p()
    devs = (C.c_int * 1)(env.local_rank)
    t0 = time.perf_counter()
    _check(lib.gorp_engine_create(blob._ptr, blob.length, devs, 1, C.byref(eng)))
    create_s = time.perf_counter() - t0
    stream = torch.cuda.current_stream().cuda_stream
    dres = _ffi.DeviceResult()
    d_hist = torch.zeros(n_bins, dtype=torch.int64, device=dev)

    # the prefix of this rank's shard on the CPU: the same generator (line i = f(seed, i)), then the oracle
    n_prefix = min(PREFIX_LINES, n_lines)
    prefix = host_lines(workload, first_line, n_prefix)
    assert (d_text[:prefix.size].cpu().numpy().view(np.uint16) == prefix).all(), "device-generated text differs from the host-generated text"
    o = gorp_oracle.Gorp(definition_of(workload))
    cores = os.cpu_count() or 1
    pst = gorp_oracle.split_lines(prefix)
    oe, osp = o.extract_batch(prefix, pst, threads=cores)

    def step(flags=0):
        _check(lib.gorp_extract_text_device(eng, 0, d_text.data_ptr(), n_units, stream, flags, C.byref(dres)))
        if world > 1:
            # the one (optional) collective of the path: all-reduce of the per-extraction histogram, every step
            (err,) = cudart.cudaMemcpyAsync(d_hist.data_ptr(), dres.d_histogram, n_bins * 8, cudart.cudaMemcpyKind.cudaMemcpyDeviceToDevice, stream)
            assert int(err) == 0, err
            sharding.allreduce_histogram(d_hist)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        step()
    torch.cuda.synchronize()
    assert dres.n_lines == n_lines, (dres.n_lines, n_lines)
    # parity at full size: rows of the shard's first lines (GPU result of the timed path) vs the oracle's rows — per-line
    # outcomes through the 64-bit hash, and the whole shard's hash for the corpus hash (identical for every GPU count)
    stride = int(dres.span_stride)
    ext_t, sp_t = parityhash.device_results(dres, dev)
    gpu_prefix = parityhash.hash_torch(first_line, ext_t[:n_prefix], sp_t[:n_prefix])
    gpu_total = parityhash.hash_torch(first_line, ext_t, sp_t)
    cpu_prefix = parityhash.hash_numpy(first_line, oe, osp[:, :stride])
    if not os.environ.get("GORP_BENCH_TIMING_ONLY"):  # kernel diagnostics that break the results on purpose (never a bench value)
        assert gpu_prefix == cpu_prefix, "parity hash mismatch on %s: gpu %x cpu %x" % (workload, gpu_prefix, cpu_prefix)
    local_hist = torch.zeros(n_bins, dtype=torch.int64, device=dev)
    (err,) = cudart.cudaMemcpyAsync(local_hist.data_ptr(), dres.d_histogram, n_bins * 8, cudart.cudaMemcpyKind.cudaMemcpyDeviceToDevice, stream)
    assert int(err) == 0, err
    torch.cuda.synchronize()
    bins = torch.where(ext_t >= 0, ext_t, torch.where(ext_t == -1, n_bins - 2, n_bins - 1)).to(torch.int64)
    assert (torch.bincount(bins, minlength=n_bins) == local_hist).all(), "histogram differs from the per-line outcomes"
    del ext_t, sp_t, bins
    names = (C.c_char_p * 16)()
    tot = (C.c_double * 16)()
    cnt, calls, launches = C.c_int(), C.c_int64(), C.c_int64()
    _check(lib.gorp_kernel_times(eng, 0, names, tot, 16, C.byref(cnt), C.byref(calls), C.byref(launches), 1))

    barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    per_step = []
    gap_ms = float(os.environ.get("GORP_BENCH_GAP_MS", "0"))  # diagnostics only: idle time between steps
    for _ in range(steps):
        if os.environ.get("GORP_BENCH_PER_STEP"):  # diagnostics only: a pair of events per step
            if gap_ms:
                torch.cuda.synchronize()
                time.sleep(gap_ms / 1e3)
            ev0 = torch.cuda.Event(enable_timing=True)
            ev0.record()
        step(_ffi.FLAG_TIME_KERNELS)
        if os.environ.get("GORP_BENCH_PER_STEP"):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            per_step.append((ev0, ev))
    e1.record()
    barrier()
    if per_step:
        print("[bench] %s ms per step:" % workload, [round(a.elapsed_time(b), 2) for a, b in per_step], file=sys.stderr)
    clocks = sampler.stop() if sampler else None
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, dres, n_bins, dev)
    ms = e0.elapsed_time(e1) / steps
    if world > 1:  # every rank holds the job-wide histogram: its sum is the job's line count
        assert int(d_hist.sum().item()) == n_lines * world, (int(d_hist.sum().item()), n_lines * world)
    _check(lib.gorp_kernel_times(eng, 0, names, tot, 16, C.byref(cnt), C.byref(calls), C.byref(launches), 1))
    kern = {}
    for i in range(cnt.value):  # a kernel that is marked twice in one call (retry) adds up
        kern[names[i].decode()] = kern.get(names[i].decode(), 0.0) + tot[i] / max(calls.value, 1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    h = torch.tensor([gpu_total & 0xFFFFFFFF, gpu_total >> 32, in_bytes], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(h, op=dist.ReduceOp.SUM)  # 64-bit modular sum over ranks: 32-bit halves, carried below
    ms_max = float(t.item())
    corpus_hash = (int(h[0].item()) + (int(h[1].item()) << 32)) & ((1 << 64) - 1)
    job_bytes = int(h[2].item())
    total_lines = n_lines * world
    peak, peak_src = hbm_peak()
    dom = max(kern, key=kern.get) if kern else None
    roof = None
    if dom:
        ach = in_bytes / (kern[dom] / 1e3) / 1e9
        tr = ncu_traffic().get(workload, {})
        per_kernel = {k: v["dram_bytes_per_text_byte"] * in_bytes for k, v in tr.items() if k in kern}
        roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": per_kernel.get(dom),
                "traffic_step": sum(per_kernel.values()) if per_kernel else None,
                "traffic_source": ("ncu dram__bytes_read.sum + dram__bytes_write.sum per text byte (%s) x bytes of this launch"
                                   % tr[dom]["source"]) if dom in tr else None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": in_bytes,
                "kernel_ms": kern[dom], "all_kernels_ms": kern,
                "whole_step_frac": (job_bytes / world / (ms_max / 1e3) / 1e9) / peak,
                "whole_step_frac_of_8TBps": (job_bytes / world / (ms_max / 1e3) / 1e9) / 8000.0,
                "whole_step_note": "job input bytes / (n_gpus x step time x HBM peak): the aggregate HBM-read roofline fraction"}
    cfg = config_dict(workload, lines_per_gpu, world, n_bins)
    if corpus_note:
        cfg["corpus"] += "; " + corpus_note
    out = {"workload": desc, "key": workload, "lines": total_lines, "lines_per_gpu": n_lines, "bytes_per_gpu": in_bytes,
           "job_bytes": job_bytes, "ms_per_step": ms_max, "value": total_lines / (ms_max / 1e3), "unit": "lines/s",
           "input_gb_per_s": job_bytes / (ms_max / 1e3) / 1e9, "steps": steps, "roofline": roof,
           "parity": {"prefix_lines_per_rank": n_prefix, "prefix_hash_gpu": "%016x" % gpu_prefix,
                      "prefix_hash_cpu_oracle": "%016x" % cpu_prefix, "prefix_equal": True,
                      "device_text_equals_host_text_on_prefix": True,
                      "corpus_hash": "%016x" % corpus_hash, "corpus_lines": total_lines,
                      "histogram_equals_per_line_outcomes": True,
                      "what": "order-independent 64-bit hash of (global line index, ext_id, spans) — gorp_b200/parityhash.py; the "
                              "corpus hash sums every rank's shard and is the same number for every GPU count over the same lines"},
           "gpu_launches": int(launches.value), "engine_create_s": create_s, "corpus_generate_s": gen_s, "config": cfg}
    # CPU baseline on rank 0: bounded sample of the same workload
    if rank == 0 and not env.args.skip_cpu:
        c_lines = min(env.args.cpu_lines, n_lines)
        ctext = prefix if c_lines <= n_prefix else host_lines(workload, first_line, c_lines)
        cst = pst if c_lines <= n_prefix else gorp_oracle.split_lines(ctext)
        t0 = time.perf_counter()
        o.extract_batch(ctext, cst, threads=cores)
        cdt = time.perf_counter() - t0
        one = 200_000
        t0 = time.perf_counter()
        o.extract_batch(prefix, (pst[0][:one], pst[1][:one]), threads=1)
        cdt1 = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": len(cst[0]) / cdt, "unit": "lines/s", "cores": cores, "kind": "port",
                               "sample": "the first %d lines (%.2f GB) of the same workload, all %d host threads; 1 thread: %.0f lines/s"
                                         % (len(cst[0]), ctext.nbytes / 1e9, cores, min(one, len(pst[0])) / cdt1),
                               "note": "C restatement of the reference's Gorp.extract loop (JVM unavailable in this image)"}
    if keep:
        return out, clocks, (eng, d_text, n_lines, n_units, in_bytes, barrier)
    del d_text
    lib.gorp_engine_destroy(eng)
    torch.cuda.empty_cache()
    return out, clocks, None


def e2e_run(env, kept, workload):
    """config #2 end to end through the host-buffer C ABI (H2D + kernels + D2H inside the timed region)."""
    torch, dist, lib, _ffi, _check = env.torch, env.dist, env.lib, env.ffi, env.check
    eng, d_text, n_lines, n_units, in_bytes, barrier = kept
    world, dev, args = env.world, env.dev, env.args
    try:
        if args.skip_e2e:
            raise RuntimeError("skipped (--skip-e2e)")
        avail_gb = 0.0
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                avail_gb = int(ln.split()[1]) / 1e6
        per_rank_gb = in_bytes / 1e9 * 1.6
        frac = 1.0 if avail_gb > per_rank_gb * world * 1.5 + 16 else max(0.01, (avail_gb - 16) / (per_rank_gb * world * 1.5))
        # the host batch = the leading part of this rank's shard (cut after a '\n'), copied out of HBM once, outside the timed region
        e2e_units = n_units
        if frac < 1.0:
            cut = int(n_units * frac)
            nl = torch.nonzero(d_text[cut:cut + 100000] == 10)
            e2e_units = cut + int(nl[0].item()) + 1
        h_text = torch.empty(e2e_units, dtype=torch.int16).pin_memory()
        h_text.copy_(d_text[:e2e_units])
        h_np = h_text.numpy().view(np.uint16)
        res = _ffi.Result()

        def e2e_step():
            _check(lib.gorp_extract_text(eng, h_np.ctypes.data, h_np.size, C.byref(res)))
            nl, ns = res.n_lines, res.n_lines * res.span_stride
            lib.gorp_result_release(eng, C.byref(res))
            return nl, ns
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            nl, ns = e2e_step()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        ll = torch.tensor([nl], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(ll, op=dist.ReduceOp.SUM)
        d2h = nl * 4 + (nl + 1) * 8 + ns * 4 + 5 * 8
        e2e = {"value": int(ll.item()) / float(tt.item()), "unit": "lines/s", "h2d_bytes_per_step": int(h_np.size * 2),
               "d2h_bytes_per_step": int(d2h), "lines_per_step_per_gpu": int(nl), "ms_per_step": float(tt.item()) * 1e3,
               "h2d_gb_per_s_per_gpu": h_np.size * 2 / float(tt.item()) / 1e9, "numa": env.numa,
               "timing": "host wall clock around gorp_extract_text (it returns after the last D2H), max over ranks"}
        # the platform's ceiling for this leg: the same pinned buffer copied host -> device by all ranks at once, nothing else
        d_scratch = torch.empty_like(d_text[:e2e_units])
        d_scratch.copy_(h_text, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            d_scratch.copy_(h_text, non_blocking=True)
        torch.cuda.synchronize()
        tc = torch.tensor([(time.perf_counter() - t0) / 2], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        e2e["h2d_ceiling_gb_per_s_per_gpu"] = h_np.size * 2 / float(tc.item()) / 1e9
        e2e["h2d_ceiling_note"] = "plain cudaMemcpyAsync of the same pinned text by all %d ranks at once (max over ranks)" % world
        del d_scratch
        # the same call fed with ISO-8859-1 bytes (what a JDK 9+ String with the LATIN1 coder holds; the synthetic corpus is
        # ASCII): gorp_extract_text_latin1 widens on the device, the host-to-device copy moves half the bytes
        if int(d_text.max().item()) < 256 and int(d_text.min().item()) >= 0:
            h8 = torch.empty(e2e_units, dtype=torch.uint8).pin_memory()
            h8.copy_(d_text[:e2e_units].to(torch.uint8))
            h8_np = h8.numpy()

            def e2e8_step():
                _check(lib.gorp_extract_text_latin1(eng, h8_np.ctypes.data, h8_np.size, C.byref(res)))
                nl8 = res.n_lines
                lib.gorp_result_release(eng, C.byref(res))
                return nl8
            assert e2e8_step() == nl
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                e2e8_step()
            torch.cuda.synchronize()
            dt8 = (time.perf_counter() - t0) / args.e2e_steps
            tt8 = torch.tensor([dt8], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt8, op=dist.ReduceOp.MAX)
            e2e["latin1_input"] = {"value": int(ll.item()) / float(tt8.item()), "unit": "lines/s", "h2d_bytes_per_step": int(h8_np.size),
                                   "d2h_bytes_per_step": int(d2h), "ms_per_step": float(tt8.item()) * 1e3,
                                   "call": "gorp_extract_text_latin1 (ISO-8859-1 bytes in, widened to UTF-16 on the device)"}
            # ... and with UTF-8 bytes (what the reference's InputLineReader reads from a log file, io/InputLineReader.java:51;
            # the ASCII corpus is its own UTF-8): validated and decoded on the device
            def e2eu_step():
                _check(lib.gorp_extract_text_utf8(eng, h8_np.ctypes.data, h8_np.size, C.byref(res)))
                nlu = res.n_lines
                lib.gorp_result_release(eng, C.byref(res))
                return nlu
            assert e2eu_step() == nl
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                e2eu_step()
            torch.cuda.synchronize()
            ttu = torch.tensor([(time.perf_counter() - t0) / args.e2e_steps], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(ttu, op=dist.ReduceOp.MAX)
            e2e["utf8_input"] = {"value": int(ll.item()) / float(ttu.item()), "unit": "lines/s", "h2d_bytes_per_step": int(h8_np.size),
                                 "d2h_bytes_per_step": int(d2h), "ms_per_step": float(ttu.item()) * 1e3,
                                 "call": "gorp_extract_text_utf8 (UTF-8 bytes in, decoded to UTF-16 on the device)"}
            h8_np = None  # (the numpy view keeps the pinned buffer alive)
            del h8
        # the List<String> form (Gorp.extractAll(List<String>), Gorp.java:145-147): the same lines as one concatenation without
        # separators plus n + 1 offsets, on a bounded share of the batch (the offsets are another 8 bytes per line of pinned memory)
        ln_lines = min(int(nl), 25_000_000)
        d_off = torch.nonzero(d_text[:e2e_units] == 10).flatten()[:ln_lines] + 1  # starts of lines 1 .. ln_lines
        cut_units = int(d_off[-1].item())
        keep = d_text[:cut_units] != 10
        h_lt = torch.empty(cut_units - ln_lines, dtype=torch.int16).pin_memory()
        h_lt.copy_(d_text[:cut_units][keep])
        h_lo = torch.zeros(ln_lines + 1, dtype=torch.int64).pin_memory()
        h_lo[1:].copy_(d_off - torch.arange(1, ln_lines + 1, device=dev))
        del d_off, keep
        lt_np, lo_np = h_lt.numpy().view(np.uint16), h_lo.numpy()

        def e2el_step():
            _check(lib.gorp_extract_lines(eng, lt_np.ctypes.data, lo_np.ctypes.data, ln_lines, C.byref(res)))
            nll = res.n_lines
            lib.gorp_result_release(eng, C.byref(res))
            return nll
        assert e2el_step() == ln_lines
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2el_step()
        torch.cuda.synchronize()
        ttl = torch.tensor([(time.perf_counter() - t0) / args.e2e_steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ttl, op=dist.ReduceOp.MAX)
        e2e["lines_form"] = {"value": ln_lines * world / float(ttl.item()), "unit": "lines/s", "lines_per_step_per_gpu": ln_lines,
                             "h2d_bytes_per_step": int(lt_np.size * 2 + lo_np.size * 8), "d2h_bytes_per_step": int(d2h * ln_lines // max(int(nl), 1)),
                             "ms_per_step": float(ttl.item()) * 1e3,
                             "call": "gorp_extract_lines (concatenated strings + offsets: the List<String> form)"}
        del h_lt, h_lo
        del h_text
    except Exception as ex:  # noqa: BLE001
        e2e = {"value": None, "unit": "lines/s", "error": str(ex)[:200]}
    return e2e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--lines-per-gpu", type=int, default=100_000_000)
    ap.add_argument("--config-lines-per-gpu", type=int, default=40_000_000, help="lines per GPU of the configs[] entries")
    ap.add_argument("--config-steps", type=int, default=10)
    ap.add_argument("--configs", default=",".join(EXTRA_CONFIGS), help="comma-separated extra configs ('' = none)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--ref-lines", type=int, default=0, help="reference arm: lines per step (0 = the config's, bounded by --ref-budget-s)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="reference arm: wall-clock budget of the whole run")
    ap.add_argument("--cpu-lines", type=int, default=16_000_000)
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs only")
    ap.add_argument("--no-clock-sampler", action="store_true", help="diagnostics: do not run nvidia-smi beside the timed region")
    ap.add_argument("--workload", default="readme", choices=sorted(WORKLOADS), help="BASELINE.json config of `value` (default: #2, the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step of `value` as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from gorp_b200 import build as gbuild
    gbuild.build()
    from gorp_b200 import _ffi
    from gorp_b200.api import Blob, _check
    try:
        from cuda.bindings import runtime as cudart
    except Exception:  # noqa: BLE001
        from cuda import cudart

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_numa(cudart, local_rank) if not os.environ.get("GORP_BENCH_NO_NUMA") else {"node": None, "disabled": True}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    env = Env()
    env.numa = numa
    env.torch, env.dist, env.lib, env.ffi, env.Blob, env.check, env.cudart = torch, dist, _ffi.lib, _ffi, Blob, _check, cudart
    env.rank, env.local_rank, env.world, env.dev, env.args = rank, local_rank, world, dev, args

    sampler = ClockSampler(local_rank)
    if not args.no_clock_sampler:
        sampler.launch()
    head, clocks, kept = device_config_run(env, args.workload, args.lines_per_gpu, args.steps, args.warmup, sampler=sampler, keep=True,
                                           dump_dir=args.dump_outputs)
    e2e = e2e_run(env, kept, args.workload)
    env.lib.gorp_engine_destroy(kept[0])
    kept = None
    torch.cuda.empty_cache()

    configs = []
    for w in [x for x in args.configs.split(",") if x and x != args.workload]:
        try:
            lines = min(args.config_lines_per_gpu, args.lines_per_gpu)
            note, steps = None, args.config_steps
            if w == "utf16mix" and args.lines_per_gpu >= 100_000_000:
                # config #5 as specified: a 100 GB corpus sharded over 2 / 4 / 8 GPUs; one GPU runs one shard of the 8-way split
                lines = CONFIG5_TOTAL_LINES // max(world, 8 if world == 1 else world)
                note = ("the 100 GB corpus (%d lines) sharded over %d GPUs" % (CONFIG5_TOTAL_LINES, world) if world > 1 else
                        "1 GPU: the first shard of the 8-way split of the 100 GB corpus (%d of %d lines)" % (lines, CONFIG5_TOTAL_LINES))
                steps = args.config_steps if lines <= 40_000_000 else max(3, args.config_steps * 40_000_000 // lines)
            c, _, _ = device_config_run(env, w, lines, steps, 3, corpus_note=note)
            configs.append(c)
        except Exception as ex:  # noqa: BLE001  (a failing extra config must not hide the headline)
            configs.append({"key": w, "workload": WORKLOADS[w][0], "error": "%s: %s" % (type(ex).__name__, str(ex)[:300])})
            torch.cuda.empty_cache()

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": head["value"], "unit": "lines/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16",
            "data": "synthetic", "input_gb_per_s": head["input_gb_per_s"],
            "config": head["config"], "roofline": head["roofline"], "cpu_baseline": head.get("cpu_baseline"), "e2e": e2e, "clocks": clocks,
            "gpu_launches": head["gpu_launches"], "parity": head["parity"],
            "configs": configs,
        }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
