#!/usr/bin/env python
"""Per-kernel time of the read organisation (load_reads: ingest + sort + dedupe), the table build and the graph stages of
one bench.py step, under torch.profiler with CUDA activities (no Nsight tools needed).

    python tools/stage_kernels.py OUT_DIR [--workloads cfg4,cfg2] [--steps 3] [--warmup 1]

For every workload: one line per kernel and stage (launches and ms per step), the library's stage timers (CUDA events,
from an unprofiled step) and the sizes the sort and table kernels depend on, printed by the library when
SAGE2GPU_STAGE_STATS is set: members of tie runs longer than the in-kernel limit, retry records of the bucketed table
build.  Writes OUT_DIR/stage_kernels_<workload>.json.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def kernel_events(prof):
    out = []
    for e in prof.events():
        if str(getattr(e, "device_type", "")).endswith("CUDA") and e.device_time_total > 0 and "Memcpy" not in e.name and "Memset" not in e.name:
            out.append((re.sub(r"\(.*", "", e.name).strip(), e.device_time_total / 1000.0))
    return out


def captured_stats(fn):
    """Run fn() with SAGE2GPU_STAGE_STATS set and return the library's `sage2gpu stats:` lines (written to fd 2)."""
    os.environ["SAGE2GPU_STAGE_STATS"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["SAGE2GPU_STAGE_STATS"]
        f.seek(0)
        text = f.read().decode(errors="replace")
    stats = {}
    for line in text.splitlines():
        if line.startswith("sage2gpu stats:"):
            parts = line.split()
            stage = parts[2]
            stats[stage] = {k: int(v) for k, v in (p.split("=") for p in parts[3:])}
        elif line.strip():
            sys.stderr.write(line + "\n")
    return stats


def run_workload(name, steps, warmup, out_dir):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    from sage2_b200 import api, synth

    reads, k = synth.config_cached(name)
    bases, offsets = synth.concat(reads)
    n = len(offsets) - 1
    d_b = torch.from_numpy(np.ascontiguousarray(bases)).cuda()
    d_o = torch.from_numpy(np.ascontiguousarray(offsets)).cuda()
    del reads, bases
    gpu = api.Sage2Gpu(0)
    stream = torch.cuda.ExternalStream(gpu.stream_ptr(), device=torch.device("cuda", 0))
    stages = [
        ("organize_reads", lambda: gpu.load_reads_ptr(d_b.data_ptr(), d_o.data_ptr(), n, k, device=True)),
        ("build_table", gpu.build_hash_table),
        ("graph", gpu.build_overlap_graph),
    ]

    def step():
        for _, fn in stages:
            fn()
        stream.synchronize()

    for _ in range(warmup):
        step()
    step()
    timers = gpu.timers()
    counters = gpu.counters()
    stats = captured_stats(step)
    per = collections.defaultdict(lambda: [0, 0.0])
    for _ in range(steps):
        for stage, fn in stages:
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn()
                stream.synchronize()
            for kname, ms in kernel_events(prof):
                per[(stage, kname)][0] += 1
                per[(stage, kname)][1] += ms
    rows = [{"stage": s, "kernel": kn, "launches_per_step": c / steps, "ms_per_step": ms / steps} for (s, kn), (c, ms) in per.items()]
    rows.sort(key=lambda r: (r["stage"], -r["ms_per_step"]))
    totals = collections.defaultdict(float)
    for r in rows:
        totals[r["stage"]] += r["ms_per_step"]
    props = torch.cuda.get_device_properties(0)
    power = None
    try:
        import subprocess
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:       # noqa: BLE001
        pass
    res = {"workload": name, "reads": n, "k": k, "gpu": props.name, "power_limit_and_max_sm_clock": power, "profiled_steps": steps,
           "stage_timers_ms": timers, "stats": stats, "unique_reads": counters["unique_reads"],
           "kernel_ms_per_step_by_stage": dict(totals), "kernels": rows}
    print(f"== {name}: {n} reads, {counters['unique_reads']} unique, {props.name} ({power})")
    print("   stage timers (ms, unprofiled step): " + ", ".join(f"{k2} {v:.2f}" for k2, v in timers.items() if v))
    for stage, st in stats.items():
        print(f"   stats {stage}: " + ", ".join(f"{k2}={v}" for k2, v in st.items()))
    for r in rows:
        if r["stage"] != "graph" or r["ms_per_step"] >= 0.2:
            print(f"   {r['stage']:<15} {r['kernel'][:60]:<60} {r['launches_per_step']:7.1f} launches {r['ms_per_step']:9.3f} ms")
    for s, t in totals.items():
        print(f"   {s:<15} kernels total {t:9.3f} ms")
    with open(os.path.join(out_dir, f"stage_kernels_{name}.json"), "w") as f:
        json.dump(res, f, indent=1)
    gpu.close()
    del d_b, d_o
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out_dir")
    ap.add_argument("--workloads", default="cfg4,cfg2")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    for name in a.workloads.split(","):
        run_workload(name, a.steps, a.warmup, a.out_dir)


if __name__ == "__main__":
    main()
