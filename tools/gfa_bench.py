"""Wall time of the device-formatted text writers on one context, in one call: sage2gpu_write_reads + sage2gpu_write_graph3
(the reference's `.reads` / `.graph3`) against sage2gpu_write_gfa (the same graph as GFA 1.0), alternated, after one warm-up
of each.  Each time is the call's host wall clock: formatting kernels, device-to-host copies and the fwrite into a temporary
directory (the page cache, not the disk).  Reports the card's name and power limit and the size of every file.

Usage: python tools/gfa_bench.py [--sets cfg2] [--reps 5] [--out DIR]   (needs a GPU)."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sage2_b200 import api, synth  # noqa: E402


def timed(fn, path) -> float:
    t0 = time.perf_counter()
    fn(path)
    dt = time.perf_counter() - t0
    os.unlink(path)
    return dt


def bench_set(name: str, reps: int, d: str) -> dict:
    reads, k = synth.config_cached(name)
    b, off = synth.concat(reads)
    g = api.Sage2Gpu(0)
    try:
        g.run_steps123(b, off, k)
        c = g.counters()
        paths = {x: os.path.join(d, "g" + x) for x in (".reads", ".graph3", ".gfa")}
        sizes = {}
        for ext, fn in ((".reads", g.write_reads), (".graph3", g.write_graph3), (".gfa", g.write_gfa)):     # warm-up
            fn(paths[ext])
            sizes[ext] = os.path.getsize(paths[ext])
            os.unlink(paths[ext])
        reads_s, graph3_s, gfa_s = [], [], []
        for _ in range(reps):
            reads_s.append(timed(g.write_reads, paths[".reads"]))
            graph3_s.append(timed(g.write_graph3, paths[".graph3"]))
            gfa_s.append(timed(g.write_gfa, paths[".gfa"]))
        both = [r + q for r, q in zip(reads_s, graph3_s)]
        r3 = lambda v: [round(x, 3) for x in v]     # noqa: E731
        return {"k": k, "unique_reads": c["unique_reads"], "edges": c["n_edges"], "bytes": sizes,
                "write_reads_s": r3(reads_s), "write_graph3_s": r3(graph3_s), "reads_plus_graph3_s": r3(both), "write_gfa_s": r3(gfa_s),
                "reads_plus_graph3_s_median": round(statistics.median(both), 3), "write_gfa_s_median": round(statistics.median(gfa_s), 3)}
    finally:
        g.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", default="cfg2")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for gfa_bench.json (default: the JSON line on stdout only)")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": card[0] if card else "unknown", "sets": {}}
    with tempfile.TemporaryDirectory() as d:
        for name in a.sets.split(","):
            res["sets"][name] = bench_set(name, a.reps, d)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "gfa_bench.json"), "w") as fo:
            json.dump(res, fo, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
