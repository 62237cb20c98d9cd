"""Compressed-input ingest: the same seeded reads as plain FASTQ, as one gzip member (inflated by host zlib) and as BGZF
(level 6, inflated on the GPU), for cfg2 and optionally a cfg4-sized set.  Reports in one call:

  - the inflate kernel alone (sage2gpu_inflate_bgzf, CUDA events; text far larger than L2, one warm-up call first):
    milliseconds and GB/s of text written;
  - `sage2gpu -M 3` wall clock on each of the three files, repeated and alternated;
  - the card's name and power limit.

Usage: python tools/bgzf_bench.py [--sets cfg2,cfg4] [--reps 3] [--out DIR]   (needs a GPU)."""
from __future__ import annotations

import argparse
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bgzf  # noqa: E402
from sage2_b200 import api, synth  # noqa: E402

BIN = os.path.join(ROOT, "sage2_b200", "sage2gpu")


def _member(t: bytes) -> bytes:
    return bgzf.member(t, 6)


def write_files(name: str, d: str) -> dict:
    reads, k = synth.config(name)
    fq = os.path.join(d, name + ".fastq")
    synth.write_fastq(fq, reads)
    del reads
    text = open(fq, "rb").read()
    t0 = time.time()
    with ProcessPoolExecutor(os.cpu_count()) as ex:
        blob = b"".join(ex.map(_member, bgzf.split(text), chunksize=64)) + bgzf.EOF_MEMBER
    t_bgzf = time.time() - t0
    open(os.path.join(d, name + ".bgzf.fastq.gz"), "wb").write(blob)
    t0 = time.time()
    with gzip.open(os.path.join(d, name + ".fastq.gz"), "wb", compresslevel=6) as f:
        f.write(text)
    t_gz = time.time() - t0
    return {"k": k, "text_bytes": len(text), "bgzf_bytes": len(blob), "gzip_bytes": os.path.getsize(os.path.join(d, name + ".fastq.gz")),
            "bgzf_write_s": round(t_bgzf, 2), "gzip_write_s": round(t_gz, 2), "blob": blob}


def inflate_kernel(blob: bytes, reps: int) -> dict:
    g = api.Sage2Gpu(0)
    try:
        g.inflate_bgzf(blob)                      # warm-up (module load, allocations)
        ms = []
        for _ in range(reps):
            out, m = g.inflate_bgzf(blob)
            ms.append(m)
        return {"text_bytes": len(out), "kernel_ms": [round(x, 3) for x in ms],
                "text_gbps_best": round(len(out) / min(ms) / 1e6, 2), "text_gbps_median": round(len(out) / sorted(ms)[len(ms) // 2] / 1e6, 2)}
    finally:
        g.close()


def cli_wall(files: dict, k: int, reps: int, d: str) -> dict:
    out = {kind: [] for kind in files}
    for r in range(reps):
        for kind, path in files.items():
            o = os.path.join(d, "o_" + kind)
            t0 = time.time()
            subprocess.run([BIN, "-f", path, "-k", str(k), "-o", o, "-p", "g", "-M", "3"], check=True)
            out[kind].append(round(time.time() - t0, 3))
            if r == reps - 1:
                out[kind + "_log_step1"] = [ln.strip() for ln in open(os.path.join(o, "g.log")) if "Parsed and uploaded" in ln or "Records split" in ln]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", default="cfg2")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for bgzf_bench.json (default: the JSON line on stdout only)")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": card[0] if card else "unknown", "zlib": zlib.ZLIB_RUNTIME_VERSION, "host_cpus": os.cpu_count(), "sets": {}}
    with tempfile.TemporaryDirectory() as d:
        for name in a.sets.split(","):
            f = write_files(name, d)
            blob = f.pop("blob")
            f["inflate"] = inflate_kernel(blob, 5)
            del blob
            files = {"plain": os.path.join(d, name + ".fastq"), "gzip": os.path.join(d, name + ".fastq.gz"),
                     "bgzf": os.path.join(d, name + ".bgzf.fastq.gz")}
            f["cli_wall_s"] = cli_wall(files, f["k"], a.reps, d)
            res["sets"][name] = f
            for p in files.values():
                os.unlink(p)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "bgzf_bench.json"), "w") as fo:
            json.dump(res, fo, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
