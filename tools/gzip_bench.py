"""Ordinary gzip ingest on the GPU: the same seeded reads as plain FASTQ, as one gzip member (level 6, as `gzip` writes it)
and as BGZF (level 6), for cfg2 and optionally a cfg4-sized set.  Reports in one call:

  - the card's name and power limit;
  - the device inflate of the gzip file alone (sage2gpu_inflate_gzip: the sum of its kernels' CUDA-event times, and the call's
    wall clock with its host round trips; one warm-up call, then the median of 5), ranges decoded and candidates rejected;
  - host zlib inflating the same file on one thread as the host program's old loop did: gzread with a 1 MiB gzbuffer into a
    reused 32 MiB buffer (libz.so.1 through ctypes), median of 3;
  - `sage2gpu -M 3` wall clock and its "Parsed and uploaded" time on the plain, gzip and BGZF files, every run, alternated;
  - the BGZF inflate kernel again (sage2gpu_inflate_bgzf), to compare with the decoder before it was shared.

Usage: python tools/gzip_bench.py [--sets cfg2,cfg4] [--reps 3] [--out DIR]   (needs a GPU)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bgzf_bench  # noqa: E402
from sage2_b200 import api  # noqa: E402

BIN = bgzf_bench.BIN


def gzip_inflate(blob: bytes, text_bytes: int, reps: int = 5) -> dict:
    g = api.Sage2Gpu(0)
    try:
        g.inflate_gzip(blob, text_bytes)          # warm-up (module load, allocations)
        ms, wall = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            out, m, ranges, confirmed, rejected = g.inflate_gzip(blob, text_bytes)
            wall.append((time.perf_counter() - t0) * 1e3)
            ms.append(m)
        km, wm = statistics.median(ms), statistics.median(wall)
        return {"text_bytes": len(out), "kernel_ms": [round(x, 2) for x in ms], "call_ms": [round(x, 2) for x in wall],
                "text_gbps_kernels_median": round(len(out) / km / 1e6, 2), "text_gbps_call_median": round(len(out) / wm / 1e6, 2),
                "ranges": ranges, "confirmed": confirmed, "rejected": rejected}
    finally:
        g.close()


def host_zlib(path: str, reps: int = 3) -> dict:
    z = C.CDLL("libz.so.1")
    z.gzopen.restype = C.c_void_p
    z.gzopen.argtypes = [C.c_char_p, C.c_char_p]
    z.gzbuffer.argtypes = [C.c_void_p, C.c_uint]
    z.gzread.argtypes = [C.c_void_p, C.c_void_p, C.c_uint]
    z.gzclose.argtypes = [C.c_void_p]
    buf = C.create_string_buffer(32 << 20)
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f = z.gzopen(path.encode(), b"r")
        z.gzbuffer(f, 1 << 20)
        n = 0
        while True:
            k = z.gzread(f, buf, 32 << 20)
            if k <= 0:
                break
            n += k
        z.gzclose(f)
        t.append(time.perf_counter() - t0)
    return {"text_bytes": n, "s": [round(x, 3) for x in t], "s_median": round(statistics.median(t), 3)}


def cli_wall(files: dict, k: int, reps: int, d: str) -> dict:
    """`sage2gpu -M 3` on each file, alternated: wall clock and the "Parsed and uploaded" seconds of every run"""
    out = {kind: {"wall_s": [], "parsed_and_uploaded_s": []} for kind in files}
    for _ in range(reps):
        for kind, path in files.items():
            o = os.path.join(d, "o_" + kind)
            t0 = time.time()
            subprocess.run([BIN, "-f", path, "-k", str(k), "-o", o, "-p", "g", "-M", "3"], check=True)
            out[kind]["wall_s"].append(round(time.time() - t0, 3))
            for ln in open(os.path.join(o, "g.log")):
                if "Parsed and uploaded" in ln:
                    out[kind]["parsed_and_uploaded_s"].append(float(ln.split(" in ")[1].split()[0]))
                if "Records split" in ln:
                    out[kind]["log_step1"] = ln.strip()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", default="cfg2")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for gzip_bench.json (default: the JSON line on stdout only)")
    a = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    res = {"card": card[0] if card else "unknown", "zlib": zlib.ZLIB_RUNTIME_VERSION, "sets": {}}
    with tempfile.TemporaryDirectory() as d:
        for name in a.sets.split(","):
            f = bgzf_bench.write_files(name, d)
            bz = f.pop("blob")
            gzb = open(os.path.join(d, name + ".fastq.gz"), "rb").read()
            f["gzip_inflate_device"] = gzip_inflate(gzb, f["text_bytes"])
            f["gzip_inflate_host_zlib_1thread"] = host_zlib(os.path.join(d, name + ".fastq.gz"))
            del gzb
            files = {"plain": os.path.join(d, name + ".fastq"), "gzip": os.path.join(d, name + ".fastq.gz"),
                     "bgzf": os.path.join(d, name + ".bgzf.fastq.gz")}
            f["cli"] = cli_wall(files, f["k"], a.reps, d)
            f["bgzf_inflate"] = bgzf_bench.inflate_kernel(bz, 5)
            del bz
            res["sets"][name] = f
            for p in files.values():
                os.unlink(p)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "gzip_bench.json"), "w") as fo:
            json.dump(res, fo, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
