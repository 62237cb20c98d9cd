#!/usr/bin/env python
"""Sector loads of the superstring scan's probes (search_fast.cu stage 1), counted on the table the library built.  No timing.

    python tools/probe_rounds.py OUT_DIR [--workloads cfg4,cfg2] [--sample 100000]

For every workload: steps 1-2 on the GPU (read organisation, table build), then on the host, for a seeded sample of unique
reads, every window's walk from its home sector (tests/table_ref.py) over the slot index the GPU holds, judged as the scan
judges a sector: the first slot whose tag matches ends the walk (found), an empty slot ends it (absent), a full sector
without a match goes on to the next one.  Printed per workload: the share of full sectors, the distribution of sector
loads per window (found / absent), and the dependent load rounds per read when a warp probes its windows
  chunked: 32 windows at a time, each chunk waiting for its slowest lane (sum over chunks of the chunk's maximum);
  queued:  one warp-wide queue, a lane taking the next window as soon as its probe ends.
A masked key's confirmation (probe_window, a key with >= 100 entries) is not counted.  Writes OUT_DIR/probe_rounds_<w>.json.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

_u = np.uint64


def window_keys(B: np.ndarray, W: int, h: int):
    """(v0, v1) of windows 0..W-1 of the reads whose 2-bit bases are the rows of B: arrays [R, W]"""
    R = B.shape[0]
    v0 = np.zeros((R, W), np.uint64)
    v1 = np.zeros((R, W), np.uint64)
    n0 = max(h - 32, 0)
    for j in range(W):
        a = np.zeros(R, np.uint64)
        for t in range(n0):
            a = (a << _u(2)) | B[:, j + t]
        b = np.zeros(R, np.uint64)
        for t in range(n0, h):
            b = (b << _u(2)) | B[:, j + t]
        v0[:, j], v1[:, j] = a, b
    return v0, v1


def sector_loads(hsh: np.ndarray, sectors: np.ndarray, nsec: int, shards: int, tag_bits: int):
    """sector loads of each probe and whether it ended on a tag match"""
    import table_ref
    base = table_ref.key_owner(hsh, shards) * nsec
    sec = table_ref.home_sector(hsh, nsec).astype(np.int64)
    tag = table_ref.slot_tag(hsh, tag_bits)
    loads = np.zeros(len(hsh), np.int64)
    found = np.zeros(len(hsh), bool)
    live = np.arange(len(hsh))
    while len(live):
        s = sectors[base[live] + sec[live]]
        loads[live] += 1
        match = ((s >> _u(40)) == tag[live, None]) & (s != 0)
        hit = match.any(axis=1)
        found[live[hit]] = True
        more = ~hit & (s[:, 3] != 0)
        live, nxt = live[more], sec[live[more]] + 1
        sec[live] = np.where(nxt == nsec, 0, nxt)
    return loads, found


def rounds(L: np.ndarray, W: np.ndarray):
    """dependent load rounds per read (rows of L: sector loads of each window, windows >= W[r] unused)"""
    R, Wmax = L.shape
    chunked = np.zeros(R, np.int64)
    for c in range(0, Wmax, 32):
        chunked += L[:, c:c + 32].max(axis=1)
    # queued: every round the idle lanes take the next windows in order, then every busy lane makes one load
    rem = np.zeros((R, 32), np.int64)
    nxt = np.zeros(R, np.int64)
    queued = np.zeros(R, np.int64)
    rows = np.arange(R)[:, None]
    while True:
        idle = rem == 0
        jn = nxt[:, None] + np.cumsum(idle, axis=1) - 1
        take = idle & (jn < W[:, None])
        rem = np.where(take, L[rows, np.minimum(jn, Wmax - 1)], rem)
        nxt += idle.sum(axis=1)
        busy = rem > 0
        if not busy.any():
            break
        queued += busy.any(axis=1)
        rem -= busy
    return chunked, queued


def run_workload(name, sample, out_dir):
    import torch
    import table_ref
    from sage2_b200 import api, synth

    reads, k = synth.config_cached(name)
    bases, offsets = synth.concat(reads)
    n = len(offsets) - 1
    d_b = torch.from_numpy(np.ascontiguousarray(bases)).cuda()
    d_o = torch.from_numpy(np.ascontiguousarray(offsets)).cuda()
    del reads, bases
    gpu = api.Sage2Gpu(0)
    gpu.load_reads_ptr(d_b.data_ptr(), d_o.data_ptr(), n, k, device=True)
    gpu.build_hash_table()
    torch.cuda.synchronize()
    c = gpu.counters()
    h = c["hash_len"]
    from sage2_b200 import multi
    v = gpu.table_view()
    slots = multi.device_view_fn(torch.device("cuda", 0))(v["slots"], v["n_slots"], "<i8").cpu().numpy().view(np.uint64)
    nsec, shards = v["sectors_per_shard"], v["shards"]
    r = gpu.reads()
    gpu.close()
    del d_b, d_o
    torch.cuda.empty_cache()

    U = len(r["length"])
    rng = np.random.default_rng(12345)
    ids = np.sort(rng.choice(U, size=min(sample, U), replace=False))
    length = r["length"][ids].astype(np.int64)
    W = length - h + 1
    Wmax = int(W.max())
    pos = (r["byte_off"][ids].astype(np.int64) * 4)[:, None] + np.arange(int(length.max()))[None, :]
    pos = np.minimum(pos, 4 * len(r["fwd"]) - 1)
    B = table_ref._bases(r["fwd"], pos)
    v0, v1 = window_keys(B, Wmax, h)
    hsh = table_ref.hash_key(v0.ravel(), v1.ravel())
    valid = (np.arange(Wmax)[None, :] < W[:, None]).ravel()
    sectors = slots.reshape(-1, 4)
    loads = np.zeros(len(hsh), np.int64)
    found = np.zeros(len(hsh), bool)
    loads[valid], found[valid] = sector_loads(hsh[valid], sectors, nsec, shards, 24)
    chunked, queued = rounds(loads.reshape(len(ids), Wmax), W)

    lv, fv = loads[valid], found[valid]
    dist = {}
    for what, sel in (("found", fv), ("absent", ~fv)):
        x = lv[sel]
        dist[what] = {"windows": int(len(x)), "mean_loads": float(x.mean()) if len(x) else 0.0,
                      **{f"p_more_than_{m}": float((x > m).mean()) if len(x) else 0.0 for m in (1, 2, 3)}}
    per_read = {"windows": float(W.mean()), "sector_loads": float(lv.sum() / len(ids)),
                "rounds_chunked": float(chunked.mean()), "rounds_queued": float(queued.mean())}
    res = {"workload": name, "unique_reads": U, "sampled_reads": int(len(ids)), "hash_len": h, "sectors": int(len(sectors)),
           "shards": shards, "distinct_keys": c.get("distinct_keys"), "load": (c.get("distinct_keys") or 0) / (4 * len(sectors)),
           "full_sectors": float((sectors[:, 3] != 0).mean()), "windows_found": float(fv.mean()),
           "loads_per_window": dist, "per_read": per_read}
    print(f"== {name}: {U} unique reads, {len(ids)} sampled, h = {h}, {len(sectors)} sectors, load {res['load']:.3f}, "
          f"full sectors {res['full_sectors']:.1%}, windows that find a key {res['windows_found']:.1%}")
    for what, d in dist.items():
        print(f"   key {what:<6} {d['windows']:>9} windows, {d['mean_loads']:.3f} loads, P(> 1 / > 2 / > 3 sectors) "
              f"{d['p_more_than_1']:.1%} / {d['p_more_than_2']:.1%} / {d['p_more_than_3']:.1%}")
    print(f"   per read: {per_read['windows']:.1f} windows, {per_read['sector_loads']:.1f} sector loads, dependent rounds "
          f"chunked {per_read['rounds_chunked']:.2f}, queued {per_read['rounds_queued']:.2f}")
    with open(os.path.join(out_dir, f"probe_rounds_{name}.json"), "w") as f:
        json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out_dir")
    ap.add_argument("--workloads", default="cfg4,cfg2")
    ap.add_argument("--sample", type=int, default=100000)
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    for name in a.workloads.split(","):
        run_workload(name, a.sample, a.out_dir)


if __name__ == "__main__":
    main()
