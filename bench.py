#!/usr/bin/env python
"""bench.py -- reads/s through SAGE2's overlap-graph build (reference steps 1-3) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg4] [--dump-outputs DIR]

A "step" is one complete pass of the hot path over one batch of synthetic reads: ingest (filter,
canonicalise, 2-bit pack), sort + dedupe, prefix/suffix table, phase A search + extension state
machine, phase B, phase-C candidates + marking, canonical edge sort.  The default workload is BASELINE.json
config #4 (100 Mbp genome with 2 % interspersed repeats, 150 bp paired-end, 50x, -k 75: 33,333,332 input reads per
step), the largest named configuration that fits one GPU; config #2 (4.6 Mbp, 100x, -k 63) is measured next to it
at N = 1 and reported under "cfg2".  Every number carries a parity gate: the digests of the resident unique reads
and of the edge list (sage2gpu_digest) are compared on every rank with those of the UNMODIFIED reference's own
`.reads` / `.graph3` files (tests/golden/golden_big.json); a mismatch prints an error instead of a value.

  value   : whole-job input reads/s with the ASCII reads already resident in HBM.
  e2e     : the same through the C ABI with HOST (pinned) buffers: H2D of the reads and D2H of the
            edge list are inside the timed region.
  roofline: the phase-A search kernel against the measured HBM copy peak (MEASURED_PEAKS.json).
  cpu_baseline / --impl reference: the UNMODIFIED reference's steps 1-3 (oracle/_ref/ref_steps123,
            built from /root/reference in the build container) on the box's host cores, on a bounded
            sample of the workload's shape (smaller genome, same read length / coverage / repeats per Mbp / k).

N > 1 (torchrun, one rank per GPU): ONE read set for the whole job, total work fixed, so scaling is
"strong".  Two layouts (DESIGN.md section 4), the headline is the faster one at this size:
  --table replicated (default): reads and table on every GPU, phase A partitioned by read id, one NCCL exchange;
  --table sharded: every GPU holds one key-hash shard of the table, the window probes are routed to their owners
            through peer-memory mailboxes (--exchange p2p: kernel stores over NVLink) or NCCL all-to-all.
The other layout is timed on the same reads and reported as `alt_table`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the tree stays as the build left it (it may be read-only): no bytecode caches from this run
sys.dont_write_bytecode = True

METRIC = "reads/sec through exact-overlap graph build (SAGE2 steps 1-3)"
UNIT = "reads/s"

# name -> (description, genome bp, read length, coverage, k, repeat copies per Mbp of a 1 kb element)
SHAPES = {
    "cfg2": ("cfg2: synthetic 4.6 Mbp random genome, 150 bp paired-end, 100x, -k 63", 4_600_000, 150, 100, 63, 0),
    "cfg4": ("cfg4: synthetic 100 Mbp genome with 2 % interspersed repeats (2,000 copies of a 1 kb element), 150 bp "
             "paired-end, 50x, -k 75", 100_000_000, 150, 50, 75, 20),
}


def make_workload(name: str, genome_size: int | None = None):
    """(reads (N, L) uint8 ASCII, k, config dict).  Full size: exactly sage2_b200.synth.config(name) -- the read set
    the goldens in tests/golden/golden_big.json were made from.  genome_size: a sample of the same shape."""
    from sage2_b200 import synth
    if name not in SHAPES or genome_size is None:
        reads, k = synth.config(name)
        cfg = {"workload": SHAPES[name][0] if name in SHAPES else name, "name": name, "k": k}
        if name in SHAPES:
            cfg.update(genome_bp=SHAPES[name][1], read_len=SHAPES[name][2], coverage=SHAPES[name][3])
        return reads, k, cfg
    desc, _, L, cov, k, rep_per_mbp = SHAPES[name]
    G = int(genome_size)
    g = synth.random_genome(G, 4600)
    if rep_per_mbp:
        g = synth.add_repeats(g, max(2, G * rep_per_mbp // 1_000_000), 1000, 101)
    reads = synth.paired_reads(g, L, cov, seed=4601, mu=450, sigma=30)
    return reads, k, {"workload": desc, "name": name, "genome_bp": G, "read_len": L, "coverage": cov, "k": k}


def cached_workload(name: str, rank: int, world: int, barrier):
    """The full-size read set, generated once per box (rank 0) and memory-mapped by everybody (sage2_b200.synth.config_cached,
    the cache the full-size tests use too)."""
    from sage2_b200 import synth
    reads, k = synth.config_cached(name, wait=barrier)
    cfg = {"workload": SHAPES[name][0] if name in SHAPES else name, "name": name, "k": k}
    if name in SHAPES:
        cfg.update(genome_bp=SHAPES[name][1], read_len=SHAPES[name][2], coverage=SHAPES[name][3])
    return reads, k, cfg


def golden_for(name: str):
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "golden_big.json"))).get(name)
    except (OSError, ValueError):
        return None


# ---- clocks ------------------------------------------------------------------------------------

class ClockSampler:
    """SM clock and throttle reasons during the timed region, read through NVML in a background thread
    (a polling `nvidia-smi -lms` subprocess was measured to stall kernel launches for tens of ms)."""

    def __init__(self, index: int, period_s: float = 0.1):
        self.rows, self.stop_flag, self.t, self.err = [], threading.Event(), None, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.period = period_s
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception as e:      # noqa: BLE001 - any NVML problem just means "no clock record"
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                  int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception as e:  # noqa: BLE001
                self.err = repr(e)
                return
            self.stop_flag.wait(self.period)

    def stop(self) -> dict:
        if self.t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: " + str(self.err)]}
        self.stop_flag.set()
        self.t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        reasons = sorted(n for n, bit in names.items() if any(r & bit for _, r in self.rows))
        sm = [c for c, _ in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max, "reasons": reasons,
                "samples": len(sm), "source": "NVML"}


# ---- the reference on the host cores -------------------------------------------------------------

def reference_run(reads, k, tmpdir: str, threads: int | None = None) -> dict:
    """One run of the unmodified reference's steps 1-3 (oracle/_ref/ref_steps123) on `reads`."""
    from oracle import oracle
    from sage2_b200 import synth
    fq = os.path.join(tmpdir, "sample.fastq")
    synth.write_fastq(fq, reads)
    env = dict(os.environ)
    # all host cores unless told otherwise (torchrun exports OMP_NUM_THREADS=1 to its ranks)
    env["OMP_NUM_THREADS"] = str(threads or os.cpu_count() or 1)
    if os.access(oracle.REF_STEPS, os.X_OK):
        out = subprocess.run([oracle.REF_STEPS, fq, str(k)], env=env, check=True, capture_output=True, text=True).stdout
        d = json.loads(out.strip().splitlines()[-1])
        d["kind"] = "reference"
        return d
    # the reference did not travel: time the C port instead
    b, off = synth.concat(reads)
    t = time.perf_counter()
    o = oracle.OracleRun(b, off, k, threads or 0)
    dt = time.perf_counter() - t
    return {"input_reads": len(reads), "unique_reads": o.U, "edges": o.n_edges, "threads": threads or os.cpu_count(),
            "t_steps123": dt, "kind": "port"}


def sample_workload(name: str, target_seconds: float, tmpdir: str):
    """A sample of the workload's shape (same read length, coverage, k, repeats per Mbp; smaller genome) sized so
    that the reference needs about target_seconds for it."""
    name = name if name in SHAPES else "cfg2"
    _, G_full, L, cov, _, _ = SHAPES[name]
    probe_reads, k, _ = make_workload(name, genome_size=150_000)
    d = reference_run(probe_reads, k, tmpdir)
    rate = d["input_reads"] / max(d["t_steps123"], 1e-3)
    want_reads = max(100_000, int(rate * target_seconds))
    G = max(150_000, min(G_full, int(want_reads * L / cov)))
    return make_workload(name, genome_size=G)


def sample_text(cfg: dict, n_reads: int, seconds: float | None = None) -> str:
    t = f" ({seconds:.1f} s)" if seconds is not None else ""
    return (f"{cfg['name']}-shaped sample: {cfg['genome_bp']} bp genome, {n_reads} reads, same read length / coverage / "
            f"repeat density / k, steps 1-3{t} without FASTQ parse / text output")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step = max(4.0, 170.0 / max(1, args.steps + args.warmup))
    times, last = [], None
    with tempfile.TemporaryDirectory(prefix="sage2_ref_") as tmp:
        reads, k, cfg = sample_workload(args.workload, min(25.0, per_step), tmp)
        for i in range(args.warmup + args.steps):
            last = reference_run(reads, k, tmp)
            if i >= args.warmup:
                times.append(last["t_steps123"])
    ms = 1000.0 * float(np.mean(times))
    value = len(reads) / (ms / 1000.0)
    full = SHAPES.get(cfg["name"], (cfg["workload"],))[0]
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "impl": "reference",
            "config": dict(cfg, workload=full, sample_reads=len(reads), sample_genome_bp=cfg["genome_bp"]),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": last.get("threads"), "kind": last["kind"],
                             "sample": sample_text(cfg, len(reads))},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "reference_breakdown_s": {k2: v for k2, v in last.items() if k2.startswith("t_")}}
    print(json.dumps(line), flush=True)


# ---- our arm -----------------------------------------------------------------------------------

def algorithmic_bytes_phase_a(c: dict, read_len: int, n_slice: int | None = None) -> float:
    """SURVEY.md 8(d) restricted to the phase-A launch: stream the packed reads once, one 32-B sector
    per window probe, one sector-rounded packed partner read per gated comparison, 16 B of extension
    records out per read."""
    U, V, probes = (n_slice if n_slice is not None else c["unique_reads"]), c["compare_calls"], c["window_probes"]
    packed = (read_len + 3) // 4
    B = 32 * ((packed + 31) // 32)
    return float(U * packed + 32 * probes + B * V + 16 * U)


class Job:
    """One workload on this rank's GPU: device-resident and host-buffer steps, timing, parity."""

    def __init__(self, args, name, torch, dist, rank, world, local):
        from sage2_b200 import api, multi, synth
        self.args, self.name, self.torch, self.dist, self.rank, self.world, self.local = args, name, torch, dist, rank, world, local
        self.api, self.multi = api, multi
        self.dev = torch.device("cuda", local)
        reads, self.k, self.cfg = cached_workload(name, rank, world, self.barrier)
        self.n_reads = len(reads)
        self.read_len = int(reads.shape[1])
        bases, offsets = synth.concat(reads)
        self.nbytes_in = int(bases.nbytes + offsets.nbytes)
        self.h_bases = torch.empty(bases.shape[0], dtype=torch.uint8).pin_memory()
        self.h_bases.numpy()[:] = bases                      # straight from the (memory-mapped) cache into pinned memory
        self.h_off = torch.from_numpy(offsets).pin_memory()
        del reads, bases
        self.d_bases = self.h_bases.cuda(non_blocking=False)
        self.d_off = self.h_off.cuda(non_blocking=False)
        # this rank's slice of the host input (N > 1, host-buffer leg): reads [lo, hi), offsets rebased to the slice
        share = -(-self.n_reads // world)
        self.sl_lo, self.sl_hi = min(self.n_reads, rank * share), min(self.n_reads, (rank + 1) * share)
        sl = offsets[self.sl_lo:self.sl_hi + 1] - offsets[self.sl_lo]
        self.h_sl_off = torch.from_numpy(np.ascontiguousarray(sl)).pin_memory()
        self.sl_byte0 = int(offsets[self.sl_lo])
        self.sl_bytes = int(offsets[self.sl_hi] - offsets[self.sl_lo])
        self.max_len = int(np.max(np.diff(offsets))) if self.n_reads else 1
        self.gpu = api.Sage2Gpu(local)
        if args.read_order is not None:
            self.gpu.set_option("read_order", {"id": 0, "minhash": 1}[args.read_order])
        self.stream = torch.cuda.ExternalStream(self.gpu.stream_ptr(), device=self.dev)
        self.comm = {"sent": 0, "h2d": 0}
        self.xstats = {}
        self.h_edges = None
        self.per_step = []
        self.gold = golden_for(name)
        self.parity_legs = []
        # the mailbox transport needs peer access between all GPUs of the job (NVLink / NVSwitch box); otherwise NCCL
        ok = True
        if world > 1:
            try:
                ok = torch.cuda.device_count() >= world and all(torch.cuda.can_device_access_peer(local, d) for d in range(world) if d != local)
            except Exception:      # noqa: BLE001
                ok = False
            t_ok = torch.tensor([1 if ok else 0], device="cuda")
            dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
            ok = bool(t_ok.item())
        self.peers_ok = ok
        self.sharded = args.table == "sharded"

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def build_graph(self):
        """Table + graph on reads this rank has already organised (the sharded layout; one GPU)."""
        gpu, args, multi = self.gpu, self.args, self.multi
        if self.sharded:       # key-hash shard per GPU, window probes routed to their owners
            gpu.build_hash_table_shard(self.rank, self.world)
            p2p = args.exchange == "p2p" and self.peers_ok      # peer-memory mailboxes (NVLink P2P stores) or NCCL all-to-all
            return multi.build_overlap_graph_sharded(gpu, self.rank, self.world, self.dev,
                                                     batch_reads=min(args.batch_reads, 1 << 19) if p2p else args.batch_reads,
                                                     stats=self.xstats, p2p=p2p)
        gpu.build_hash_table()
        return multi.build_overlap_graph(gpu, self.rank, self.world, self.dev)

    def steps123(self, bases_ptr, off_ptr, on_device):
        """Steps 1-3 on input every rank can see.  Replicated table over several GPUs: every stage partitioned (key range of
        the reads, key-hash shard of the table, id slice of the search), results all-gathered (multi.partitioned_graph_steps)."""
        if self.world > 1 and not self.sharded and not self.args.replicate_stages:
            return self.multi.build_partitioned(self.gpu, self.rank, self.world, self.dev, bases_ptr, off_ptr, self.n_reads, self.k, on_device,
                                                stats=self.xstats)
        self.gpu.load_reads_ptr(bases_ptr, off_ptr, self.n_reads, self.k, device=on_device)
        return self.build_graph()

    def step_device(self):
        self.comm["sent"] = self.steps123(self.d_bases.data_ptr(), self.d_off.data_ptr(), True)

    def step_host(self):
        # the call a user of the C ABI makes: host buffers in, edge list back in host memory
        torch, gpu = self.torch, self.gpu
        if self.world == 1:
            self.steps123(self.h_bases.data_ptr(), self.h_off.data_ptr(), False)
            self.comm["h2d"] = self.nbytes_in
        elif not self.sharded and not self.args.replicate_stages:
            # each rank moves and packs 1/N of the input; the PACKED records are all-gathered over NVLink (4 x fewer bytes than
            # the characters), every later stage is partitioned (multi.partitioned_slice_steps)
            self.multi.build_partitioned_slices(gpu, self.rank, self.world, self.dev, self.h_bases.data_ptr() + self.sl_byte0,
                                                self.h_sl_off.data_ptr(), self.sl_hi - self.sl_lo, self.k, False, self.max_len, stats=self.xstats)
            self.comm["h2d"] = self.sl_bytes + 8 * (self.sl_hi - self.sl_lo + 1)
        else:       # each rank moves 1/N of the input over PCIe, NVLink all-gather of the characters completes it
            # (on torch's own stream: pinned tensors must not be tied to the library's stream, which dies first)
            tb, to, self.comm["h2d"] = self.multi.upload_partitioned(self.h_bases, self.h_off, self.rank, self.world, self.dev)
            torch.cuda.current_stream(self.dev).synchronize()
            self.steps123(tb.data_ptr(), to.data_ptr(), True)
        if self.h_edges is None:
            self.h_edges = torch.empty(2 * max(1, gpu.counters()["n_edges"]), dtype=torch.int64).pin_memory()
        gpu.edges_packed_into(self.h_edges.data_ptr(), self.h_edges.numel() // 2)

    def check_parity(self, leg: str):
        """Digests of this rank's resident result against the unmodified reference's files; every rank, every leg."""
        d = self.gpu.digest()
        c = self.gpu.counters()
        g = self.gold
        if g is None:
            ok = None
        else:
            ok = (d["edges"] == g["edges_digest"] and d["reads"] == g["reads_digest"] and c["n_edges"] == g["n_edges"]
                  and c["unique_reads"] == g["unique_reads"])
        all_ok = ok
        if self.world > 1 and ok is not None:
            t = self.torch.tensor([1 if ok else 0], device="cuda")
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
            all_ok = bool(t.item())
        self.parity_legs.append({"leg": leg, "table": "sharded" if self.sharded else "replicated", "ok": all_ok,
                                 "edges_digest": f"{d['edges']:016x}", "reads_digest": f"{d['reads']:016x}",
                                 "n_edges": c["n_edges"], "unique_reads": c["unique_reads"]})
        return all_ok

    def parity(self) -> dict:
        g = self.gold
        oks = [x["ok"] for x in self.parity_legs]
        out = {"ok": (all(oks) if oks and all(o is not None for o in oks) else None), "ranks_checked": self.world,
               "legs": self.parity_legs}
        if g is None:
            out["reason"] = f"no golden for workload {self.name} in tests/golden/golden_big.json"
        else:
            out["golden"] = {"source": "unmodified reference `SAGE2 -s -M 3` (tests/golden/make_golden_big.py)",
                             "edges_digest": f"{g['edges_digest']:016x}", "reads_digest": f"{g['reads_digest']:016x}",
                             "graph3_md5": g["graph3_md5"], "reads_md5": g["reads_md5"], "n_edges": g["n_edges"]}
        return out

    def timed(self, fn, steps):
        torch, gpu, api = self.torch, self.gpu, self.api
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        l0 = api.kernel_launches()
        t0 = time.perf_counter()
        ev0.record(self.stream)
        stage = {}
        marks = [ev0]
        for _ in range(steps):
            fn()
            for kk, vv in gpu.timers().items():
                stage[kk] = stage.get(kk, 0.0) + vv
            marks.append(torch.cuda.Event(enable_timing=True))
            marks[-1].record(self.stream)
        ev1.record(self.stream)
        self.barrier()
        wall_ms = (time.perf_counter() - t0) * 1000.0
        dev_ms = ev0.elapsed_time(ev1)
        self.per_step.append([round(a.elapsed_time(b), 3) for a, b in zip(marks[:-1], marks[1:])])
        t = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), api.kernel_launches() - l0, {a: b / steps for a, b in stage.items()}

    def dump_outputs(self, out_dir: str, max_rows: int = 1 << 19, seed: int = 0):
        """What the last step left on this GPU, as float64 .npy files (38 MB at most; row samples are seeded, so two runs
        of the same workload pick the same rows):
          edges.npy     sampled rows of the edge list, in order: [row, from, to, type, delta, delta_twin]
          reads.npy     sampled unique reads, in id order: [id, length, frequency]
          counters.npy  good_reads, unique_reads, n_edges, contained_ext, contained_size, left_to_explore,
                        edges_inserted_c, transitive_removed
          digests.npy   digests of the whole edge list and of all reads (tests/digest.py), each as [high 32 bits, low 32 bits]"""
        def sample(n):
            if n <= max_rows:
                return np.arange(n)
            return np.sort(np.random.default_rng(seed).choice(n, size=max_rows, replace=False))

        def save(name, *cols):      # one column: a vector; several: a table with one row per sampled item
            a = np.stack([np.asarray(c, np.float64) for c in cols], axis=1) if len(cols) > 1 else cols[0]
            np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))

        os.makedirs(out_dir, exist_ok=True)
        gpu = self.gpu
        e = gpu.edges()
        rows = sample(len(e))
        e = e[rows]
        save("edges", rows, e["from"], e["to"], e["type"], e["delta"], e["delta_twin"])
        r = gpu.reads()
        rows = sample(len(r["length"]))
        save("reads", rows + 1, r["length"][rows], r["frequency"][rows])
        c = gpu.counters()
        save("counters", [c[n] for n in ("good_reads", "unique_reads", "n_edges", "contained_ext", "contained_size",
                                         "left_to_explore", "edges_inserted_c", "transitive_removed")])
        d = gpu.digest()
        save("digests", [d["edges"] >> 32, d["edges"] & 0xFFFFFFFF, d["reads"] >> 32, d["reads"] & 0xFFFFFFFF])

    def measure(self, steps: int, warmup: int, with_alt: bool, sample_clocks: bool, dump_dir: str | None = None) -> dict:
        args, gpu, world = self.args, self.gpu, self.world
        for _ in range(max(3, warmup)):
            self.step_device()
        self.xstats.clear()
        sampler = ClockSampler(self.local) if sample_clocks and self.rank == 0 and not os.environ.get("SAGE2_BENCH_NO_SAMPLER") else None
        dev_ms, wall_ms, launches, stage = self.timed(self.step_device, steps)
        counters = gpu.counters()
        clocks = sampler.stop() if sampler else None
        xwall = {kk: (vv / steps) for kk, vv in self.xstats.items()} if self.xstats else None
        self.check_parity("device_resident")
        if dump_dir and self.rank == 0:
            self.dump_outputs(dump_dir)
        self.step_host()
        e2e_dev_ms, e2e_wall_ms, _, _ = self.timed(self.step_host, steps)
        self.check_parity("e2e")
        n_edges = gpu.counters()["n_edges"]
        main_sent = self.comm["sent"]

        # N > 1: the other table layout on the same reads, device-resident, reported next to the headline (DESIGN.md section 4)
        alt = None
        if world > 1 and with_alt:
            self.sharded = not self.sharded
            try:
                self.xstats.clear()
                for _ in range(3):
                    self.step_device()
                self.xstats.clear()
                a_ms, _, a_launches, a_stage = self.timed(self.step_device, steps)
                self.check_parity("alt_table")
                alt = {"table": "sharded" if self.sharded else "replicated",
                       "exchange": (args.exchange if self.peers_ok else "nccl") if self.sharded else "nccl",
                       "ms_per_step": a_ms / steps,
                       "value": self.n_reads / (a_ms / steps / 1000.0), "unit": UNIT, "sent_bytes_per_rank_and_step": self.comm["sent"],
                       "gpu_launches": a_launches, "stage_ms": a_stage,
                       "exchange_wall_ms_per_step": {kk: (vv / steps) for kk, vv in self.xstats.items()}}
            except Exception as ex:      # noqa: BLE001 - the headline above stands; the failure is reported, not hidden
                alt = {"table": "sharded" if self.sharded else "replicated", "error": repr(ex)[:300]}
            self.sharded = not self.sharded
            self.comm["sent"] = main_sent
        return dict(dev_ms=dev_ms, wall_ms=wall_ms, launches=launches, stage=stage, counters=counters, clocks=clocks,
                    e2e_dev_ms=e2e_dev_ms, n_edges=n_edges, alt=alt, steps=steps, xwall=xwall)

    def roofline(self, m: dict, with_gather: bool) -> dict:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        counters, stage = m["counters"], m["stage"]
        n_slice = min(counters["unique_reads"], -(-counters["unique_reads"] // self.world))      # rank 0's share of the reads
        abytes = algorithmic_bytes_phase_a(counters, self.read_len or counters["avg_len"], n_slice)
        traffic = None
        try:        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu --set full capture
            prof = json.load(open(os.path.join(ROOT, "profiles", "phase_a_traffic.json")))
            prof = prof.get(self.name, prof if prof.get("workload") == self.name else None)
            if self.world == 1 and prof:
                traffic = float(prof["dram_bytes_per_launch"])
        except (OSError, ValueError, KeyError, AttributeError):
            pass
        gather = None
        if with_gather:
            # the random-access ceiling of this GPU, measured now (DESIGN.md section 3): uniformly random 64-byte blocks
            # fetched by lane pairs / 32-byte sectors by single lanes over 8 GiB
            gather = {"gbs_64B_blocks": self.gpu.measure_gather(8 << 30, 64, 1 << 27, 2),
                      "gbs_32B_sectors": self.gpu.measure_gather(8 << 30, 32, 1 << 27, 1), "footprint_gib": 8}
        ka_ms = stage["phase_a_kernel"]
        achieved = abytes / (ka_ms / 1000.0) / 1e9
        return {"bound": "hbm", "kernel": "phase_a_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)",
                "algorithmic_bytes_per_launch": abytes, "kernel_ms": ka_ms,
                "kernel_share_of_step": ka_ms / (m["dev_ms"] / m["steps"]), "random_gather_peak": gather}

    def close(self):
        self.torch.cuda.synchronize()
        self.gpu.close()
        self.h_bases = self.h_off = self.d_bases = self.d_off = self.h_edges = None


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # N > 1: ONE read set for the whole job (same bytes on every rank); phase A is partitioned by read id and followed
    # by one NCCL exchange (sage2_b200/multi.py); reads and table are replicated (SURVEY.md 8(e), DESIGN.md section 4)
    job = Job(args, args.workload, torch, dist, rank, world, local)
    m = job.measure(args.steps, args.warmup, with_alt=not args.no_alt_table, sample_clocks=True, dump_dir=args.dump_outputs)
    parity = job.parity()
    roofline = job.roofline(m, with_gather=not args.no_gather) if rank == 0 else None
    n_reads, cfg, comm, sharded, per_step = job.n_reads, job.cfg, dict(job.comm), job.sharded, job.per_step
    nbytes_in = job.nbytes_in
    job.close()

    # N = 1: BASELINE config #2 next to the headline workload
    extra = None
    if world == 1 and args.workload != "cfg2" and not args.no_cfg2:
        j2 = Job(args, "cfg2", torch, dist, rank, world, local)
        m2 = j2.measure(args.steps, 3, with_alt=False, sample_clocks=False)
        r2 = j2.roofline(m2, with_gather=False)
        ms2 = m2["dev_ms"] / m2["steps"]
        extra = {"workload": j2.cfg["workload"], "reads_per_step": j2.n_reads, "ms_per_step": ms2, "value": j2.n_reads / (ms2 / 1000.0),
                 "unit": UNIT, "e2e": {"value": j2.n_reads / (m2["e2e_dev_ms"] / m2["steps"] / 1000.0), "unit": UNIT,
                                       "ms_per_step": m2["e2e_dev_ms"] / m2["steps"], "h2d_bytes_per_step": j2.nbytes_in,
                                       "d2h_bytes_per_step": int(16 * m2["n_edges"])},
                 "roofline": r2, "stage_ms": m2["stage"], "gpu_launches": m2["launches"], "parity": j2.parity()}
        j2.close()

    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    if parity["ok"] is False or (extra and extra["parity"]["ok"] is False):
        print(json.dumps({"metric": METRIC, "error": "PARITY FAILED: the result differs from the unmodified reference's; no value reported",
                          "n_gpus": world, "parity": parity, "cfg2_parity": extra["parity"] if extra else None}), flush=True)
        sys.exit(1)

    steps = m["steps"]
    ms_per_step = m["dev_ms"] / steps
    value = n_reads / (ms_per_step / 1000.0)             # one job: every rank worked on the same n_reads
    e2e_value = n_reads / (m["e2e_dev_ms"] / steps / 1000.0)
    counters, stage = m["counters"], m["stage"]

    # reference's CPU path on a bounded sample of the same workload (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        with tempfile.TemporaryDirectory(prefix="sage2_cpu_") as tmp:
            s_reads, s_k, s_cfg = sample_workload(args.workload, 15.0, tmp)
            d = reference_run(s_reads, s_k, tmp)
        cpu = {"value": d["input_reads"] / d["t_steps123"], "unit": UNIT, "cores": d.get("threads"), "kind": d["kind"],
               "sample": sample_text(s_cfg, len(s_reads), d["t_steps123"]),
               "breakdown_s": {k2: v for k2, v in d.items() if k2.startswith("t_")}}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": dict(cfg, parallelism=(
                           (f"{world} GPU(s): reads replicated, table sharded by key hash, window probes routed to their owners "
                            f"({'kernel stores into peer-memory mailboxes over NVLink' if args.exchange == 'p2p' else 'NCCL all-to-all'}), "
                            f"phase A partitioned by read id ({comm['sent']} B sent per rank and step)") if sharded else
                           "single GPU" if world == 1 else
                           (f"{world} GPUs: every stage partitioned (reads organised by key range, table built by key-hash shard, phase A "
                            f"by read id), reads / table / phase-A arrays all-gathered over NVLink ({comm['sent']} B contributed per rank)")
                           if not args.replicate_stages else
                           f"{world} GPUs: reads + table replicated, phase A partitioned by read id, "
                           f"one NCCL exchange (all-gather + all-reduce MAX, {comm['sent']} B sent per rank)"),
                       table=args.table, read_order=args.read_order or "default",
                       reads_per_step=n_reads, l2_policy=f"inputs ({nbytes_in >> 20} MB ASCII + working set) larger than the 126 MB L2",
                       timing="CUDA events on the library stream around all steps, max over ranks"),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(comm["h2d"]) * world,
                "d2h_bytes_per_step": int(16 * m["n_edges"]), "ms_per_step": m["e2e_dev_ms"] / steps},
        "gpu_launches": m["launches"],
        "clocks": m["clocks"],
        "parity": parity,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "edges_per_sec": counters["n_edges"] / (ms_per_step / 1000.0),
        "wall_ms_per_step": m["wall_ms"] / steps,
        "stage_ms": stage,
        "alt_table": m["alt"],
        "exchange_wall_ms_per_step": m.get("xwall"),
        "cfg2": extra,
        "per_step_ms": {"device_resident": per_step[0], "e2e": per_step[1]},
        "counters": {kk: counters[kk] for kk in ("good_reads", "unique_reads", "distinct_keys", "keys_over_threshold", "compare_calls",
                                                  "window_probes", "n_edges", "left_to_explore", "record_words", "slow_path_reads",
                                                  "phase_c_on_device")},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", help="cfg4 (default), cfg2, cfg3-40/60/90, cfg1, cfg4mini")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg2", action="store_true", help="N = 1: do not also measure BASELINE config #2")
    ap.add_argument("--table", default="replicated", choices=["replicated", "sharded"],
                    help="N > 1: every GPU holds the whole table, or one key-hash shard of it with routed probes (SURVEY 8(e))")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="--table sharded: routed probes through peer-memory mailboxes (kernel stores over NVLink) or NCCL all-to-all")
    ap.add_argument("--replicate-stages", action="store_true",
                    help="N > 1, replicated table: every rank organises all reads and builds the whole table (the round-1 layout)")
    ap.add_argument("--no-alt-table", action="store_true", help="N > 1: do not also time the other table layout")
    ap.add_argument("--batch-reads", type=int, default=1 << 20, help="reads per routed batch (--table sharded)")
    ap.add_argument("--no-gather", action="store_true", help="skip the random-gather ceiling microbenchmark")
    ap.add_argument("--read-order", default=None, choices=["id", "minhash"], help="phase-A schedule (default: the library's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload computed to DIR/*.npy (Job.dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
