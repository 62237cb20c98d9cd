"""GPU parity on reads longer than 152 bases (and of 56): every record stride the kernels are instantiated for.

The longest read of a set decides the record width SW (2 to 32 words) and the storage stride of the unique reads (4, 8, 16
or 32 words).  Packing, the unique write, phase A (general kernel and superstring scan), the sharded routing, phase C, the
`.reads` writer and the step-6 mapping all have code that depends on it.  The sets of tests/long_datasets.py cover each
width; test_long_reads_emul.py pins the CPU emulation of core.cuh to the oracle on the same sets, so a difference here is in
the CUDA code."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import datasets
import digest
import long_datasets
from long_datasets import SW
from oracle import oracle
from sage2_b200 import api, multi, synth
from test_gpu_parity import _compare, _check_edges_are_exact_overlaps, _decode
from test_gpu_sharded import _sharded
from test_long_reads_emul import record_words

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
NAMES = list(long_datasets.LONG_DATASETS)
EDGE_FIELDS = ("from", "to", "type", "delta", "delta_twin")


@functools.lru_cache(maxsize=None)
def _ref(name):
    reads, k = long_datasets.get(name)
    reads = synth.to_list(reads)
    b, off = synth.concat(reads)
    return reads, k, b, off, oracle.OracleRun(b, off, k)


def _run(name, **options):
    _, k, b, off, _ = _ref(name)
    gpu = api.Sage2Gpu(0)
    for key, value in options.items():
        gpu.set_option(key, value)
    gpu.run_steps123(b, off, k)
    return gpu


def _same_edges(gpu, o):
    e = gpu.edges()
    assert len(e) == o.n_edges
    for f in EDGE_FIELDS:
        np.testing.assert_array_equal(e[f], o.edges[f])


def _same_reads(gpu, o):
    r = gpu.reads()
    np.testing.assert_array_equal(r["length"], o.length[1:])
    np.testing.assert_array_equal(r["frequency"], o.frequency[1:])
    np.testing.assert_array_equal(r["fwd"], o.fwd)
    np.testing.assert_array_equal(r["rc"], o.rc)


def _reads_digest(gpu):
    """tests/digest.py over the unique reads as the C ABI returns them."""
    r = gpu.reads()
    U = len(r["length"])
    rows = [bytes(np.frombuffer(b"ACGT", np.uint8)[_decode(r["fwd"][int(r["byte_off"][i]):int(r["byte_off"][i + 1])], int(r["length"][i]))])
            for i in range(U)]
    return digest.finish(digest.reads_digest_ragged(np.arange(1, U + 1), r["frequency"], r["length"], rows), U)


# ---- a. every stage, the files, the digests -------------------------------------------------------------------------

@pytest.mark.parametrize("name", NAMES)
def test_every_stage_equals_oracle(name, tmp_path):
    _, k, _, _, o = _ref(name)
    gpu = _run(name)
    c = gpu.counters()
    assert c["record_words"] == SW[name]
    _compare(o, gpu)
    gpu.write_reads(str(tmp_path / "g.reads"))
    gpu.write_graph3(str(tmp_path / "g.graph3"))
    o.write_reads(str(tmp_path / "o.reads"))
    o.write_graph3(str(tmp_path / "o.graph3"))
    for ext in ("reads", "graph3"):
        assert (tmp_path / f"g.{ext}").read_bytes() == (tmp_path / f"o.{ext}").read_bytes(), ext
    d = gpu.digest()
    assert d["edges"] == digest.edges_digest_total(gpu.edges())
    assert d["reads"] == _reads_digest(gpu)
    assert _check_edges_are_exact_overlaps(gpu, k, sample=1000) > 0


# ---- b. phase A: with and without the superstring scan, in min-hash order, both table builds --------------------------

@pytest.mark.parametrize("name", NAMES)
def test_phase_a_variants_equal_oracle(name, monkeypatch):
    reads, k, _, _, o = _ref(name)
    gpu = _run(name)
    fast = gpu.counters()["fast_path_reads"]
    # the superstring scan is instantiated up to 8 words and takes reads of at most 128 windows of h = min(k, 64) bases
    # (search_fast.cu kFastWindows): it certifies most such reads of these sets; above 8 words the general kernel takes all
    scan_reads = sum(1 for r in reads if len(r) - min(k, 64) + 1 <= 128) if SW[name] <= 8 else 0
    if scan_reads:
        assert fast > 0, fast
    else:
        assert fast == 0, fast
    gpu = _run(name, fast_scan=0)
    assert gpu.counters()["fast_path_reads"] == 0
    _compare(o, gpu)
    _compare(o, _run(name, read_order=1))
    for how in ("direct", "bucketed"):
        monkeypatch.setenv("SAGE2GPU_TABLE_BUILD", how)
        _compare(o, _run(name))


# ---- c. phase C on the device and through the host walk ---------------------------------------------------------------

def test_phase_c_device_and_host_walk_agree(monkeypatch):
    """Fixed-length sets have a symmetric candidate set: phase C runs wholly on the device (phase_c_on_device == 1) at every
    storage stride from 8 to 32 words; forcing the host walk must give the same edges, the oracle's."""
    on_device = {}
    for name in ("f153", "f248", "f504", "f1016"):
        o = _ref(name)[4]
        monkeypatch.delenv("SAGE2GPU_PHASE_C_HOST", raising=False)
        gpu = _run(name)
        c = gpu.counters()
        assert (c["edges_inserted_c"], c["transitive_removed"]) == (o.edges_inserted_c, o.transitive_removed)
        on_device[name] = c["phase_c_on_device"]
        e1 = gpu.edges().copy()
        _same_edges(gpu, o)
        monkeypatch.setenv("SAGE2GPU_PHASE_C_HOST", "1")
        gpu = _run(name)
        c = gpu.counters()
        assert c["phase_c_on_device"] == 0
        assert (c["edges_inserted_c"], c["transitive_removed"]) == (o.edges_inserted_c, o.transitive_removed)
        np.testing.assert_array_equal(e1, gpu.edges())
    assert on_device == {"f153": 1, "f248": 1, "f504": 1, "f1016": 1}, on_device


# ---- d. the partitioned build -----------------------------------------------------------------------------------------

def _check_ranks(gpus, o):
    assert sum(g.counters()["compare_calls"] for g in gpus) == o.compare_calls
    for g in gpus:
        c = g.counters()
        assert c["unique_reads"] == o.U and c["distinct_keys"] == o.distinct_keys and c["keys_over_threshold"] == o.keys_over_threshold
        _same_reads(g, o)
        _same_edges(g, o)
        np.testing.assert_array_equal(g.extensions()["explored"], o.explored_b[1:])


@pytest.mark.parametrize("name", ["v377", "short_in_wide"])
def test_partitioned_build_equals_oracle(name):
    _, k, b, off, o = _ref(name)
    dev = torch.device("cuda", 0)
    tb, to = torch.from_numpy(b).to(dev), torch.from_numpy(off).to(dev)
    torch.cuda.synchronize()
    world = 3
    gpus = [api.Sage2Gpu(0) for _ in range(world)]
    multi.run_local([multi.partitioned_graph_steps(g, r, world, multi.device_view_fn(dev), tb.data_ptr(), to.data_ptr(), len(off) - 1, k, True)
                     for r, g in enumerate(gpus)])
    for g in gpus:
        assert g.counters()["record_words"] == SW[name]
    _check_ranks(gpus, o)


@pytest.mark.parametrize("name", ["v377", "short_in_wide"])
def test_partitioned_slices_pack_at_the_stride_of_the_whole_set(name):
    """Host-cut slices, only the middle one holding the reads that need the widest record: the other slices would pack at a
    narrower stride on their own, but every slice must pack at the stride of the longest read of all of them."""
    reads, k, _, _, _ = _ref(name)
    longest = max(len(r) for r in reads)
    top = [r for r in reads if record_words(len(r)) == SW[name]]
    rest = [r for r in reads if record_words(len(r)) < SW[name]]
    third = len(rest) // 3
    slices = [rest[:third], rest[third:2 * third] + top, rest[2 * third:]]
    assert record_words(max(len(r) for r in slices[0])) < SW[name] and record_words(max(len(r) for r in slices[2])) < SW[name]
    b, off = synth.concat([r for s in slices for r in s])
    o = oracle.OracleRun(b, off, k)
    world = len(slices)
    host = [synth.concat(s) for s in slices]
    view = multi.device_view_fn(torch.device("cuda", 0))
    gpus = [api.Sage2Gpu(0) for _ in range(world)]
    multi.run_local([multi.partitioned_slice_steps(g, r, world, view, host[r][0].ctypes.data, host[r][1].ctypes.data, len(slices[r]), k, False, longest)
                     for r, g in enumerate(gpus)])
    for g in gpus:
        assert g.counters()["record_words"] == SW[name]
    _check_ranks(gpus, o)
    # a maximum below the slice's longest read is refused, not packed into too narrow a record
    hb, ho = host[1]
    with pytest.raises(api.Sage2GpuError, match="longer than the maximum"):
        api.Sage2Gpu(0).pack_slice(hb.ctypes.data, ho.ctypes.data, len(slices[1]), k, False, longest - 1)


# ---- e. the sharded table ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,world", [("hicopy250", 2), ("v505", 3)])
@pytest.mark.parametrize("p2p", [False, True])
def test_sharded_table_equals_oracle(name, world, p2p):
    o, gpus = _sharded(name, world, p2p=p2p)
    assert all(g.counters()["record_words"] == SW[name] for g in gpus)
    assert sum(g.counters()["compare_calls"] for g in gpus) == o.compare_calls
    for g in gpus:
        _same_edges(g, o)
        np.testing.assert_array_equal(g.extensions()["explored"], o.explored_b[1:])


# ---- f. the streamed upload -------------------------------------------------------------------------------------------

def test_streamed_upload_equals_one_shot():
    reads, k, b, off, o = _ref("short_in_wide")
    first_long = next(i for i, r in enumerate(reads) if len(r) > 100)
    chunk = max(1, first_long // 2)           # the first chunks hold 100-base reads only
    assert max(len(r) for r in reads[:chunk]) <= 100
    gpu = api.Sage2Gpu(0)
    gpu.load_reads_chunked(b, off, k, reads_per_chunk=chunk)
    gpu.build_hash_table()
    gpu.build_overlap_graph()
    assert gpu.counters()["record_words"] == 32
    _compare(o, gpu)
    np.testing.assert_array_equal(gpu.edges(), _run("short_in_wide").edges())


# ---- g. step-6 mapping ------------------------------------------------------------------------------------------------

_COMP = {65: 84, 67: 71, 71: 67, 84: 65, 97: 116, 99: 103, 103: 99, 116: 97, 78: 78}


def _long_queries(reads, seed):
    """Queries around the widest lengths: the longest reads as they are, reverse-complemented, lower-cased, with one
    substitution or an N, cut by one base, and extended past the record stride and past 1016 bases."""
    rng = np.random.default_rng(seed)
    longest = max(len(r) for r in reads)
    top = [r for r in reads if len(r) >= longest - 8]
    out = []
    for r in top[:40]:
        p = int(rng.integers(0, len(r)))
        sub = r[:p] + bytes([b"ACGT"[(b"ACGT".find(r[p:p + 1]) + 1) % 4]]) + r[p + 1:]
        out += [r, bytes(_COMP[c] for c in reversed(r)), r.lower(), sub, r[:p] + b"N" + r[p + 1:], r[:-1], r[1:]]
        for n in (longest + 1, 1016, 1017, 1300):
            ext = (r * (n // len(r) + 1))[:n]
            out += [ext, bytes(_COMP[c] for c in reversed(ext))]
    return out


@pytest.mark.parametrize("name", ["f56", "f248", "v377", "short_in_wide"])
def test_map_reads_equals_oracle(name):
    reads, k, b, off, o = _ref(name)
    queries = datasets.map_queries_of(reads, n=3000, seed=41) + _long_queries(reads, 42)
    qlen = np.array([len(q) for q in queries])
    assert (qlen > 32 * SW[name] - 8).any() and (qlen > 1016).any()
    qb, qoff = synth.concat(queries)
    want_ids, want_good = o.map_reads(qb, qoff, k)
    assert (want_ids > 0).sum() > 500 and (want_ids < 0).sum() > 500
    gpu = api.Sage2Gpu(0)
    gpu.load_reads(b, off, k)
    assert gpu.counters()["record_words"] == SW[name]
    ids, good, _ = gpu.map_reads(qb, qoff)
    np.testing.assert_array_equal(good, want_good)
    np.testing.assert_array_equal(ids, want_ids)


# ---- h. the length limit ----------------------------------------------------------------------------------------------

def test_reads_up_to_1016_bases_and_no_longer():
    reads, k, _, _, _ = _ref("f1016")
    assert max(len(r) for r in reads) == 1016          # loads, and is checked in full by the tests above
    gpu = api.Sage2Gpu(0)
    too_long = reads[:50] + [reads[50] + b"A"] + reads[51:100]
    b, off = synth.concat(too_long)
    with pytest.raises(api.Sage2GpuError, match="longer than 1016 bases"):
        gpu.load_reads(b, off, k)
    _, k, b, off, o = _ref("f153")       # the context still works
    gpu.run_steps123(b, off, k)
    _compare(o, gpu)


# ---- i. the warp-per-read pack at SW <= 8 -----------------------------------------------------------------------------

_PACK_WARP = r"""
import sys
sys.path[:0] = [{root!r}, {here!r}]
import numpy as np
import torch
from torch.profiler import profile, ProfilerActivity
import long_datasets
from oracle import oracle
from sage2_b200 import api, synth
for name in ("f56", "f248"):
    reads, k = long_datasets.get(name)
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    gpu = api.Sage2Gpu(0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gpu.load_reads(b, off, k)
        torch.cuda.synchronize()
    names = {{e.name for e in prof.events()}}
    assert any("pack_kernel" in n for n in names) and not any("pack_thread_kernel" in n for n in names), sorted(names)
    c = gpu.counters()
    assert c["record_words"] == long_datasets.SW[name] and c["unique_reads"] == o.U
    r = gpu.reads()
    np.testing.assert_array_equal(r["length"], o.length[1:])
    np.testing.assert_array_equal(r["frequency"], o.frequency[1:])
    np.testing.assert_array_equal(r["fwd"], o.fwd)
    np.testing.assert_array_equal(r["rc"], o.rc)
    print(name, "ok")
"""


def test_warp_per_read_pack_at_narrow_strides():
    """SAGE2GPU_PACK_WARP is read once per process: a child process packs f56 (SW 2) and f248 (SW 8) with the warp-per-read
    kernel, which otherwise only runs above 8 words."""
    root = os.path.dirname(HERE)
    env = dict(os.environ, SAGE2GPU_PACK_WARP="1")
    out = subprocess.run([sys.executable, "-c", _PACK_WARP.format(root=root, here=HERE)], env=env, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "f56 ok" in out.stdout and "f248 ok" in out.stdout
