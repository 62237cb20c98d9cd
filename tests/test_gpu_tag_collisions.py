"""GPU parity with narrow slot tags: every search path that resolves a tag collision, run on every data set.

A slot keeps 24 bits of its key's hash as a tag (csrc/core.cuh); a tag match that is not the key is a collision, and the
table build, the superstring scan, the general kernel (restart with verified probes), phase C's probes, masked keys and the
routed probes of the sharded layout each have code for it.  With 24 bits these paths almost never run on small sets, so the
library and the `sage2gpu` program are built again with SG_SLOT_TAG_BITS = 0 (every occupied slot matches every probe: only
the key compare separates keys) and 8 (a fraction of the reads meet a collision), into tests/_build/tag<N>/.  Every stage
must still give the oracle's results, and the built table must pass the reference check of tests/table_ref.py.

Each variant runs in a child process of its own (a process loads one libsage2gpu); the product build is checked against the
same reference here too."""
import functools
import hashlib
import json
import multiprocessing
import os
import re
import subprocess

import numpy as np
import pytest

import datasets
import long_datasets
import table_ref
from sage2_b200 import api

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "sage2_b200", "csrc")
WIDTHS = [0, 8]
SMALL = ["clean", "k31", "k70", "k64", "err", "rep", "hicopy", "deep", "varlen", "varlen_err", "deep_varlen",
         "tandem", "mixed", "adapter", "empty", "allbad", "single"]
LONG = list(long_datasets.LONG_DATASETS)
BUILDS = ["direct", "bucketed"]
CASE_TIMEOUT_S = 900


def _variant_dir(bits):
    return os.path.join(HERE, "_build", f"tag{bits}")


def _build_variants():
    """make of each variant in its own object directory (make rebuilds what a newer source under csrc/ invalidates)"""
    procs = []
    for bits in WIDTHS:
        d = _variant_dir(bits)
        os.makedirs(d, exist_ok=True)
        procs.append(subprocess.Popen(["make", "-C", CSRC, "-j16", f"BUILD={d}/obj", f"OUT={d}/libsage2gpu.so", f"HOSTBIN={d}/sage2gpu",
                                       f"EXTRA_NVFLAGS=-DSG_SLOT_TAG_BITS={bits}"], stdout=subprocess.DEVNULL))
    for p in procs:
        assert p.wait(timeout=1800) == 0, "variant build failed"


def _init_child(lib_path):
    api.LIB_PATH = lib_path


@pytest.fixture(scope="module")
def variants():
    _build_variants()
    ctx = multiprocessing.get_context("spawn")
    pools = {bits: ctx.Pool(1, initializer=_init_child, initargs=(os.path.join(_variant_dir(bits), "libsage2gpu.so"),))
             for bits in WIDTHS}
    try:
        yield pools
    finally:
        for p in pools.values():
            p.terminate()
            p.join()


def _in_child(pools, bits, fn, *args):
    """fn(bits, *args) in the child that loaded the variant's library; its exception (with the child's traceback) fails here"""
    res = pools[bits].apply_async(fn, (bits, *args))
    try:
        return res.get(timeout=CASE_TIMEOUT_S)
    except multiprocessing.TimeoutError:
        pools[bits].terminate()
        pytest.fail(f"{fn.__name__}{args} at {bits} tag bits did not finish in {CASE_TIMEOUT_S} s")


# ---- what the children run --------------------------------------------------------------------------------------------

@functools.lru_cache(maxsize=None)
def _ref(name):
    from oracle import oracle
    from sage2_b200 import synth
    if name in datasets.DATASETS:
        reads, k = datasets.get(name)
    else:
        reads, k = long_datasets.get(name)
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    return b, off, k, o, table_ref.Keys.from_oracle(o)


def _host(ptr, n, typestr):
    import torch
    from sage2_b200 import multi
    torch.cuda.synchronize()
    return multi.device_view_fn(torch.device("cuda", 0))(ptr, n, typestr).cpu().numpy()


def check_gpu_table(gpu, keys, bits, rank=0, world=1):
    """the table `gpu` holds against table_ref.check_table"""
    v = gpu.table_view()
    slots = _host(v["slots"], v["n_slots"], "<i8").view(np.uint64)
    entries = _host(v["entries"], v["n_entries"], "<i4").view(np.uint32)
    if keys.U == 0:
        return {"keys": 0, "passed_same_tag": 0}
    return table_ref.check_table(keys, slots, entries, v["sectors_per_shard"], v["shards"], bits, rank, world)


def _gpu(b, off, k, **options):
    g = api.Sage2Gpu(0)
    for key, value in options.items():
        g.set_option(key, value)
    g.run_steps123(b, off, k)
    return g


def _with_env(name, value):
    if value is None:
        os.environ.pop(name, None)
    else:
        os.environ[name] = value


def run_set(bits, name):
    """every stage of one set: both table builds x superstring scan on / off, min-hash order, the host walk of phase C"""
    from test_gpu_parity import _compare
    b, off, k, o, keys = _ref(name)
    st = {}
    try:
        for how in BUILDS:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            for fast in (1, 0):
                g = _gpu(b, off, k, fast_scan=fast)
                _compare(o, g)
                c = g.counters()
                st[f"{how}_fast{fast}"] = {x: c[x] for x in ("fast_path_reads", "unique_reads", "probe_restarts")}
            st[f"{how}_table"] = check_gpu_table(g, keys, bits)
        _with_env("SAGE2GPU_TABLE_BUILD", None)
        _compare(o, _gpu(b, off, k, read_order=1))
        if name in ("varlen_err", "err"):
            _with_env("SAGE2GPU_PHASE_C_HOST", "1")
            g = _gpu(b, off, k)
            assert g.counters()["phase_c_on_device"] == 0
            _compare(o, g)
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)
        _with_env("SAGE2GPU_PHASE_C_HOST", None)
    return st


def run_long(bits, name):
    from test_gpu_parity import _compare
    b, off, k, o, keys = _ref(name)
    st = {}
    try:
        for how in BUILDS:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            g = _gpu(b, off, k)
            _compare(o, g)
            st[how] = check_gpu_table(g, keys, bits)
        _compare(o, _gpu(b, off, k, fast_scan=0))
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)
    return st


def run_partitioned_phase_a(bits, name, world):
    """world contexts on one GPU with the same reads and table, each searching its slice of phase A (test_gpu_parity)"""
    from test_gpu_parity import test_partitioned_phase_a_slices_compose
    test_partitioned_phase_a_slices_compose(name, world)
    return {}


def run_partitioned_build(bits, name, world):
    """every stage partitioned over `world` contexts: the gathered table (`world` shards) checked on every rank"""
    import torch
    from sage2_b200 import multi
    b, off, k, o, keys = _ref(name)
    dev = torch.device("cuda", 0)
    tb, to = torch.from_numpy(b).to(dev), torch.from_numpy(off).to(dev)
    torch.cuda.synchronize()
    st = {}
    try:
        for how in BUILDS:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            gpus = [api.Sage2Gpu(0) for _ in range(world)]
            multi.run_local([multi.partitioned_graph_steps(g, r, world, multi.device_view_fn(dev), tb.data_ptr(), to.data_ptr(), len(off) - 1, k, True)
                             for r, g in enumerate(gpus)])
            assert sum(g.counters()["compare_calls"] for g in gpus) == o.compare_calls
            for g in gpus:
                assert g.table_view()["shards"] == world
                st[how] = check_gpu_table(g, keys, bits)
                e = g.edges()
                assert len(e) == o.n_edges
                for f in ("from", "to", "type", "delta", "delta_twin"):
                    np.testing.assert_array_equal(e[f], o.edges[f])
                np.testing.assert_array_equal(g.extensions()["explored"], o.explored_b[1:])
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)
    return st


def run_sharded(bits, name, world, p2p):
    """the sharded layout (probes routed to the shard that owns the key) over one transport; every shard checked"""
    from test_gpu_sharded import _sharded
    b, off, k, o, keys = _ref(name)
    st = {}
    try:
        for how in BUILDS:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            o, gpus = _sharded(name, world, p2p=p2p)
            assert sum(g.counters()["compare_calls"] for g in gpus) == o.compare_calls
            held = 0
            for r, g in enumerate(gpus):
                held += check_gpu_table(g, keys, bits, r, world)["keys"]
                e = g.edges()
                assert len(e) == o.n_edges
                for f in ("from", "to", "type", "delta", "delta_twin"):
                    np.testing.assert_array_equal(e[f], o.edges[f])
                np.testing.assert_array_equal(g.extensions()["explored"], o.explored_b[1:])
            assert held == keys.K
            st[how] = {"probe_restarts": sum(g.counters()["probe_restarts"] for g in gpus)}
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)
    return st


# ---- the tests --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", SMALL)
@pytest.mark.parametrize("bits", WIDTHS)
def test_small_sets_equal_oracle(variants, bits, name):
    st = _in_child(variants, bits, run_set, name)
    if name == "clean" and bits == 8:
        # the collision paths ran: the superstring scan passed reads on, the general kernel restarted reads, and tag
        # matches of other keys lay on the walks of the build
        f = st["direct_fast1"]
        assert 0 < f["fast_path_reads"] < f["unique_reads"], f
        for how in BUILDS:
            for fast in (0, 1):
                assert st[f"{how}_fast{fast}"]["probe_restarts"] > 0, (how, fast, st)
            assert st[f"{how}_table"]["passed_same_tag"] > 0, st


@pytest.mark.parametrize("name", LONG)
@pytest.mark.parametrize("bits", WIDTHS)
def test_long_reads_equal_oracle(variants, bits, name):
    """every record width from 2 to 32 words"""
    _in_child(variants, bits, run_long, name)


@pytest.mark.parametrize("name,world", [("rep", 2), ("deep_varlen", 3), ("varlen_err", 4)])
@pytest.mark.parametrize("bits", WIDTHS)
def test_partitioned_phase_a(variants, bits, name, world):
    _in_child(variants, bits, run_partitioned_phase_a, name, world)


@pytest.mark.parametrize("name", ["varlen_err", "hicopy"])
@pytest.mark.parametrize("bits", WIDTHS)
def test_partitioned_build_gathered_table(variants, bits, name):
    _in_child(variants, bits, run_partitioned_build, name, 3)


@pytest.mark.parametrize("name,world", [("rep", 2), ("hicopy", 3), ("mixed", 4)])
@pytest.mark.parametrize("p2p", [False, True])
@pytest.mark.parametrize("bits", WIDTHS)
def test_sharded_layout(variants, bits, name, world, p2p):
    st = _in_child(variants, bits, run_sharded, name, world, p2p)
    if bits == 0:     # every routed tag probe takes the first occupied slot: reads go through the verified redo pass
        for how in BUILDS:
            assert st[how]["probe_restarts"] > 0, st


def _verified_pass_ran(st):
    for how in BUILDS:
        assert st[how]["probe_restarts"] > 0, st


def test_mailbox_tag_collisions(variants):
    """The peer-memory transport at 0 tag bits (varlen_err, 2 shards): the reads whose routed tag probes met another key
    go through the verified pass, and every rank ends with the oracle's compare count, edges and explored states."""
    _verified_pass_ran(_in_child(variants, 0, run_sharded, "varlen_err", 2, True))


def test_tag_collisions_take_the_verified_pass(variants):
    """The same over the all-to-all transport."""
    _verified_pass_ran(_in_child(variants, 0, run_sharded, "varlen_err", 2, False))


def test_sharded_tag_collisions_at_the_widest_stride(variants):
    """The verified pass of the routed kernel at SW > 8 (one resident block), at both tag widths."""
    for bits in WIDTHS:
        _verified_pass_ran(_in_child(variants, bits, run_sharded, "v505", 2, False))


def test_cli_sharded_layout_takes_the_verified_pass(variants, tmp_path):
    """`sage2gpu --devices` in the sharded layout at 0 tag bits: the reads that met a collision are routed once more with
    exact keys, and the files are the reference's bytes"""
    from sage2_b200 import synth
    gold = json.load(open(os.path.join(HERE, "golden", "golden.json")))["varlen_err"]
    reads, k = datasets.get("varlen_err")
    fq = tmp_path / "in.fastq"
    synth.write_fastq(str(fq), reads)
    out = tmp_path / "out"
    env = dict(os.environ, SAGE2GPU_TABLE_LAYOUT="sharded")
    subprocess.run([os.path.join(_variant_dir(0), "sage2gpu"), "-f", str(fq), "-k", str(k), "-o", str(out), "-p", "g", "-M", "3",
                    "--devices", "0,0"], check=True, env=env, timeout=CASE_TIMEOUT_S)
    md5 = lambda p: hashlib.md5(open(p, "rb").read()).hexdigest()
    assert (md5(out / "g.reads"), md5(out / "g.graph3")) == (gold["reads_md5"], gold["graph3_md5"])
    log = open(out / "g.log").read()
    assert "Table layout: sharded" in log
    assert int(re.search(r"reads of the verified redo pass \(max over the contexts\): (\d+)", log).group(1)) > 0


# ---- the product's own table (24-bit tags) against the reference --------------------------------------------------------

@pytest.mark.parametrize("how", BUILDS)
def test_product_table_equals_reference(how, monkeypatch):
    from sage2_b200 import synth
    monkeypatch.setenv("SAGE2GPU_TABLE_BUILD", how)
    for name in SMALL:
        b, off, k, o, keys = _ref(name)
        g = api.Sage2Gpu(0)
        g.load_reads(b, off, k)
        g.build_hash_table()
        st = check_gpu_table(g, keys, 24)
        assert st["keys"] == o.distinct_keys == g.counters()["distinct_keys"]
    # cfg2 at full size (2.2 M unique reads): the keys from the reads the GPU holds, which the reference's digest pins
    from test_gpu_parity import BIG
    reads, k = synth.config_cached("cfg2")
    b, off = synth.concat(reads)
    g = api.Sage2Gpu(0)
    g.load_reads(b, off, k)
    g.build_hash_table()
    assert g.digest(edges=False)["reads"] == BIG["cfg2"]["reads_digest"]
    keys = table_ref.Keys.from_reads(g.reads(), min(k, 64))
    st = check_gpu_table(g, keys, 24)
    assert st["keys"] == g.counters()["distinct_keys"]
    assert keys.over_threshold == g.counters()["keys_over_threshold"] == BIG["cfg2"]["over_threshold"]
