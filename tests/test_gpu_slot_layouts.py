"""GPU parity on the read sets of tests/slot_layouts.py: probe walks that wrap past the end of the slot index or of a
shard, long runs of full sectors, and a chain across the seam of two bucket slot ranges of the bucketed build.

Every walk of the pipeline meets these chains: the direct build (table_insert_kernel), the bucketed build's claim and retry
rounds, the superstring scan's warp-wide probe queue (phase_a_fast_kernel), the general kernel's probe_window, and the
routed probes of the sharded layout (answer_one).  Every configuration must give the oracle's results, and every table built
must pass the reference check (table_ref.check_table) at the planned geometry and show the planned chains: the same
occupied slots as the reference build and as many wrapped keys per shard (both independent of the order the keys were
inserted in), and the set's premise (slot_layouts.check_premise)."""
import functools
import os
import subprocess

import numpy as np
import pytest
import torch

import slot_layouts as sl
import table_ref
from oracle import oracle
from sage2_b200 import api, multi, synth
from test_gpu_parity import _compare
from test_gpu_tag_collisions import WIDTHS, _in_child, variants  # noqa: F401  (variants: the fixture of the tag variants)

pytestmark = pytest.mark.gpu

SETS = sl.set_names()
SHARD_SETS = [s for s in SETS if s.startswith("shard_ends")]
BUILDS = ["direct", "bucketed"]


@functools.lru_cache(maxsize=None)
def _ref(set_name):
    p = sl.get(*sl.parse(set_name))
    b, off = synth.concat(p.reads)
    o = oracle.OracleRun(b, off, p.k)
    keys, lay = sl.reference(p, o)
    return p, b, off, o, keys, lay


def _host(ptr, n, typestr):
    torch.cuda.synchronize()
    return multi.device_view_fn(torch.device("cuda", 0))(ptr, n, typestr).cpu().numpy()


def check_layout(g, set_name, bits=24, rank=0, world=1):
    """The table `g` holds: a table of the set's keys (table_ref.check_table with `bits` tag bits), at the geometry planned
    for it, and -- where that geometry is the plan's own -- with the reference build's occupied slots and wrapped keys and
    the set's premise.  world > 1: shard `rank` of the sharded layout."""
    p, b, off, o, keys, ref = _ref(set_name)
    v = g.table_view()
    slots = _host(v["slots"], v["n_slots"], "<i8").view(np.uint64)
    entries = _host(v["entries"], v["n_entries"], "<i4").view(np.uint32)
    shards, nsec = v["shards"], v["sectors_per_shard"]
    W = max(shards, world)
    assert nsec == sl.table_sectors(p.U, W), (nsec, p.U, W)
    st = table_ref.check_table(keys, slots, entries, nsec, shards, bits, rank, world)
    if W != p.world:
        return st
    if world > 1:        # one shard of the sharded layout: the slots of shard `rank` of the reference's gathered table
        seg = slice(rank * 4 * nsec, (rank + 1) * 4 * nsec)
        np.testing.assert_array_equal(slots != 0, ref.slots[seg] != 0)
        mine = sl.Layout(keys, slots, entries, nsec, 1)
        assert int(mine.wrapped().sum()) == ref.wrapped_per_shard()[rank]
        return st
    lay = sl.Layout(keys, slots, entries, nsec, shards)
    np.testing.assert_array_equal(slots != 0, ref.slots != 0)
    assert lay.wrapped_per_shard() == ref.wrapped_per_shard()
    st.update(sl.check_premise(p, o, lay, sequential=False))
    return st


def _with_env(name, value):
    if value is None:
        os.environ.pop(name, None)
    else:
        os.environ[name] = value


def _gpu(b, off, k, **options):
    g = api.Sage2Gpu(0)
    for key, value in options.items():
        g.set_option(key, value)
    g.run_steps123(b, off, k)
    return g


def run_one_context(set_name, bits=24, orders=(0, 1), phase_c_host=True):
    """both table builds x superstring scan on / off x read order; phase C through the host walk once"""
    p, b, off, o, keys, ref = _ref(set_name)
    st = {}
    try:
        for how in BUILDS:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            for fast in (1, 0):
                for order in orders:
                    g = _gpu(b, off, p.k, fast_scan=fast, read_order=order)
                    _compare(o, g)
                    st[how, fast, order] = g.counters()["fast_path_reads"]
            st[how] = check_layout(g, set_name, bits)
        _with_env("SAGE2GPU_TABLE_BUILD", None)
        if phase_c_host:
            _with_env("SAGE2GPU_PHASE_C_HOST", "1")
            g = _gpu(b, off, p.k)
            assert g.counters()["phase_c_on_device"] == 0
            _compare(o, g)
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)
        _with_env("SAGE2GPU_PHASE_C_HOST", None)
    return st


def _same_graph(o, gpus):
    assert sum(g.counters()["compare_calls"] for g in gpus) == o.compare_calls
    for g in gpus:
        e = g.edges()
        assert len(e) == o.n_edges
        for f in ("from", "to", "type", "delta", "delta_twin"):
            np.testing.assert_array_equal(e[f], o.edges[f])
        np.testing.assert_array_equal(g.extensions()["explored"], o.explored_b[1:])


def run_partitioned(set_name, bits=24):
    """every stage partitioned over the plan's world: the gathered table (world shards back to back) on every rank"""
    p, b, off, o, keys, ref = _ref(set_name)
    dev = torch.device("cuda", 0)
    tb, to = torch.from_numpy(b).to(dev), torch.from_numpy(off).to(dev)
    torch.cuda.synchronize()
    try:
        for how in BUILDS:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            gpus = [api.Sage2Gpu(0) for _ in range(p.world)]
            multi.run_local([multi.partitioned_graph_steps(g, r, p.world, multi.device_view_fn(dev), tb.data_ptr(), to.data_ptr(), len(off) - 1,
                                                           p.k, True) for r, g in enumerate(gpus)])
            _same_graph(o, gpus)
            for g in gpus:
                assert g.table_view()["shards"] == p.world
                check_layout(g, set_name, bits)
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)


def run_sharded(set_name, p2p, bits=24, builds=BUILDS):
    """the sharded layout at the plan's world: probes routed to the shard that owns the key; every shard checked"""
    p, b, off, o, keys, ref = _ref(set_name)
    world = p.world
    restarts = 0
    try:
        for how in builds:
            _with_env("SAGE2GPU_TABLE_BUILD", how)
            gpus = []
            for r in range(world):
                g = api.Sage2Gpu(0)
                g.load_reads(b, off, p.k)
                g.build_hash_table_shard(r, world)
                gpus.append(g)
            batch = 1000           # several routed batches
            if p2p:
                multi.run_local([multi.mailbox_steps(g, r, world, batch) for r, g in enumerate(gpus)])
            multi.run_local([multi.sharded_graph_steps(g, r, world, multi.device_view_fn(torch.device("cuda", 0)), batch, p2p=p2p)
                             for r, g in enumerate(gpus)])
            _same_graph(o, gpus)
            held = 0
            for r, g in enumerate(gpus):
                held += check_layout(g, set_name, bits, r, world)["keys"]
            assert held == keys.K
            restarts += sum(g.counters()["probe_restarts"] for g in gpus)
    finally:
        _with_env("SAGE2GPU_TABLE_BUILD", None)
    return restarts


# ---- the tests --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("set_name", SETS)
def test_one_context_equals_oracle(set_name):
    st = run_one_context(set_name)
    for how in BUILDS:
        for order in (0, 1):
            assert st[how, 1, order] > 0, (how, order, st)       # the scan's probe queue ran on these chains
    p = sl.get(*sl.parse(set_name))
    if p.world == 1:
        assert st["direct"]["wrapped"] == st["bucketed"]["wrapped"]


@pytest.mark.parametrize("set_name", SHARD_SETS)
def test_partitioned_gathered_table_equals_oracle(set_name):
    run_partitioned(set_name)


@pytest.mark.parametrize("p2p", [False, True])
@pytest.mark.parametrize("set_name", SHARD_SETS)
def test_sharded_layout_equals_oracle(set_name, p2p):
    run_sharded(set_name, p2p)


@pytest.mark.parametrize("layout", ["replicated", "sharded"])
@pytest.mark.parametrize("k", sl.KS)
def test_cli_wrap_end_equals_oracle_files(k, layout, tmp_path):
    """`sage2gpu --devices 0,0` on wrap_end written as FASTA: the `.reads` / `.graph3` bytes of the oracle"""
    from test_gpu_cli import BIN
    p, b, off, o, keys, ref = _ref(f"wrap_end_k{k}")
    fa = tmp_path / "in.fa"
    with open(fa, "wb") as f:
        for i, s in enumerate(p.reads):
            f.write(b">r%d\n%s\n" % (i, s))
    o.write_reads(str(tmp_path / "o.reads"))
    o.write_graph3(str(tmp_path / "o.graph3"))
    out = tmp_path / "out"
    env = dict(os.environ, SAGE2GPU_TABLE_LAYOUT=layout)
    subprocess.run([BIN, "-f", str(fa), "-k", str(k), "-o", str(out), "-p", "g", "-M", "3", "--devices", "0,0"], check=True, env=env,
                   timeout=600)
    for ext in ("reads", "graph3"):
        assert open(out / f"g.{ext}", "rb").read() == open(tmp_path / f"o.{ext}", "rb").read(), ext
    assert f"Table layout: {layout}" in open(out / "g.log").read()


# ---- narrow slot tags: the variant builds of test_gpu_tag_collisions.py ---------------------------------------------------
# At 8 and 0 tag bits a wrapped chain holds other keys with the same tag, so every walk has to tell them apart after the
# wrap: the scan's punt, probe_window in exact mode, the retry round's record compare and the routed proof.  Each variant
# runs in a child process that loaded its library (the fixture `variants` of test_gpu_tag_collisions.py).

TAG_SETS = [s for s in SETS if s.startswith(("wrap_end", "shard_ends"))]


def run_narrow_tags(bits, set_name):
    """one context with both builds, scan on / off; where the set is planned for shards, the gathered table and the sharded
    layout over both transports.  Every table checked at `bits` tag bits."""
    st = run_one_context(set_name, bits, orders=(0,), phase_c_host=False)
    if sl.world_of(sl.parse(set_name)[0]) > 1:
        run_partitioned(set_name, bits)
        st["restarts"] = run_sharded(set_name, False, bits) + run_sharded(set_name, True, bits, builds=["direct"])
    return st


@pytest.mark.parametrize("set_name", TAG_SETS)
@pytest.mark.parametrize("bits", WIDTHS)
def test_narrow_tags_equal_oracle(variants, bits, set_name):
    st = _in_child(variants, bits, run_narrow_tags, set_name)
    for how in BUILDS:
        assert st[how]["passed_same_tag"] > 0, st         # walks of the build pass another key with the same tag
    if "restarts" in st and bits == 0:
        assert st["restarts"] > 0, st                     # the routed tag probes met other keys: the verified pass ran
