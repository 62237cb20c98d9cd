"""GPU parity of the sharded-table build (SURVEY.md 8(e); include/sage2gpu.h "The table sharded by key hash"):
`world` contexts on ONE GPU hold one key-hash shard each, the exchanges of sage2_b200/multi.py are done in memory
(run_local), and every rank must end with the oracle's state: extension records, explored states, counters and
the edge list.  The same steps over NCCL on two real GPUs are in test_gpu_multi.py."""
import os

import numpy as np
import pytest
import torch

import datasets
import long_datasets
from oracle import oracle
from sage2_b200 import api, multi, synth
from test_gpu_parity import _compare, BIG

pytestmark = pytest.mark.gpu


def _sharded(name, world, batch_reads=1 << 19, p2p=False):
    if name in datasets.DATASETS:
        reads, k = datasets.get(name)
    elif name in long_datasets.LONG_DATASETS:
        reads, k = long_datasets.get(name)
    else:
        reads, k = synth.config(name)
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    dev = torch.device("cuda", 0)
    gpus = []
    for r in range(world):
        g = api.Sage2Gpu(0)
        g.load_reads(b, off, k)
        g.build_hash_table_shard(r, world)
        gpus.append(g)
    view = multi.device_view_fn(dev)
    if p2p:      # mailboxes of the other contexts: plain device pointers inside one process
        batch_reads = min(batch_reads, 1 << 14)
        multi.run_local([multi.mailbox_steps(g, r, world, batch_reads) for r, g in enumerate(gpus)])
    multi.run_local([multi.sharded_graph_steps(g, r, world, view, batch_reads, p2p=p2p) for r, g in enumerate(gpus)])
    return o, gpus


@pytest.mark.parametrize("name,world", [("clean", 1), ("rep", 2), ("hicopy", 3), ("deep", 2), ("varlen_err", 3), ("mixed", 4),
                                        ("tandem", 2), ("empty", 2), ("single", 3)])
def test_sharded_table_over_mailboxes_equals_oracle(name, world):
    """The peer-memory transport: queries stored by the routing kernel into the owners' mailboxes, answers copied back."""
    o, gpus = _sharded(name, world, p2p=True)
    assert sum(g.counters()["compare_calls"] for g in gpus) == o.compare_calls
    for g in gpus:
        e = g.edges()
        assert len(e) == o.n_edges
        for f in ("from", "to", "type", "delta", "delta_twin"):
            np.testing.assert_array_equal(e[f], o.edges[f])
        np.testing.assert_array_equal(g.extensions()["explored"], o.explored_b[1:])


@pytest.mark.parametrize("name,world", [("clean", 1), ("rep", 2), ("k70", 3), ("hicopy", 2), ("deep", 2), ("varlen_err", 3),
                                        ("deep_varlen", 2), ("tandem", 2), ("mixed", 4), ("err", 8), ("k31", 2),
                                        ("empty", 2), ("allbad", 2), ("single", 3)])
def test_sharded_table_equals_oracle(name, world):
    o, gpus = _sharded(name, world)
    calls = sum(g.counters()["compare_calls"] for g in gpus)
    keys = sum(g.counters()["distinct_keys"] for g in gpus)
    over = sum(g.counters()["keys_over_threshold"] for g in gpus)
    assert (calls, keys, over) == (o.compare_calls, o.distinct_keys, o.keys_over_threshold)
    for g in gpus:
        c = g.counters()
        c0 = dict(c)
        # per-rank counters that are sums over the ranks are checked above; patch them so _compare can check the rest
        g.counters = lambda c0=c0: {**c0, "compare_calls": o.compare_calls, "distinct_keys": o.distinct_keys,
                                    "keys_over_threshold": o.keys_over_threshold}
        _compare(o, g)


def test_small_batches_and_uneven_slices():
    o, gpus = _sharded("rep", 3, batch_reads=1000)
    for g in gpus:
        e = g.edges()
        assert len(e) == o.n_edges
        for f in ("from", "to", "type", "delta", "delta_twin"):
            np.testing.assert_array_equal(e[f], o.edges[f])


def test_sharded_context_refuses_the_local_search():
    reads, k = datasets.get("clean")
    b, off = synth.concat(reads)
    g = api.Sage2Gpu(0)
    g.load_reads(b, off, k)
    g.build_hash_table_shard(1, 2)
    with pytest.raises(api.Sage2GpuError):
        g.build_overlap_graph()


def test_cfg2_sharded_full_size():
    """cfg2 at full size over 4 shards on one GPU: the edge list equals the single-table build's AND the unmodified
    reference's (digests of its own `.reads` / `.graph3`, tests/golden/golden_big.json)."""
    reads, k = synth.config_cached("cfg2")
    b, off = synth.concat(reads)
    ref = api.Sage2Gpu(0)
    ref.run_steps123(b, off, k)
    want = ref.edges()
    want_calls = ref.counters()["compare_calls"]
    del ref
    world = 4
    gpus = []
    for r in range(world):
        g = api.Sage2Gpu(0)
        g.load_reads(b, off, k)
        g.build_hash_table_shard(r, world)
        gpus.append(g)
    view = multi.device_view_fn(torch.device("cuda", 0))
    multi.run_local([multi.sharded_graph_steps(g, r, world, view) for r, g in enumerate(gpus)])
    assert sum(g.counters()["compare_calls"] for g in gpus) == want_calls
    for g in gpus[:2]:
        e = g.edges()
        assert len(e) == len(want)
        for f in ("from", "to", "type", "delta", "delta_twin"):
            np.testing.assert_array_equal(e[f], want[f])
    for g in gpus:
        d = g.digest()
        assert d["edges"] == BIG["cfg2"]["edges_digest"] and d["reads"] == BIG["cfg2"]["reads_digest"]


def _host_gib():
    try:
        import psutil
        return psutil.virtual_memory().available / 2 ** 30
    except Exception:
        return 0.0


@pytest.mark.skipif(_host_gib() < 40, reason="cfg4 needs about 25 GiB of host memory for its 33 M synthetic reads")
def test_cfg4_sharded_equals_single_table():
    """cfg4 at full size (33.3 M reads, 27.9 M unique, 2 % repeats: masked keys, 94,560 reads left for phase C, host walk):
    the sharded build (one shard, peer-memory transport, 54 routed batches) gives the single-table build's edge list."""
    reads, k = synth.config_cached("cfg4")
    b, off = synth.concat(reads)
    del reads
    g = api.Sage2Gpu(0)
    g.run_steps123(b, off, k)
    want = g.edges()
    want_calls = g.counters()["compare_calls"]
    g.build_hash_table_shard(0, 1)
    multi.build_overlap_graph_sharded(g, 0, 1, torch.device("cuda", 0), batch_reads=1 << 19, p2p=True)
    c = g.counters()
    assert c["compare_calls"] == want_calls and c["n_edges"] == len(want)
    got = g.edges()
    for f in ("from", "to", "type", "delta", "delta_twin"):
        np.testing.assert_array_equal(got[f], want[f])
    if "cfg4" in BIG:      # ... and the unmodified reference's own result
        d = g.digest()
        assert d["edges"] == BIG["cfg4"]["edges_digest"] and d["reads"] == BIG["cfg4"]["reads_digest"]
        assert c["n_edges"] == BIG["cfg4"]["n_edges"]
