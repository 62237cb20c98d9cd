"""The read sets of tests/slot_layouts.py without a GPU: each shows, on the reference table at the planned geometry, the
edge it was planned for (so that a change to the hashing or the sizing that quietly removes it fails here), and the CPU
emulation of the pipeline equals the oracle on it, in one context and as a sharded table."""
import functools

import numpy as np
import pytest

import emul
import slot_layouts as sl
import table_ref
from oracle import oracle
from sage2_b200 import multi, synth
from test_host_emulation import compare_stage_outputs
from test_sharded_emul import _check

# csrc/table.cu at the planned 3000 unique reads: 4U keys, load factor <= 2/3, a shard 1/world of it plus 10 %
PLANNED_NSEC = {1: 4500, 2: 2476, 3: 1651}
SETS = sl.set_names()


@functools.lru_cache(maxsize=None)
def _oracle(set_name):
    p = sl.get(*sl.parse(set_name))
    b, off = synth.concat(p.reads)
    return p, b, off, oracle.OracleRun(b, off, p.k)


def test_planned_geometry():
    assert sl.U_PLAN == 3000
    for w, n in PLANNED_NSEC.items():
        assert sl.table_sectors(sl.U_PLAN, w) == n


@pytest.mark.parametrize("set_name", SETS)
def test_reference_table_shows_the_premise(set_name):
    p, b, off, o = _oracle(set_name)
    assert p.nsec == PLANNED_NSEC[p.world]
    keys, lay = sl.reference(p, o)
    assert lay.dist.max() >= 6
    st = sl.check_premise(p, o, lay, sequential=True)
    if p.world > 1:      # the shards of the sharded layout: the same keys in the same places
        for r in range(p.world):
            slots, entries = table_ref.build_sequential(keys, p.nsec, rank=r, world=p.world)
            table_ref.check_table(keys, slots, entries, p.nsec, rank=r, world=p.world)
            np.testing.assert_array_equal(slots != 0, lay.slots[r * 4 * p.nsec:(r + 1) * 4 * p.nsec] != 0)


@pytest.mark.parametrize("set_name", SETS)
def test_emulation_equals_oracle(set_name):
    p, b, off, o = _oracle(set_name)
    e = emul.EmuRun(b, off, p.k)
    assert (e.distinct, e.over, e.compare_calls) == (o.distinct_keys, o.keys_over_threshold, o.compare_calls)
    compare_stage_outputs(o, e.U, e.len, e.freq, e.F, e.RC, e.extR, e.extL, e.explored_b, e.edges, e.explored_a)


@pytest.mark.parametrize("set_name", SETS)
def test_sharded_emulation_equals_oracle(set_name):
    p, b, off, o = _oracle(set_name)
    world = max(p.world, 2)
    shards = []
    for r in range(world):
        s = emul.EmuShard(b, off, p.k)
        s.build_hash_table_shard(r, world)
        shards.append(s)
    multi.run_local([multi.sharded_graph_steps(s, r, world, multi.host_view, 1000) for r, s in enumerate(shards)],
                    views_of=lambda r, bufs: emul.host_phase_a_views(bufs, world))
    assert sum(s.counters()["compare_calls"] for s in shards) == o.compare_calls
    assert sum(s.counters()["distinct_keys"] for s in shards) == o.distinct_keys
    for s in shards:
        _check(s.edges(), o)
        s.close()
