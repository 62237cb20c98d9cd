"""The CPU emulation of core.cuh (tests/host_emul.cpp) against the oracle on the long-read sets of tests/long_datasets.py:
every record stride from 2 to 32 words.  The GPU runs of the same sets are in test_gpu_long_reads.py."""
import numpy as np
import pytest

import emul
import long_datasets
from oracle import oracle
from sage2_b200 import synth
from test_host_emulation import compare_stage_outputs

STRIDES = (2, 3, 4, 5, 6, 8, 12, 16, 32)


def record_words(max_len: int) -> int:
    """reads.cu: words_for_len rounded up to a stride the kernels are instantiated for."""
    sw = max(2, (2 * max_len + 16 + 63) // 64)
    return next(s for s in STRIDES if s >= sw)


def test_sets_cover_every_wide_stride():
    got = {}
    for name in long_datasets.LONG_DATASETS:
        reads, _ = long_datasets.get(name)
        got[name] = record_words(max(len(r) for r in synth.to_list(reads)))
    assert got == long_datasets.SW
    assert set(got.values()) == {2, 6, 8, 12, 16, 32}


@pytest.mark.parametrize("name", list(long_datasets.LONG_DATASETS))
def test_emulated_pipeline_equals_oracle_on_long_reads(name):
    reads, k = long_datasets.get(name)
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    e = emul.EmuRun(b, off, k)
    assert o.U > 500 and o.n_edges > 500 and o.edges_inserted_c > 0
    if name == "hicopy250":
        assert o.keys_over_threshold > 0
    assert e.N == o.N
    assert e.over == o.keys_over_threshold
    assert e.distinct == o.distinct_keys
    assert e.compare_calls == o.compare_calls
    assert (e.contained, e.contained_size) == (o.contained_ext, o.contained_size)
    assert (e.inserted, e.removed) == (o.edges_inserted_c, o.transitive_removed)
    compare_stage_outputs(o, e.U, e.len, e.freq, e.F, e.RC, e.extR, e.extL, e.explored_b, e.edges, e.explored_a)


def test_records_of_every_stride_pack_and_reverse_complement():
    """core.cuh pack / revcomp at lengths around every stride boundary, in the widest record (32 words) too."""
    rng = np.random.default_rng(12)
    L = emul.lib()
    for length in (56, 57, 152, 153, 184, 185, 248, 249, 376, 377, 504, 505, 1015, 1016):
        s = bytes(rng.choice(list(b"ACGT"), size=length).astype(np.uint8))
        for SW in {record_words(length), 32}:
            f, r, want = (np.zeros(SW, np.uint64) for _ in range(3))
            L.hemu_pack(s, length, SW, f.ctypes.data, 0)
            L.hemu_pack(s, length, SW, want.ctypes.data, 1)
            L.hemu_revcomp(f.ctypes.data, r.ctypes.data, SW, length)
            np.testing.assert_array_equal(r, want)
            packed = np.zeros((length + 3) // 4, np.uint8)
            oracle.lib().sgo_chars_to_bytes(s, length, packed.ctypes.data)
            np.testing.assert_array_equal(emul.records_to_bytes(f[None, :], np.array([length])), packed)
