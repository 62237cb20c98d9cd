"""CPU tests of tests/table_ref.py, the reference the GPU table is checked against: its keys agree with the oracle, a table
built one key at a time passes the check at every tag width and layout, and each kind of broken table fails it."""
import numpy as np
import pytest

import datasets
import table_ref
from oracle import oracle
from sage2_b200 import synth


def _keys(reads, k):
    b, off = synth.concat(reads)
    o = oracle.OracleRun(b, off, k)
    return table_ref.Keys.from_oracle(o), o


def _small():
    """~600 reads of a random genome and 130 reads that share their first 40 bases: one masked key (>= 100 entries)."""
    g = synth.random_genome(6_000, 41)
    reads = synth.to_list(synth.paired_reads(g, 100, 10, seed=42, mu=300, sigma=20, err_rate=0.002))
    rng = np.random.default_rng(43)
    head = b"ACGTTGCAAGCTTGCATGCCTGCAGGTCGACTCTAGAGGA"
    reads += [head + bytes(rng.choice(list(b"ACGT"), size=60).astype(np.uint8)) for _ in range(130)]
    return _keys(reads, 40)[0]


@pytest.fixture(scope="module")
def small():
    return _small()


@pytest.mark.parametrize("name", ["clean", "k31", "k70", "hicopy", "mixed", "varlen_err"])
def test_keys_agree_with_the_oracle(name):
    keys, o = _keys(*datasets.get(name))
    assert keys.K == o.distinct_keys
    assert keys.over_threshold == o.keys_over_threshold
    # the keys are the bases the type names: check a few against the reads themselves
    rid = np.arange(0, keys.U, max(1, keys.U // 50))
    codes = {0: o.fwd, 2: o.rc}
    for r in rid:
        L, s = int(o.length[r + 1]), int(o.byte_off[r + 1])
        for t in range(4):
            bits = np.unpackbits(codes[t & 2][s:s + (L + 3) // 4])
            seq = (bits[0:2 * L:2] * 2 + bits[1:2 * L:2]).astype(np.uint64)
            key = seq[L - o.hash_len:] if t & 1 else seq[:o.hash_len]
            v = 0
            for c in key:
                v = (v << 2) | int(c)
            assert (int(keys.v0[4 * r + t]) << 64 | int(keys.v1[4 * r + t])) == (v >> 64) << 64 | (v & table_ref.M64)


def test_hash_functions_match_their_definition():
    """mix64 / hash_key / home_sector against Python integers."""
    def mix(x):
        x ^= x >> 33; x = x * 0xff51afd7ed558ccd & table_ref.M64; x ^= x >> 33; x = x * 0xc4ceb9fe1a85ec53 & table_ref.M64
        return x ^ (x >> 33)
    rng = np.random.default_rng(7)
    v0 = rng.integers(0, 1 << 63, 200, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    v1 = rng.integers(0, 1 << 63, 200, dtype=np.uint64)
    h = table_ref.hash_key(v0, v1)
    for a, b, x in zip(v0.tolist(), v1.tolist(), h.tolist()):
        assert x == mix(b ^ mix((a + 0x9e3779b97f4a7c15) & table_ref.M64))
    for nsec in (256, 1001, (1 << 32) - 1):
        assert table_ref.home_sector(h, nsec).tolist() == [x * nsec >> 64 for x in h.tolist()]


@pytest.mark.parametrize("tag_bits", [24, 8, 0])
@pytest.mark.parametrize("shards,world", [(1, 1), (3, 1), (1, 2)])
def test_sequential_table_passes(small, tag_bits, shards, world):
    nsec = max(256, (6 * small.U + 3) // 4 // max(shards, world))
    for rank in range(world):
        slots, entries = table_ref.build_sequential(small, nsec, shards, tag_bits, rank, world)
        st = table_ref.check_table(small, slots, entries, nsec, shards, tag_bits, rank, world)
        assert st["keys"] == int((table_ref.key_owner(small.hash, world) == rank).sum())
        if tag_bits == 0:
            assert st["passed_same_tag"] > 0


# ---- each corruption is caught ------------------------------------------------------------------------------------

@pytest.fixture
def table(small):
    # a full index (load ~0.9): keys are displaced from their home sectors
    nsec = (small.K * 10 // 9 + 3) // 4
    slots, entries = table_ref.build_sequential(small, nsec, 1, 24)
    table_ref.check_table(small, slots, entries, nsec)
    return small, slots, entries, nsec


def _key_slot(keys, slots, entries, pred):
    """first occupied slot index whose key satisfies pred(key id, slot index)"""
    for s in np.flatnonzero(slots):
        w = int(slots[s])
        c, p = (w >> 33) & 127, w & ((1 << 33) - 1)
        e = int(entries[p]) if 2 <= c < 100 else p
        key = int(keys.key_of_entry[e])
        if pred(key, int(s)):
            return key, int(s)
    raise AssertionError("no such slot")


def _first_free(slots, sec):
    row = slots[4 * sec:4 * sec + 4]
    free = np.flatnonzero(row == 0)
    return 4 * sec + int(free[0]) if len(free) else None


def test_catches_a_duplicated_key_slot(table):
    keys, slots, entries, nsec = table
    _, s = _key_slot(keys, slots, entries, lambda k, s: keys.n[k] == 1)
    free = next(f for f in (_first_free(slots, x) for x in range(nsec)) if f is not None)
    slots[free] = slots[s]
    with pytest.raises(AssertionError, match="more than one slot"):
        table_ref.check_table(keys, slots, entries, nsec)


def test_catches_a_hole_before_a_key(table):
    keys, slots, entries, nsec = table
    home = table_ref.home_sector(keys.hash, nsec).astype(np.int64)

    def movable(k, s):      # last occupied slot of its home sector, and the next sector has room
        sec = s // 4
        return sec == home[k] and (s % 4 == 3 or slots[s + 1] == 0) and _first_free(slots, (sec + 1) % nsec) is not None
    _, s = _key_slot(keys, slots, entries, movable)
    dst = _first_free(slots, (s // 4 + 1) % nsec)
    slots[dst], slots[s] = slots[s], 0
    with pytest.raises(AssertionError, match="empty slot before"):
        table_ref.check_table(keys, slots, entries, nsec)


def test_catches_a_run_out_of_order(table):
    keys, slots, entries, nsec = table
    _, s = _key_slot(keys, slots, entries, lambda k, s: 2 <= keys.n[k] < 100)
    p = int(slots[s]) & ((1 << 33) - 1)
    entries[p], entries[p + 1] = entries[p + 1], entries[p]
    with pytest.raises(AssertionError, match="out of place"):
        table_ref.check_table(keys, slots, entries, nsec)


def test_catches_a_wrong_masked_representative(table):
    keys, slots, entries, nsec = table
    masked, s = _key_slot(keys, slots, entries, lambda k, s: keys.n[k] >= 100)
    other = int(np.flatnonzero(keys.key_of_entry != masked)[0])
    slots[s] = (int(slots[s]) & ~((1 << 33) - 1)) | other
    with pytest.raises(AssertionError, match="more than one slot|owns no slot"):
        table_ref.check_table(keys, slots, entries, nsec)


def test_catches_a_key_in_the_wrong_shard(small):
    nsec = max(256, small.K // 4)
    slots, entries = table_ref.build_sequential(small, nsec, 2, 24)
    table_ref.check_table(small, slots, entries, nsec, shards=2)
    owner = table_ref.key_owner(small.hash, 2)
    home = table_ref.home_sector(small.hash, nsec).astype(np.int64)

    def movable(k, s):      # a key of shard 0, last in its sector, whose home sector in shard 1 has room
        return owner[k] == 0 and (s % 4 == 3 or slots[s + 1] == 0) and _first_free(slots, nsec + home[k]) is not None
    key, s = _key_slot(small, slots, entries, movable)
    dst = _first_free(slots, nsec + home[key])
    slots[dst], slots[s] = slots[s], 0
    with pytest.raises(AssertionError, match="wrong shard"):
        table_ref.check_table(small, slots, entries, nsec, shards=2)
    # the sharded layout: a shard that holds a key another rank owns
    slots, entries = table_ref.build_sequential(small, nsec, 1, 24, rank=0, world=2)
    theirs, _ = table_ref.build_sequential(small, nsec, 1, 24, rank=1, world=2)
    for s in np.flatnonzero(theirs):
        w = int(theirs[s])
        if (w >> 33) & 127 == 1 and slots[s] == 0 and (s % 4 == 0 or slots[s - 1] != 0):
            slots[s] = w
            break
    else:
        pytest.fail("no free place for a key of the other shard")
    with pytest.raises(AssertionError, match="other shards"):
        table_ref.check_table(small, slots, entries, nsec, rank=0, world=2)
