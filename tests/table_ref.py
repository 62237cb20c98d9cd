"""Reference of the prefix/suffix table (csrc/table.cu, csrc/core.cuh), restated from its definitions in numpy.

TEST INFRASTRUCTURE.  It does not include core.cuh: the constants and hash functions below are written out again so that a
change to the product's hashing or slot layout shows up as a difference here.

The table of a unique read set holds, for every read (0-based rid) and type t (0 fwd prefix, 1 fwd suffix, 2 revcomp
prefix, 3 revcomp suffix), the entry 4 * rid + t under the key of h = min(k, 64) bases that the type names.  The slot index
keeps one 64-bit slot per distinct key, grouped in sectors of 4:
    [63:40] tag = the low `tag_bits` bits of hash_key(v0, v1)   [39:33] min(n, 127)   [32:0] payload
with payload = the key's only entry (n = 1), an offset into entries[] where the key's n entries sit sorted (2 <= n <= 99),
or one of the key's entries (n >= 100, a masked key).  A key lives in the first slot that was free on the walk from its home
sector (mulhi(hash, sectors)), wrapping inside the shard that owns it.

check_table() tests these invariants, none of which depends on the order the keys were inserted in; build_sequential() is a
plain one-key-at-a-time inserter that satisfies them.
"""
from __future__ import annotations

import numpy as np

M64 = (1 << 64) - 1
THRESHOLD = 100          # hashTable.cpp:76: a key with this many entries is masked
SLOTS_PER_SECTOR = 4
PAYLOAD_MASK = np.uint64((1 << 33) - 1)

_u = np.uint64


def mix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        x = x ^ (x >> _u(33))
        x = x * _u(0xff51afd7ed558ccd)
        x = x ^ (x >> _u(33))
        x = x * _u(0xc4ceb9fe1a85ec53)
        return x ^ (x >> _u(33))


def hash_key(v0: np.ndarray, v1: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        return mix64(v1 ^ mix64(v0 + _u(0x9e3779b97f4a7c15)))


def home_sector(hsh: np.ndarray, nsec: int) -> np.ndarray:
    """high 64 bits of the 128-bit product hsh * nsec (nsec < 2^32)"""
    assert 0 < nsec < (1 << 32)
    n = _u(nsec)
    hi, lo = hsh >> _u(32), hsh & _u(0xFFFFFFFF)
    return (hi * n + ((lo * n) >> _u(32))) >> _u(32)


def slot_tag(hsh: np.ndarray, tag_bits: int) -> np.ndarray:
    return hsh & _u((1 << tag_bits) - 1)


def key_owner(hsh: np.ndarray, world: int) -> np.ndarray:
    """shard of a key: hash bits 24..33 modulo the number of shards"""
    if world <= 1:
        return np.zeros(len(hsh), np.int64)
    return (((hsh >> _u(24)) & _u(0x3FF)) % _u(world)).astype(np.int64)


def _bases(packed: np.ndarray, pos: np.ndarray) -> np.ndarray:
    """2-bit code of base `pos` of the reference's byte layout (4 bases per byte, first base in the top bits)"""
    return ((packed[pos >> 2] >> (6 - 2 * (pos & 3)).astype(np.uint8)) & 3).astype(np.uint64)


def _fold(packed: np.ndarray, start: np.ndarray, n: int) -> np.ndarray:
    v = np.zeros(len(start), np.uint64)
    for t in range(n):
        v = (v << _u(2)) | _bases(packed, start + t)
    return v


class Keys:
    """The 4U entries of a unique read set grouped by key (key ids in (hash, v0) order).

    fwd / rc: the reads in the reference's byte layout, read i at bytes [starts[i], ...); length: bases per read."""

    def __init__(self, fwd: np.ndarray, rc: np.ndarray, starts: np.ndarray, length: np.ndarray, h: int):
        length = np.asarray(length, np.int64)
        U = self.U = len(length)
        self.h = h
        assert U == 0 or length.min() >= h, "every unique read is at least h bases long"
        base0 = np.asarray(starts, np.int64)[:U] * 4
        v0 = np.zeros(4 * U, np.uint64)
        v1 = np.zeros(4 * U, np.uint64)
        for t in range(4):
            packed = rc if t & 2 else fwd
            s = base0 + (length - h if t & 1 else 0)
            if h <= 32:
                v1[t::4] = _fold(packed, s, h)
            else:
                v0[t::4] = _fold(packed, s, h - 32)
                v1[t::4] = _fold(packed, s + h - 32, 32)
        self.v0, self.v1 = v0, v1
        hsh = hash_key(v0, v1)
        # hash_key is a bijection of v1 for a fixed v0, so (hash, v0) identifies a key
        order = np.lexsort((np.arange(4 * U), v0, hsh))
        self.sorted_entries = order.astype(np.uint32)           # every key's entries, ascending = (rid, type) order
        new = np.ones(4 * U, bool)
        if U:
            new[1:] = (hsh[order][1:] != hsh[order][:-1]) | (v0[order][1:] != v0[order][:-1])
        self.first = np.flatnonzero(new)                         # key id -> its first position in sorted_entries
        K = self.K = len(self.first)
        self.n = np.diff(np.append(self.first, 4 * U))           # entries per key
        self.hash = hsh[order][self.first] if U else np.zeros(0, np.uint64)
        self.key_of_entry = np.empty(4 * U, np.int64)
        self.key_of_entry[order] = np.cumsum(new) - 1
        self.over_threshold = int((self.n >= THRESHOLD).sum())
        assert K == 0 or self.key_of_entry.max() == K - 1

    @classmethod
    def from_oracle(cls, o) -> "Keys":
        """oracle.OracleRun: 1-based arrays (byte_off[i] = first byte of read i)"""
        return cls(o.fwd, o.rc, o.byte_off[1:o.U + 1], o.length[1:], o.hash_len)

    @classmethod
    def from_reads(cls, r: dict, h: int) -> "Keys":
        """Sage2Gpu.reads(): 0-based arrays"""
        return cls(r["fwd"], r["rc"], r["byte_off"][:-1], r["length"], h)


def _slot_word(tag, count, payload) -> int:
    return (int(tag) << 40) | (min(int(count), 127) << 33) | int(payload)


def build_sequential(keys: Keys, nsec: int, shards: int = 1, tag_bits: int = 24, rank: int = 0, world: int = 1):
    """(slots, entries) of a table built one key at a time in key-id order.  shards > 1: the gathered layout (a key lives in
    shard key_owner(hash, shards)); world > 1: the shard `rank` of the sharded layout (only the keys it owns)."""
    slots = np.zeros(shards * nsec * SLOTS_PER_SECTOR, np.uint64)
    owner = key_owner(keys.hash, shards)
    home = home_sector(keys.hash, nsec).astype(np.int64)
    tags = slot_tag(keys.hash, tag_bits)
    owned = key_owner(keys.hash, world) == rank
    where = np.full(keys.K, -1, np.int64)
    for key in np.flatnonzero(owned):
        base, sec = int(owner[key]) * nsec, int(home[key])
        for _ in range(nsec):
            row = slots[(base + sec) * SLOTS_PER_SECTOR:(base + sec + 1) * SLOTS_PER_SECTOR]
            free = np.flatnonzero(row == 0)
            if len(free):
                where[key] = (base + sec) * SLOTS_PER_SECTOR + int(free[0])
                break
            sec = (sec + 1) % nsec
        assert where[key] >= 0, "slot index full"
        slots[where[key]] = 1           # occupied; the word is written below
    runs = []
    for s in np.sort(where[where >= 0]):
        key = int(np.flatnonzero(where == s)[0])
        n, f = int(keys.n[key]), int(keys.first[key])
        mine = keys.sorted_entries[f:f + n]
        if 2 <= n < THRESHOLD:
            slots[s] = _slot_word(tags[key], n, sum(len(r) for r in runs))
            runs.append(mine)
        else:
            slots[s] = _slot_word(tags[key], n, mine[0])
    entries = np.concatenate(runs).astype(np.uint32) if runs else np.zeros(0, np.uint32)
    return slots, entries


def check_table(keys: Keys, slots: np.ndarray, entries: np.ndarray, nsec: int, shards: int = 1, tag_bits: int = 24,
                rank: int = 0, world: int = 1) -> dict:
    """Assert that (slots, entries) is a table of `keys`.  shards > 1: gathered layout; world > 1: shard `rank` of the sharded
    layout.  Returns {"keys": keys held, "passed_same_tag": keys whose probe walk passes a slot of another key with the
    same tag (the collisions a search has to resolve)}."""
    slots = np.asarray(slots, np.uint64)
    entries = np.asarray(entries, np.uint32)
    assert len(slots) == shards * nsec * SLOTS_PER_SECTOR, (len(slots), shards, nsec)
    owned = key_owner(keys.hash, world) == rank
    K = int(owned.sum())

    occ = (slots != 0).reshape(-1, SLOTS_PER_SECTOR)
    bad = np.flatnonzero((occ[:, 1:] & ~occ[:, :-1]).any(axis=1))
    assert len(bad) == 0, f"empty slots are not a suffix of sector {bad[:5]}"

    at = np.flatnonzero(slots)
    word = slots[at]
    tag = word >> _u(40)
    cnt = ((word >> _u(33)) & _u(127)).astype(np.int64)
    pay = (word & PAYLOAD_MASK).astype(np.int64)

    # the key of every slot, through the entry its payload names
    run = (cnt >= 2) & (cnt < THRESHOLD)
    assert (pay[run] + cnt[run] <= len(entries)).all(), "entry run past the end of entries[]"
    assert (pay[~run] < 4 * keys.U).all(), "payload is not an entry"
    ent = pay.copy()
    ent[run] = entries[pay[run]]
    assert (ent < 4 * keys.U).all(), "run starts with something that is not an entry"
    key = keys.key_of_entry[ent]
    held = np.bincount(key, minlength=keys.K)
    stray = np.flatnonzero(held[~owned] if world > 1 else np.zeros(0, int))
    assert len(stray) == 0, f"{len(stray)} keys of other shards held by shard {rank} of {world}"
    twice = np.flatnonzero(held > 1)
    assert len(twice) == 0, f"{len(twice)} keys own more than one slot (e.g. key of entry {keys.sorted_entries[keys.first[twice[0]]]})"
    assert len(at) == K, f"{len(at)} occupied slots for {K} distinct keys"
    assert (held[owned] == 1).all(), "a key owns no slot"

    n = keys.n[key]
    assert (tag == slot_tag(keys.hash[key], tag_bits)).all(), "slot tag differs from the key's tag"
    assert (cnt == np.minimum(n, 127)).all(), "slot count differs from min(entries of the key, 127)"
    one = n == 1
    assert (pay[one] == keys.sorted_entries[keys.first[key[one]]]).all(), "single-entry slot names another entry"
    assert (run == ((n >= 2) & (n < THRESHOLD))).all()

    # 2..99 entries: the runs tile entries[] in some order, each the key's entries sorted by (rid, type)
    o = np.argsort(pay[run], kind="stable")
    starts, lens, rkey = pay[run][o], n[run][o], key[run][o]
    ends = np.cumsum(lens)
    assert int(ends[-1] if len(ends) else 0) == len(entries), f"runs cover {int(ends[-1]) if len(ends) else 0} of {len(entries)} entries"
    assert (starts == ends - lens).all(), "entry runs overlap or leave a gap"
    want = keys.sorted_entries[np.repeat(keys.first[rkey] - starts, lens) + np.arange(len(entries))] if len(entries) else entries
    bad = np.flatnonzero(entries != want)
    assert len(bad) == 0, f"entries[{bad[0] if len(bad) else 0}] out of place: a run is not the key's entries in (rid, type) order"

    # shard, then the walk from the home sector: no empty slot before the key's slot
    hsh = keys.hash[key]
    shard = at // (nsec * SLOTS_PER_SECTOR)
    assert (shard == key_owner(hsh, shards)).all(), "key in the wrong shard"
    home = home_sector(hsh, nsec).astype(np.int64)
    sec = at // SLOTS_PER_SECTOR - shard * nsec
    dist = ((sec - home) % nsec) * SLOTS_PER_SECTOR + at % SLOTS_PER_SECTOR
    ktag = slot_tag(hsh, tag_bits)
    passed = np.zeros(len(at), bool)
    for p in range(int(dist.max()) if len(dist) else 0):
        a = np.flatnonzero(dist > p)
        s = slots[(shard[a] * nsec + (home[a] + p // SLOTS_PER_SECTOR) % nsec) * SLOTS_PER_SECTOR + p % SLOTS_PER_SECTOR]
        assert (s != 0).all(), f"empty slot before the slot of {int((s == 0).sum())} keys on their walk from the home sector"
        passed[a] |= (s >> _u(40)) == ktag[a]
    return {"keys": K, "passed_same_tag": int(passed.sum())}
